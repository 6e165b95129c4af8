// Voronoi neighbour lists of periodic structures in fp64: pymatgen's VoronoiNN(weight="solid_angle").get_voronoi_polyhedra
// + _extract_nn_info as called by the reference's compute_voronoi_neighbor (scann/utils/voronoi_neighbor.py:11-61).
//
// One warp per centre.  The cell of centre x_i within the point set S = {x_j + n L : |x_j + n L - x_i| <= cutoff} is
// built by clipping: it starts as a cube of half-size H = 1e5 * cutoff around x_i and is cut by the bisector plane of each
// point of S in ascending distance, until the next point is farther than twice the largest vertex distance (the
// security radius: a plane at distance d/2 cannot cut a cell whose vertices all lie within d/2, so every later point
// leaves the cell unchanged and the result is exact for S).
//
// Representation (the simple-polytope form of Ray et al., "Meshless Voronoi on the GPU", 2018, stored per facet
// rather than per dual triangle): every facet owns a slot holding its plane n.x <= w and its polygon as a cyclic list
// of edge labels, label k = the slot of the neighbouring facet across edge k -> k+1, counter-clockwise seen from
// outside.  Vertex k of facet s is the intersection of the three planes (s, label k-1, label k), so no coordinate is
// stored: every vertex is recomputed from its three planes, always with the planes in ascending slot order, so the
// three facets that share a vertex compute it bit for bit alike and classify it alike against a new plane.  That
// consistency keeps the combinatorics valid when four or more planes meet in a point (ideal lattices): such a point
// is a cluster of coincident degree-3 vertices joined by zero-length edges, and a facet that only touches the cell in
// that point collapses to coincident vertices (solid angle 0, dropped as pymatgen drops weight 0).
// Cutting by plane p: each facet whose vertices lie partly outside keeps its inside run plus two new vertices; the
// new facet's boundary is the cycle f -> succ(f) where succ(f) is the label of the edge along which f leaves p's
// half-space -- no geometry, only labels.
//
// Box size: a facet with an edge on the box (a label < 6) is unbounded in S: Qhull's "-1" vertex.  A bounded facet of
// S reaches the box only through a Voronoi vertex farther than H = 1e5 * cutoff from x_i, i.e. the centre of an empty
// sphere of that radius through x_i and three points within cutoff of it; those four points would have to be coplanar
// to about cutoff / 2e5 (7e-5 Angstrom at 13 Angstrom), far below what Qhull resolves as distinct.  The box vertices
// themselves never enter a result: a finite cell has none left, and a facet that touches the box is infinite.
// Precision: vertices come from 3x3 solves on planes of magnitude |x_j - x_i|, not from interpolation along edges,
// so the box size does not limit the accuracy of the finite cell.
#include <type_traits>

#include "common.cuh"

#define SCANN_ERR_VORONOI_COINCIDENT 32
#define SCANN_ERR_VORONOI_CAPACITY 64
#define SCANN_ERR_VORONOI_NO_FACET 128
#define SCANN_ERR_VORONOI_TOPOLOGY 256
#define VOR_INFINITE 1          // per-centre flag: the cell has an unbounded facet in S (host retries / drops it)

// The cell search comes in two forms, the same code at two capacities (vor_cells_kernel<F, V, WARPS>):
#define VOR_FMAX 64             // narrow form: facet slots per cell, slots 0..5 = the box
#define VOR_VMAX 32             //   vertices per facet
#define VOR_WARPS 4             //   centres per CTA
#define VOR_FMAX_WIDE 256       // wide form, for the centres whose cell overflows the narrow one (labels stay uint8_t)
#define VOR_VMAX_WIDE 64        //   vertices per facet (64-bit vertex masks)
#define VOR_WARPS_WIDE 1        //   centres per CTA: ~33 KB of shared memory per warp
#define VOR_CB 128              // candidates per distance band
#define VOR_IMG_MAX 511         // |n_k| of a packed image (10 bits per component)

struct VorFacet {               // one finite facet of a centre's cell (32 bytes; ScannVoronoiFacet in the header)
    double solid_angle, normalized, distance;
    int32_t site, image;        // image = (n0 + 512) | (n1 + 512) << 10 | (n2 + 512) << 20
};

// a set of vertices of one facet: one bit per vertex
template <int V> using VorMask = typename std::conditional<(V > 32), uint64_t, uint32_t>::type;
__device__ __forceinline__ int vor_popc(uint32_t m) { return __popc(m); }
__device__ __forceinline__ int vor_popc(uint64_t m) { return __popcll(m); }
__device__ __forceinline__ int vor_hibit(uint32_t m) { return 31 - __clz(m); }
__device__ __forceinline__ int vor_hibit(uint64_t m) { return 63 - __clzll(m); }

// One centre's cell: F facet slots of up to V vertices.
template <int F, int V>
struct VorWarp {
    double4 pl[F];              // facet plane: n.x <= w with x relative to the centre
    double cd2[VOR_CB];         // candidates of the current band
    int cj[VOR_CB], cimg[VOR_CB];
    int fsite[F], fimg[F];
    VorMask<V> omask[F];        // vertices outside the plane being inserted
    double edge[32];
    int hist[32];
    int ncol;
    uint8_t order[VOR_CB];
    uint8_t lab[F][V];
    uint8_t tmp[32][V];
    uint8_t nv[F];
    uint8_t succ[F];
};

__device__ __forceinline__ double3 d3sub(double3 a, double3 b) { return make_double3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ double d3dot(double3 a, double3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ double3 d3cross(double3 a, double3 b) {
    return make_double3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
// explicitly rounded forms (never contracted differently at different call sites): the quantities that decide a
// vertex's side of a plane or a candidate's band must come out bit for bit alike wherever they are computed
__device__ __forceinline__ double x3dot(double3 a, double3 b) {
    return __fma_rn(a.x, b.x, __fma_rn(a.y, b.y, __dmul_rn(a.z, b.z)));
}
__device__ __forceinline__ double3 x3cross(double3 a, double3 b) {
    return make_double3(__fma_rn(a.y, b.z, -__dmul_rn(a.z, b.y)), __fma_rn(a.z, b.x, -__dmul_rn(a.x, b.z)),
                        __fma_rn(a.x, b.y, -__dmul_rn(a.y, b.x)));
}

// Vertex of the planes of slots a, b, c, solved with the slots in ascending order, so that every facet sharing the
// vertex gets the same bits.
__device__ __forceinline__ double3 vor_vertex(const double4* pl, int a, int b, int c) {
    int s0 = min(a, min(b, c)), s2 = max(a, max(b, c)), s1 = a + b + c - s0 - s2;
    double4 P = pl[s0], Q = pl[s1], R = pl[s2];
    double3 p = make_double3(P.x, P.y, P.z), q = make_double3(Q.x, Q.y, Q.z), r = make_double3(R.x, R.y, R.z);
    double3 qr = x3cross(q, r), rp = x3cross(r, p), pq = x3cross(p, q);
    double inv = __drcp_rn(x3dot(p, qr));
    return make_double3(__dmul_rn(__fma_rn(P.w, qr.x, __fma_rn(Q.w, rp.x, __dmul_rn(R.w, pq.x))), inv),
                        __dmul_rn(__fma_rn(P.w, qr.y, __fma_rn(Q.w, rp.y, __dmul_rn(R.w, pq.y))), inv),
                        __dmul_rn(__fma_rn(P.w, qr.z, __fma_rn(Q.w, rp.z, __dmul_rn(R.w, pq.z))), inv));
}

// displacement x_j + n L - x_i (xyz) and its squared length (w): one definition for every pass over the candidates
__device__ __forceinline__ double4 vor_disp(const double* X, const double* L, double3 xi, int j, int n0, int n1, int n2) {
    double dx = __dadd_rn(__dadd_rn(X[3 * j], -xi.x), __fma_rn(n0, L[0], __fma_rn(n1, L[3], __dmul_rn(n2, L[6]))));
    double dy = __dadd_rn(__dadd_rn(X[3 * j + 1], -xi.y), __fma_rn(n0, L[1], __fma_rn(n1, L[4], __dmul_rn(n2, L[7]))));
    double dz = __dadd_rn(__dadd_rn(X[3 * j + 2], -xi.z), __fma_rn(n0, L[2], __fma_rn(n1, L[5], __dmul_rn(n2, L[8]))));
    return make_double4(dx, dy, dz, x3dot(make_double3(dx, dy, dz), make_double3(dx, dy, dz)));
}

__device__ __forceinline__ int vor_pack(int n0, int n1, int n2) {
    return (n0 + 512) | ((n1 + 512) << 10) | ((n2 + 512) << 20);
}

// Runs `fn(j, n0, n1, n2)` for every (site, image) whose image box can reach within `reach` of the centre, spread
// over the lanes.  lo / hi: the image range of site j along each lattice direction.
template <typename F>
__device__ __forceinline__ void vor_for_each_image(const double* X, const double* B, double3 xi, double3 reach,
                                                   int a0, int a1, int lane, F fn) {
    for (int j = a0; j < a1; ++j) {
        double3 d = make_double3(X[3 * j] - xi.x, X[3 * j + 1] - xi.y, X[3 * j + 2] - xi.z);
        int lo[3], cnt[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            double f = d.x * B[k] + d.y * B[3 + k] + d.z * B[6 + k];      // fractional coordinate k of x_j - x_i
            const double rk = k == 0 ? reach.x : k == 1 ? reach.y : reach.z;
            lo[k] = (int)floor(-rk - f);
            cnt[k] = (int)ceil(rk - f) - lo[k] + 1;
        }
        int total = cnt[0] * cnt[1] * cnt[2];
        for (int t = lane; t < total; t += 32) {
            int n2 = t % cnt[2], r = t / cnt[2];
            fn(j, lo[0] + r / cnt[1], lo[1] + r % cnt[1], lo[2] + n2);
        }
    }
}

// One warp per centre; lane l owns facet slots l, l + 32, ... (F / 32 of them).  The free slot a cut takes is the lowest
// free one, so a cell that fits in the narrow form gets the same slots, hence the same bits, from either form.
template <int F, int V, int WARPS>
__global__ void __launch_bounds__(32 * WARPS) vor_cells_kernel(
        const double* __restrict__ lattice, const double* __restrict__ coords, const int32_t* __restrict__ sa_off,
        const int32_t* __restrict__ centre_atom, const int32_t* __restrict__ centre_struct,
        const double* __restrict__ cutoff, int n_centres, int allow_pathological, int cap, VorFacet* __restrict__ slots,
        int32_t* __restrict__ slot_count, int32_t* __restrict__ centre_flags, int32_t* __restrict__ status) {
    static_assert(F % 32 == 0 && F <= 256 && V <= 64, "slot labels are uint8_t, vertex masks at most 64 bits");
    static_assert(sizeof(VorWarp<F, V>) * WARPS <= 48 * 1024, "static shared memory of a CTA");
    constexpr int P = F / 32;           // facet slots per lane
    using M = VorMask<V>;
    __shared__ VorWarp<F, V> sm[WARPS];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int c = blockIdx.x * WARPS + w;
    if (c >= n_centres) return;
    VorWarp<F, V>& W = sm[w];
    const int i = centre_atom[c], s = centre_struct[c];
    const int a0 = sa_off[s], a1 = sa_off[s + 1];
    double L[9], B[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) L[k] = lattice[9 * s + k];
    {   // B = L^-1 (rows of L are the lattice vectors; fractional = x B)
        double c0 = L[4] * L[8] - L[5] * L[7], c1 = L[5] * L[6] - L[3] * L[8], c2 = L[3] * L[7] - L[4] * L[6];
        double inv = 1.0 / (L[0] * c0 + L[1] * c1 + L[2] * c2);
        B[0] = c0 * inv; B[1] = (L[2] * L[7] - L[1] * L[8]) * inv; B[2] = (L[1] * L[5] - L[2] * L[4]) * inv;
        B[3] = c1 * inv; B[4] = (L[0] * L[8] - L[2] * L[6]) * inv; B[5] = (L[2] * L[3] - L[0] * L[5]) * inv;
        B[6] = c2 * inv; B[7] = (L[1] * L[6] - L[0] * L[7]) * inv; B[8] = (L[0] * L[4] - L[1] * L[3]) * inv;
    }
    const double3 xi = make_double3(coords[3 * i], coords[3 * i + 1], coords[3 * i + 2]);
    const double cut = cutoff[c], cut2 = cut * cut;
    const double3 reach = make_double3(cut * sqrt(B[0] * B[0] + B[3] * B[3] + B[6] * B[6]),
                                       cut * sqrt(B[1] * B[1] + B[4] * B[4] + B[7] * B[7]),
                                       cut * sqrt(B[2] * B[2] + B[5] * B[5] + B[8] * B[8]));
    int err = 0;

    // ---- the box: slot 2a (+axis a) / 2a+1 (-axis a); polygons counter-clockwise seen from outside
    const double H = 1e5 * fmax(cut, 1.0);
    for (int t = lane; t < F; t += 32) W.nv[t] = 0;
    __syncwarp();
    if (lane < 6) {
        int a = lane >> 1, pos = (lane & 1) == 0, b = (a + 1) % 3, cc = (a + 2) % 3;
        double n[3] = {0.0, 0.0, 0.0};
        n[a] = pos ? 1.0 : -1.0;
        W.pl[lane] = make_double4(n[0], n[1], n[2], H);
        uint8_t lb[4];
        if (pos) { lb[0] = 2 * cc + 1; lb[1] = 2 * b; lb[2] = 2 * cc; lb[3] = 2 * b + 1; }
        else     { lb[0] = 2 * b + 1; lb[1] = 2 * cc; lb[2] = 2 * b; lb[3] = 2 * cc + 1; }
        for (int k = 0; k < 4; ++k) W.lab[lane][k] = lb[k];
        W.nv[lane] = 4;
    }
    __syncwarp();

    // ---- candidates in ascending distance, in bands of at most VOR_CB
    double lo2 = -1.0;                    // the current band is (lo2, hi2]
    bool done = false;
    for (int band = 0; band < 4096 && !done && !err; ++band) {
        if (lo2 >= cut2) break;
        double hi2 = cut2;
        int n_in = 0;
        for (int refine = 0; refine < 64; ++refine) {
            const double base = fmax(lo2, 0.0);
            if (lane < 32) {
                W.edge[lane] = lane == 31 ? hi2 : base + (hi2 - base) * (lane + 1) / 32.0;
                W.hist[lane] = 0;
            }
            __syncwarp();
            int coinc = 0;
            vor_for_each_image(coords, B, xi, reach, a0, a1, lane, [&](int j, int n0, int n1, int n2) {
                if (j == i && n0 == 0 && n1 == 0 && n2 == 0) return;
                const double d2 = vor_disp(coords, L, xi, j, n0, n1, n2).w;
                if (d2 <= lo2 || d2 > hi2) return;
                if (d2 < 1e-16) coinc = 1;
                int b = 0;                                  // first edge >= d2
#pragma unroll
                for (int step = 16; step > 0; step >>= 1)
                    if (W.edge[b + step - 1] < d2) b += step;
                atomicAdd(&W.hist[b], 1);
            });
            __syncwarp();
            if (__any_sync(0xffffffffu, coinc)) { err |= SCANN_ERR_VORONOI_COINCIDENT; break; }
            int h = W.hist[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {              // inclusive prefix sum over the bins
                int v = __shfl_up_sync(0xffffffffu, h, o);
                if (lane >= o) h += v;
            }
            unsigned fit = __ballot_sync(0xffffffffu, h <= VOR_CB);
            if (fit == 0) {                                 // the first bin alone overflows: narrow the band
                double nh = W.edge[0];
                __syncwarp();
                if (!(nh < hi2) || nh - base <= 1e-14 * nh) { err |= SCANN_ERR_VORONOI_CAPACITY; break; }
                hi2 = nh;
                continue;
            }
            int last = 31 - __clz(fit);                     // counts are monotone: fit is a prefix of the lanes
            hi2 = W.edge[last];
            n_in = __shfl_sync(0xffffffffu, h, last);
            __syncwarp();
            break;
        }
        if (err) break;
        // collect (lo2, hi2]
        if (lane == 0) W.ncol = 0;
        __syncwarp();
        int big = 0;
        vor_for_each_image(coords, B, xi, reach, a0, a1, lane, [&](int j, int n0, int n1, int n2) {
            if (j == i && n0 == 0 && n1 == 0 && n2 == 0) return;
            const double d2 = vor_disp(coords, L, xi, j, n0, n1, n2).w;
            if (d2 <= lo2 || d2 > hi2) return;
            if (max(abs(n0), max(abs(n1), abs(n2))) > VOR_IMG_MAX) { big = 1; return; }
            int slot = atomicAdd(&W.ncol, 1);
            if (slot < VOR_CB) { W.cd2[slot] = d2; W.cj[slot] = j; W.cimg[slot] = vor_pack(n0, n1, n2); }
        });
        __syncwarp();
        const int ncol = W.ncol;
        if (__any_sync(0xffffffffu, big) || ncol != n_in) { err |= SCANN_ERR_VORONOI_CAPACITY; break; }
        // rank sort by (distance, site, image): keys are unique
        for (int t = lane; t < ncol; t += 32) {
            double d = W.cd2[t];
            int jj = W.cj[t], im = W.cimg[t], r = 0;
            for (int u = 0; u < ncol; ++u) {
                double du = W.cd2[u];
                r += du < d || (du == d && (W.cj[u] < jj || (W.cj[u] == jj && W.cimg[u] < im)));
            }
            W.order[r] = (uint8_t)t;
        }
        __syncwarp();

        for (int q = 0; q < ncol && !err; ++q) {
            const int t = W.order[q];
            const int jj = W.cj[t], im = W.cimg[t];
            const int n0 = (im & 1023) - 512, n1 = ((im >> 10) & 1023) - 512, n2 = ((im >> 20) & 1023) - 512;
            const double4 ed = vor_disp(coords, L, xi, jj, n0, n1, n2);
            const double3 e = make_double3(ed.x, ed.y, ed.z);
            const double d2 = ed.w, off = 0.5 * d2;
            // A vertex counts as outside only beyond 1e-11 |e| (|e| + |v|_1), a few hundred times the rounding of
            // v.e - |e|^2/2: vertices that lie on the plane up to rounding -- a cluster where many planes meet (the centre
            // of a cospherical shell), or a line shared by the planes of coplanar neighbours (a fullerene's rings), out to
            // where it meets the box -- then stay inside together instead of splitting the outside region or cutting
            // along a line of dependent planes.  A cut that shallow changes no solid angle by more than ~1e-10 relative.
            const double tol = 1e-11 * sqrt(d2);
            // classify every vertex against the new plane; largest vertex distance of the current cell
            double r2 = 0.0;
            int nonfinite = 0;
            for (int h = 0; h < P; ++h) {
                const int f = lane + 32 * h, n = W.nv[f];
                M m = 0;
                for (int k = 0; k < n; ++k) {
                    double3 v = vor_vertex(W.pl, f, W.lab[f][k == 0 ? n - 1 : k - 1], W.lab[f][k]);
                    r2 = fmax(r2, x3dot(v, v));
                    const double scale = __dmul_rn(tol, __dadd_rn(sqrt(d2), fabs(v.x) + fabs(v.y) + fabs(v.z)));
                    if (!(fabs(v.x) + fabs(v.y) + fabs(v.z) < INFINITY)) nonfinite = 1;     // planes without one point
                    if (__dadd_rn(x3dot(v, e), -off) > scale) m |= M(1) << k;
                }
                W.omask[f] = m;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) r2 = fmax(r2, __shfl_xor_sync(0xffffffffu, r2, o));
            if (__any_sync(0xffffffffu, nonfinite)) { err |= SCANN_ERR_VORONOI_TOPOLOGY; break; }
            if (d2 > 4.0 * r2) { done = true; break; }      // security radius reached: S adds nothing more
            bool any = false;
            for (int h = 0; h < P; ++h) any |= W.omask[lane + 32 * h] != 0;
            if (!__any_sync(0xffffffffu, any)) continue;
            // a free slot for the new facet (free before this cut): the lowest one
            int p;
            if constexpr (P == 2) {                           // the narrow form as it always was: the same SASS
                bool fr0 = lane >= 6 && W.nv[lane] == 0, fr1 = W.nv[lane + 32] == 0;
                unsigned b0 = __ballot_sync(0xffffffffu, fr0), b1 = __ballot_sync(0xffffffffu, fr1);
                if (!b0 && !b1) { err |= SCANN_ERR_VORONOI_CAPACITY; break; }
                p = b0 ? __ffs(b0) - 1 : 32 + __ffs(b1) - 1;
            } else {
                p = -1;
                for (int h = P - 1; h >= 0; --h) {
                    const unsigned b = __ballot_sync(0xffffffffu, (h > 0 || lane >= 6) && W.nv[lane + 32 * h] == 0);
                    if (b) p = 32 * h + __ffs(b) - 1;
                }
                if (p < 0) { err |= SCANN_ERR_VORONOI_CAPACITY; break; }
            }
            // cut every facet: the inside run plus the entry and exit vertices
            int bad = 0, npart = 0, first = -1;
            for (int h = 0; h < P; ++h) {
                const int f = lane + 32 * h, n = W.nv[f];
                const M m = W.omask[f];
                if (m == 0 || n == 0) continue;
                const M full = n == V ? ~M(0) : (M(1) << n) - M(1);
                if (m == full) { W.nv[f] = 0; continue; }
                int runs = 0, kx = 0;
                for (int k = 0; k < n; ++k) {
                    int k1 = k + 1 == n ? 0 : k + 1;
                    if (!((m >> k) & 1) && ((m >> k1) & 1)) { ++runs; kx = k; }
                }
                const int nin = n - vor_popc(m);
                if (runs != 1) { bad |= SCANN_ERR_VORONOI_TOPOLOGY; continue; }
                if (nin + 2 > V) { bad |= SCANN_ERR_VORONOI_CAPACITY; continue; }
                int kin = kx - nin + 1;                       // first inside vertex of the run ending at kx
                if (kin < 0) kin += n;
                int o = 0;
                W.tmp[lane][o++] = W.lab[f][kin == 0 ? n - 1 : kin - 1];      // entry vertex
                for (int k = kin, c2 = 0; c2 < nin; ++c2, k = k + 1 == n ? 0 : k + 1) W.tmp[lane][o++] = W.lab[f][k];
                W.tmp[lane][o++] = (uint8_t)p;                                 // exit vertex
                W.succ[f] = W.lab[f][kx];
                for (int k = 0; k < o; ++k) W.lab[f][k] = W.tmp[lane][k];
                W.nv[f] = (uint8_t)o;
                ++npart;
                if (first < 0) first = f;
            }
            bad = __reduce_or_sync(0xffffffffu, bad);
            npart = __reduce_add_sync(0xffffffffu, npart);
            first = __reduce_min_sync(0xffffffffu, first < 0 ? 0x7fffffff : first);
            __syncwarp();
            if (!bad && npart == 0) bad = SCANN_ERR_VORONOI_TOPOLOGY;
            if (bad) { err |= bad; break; }
            if (lane == 0) {                                  // the new facet's boundary: f -> succ(f)
                int f = first, k = 0;
                do { if (k < V) W.lab[p][k] = (uint8_t)f; ++k; f = W.succ[f]; } while (f != first && k <= F);
                if (k > V) err |= SCANN_ERR_VORONOI_CAPACITY;
                else if (f != first || k != npart) err |= SCANN_ERR_VORONOI_TOPOLOGY;
                W.nv[p] = err ? 0 : (uint8_t)k;
                W.pl[p] = make_double4(e.x, e.y, e.z, off);
                W.fsite[p] = jj - a0;
                W.fimg[p] = im;
            }
            err = __shfl_sync(0xffffffffu, err, 0);
            __syncwarp();
        }
        lo2 = hi2;
    }

    // ---- finite facets: solid angle (pymatgen's fan formula), distance, site, image
    int flags = 0, nkeep = 0;
    double sa[P] = {};
    bool keep[P] = {};
    if (!err) {
        bool inf = false;
        for (int h = 0; h < P; ++h) {
            const int f = lane + 32 * h, n = W.nv[f];
            if (f < 6 || n == 0) continue;
            bool touches = false;
            for (int k = 0; k < n; ++k) touches |= W.lab[f][k] < 6;
            if (touches) { inf = true; continue; }
            // drop coincident consecutive vertices (a cluster of degree-3 vertices is one point of the cell)
            const double tol2 = 1e-18 * W.pl[f].w * 2.0;      // (1e-9 * |x_j - x_i|)^2
            M kept = 0;
            double3 v0 = vor_vertex(W.pl, f, W.lab[f][n - 1], W.lab[f][0]), prev = v0;
            kept = 1;
            int nk = 1, lastk = 0;
            for (int k = 1; k < n; ++k) {
                double3 v = vor_vertex(W.pl, f, W.lab[f][k - 1], W.lab[f][k]), dv = d3sub(v, prev);
                if (d3dot(dv, dv) > tol2) { kept |= M(1) << k; prev = v; ++nk; lastk = k; }
            }
            while (nk > 1) {                                  // trailing vertices that coincide with the first
                double3 v = vor_vertex(W.pl, f, W.lab[f][lastk - 1], W.lab[f][lastk]), dv = d3sub(v, v0);
                if (d3dot(dv, dv) > tol2) break;
                kept &= ~(M(1) << lastk);
                --nk;
                lastk = vor_hibit(kept);
            }
            if (nk < 3) continue;
            double3 r0 = v0, rk = v0;
            double n0 = sqrt(d3dot(r0, r0)), nkk = n0, ang = 0.0;
            int seen = 0;
            for (int k = 1; k < n; ++k) {
                if (!((kept >> k) & 1)) continue;
                double3 r1 = vor_vertex(W.pl, f, W.lab[f][k - 1], W.lab[f][k]);
                double n1 = sqrt(d3dot(r1, r1));
                if (seen++) {
                    double tp = fabs(d3dot(r0, d3cross(rk, r1)));
                    double de = n0 * nkk * n1 + n1 * d3dot(r0, rk) + nkk * d3dot(r0, r1) + n0 * d3dot(rk, r1);
                    double a = de == 0.0 ? (tp > 0.0 ? 0.5 * M_PI : -0.5 * M_PI) : atan(tp / de);
                    ang += (a > 0.0 ? a : a + M_PI) * 2.0;
                }
                rk = r1;
                nkk = n1;
            }
            sa[h] = ang;
            keep[h] = ang > 0.0;
        }
        if (__any_sync(0xffffffffu, inf)) flags |= VOR_INFINITE;
        double mx = sa[0];
        for (int h = 1; h < P; ++h) mx = fmax(mx, sa[h]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        const bool emit = allow_pathological || !(flags & VOR_INFINITE);
        if (emit) {
            int base = 0;
            for (int h = 0; h < P; ++h) {
                unsigned bal = __ballot_sync(0xffffffffu, keep[h]);
                if (keep[h]) {
                    const int k = base + __popc(bal & ((1u << lane) - 1u));
                    const int f = lane + 32 * h;
                    if (k < cap) {
                        VorFacet r;
                        r.solid_angle = sa[h];
                        r.normalized = sa[h] / mx;
                        r.distance = sqrt(2.0 * W.pl[f].w);
                        r.site = W.fsite[f];
                        r.image = W.fimg[f];
                        slots[(size_t)c * cap + k] = r;
                    }
                }
                base += __popc(bal);
            }
            nkeep = base;
            if (nkeep > cap) err |= SCANN_ERR_VORONOI_CAPACITY;
            else if (nkeep == 0) err |= SCANN_ERR_VORONOI_NO_FACET;
        }
    }
    if (lane == 0) {
        slot_count[c] = err ? 0 : min(nkeep, cap);
        centre_flags[c] = flags | err;
        if (err) atomicOr(status, err);
    }
}

// ---- per-centre slots -> CSR: off[c] = sum of the counts before c (one CTA), then a parallel copy
__global__ void __launch_bounds__(1024) vor_scan_kernel(const int32_t* __restrict__ count, int n, int32_t* __restrict__ off) {
    __shared__ int wsum[32];
    __shared__ int carry;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    if (t == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < n; base += 1024) {
        int v = base + t < n ? count[base + t] : 0, x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) wsum[w] = x;
        __syncthreads();
        if (w == 0) {
            int s = wsum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int y = __shfl_up_sync(0xffffffffu, s, o);
                if (lane >= o) s += y;
            }
            wsum[lane] = s;
        }
        __syncthreads();
        const int incl = x + (w ? wsum[w - 1] : 0) + carry;
        if (base + t < n) off[base + t] = incl - v;
        __syncthreads();
        if (t == 1023) carry = incl;
        __syncthreads();
    }
    if (t == 0) off[n] = carry;
}

__global__ void vor_compact_kernel(const VorFacet* __restrict__ slots, const int32_t* __restrict__ count,
                                   const int32_t* __restrict__ off, int n, int cap, VorFacet* __restrict__ rec) {
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (c >= n) return;
    const int k = count[c], o = off[c];
    for (int t = lane; t < k; t += 32) rec[o + t] = slots[(size_t)c * cap + t];
}

// Byte size of the result blob of n centres with `cap` slots each (include/scann_b200.h).
static size_t vor_header_bytes(int n) { return (((size_t)(2 * n + 1) * 4) + 31) / 32 * 32; }

extern "C" int scann_voronoi_neighbors(const double* lattice, const double* coords, const int32_t* struct_atom_off,
                                       const int32_t* centre_atom, const int32_t* centre_struct, const double* cutoff,
                                       int n_centres, int allow_pathological, int cap, void* slots, int32_t* slot_count,
                                       void* blob, void* host_blob, int32_t* status, void* stream) {
    if (n_centres < 0 || cap <= 0 || cap > VOR_FMAX_WIDE) {
        scann_set_error("scann_voronoi_neighbors: n_centres %d, cap %d (1..%d)", n_centres, cap, VOR_FMAX_WIDE);
        return 1;
    }
    if (n_centres == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    int32_t* off = (int32_t*)blob;
    int32_t* flags = off + n_centres + 1;
    VorFacet* rec = (VorFacet*)((char*)blob + vor_header_bytes(n_centres));
    if (cap <= VOR_FMAX)        // the narrow form
        vor_cells_kernel<VOR_FMAX, VOR_VMAX, VOR_WARPS><<<(n_centres + VOR_WARPS - 1) / VOR_WARPS, 32 * VOR_WARPS, 0, st>>>(
            lattice, coords, struct_atom_off, centre_atom, centre_struct, cutoff, n_centres, allow_pathological, cap,
            (VorFacet*)slots, slot_count, flags, status);
    else                        // the wide form
        vor_cells_kernel<VOR_FMAX_WIDE, VOR_VMAX_WIDE, VOR_WARPS_WIDE>
            <<<(n_centres + VOR_WARPS_WIDE - 1) / VOR_WARPS_WIDE, 32 * VOR_WARPS_WIDE, 0, st>>>(
            lattice, coords, struct_atom_off, centre_atom, centre_struct, cutoff, n_centres, allow_pathological, cap,
            (VorFacet*)slots, slot_count, flags, status);
    vor_scan_kernel<<<1, 1024, 0, st>>>(slot_count, n_centres, off);
    vor_compact_kernel<<<(n_centres + 7) / 8, 256, 0, st>>>((const VorFacet*)slots, slot_count, off, n_centres, cap, rec);
    if (int rc = scann_check_launch("scann_voronoi_neighbors")) return rc;
    if (host_blob) {
        size_t bytes = vor_header_bytes(n_centres) + (size_t)n_centres * cap * sizeof(VorFacet);
        cudaError_t e = cudaMemcpyAsync(host_blob, blob, bytes, cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) {
            scann_set_error("scann_voronoi_neighbors: copy of the result: %s", cudaGetErrorString(e));
            return 2;
        }
    }
    return 0;
}

// ---- facet records -> the model's neighbour lists ---------------------------------------------------------------
// What the host does per centre between the cell search and the model's input (voronoi.py voronoi_polyhedra +
// compute_voronoi_neighbors, DataIterator): order the facets by (distance, site, n0, n1, n2), keep distance <= d_thresh
// and normalised solid angle >= w_thresh (fp64), and write (site, (float)weight, (float)distance).
#define VOR_SEL_WARPS 8
#define VOR_SEL 64              // staging slots per atom row: the most neighbours an atom keeps
#define VOR_SEL_MAX VOR_FMAX_WIDE   // records per centre (the wide cell search's capacity)

// Facet a before facet b in the host's np.lexsort order.  The image components compare as stored: (x & 1023) and
// (x & 1023) - 512 order alike, but the packed word itself would compare n2 first.
__device__ __forceinline__ bool vor_before(double da, int sa, int ia, double db, int sb, int ib) {
    if (da != db) return da < db;
    if (sa != sb) return sa < sb;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int na = (ia >> (10 * k)) & 1023, nb = (ib >> (10 * k)) & 1023;
        if (na != nb) return na < nb;
    }
    return false;
}

// The select of a centre with more records than two per lane: each lane ranks its records against all of the centre's
// records in global memory (rare: only centres of the wide cell search).  Out of line, so that it leaves the register
// allocation of the two-per-lane code alone.
__device__ __noinline__ void vor_select_wide(const VorFacet* __restrict__ rec, int k, double d_thresh, double w_thresh,
                                             int column, int lane, int r, int32_t* __restrict__ sel_count,
                                             int32_t* __restrict__ sel_idx, float* __restrict__ sel_w,
                                             float* __restrict__ sel_d, int32_t* __restrict__ status) {
    const size_t row = (size_t)r * VOR_SEL;
    int kept = 0;
    for (int i = lane; i < k; i += 32) {
        const VorFacet ri = rec[i];
        if (!(ri.distance <= d_thresh && ri.normalized >= w_thresh)) continue;
        int rank = 0;
        for (int j = 0; j < k; ++j) {
            const double dj = rec[j].distance;
            if (j == i || !(dj <= d_thresh && rec[j].normalized >= w_thresh)) continue;
            const int sj = rec[j].site, ij = rec[j].image;
            rank += vor_before(dj, sj, ij, ri.distance, ri.site, ri.image) ||
                    (j < i && !vor_before(ri.distance, ri.site, ri.image, dj, sj, ij));
        }
        if (rank < VOR_SEL) {
            sel_idx[row + rank] = ri.site;
            sel_w[row + rank] = __double2float_rn(column ? ri.normalized : ri.solid_angle);
            sel_d[row + rank] = __double2float_rn(ri.distance);
        }
        ++kept;
    }
    kept = __reduce_add_sync(0xffffffffu, kept);
    if (lane == 0) {
        sel_count[r] = kept;                    // the true count: more than VOR_SEL is an error the host reports
        if (kept > VOR_SEL) atomicOr(status, SCANN_ERR_VORONOI_CAPACITY);
    }
}

// One warp per centre; the rank of a kept record is the number of kept records before it in the host's order (ties,
// which would be one facet listed twice, by record position: a stable sort).  Up to 64 records: two per lane, ranked
// in shared memory.  65..256 records (a centre of the wide cell search): a loop over the lane's records, ranked against
// the records in global memory; more than 64 kept ones write their true count and set the capacity bit.
// Min. blocks 1: with the out-of-line call and no min. blocks, ptxas (CUDA 12.9, sm_100a) gives the kernel 32 registers
// and spills 8 bytes; with it, 40 registers and no spill.
__global__ void __launch_bounds__(32 * VOR_SEL_WARPS, 1) vor_select_kernel(
        const int32_t* __restrict__ off, const VorFacet* __restrict__ rec, const int32_t* __restrict__ centre_row, int n,
        double d_thresh, double w_thresh, int column, int32_t* __restrict__ sel_count, int32_t* __restrict__ sel_idx,
        float* __restrict__ sel_w, float* __restrict__ sel_d, int32_t* __restrict__ status) {
    __shared__ double s_d[VOR_SEL_WARPS][VOR_SEL];
    __shared__ int s_site[VOR_SEL_WARPS][VOR_SEL], s_img[VOR_SEL_WARPS][VOR_SEL];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int c = blockIdx.x * VOR_SEL_WARPS + w;
    if (c >= n) return;                         // whole warps only: the kernel has no block-level barrier
    const int o = off[c];
    int k = off[c + 1] - o;
    if (k > VOR_SEL_MAX) {
        if (lane == 0) atomicOr(status, SCANN_ERR_VORONOI_CAPACITY);
        k = VOR_SEL_MAX;
    }
    if (k > VOR_SEL) {                          // warp-uniform
        vor_select_wide(rec + o, k, d_thresh, w_thresh, column, lane, centre_row[c], sel_count, sel_idx, sel_w, sel_d,
                        status);
        return;
    }
    VorFacet r[2];
    bool keep[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int i = lane + 32 * h;
        keep[h] = false;
        if (i < k) {
            r[h] = rec[o + i];
            keep[h] = r[h].distance <= d_thresh && r[h].normalized >= w_thresh;
            // a dropped record takes no part in the ranking: site -1 marks it
            s_d[w][i] = r[h].distance;
            s_site[w][i] = keep[h] ? r[h].site : -1;
            s_img[w][i] = r[h].image;
        }
    }
    __syncwarp();
    const size_t row = (size_t)centre_row[c] * VOR_SEL;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int i = lane + 32 * h;
        if (!keep[h]) continue;
        const double di = r[h].distance;
        const int si = r[h].site, ii = r[h].image;
        int rank = 0;
        for (int j = 0; j < k; ++j) {
            const int sj = s_site[w][j];
            if (sj < 0 || j == i) continue;
            const double dj = s_d[w][j];
            const int ij = s_img[w][j];
            rank += vor_before(dj, sj, ij, di, si, ii) || (j < i && !vor_before(di, si, ii, dj, sj, ij));
        }
        sel_idx[row + rank] = si;
        sel_w[row + rank] = __double2float_rn(column ? r[h].normalized : r[h].solid_angle);
        sel_d[row + rank] = __double2float_rn(di);
    }
    const int kept = __popc(__ballot_sync(0xffffffffu, keep[0])) + __popc(__ballot_sync(0xffffffffu, keep[1]));
    if (lane == 0) sel_count[centre_row[c]] = kept;
}

extern "C" int scann_voronoi_select(const void* blob, const int32_t* centre_row, int n_centres, double d_thresh,
                                    double w_thresh, int weight_column, int32_t* sel_count, int32_t* sel_idx,
                                    float* sel_w, float* sel_d, int32_t* status, void* stream) {
    if (n_centres < 0 || (weight_column != 0 && weight_column != 1)) {
        scann_set_error("scann_voronoi_select: n_centres %d, weight_column %d (0 or 1)", n_centres, weight_column);
        return 1;
    }
    if (n_centres == 0) return 0;
    const int32_t* off = (const int32_t*)blob;
    const VorFacet* rec = (const VorFacet*)((const char*)blob + vor_header_bytes(n_centres));
    vor_select_kernel<<<(n_centres + VOR_SEL_WARPS - 1) / VOR_SEL_WARPS, 32 * VOR_SEL_WARPS, 0, (cudaStream_t)stream>>>(
        off, rec, centre_row, n_centres, d_thresh, w_thresh, weight_column, sel_count, sel_idx, sel_w, sel_d, status);
    return scann_check_launch("scann_voronoi_select");
}

// One warp per atom of the batch: its selected neighbours -> nbr_idx / nbr_w / nbr_d at atom_nbr_off[atom]; lane 0
// raises the structure's largest count (integer atomics: the result does not depend on the order).  The first threads
// also write the batch's struct_atom_off and z.
__global__ void vor_batch_fill_kernel(const int32_t* __restrict__ sa, const int32_t* __restrict__ z, int s0, int n_structs,
                                      int a0, int A, const int32_t* __restrict__ sel_count, const int32_t* __restrict__ sel_idx,
                                      const float* __restrict__ sel_w, const float* __restrict__ sel_d,
                                      const int32_t* __restrict__ an, int32_t* __restrict__ sa_out,
                                      int32_t* __restrict__ z_out, int32_t* __restrict__ idx_out,
                                      float* __restrict__ w_out, float* __restrict__ d_out, int32_t* __restrict__ sizes) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t <= n_structs) sa_out[t] = sa[s0 + t] - a0;
    const int a = t >> 5, lane = t & 31;
    if (a >= A) return;
    const int row = a0 + a, k = sel_count[row], p = an[a];
    for (int i = lane; i < min(k, VOR_SEL); i += 32) {    // k > VOR_SEL: select has flagged the centre
        idx_out[p + i] = sel_idx[(size_t)row * VOR_SEL + i];
        w_out[p + i] = sel_w[(size_t)row * VOR_SEL + i];
        d_out[p + i] = sel_d[(size_t)row * VOR_SEL + i];
    }
    if (lane == 0) {
        z_out[a] = z[row];
        int lo = s0, hi = s0 + n_structs - 1;           // structure of the atom: last s with sa[s] <= row
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (sa[mid] <= row) lo = mid; else hi = mid - 1;
        }
        atomicMax(&sizes[lo - s0], k);
        atomicAdd(&sizes[n_structs + lo - s0], k);
    }
}

extern "C" int scann_voronoi_batch_csr(const int32_t* struct_atom_off, const int32_t* z, int s0, int n_structs,
                                       int atom0, int n_atoms, const int32_t* sel_count, const int32_t* sel_idx,
                                       const float* sel_w, const float* sel_d, void* csr, long long off_sa,
                                       long long off_an, long long off_z, long long off_idx, long long off_w,
                                       long long off_d, int32_t* sizes, void* stream) {
    if (n_structs <= 0 || n_atoms < 0 || s0 < 0 || atom0 < 0) {
        scann_set_error("scann_voronoi_batch_csr: s0 %d, n_structs %d, atom0 %d, n_atoms %d", s0, n_structs, atom0,
                        n_atoms);
        return 1;
    }
    cudaStream_t st = (cudaStream_t)stream;
    char* p = (char*)csr;
    int32_t* an = (int32_t*)(p + off_an);
    cudaError_t e = cudaMemsetAsync(sizes, 0, sizeof(int32_t) * 2 * (size_t)n_structs, st);
    if (e != cudaSuccess) {
        scann_set_error("scann_voronoi_batch_csr: %s", cudaGetErrorString(e));
        return 2;
    }
    vor_scan_kernel<<<1, 1024, 0, st>>>(sel_count + atom0, n_atoms, an);
    const long long threads = max((long long)n_atoms * 32, (long long)n_structs + 1);
    vor_batch_fill_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(
        struct_atom_off, z, s0, n_structs, atom0, n_atoms, sel_count, sel_idx, sel_w, sel_d, an, (int32_t*)(p + off_sa),
        (int32_t*)(p + off_z), (int32_t*)(p + off_idx), (float*)(p + off_w), (float*)(p + off_d), sizes);
    return scann_check_launch("scann_voronoi_batch_csr");
}
