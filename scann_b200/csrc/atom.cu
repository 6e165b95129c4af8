// Per-atom ("row") kernels: input embedding, geometry initialisation, blocked dense GEMM with
// fused epilogues, weight-gradient GEMM, LayerNorm backward, small utilities.
//
// fp32 SIMT implementations.  Row r = b*M + m addresses atom m of structure b; every
// per-atom tensor is [R,128] row-major.  Weight blocks are [128,128] row-major (Keras Dense
// kernels are [in,out], used as x @ W + b; the 384x128 filter_geo kernel is three stacked
// blocks, attention.py:142-151).
#include "common.cuh"

// ---------------------------------------------------------------------------------------------
// Input embedding: x0 = swish([emb[Z] | ring @ Wr + br] @ We + be)      (scann_model.py:361-374)
// ---------------------------------------------------------------------------------------------
#define EMB_ROWS 8
__global__ void __launch_bounds__(128) embed_fwd_kernel(const int32_t* __restrict__ atomic,
                                                        const float* __restrict__ ring, int R, int E, int n_atoms,
                                                        const float* __restrict__ emb, const float* __restrict__ Wr,
                                                        const float* __restrict__ br, const float* __restrict__ We,
                                                        const float* __restrict__ be, float* __restrict__ t0,
                                                        float* __restrict__ x0, int32_t* __restrict__ status,
                                                        const ScannDropCtl* __restrict__ drop,
                                                        const float* __restrict__ emb_rows) {
    extern __shared__ float s_cat[];   // [EMB_ROWS][Kin]
    const int Kin = E + (ring ? 10 : 0);
    const int r0 = blockIdx.x * EMB_ROWS;
    pdl_wait();
    pdl_trigger();      // only after the own wait: at most one kernel ahead becomes resident early
    for (int i = threadIdx.x; i < EMB_ROWS * Kin; i += blockDim.x) {
        int rr = i / Kin, k = i % Kin, r = r0 + rr;
        float v = 0.f;
        if (r < R) {
            if (k < E && emb_rows) {
                v = emb_rows[(size_t)r * E + k];            // feature == "cgcnn": Dense(92 -> E) output of this row
            } else if (k < E) {
                int z = atomic[r];
                if (z < 0 || z >= n_atoms) { atomicOr(status, SCANN_ERR_BAD_ATOMIC); z = 0; }
                v = emb[(size_t)z * E + k];
            } else {
                int kk = k - E;
                v = br[kk] + ring[(size_t)r * 2] * Wr[kk] + ring[(size_t)r * 2 + 1] * Wr[10 + kk];
            }
        }
        s_cat[i] = v;
    }
    __syncthreads();
    const int n = threadIdx.x;
    float acc[EMB_ROWS];
    const float b = be[n];
#pragma unroll
    for (int i = 0; i < EMB_ROWS; ++i) acc[i] = b;
    for (int k = 0; k < Kin; ++k) {
        float w = __ldg(We + (size_t)k * SCANN_D + n);
#pragma unroll
        for (int i = 0; i < EMB_ROWS; ++i) acc[i] = fmaf(s_cat[i * Kin + k], w, acc[i]);
    }
#pragma unroll
    for (int i = 0; i < EMB_ROWS; ++i) {
        int r = r0 + i;
        if (r < R) {
            if (t0) t0[(size_t)r * SCANN_D + n] = acc[i];
            x0[(size_t)r * SCANN_D + n] = swish_f(acc[i]) * drop_mult(drop, 0u, (uint32_t)r * SCANN_D + n);
        }
    }
}

// Backward, stage 1: d_t0 = d_x0 * swish'(t0); per-species sums G[z][:] += d_t0[r][:],
// G[n_atoms+0][:] = sum over all rows (= d be), G[n_atoms+1+c][:] += ring[r][c] * d_t0[r][:].
__global__ void __launch_bounds__(128) embed_bwd_gather_kernel(const int32_t* __restrict__ atomic,
                                                               const float* __restrict__ ring, int R, int n_atoms,
                                                               const float* __restrict__ t0,
                                                               const float* __restrict__ dx0, float* __restrict__ G,
                                                               int rows_per_cta, const ScannDropCtl* __restrict__ drop) {
    const int n = threadIdx.x;
    int r0 = blockIdx.x * rows_per_cta, r1 = min(R, r0 + rows_per_cta);
    float all = 0.f, g0 = 0.f, g1 = 0.f;
    float run = 0.f;
    int zrun = -1;
    // rows in batches of 8: the loads of a batch are independent and issued together (the run-length logic with
    // its atomics otherwise keeps the compiler from overlapping them: 32 dependent round trips per thread)
    for (int rb = r0; rb < r1; rb += 8) {
        float dv[8], tv[8];
        int zv[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int r = min(rb + q, r1 - 1);
            dv[q] = dx0[(size_t)r * SCANN_D + n];
            tv[q] = t0[(size_t)r * SCANN_D + n];
            zv[q] = atomic[r];
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int r = rb + q;
            if (r >= r1) break;
            const float d = dv[q] * drop_mult(drop, 0u, (uint32_t)r * SCANN_D + n) * swish_grad_f(tv[q]);
            int z = zv[q];
            z = (z < 0 || z >= n_atoms) ? 0 : z;
            if (z != zrun) {
                if (zrun >= 0) atomicAdd(G + (size_t)zrun * SCANN_D + n, run);
                zrun = z;
                run = 0.f;
            }
            run += d;
            all += d;
            if (ring) {
                g0 = fmaf(ring[(size_t)r * 2], d, g0);
                g1 = fmaf(ring[(size_t)r * 2 + 1], d, g1);
            }
        }
    }
    if (zrun >= 0) atomicAdd(G + (size_t)zrun * SCANN_D + n, run);
    atomicAdd(G + (size_t)n_atoms * SCANN_D + n, all);
    if (ring) {
        atomicAdd(G + (size_t)(n_atoms + 1) * SCANN_D + n, g0);
        atomicAdd(G + (size_t)(n_atoms + 2) * SCANN_D + n, g1);
    }
}

// Deterministic form of stage 1: thread n owns column n of every per-species row of the CTA's partial G (shared
// memory, rows in order, no atomics); the partial goes to slot blockIdx.x of Gs ([grid][n_atoms + 3][128]).
__global__ void __launch_bounds__(128) embed_bwd_gather_det_kernel(const int32_t* __restrict__ atomic,
                                                                   const float* __restrict__ ring, int R, int n_atoms,
                                                                   const float* __restrict__ t0,
                                                                   const float* __restrict__ dx0, float* __restrict__ Gs,
                                                                   int rows_per_cta, const ScannDropCtl* __restrict__ drop) {
    extern __shared__ float s_g[];                       // [n_atoms + 3][128]
    const int n = threadIdx.x, nrow = n_atoms + 3;
    for (int z = 0; z < nrow; ++z) s_g[z * SCANN_D + n] = 0.f;
    const int r0 = blockIdx.x * rows_per_cta, r1 = min(R, r0 + rows_per_cta);
    for (int r = r0; r < r1; ++r) {
        const float d = dx0[(size_t)r * SCANN_D + n] * drop_mult(drop, 0u, (uint32_t)r * SCANN_D + n) *
                        swish_grad_f(t0[(size_t)r * SCANN_D + n]);
        int z = atomic[r];
        z = (z < 0 || z >= n_atoms) ? 0 : z;
        s_g[z * SCANN_D + n] += d;
        s_g[n_atoms * SCANN_D + n] += d;
        if (ring) {
            s_g[(n_atoms + 1) * SCANN_D + n] = fmaf(ring[(size_t)r * 2], d, s_g[(n_atoms + 1) * SCANN_D + n]);
            s_g[(n_atoms + 2) * SCANN_D + n] = fmaf(ring[(size_t)r * 2 + 1], d, s_g[(n_atoms + 2) * SCANN_D + n]);
        }
    }
    float* slot = Gs + (size_t)blockIdx.x * nrow * SCANN_D;
    for (int z = 0; z < nrow; ++z) slot[z * SCANN_D + n] = s_g[z * SCANN_D + n];
}

// G[i] = sum over the nslots slots of Gs, in slot order (eight loads in flight)
__global__ void __launch_bounds__(128) embed_bwd_slot_sum_kernel(const float* __restrict__ Gs, int nslots, int count,
                                                                 float* __restrict__ G) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    float s = 0.f;
    int k = 0;
    for (; k + 8 <= nslots; k += 8) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = Gs[(size_t)(k + u) * count + i];
#pragma unroll
        for (int u = 0; u < 8; ++u) s += v[u];
    }
    for (; k < nslots; ++k) s += Gs[(size_t)k * count + i];
    G[i] = s;
}

// Backward, stage 2 (tiny): dWe = [emb^T G ; br (x) G_all + Wr^T G2], dbe = G_all,
// d_emb = G We[:E]^T, dWr = G2 We[E:]^T, dbr = G_all We[E:]^T.  Gradients are ACCUMULATED.
__global__ void __launch_bounds__(128) embed_bwd_final_kernel(int E, int n_atoms, int has_ring,
                                                              const float* __restrict__ emb,
                                                              const float* __restrict__ Wr,
                                                              const float* __restrict__ br,
                                                              const float* __restrict__ We,
                                                              const float* __restrict__ G, float* __restrict__ d_emb,
                                                              float* __restrict__ dWr, float* __restrict__ dbr,
                                                              float* __restrict__ dWe, float* __restrict__ dbe) {
    const int n = threadIdx.x;
    const int Kin = E + (has_ring ? 10 : 0);
    const float* Gall = G + (size_t)n_atoms * SCANN_D;
    const float* G2 = G + (size_t)(n_atoms + 1) * SCANN_D;
    // block b handles row k of dWe (k < Kin), then the small dot-product outputs
    for (int k = blockIdx.x; k < Kin; k += gridDim.x) {
        float acc = 0.f;
        if (k < E) {
            for (int z = 0; z < n_atoms; ++z) acc = fmaf(emb[(size_t)z * E + k], G[(size_t)z * SCANN_D + n], acc);
        } else {
            int kk = k - E;
            acc = br[kk] * Gall[n] + Wr[kk] * G2[n] + Wr[10 + kk] * G2[SCANN_D + n];
        }
        dWe[(size_t)k * SCANN_D + n] += acc;
    }
    if (blockIdx.x == 0) dbe[n] += Gall[n];
    // dot products of length 128 across the block: outputs (z,k<E), (c,kk), (kk)
    __shared__ float s_red[4];
    int n_out = n_atoms * E + (has_ring ? 30 : 0);
    for (int o = blockIdx.x; o < n_out; o += gridDim.x) {
        const float* gv;
        const float* wv;
        float* dst;
        if (o < n_atoms * E) {
            int z = o / E, k = o % E;
            gv = G + (size_t)z * SCANN_D;
            wv = We + (size_t)k * SCANN_D;
            dst = d_emb + (size_t)z * E + k;
        } else {
            int q = o - n_atoms * E;   // 0..19 -> dWr[c][kk], 20..29 -> dbr[kk]
            int kk = q % 10, c = q / 10;
            gv = (c < 2) ? (G2 + (size_t)c * SCANN_D) : Gall;
            wv = We + (size_t)(E + kk) * SCANN_D;
            dst = (c < 2) ? (dWr + c * 10 + kk) : (dbr + kk);
        }
        float p = warp_sum(gv[n] * wv[n]);
        if ((n & 31) == 0) s_red[n >> 5] = p;
        __syncthreads();
        if (n == 0) *dst += s_red[0] + s_red[1] + s_red[2] + s_red[3];
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// feature == "cgcnn" (scann_model.py:364-365): embed_atom = Dense(92 -> E) over per-atom feature vectors instead
// of an Embedding lookup.  Small general kernels (this variant is rare; nothing here is performance critical).
// ---------------------------------------------------------------------------------------------
#define CG_KMAX 144        // embedding_dim (<= 128) + 10 ring columns, rounded up: row stride of d_cat
// out[r, k] = sum_f A[r, f] W[f, k] + b[k]      (A [R,F], W [F,K], K <= 128)
__global__ void __launch_bounds__(128) small_dense_fwd_kernel(const float* __restrict__ A, const float* __restrict__ W,
                                                              const float* __restrict__ b, int R, int F, int K,
                                                              float* __restrict__ out) {
    pdl_wait();
    pdl_trigger();
    const int k = threadIdx.x;
    for (int r = blockIdx.x; r < R; r += gridDim.x) {
        if (k >= K) continue;
        float acc = b ? b[k] : 0.f;
        for (int f = 0; f < F; ++f) acc = fmaf(A[(size_t)r * F + f], W[(size_t)f * K + k], acc);
        out[(size_t)r * K + k] = acc;
    }
}
// General embedding backward, stage 1 (32 rows per CTA): d_t0 = dx0 * dropout * swish'(t0);
// dWe[k, :] += cat[r, k] d_t0[r, :], dbe += d_t0, d_cat[r, k] = <d_t0[r, :], We[k, :]>  with
// cat[r, :] = [emb_rows[r, :E] | br + ring[r] @ Wr].
// DET (deterministic mode): the CTA's dWe rows and dbe go to its slot of dWe, a [grid][(Kin + 1) * 128] array
// (dWe rows, then dbe; dbe unused).
template <bool DET>
__global__ void __launch_bounds__(128) embed_bwd_rows_kernel(const float* __restrict__ emb_rows,
                                                             const float* __restrict__ ring, int R, int E,
                                                             const float* __restrict__ Wr, const float* __restrict__ br,
                                                             const float* __restrict__ We, const float* __restrict__ t0,
                                                             const float* __restrict__ dx0, float* __restrict__ d_cat,
                                                             float* __restrict__ dWe, float* __restrict__ dbe,
                                                             const ScannDropCtl* __restrict__ drop) {
    __shared__ float s_dt[32][SCANN_D];
    __shared__ float s_cat[32][CG_KMAX];
    const int n = threadIdx.x, Kin = E + (ring ? 10 : 0);
    const int r0 = blockIdx.x * 32;
    float bsum = 0.f;
    for (int i = 0; i < 32; ++i) {
        const int r = r0 + i;
        float d = 0.f;
        if (r < R)
            d = dx0[(size_t)r * SCANN_D + n] * drop_mult(drop, 0u, (uint32_t)r * SCANN_D + n) *
                swish_grad_f(t0[(size_t)r * SCANN_D + n]);
        s_dt[i][n] = d;
        bsum += d;
        for (int k = n; k < Kin; k += 128) {
            float c = 0.f;
            if (r < R) {
                if (k < E) c = emb_rows[(size_t)r * E + k];
                else { const int kk = k - E; c = br[kk] + ring[(size_t)r * 2] * Wr[kk] + ring[(size_t)r * 2 + 1] * Wr[10 + kk]; }
            }
            s_cat[i][k] = c;
        }
    }
    __syncthreads();
    float* slot = dWe + (size_t)blockIdx.x * (Kin + 1) * SCANN_D;
    if constexpr (DET) slot[(size_t)Kin * SCANN_D + n] = bsum;
    else atomicAdd(dbe + n, bsum);
    for (int k = 0; k < Kin; ++k) {
        float acc = 0.f;
#pragma unroll 8
        for (int i = 0; i < 32; ++i) acc = fmaf(s_cat[i][k], s_dt[i][n], acc);
        if constexpr (DET) slot[(size_t)k * SCANN_D + n] = acc;
        else atomicAdd(dWe + (size_t)k * SCANN_D + n, acc);
    }
    // d_cat[r, k]: thread k, loop over the CTA's rows
    for (int k = n; k < Kin; k += 128) {
        for (int i = 0; i < 32 && r0 + i < R; ++i) {
            float acc = 0.f;
            for (int c = 0; c < SCANN_D; ++c) acc = fmaf(s_dt[i][c], We[(size_t)k * SCANN_D + c], acc);
            d_cat[(size_t)(r0 + i) * CG_KMAX + k] = acc;
        }
    }
}
// stage 2: dW_emb[f, k] += sum_r A92[r, f] d_cat[r, k] ; db_emb[k] += sum_r d_cat[r, k] ; ring Dense likewise.
// grid = F + 1 (+ 3 with ring) CTAs, 128 threads (k).
__global__ void __launch_bounds__(128) embed_bwd_cols_kernel(const float* __restrict__ A92, const float* __restrict__ ring,
                                                            int R, int F, int E, const float* __restrict__ d_cat,
                                                            float* __restrict__ dWemb, float* __restrict__ dbemb,
                                                            float* __restrict__ dWr, float* __restrict__ dbr) {
    const int k = threadIdx.x, f = blockIdx.x;
    float acc = 0.f;
    if (f <= F) {
        if (k >= E) return;
        for (int r = 0; r < R; ++r) acc = fmaf(f < F ? A92[(size_t)r * F + f] : 1.0f, d_cat[(size_t)r * CG_KMAX + k], acc);
        if (f < F) dWemb[(size_t)f * E + k] += acc; else dbemb[k] += acc;
    } else {
        const int c = f - F - 1;          // 0, 1: ring rows of Wr ; 2: br
        if (k >= 10) return;
        for (int r = 0; r < R; ++r) acc = fmaf(c < 2 ? ring[(size_t)r * 2 + c] : 1.0f, d_cat[(size_t)r * CG_KMAX + E + k], acc);
        if (c < 2) dWr[c * 10 + k] += acc; else dbr[k] += acc;
    }
}
// Batches that carry atomic numbers: embed_atom's output for an atom is row Z of emb_table = table @ W + b, so its
// gradients are dW[f, k] += sum_z table[z, f] d_emb[z, k] and db[k] += sum_z d_emb[z, k], with d_emb the per-element
// sums of embed_bwd_final_kernel.  grid = F + 1 CTAs (the last one: db), thread k; z ascending (deterministic).
__global__ void __launch_bounds__(128) cgcnn_table_bwd_kernel(const float* __restrict__ table,
                                                              const float* __restrict__ d_emb, int Z, int F, int E,
                                                              float* __restrict__ dW, float* __restrict__ db) {
    const int k = threadIdx.x, f = blockIdx.x;
    if (k >= E) return;
    float acc = 0.f;
    if (f < F) {
        for (int z = 0; z < Z; ++z) acc = fmaf(table[(size_t)z * F + f], d_emb[(size_t)z * E + k], acc);
        dW[(size_t)f * E + k] += acc;
    } else {
        for (int z = 0; z < Z; ++z) acc += d_emb[(size_t)z * E + k];
        db[k] += acc;
    }
}

// ---------------------------------------------------------------------------------------------
// Geometry initialisation (g_update): g0 = swish(rbf_d Wd + bd) * swish(rbf_w Ww + bw)
// rbf_x[k] = exp(-(x - c_k)^2 / 0.25)                 (scann_model.py:378-389, custom_layers.py:55-65)
// and the geometry filter of a g_update = False layer: g' = swish(rbf_d Wf + bf) * w   (attention.py:155)
// ---------------------------------------------------------------------------------------------
// The four kernels below walk the pair rows in CHUNKS of GEOM_CR = 64 rows, whatever the tile stride of the plan
// (rows = ntiles * stride, a multiple of 32; padding rows have pair_c < 0 and may sit anywhere in a chunk).  Per chunk:
// four threads per row fetch the row's (centre, distance, weight) with unconditional loads -- one round trip -- and
// write its Gaussians as 16-byte vectors; after ONE barrier thread (n = tid % 128, half = tid / 128) runs over the rows
// half, half + 2, ... with its weight column in registers and the Gaussians read as LDS.128 broadcasts.
// (Round 2, first form: one 32-row tile per round, 32 threads fetching centre -> distance / weight as two dependent
// round trips, three barriers per tile, an integer division per Gaussian: noupdate_geom_fwd 72 us and noupdate_geom_bwd
// 194 us per layer on the PtGP shape (132 031 pairs), a third of that train step -- gpurun_out/r02ch_launches.csv.)
#define GEOM_CR 64

template <int NC>   // 20: Gaussians of the distance; 40: distance | Voronoi weight
__device__ __forceinline__ void geom_stage_chunk(float (*s_rbf)[2 * SCANN_RBF], int* s_c, float* s_w,
                                                 const int32_t* __restrict__ pair_c, const float* __restrict__ pair_d,
                                                 const float* __restrict__ pair_w, const float* __restrict__ cd,
                                                 const float* __restrict__ cw, size_t base, int nrows) {
    const int row = threadIdx.x & (GEOM_CR - 1), part = threadIdx.x >> 6;
    int c = -1;
    float d = 0.f, w = 0.f;
    if (row < nrows) { c = pair_c[base + row]; d = pair_d[base + row]; w = pair_w[base + row]; }
    if (part == 0) { s_c[row] = c; s_w[row] = c >= 0 ? w : 0.f; }
    for (int j = part; j < NC / 4; j += 4) {                 // 16-byte vector j of the row: Gaussians 4j .. 4j + 3
        const bool dist = 4 * j < SCANN_RBF;
        const float x = dist ? d : w;
        const float* cc = dist ? cd + 4 * j : cw + (4 * j - SCANN_RBF);
        const float d0 = x - cc[0], d1 = x - cc[1], d2 = x - cc[2], d3 = x - cc[3];
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c >= 0) v = make_float4(expf(-(d0 * d0) / 0.25f), expf(-(d1 * d1) / 0.25f), expf(-(d2 * d2) / 0.25f),
                                    expf(-(d3 * d3) / 0.25f));
        *reinterpret_cast<float4*>(&s_rbf[row][4 * j]) = v;
    }
    __syncthreads();
}
// rows of chunk ch and its first row
#define GEOM_CHUNK_LOOP(NT, STRIDE)                                                                       \
    const long long total_rows = (long long)(NT) * (STRIDE);                                              \
    const int nchunks = (int)((total_rows + GEOM_CR - 1) / GEOM_CR);                                      \
    for (int ch = blockIdx.x; ch < nchunks; ch += gridDim.x)
#define GEOM_CHUNK_ROWS(ch) ((int)(total_rows - (long long)(ch) * GEOM_CR < GEOM_CR ? total_rows - (long long)(ch) * GEOM_CR : GEOM_CR))

__global__ void __launch_bounds__(256) geom_init_fwd_kernel(const int32_t* __restrict__ ntiles, int stride,
                                                            const int32_t* __restrict__ pair_c,
                                                            const float* __restrict__ pair_d,
                                                            const float* __restrict__ pair_w,
                                                            const float* __restrict__ cd, const float* __restrict__ cw,
                                                            const float* __restrict__ Wd, const float* __restrict__ bd,
                                                            const float* __restrict__ Ww, const float* __restrict__ bw,
                                                            float* __restrict__ g0) {
    __shared__ __align__(16) float s_rbf[GEOM_CR][2 * SCANN_RBF];    // rows read as LDS.128 broadcasts
    __shared__ int s_c[GEOM_CR];
    __shared__ float s_w[GEOM_CR];
    const int n = threadIdx.x & 127, half = threadIdx.x >> 7;
    float wd[SCANN_RBF], ww[SCANN_RBF];
#pragma unroll
    for (int k = 0; k < SCANN_RBF; ++k) {
        wd[k] = Wd[k * SCANN_D + n];
        ww[k] = Ww[k * SCANN_D + n];
    }
    const float bdn = bd[n], bwn = bw[n];
    pdl_wait();                                   // weights above are parameters; the plan is a predecessor's output
    const int nt = *ntiles;
    GEOM_CHUNK_LOOP(nt, stride) {
        const size_t base = (size_t)ch * GEOM_CR;
        const int nrows = GEOM_CHUNK_ROWS(ch);
        __syncthreads();
        if (ch + (int)gridDim.x >= nchunks) pdl_trigger();          // last chunk of this CTA: let the next kernel set up
        geom_stage_chunk<2 * SCANN_RBF>(s_rbf, s_c, s_w, pair_c, pair_d, pair_w, cd, cw, base, nrows);
#pragma unroll 4
        for (int row = half; row < nrows; row += 2) {                // padding rows: Gaussians are zero, result selected away
            float a = bdn, b = bwn;
            const float4* rb = reinterpret_cast<const float4*>(s_rbf[row]);
#pragma unroll
            for (int k4 = 0; k4 < SCANN_RBF / 4; ++k4) {
                const float4 rd = rb[k4], rw = rb[SCANN_RBF / 4 + k4];
                a = fmaf(rd.x, wd[4 * k4], a); a = fmaf(rd.y, wd[4 * k4 + 1], a);
                a = fmaf(rd.z, wd[4 * k4 + 2], a); a = fmaf(rd.w, wd[4 * k4 + 3], a);
                b = fmaf(rw.x, ww[4 * k4], b); b = fmaf(rw.y, ww[4 * k4 + 1], b);
                b = fmaf(rw.z, ww[4 * k4 + 2], b); b = fmaf(rw.w, ww[4 * k4 + 3], b);
            }
            g0[(base + row) * SCANN_D + n] = s_c[row] >= 0 ? swish_fast(a) * swish_fast(b) : 0.f;
        }
    }
    pdl_trigger();
}

// Backward: accumulates dWd, dbd, dWw, dbw from d_g0 (no gradient flows to distances/weights).
// DET (deterministic mode): every half-CTA stores its partial sums into slot 2 * blockIdx.x + half of dWd, a
// [2 * grid][GEOM_BWD_SLOT] array laid out as dWd | dWw | dbd | dbw (dbd, dWw, dbw unused).
#define GEOM_BWD_SLOT (2 * SCANN_RBF * SCANN_D + 2 * SCANN_D)
template <bool DET>
__global__ void __launch_bounds__(256, 2) geom_init_bwd_kernel(const int32_t* __restrict__ ntiles, int stride,
                                                            const int32_t* __restrict__ pair_c,
                                                            const float* __restrict__ pair_d,
                                                            const float* __restrict__ pair_w,
                                                            const float* __restrict__ cd, const float* __restrict__ cw,
                                                            const float* __restrict__ Wd, const float* __restrict__ bd,
                                                            const float* __restrict__ Ww, const float* __restrict__ bw,
                                                            const float* __restrict__ dg0, float* __restrict__ dWd,
                                                            float* __restrict__ dbd, float* __restrict__ dWw,
                                                            float* __restrict__ dbw) {
    __shared__ __align__(16) float s_rbf[GEOM_CR][2 * SCANN_RBF];    // rows read as LDS.128 broadcasts
    __shared__ int s_c[GEOM_CR];
    __shared__ float s_w[GEOM_CR];
    const int n = threadIdx.x & 127, half = threadIdx.x >> 7;
    float wd[SCANN_RBF], ww[SCANN_RBF], gd[SCANN_RBF], gw[SCANN_RBF];
#pragma unroll
    for (int k = 0; k < SCANN_RBF; ++k) {
        wd[k] = Wd[k * SCANN_D + n];
        ww[k] = Ww[k * SCANN_D + n];
        gd[k] = 0.f;
        gw[k] = 0.f;
    }
    const float bdn = bd[n], bwn = bw[n];
    float gbd = 0.f, gbw = 0.f;
    pdl_wait();
    const int nt = *ntiles;
    GEOM_CHUNK_LOOP(nt, stride) {
        const size_t base = (size_t)ch * GEOM_CR;
        const int nrows = GEOM_CHUNK_ROWS(ch);
        __syncthreads();
        if (ch + (int)gridDim.x >= nchunks) pdl_trigger();          // last chunk of this CTA: let the next kernel set up
        geom_stage_chunk<2 * SCANN_RBF>(s_rbf, s_c, s_w, pair_c, pair_d, pair_w, cd, cw, base, nrows);
        // the gradient rows of this thread's half are independent loads: keep 8 in flight.  (Batches of 4 with the next
        // batch prefetched -- the form that pays in noupdate_geom_bwd_kernel -- are neutral here: 128 registers either way,
        // gpurun_out/r02da_ab.log.)
        for (int r8 = half; r8 < nrows; r8 += 16) {
            float dv[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) dv[q] = r8 + 2 * q < nrows ? dg0[(base + r8 + 2 * q) * SCANN_D + n] : 0.f;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int row = r8 + 2 * q;
                if (row >= nrows || s_c[row] < 0) continue;
                float a = bdn, b = bwn;
                const float4* rb = reinterpret_cast<const float4*>(s_rbf[row]);
#pragma unroll
                for (int k4 = 0; k4 < SCANN_RBF / 4; ++k4) {
                    const float4 rd = rb[k4], rw = rb[SCANN_RBF / 4 + k4];
                    a = fmaf(rd.x, wd[4 * k4], a); a = fmaf(rd.y, wd[4 * k4 + 1], a);
                    a = fmaf(rd.z, wd[4 * k4 + 2], a); a = fmaf(rd.w, wd[4 * k4 + 3], a);
                    b = fmaf(rw.x, ww[4 * k4], b); b = fmaf(rw.y, ww[4 * k4 + 1], b);
                    b = fmaf(rw.z, ww[4 * k4 + 2], b); b = fmaf(rw.w, ww[4 * k4 + 3], b);
                }
                const float sa = sigmoid_fast(a), sb = sigmoid_fast(b);
                const float da = dv[q] * (b * sb) * (sa * (1.0f + a * (1.0f - sa)));
                const float db = dv[q] * (a * sa) * (sb * (1.0f + b * (1.0f - sb)));
                gbd += da;
                gbw += db;
                // the Gaussians are read again (shared-memory broadcasts) rather than kept: 40 registers less,
                // two CTAs per SM
#pragma unroll
                for (int k4 = 0; k4 < SCANN_RBF / 4; ++k4) {
                    const float4 rd = rb[k4], rw = rb[SCANN_RBF / 4 + k4];
                    gd[4 * k4] = fmaf(rd.x, da, gd[4 * k4]); gd[4 * k4 + 1] = fmaf(rd.y, da, gd[4 * k4 + 1]);
                    gd[4 * k4 + 2] = fmaf(rd.z, da, gd[4 * k4 + 2]); gd[4 * k4 + 3] = fmaf(rd.w, da, gd[4 * k4 + 3]);
                    gw[4 * k4] = fmaf(rw.x, db, gw[4 * k4]); gw[4 * k4 + 1] = fmaf(rw.y, db, gw[4 * k4 + 1]);
                    gw[4 * k4 + 2] = fmaf(rw.z, db, gw[4 * k4 + 2]); gw[4 * k4 + 3] = fmaf(rw.w, db, gw[4 * k4 + 3]);
                }
            }
        }
    }
    pdl_trigger();
    if constexpr (DET) {
        float* slot = dWd + ((size_t)blockIdx.x * 2 + half) * GEOM_BWD_SLOT;
#pragma unroll
        for (int k = 0; k < SCANN_RBF; ++k) {
            slot[k * SCANN_D + n] = gd[k];
            slot[(SCANN_RBF + k) * SCANN_D + n] = gw[k];
        }
        slot[2 * SCANN_RBF * SCANN_D + n] = gbd;
        slot[2 * SCANN_RBF * SCANN_D + SCANN_D + n] = gbw;
    } else if ((long long)blockIdx.x * GEOM_CR < (long long)nt * stride) {
#pragma unroll
        for (int k = 0; k < SCANN_RBF; ++k) {
            atomicAdd(dWd + k * SCANN_D + n, gd[k]);
            atomicAdd(dWw + k * SCANN_D + n, gw[k]);
        }
        atomicAdd(dbd + n, gbd);
        atomicAdd(dbw + n, gbw);
    }
}

// g_update = False, forward (attention.py:155): g' = swish(rbf(d) @ Wf + bf) * w  as a [rows,128] tensor -- the geometry
// operand of the pipelined attention kernels (la_pipe.cu / la_pipe_bwd.cu), which take it tile by tile through TMA.
// (The round-1 attention kernel la_attn_fwd_tc computes the same expression on the fly inside its tile loop; the
// pipelined kernels' consumers have no issue slots left for 20 more fused multiply-adds per element, profiles/r02_summary.md.)
// Padding rows of a tile are written as zeros.
__global__ void __launch_bounds__(256) noupdate_geom_fwd_kernel(const int32_t* __restrict__ ntiles, int stride,
                                                                const int32_t* __restrict__ pair_c,
                                                                const float* __restrict__ pair_d,
                                                                const float* __restrict__ pair_w,
                                                                const float* __restrict__ cd,
                                                                const float* __restrict__ Wf, const float* __restrict__ bf,
                                                                float* __restrict__ g) {
    __shared__ __align__(16) float s_rbf[GEOM_CR][2 * SCANN_RBF];
    __shared__ int s_c[GEOM_CR];
    __shared__ float s_w[GEOM_CR];
    const int n = threadIdx.x & 127, half = threadIdx.x >> 7;
    float wf[SCANN_RBF];
#pragma unroll
    for (int k = 0; k < SCANN_RBF; ++k) wf[k] = Wf[k * SCANN_D + n];
    const float bfn = bf[n];
    pdl_wait();                                   // weights above are parameters; the plan is a predecessor's output
    const int nt = *ntiles;
    GEOM_CHUNK_LOOP(nt, stride) {
        const size_t base = (size_t)ch * GEOM_CR;
        const int nrows = GEOM_CHUNK_ROWS(ch);
        __syncthreads();
        if (ch + (int)gridDim.x >= nchunks) pdl_trigger();
        geom_stage_chunk<SCANN_RBF>(s_rbf, s_c, s_w, pair_c, pair_d, pair_w, cd, cd, base, nrows);
#pragma unroll 4
        for (int row = half; row < nrows; row += 2) {
            float a = bfn;
            const float4* rb = reinterpret_cast<const float4*>(s_rbf[row]);
#pragma unroll
            for (int k4 = 0; k4 < SCANN_RBF / 4; ++k4) {
                const float4 rd = rb[k4];
                a = fmaf(rd.x, wf[4 * k4], a); a = fmaf(rd.y, wf[4 * k4 + 1], a);
                a = fmaf(rd.z, wf[4 * k4 + 2], a); a = fmaf(rd.w, wf[4 * k4 + 3], a);
            }
            g[(base + row) * SCANN_D + n] = s_c[row] >= 0 ? swish_fast(a) * s_w[row] : 0.f;
        }
    }
    pdl_trigger();
}

// g_update = False (attention.py:155): g' = swish(rbf(d) @ Wf + bf) * w is recomputed in every layer; its only
// trainable inputs are Wf [20,128] and bf.  dWf += rbf^T d_pre, dbf += sum d_pre with
// d_pre = dg' * w * swish'(pre), pre = rbf @ Wf + bf (recomputed here from the 8 bytes/pair of raw geometry).
// DET (deterministic mode): every half-CTA stores its partial sums into slot 2 * blockIdx.x + half of dWf, a
// [2 * grid][NOUP_BWD_SLOT] array laid out as dWf (20 x 128) | dbf (dbf unused).
#define NOUP_BWD_SLOT ((SCANN_RBF + 1) * SCANN_D)
template <bool DET>
__global__ void __launch_bounds__(256, 2) noupdate_geom_bwd_kernel(const int32_t* __restrict__ ntiles, int stride,
                                                                const int32_t* __restrict__ pair_c,
                                                                const float* __restrict__ pair_d,
                                                                const float* __restrict__ pair_w,
                                                                const float* __restrict__ cd,
                                                                const float* __restrict__ Wf, const float* __restrict__ bf,
                                                                const float* __restrict__ dg, float* __restrict__ dWf,
                                                                float* __restrict__ dbf) {
    __shared__ __align__(16) float s_rbf[GEOM_CR][2 * SCANN_RBF];
    __shared__ int s_c[GEOM_CR];
    __shared__ float s_w[GEOM_CR];
    const int n = threadIdx.x & 127, half = threadIdx.x >> 7;
    float wf[SCANN_RBF], gf[SCANN_RBF];
#pragma unroll
    for (int k = 0; k < SCANN_RBF; ++k) { wf[k] = Wf[k * SCANN_D + n]; gf[k] = 0.f; }
    const float bfn = bf[n];
    float gb = 0.f;
    pdl_wait();
    const int nt = *ntiles;
    GEOM_CHUNK_LOOP(nt, stride) {
        const size_t base = (size_t)ch * GEOM_CR;
        const int nrows = GEOM_CHUNK_ROWS(ch);
        __syncthreads();
        if (ch + (int)gridDim.x >= nchunks) pdl_trigger();
        geom_stage_chunk<SCANN_RBF>(s_rbf, s_c, s_w, pair_c, pair_d, pair_w, cd, cd, base, nrows);
        // gradient rows in batches of 8, the NEXT batch's loads issued before the current one is consumed (they were one
        // exposed HBM round trip per batch: 4 of the ~10 us a chunk took, gpurun_out/r02cz_launches_ptgp.csv)
        float nx[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) nx[q] = half + 2 * q < nrows ? dg[(base + half + 2 * q) * SCANN_D + n] : 0.f;
        for (int r8 = half; r8 < nrows; r8 += 16) {
            float dv[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) dv[q] = nx[q];
#pragma unroll
            for (int q = 0; q < 8; ++q) nx[q] = r8 + 16 + 2 * q < nrows ? dg[(base + r8 + 16 + 2 * q) * SCANN_D + n] : 0.f;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int row = r8 + 2 * q;
                if (row >= nrows || s_c[row] < 0) continue;
                float a = bfn;
                const float4* rb = reinterpret_cast<const float4*>(s_rbf[row]);
                float4 rd[SCANN_RBF / 4];
#pragma unroll
                for (int k4 = 0; k4 < SCANN_RBF / 4; ++k4) {
                    rd[k4] = rb[k4];
                    a = fmaf(rd[k4].x, wf[4 * k4], a); a = fmaf(rd[k4].y, wf[4 * k4 + 1], a);
                    a = fmaf(rd[k4].z, wf[4 * k4 + 2], a); a = fmaf(rd[k4].w, wf[4 * k4 + 3], a);
                }
                const float da = dv[q] * s_w[row] * swish_grad_fast(a);
                gb += da;
#pragma unroll
                for (int k4 = 0; k4 < SCANN_RBF / 4; ++k4) {
                    gf[4 * k4] = fmaf(rd[k4].x, da, gf[4 * k4]); gf[4 * k4 + 1] = fmaf(rd[k4].y, da, gf[4 * k4 + 1]);
                    gf[4 * k4 + 2] = fmaf(rd[k4].z, da, gf[4 * k4 + 2]); gf[4 * k4 + 3] = fmaf(rd[k4].w, da, gf[4 * k4 + 3]);
                }
            }
        }
    }
    pdl_trigger();
    if constexpr (DET) {
        float* slot = dWf + ((size_t)blockIdx.x * 2 + half) * NOUP_BWD_SLOT;
#pragma unroll
        for (int k = 0; k < SCANN_RBF; ++k) slot[k * SCANN_D + n] = gf[k];
        slot[SCANN_RBF * SCANN_D + n] = gb;
    } else if ((long long)blockIdx.x * GEOM_CR < (long long)nt * stride) {
#pragma unroll
        for (int k = 0; k < SCANN_RBF; ++k) atomicAdd(dWf + k * SCANN_D + n, gf[k]);
        atomicAdd(dbf + n, gb);
    }
}

// ---------------------------------------------------------------------------------------------
// Blocked dense GEMM:  C[r, nb*128 + c] = epi( sum_kb A_kb[r,:] @ W[kb*nblk+nb] + bias[nb] )
// A_kb: [R,128] with row stride lda; W blocks: [128,128] row-major.
// 32 rows x 128 cols per CTA, 256 threads, 4x4 register tile.
// ---------------------------------------------------------------------------------------------
#define DENSE_BM 32
#define DENSE_LDS 132
struct DenseArgs {
    const float* A[3];
    int lda;
    const float* W[9];      // [kblk][nblk]
    const float* bias[3];   // per n-block, nullable
    int kblk, nblk;
    int R;
    float* C;
    int ldc;
    int mode;               // 0 none | 1 swish | 2 multiply by swish'(pre_in) | 3 LayerNorm
    const float* resid;     // nullable, added before the activation / LayerNorm
    int ldres;
    const float* pre_in;    // mode 2
    float* pre_out;         // mode 1: pre-activation ; mode 3: pre-LayerNorm value (nullable)
    const float* gamma;
    const float* beta;
};

__global__ void __launch_bounds__(256) dense_kernel(const DenseArgs a) {
    __shared__ float s_a[DENSE_BM][DENSE_LDS];
    const int tid = threadIdx.x, ty = tid >> 5, tx = tid & 31;
    const int r0 = blockIdx.x * DENSE_BM, nb = blockIdx.y;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int kb = 0; kb < a.kblk; ++kb) {
        const float* A = a.A[kb];
        __syncthreads();
        for (int i = tid; i < DENSE_BM * 32; i += 256) {
            int rr = i >> 5, c4 = (i & 31) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r0 + rr < a.R) v = ld4(A + (size_t)(r0 + rr) * a.lda + c4);
            st4(&s_a[rr][c4], v);
        }
        __syncthreads();
        const float* W = a.W[kb * a.nblk + nb] + tx * 4;
#pragma unroll 2
        for (int k0 = 0; k0 < SCANN_D; k0 += 4) {
            float4 av[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) av[i] = ld4(&s_a[ty * 4 + i][k0]);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                float4 b = ldg4(W + (size_t)(k0 + kk) * SCANN_D);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    float x = kk == 0 ? av[i].x : kk == 1 ? av[i].y : kk == 2 ? av[i].z : av[i].w;
                    acc[i][0] = fmaf(x, b.x, acc[i][0]);
                    acc[i][1] = fmaf(x, b.y, acc[i][1]);
                    acc[i][2] = fmaf(x, b.z, acc[i][2]);
                    acc[i][3] = fmaf(x, b.w, acc[i][3]);
                }
            }
        }
    }
    // epilogue
    const int c0 = tx * 4;
    float4 bias = make_float4(0.f, 0.f, 0.f, 0.f);
    if (a.bias[nb]) bias = ldg4(a.bias[nb] + c0);
    float4 gam = make_float4(0.f, 0.f, 0.f, 0.f), bet = gam;
    if (a.mode == 3) { gam = ldg4(a.gamma + c0); bet = ldg4(a.beta + c0); }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = r0 + ty * 4 + i;
        const bool ok = r < a.R;           // warp-uniform (ty is the warp index)
        float v[4] = {acc[i][0] + bias.x, acc[i][1] + bias.y, acc[i][2] + bias.z, acc[i][3] + bias.w};
        if (a.resid && ok) {
            float4 rv = ld4(a.resid + (size_t)r * a.ldres + nb * SCANN_D + c0);
            v[0] += rv.x; v[1] += rv.y; v[2] += rv.z; v[3] += rv.w;
        }
        if (a.mode == 1) {
            if (a.pre_out && ok) st4(a.pre_out + (size_t)r * a.ldc + nb * SCANN_D + c0, make_float4(v[0], v[1], v[2], v[3]));
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = swish_f(v[j]);
        } else if (a.mode == 2) {
            if (ok) {
                float4 p = ld4(a.pre_in + (size_t)r * a.ldc + nb * SCANN_D + c0);
                v[0] *= swish_grad_f(p.x); v[1] *= swish_grad_f(p.y);
                v[2] *= swish_grad_f(p.z); v[3] *= swish_grad_f(p.w);
            }
        } else if (a.mode == 3) {
            if (a.pre_out && ok) st4(a.pre_out + (size_t)r * a.ldc + c0, make_float4(v[0], v[1], v[2], v[3]));
            float mean = warp_sum(v[0] + v[1] + v[2] + v[3]) * (1.0f / SCANN_D);
            float d0 = v[0] - mean, d1 = v[1] - mean, d2 = v[2] - mean, d3 = v[3] - mean;
            float var = warp_sum(d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3) * (1.0f / SCANN_D);
            float inv = rsqrtf(var + SCANN_LN_EPS);
            v[0] = d0 * inv * gam.x + bet.x; v[1] = d1 * inv * gam.y + bet.y;
            v[2] = d2 * inv * gam.z + bet.z; v[3] = d3 * inv * gam.w + bet.w;
        }
        if (ok) st4(a.C + (size_t)r * a.ldc + nb * SCANN_D + c0, make_float4(v[0], v[1], v[2], v[3]));
    }
}

// ---------------------------------------------------------------------------------------------
// Weight gradient:  dW[kb*nblk+nb] += A_kb^T @ G_nb   (reduction over rows), db[nb] += colsum(G_nb)
// 64x64 output sub-tile per CTA, rows split across blockIdx.x, atomics into dW.
// ---------------------------------------------------------------------------------------------
struct WgradArgs {
    const float* A[3];
    int lda;
    const float* G[3];
    int ldg;
    int kblk, nblk, R, rows_per_cta;
    float* dW[9];
    float* db[3];           // nullable
};

__global__ void __launch_bounds__(256) wgrad_kernel(const WgradArgs a) {
    __shared__ float s_a[16][64];
    __shared__ float s_g[16][64];
    const int tid = threadIdx.x;
    const int sub = blockIdx.y, m0 = (sub >> 1) * 64, n0 = (sub & 1) * 64;
    const int kb = blockIdx.z / a.nblk, nb = blockIdx.z % a.nblk;
    const float* A = a.A[kb] + m0;
    const float* G = a.G[nb] + n0;
    const int r_lo = blockIdx.x * a.rows_per_cta, r_hi = min(a.R, r_lo + a.rows_per_cta);
    const int tm = (tid >> 4) * 4, tn = (tid & 15) * 4;
    float acc[4][4];
    float bsum[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    const int lr = tid >> 4, lc = (tid & 15) * 4;
    for (int r = r_lo; r < r_hi; r += 16) {
        float4 va = make_float4(0.f, 0.f, 0.f, 0.f), vg = va;
        if (r + lr < r_hi) {
            va = ld4(A + (size_t)(r + lr) * a.lda + lc);
            vg = ld4(G + (size_t)(r + lr) * a.ldg + lc);
        }
        __syncthreads();
        st4(&s_a[lr][lc], va);
        st4(&s_g[lr][lc], vg);
        __syncthreads();
#pragma unroll
        for (int rr = 0; rr < 16; ++rr) {
            float4 x = ld4(&s_a[rr][tm]);
            float4 g = ld4(&s_g[rr][tn]);
            float xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                acc[i][0] = fmaf(xs[i], g.x, acc[i][0]);
                acc[i][1] = fmaf(xs[i], g.y, acc[i][1]);
                acc[i][2] = fmaf(xs[i], g.z, acc[i][2]);
                acc[i][3] = fmaf(xs[i], g.w, acc[i][3]);
            }
            if (tm == 0) { bsum[0] += g.x; bsum[1] += g.y; bsum[2] += g.z; bsum[3] += g.w; }
        }
    }
    float* dW = a.dW[kb * a.nblk + nb];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) atomicAdd(dW + (size_t)(m0 + tm + i) * SCANN_D + n0 + tn + j, acc[i][j]);
    if (tm == 0 && m0 == 0 && kb == 0 && a.db[nb]) {
#pragma unroll
        for (int j = 0; j < 4; ++j) atomicAdd(a.db[nb] + n0 + tn + j, bsum[j]);
    }
}

// ---------------------------------------------------------------------------------------------
// LayerNorm backward (one warp per row): dv = inv * (dxh - mean(dxh) - xh * mean(dxh*xh)),
// dxh = dy * gamma, xh = (v - mean) * inv ;  dgamma += dy*xh ; dbeta += dy.
// Optionally writes dv to a second destination as well (dv2, row stride ld2).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ln_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ v,
                                                     const float* __restrict__ gamma, int R, float* __restrict__ dv,
                                                     float* __restrict__ dv2, int ld2, float* __restrict__ dgamma,
                                                     float* __restrict__ dbeta) {
    __shared__ float s_g[SCANN_D], s_b[SCANN_D];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    if (threadIdx.x < SCANN_D) { s_g[threadIdx.x] = 0.f; s_b[threadIdx.x] = 0.f; }
    __syncthreads();
    const float4 gam = ldg4(gamma + lane * 4);
    pdl_wait();
    pdl_trigger();
    float ag[4] = {0.f, 0.f, 0.f, 0.f}, ab[4] = {0.f, 0.f, 0.f, 0.f};
    for (int r = blockIdx.x * nwarp + warp; r < R; r += gridDim.x * nwarp) {
        float4 x = ld4(v + (size_t)r * SCANN_D + lane * 4);
        float4 d = ld4(dy + (size_t)r * SCANN_D + lane * 4);
        float mean = warp_sum(x.x + x.y + x.z + x.w) * (1.0f / SCANN_D);
        float c0 = x.x - mean, c1 = x.y - mean, c2 = x.z - mean, c3 = x.w - mean;
        float var = warp_sum(c0 * c0 + c1 * c1 + c2 * c2 + c3 * c3) * (1.0f / SCANN_D);
        float inv = rsqrtf(var + SCANN_LN_EPS);
        float h0 = c0 * inv, h1 = c1 * inv, h2 = c2 * inv, h3 = c3 * inv;
        float e0 = d.x * gam.x, e1 = d.y * gam.y, e2 = d.z * gam.z, e3 = d.w * gam.w;
        float m1 = warp_sum(e0 + e1 + e2 + e3) * (1.0f / SCANN_D);
        float m2 = warp_sum(e0 * h0 + e1 * h1 + e2 * h2 + e3 * h3) * (1.0f / SCANN_D);
        float4 o = make_float4(inv * (e0 - m1 - h0 * m2), inv * (e1 - m1 - h1 * m2), inv * (e2 - m1 - h2 * m2),
                               inv * (e3 - m1 - h3 * m2));
        st4(dv + (size_t)r * SCANN_D + lane * 4, o);
        if (dv2) st4(dv2 + (size_t)r * ld2 + lane * 4, o);
        ag[0] += d.x * h0; ag[1] += d.y * h1; ag[2] += d.z * h2; ag[3] += d.w * h3;
        ab[0] += d.x; ab[1] += d.y; ab[2] += d.z; ab[3] += d.w;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        atomicAdd(&s_g[lane * 4 + j], ag[j]);
        atomicAdd(&s_b[lane * 4 + j], ab[j]);
    }
    __syncthreads();
    if (threadIdx.x < SCANN_D) {
        atomicAdd(dgamma + threadIdx.x, s_g[threadIdx.x]);
        atomicAdd(dbeta + threadIdx.x, s_b[threadIdx.x]);
    }
}

// ---------------------------------------------------------------------------------------------
// Atoms without a single valid neighbour: context = q, out = LN(q)      (attention.py:206-214)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) la_nopair_fwd_kernel(const int32_t* __restrict__ cnt,
                                                            const float* __restrict__ proj, int R,
                                                            const float* __restrict__ gamma,
                                                            const float* __restrict__ beta,
                                                            float* __restrict__ ctx_pre, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    pdl_wait();
    pdl_trigger();      // only after the own wait: at most one kernel ahead becomes resident early
    if (r >= R || cnt[r] != 0) return;
    float4 q = ld4(proj + (size_t)r * 3 * SCANN_D + 2 * SCANN_D + lane * 4);
    if (ctx_pre) st4(ctx_pre + (size_t)r * SCANN_D + lane * 4, q);
    float mean = warp_sum(q.x + q.y + q.z + q.w) * (1.0f / SCANN_D);
    float c0 = q.x - mean, c1 = q.y - mean, c2 = q.z - mean, c3 = q.w - mean;
    float var = warp_sum(c0 * c0 + c1 * c1 + c2 * c2 + c3 * c3) * (1.0f / SCANN_D);
    float inv = rsqrtf(var + SCANN_LN_EPS);
    float4 g = ldg4(gamma + lane * 4), b = ldg4(beta + lane * 4);
    st4(out + (size_t)r * SCANN_D + lane * 4,
        make_float4(c0 * inv * g.x + b.x, c1 * inv * g.y + b.y, c2 * inv * g.z + b.z, c3 * inv * g.w + b.w));
}

// ---------------------------------------------------------------------------------------------
// Transpose a list of 128x128 blocks of the parameter arena into the transposed arena.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) transpose_blocks_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                               const int32_t* __restrict__ offsets) {
    // one CTA per 32x32 sub-tile (blockIdx.y): 16 x as many CTAs as blocks, each a single load / store round (the first
    // form walked the 16 sub-tiles of a block in one CTA, two barriers each: 37 us for 53 blocks on the side stream)
    __shared__ float s[32][33];
    const size_t off = (size_t)offsets[blockIdx.x];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int t = blockIdx.y;
    const int bi = (t >> 2) * 32, bj = (t & 3) * 32;
    for (int i = ty; i < 32; i += 8) s[i][tx] = src[off + (size_t)(bi + i) * SCANN_D + bj + tx];
    __syncthreads();
    for (int i = ty; i < 32; i += 8) dst[off + (size_t)(bj + i) * SCANN_D + bi + tx] = s[tx][i];
}

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" int scann_embed_forward(const int32_t* atomic, const float* ring, int R, int E, int n_atoms,
                                   const float* emb, const float* Wr, const float* br, const float* We,
                                   const float* be, float* t0, float* x0, int32_t* status, const void* drop_ctl,
                                   const float* emb_rows, void* stream) {
    int Kin = E + (ring ? 10 : 0);
    size_t smem = (size_t)EMB_ROWS * Kin * sizeof(float);
    scann_launch(embed_fwd_kernel, dim3((R + EMB_ROWS - 1) / EMB_ROWS), dim3(128), smem, stream, atomic, ring, R, E, n_atoms,
                 emb, Wr, br, We, be, t0, x0, status, (const ScannDropCtl*)drop_ctl, emb_rows);
    return scann_check_launch("scann_embed_forward");
}

extern "C" int scann_embed_backward(const int32_t* atomic, const float* ring, int R, int E, int n_atoms,
                                    const float* emb, const float* Wr, const float* br, const float* We,
                                    const float* t0, const float* dx0, float* G_ws, float* d_emb, float* dWr,
                                    float* dbr, float* dWe, float* dbe, const void* drop_ctl, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    cudaMemsetAsync(G_ws, 0, (size_t)(n_atoms + 3) * SCANN_D * sizeof(float), st);
    int rows_per_cta = 16;
    embed_bwd_gather_kernel<<<(R + rows_per_cta - 1) / rows_per_cta, 128, 0, st>>>(atomic, ring, R, n_atoms, t0, dx0,
                                                                                  G_ws, rows_per_cta,
                                                                                  (const ScannDropCtl*)drop_ctl);
    embed_bwd_final_kernel<<<64, 128, 0, st>>>(E, n_atoms, ring ? 1 : 0, emb, Wr, br, We, G_ws, d_emb, dWr, dbr, dWe,
                                               dbe);
    return scann_check_launch("scann_embed_backward");
}

extern "C" int scann_device_sm_count(void);

// Deterministic form: G_slots = [scann_embed_backward_det_slots(R)][n_atoms + 3][128] floats of workspace.  Rows per CTA
// are chosen so that the slots fill about two waves of CTAs: enough parallelism, slot traffic bounded by the SM count.
static int embed_det_rows(int R) {
    static int sms = 0;
    if (sms == 0) sms = scann_device_sm_count();
    const int ctas = 2 * (sms > 0 ? sms : 148);
    const int rows = (R + ctas - 1) / ctas;
    return rows < 16 ? 16 : rows;
}

extern "C" int scann_embed_backward_det(const int32_t* atomic, const float* ring, int R, int E, int n_atoms,
                                        const float* emb, const float* Wr, const float* br, const float* We,
                                        const float* t0, const float* dx0, float* G_ws, float* G_slots, float* d_emb,
                                        float* dWr, float* dbr, float* dWe, float* dbe, const void* drop_ctl, void* stream) {
    if (R <= 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int nrow = n_atoms + 3, rows = embed_det_rows(R), nslots = (R + rows - 1) / rows;
    const size_t smem = (size_t)nrow * SCANN_D * sizeof(float);
    if (smem > 200 * 1024) { scann_set_error("embed_backward_det: n_atoms=%d too large", n_atoms); return 1; }
    static size_t configured = 48 * 1024;             // dynamic shared memory the kernel is opted in to
    if (smem > configured) {
        if (cudaFuncSetAttribute(embed_bwd_gather_det_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) !=
            cudaSuccess) {
            scann_set_error("embed_backward_det: shared-memory opt-in failed");
            return 1;
        }
        configured = 200 * 1024;
    }
    embed_bwd_gather_det_kernel<<<nslots, 128, smem, st>>>(atomic, ring, R, n_atoms, t0, dx0, G_slots, rows,
                                                           (const ScannDropCtl*)drop_ctl);
    embed_bwd_slot_sum_kernel<<<nrow, 128, 0, st>>>(G_slots, nslots, nrow * SCANN_D, G_ws);
    embed_bwd_final_kernel<<<64, 128, 0, st>>>(E, n_atoms, ring ? 1 : 0, emb, Wr, br, We, G_ws, d_emb, dWr, dbr, dWe,
                                               dbe);
    return scann_check_launch("scann_embed_backward_det");
}

// Slots of the G workspace scann_embed_backward_det needs for R atom rows.
extern "C" int scann_embed_backward_det_slots(int R) { return R <= 0 ? 0 : (R + embed_det_rows(R) - 1) / embed_det_rows(R); }

// feature == "cgcnn": emb_rows [R,E] = atomic92 [R,92] @ embed_atom/kernel + bias (feeds scann_embed_forward).
extern "C" int scann_cgcnn_embed_forward(const float* atomic92, const float* W, const float* b, int R, int F, int E,
                                         float* emb_rows, void* stream) {
    if (E > 128 || E < 1 || F < 1) { scann_set_error("cgcnn_embed_forward: bad sizes F=%d E=%d", F, E); return 1; }
    if (R <= 0) return 0;
    scann_launch(small_dense_fwd_kernel, dim3(R < 592 ? R : 592), dim3(128), 0, stream, atomic92, W, b, R, F, E, emb_rows);
    return scann_check_launch("scann_cgcnn_embed_forward");
}

// Backward of the cgcnn embedding path: gradients of dense_embed (dWe, dbe), embed_atom Dense (dWemb, dbemb) and
// extra_embed (dWr, dbr, nullable) ACCUMULATED; d_cat_ws: R*144 floats of workspace.
extern "C" int scann_cgcnn_embed_backward(const float* atomic92, const float* emb_rows, const float* ring, int R, int F,
                                          int E, const float* Wr, const float* br, const float* We, const float* t0,
                                          const float* dx0, float* d_cat_ws, float* dWemb, float* dbemb, float* dWr,
                                          float* dbr, float* dWe, float* dbe, const void* drop_ctl, void* stream) {
    if (E > 128) { scann_set_error("cgcnn_embed_backward: embedding width %d too large", E); return 1; }
    if (R <= 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    embed_bwd_rows_kernel<false><<<(R + 31) / 32, 128, 0, st>>>(emb_rows, ring, R, E, Wr, br, We, t0, dx0, d_cat_ws, dWe, dbe,
                                                              (const ScannDropCtl*)drop_ctl);
    embed_bwd_cols_kernel<<<F + 1 + (ring ? 3 : 0), 128, 0, st>>>(atomic92, ring, R, F, E, d_cat_ws, dWemb, dbemb, dWr, dbr);
    return scann_check_launch("scann_cgcnn_embed_backward");
}

// Deterministic form: dense_embed's gradients go to slots [(R + 31) / 32][(E + (ring ? 10 : 0) + 1) * 128] (kernel rows,
// then bias; scann_slot_reduce adds them up); the embed_atom / extra_embed gradients are written by one thread each.
extern "C" int scann_cgcnn_embed_backward_det(const float* atomic92, const float* emb_rows, const float* ring, int R, int F,
                                              int E, const float* Wr, const float* br, const float* We, const float* t0,
                                              const float* dx0, float* d_cat_ws, float* dWemb, float* dbemb, float* dWr,
                                              float* dbr, float* slots, const void* drop_ctl, void* stream) {
    if (E > 128) { scann_set_error("cgcnn_embed_backward: embedding width %d too large", E); return 1; }
    if (R <= 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    embed_bwd_rows_kernel<true><<<(R + 31) / 32, 128, 0, st>>>(emb_rows, ring, R, E, Wr, br, We, t0, dx0, d_cat_ws, slots,
                                                             (float*)nullptr, (const ScannDropCtl*)drop_ctl);
    embed_bwd_cols_kernel<<<F + 1 + (ring ? 3 : 0), 128, 0, st>>>(atomic92, ring, R, F, E, d_cat_ws, dWemb, dbemb, dWr, dbr);
    return scann_check_launch("scann_cgcnn_embed_backward_det");
}

// embed_atom's gradients from the per-element gradient d_emb [Z_rows, E] of emb_table = table @ W + b, ACCUMULATED
// into dW [F, E] and db [E].  One thread per output element, z ascending: the same bits in both training modes.
extern "C" int scann_cgcnn_table_backward(const float* table, const float* d_emb, int Z_rows, int F, int E, float* dW,
                                          float* db, void* stream) {
    if (F != 92 || E < 1 || E > 128 || Z_rows < 1) {
        scann_set_error("cgcnn_table_backward: bad sizes Z_rows=%d F=%d E=%d (F must be 92, E in 1..128, Z_rows >= 1)",
                        Z_rows, F, E);
        return 1;
    }
    cgcnn_table_bwd_kernel<<<F + 1, 128, 0, (cudaStream_t)stream>>>(table, d_emb, Z_rows, F, E, dW, db);
    return scann_check_launch("scann_cgcnn_table_backward");
}

extern "C" int scann_geom_init_forward(const int32_t* ntiles, int grid, int tile_stride, const int32_t* pair_c, const float* pair_d,
                                       const float* pair_w, const float* centers_d, const float* centers_w,
                                       const float* Wd, const float* bd, const float* Ww, const float* bw, float* g0,
                                       void* stream) {
    if (tile_stride != 32 && tile_stride != 64 && tile_stride != 128) { scann_set_error("geom_init: tile_stride must be 64 or 128"); return 1; }
    scann_launch(geom_init_fwd_kernel, dim3(grid), dim3(256), 0, stream, ntiles, tile_stride, pair_c, pair_d, pair_w, centers_d, centers_w,
                 Wd, bd, Ww, bw, g0);
    return scann_check_launch("scann_geom_init_forward");
}

extern "C" int scann_geom_init_backward(const int32_t* ntiles, int grid, int tile_stride, const int32_t* pair_c, const float* pair_d,
                                        const float* pair_w, const float* centers_d, const float* centers_w,
                                        const float* Wd, const float* bd, const float* Ww, const float* bw,
                                        const float* dg0, float* dWd, float* dbd, float* dWw, float* dbw,
                                        void* stream) {
    if (tile_stride != 32 && tile_stride != 64 && tile_stride != 128) { scann_set_error("geom_init: tile_stride must be 64 or 128"); return 1; }
    scann_launch(geom_init_bwd_kernel<false>, dim3(grid), dim3(256), 0, stream, ntiles, tile_stride, pair_c, pair_d, pair_w, centers_d, centers_w,
                 Wd, bd, Ww, bw, dg0, dWd, dbd, dWw, dbw);
    return scann_check_launch("scann_geom_init_backward");
}

// Deterministic form: slots = [2 * grid][2 * 20 * 128 + 2 * 128] partial sums (dWd | dWw | dbd | dbw per half-CTA), to be
// added up in slot order (scann_slot_reduce).
extern "C" int scann_geom_init_backward_det(const int32_t* ntiles, int grid, int tile_stride, const int32_t* pair_c,
                                            const float* pair_d, const float* pair_w, const float* centers_d,
                                            const float* centers_w, const float* Wd, const float* bd, const float* Ww,
                                            const float* bw, const float* dg0, float* slots, void* stream) {
    if (tile_stride != 32 && tile_stride != 64 && tile_stride != 128) { scann_set_error("geom_init: tile_stride must be 64 or 128"); return 1; }
    scann_launch(geom_init_bwd_kernel<true>, dim3(grid), dim3(256), 0, stream, ntiles, tile_stride, pair_c, pair_d, pair_w, centers_d,
                 centers_w, Wd, bd, Ww, bw, dg0, slots, (float*)nullptr, (float*)nullptr, (float*)nullptr);
    return scann_check_launch("scann_geom_init_backward_det");
}

// g' = swish(rbf(d) @ Wf + bf) * w of a g_update = False layer as a [tile_cap * tile_stride, 128] tensor (see
// noupdate_geom_fwd_kernel): the geometry input of scann_la_forward_pipe / scann_la_backward_pipe for such a layer.
extern "C" int scann_noupdate_geom_forward(const int32_t* ntiles, int grid, int tile_stride, const int32_t* pair_c,
                                           const float* pair_d, const float* pair_w, const float* centers_d,
                                           const float* Wf, const float* bf, float* g_out, void* stream) {
    if (tile_stride != 32 && tile_stride != 64 && tile_stride != 128) { scann_set_error("noupdate_geom_forward: tile_stride must be 32, 64 or 128"); return 1; }
    if (grid <= 0) return 0;
    scann_launch(noupdate_geom_fwd_kernel, dim3(grid), dim3(256), 0, stream, ntiles, tile_stride, pair_c, pair_d, pair_w,
                 centers_d, Wf, bf, g_out);
    return scann_check_launch("scann_noupdate_geom_forward");
}

// Weight gradient of the g_update = False geometry (see noupdate_geom_bwd_kernel): dWf [20,128], dbf [128]
// accumulated from dg = gradient w.r.t. g' ([rows,128], left by scann_la_backward_noupdate_tc).
extern "C" int scann_noupdate_geom_backward(const int32_t* ntiles, int grid, int tile_stride, const int32_t* pair_c,
                                            const float* pair_d, const float* pair_w, const float* centers_d,
                                            const float* Wf, const float* bf, const float* dg, float* dWf, float* dbf,
                                            void* stream) {
    if (tile_stride != 32 && tile_stride != 64 && tile_stride != 128) { scann_set_error("noupdate_geom_backward: tile_stride must be 64 or 128"); return 1; }
    scann_launch(noupdate_geom_bwd_kernel<false>, dim3(grid), dim3(256), 0, stream, ntiles, tile_stride, pair_c, pair_d, pair_w,
                 centers_d, Wf, bf, dg, dWf, dbf);
    return scann_check_launch("scann_noupdate_geom_backward");
}

// Deterministic form: slots = [2 * grid][21 * 128] partial sums (dWf | dbf per half-CTA), added up in slot order by
// scann_slot_reduce.
extern "C" int scann_noupdate_geom_backward_det(const int32_t* ntiles, int grid, int tile_stride, const int32_t* pair_c,
                                                const float* pair_d, const float* pair_w, const float* centers_d,
                                                const float* Wf, const float* bf, const float* dg, float* slots,
                                                void* stream) {
    if (tile_stride != 32 && tile_stride != 64 && tile_stride != 128) { scann_set_error("noupdate_geom_backward: tile_stride must be 64 or 128"); return 1; }
    scann_launch(noupdate_geom_bwd_kernel<true>, dim3(grid), dim3(256), 0, stream, ntiles, tile_stride, pair_c, pair_d, pair_w,
                 centers_d, Wf, bf, dg, slots, (float*)nullptr);
    return scann_check_launch("scann_noupdate_geom_backward_det");
}

// Generic blocked dense: see DenseArgs.  A/W/bias arrays hold kblk / kblk*nblk / nblk entries.
extern "C" int scann_dense_forward(const float* const* A, int lda, const float* const* W, const float* const* bias,
                                   int kblk, int nblk, int R, float* C, int ldc, int mode, const float* resid,
                                   int ldres, const float* pre_in, float* pre_out, const float* gamma,
                                   const float* beta, void* stream) {
    if (kblk < 1 || kblk > 3 || nblk < 1 || nblk > 3) { scann_set_error("dense: kblk/nblk must be in 1..3"); return 1; }
    if (mode == 3 && nblk != 1) { scann_set_error("dense: LayerNorm epilogue needs nblk == 1"); return 1; }
    if (R <= 0) return 0;
    DenseArgs a;
    for (int i = 0; i < 3; ++i) { a.A[i] = i < kblk ? A[i] : nullptr; a.bias[i] = (bias && i < nblk) ? bias[i] : nullptr; }
    for (int i = 0; i < 9; ++i) a.W[i] = i < kblk * nblk ? W[i] : nullptr;
    a.lda = lda; a.kblk = kblk; a.nblk = nblk; a.R = R; a.C = C; a.ldc = ldc; a.mode = mode;
    a.resid = resid; a.ldres = ldres; a.pre_in = pre_in; a.pre_out = pre_out; a.gamma = gamma; a.beta = beta;
    dim3 grid((R + DENSE_BM - 1) / DENSE_BM, nblk);
    dense_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(a);
    return scann_check_launch("scann_dense_forward");
}

extern "C" int scann_dense_wgrad(const float* const* A, int lda, const float* const* G, int ldg, int kblk, int nblk,
                                 int R, float* const* dW, float* const* db, void* stream) {
    if (kblk < 1 || kblk > 3 || nblk < 1 || nblk > 3) { scann_set_error("wgrad: kblk/nblk must be in 1..3"); return 1; }
    if (R <= 0) return 0;
    WgradArgs a;
    for (int i = 0; i < 3; ++i) {
        a.A[i] = i < kblk ? A[i] : nullptr;
        a.G[i] = i < nblk ? G[i] : nullptr;
        a.db[i] = (db && i < nblk) ? db[i] : nullptr;
    }
    for (int i = 0; i < 9; ++i) a.dW[i] = i < kblk * nblk ? dW[i] : nullptr;
    a.lda = lda; a.ldg = ldg; a.kblk = kblk; a.nblk = nblk; a.R = R;
    // aim for ~2 waves of CTAs over 148 SMs
    int per = kblk * nblk * 4;
    int chunks = (296 + per - 1) / per;
    int rows = (R + chunks - 1) / chunks;
    rows = ((rows + 15) / 16) * 16;
    if (rows < 64) rows = 64;
    a.rows_per_cta = rows;
    dim3 grid((R + rows - 1) / rows, 4, kblk * nblk);
    wgrad_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(a);
    return scann_check_launch("scann_dense_wgrad");
}

extern "C" int scann_layernorm_backward(const float* dy, const float* v, const float* gamma, int R, float* dv,
                                        float* dv2, int ld2, float* dgamma, float* dbeta, void* stream) {
    if (R <= 0) return 0;
    int grid = (R + 31) / 32;
    if (grid > 592) grid = 592;
    scann_launch(ln_bwd_kernel, dim3(grid), dim3(256), 0, stream, dy, v, gamma, R, dv, dv2, ld2, dgamma, dbeta);
    return scann_check_launch("scann_layernorm_backward");
}

extern "C" int scann_la_nopair_forward(const int32_t* cnt, const float* proj, int R, const float* gamma,
                                       const float* beta, float* ctx_pre, float* out, void* stream) {
    if (R <= 0) return 0;
    scann_launch(la_nopair_fwd_kernel, dim3((R + 7) / 8), dim3(256), 0, stream, cnt, proj, R, gamma, beta, ctx_pre, out);
    return scann_check_launch("scann_la_nopair_forward");
}

extern "C" int scann_transpose_blocks(const float* src, float* dst, const int32_t* offsets, int nblocks,
                                      void* stream) {
    if (nblocks <= 0) return 0;
    transpose_blocks_kernel<<<dim3(nblocks, 16), 256, 0, (cudaStream_t)stream>>>(src, dst, offsets);
    return scann_check_launch("scann_transpose_blocks");
}
