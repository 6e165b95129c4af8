// Batch plan: padded [B,M,N] neighbour lists -> tile-padded packed pair layout.
//
// The reference keeps every (atom, neighbour-slot) pair of the padded batch and masks
// the invalid ones (scann/utils/datagenerator.py:80-101, scann/layers/attention.py:186-206).
// Masked slots never reach a model output (their softmax weight is exactly 0 in fp32 and
// the context sum multiplies by the mask again), so the kernels only materialise VALID
// pairs.  Pairs of one centre atom stay contiguous (slot order preserved) and are grouped
// into tiles of at most `tile_rows` (<= tile_stride) rows that never split an atom; the caller picks
// tile_rows so that the tile count fills whole waves of SMs (the kernels' cost per tile is roughly
// proportional to its rows).  Tile t owns rows [t*tile_stride, (t+1)*tile_stride) of every per-pair tensor
// (tile_stride = 128, or 64 when the local-attention kernels run two warp groups per CTA); unused rows are
// padding (pair_c = -1).
#include "common.cuh"

#define PLAN_GSZ 128   // atom rows per greedy group (one thread walks one group)

__global__ void plan_count_kernel(const uint8_t* __restrict__ nmask, const int32_t* __restrict__ nbr,
                                  int R, int M, int N, int32_t* __restrict__ cnt, int32_t* __restrict__ status) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    const uint8_t* m = nmask + (size_t)r * N;
    const int32_t* j = nbr + (size_t)r * N;
    int c = 0, bad = 0;
    for (int n = 0; n < N; ++n) {
        if (m[n]) {
            ++c;
            int v = j[n];
            bad |= (v < 0) | (v >= M);
        }
    }
    if (c > SCANN_TILE) { atomicOr(status, SCANN_ERR_TOO_MANY_NBRS); c = 0; }
    if (bad) { atomicOr(status, SCANN_ERR_BAD_NEIGHBOR); c = 0; }
    cnt[r] = c;
}

// One thread per group of PLAN_GSZ consecutive atom rows: greedy first-fit in order.
// rowptr[r] <- local_tile*128 + offset (group-local); gtiles[g] <- tiles used by the group.
__global__ void plan_group_kernel(const int32_t* __restrict__ cnt, int R, int ngroups, int tile_rows, int tile_stride,
                                  int32_t* __restrict__ rowptr, int32_t* __restrict__ gtiles,
                                  int32_t* __restrict__ gcount) {
    __shared__ int32_t s_cnt[32 * (PLAN_GSZ + 1)];
    int g0 = blockIdx.x * 32;
    for (int i = threadIdx.x; i < 32 * PLAN_GSZ; i += blockDim.x) {
        int g = i / PLAN_GSZ, a = i % PLAN_GSZ;
        int r = (g0 + g) * PLAN_GSZ + a;
        s_cnt[g * (PLAN_GSZ + 1) + a] = (r < R) ? cnt[r] : 0;
    }
    __syncthreads();
    int g = g0 + threadIdx.x;
    if (threadIdx.x >= 32 || g >= ngroups) return;
    int32_t* sc = s_cnt + threadIdx.x * (PLAN_GSZ + 1);
    int tile = 0, fill = 0, any = 0, pairs = 0;
    for (int a = 0; a < PLAN_GSZ; ++a) {
        int c = sc[a];
        pairs += c;
        if (c == 0) { sc[a] = -1; continue; }
        if (fill + c > tile_rows && fill > 0) { ++tile; fill = 0; }
        sc[a] = tile * tile_stride + fill;
        fill += c;
        any = 1;
    }
    gtiles[g] = any ? tile + 1 : 0;
    if (gcount) gcount[g] = pairs;
    __syncwarp();
    for (int a = 0; a < PLAN_GSZ; ++a) {
        int r = g * PLAN_GSZ + a;
        if (r < R) rowptr[r] = sc[a];
    }
}

// Exclusive scan of gtiles (single CTA) -> gbase ; total -> ntiles.
__global__ void plan_scan_kernel(const int32_t* __restrict__ gtiles, int ngroups, int tile_cap,
                                 int32_t* __restrict__ gbase, int32_t* __restrict__ ntiles,
                                 int32_t* __restrict__ status, const int32_t* __restrict__ gcount,
                                 int32_t* __restrict__ gcbase, int32_t* __restrict__ nvalid) {
    __shared__ int32_t s_part[1024];
    __shared__ int32_t s_cpart[1024];
    int per = (ngroups + blockDim.x - 1) / blockDim.x;
    int lo = threadIdx.x * per, hi = min(lo + per, ngroups);
    int sum = 0, csum = 0;
    for (int g = lo; g < hi; ++g) { sum += gtiles[g]; if (gcount) csum += gcount[g]; }
    s_part[threadIdx.x] = sum;
    s_cpart[threadIdx.x] = csum;
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0, crun = 0;
        for (int i = 0; i < (int)blockDim.x; ++i) {
            int v = s_part[i]; s_part[i] = run; run += v;
            int c = s_cpart[i]; s_cpart[i] = crun; crun += c;
        }
        if (run > tile_cap) { atomicOr(status, SCANN_ERR_TILE_OVERFLOW); run = 0; crun = 0; }
        *ntiles = run;
        if (nvalid) *nvalid = crun;
    }
    __syncthreads();
    int run = s_part[threadIdx.x], crun = s_cpart[threadIdx.x];
    for (int g = lo; g < hi; ++g) {
        gbase[g] = run; run += gtiles[g];
        if (gcount) { gcbase[g] = crun; crun += gcount[g]; }
    }
}

__global__ void plan_fill_kernel(const uint8_t* __restrict__ nmask, const int32_t* __restrict__ nbr,
                                 const float* __restrict__ dist, const float* __restrict__ weight,
                                 const int32_t* __restrict__ cnt, const int32_t* __restrict__ gbase,
                                 const int32_t* __restrict__ ntiles, int R, int M, int N, int tile_stride,
                                 int32_t* __restrict__ rowptr, int32_t* __restrict__ tile_a0,
                                 int32_t* __restrict__ tile_a1, int32_t* __restrict__ pair_c,
                                 int32_t* __restrict__ pair_j, int32_t* __restrict__ pair_slot,
                                 float* __restrict__ pair_d, float* __restrict__ pair_w,
                                 int32_t* __restrict__ valid_rows, int32_t* __restrict__ valid_j,
                                 const int32_t* __restrict__ gcbase) {
    // one CTA = one plan group (blockDim = PLAN_GSZ): the compact position of an atom's pairs is the group's base
    // plus the exclusive prefix of cnt inside the group, so the compact list follows the tile order (sequential
    // reads for its consumers)
    __shared__ int32_t s_wsum[PLAN_GSZ / 32];
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    int c = r < R ? cnt[r] : 0;
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int v = __shfl_up_sync(0xffffffffu, incl, o);
        if ((int)(threadIdx.x & 31) >= o) incl += v;
    }
    if ((threadIdx.x & 31) == 31) s_wsum[threadIdx.x >> 5] = incl;
    __syncthreads();
    int wbase = 0;
    for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) wbase += s_wsum[w];
    const int vbase = valid_rows ? gcbase[blockIdx.x] + wbase + incl - c : 0;
    if (r >= R) return;
    if (c == 0 || *ntiles == 0) { rowptr[r] = 0; return; }
    int rp = gbase[r / PLAN_GSZ] * tile_stride + rowptr[r];
    rowptr[r] = rp;
    int tile = rp / tile_stride;
    if (rp % tile_stride == 0) tile_a0[tile] = r;
    atomicMax(&tile_a1[tile], r + 1);
    int b = r / M;
    const uint8_t* m = nmask + (size_t)r * N;
    int k = 0;
    for (int n = 0; n < N; ++n) {
        if (m[n]) {
            size_t s = (size_t)r * N + n;
            int p = rp + k;
            if (valid_rows) { valid_rows[vbase + k] = p; valid_j[vbase + k] = b * M + nbr[s]; }
            ++k;
            pair_c[p] = r;
            pair_j[p] = b * M + nbr[s];
            pair_slot[p] = (int32_t)s;
            pair_d[p] = dist[s];
            pair_w[p] = weight[s];
        }
    }
}

// The four kernels above in ONE launch of one CTA per plan group (PLAN_GSZ atom rows, one thread per row).  As
// separate launches the plan costs ~45 us of a 1.2 ms QM9 train step and of a 0.4 ms inference step (four dependent
// launches, two of them single-CTA serial loops); here a CTA counts its rows, thread 0 packs them greedily out of
// shared memory, the CTA publishes (tiles, pairs) of its group and picks up the sums over the lower groups
// (decoupled look-back: a CTA only ever waits for CTAs with a smaller index, which the hardware schedules first),
// then fills its own pairs.  Same algorithm, same plan (tests/test_gpu_parity.py::
// test_plan_gathers_and_masks_bit_exact runs both forms).
//
// sync[0] = epoch, sync[1] = ticket, sync[2 + g] = published word of group g, 64 bit:
// (epoch + 1) << 32 | pairs << 12 | tiles.  Words of earlier launches carry an older epoch, so nothing has to be
// cleared between launches (the buffer is zeroed once, when it is allocated); the last CTA to finish advances
// the epoch.
__global__ void __launch_bounds__(PLAN_GSZ) plan_chain_kernel(
    const uint8_t* __restrict__ nmask, const int32_t* __restrict__ nbr, const float* __restrict__ dist,
    const float* __restrict__ weight, int R, int M, int N, int ngroups, int tile_cap, int tile_rows, int tile_stride,
    int32_t* __restrict__ cnt, int32_t* __restrict__ rowptr, int32_t* __restrict__ tile_a0, int32_t* __restrict__ tile_a1,
    int32_t* __restrict__ ntiles, int32_t* __restrict__ pair_c, int32_t* __restrict__ pair_j,
    int32_t* __restrict__ pair_slot, float* __restrict__ pair_d, float* __restrict__ pair_w,
    int32_t* __restrict__ valid_rows, int32_t* __restrict__ valid_j, int32_t* __restrict__ nvalid,
    unsigned long long* __restrict__ sync, int32_t* __restrict__ status) {
    __shared__ int32_t s_cnt[PLAN_GSZ];
    __shared__ int32_t s_rp[PLAN_GSZ];            // (pairs of the group before the atom) << 16 | group-local row
    __shared__ int32_t s_red[2][PLAN_GSZ / 32];
    __shared__ int32_t s_own[2], s_base[2];
    const int tid = threadIdx.x, g = blockIdx.x, r = g * PLAN_GSZ + tid;
    const unsigned epoch = (unsigned)*reinterpret_cast<volatile unsigned long long*>(sync) + 1u;
    // ---- valid neighbours of this thread's atom row
    int c = 0;
    if (r < R) {
        const uint8_t* m = nmask + (size_t)r * N;
        const int32_t* j = nbr + (size_t)r * N;
        int bad = 0;
        // unconditional loads, selected afterwards: a load behind `if (m[n])` would make every slot a dependent
        // round trip through L2
#pragma unroll 4
        for (int n = 0; n < N; ++n) {
            const int mm = m[n], v = j[n];
            if (mm) {
                ++c;
                bad |= (v < 0) | (v >= M);
            }
        }
        if (c > SCANN_TILE) { atomicOr(status, SCANN_ERR_TOO_MANY_NBRS); c = 0; }
        if (bad) { atomicOr(status, SCANN_ERR_BAD_NEIGHBOR); c = 0; }
        cnt[r] = c;
    }
    s_cnt[tid] = c;
    __syncthreads();
    // ---- greedy first-fit in row order (thread 0), publish the group's totals
    if (tid == 0) {
        int tile = 0, fill = 0, any = 0, pairs = 0;
#pragma unroll 8
        for (int a = 0; a < PLAN_GSZ; ++a) {
            const int ca = s_cnt[a];
            if (ca != 0) {
                if (fill + ca > tile_rows && fill > 0) { ++tile; fill = 0; }
                s_rp[a] = (pairs << 16) | (tile * tile_stride + fill);
                fill += ca;
                pairs += ca;
                any = 1;
            }
        }
        const int tiles = any ? tile + 1 : 0;
        s_own[0] = tiles;
        s_own[1] = pairs;
        const unsigned long long word = ((unsigned long long)epoch << 32) | ((unsigned long long)pairs << 12) | (unsigned)tiles;
        asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(sync + 2 + g), "l"(word) : "memory");
    }
    // ---- look back: sums over the groups below this one (thread i waits for group i)
    int bt = 0, bp = 0;
    for (int i = tid; i < g; i += PLAN_GSZ) {
        unsigned long long w;
        do {
            asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(w) : "l"(sync + 2 + i) : "memory");
        } while ((unsigned)(w >> 32) != epoch);
        bt += (int)(w & 0xfffu);
        bp += (int)((w >> 12) & 0xfffffu);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        bt += __shfl_xor_sync(0xffffffffu, bt, o);
        bp += __shfl_xor_sync(0xffffffffu, bp, o);
    }
    if ((tid & 31) == 0) { s_red[0][tid >> 5] = bt; s_red[1][tid >> 5] = bp; }
    __syncthreads();
    if (tid == 0) {
        int t = 0, p = 0;
        for (int w = 0; w < PLAN_GSZ / 32; ++w) { t += s_red[0][w]; p += s_red[1][w]; }
        s_base[0] = t;
        s_base[1] = p;
    }
    __syncthreads();
    const int gbase = s_base[0], gcbase = s_base[1];
    const bool overflow = gbase + s_own[0] > tile_cap;
    if (g == ngroups - 1 && tid == 0) {          // the last group knows the totals
        int run = gbase + s_own[0], crun = gcbase + s_own[1];
        if (run > tile_cap) { run = 0; crun = 0; }
        *ntiles = run;
        if (valid_rows) *nvalid = crun;
    }
    if (overflow && tid == 0) atomicOr(status, SCANN_ERR_TILE_OVERFLOW);
    // ---- the pairs of this thread's atom into its tile rows (and the compact list, which follows the tile order)
    if (r < R) {
        if (c == 0 || overflow) {
            rowptr[r] = 0;
        } else {
            const int packed = s_rp[tid];
            const int rp = gbase * tile_stride + (packed & 0xffff);
            const int vbase = gcbase + (packed >> 16);
            rowptr[r] = rp;
            const int tile = rp / tile_stride;
            if (rp % tile_stride == 0) tile_a0[tile] = r;
            atomicMax(&tile_a1[tile], r + 1);
            const int b = r / M;
            const uint8_t* m = nmask + (size_t)r * N;
            int k = 0;
#pragma unroll 4
            for (int n = 0; n < N; ++n) {
                const size_t s = (size_t)r * N + n;
                const int mm = m[n], jn = nbr[s];
                const float dn = dist[s], wn = weight[s];
                if (mm) {
                    const int p = rp + k;
                    const int j = b * M + jn;
                    if (valid_rows) { valid_rows[vbase + k] = p; valid_j[vbase + k] = j; }
                    ++k;
                    pair_c[p] = r;
                    pair_j[p] = j;
                    pair_slot[p] = (int32_t)s;
                    pair_d[p] = dn;
                    pair_w[p] = wn;
                }
            }
        }
    }
    // ---- the last CTA to get here advances the epoch (every published word of this launch has been consumed:
    // a CTA passes its look-back before it takes a ticket)
    __syncthreads();
    if (tid == 0) {
        const unsigned long long t = atomicAdd(sync + 1, 1ull);
        if (t == (unsigned long long)(ngroups - 1)) {
            sync[1] = 0ull;
            __threadfence();
            *reinterpret_cast<volatile unsigned long long*>(sync) = (unsigned long long)epoch;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Ragged (CSR) batch -> padded device buffers: DataIterator.__getitem__ (scann/utils/datagenerator.py:69-135) on
// the device.  One thread per padded neighbour slot (b, m, n), so that the [R, N] stores of a warp are contiguous;
// the n == 0 thread of a row also writes the row's atom fields.  Neighbour value 1000 is the reference's padding
// marker (mask = idx != 1000, index reset to 0; datagenerator.py:82-90); weights / distances are zero padded;
// atom_mask = Z != 0.
// kGather = false (scann_pack_batch): batch structure b is structure b of the CSR batch (offsets from 0, one blob
// copied from the host).  kGather = true (scann_gather_batch): batch structure b is structure sel[b] of a
// device-resident data set, and target[b] = tgt[sel[b]].
// ---------------------------------------------------------------------------------------------
template <bool kGather>
__global__ void pack_batch_kernel(const int32_t* __restrict__ sel, const int32_t* __restrict__ sa,
                                  const int32_t* __restrict__ an, const int32_t* __restrict__ z,
                                  const int32_t* __restrict__ idx, const float* __restrict__ w,
                                  const float* __restrict__ d, const int32_t* __restrict__ ring,
                                  const float* __restrict__ tgt, int B, int M, int N,
                                  int32_t* __restrict__ atomic, uint8_t* __restrict__ atom_mask,
                                  int32_t* __restrict__ nbr, uint8_t* __restrict__ nmask, float* __restrict__ weight,
                                  float* __restrict__ dist, float* __restrict__ ring_out, float* __restrict__ target) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (tgt && t < B) target[t] = tgt[kGather ? sel[t] : t];
    if (t >= B * M * N) return;
    const int r = t / N, n = t - r * N;
    const int b = r / M, m = r - b * M;
    const int s = kGather ? sel[b] : b;
    const int a0 = sa[s], n_at = sa[s + 1] - a0;
    int p0 = 0, k = 0, a = -1;
    if (m < n_at) { a = a0 + m; p0 = an[a]; k = an[a + 1] - p0; }
    if (n == 0) {
        const int Z = a >= 0 ? z[a] : 0;
        atomic[r] = Z;
        atom_mask[r] = Z != 0;
        if (ring_out) {
            ring_out[(size_t)r * 2] = a >= 0 ? (float)ring[(size_t)a * 2] : 0.f;
            ring_out[(size_t)r * 2 + 1] = a >= 0 ? (float)ring[(size_t)a * 2 + 1] : 0.f;
        }
    }
    int j = 0;
    bool valid = false;
    float wv = 0.f, dv = 0.f;
    if (n < k) {
        j = idx[p0 + n];
        valid = j != 1000;
        if (!valid) j = 0;
        wv = w[p0 + n];
        dv = d[p0 + n];
    }
    nbr[t] = j; nmask[t] = valid; weight[t] = wv; dist[t] = dv;
}

static int pack_shape_ok(const char* who, int B, int M, int N) {
    if (B <= 0 || M <= 0 || N <= 0) { scann_set_error("%s: bad shape B=%d M=%d N=%d", who, B, M, N); return 0; }
    if ((long long)B * M * N > 0x7fffffffLL) {
        scann_set_error("%s: B*M*N = %lld neighbour slots exceed int32", who, (long long)B * M * N);
        return 0;
    }
    return 1;
}

// csr: device blob; off_*: byte offsets of struct_atom_off [B+1], atom_nbr_off [A+1], z [A], nbr_idx / nbr_w / nbr_d [P],
// ring [A,2] int32 (or < 0), target [B] (or < 0).  Outputs: the padded arrays of the reference's input dict.
extern "C" int scann_pack_batch(const void* csr, long long off_sa, long long off_an, long long off_z, long long off_idx,
                                long long off_w, long long off_d, long long off_ring, long long off_target, int B, int M,
                                int N, int32_t* atomic, uint8_t* atom_mask, int32_t* neighbors, uint8_t* neighbor_mask,
                                float* weight, float* dist, float* ring_out, float* target, void* stream) {
    if (!pack_shape_ok("pack_batch", B, M, N)) return 1;
    const char* p = (const char*)csr;
    const int T = B * M * N;
    pack_batch_kernel<false><<<(max(T, B) + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        nullptr, (const int32_t*)(p + off_sa), (const int32_t*)(p + off_an), (const int32_t*)(p + off_z),
        (const int32_t*)(p + off_idx), (const float*)(p + off_w), (const float*)(p + off_d),
        off_ring >= 0 ? (const int32_t*)(p + off_ring) : nullptr, off_target >= 0 ? (const float*)(p + off_target) : nullptr,
        B, M, N, atomic, atom_mask, neighbors, neighbor_mask, weight, dist, off_ring >= 0 ? ring_out : nullptr, target);
    return scann_check_launch("scann_pack_batch");
}

extern "C" int scann_gather_batch(const int32_t* struct_atom_off, const int32_t* atom_nbr_off, const int32_t* z,
                                  const int32_t* nbr_idx, const float* nbr_w, const float* nbr_d, const int32_t* ring,
                                  const float* target_in, const int32_t* sel, int B, int M, int N, int32_t* atomic,
                                  uint8_t* atom_mask, int32_t* neighbors, uint8_t* neighbor_mask, float* weight,
                                  float* dist, float* ring_out, float* target, void* stream) {
    if (!pack_shape_ok("gather_batch", B, M, N)) return 1;
    if (!sel) { scann_set_error("gather_batch: sel is NULL"); return 1; }
    const int T = B * M * N;
    pack_batch_kernel<true><<<(max(T, B) + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        sel, struct_atom_off, atom_nbr_off, z, nbr_idx, nbr_w, nbr_d, ring, target_in, B, M, N, atomic, atom_mask,
        neighbors, neighbor_mask, weight, dist, ring ? ring_out : nullptr, target_in ? target : nullptr);
    return scann_check_launch("scann_gather_batch");
}

extern "C" int scann_plan_build(const uint8_t* neighbor_mask, const int32_t* neighbors, const float* dist,
                                const float* weight, int B, int M, int N, int tile_cap, int tile_rows,
                                int tile_stride, int32_t* cnt,
                                int32_t* rowptr, int32_t* tile_a0, int32_t* tile_a1, int32_t* ntiles,
                                int32_t* pair_c, int32_t* pair_j, int32_t* pair_slot, float* pair_d,
                                float* pair_w, int32_t* valid_rows, int32_t* valid_j, int32_t* nvalid, int32_t* scratch,
                                int scratch_len,
                                int32_t* status, void* stream_) {
    cudaStream_t st = (cudaStream_t)stream_;
    long long Rll = (long long)B * M;
    if (Rll <= 0 || N <= 0 || Rll * N > 0x7fffffffLL) { scann_set_error("plan: bad shape B=%d M=%d N=%d", B, M, N); return 1; }
    if (tile_stride != 32 && tile_stride != 64 && tile_stride != SCANN_TILE) { scann_set_error("plan: tile_stride must be 32, 64 or 128"); return 1; }
    if (tile_rows < 1 || tile_rows > tile_stride) { scann_set_error("plan: tile_rows must be in 1..tile_stride"); return 1; }
    int R = (int)Rll;
    int ngroups = (R + PLAN_GSZ - 1) / PLAN_GSZ;
    if (valid_rows && !valid_j) { scann_set_error("plan: valid_rows needs valid_j"); return 1; }
    const int need = (valid_rows ? 4 : 2) * ngroups;
    if (scratch_len < need) { scann_set_error("plan: scratch too small (%d < %d)", scratch_len, need); return 1; }
    int32_t* gtiles = scratch;
    int32_t* gbase = scratch + ngroups;
    int32_t* gcount = valid_rows ? scratch + 2 * ngroups : nullptr;
    int32_t* gcbase = valid_rows ? scratch + 3 * ngroups : nullptr;
    size_t rows = (size_t)tile_cap * tile_stride;
    // padding rows are recognised by pair_c < 0; every consumer guards on it, so the other
    // per-pair arrays need no initialisation.  tile_a1 is built with atomicMax.
    cudaMemsetAsync(pair_c, 0xFF, rows * sizeof(int32_t), st);
    cudaMemsetAsync(tile_a1, 0, (size_t)tile_cap * sizeof(int32_t), st);
    // one launch (decoupled look-back over the plan groups) when the caller's scratch has room for the 64-bit
    // words behind the 4 * ngroups ints of the four-kernel form (and the buffer is 8-byte aligned)
    const int sync_off = (4 * ngroups + 1) & ~1;
    if (!scann_plan_unfused() && scratch_len >= sync_off + 2 * (ngroups + 2) && ((uintptr_t)scratch & 7) == 0 &&
        ngroups < 4096) {
        plan_chain_kernel<<<ngroups, PLAN_GSZ, 0, st>>>(neighbor_mask, neighbors, dist, weight, R, M, N, ngroups, tile_cap,
                                                       tile_rows, tile_stride, cnt, rowptr, tile_a0, tile_a1, ntiles, pair_c,
                                                       pair_j, pair_slot, pair_d, pair_w, valid_rows, valid_j,
                                                       valid_rows ? nvalid : nullptr,
                                                       reinterpret_cast<unsigned long long*>(scratch + sync_off), status);
        return scann_check_launch("scann_plan_build");
    }
    plan_count_kernel<<<(R + 255) / 256, 256, 0, st>>>(neighbor_mask, neighbors, R, M, N, cnt, status);
    plan_group_kernel<<<(ngroups + 31) / 32, 128, 0, st>>>(cnt, R, ngroups, tile_rows, tile_stride, rowptr, gtiles, gcount);
    plan_scan_kernel<<<1, 1024, 0, st>>>(gtiles, ngroups, tile_cap, gbase, ntiles, status, gcount, gcbase,
                                         valid_rows ? nvalid : nullptr);
    plan_fill_kernel<<<(R + PLAN_GSZ - 1) / PLAN_GSZ, PLAN_GSZ, 0, st>>>(neighbor_mask, neighbors, dist, weight, cnt, gbase, ntiles, R, M,
                                                     N, tile_stride, rowptr, tile_a0, tile_a1, pair_c, pair_j, pair_slot, pair_d,
                                                     pair_w, valid_rows, valid_j, gcbase);
    return scann_check_launch("scann_plan_build");
}

// ---------------------------------------------------------------------------------------------
// Local-attention scores: pair-plan order -> the user's layouts.  The forward kernels store the softmax of every
// valid pair through their `attn` pointer, [rows, 8] per layer in plan order (layer l at attn + l * rows * 8).
// ---------------------------------------------------------------------------------------------

// out [L][B][8][M][N], the first output of LocalAttention.call (scann/layers/attention.py:186-189, :216).  One thread
// per padded slot (b, m, n) and layer (blockIdx.y): it reads the slot's 8 heads in one 32-byte row and writes them to
// 8 planes, so the stores of a warp are contiguous in n and m.  The plan keeps an atom's pairs contiguous and in slot
// order (plan_fill_kernel), so valid slot n of row r is plan row rowptr[r] + (valid slots of row r before n).
__global__ void attn_to_padded_kernel(const float* __restrict__ attn, long long rows, const int32_t* __restrict__ cnt,
                                      const int32_t* __restrict__ rowptr, const uint8_t* __restrict__ nmask, int B,
                                      int M, int N, float* __restrict__ out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int T = B * M * N;
    if (t >= T) return;
    const int l = blockIdx.y;
    const int r = t / N, n = t - r * N;
    const int b = r / M, mn = t - b * M * N;
    const size_t plane = (size_t)M * N;
    float* o = out + ((size_t)l * B + b) * 8 * plane + mn;
    const int c = cnt[r];
    if (c == 0) {
        // no valid neighbour: the mask adds -1e9 to every logit, which absorbs |s| < 32 in fp32, so the softmax of
        // the N equal logits is uniform
        const float u = 1.0f / (float)N;
#pragma unroll
        for (int h = 0; h < 8; ++h) o[h * plane] = u;
        return;
    }
    const uint8_t* m = nmask + (size_t)r * N;
    if (!m[n]) {
#pragma unroll
        for (int h = 0; h < 8; ++h) o[h * plane] = 0.0f;
        return;
    }
    int k = 0;
    for (int j = 0; j < n; ++j) k += m[j] != 0;
    const float4* a = reinterpret_cast<const float4*>(attn + ((size_t)l * rows + rowptr[r] + k) * 8);
    const float4 a0 = a[0], a1 = a[1];
    o[0] = a0.x; o[plane] = a0.y; o[2 * plane] = a0.z; o[3 * plane] = a0.w;
    o[4 * plane] = a1.x; o[5 * plane] = a1.y; o[6 * plane] = a1.z; o[7 * plane] = a1.w;
}

// out [L][8][ld]: the compact list of the plan (valid_rows, nvalid) holds the valid pairs in atom-row order and, per
// atom, in slot order, so entry i of the list is pair i of the batch's CSR neighbour lists whenever those lists carry
// no padding marker.  One thread per list entry and layer.
__global__ void attn_to_csr_kernel(const float* __restrict__ attn, long long rows, const int32_t* __restrict__ valid_rows,
                                   const int32_t* __restrict__ nvalid, int ld, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ld || i >= *nvalid) return;
    const int l = blockIdx.y;
    const float4* a = reinterpret_cast<const float4*>(attn + ((size_t)l * rows + valid_rows[i]) * 8);
    const float4 a0 = a[0], a1 = a[1];
    float* o = out + (size_t)l * 8 * ld + i;
    o[0] = a0.x; o[(size_t)ld] = a0.y; o[2 * (size_t)ld] = a0.z; o[3 * (size_t)ld] = a0.w;
    o[4 * (size_t)ld] = a1.x; o[5 * (size_t)ld] = a1.y; o[6 * (size_t)ld] = a1.z; o[7 * (size_t)ld] = a1.w;
}

static int attn_args_ok(const char* who, const float* attn, int L, long long rows, const float* out) {
    if (L <= 0 || L > 65535) { scann_set_error("%s: bad layer count L=%d", who, L); return 0; }
    if (rows <= 0 || rows > 0x7fffffffLL) { scann_set_error("%s: bad plan row count %lld", who, rows); return 0; }
    if (!attn || !out) { scann_set_error("%s: attn / out is NULL", who); return 0; }
    if ((uintptr_t)attn & 15) { scann_set_error("%s: attn must be 16-byte aligned", who); return 0; }
    return 1;
}

extern "C" int scann_attn_to_padded(const float* attn, int L, long long rows, const int32_t* cnt, const int32_t* rowptr,
                                    const uint8_t* neighbor_mask, int B, int M, int N, float* out, void* stream) {
    if (!attn_args_ok("attn_to_padded", attn, L, rows, out)) return 1;
    if (!pack_shape_ok("attn_to_padded", B, M, N)) return 1;
    if ((long long)B * 8 * M * N > 0x7fffffffLL) {
        scann_set_error("attn_to_padded: B*8*M*N = %lld scores per layer exceed int32", (long long)B * 8 * M * N);
        return 1;
    }
    if (!cnt || !rowptr || !neighbor_mask) { scann_set_error("attn_to_padded: cnt / rowptr / neighbor_mask is NULL"); return 1; }
    const int T = B * M * N;
    attn_to_padded_kernel<<<dim3((T + 255) / 256, L), 256, 0, (cudaStream_t)stream>>>(attn, rows, cnt, rowptr,
                                                                                      neighbor_mask, B, M, N, out);
    return scann_check_launch("scann_attn_to_padded");
}

extern "C" int scann_attn_to_csr(const float* attn, int L, long long rows, const int32_t* valid_rows,
                                 const int32_t* nvalid, int ld, float* out, void* stream) {
    if (!attn_args_ok("attn_to_csr", attn, L, rows, out)) return 1;
    if (ld <= 0) { scann_set_error("attn_to_csr: bad ld=%d", ld); return 1; }
    if (!valid_rows || !nvalid) { scann_set_error("attn_to_csr: valid_rows / nvalid is NULL"); return 1; }
    attn_to_csr_kernel<<<dim3((ld + 255) / 256, L), 256, 0, (cudaStream_t)stream>>>(attn, rows, valid_rows, nvalid, ld, out);
    return scann_check_launch("scann_attn_to_csr");
}
