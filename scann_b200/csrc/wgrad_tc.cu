// All weight-gradient GEMMs of one train step in ONE persistent launch (tcgen05, kind::tf32, 3xTF32).
//
// Every Dense kernel gradient of the graph is a reduction over rows, dW = X^T Y (TF autodiff of the Dense /
// einsum layers in scann/layers/attention.py:118-216 and scann/models/scann_model.py:424-447 inside keras fit):
//   * per pair  : key/kernel      += (x[j] * g')^T d_k        filter_geo rows 128..255 += g^T d_pre
//   * per atom  : filter_geo rows 0..127 / 256..383, query, ResidualNorm dense / dense_1, after_Lc,
//                 GlobalAttention query / key, bf_property  (+ the bias gradients = column sums of Y)
// They only feed the optimiser, so nothing in the backward chain waits for them.  Launched layer by layer on
// a side stream they cost more SM time than they hide (measured: 0.42 of the 1.59 ms step is lost to them,
// mostly per-launch partial-sum traffic: 148 CTAs x 64 KB x 2 per layer and wave quantisation).  Here the
// ~50 problems are concatenated into one list of 32-row units, the list is cut into equal contiguous ranges,
// one per CTA, and a CTA accumulates a problem's units in tensor memory and flushes each accumulator ONCE with
// vector atomics (red.global.add.v4.f32) straight into the gradient arena: no partial buffers, no reduce
// kernels, perfect balance.
//
// Operands are the MN-major SWIZZLE_128B_BASE32B images of tc_common.cuh (K = pair / atom rows).
#include "common.cuh"
#include "tc_common.cuh"

#define WG_THREADS 512
#define WG_WARPS 16
#define WG_MAX_PROBLEMS 96

// Mirrors ScannWgradProblem in include/scann_b200.h.
struct WgProblem {
    const float* X;      // [rows, ldx] left operand rows
    const float* Y;      // [rows, ldy] right operand rows
    const float* xg;     // pair problems: X rows are multiplied by xg[pair_j[row], :] ([R,128]); else NULL
    float* dW;           // [128,128], accumulated
    float* db;           // [128] += column sums of Y, nullable
    int ldx, ldy;
    int rows;            // >= 0: atom problem with this many rows ; < 0: pair problem (rows = ntiles * stride,
                         //       rows whose pair_c < 0 are padding)
    int pad;
};

struct WgArgs {
    const WgProblem* prob;
    int nprob;
    const int32_t* ntiles;
    int stride;
    const int32_t* pair_c;
    const int32_t* pair_j;
    const int32_t* valid_rows;   // compact list of the valid pair rows (scann_plan_build), nullable
    const int32_t* valid_j;      // neighbour atom row of each compact entry
    const int32_t* nvalid;       // its length (device)
    float* slots;                // deterministic form: [grid][2][128*128] partial dW of the shared problems
    float* bslots;               //                     [grid][2][128]     partial db
};

__device__ __forceinline__ void wg_split_store(uint8_t* sHi, uint8_t* sLo, uint32_t off, float4 v) {
    float4 h, l;
    tf32_split(v.x, h.x, l.x); tf32_split(v.y, h.y, l.y); tf32_split(v.z, h.z, l.z); tf32_split(v.w, h.w, l.w);
    *reinterpret_cast<float4*>(sHi + off) = h;
    *reinterpret_cast<float4*>(sLo + off) = l;
}

#define WG_UR 32                       // rows per unit (= K extent of one MMA group)
#define WG_NIMG 2                      // operand image sets: the split of unit u+1 overlaps the MMAs of unit u
#define WG_RPW (WG_UR / WG_WARPS)      // rows per warp per unit
#define WG_MNB ((uint32_t)WG_UR * 128u)          // one column block of an MN-major image: [UR rows x 32 columns]
#define WG_MNT (4u * WG_MNB)                     // one image [UR x 128] fp32 = 32 KB

__device__ __forceinline__ uint32_t wg_mn_off(int r, int c) {
    return (uint32_t)(c >> 5) * WG_MNB + (uint32_t)r * 128u + (((((uint32_t)c >> 3) & 3u) ^ ((uint32_t)r & 3u)) << 5) +
           ((uint32_t)c & 7u) * 4u;
}
__device__ __forceinline__ uint64_t wg_mn_desc(uint32_t saddr) { return tc_desc(saddr, WG_MNB, 512u) | ((uint64_t)1 << 61); }

// The problem a cursor currently points at, cached in registers: the table lives in shared memory and the shared-
// memory data pipe is this kernel's busiest unit (ncu, first version: LSU wavefronts 64 % + tensor-core operand
// reads 22 % of its peak), so it is only touched when a unit crosses a problem boundary (~50 times per CTA).
struct WgCursor {
    int p, ubase, uend;            // problem index, its first unit, one past its last unit
    const float *X, *Y, *xg;
    int ldx, ldy, nrows;
    bool pair;
};
// The raw operand rows of one unit, held in registers from the moment their loads are issued (two units ahead of
// their use) until they are split into the operand images.
struct WgRegs {
    float4 x[WG_RPW], y[WG_RPW], nb[WG_RPW];
    bool has_xg;
};

// Pipeline per CTA.  The inputs come from HBM (6 % L2 hit rate measured), so the loads of the next units must be
// in flight while the current one is split and multiplied:
//   LDG.128 of units u+1, u+2 in registers (64 KB in flight per SM) | regs(u) -> hi/lo split -> 4 MN-major images
//   (set u % 2) -> MMAs;  the split of unit u+1 overlaps the MMAs of unit u.
// The first version staged the raw rows through shared memory with cp.async; per unit that cost 256 wavefronts
// for the copies, 256 for reading them back and ~200 for the dummy LDS the compiler wraps around LDGSTS, on top of
// the 512 (split stores) + 752 (tensor-core reads) that are inherent: the kernel ran at 2.4 TB/s, bound by the
// shared-memory pipe, not by HBM.
// DET (deterministic mode, DESIGN.md section 4.7): a problem that lies entirely inside this CTA's unit range is STORED
// into dW / db; the first and the last problem of the range, which neighbouring CTAs may share, go to the CTA's two
// slots (slot 0: a problem that started before the range, slot 1: one that continues behind it), summed in CTA order
// by scann_wgrad_batch_reduce.  The bias column sums of the warps are combined in warp order.
template <bool DET>
__global__ void __launch_bounds__(WG_THREADS, 1) wgrad_batch_tc_kernel(const WgArgs a) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    // the BASE32B swizzle is a function of the absolute shared address: align the images to 1024 bytes
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    __shared__ uint64_t bars[WG_NIMG];
    __shared__ uint32_t tmem_base_s;
    __shared__ float s_db[SCANN_D];
    __shared__ int s_units[WG_MAX_PROBLEMS + 1];        // exclusive prefix of units per problem
    __shared__ WgProblem s_prob[WG_MAX_PROBLEMS];       // the problem table
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // pair problems run over the compact list of valid rows when the plan provides it (independent of how
    // sparsely the tiles are filled), else over all tile slots with the padding rows skipped
    const int pair_rows = a.valid_rows ? *a.nvalid : *a.ntiles * a.stride;
    for (int i = tid; i < a.nprob * (int)(sizeof(WgProblem) / 8); i += WG_THREADS)
        reinterpret_cast<uint64_t*>(s_prob)[i] = reinterpret_cast<const uint64_t*>(a.prob)[i];
    __syncthreads();
    if (tid == 0) {
        int run = 0;
        for (int p = 0; p < a.nprob; ++p) {
            s_units[p] = run;
            const int rows = s_prob[p].rows >= 0 ? s_prob[p].rows : pair_rows;
            run += (rows + WG_UR - 1) / WG_UR;
        }
        s_units[a.nprob] = run;
    }
    if (tid < SCANN_D) s_db[tid] = 0.f;
    if (warp == 0) tmem_alloc(&tmem_base_s, 256);
    if (tid < WG_NIMG) mbar_init(&bars[tid], 1);
    if (tid == 0) mbar_fence_init();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const int total = s_units[a.nprob];
    const long long G = gridDim.x;
    const int u_lo = (int)((long long)total * blockIdx.x / G), u_hi = (int)((long long)total * (blockIdx.x + 1) / G);
    const uint32_t t_dm = tmem_base_s, t_dc = tmem_base_s + 128;
    const uint32_t idesc = tc_idesc_tf32(128, 128, true, true);
    uint32_t phase[WG_NIMG];
    bool pending[WG_NIMG];          // an MMA group reading image set b is in flight (not yet waited for)
#pragma unroll
    for (int b = 0; b < WG_NIMG; ++b) { phase[b] = 0; pending[b] = false; }
    bool first = true;              // no MMA has been issued into the accumulators of the current problem
    float4 colsum = make_float4(0.f, 0.f, 0.f, 0.f);

    auto seek = [&](WgCursor& c, int u) {           // make c describe the problem of unit u (u < total)
        if (u < c.uend) return;
        while (u >= c.uend) { ++c.p; c.ubase = c.uend; c.uend = s_units[c.p + 1]; }
        const WgProblem& pr = s_prob[c.p];
        c.X = pr.X; c.Y = pr.Y; c.xg = pr.xg; c.ldx = pr.ldx; c.ldy = pr.ldy;
        c.pair = pr.rows < 0;
        c.nrows = c.pair ? pair_rows : pr.rows;
    };
    WgCursor ci{-1, 0, 0, nullptr, nullptr, nullptr, 0, 0, 0, false};      // indices are fetched for its unit
    WgCursor cl = ci;                                                      // loads are issued for its unit
    int pc = -1, pc_uend = 0;                                              // problem being multiplied

    // Source rows (and neighbour rows) of the unit that will be loaded NEXT, fetched one call ahead: otherwise
    // every load would start with a dependent L2 round trip.
    int src[WG_RPW], nbj[WG_RPW];
    auto fetch_idx = [&](int u) {
#pragma unroll
        for (int i = 0; i < WG_RPW; ++i) { src[i] = -1; nbj[i] = 0; }
        if (u >= u_hi) return;
        seek(ci, u);
        const int rowbase = (u - ci.ubase) * WG_UR;
#pragma unroll
        for (int i = 0; i < WG_RPW; ++i) {
            const int r = rowbase + warp + WG_WARPS * i;
            if (r < ci.nrows) {
                src[i] = r;
                if (ci.pair) {
                    if (a.valid_rows) {
                        src[i] = a.valid_rows[r];
                        if (ci.xg) nbj[i] = a.valid_j[r];         // independent of the load above: one round trip
                    } else {
                        if (a.pair_c[r] < 0) src[i] = -1;
                        if (ci.xg) nbj[i] = a.pair_j[r];
                    }
                }
            }
        }
    };
    // issue the loads of unit u into `s` (zeros for rows that do not exist), then fetch the indices of unit u + 1
    auto issue_load = [&](int u, WgRegs& s) {
        s.has_xg = false;
#pragma unroll
        for (int i = 0; i < WG_RPW; ++i) {
            s.x[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            s.y[i] = s.x[i];
            s.nb[i] = s.x[i];
        }
        if (u >= u_hi) return;
        seek(cl, u);
        s.has_xg = cl.xg != nullptr;
#pragma unroll
        for (int i = 0; i < WG_RPW; ++i) {
            if (src[i] >= 0) {
                s.x[i] = ld4(cl.X + (size_t)src[i] * cl.ldx + lane * 4);
                s.y[i] = ld4(cl.Y + (size_t)src[i] * cl.ldy + lane * 4);
                if (s.has_xg) s.nb[i] = ld4(cl.xg + (size_t)nbj[i] * SCANN_D + lane * 4);
            }
        }
        fetch_idx(u + 1);
    };
    // accumulators -> gradient arena (vector atomics), column sums -> bias gradient
    auto flush = [&](const WgProblem& pr) {
#pragma unroll
        for (int b = 0; b < WG_NIMG; ++b)
            if (pending[b]) { mbar_wait(&bars[b], phase[b]); phase[b] ^= 1; tc_fence_after(); pending[b] = false; }
        if (!first) {
            const int m = (warp & 3) * 32 + lane, nbase = (warp >> 2) * 32;
            // (DET) owned problem: dW itself; shared problem: this CTA's slot
            float* dW = pr.dW;
            float* db = pr.db;
            if constexpr (DET) {
                const int slot = (int)blockIdx.x * 2 + (s_units[pc] < u_lo ? 0 : 1);
                if (!(s_units[pc] >= u_lo && s_units[pc + 1] <= u_hi)) {
                    dW = a.slots + (size_t)slot * SCANN_D * SCANN_D;
                    db = a.bslots + (size_t)slot * SCANN_D;
                }
            }
            const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                float v[16], c[16];
                tmem_ld16(t_dm + lane_base + nbase + h * 16, v);
                tmem_ld16(t_dc + lane_base + nbase + h * 16, c);
                tmem_ld_wait();
#pragma unroll
                for (int q = 0; q < 16; q += 4) {
                    if constexpr (DET)
                        st4(dW + (size_t)m * SCANN_D + nbase + h * 16 + q,
                            make_float4(v[q] + c[q], v[q + 1] + c[q + 1], v[q + 2] + c[q + 2], v[q + 3] + c[q + 3]));
                    else
                        red_add4(pr.dW + (size_t)m * SCANN_D + nbase + h * 16 + q, v[q] + c[q], v[q + 1] + c[q + 1],
                                 v[q + 2] + c[q + 2], v[q + 3] + c[q + 3]);
                }
            }
            if constexpr (DET) {
                if (pr.db) {
                    for (int w = 0; w < WG_WARPS; ++w) {
                        if (warp == w) {
                            s_db[lane * 4 + 0] += colsum.x; s_db[lane * 4 + 1] += colsum.y;
                            s_db[lane * 4 + 2] += colsum.z; s_db[lane * 4 + 3] += colsum.w;
                        }
                        __syncthreads();
                    }
                }
                tc_fence_before();
                __syncthreads();             // every warp has read the accumulators; s_db is complete
                tc_fence_after();
                if (pr.db && tid < SCANN_D) {
                    db[tid] = s_db[tid];
                    s_db[tid] = 0.f;
                }
                __syncthreads();
            } else {
                if (pr.db) {
                    atomicAdd(&s_db[lane * 4 + 0], colsum.x); atomicAdd(&s_db[lane * 4 + 1], colsum.y);
                    atomicAdd(&s_db[lane * 4 + 2], colsum.z); atomicAdd(&s_db[lane * 4 + 3], colsum.w);
                }
                tc_fence_before();
                __syncthreads();                 // every warp has read the accumulators; s_db is complete
                tc_fence_after();
                if (pr.db && tid < SCANN_D) { atomicAdd(pr.db + tid, s_db[tid]); s_db[tid] = 0.f; }
                __syncthreads();
            }
        }
        first = true;
        colsum = make_float4(0.f, 0.f, 0.f, 0.f);
    };
    // one unit: registers -> operand images of set ib, refill the registers with unit u + 2, MMAs
    auto step = [&](int u, WgRegs& s, const int ib) {
        if (u >= pc_uend) {                  // next problem: hand over what was accumulated for the previous one
            while (u >= pc_uend) {
                if (pc >= 0) flush(s_prob[pc]);
                ++pc;
                pc_uend = s_units[pc + 1];
            }
        }
        uint8_t* sXh = smem + (size_t)ib * 4 * WG_MNT;
        uint8_t* sXl = sXh + WG_MNT;
        uint8_t* sYh = sXh + 2 * WG_MNT;
        uint8_t* sYl = sXh + 3 * WG_MNT;
        if (pending[ib]) {                   // the MMAs of unit u - 2 still read this image set
            mbar_wait(&bars[ib], phase[ib]);
            phase[ib] ^= 1;
            tc_fence_after();
            pending[ib] = false;
        }
#pragma unroll
        for (int i = 0; i < WG_RPW; ++i) {
            float4 xv = s.x[i];
            const float4 yv = s.y[i];
            if (s.has_xg) xv = make_float4(xv.x * s.nb[i].x, xv.y * s.nb[i].y, xv.z * s.nb[i].z, xv.w * s.nb[i].w);
            colsum = make_float4(colsum.x + yv.x, colsum.y + yv.y, colsum.z + yv.z, colsum.w + yv.w);
            const uint32_t off = wg_mn_off(warp + WG_WARPS * i, lane * 4);
            wg_split_store(sXh, sXl, off, xv);
            wg_split_store(sYh, sYl, off, yv);
        }
        issue_load(u + 2, s);                // the registers are free again: two units stay in flight
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        // (Round 2 experiments, both slower: the three products issued by three warps into three accumulators -- step
        // +35 us, 122 -> 157 us for this launch; eight splitter warps + a dedicated MMA warp behind named barriers -- 168
        // registers and 800 bytes of spills.  Kept: one issuing lane, two image sets.
        // Second session: the __syncthreads replaced by an mbarrier hand-over (every warp arrives on ready[set] and goes
        // on, warp 0 waits for the 16 arrives and issues; no CTA-wide barrier in the unit loop although the ncu source
        // page has 13.5 % of the samples there, gpurun_out/r02cb_prof.ncu-rep): 132 -> 157 us for this launch, QM9 step
        // 0.977 -> 0.999 ms, MP2018 1.752 -> 1.80 ms (profiles/r02_ab_wgrad_handover.log) -- the same 157 us as the
        // three-warp form: warps that drift apart cost more than the barrier.  A 17th, dedicated MMA warp leaves 96
        // registers per thread (five warps on one scheduler): 1 182 bytes of spills, not measured.  The kernel executes
        // 289 warp-instructions per warp and unit (cursor / index bookkeeping around 12 loads and 16 split stores) at
        // 48 % issue-slot use with shared memory at 26 % and DRAM at 44 %: instruction latency, not a pipe, bounds it.)
        if (warp == 0 && tc_elect_one()) {
            tc_fence_after();
            const uint64_t dxh = wg_mn_desc(smem_u32(sXh)), dxl = wg_mn_desc(smem_u32(sXl)), dyh = wg_mn_desc(smem_u32(sYh)),
                           dyl = wg_mn_desc(smem_u32(sYl));
#pragma unroll
            for (int ks = 0; ks < WG_UR / 8; ++ks)     // K-step = 8 rows = 1024 bytes of each image
                tc_mma_ss(t_dm, dxh + (uint64_t)(ks * 64), dyh + (uint64_t)(ks * 64), idesc, !(first && ks == 0));
#pragma unroll
            for (int ks = 0; ks < WG_UR / 8; ++ks)
                tc_mma_ss(t_dc, dxh + (uint64_t)(ks * 64), dyl + (uint64_t)(ks * 64), idesc, !(first && ks == 0));
#pragma unroll
            for (int ks = 0; ks < WG_UR / 8; ++ks)
                tc_mma_ss(t_dc, dxl + (uint64_t)(ks * 64), dyh + (uint64_t)(ks * 64), idesc, true);
            tc_commit(&bars[ib]);
        }
        pending[ib] = true;
        first = false;
    };

    WgRegs ra, rb;
    fetch_idx(u_lo);
    issue_load(u_lo, ra);
    issue_load(u_lo + 1, rb);
#pragma unroll 1
    for (int u = u_lo; u < u_hi; u += 2) {
        step(u, ra, 0);
        if (u + 1 < u_hi) step(u + 1, rb, 1);
    }
    if (u_hi > u_lo) flush(s_prob[pc]);
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base_s, 256);
}

#define WG_SMEM (WG_NIMG * 4 * WG_MNT + 1024)

// Sums the slots of every problem that several CTAs of a deterministic scann_wgrad_batch_tc_det launch of `grid` CTAs
// shared, in CTA order, and stores the result into dW / db.  One CTA per (problem, 2048 elements of dW).
__global__ void __launch_bounds__(256) wgrad_slot_reduce_kernel(const WgProblem* __restrict__ prob, int nprob, int grid,
                                                                const int32_t* __restrict__ ntiles, int stride,
                                                                const int32_t* __restrict__ nvalid,
                                                                const float* __restrict__ slots,
                                                                const float* __restrict__ bslots) {
    __shared__ int s_ub, s_ue, s_total;
    pdl_wait();
    const int p = blockIdx.y;
    if (threadIdx.x == 0) {
        const int pair_rows = nvalid ? *nvalid : *ntiles * stride;
        int run = 0, ub = 0, ue = 0;
        for (int q = 0; q < nprob; ++q) {
            if (q == p) ub = run;
            const int rows = prob[q].rows >= 0 ? prob[q].rows : pair_rows;
            run += (rows + WG_UR - 1) / WG_UR;
            if (q == p) ue = run;
        }
        s_ub = ub; s_ue = ue; s_total = run;
    }
    __syncthreads();
    const int ub = s_ub, ue = s_ue;
    const long long total = s_total, G = grid;
    if (ub >= ue) return;
    auto lo = [&](long long c) { return (int)(total * c / G); };
    int c0 = (int)((long long)ub * G / total);                  // the CTA whose range holds unit ub
    while (c0 + 1 < grid && lo(c0 + 1) <= ub) ++c0;
    while (c0 > 0 && lo(c0) > ub) --c0;
    if (lo(c0 + 1) >= ue) return;                                // one CTA owns the problem: it stored dW itself
    const WgProblem pr = prob[p];
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) * 8;  // 8 consecutive elements of dW per thread
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, bacc = 0.f;
    const bool bias = pr.db && blockIdx.x == 0 && threadIdx.x < SCANN_D;
    for (int c = c0; c < grid && lo(c) < ue; ++c) {
        if (lo(c) == lo(c + 1)) continue;                         // a CTA without units
        const size_t slot = (size_t)c * 2 + (ub < lo(c) ? 0 : 1);
        const float4 v0 = ld4(slots + slot * SCANN_D * SCANN_D + i), v1 = ld4(slots + slot * SCANN_D * SCANN_D + i + 4);
        acc[0] += v0.x; acc[1] += v0.y; acc[2] += v0.z; acc[3] += v0.w;
        acc[4] += v1.x; acc[5] += v1.y; acc[6] += v1.z; acc[7] += v1.w;
        if (bias) bacc += bslots[slot * SCANN_D + threadIdx.x];
    }
    st4(pr.dW + i, make_float4(acc[0], acc[1], acc[2], acc[3]));
    st4(pr.dW + i + 4, make_float4(acc[4], acc[5], acc[6], acc[7]));
    if (bias) pr.db[threadIdx.x] = bacc;
    pdl_trigger();
}

template <bool DET>
static int wgrad_batch_launch(int grid, const void* problems_dev, int nprob, const int32_t* ntiles, int tile_stride,
                              const int32_t* pair_c, const int32_t* pair_j, const int32_t* valid_rows,
                              const int32_t* valid_j, const int32_t* nvalid, float* slots, float* bslots, void* stream) {
    if (nprob < 1 || nprob > WG_MAX_PROBLEMS) { scann_set_error("wgrad_batch_tc: nprob must be in 1..%d", WG_MAX_PROBLEMS); return 1; }
    if (tile_stride != 32 && tile_stride != 64 && tile_stride != 128) { scann_set_error("wgrad_batch_tc: tile_stride must be 32, 64 or 128"); return 1; }
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(wgrad_batch_tc_kernel<DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WG_SMEM);
        if (e != cudaSuccess) { scann_set_error("wgrad_batch_tc: smem opt-in failed: %s", cudaGetErrorString(e)); return 1; }
        configured = true;
    }
    if (grid <= 0) return 0;
    WgArgs a{(const WgProblem*)problems_dev, nprob, ntiles, tile_stride, pair_c, pair_j, valid_rows, valid_j,
             valid_rows ? nvalid : nullptr, slots, bslots};
    wgrad_batch_tc_kernel<DET><<<grid, WG_THREADS, WG_SMEM, (cudaStream_t)stream>>>(a);
    return scann_check_launch("scann_wgrad_batch_tc");
}

// problems: DEVICE array of nprob ScannWgradProblem (include/scann_b200.h).  Gradients are accumulated
// (atomics) into dW / db, which the caller zeroes at the start of the step.
extern "C" int scann_wgrad_batch_tc(int grid, const void* problems_dev, int nprob, const int32_t* ntiles, int tile_stride,
                                    const int32_t* pair_c, const int32_t* pair_j, const int32_t* valid_rows,
                                    const int32_t* valid_j, const int32_t* nvalid, void* stream) {
    return wgrad_batch_launch<false>(grid, problems_dev, nprob, ntiles, tile_stride, pair_c, pair_j, valid_rows, valid_j,
                                     nvalid, nullptr, nullptr, stream);
}

// Deterministic form: dW / db are STORED (each is written by exactly one problem); slots [grid][2][128*128] and
// bslots [grid][2][128] hold the partial sums of the problems that several CTAs share, which
// scann_wgrad_batch_reduce (same grid, table and plan) adds up afterwards.
extern "C" int scann_wgrad_batch_tc_det(int grid, const void* problems_dev, int nprob, const int32_t* ntiles, int tile_stride,
                                        const int32_t* pair_c, const int32_t* pair_j, const int32_t* valid_rows,
                                        const int32_t* valid_j, const int32_t* nvalid, float* slots, float* bslots,
                                        void* stream) {
    if (!slots || !bslots) { scann_set_error("wgrad_batch_tc_det: slots and bslots are required"); return 1; }
    return wgrad_batch_launch<true>(grid, problems_dev, nprob, ntiles, tile_stride, pair_c, pair_j, valid_rows, valid_j,
                                    nvalid, slots, bslots, stream);
}

// Longest problem table one scann_wgrad_batch_tc / _det / reduce launch takes (the table is staged in shared memory);
// a longer one is cut into several launches.
extern "C" int scann_wgrad_batch_max_problems(void) { return WG_MAX_PROBLEMS; }

extern "C" int scann_wgrad_batch_reduce(int grid, const void* problems_dev, int nprob, const int32_t* ntiles, int tile_stride,
                                        const int32_t* valid_rows, const int32_t* nvalid, const float* slots,
                                        const float* bslots, void* stream) {
    if (nprob < 1 || nprob > WG_MAX_PROBLEMS) { scann_set_error("wgrad_batch_reduce: nprob must be in 1..%d", WG_MAX_PROBLEMS); return 1; }
    if (grid <= 0) return 0;
    scann_launch(wgrad_slot_reduce_kernel, dim3(SCANN_D * SCANN_D / (256 * 8), nprob), dim3(256), 0, stream,
                 (const WgProblem*)problems_dev, nprob, grid, ntiles, tile_stride, valid_rows ? nvalid : (const int32_t*)nullptr,
                 slots, bslots);
    return scann_check_launch("scann_wgrad_batch_reduce");
}
