// Chains of per-atom Dense layers in ONE kernel (tcgen05, kind::tf32, 3xTF32).
//
// Between two local-attention layers the reference runs, per atom row and with no interaction between rows,
//   forward :  ResidualNorm = LN(h + Dense(swish(Dense(h))))  (attention.py:25-40), then the next layer's
//              projections x @ [W1 | W3 | Wq] (attention.py:141-161) and "context = q" for atoms without
//              a neighbour (attention.py:206-214);
//   backward:  d_x = [s_pre | t | dq] @ [W1 | W3 | Wq]^T + scatter, LayerNorm backward, the two ResidualNorm
//              Dense layers transposed (with swish'), LayerNorm backward of the attention output.
// As separate launches these are 4-5 kernels of a few microseconds each on the critical path of the step
// (measured in the captured graph: ~8 us per kernel, ~60 of them = 0.57 of the 1.70 ms QM9 train step).
// Because rows are independent, a CTA can carry its TR rows through the WHOLE chain: the output of one step
// is written (hi/lo tf32 split) straight into the shared-memory operand image of the next step, only the
// 128x128 weight block is swapped in tensor memory between steps, and every intermediate that the weight-
// gradient kernels need is still stored to global memory by the epilogues.
//
// Per step:  V = sum_kb A_kb @ W_kb + bias (+ resid)  ->  epilogue `mode`  ->  C (and C2), optional image.
// Tensor-core layout as in dense_tc.cu: W^T stationary in tensor memory (M x K operand, hi/lo = 256 columns),
// the TR-row activation tile is the N x K operand (canonical K-major image), D^T in tensor memory (main and
// correction accumulators), transposed through shared memory, row-group epilogue (8 lanes per row).
#include "common.cuh"
#include "tc_common.cuh"

#define CH_THREADS 256
#define CH_MAX_STEPS 6
extern "C" int scann_device_sm_count(void);

// phase timestamps of CTA 0 (clock64), read back with scann_debug_clocks_chain: development builds only
// (SCANN_NVCC_DEFS=-DSCANN_DEV_PROBES); the production kernels carry no timestamp stores
#ifdef SCANN_DEV_PROBES
__device__ long long g_dbg_clk_chain[64];
#define CCLK(i) do { if (blockIdx.x == 0 && threadIdx.x == 0 && (i) < 64) g_dbg_clk_chain[i] = clock64(); } while (0)
#else
#define CCLK(i) do { } while (0)
#endif

// Mirrors ScannChainStep in include/scann_b200.h (same field order).
struct ChainStep {
    const float* A[3];      // kblk global inputs [R, lda]; A[0] == NULL: operand = image left by the previous step
    const float* W[3];      // kblk weight blocks [128,128] row-major ([in,out])
    const float* bias;      // [128] nullable
    const float* resid;     // [R, ldres] nullable, added before the epilogue
    const float* pre_in;    // mode 2: pre-activation [R, ldpre] ; mode 4: forward pre-LayerNorm value [R, ldpre]
    float* pre_out;         // mode 1: pre-activation, mode 3: pre-LayerNorm value, [R, ldpre] nullable
    const float* gamma;     // modes 3, 4 (and the no-pair fix-up)
    const float* beta;      // mode 3 (and the no-pair fix-up)
    float* dgamma;          // mode 4: accumulated (atomics)
    float* dbeta;
    float* C;               // [R, ldc] nullable
    float* C2;              // second copy of the output, [R, ldc2] nullable
    const int32_t* cnt;     // no-pair fix-up (nullable): rows with cnt[r] == 0 get np_ctx[r] = V, np_out[r] = LN(V)
    float* np_ctx;          // [R,128] nullable
    float* np_out;          // [R,128]
    const ScannDropCtl* drop;   // nullable.  modes 0-3: (sum + bias) is multiplied by the dropout mask of `drop_site`
                                // before the residual is added.  mode 4: C <- out, C2 and the image <- out * mask.
    int lda, ldres, ldpre, ldc, ldc2;
    int kblk;               // 1..3
    int mode;               // 0 none | 1 swish | 2 * swish'(pre_in) | 3 LayerNorm | 4 LayerNorm backward
    int to_image;           // the output becomes the next step's operand
    int drop_site;          // dropout site id (mask index = row * 128 + column)
    int pad;
};
struct ChainArgs {
    int nsteps, R;
    ChainStep s[CH_MAX_STEPS];
};

// weight block W[k][n] -> registers of thread (n = output feature, 64 consecutive k): all 64 loads in flight
__device__ __forceinline__ void chain_weight_load(const float* __restrict__ W, float (&w)[64], int warp, int lane) {
    const int n = (warp & 3) * 32 + lane, kbase = (warp >> 2) * 64;
#pragma unroll
    for (int q = 0; q < 64; ++q) w[q] = __ldg(W + (size_t)(kbase + q) * SCANN_D + n);
}
// registers -> tensor memory as A[M = n][K = k], hi and lo tf32 parts
__device__ __forceinline__ void chain_weight_store(const float (&w)[64], uint32_t t_whi, uint32_t t_wlo, int warp) {
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const int kbase = (warp >> 2) * 64;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        float hi[16], lo[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) tf32_split(w[g * 16 + q], hi[q], lo[q]);
        tmem_st16(t_whi + lane_base + kbase + g * 16, hi);
        tmem_st16(t_wlo + lane_base + kbase + g * 16, lo);
    }
}
__device__ __forceinline__ void chain_weight_to_tmem(const float* __restrict__ W, uint32_t t_whi, uint32_t t_wlo, int warp,
                                                     int lane) {
    float w[64];
    chain_weight_load(W, w, warp, lane);
    chain_weight_store(w, t_whi, t_wlo, warp);
}

// DET (deterministic mode, DESIGN.md section 4.7): the warps add their LayerNorm-backward column sums into shared memory
// one warp after the other, and the CTA stores them into its slot (dgamma / dbeta point to [grid][128] slot arrays).
template <int TR, bool DET>
__global__ void __launch_bounds__(CH_THREADS, 1) dense_chain_kernel(const __grid_constant__ ChainArgs a) {
    constexpr int XIT = TR / 8;                         // LDG.128 per thread for one activation tile
    constexpr uint32_t IMG = (TR / 8) * TC_RG_STRIDE;   // bytes of one K-major image of TR rows
    constexpr int STEPS = TR / (CH_THREADS / 32) / 4;   // row-group steps per warp in the epilogue
    // with 32-row tiles the registers allow fetching the NEXT step's weight block while the epilogue runs
    constexpr bool WPREF = TR == 32;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* sXhi = smem;
    uint8_t* sXlo = smem + IMG;
    uint8_t* sS = smem + 2 * IMG;
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_base_s;
    __shared__ float s_dg[SCANN_D], s_db[SCANN_D];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int r0 = blockIdx.x * TR;
    if (warp == 0) tmem_alloc(&tmem_base_s, 512);
    // (Issuing the three products of 3xTF32 from three warps into three accumulators was tried in round 2: no change
    // of the step time -- the chain's GEMM steps are not bound by MMA issue -- and 1.1e-5 instead of 8e-6 on the
    // QM9 golden: kept as it was.)
    if (tid == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;
    const uint32_t t_whi = tmem, t_wlo = tmem + 128, t_dm = tmem + 256, t_dc = tmem + 256 + TR;
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t idesc = tc_idesc_tf32(128, TR, false, false);
    const int l8 = lane & 7, rsub = lane >> 3;
    uint32_t phase = 0;
    // the first weight block only depends on parameters: stage it before waiting for the predecessor kernel
    CCLK(0);
    chain_weight_to_tmem(a.s[0].W[0], t_whi, t_wlo, warp, lane);
    CCLK(1);
    pdl_wait();
    CCLK(2);

    float wnext[64];                 // only live when WPREF
    bool have_next = false;
#pragma unroll 1
    for (int si = 0; si < a.nsteps; ++si) {
        const ChainStep& st = a.s[si];
        // parameters of the epilogue: issue the loads now, they are needed after the MMA
        float4 bias[4], gam[4], bet[4];
#pragma unroll
        for (int it = 0; it < 4; ++it) {
            const int c0 = (l8 + 8 * it) * 4;
            bias[it] = st.bias ? ldg4(st.bias + c0) : make_float4(0.f, 0.f, 0.f, 0.f);
            gam[it] = st.gamma ? ldg4(st.gamma + c0) : bias[it];
            bet[it] = st.beta ? ldg4(st.beta + c0) : bias[it];
        }
        // ------------------------------------------------------------------ GEMM: D^T = sum_kb W_kb^T X_kb^T
        float4 rv0[4], pv0[4];
#pragma unroll 1
        for (int kb = 0; kb < st.kblk; ++kb) {
            const float* A = st.A[kb];
            float4 xv[XIT];
            if (A) {
#pragma unroll
                for (int it = 0; it < XIT; ++it) {
                    const int i = tid + it * CH_THREADS, r = i >> 5, c4 = i & 31;
                    xv[it] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (r0 + r < a.R) xv[it] = ld4(A + (size_t)(r0 + r) * st.lda + c4 * 4);
                }
            }
            if (WPREF && kb == 0 && have_next) { /* staged behind the previous step's epilogue */ }
            else if (si > 0 || kb > 0) chain_weight_to_tmem(st.W[kb], t_whi, t_wlo, warp, lane);
            if (A) {
#pragma unroll
                for (int it = 0; it < XIT; ++it) {
                    const int i = tid + it * CH_THREADS, r = i >> 5, c4 = i & 31;
                    float4 v = xv[it], h, l;
                    tf32_split(v.x, h.x, l.x); tf32_split(v.y, h.y, l.y);
                    tf32_split(v.z, h.z, l.z); tf32_split(v.w, h.w, l.w);
                    const uint32_t off = tc_off4(r, c4);
                    *reinterpret_cast<float4*>(sXhi + off) = h;
                    *reinterpret_cast<float4*>(sXlo + off) = l;
                }
            }
            tmem_st_wait();
            fence_async_smem();
            tc_fence_before();
            __syncthreads();
            if (kb == 0) CCLK(3 + si * 4);
            if (warp == 0 && tc_elect_one()) {
                tc_fence_after();
                const uint64_t dh = tc_desc_kmajor(smem_u32(sXhi), 0), dl = tc_desc_kmajor(smem_u32(sXlo), 0);
                const bool first = kb == 0;
#pragma unroll
                for (int ks = 0; ks < 16; ++ks)
                    tc_mma_ts(t_dm, t_whi + ks * 8, dh + ks * TC_KSTEP_DESC, idesc, !(first && ks == 0));
#pragma unroll
                for (int ks = 0; ks < 16; ++ks)
                    tc_mma_ts(t_dc, t_wlo + ks * 8, dh + ks * TC_KSTEP_DESC, idesc, !(first && ks == 0));
#pragma unroll
                for (int ks = 0; ks < 16; ++ks) tc_mma_ts(t_dc, t_whi + ks * 8, dl + ks * TC_KSTEP_DESC, idesc, true);
                tc_commit(&bar);
            }
            if (WPREF && kb == st.kblk - 1) {
                // while the tensor core works: the next step's first weight block -> registers ...
                have_next = si + 1 < a.nsteps;
                if (have_next) chain_weight_load(a.s[si + 1].W[0], wnext, warp, lane);
            }
            if (kb == st.kblk - 1) {
                // ... and the global rows the first epilogue step needs
                const int rr = warp * (TR / (CH_THREADS / 32)) + rsub, r = r0 + rr;
#pragma unroll
                for (int it = 0; it < 4; ++it) {
                    rv0[it] = make_float4(0.f, 0.f, 0.f, 0.f);
                    pv0[it] = rv0[it];
                    if (r < a.R) {
                        if (st.resid) rv0[it] = ld4(st.resid + (size_t)r * st.ldres + (l8 + 8 * it) * 4);
                        if (st.mode == 2 || st.mode == 4) pv0[it] = ld4(st.pre_in + (size_t)r * st.ldpre + (l8 + 8 * it) * 4);
                    }
                }
            }
            mbar_wait(&bar, phase);
            phase ^= 1;
            tc_fence_after();
            __syncthreads();
        }
        CCLK(4 + si * 4);
        if (si == a.nsteps - 1) pdl_trigger();      // only the last epilogue is left
        // ------------------------------------------------------------------ epilogue 1: D^T -> S[r][n]
        {
            const int n = (warp & 3) * 32 + lane, rbase = (warp >> 2) * (TR / 2);
#pragma unroll 1
            for (int rr = rbase; rr < rbase + TR / 2; rr += 16) {
                float m[16], c[16];
                tmem_ld16(t_dm + lane_base + rr, m);
                tmem_ld16(t_dc + lane_base + rr, c);
                tmem_ld_wait();
#pragma unroll
                for (int q = 0; q < 16; ++q) *reinterpret_cast<float*>(sS + tc_off(rr + q, n)) = m[q] + c[q];
            }
        }
        if (st.mode == 4 && tid < SCANN_D) { s_dg[tid] = 0.f; s_db[tid] = 0.f; }
        if (WPREF && have_next) chain_weight_store(wnext, t_whi, t_wlo, warp);   // drains behind the row epilogue
        tc_fence_before();
        __syncthreads();
        CCLK(5 + si * 4);
        // ------------------------------------------------------------------ epilogue 2: row groups
        const int mode = st.mode;
        float dgam[4][4], dbet[4][4];
#pragma unroll
        for (int it = 0; it < 4; ++it)
#pragma unroll
            for (int q = 0; q < 4; ++q) { dgam[it][q] = 0.f; dbet[it][q] = 0.f; }
#pragma unroll 1
        for (int step = 0; step < STEPS; ++step) {
            const int rr = warp * (TR / (CH_THREADS / 32)) + step * 4 + rsub, r = r0 + rr;
            const bool ok = r < a.R;
            float v[4][4];
#pragma unroll
            for (int it = 0; it < 4; ++it) {
                const int c4 = l8 + 8 * it, c0 = c4 * 4;
                const float4 acc = *reinterpret_cast<const float4*>(sS + tc_off4(rr, c4));
                float4 rv = rv0[it];
                if (step > 0) {
                    rv = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (st.resid && ok) rv = ld4(st.resid + (size_t)r * st.ldres + c0);
                }
                float d0 = 1.f, d1 = 1.f, d2 = 1.f, d3 = 1.f;
                if (st.drop && mode != 4) {
                    const uint32_t idx = (uint32_t)r * SCANN_D + c0;
                    d0 = drop_mult(st.drop, st.drop_site, idx); d1 = drop_mult(st.drop, st.drop_site, idx + 1);
                    d2 = drop_mult(st.drop, st.drop_site, idx + 2); d3 = drop_mult(st.drop, st.drop_site, idx + 3);
                }
                v[it][0] = (acc.x + bias[it].x) * d0 + rv.x; v[it][1] = (acc.y + bias[it].y) * d1 + rv.y;
                v[it][2] = (acc.z + bias[it].z) * d2 + rv.z; v[it][3] = (acc.w + bias[it].w) * d3 + rv.w;
            }
            if (mode == 1) {
#pragma unroll
                for (int it = 0; it < 4; ++it) {
                    if (st.pre_out && ok)
                        st4(st.pre_out + (size_t)r * st.ldpre + (l8 + 8 * it) * 4,
                            make_float4(v[it][0], v[it][1], v[it][2], v[it][3]));
#pragma unroll
                    for (int q = 0; q < 4; ++q) v[it][q] = swish_fast(v[it][q]);
                }
            } else if (mode == 2) {
#pragma unroll
                for (int it = 0; it < 4; ++it) {
                    float4 p = pv0[it];
                    if (step > 0) {
                        p = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (ok) p = ld4(st.pre_in + (size_t)r * st.ldpre + (l8 + 8 * it) * 4);
                    }
                    v[it][0] *= swish_grad_fast(p.x); v[it][1] *= swish_grad_fast(p.y);
                    v[it][2] *= swish_grad_fast(p.z); v[it][3] *= swish_grad_fast(p.w);
                }
            } else if (mode == 3) {
                float s1 = 0.f;
#pragma unroll
                for (int it = 0; it < 4; ++it) {
                    if (st.pre_out && ok)
                        st4(st.pre_out + (size_t)r * st.ldpre + (l8 + 8 * it) * 4,
                            make_float4(v[it][0], v[it][1], v[it][2], v[it][3]));
                    s1 += v[it][0] + v[it][1] + v[it][2] + v[it][3];
                }
                // shifted one-pass moments: shift = mean of the row's first 16-column slice
                const float sh = __shfl_sync(0xffffffffu, s1, lane & 24) * (1.0f / 16.0f);
                float m1 = 0.f, m2 = 0.f;
#pragma unroll
                for (int it = 0; it < 4; ++it)
#pragma unroll
                    for (int q = 0; q < 4; ++q) { v[it][q] -= sh; m1 += v[it][q]; m2 = fmaf(v[it][q], v[it][q], m2); }
                oct_sum2(m1, m2);
                m1 *= (1.0f / SCANN_D);
                const float inv = rsqrtf(fmaxf(m2 * (1.0f / SCANN_D) - m1 * m1, 0.f) + SCANN_LN_EPS);
#pragma unroll
                for (int it = 0; it < 4; ++it) {
                    v[it][0] = (v[it][0] - m1) * inv * gam[it].x + bet[it].x;
                    v[it][1] = (v[it][1] - m1) * inv * gam[it].y + bet[it].y;
                    v[it][2] = (v[it][2] - m1) * inv * gam[it].z + bet[it].z;
                    v[it][3] = (v[it][3] - m1) * inv * gam[it].w + bet[it].w;
                }
            } else if (mode == 4) {
                // LayerNorm backward: v = upstream gradient dy, pre_in = forward pre-LN value
                float x[4][4];
                float s1 = 0.f;
#pragma unroll
                for (int it = 0; it < 4; ++it) {
                    float4 p = pv0[it];
                    if (step > 0) {
                        p = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (ok) p = ld4(st.pre_in + (size_t)r * st.ldpre + (l8 + 8 * it) * 4);
                    }
                    x[it][0] = p.x; x[it][1] = p.y; x[it][2] = p.z; x[it][3] = p.w;
                    s1 += p.x + p.y + p.z + p.w;
                }
                float d0 = 0.f;
                oct_sum2(s1, d0);
                const float mean = s1 * (1.0f / SCANN_D);
                float var = 0.f, dummy = 0.f;
#pragma unroll
                for (int it = 0; it < 4; ++it)
#pragma unroll
                    for (int q = 0; q < 4; ++q) { x[it][q] -= mean; var = fmaf(x[it][q], x[it][q], var); }
                oct_sum2(var, dummy);
                const float inv = rsqrtf(var * (1.0f / SCANN_D) + SCANN_LN_EPS);
                const float g[4][4] = {{gam[0].x, gam[0].y, gam[0].z, gam[0].w}, {gam[1].x, gam[1].y, gam[1].z, gam[1].w},
                                       {gam[2].x, gam[2].y, gam[2].z, gam[2].w}, {gam[3].x, gam[3].y, gam[3].z, gam[3].w}};
                float t1 = 0.f, t2 = 0.f;
#pragma unroll
                for (int it = 0; it < 4; ++it)
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        x[it][q] *= inv;                                    // x_hat
                        const float dy = ok ? v[it][q] : 0.f;
                        dgam[it][q] = fmaf(dy, x[it][q], dgam[it][q]);
                        dbet[it][q] += dy;
                        v[it][q] = dy * g[it][q];                           // d x_hat
                        t1 += v[it][q];
                        t2 = fmaf(v[it][q], x[it][q], t2);
                    }
                oct_sum2(t1, t2);
                t1 *= (1.0f / SCANN_D);
                t2 *= (1.0f / SCANN_D);
#pragma unroll
                for (int it = 0; it < 4; ++it)
#pragma unroll
                    for (int q = 0; q < 4; ++q) v[it][q] = inv * (v[it][q] - t1 - x[it][q] * t2);
            }
            if (ok && st.C) {
#pragma unroll
                for (int it = 0; it < 4; ++it)
                    st4(st.C + (size_t)r * st.ldc + (l8 + 8 * it) * 4, make_float4(v[it][0], v[it][1], v[it][2], v[it][3]));
            }
            if (mode == 4 && st.drop) {
                // gradient through the dropout that follows the Dense of the next (transposed) step
#pragma unroll
                for (int it = 0; it < 4; ++it) {
                    const uint32_t idx = (uint32_t)r * SCANN_D + (l8 + 8 * it) * 4;
#pragma unroll
                    for (int q = 0; q < 4; ++q) v[it][q] *= drop_mult(st.drop, st.drop_site, idx + q);
                }
            }
            if (ok && st.C2) {
#pragma unroll
                for (int it = 0; it < 4; ++it)
                    st4(st.C2 + (size_t)r * st.ldc2 + (l8 + 8 * it) * 4, make_float4(v[it][0], v[it][1], v[it][2], v[it][3]));
            }
            if (st.to_image) {
#pragma unroll
                for (int it = 0; it < 4; ++it) {
                    float4 h, l;
                    tf32_split(ok ? v[it][0] : 0.f, h.x, l.x); tf32_split(ok ? v[it][1] : 0.f, h.y, l.y);
                    tf32_split(ok ? v[it][2] : 0.f, h.z, l.z); tf32_split(ok ? v[it][3] : 0.f, h.w, l.w);
                    const uint32_t off = tc_off4(rr, l8 + 8 * it);
                    *reinterpret_cast<float4*>(sXhi + off) = h;
                    *reinterpret_cast<float4*>(sXlo + off) = l;
                }
            }
            if (st.cnt) {
                // atoms without a valid neighbour: context = q, out = LayerNorm(q)   (attention.py:206-214)
                const bool nop = ok && st.cnt[r] == 0;
                if (__any_sync(0xffffffffu, nop)) {
                    float m1 = 0.f, m2 = 0.f;
#pragma unroll
                    for (int it = 0; it < 4; ++it)
#pragma unroll
                        for (int q = 0; q < 4; ++q) m1 += v[it][q];
                    oct_sum2(m1, m2);
                    m1 *= (1.0f / SCANN_D);
                    float dd = 0.f;
#pragma unroll
                    for (int it = 0; it < 4; ++it)
#pragma unroll
                        for (int q = 0; q < 4; ++q) { const float d = v[it][q] - m1; m2 = fmaf(d, d, m2); }
                    oct_sum2(m2, dd);
                    const float inv = rsqrtf(m2 * (1.0f / SCANN_D) + SCANN_LN_EPS);
                    if (nop) {
#pragma unroll
                        for (int it = 0; it < 4; ++it) {
                            const int c0 = (l8 + 8 * it) * 4;
                            if (st.np_ctx)
                                st4(st.np_ctx + (size_t)r * SCANN_D + c0, make_float4(v[it][0], v[it][1], v[it][2], v[it][3]));
                            st4(st.np_out + (size_t)r * SCANN_D + c0,
                                make_float4((v[it][0] - m1) * inv * gam[it].x + bet[it].x,
                                            (v[it][1] - m1) * inv * gam[it].y + bet[it].y,
                                            (v[it][2] - m1) * inv * gam[it].z + bet[it].z,
                                            (v[it][3] - m1) * inv * gam[it].w + bet[it].w));
                        }
                    }
                }
            }
        }
        if (mode == 4) {
            // column sums over this CTA's rows -> shared -> global
            float cg[4][4], cb[4][4];
#pragma unroll
            for (int it = 0; it < 4; ++it)
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    float dg = dgam[it][q], db = dbet[it][q];
                    dg += __shfl_xor_sync(0xffffffffu, dg, 8);  db += __shfl_xor_sync(0xffffffffu, db, 8);
                    dg += __shfl_xor_sync(0xffffffffu, dg, 16); db += __shfl_xor_sync(0xffffffffu, db, 16);
                    if constexpr (DET) {
                        cg[it][q] = dg; cb[it][q] = db;
                    } else if (rsub == 0) {
                        atomicAdd(&s_dg[(l8 + 8 * it) * 4 + q], dg);
                        atomicAdd(&s_db[(l8 + 8 * it) * 4 + q], db);
                    }
                }
            if constexpr (DET) {
                for (int w = 0; w < CH_THREADS / 32; ++w) {
                    if (warp == w && rsub == 0) {
#pragma unroll
                        for (int it = 0; it < 4; ++it)
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                s_dg[(l8 + 8 * it) * 4 + q] += cg[it][q];
                                s_db[(l8 + 8 * it) * 4 + q] += cb[it][q];
                            }
                    }
                    __syncthreads();
                }
                if (tid < SCANN_D) {
                    st.dgamma[(size_t)blockIdx.x * SCANN_D + tid] = s_dg[tid];
                    st.dbeta[(size_t)blockIdx.x * SCANN_D + tid] = s_db[tid];
                }
            } else {
                __syncthreads();
                if (tid < SCANN_D) {
                    atomicAdd(st.dgamma + tid, s_dg[tid]);
                    atomicAdd(st.dbeta + tid, s_db[tid]);
                }
            }
        }
        __syncthreads();        // S and the images are rewritten / read by the next step
        CCLK(6 + si * 4);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

#ifdef SCANN_DEV_PROBES
extern "C" int scann_debug_clocks_chain(long long* host_out64) {
    cudaError_t e = cudaMemcpyFromSymbol(host_out64, g_dbg_clk_chain, sizeof(long long) * 64);
    if (e != cudaSuccess) { scann_set_error("debug_clocks_chain: %s", cudaGetErrorString(e)); return 1; }
    return 0;
}
#endif

// Host-side mirror of the public struct (include/scann_b200.h): identical layout to ChainStep.
template <bool DET>
static int chain_run(const void* steps_host, int nsteps, int R, void* stream) {
    if (nsteps < 1 || nsteps > CH_MAX_STEPS) { scann_set_error("dense_chain: nsteps must be in 1..%d", CH_MAX_STEPS); return 1; }
    if (R <= 0) return 0;
    ChainArgs a;
    a.nsteps = nsteps;
    a.R = R;
    const ChainStep* s = (const ChainStep*)steps_host;
    for (int i = 0; i < nsteps; ++i) {
        a.s[i] = s[i];
        const ChainStep& t = a.s[i];
        if (t.kblk < 1 || t.kblk > 3 || t.mode < 0 || t.mode > 4) { scann_set_error("dense_chain: step %d: bad kblk/mode", i); return 1; }
        if (!t.A[0] && i == 0) { scann_set_error("dense_chain: step 0 has no input"); return 1; }
        if (!t.A[0] && t.kblk != 1) { scann_set_error("dense_chain: step %d: an image operand needs kblk == 1", i); return 1; }
        for (int kb = 0; kb < t.kblk; ++kb)
            if (!t.W[kb] || (kb > 0 && !t.A[kb])) { scann_set_error("dense_chain: step %d: missing operand %d", i, kb); return 1; }
        if ((t.mode == 2 || t.mode == 4) && !t.pre_in) { scann_set_error("dense_chain: step %d: mode needs pre_in", i); return 1; }
        if ((t.mode == 3 || t.mode == 4) && !t.gamma) { scann_set_error("dense_chain: step %d: mode needs gamma", i); return 1; }
        if (t.mode == 3 && !t.beta) { scann_set_error("dense_chain: step %d: LayerNorm needs beta", i); return 1; }
        if (t.mode == 4 && (!t.dgamma || !t.dbeta)) { scann_set_error("dense_chain: step %d: LayerNorm backward needs dgamma/dbeta", i); return 1; }
        if (t.cnt && (!t.np_out || !t.gamma || !t.beta)) { scann_set_error("dense_chain: step %d: no-pair fix-up needs np_out/gamma/beta", i); return 1; }
    }
    for (int i = nsteps; i < CH_MAX_STEPS; ++i) a.s[i] = ChainStep{};
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(dense_chain_kernel<128, DET>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)(3 * TC_TILE_BYTES));
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(dense_chain_kernel<64, DET>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)(3 * TC_TILE_BYTES / 2));
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(dense_chain_kernel<32, DET>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)(3 * TC_TILE_BYTES / 4));
        if (e != cudaSuccess) { scann_set_error("dense_chain: smem opt-in failed: %s", cudaGetErrorString(e)); return 1; }
        configured = true;
    }
    static int sms = 0;
    if (sms == 0) sms = scann_device_sm_count();
    int tr = 128;
    if ((R + 31) / 32 <= sms) tr = 32;
    else if ((R + 63) / 64 <= sms) tr = 64;
    dim3 grid((R + tr - 1) / tr);
    const size_t smem = 3 * (size_t)(tr / 8) * TC_RG_STRIDE;
    if (tr == 32) scann_launch(dense_chain_kernel<32, DET>, grid, dim3(CH_THREADS), smem, stream, a);
    else if (tr == 64) scann_launch(dense_chain_kernel<64, DET>, grid, dim3(CH_THREADS), smem, stream, a);
    else scann_launch(dense_chain_kernel<128, DET>, grid, dim3(CH_THREADS), smem, stream, a);
    return scann_check_launch("scann_dense_chain");
}

extern "C" int scann_dense_chain(const void* steps_host, int nsteps, int R, void* stream) {
    return chain_run<false>(steps_host, nsteps, R, stream);
}

// Deterministic form: dgamma / dbeta of every mode-4 step are [scann_dense_chain_grid(R)][128] slot arrays.
extern "C" int scann_dense_chain_det(const void* steps_host, int nsteps, int R, void* stream) {
    return chain_run<true>(steps_host, nsteps, R, stream);
}

// CTAs of one scann_dense_chain launch over R rows.
extern "C" int scann_dense_chain_grid(int R) {
    static int sms = 0;
    if (sms == 0) sms = scann_device_sm_count();
    if (R <= 0) return 0;
    const int tr = (R + 31) / 32 <= sms ? 32 : ((R + 63) / 64 <= sms ? 64 : 128);
    return (R + tr - 1) / tr;
}
