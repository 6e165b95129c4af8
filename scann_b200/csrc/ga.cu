// Global attention + property head, one CTA per structure.
//
// Restates GlobalAttention.call (scann/layers/attention.py:267-318) for v_proj=False,
// kq_proj=True and the head Dense layers (scann/models/scann_model.py:437-447).
// The reference builds the [M,M] energy matrix, zeroes its diagonal and sums over the
// query axis (:279-292); with m in {0,1} that equals
//     s_i = m_i * k_i . (Q - m_i q_i),   Q = sum_j m_j q_j
// so no M x M matrix is formed (O(M*D) work).  ga = softmax_i(s/||s|| - 1e9 (1-m)) is the
// ga_score output; ctx = sum_i m_i ga_i k_i feeds bf_property -> predict_property.
#include "common.cuh"

#define GA_THREADS 128

__device__ __forceinline__ float block_sum_128(float v, float* s_red) {
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    return s_red[0] + s_red[1] + s_red[2] + s_red[3];
}
__device__ __forceinline__ float block_max_128(float v, float* s_red) {
    v = warp_max(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    return fmaxf(fmaxf(s_red[0], s_red[1]), fmaxf(s_red[2], s_red[3]));
}

// Shared forward part: fills s_Q[128], s_s[M] (normalised scores), s_ga[M]; returns ||s|| (or 1).
__device__ float ga_scores(const float* __restrict__ qk, const uint8_t* __restrict__ mask, int M, int norm,
                           float* s_Q, float* s_s, float* s_ga, float* s_red) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // loads are unconditional and selected afterwards (rows of padded atoms exist and are finite or not, the
    // select drops them): a load guarded by the mask byte would make every iteration a dependent round trip
    float Q = 0.f;
#pragma unroll 8
    for (int i = 0; i < M; ++i) {
        const float q = qk[(size_t)i * 2 * SCANN_D + tid];
        Q += mask[i] ? q : 0.f;
    }
    s_Q[tid] = Q;
    __syncthreads();
    const float4 Q4 = ld4(s_Q + lane * 4);
#pragma unroll 4
    for (int i = warp; i < M; i += GA_THREADS / 32) {
        const float4 q = ld4(qk + (size_t)i * 2 * SCANN_D + lane * 4);
        const float4 k = ld4(qk + (size_t)i * 2 * SCANN_D + SCANN_D + lane * 4);
        float v = k.x * (Q4.x - q.x) + k.y * (Q4.y - q.y) + k.z * (Q4.z - q.z) + k.w * (Q4.w - q.w);
        v = warp_sum(mask[i] ? v : 0.f);
        if (lane == 0) s_s[i] = v;
    }
    __syncthreads();
    float nrm = 1.0f;
    if (norm) {
        float p = 0.f;
        for (int i = tid; i < M; i += GA_THREADS) p += s_s[i] * s_s[i];
        nrm = sqrtf(block_sum_128(p, s_red));
        for (int i = tid; i < M; i += GA_THREADS) s_s[i] = s_s[i] / nrm;   // 0/0 -> NaN as tf.linalg.normalize
        __syncthreads();
    }
    float mx = -INFINITY;
    for (int i = tid; i < M; i += GA_THREADS) {
        float l = s_s[i] + (mask[i] ? 0.f : -1e9f);
        s_ga[i] = l;
        mx = fmaxf(mx, l);
    }
    mx = block_max_128(mx, s_red);
    float se = 0.f;
    for (int i = tid; i < M; i += GA_THREADS) {
        float e = expf(s_ga[i] - mx);
        s_ga[i] = e;
        se += e;
    }
    se = block_sum_128(se, s_red);
    for (int i = tid; i < M; i += GA_THREADS) s_ga[i] = s_ga[i] / se;
    __syncthreads();
    return nrm;
}

__global__ void __launch_bounds__(GA_THREADS) ga_head_fwd_kernel(const float* __restrict__ qk,
                                                                 const uint8_t* __restrict__ atom_mask, int M,
                                                                 int norm, const float* __restrict__ Wb,
                                                                 const float* __restrict__ bb,
                                                                 const float* __restrict__ wp,
                                                                 const float* __restrict__ bp, int mrelu,
                                                                 float* __restrict__ ga, float* __restrict__ y,
                                                                 float* __restrict__ ctx_out,
                                                                 float* __restrict__ tb_out) {
    extern __shared__ __align__(16) float sm[];
    float* s_Q = sm;                 // 128
    float* s_ctx = s_Q + SCANN_D;    // 128
    float* s_red = s_ctx + SCANN_D;  // 4
    float* s_s = s_red + 4;          // M
    float* s_ga = s_s + M;           // M
    const int b = blockIdx.x, tid = threadIdx.x;
    const float* qkb = qk + (size_t)b * M * 2 * SCANN_D;
    const uint8_t* mb = atom_mask + (size_t)b * M;
    pdl_wait();
    pdl_trigger();      // only after the own wait: at most one kernel ahead becomes resident early
    ga_scores(qkb, mb, M, norm, s_Q, s_s, s_ga, s_red);
    for (int i = tid; i < M; i += GA_THREADS) ga[(size_t)b * M + i] = s_ga[i];
    float c = 0.f;
#pragma unroll 8
    for (int i = 0; i < M; ++i) {
        const float k = qkb[(size_t)i * 2 * SCANN_D + SCANN_D + tid];
        c = fmaf(s_ga[i], mb[i] ? k : 0.f, c);
    }
    s_ctx[tid] = c;
    if (ctx_out) ctx_out[(size_t)b * SCANN_D + tid] = c;
    __syncthreads();
    float t = bb[tid];
#pragma unroll 16
    for (int d = 0; d < SCANN_D; ++d) t = fmaf(s_ctx[d], __ldg(Wb + (size_t)d * SCANN_D + tid), t);
    if (tb_out) tb_out[(size_t)b * SCANN_D + tid] = t;
    float yy = block_sum_128(swish_f(t) * wp[tid], s_red) + bp[0];
    if (mrelu) yy = fmaxf(yy, 0.f);      // mrelu forward (custom_layers.py:15)
    if (tid == 0) y[b] = yy;
}

// Backward of head + global attention for one structure (SURVEY.md appendix A).
// dy[b] is the upstream gradient of y[b] (mrelu has an identity gradient, custom_layers.py:12-13).
// DET (deterministic mode): the head gradient of structure b is stored into slot b (dwp: [B][128], dbp: [B]).
template <bool DET>
__global__ void __launch_bounds__(GA_THREADS) ga_head_bwd_kernel(
    const float* __restrict__ qk, const uint8_t* __restrict__ atom_mask, int M, int norm,
    const float* __restrict__ WbT, const float* __restrict__ wp, const float* __restrict__ tb,
    const float* __restrict__ dy, float* __restrict__ d_qk, float* __restrict__ d_tb, float* __restrict__ dwp,
    float* __restrict__ dbp) {
    extern __shared__ __align__(16) float sm[];
    float* s_Q = sm;                  // 128
    float* s_dctx = s_Q + SCANN_D;    // 128
    float* s_dtb = s_dctx + SCANN_D;  // 128
    float* s_red = s_dtb + SCANN_D;   // 4
    float* s_s = s_red + 4;           // M   normalised scores
    float* s_ga = s_s + M;            // M
    float* s_ds = s_ga + M;           // M   d_ga -> d_t -> d_s
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float* qkb = qk + (size_t)b * M * 2 * SCANN_D;
    float* dqkb = d_qk + (size_t)b * M * 2 * SCANN_D;
    const uint8_t* mb = atom_mask + (size_t)b * M;
    pdl_wait();
    pdl_trigger();      // only after the own wait: at most one kernel ahead becomes resident early
    const float g = dy[b];
    // head
    {
        float t = tb[(size_t)b * SCANN_D + tid];
        float hid = swish_f(t);
        if constexpr (DET) {
            dwp[(size_t)b * SCANN_D + tid] = g * hid;
            if (tid == 0) dbp[b] = g;
        } else {
            atomicAdd(dwp + tid, g * hid);
            if (tid == 0) atomicAdd(dbp, g);
        }
        float dt = g * wp[tid] * swish_grad_f(t);
        s_dtb[tid] = dt;
        d_tb[(size_t)b * SCANN_D + tid] = dt;
    }
    __syncthreads();
    {
        float dc = 0.f;
#pragma unroll 16
        for (int n = 0; n < SCANN_D; ++n) dc = fmaf(s_dtb[n], __ldg(WbT + (size_t)n * SCANN_D + tid), dc);
        s_dctx[tid] = dc;
    }
    const float nrm = ga_scores(qkb, mb, M, norm, s_Q, s_s, s_ga, s_red);   // syncs inside, s_dctx visible after
    // d_ga_i = m_i <d_ctx, k_i>
    {
        const float4 dc4 = ld4(s_dctx + lane * 4);
#pragma unroll 4
        for (int i = warp; i < M; i += GA_THREADS / 32) {
            const float4 k = ld4(qkb + (size_t)i * 2 * SCANN_D + SCANN_D + lane * 4);
            float v = k.x * dc4.x + k.y * dc4.y + k.z * dc4.z + k.w * dc4.w;
            v = warp_sum(mb[i] ? v : 0.f);
            if (lane == 0) s_ds[i] = v;
        }
    }
    __syncthreads();
    float p = 0.f;
    for (int i = tid; i < M; i += GA_THREADS) p = fmaf(s_ga[i], s_ds[i], p);
    const float dot = block_sum_128(p, s_red);
    for (int i = tid; i < M; i += GA_THREADS) s_ds[i] = s_ga[i] * (s_ds[i] - dot);     // d_t
    __syncthreads();
    if (norm) {
        float q = 0.f;
        for (int i = tid; i < M; i += GA_THREADS) q = fmaf(s_s[i], s_ds[i], q);
        const float sd = block_sum_128(q, s_red);
        for (int i = tid; i < M; i += GA_THREADS) s_ds[i] = (s_ds[i] - s_s[i] * sd) / nrm;
        __syncthreads();
    }
    for (int i = tid; i < M; i += GA_THREADS)
        if (!mb[i]) s_ds[i] = 0.f;
    __syncthreads();
    // d_Q[d] = sum_i d_s_i m_i k_i[d]
    const float Q = s_Q[tid], dctx = s_dctx[tid];
    float dQ = 0.f;
#pragma unroll 8
    for (int i = 0; i < M; ++i) {
        const float k = qkb[(size_t)i * 2 * SCANN_D + SCANN_D + tid];
        dQ = fmaf(s_ds[i], mb[i] ? k : 0.f, dQ);            // s_ds is 0 for masked atoms, k may be anything
    }
#pragma unroll 4
    for (int i = 0; i < M; ++i) {
        const float q = qkb[(size_t)i * 2 * SCANN_D + tid], k = qkb[(size_t)i * 2 * SCANN_D + SCANN_D + tid];
        float dq = 0.f, dk = 0.f;
        if (mb[i]) {
            dk = s_ga[i] * dctx + s_ds[i] * (Q - q);
            dq = dQ - s_ds[i] * k;
        }
        dqkb[(size_t)i * 2 * SCANN_D + tid] = dq;
        dqkb[(size_t)i * 2 * SCANN_D + SCANN_D + tid] = dk;
    }
}

// =============================================================================================
// Staged form (round 2): the default whenever a structure's [M, 256] query | key block fits shared memory.
//
// The kernels above walk the block four times out of global memory, every walk a dependent chain of round trips
// (16.7 / 21.5 us under ncu for 1-2 MB of data at QM9 / 128: 0.02-0.04 of the HBM roofline, profiles/r02_launches_final.md),
// and the 128 x 128 head GEMV is 128 dependent fused multiply-adds behind 8 batches of L2 loads.  Here
//   * 512 threads copy the block into shared memory ONCE (coalesced 16-byte loads, all of a thread's loads in flight
//     together: one round trip), every later pass reads shared memory;
//   * column sums over atoms (Q, context, dQ) and the GEMV are split four ways (quarter kq = tid / 128 owns the rows
//     i = kq, kq + 4, ... / the 32 reduction indices 32 kq ..), partials combined through s_part;
//   * this thread's 32 head weights are loaded BEFORE the PDL wait (parameters: rule (1) of common.cuh);
//   * the M-vector phases (norm, softmax, its backward) run in warp 0 with shuffles: no block-wide reductions.
// Same formulas, same NaN behaviour for a single-atom structure (0 / 0 as tf.linalg.normalize).
// =============================================================================================
#define GA2_THREADS 512
#define GA2_SMEM_MAX (200 * 1024)

__device__ __forceinline__ float ga2_comb(const float* s_part, int col) {
    return (s_part[col] + s_part[128 + col]) + (s_part[256 + col] + s_part[384 + col]);
}

__device__ __forceinline__ void ga2_stage(const float* __restrict__ qkb, const uint8_t* __restrict__ mb, int M,
                                          float* s_qk, float* s_m) {
    const int tid = threadIdx.x, n4 = M * 64;
    const float4* src = reinterpret_cast<const float4*>(qkb);
    float4* dst = reinterpret_cast<float4*>(s_qk);
    for (int i0 = tid; i0 < n4; i0 += 4 * GA2_THREADS) {
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (i0 + u * GA2_THREADS < n4) v[u] = src[i0 + u * GA2_THREADS];
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (i0 + u * GA2_THREADS < n4) dst[i0 + u * GA2_THREADS] = v[u];
    }
    for (int i = tid; i < M; i += GA2_THREADS) s_m[i] = mb[i] ? 1.0f : 0.0f;
}

// fills s_Q[128], s_s[M] (normalised scores), s_ga[M]; returns ||s|| (or 1).  Ends with a block barrier.
__device__ __forceinline__ float ga2_scores(int M, int norm, const float* s_qk, const float* s_m, float* s_part,
                                            float* s_Q, float* s_s, float* s_ga, float* s_sc) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, col = tid & 127, kq = tid >> 7;
    float acc = 0.f;
    for (int i = kq; i < M; i += 4) acc += s_m[i] != 0.f ? s_qk[i * 256 + col] : 0.f;    // select, not multiply: padded rows may hold anything
    s_part[kq * 128 + col] = acc;
    __syncthreads();
    if (tid < 128) s_Q[tid] = ga2_comb(s_part, tid);
    __syncthreads();
    const float4 Q4 = ld4(s_Q + lane * 4);
    for (int i = warp; i < M; i += GA2_THREADS / 32) {
        const float4 q = ld4(s_qk + i * 256 + lane * 4), k = ld4(s_qk + i * 256 + 128 + lane * 4);
        float v = k.x * (Q4.x - q.x) + k.y * (Q4.y - q.y) + k.z * (Q4.z - q.z) + k.w * (Q4.w - q.w);
        v = warp_sum(s_m[i] != 0.f ? v : 0.f);
        if (lane == 0) s_s[i] = v;
    }
    __syncthreads();
    if (warp == 0) {                       // lane l owns the atoms i = l, l + 32, ... in every phase
        float nrm = 1.0f;
        if (norm) {
            float p = 0.f;
            for (int i = lane; i < M; i += 32) p += s_s[i] * s_s[i];
            nrm = sqrtf(warp_sum(p));
            for (int i = lane; i < M; i += 32) s_s[i] = s_s[i] / nrm;              // 0/0 -> NaN as tf.linalg.normalize
        }
        float mx = -INFINITY;
        for (int i = lane; i < M; i += 32) {
            const float l = s_s[i] + (s_m[i] != 0.f ? 0.f : -1e9f);
            s_ga[i] = l;
            mx = fmaxf(mx, l);
        }
        mx = warp_max(mx);
        float se = 0.f;
        for (int i = lane; i < M; i += 32) {
            const float e = expf(s_ga[i] - mx);
            s_ga[i] = e;
            se += e;
        }
        se = warp_sum(se);
        for (int i = lane; i < M; i += 32) s_ga[i] = s_ga[i] / se;
        if (lane == 0) s_sc[0] = nrm;
    }
    __syncthreads();
    return s_sc[0];
}

__global__ void __launch_bounds__(GA2_THREADS, 1) ga_head_fwd_staged_kernel(
    const float* __restrict__ qk, const uint8_t* __restrict__ atom_mask, int M, int norm, const float* __restrict__ Wb,
    const float* __restrict__ bb, const float* __restrict__ wp, const float* __restrict__ bp, int mrelu,
    float* __restrict__ ga, float* __restrict__ y, float* __restrict__ ctx_out, float* __restrict__ tb_out) {
    extern __shared__ __align__(16) float sm[];
    const int Mp = (M + 3) & ~3;
    float* s_qk = sm;                          // M x 256
    float* s_part = s_qk + (size_t)M * 256;    // 4 x 128
    float* s_Q = s_part + 512;                 // 128
    float* s_ctx = s_Q + SCANN_D;              // 128
    float* s_s = s_ctx + SCANN_D;              // Mp
    float* s_ga = s_s + Mp;                    // Mp
    float* s_m = s_ga + Mp;                    // Mp
    float* s_sc = s_m + Mp;                    // 8
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, col = tid & 127, kq = tid >> 7;
    float wb[32];
#pragma unroll
    for (int d = 0; d < 32; ++d) wb[d] = __ldg(Wb + (size_t)(kq * 32 + d) * SCANN_D + col);
    const float bbc = bb[col], wpc = wp[col], bp0 = bp[0];
    pdl_wait();
    pdl_trigger();      // only after the own wait: at most one kernel ahead becomes resident early
    ga2_stage(qk + (size_t)b * M * 2 * SCANN_D, atom_mask + (size_t)b * M, M, s_qk, s_m);
    __syncthreads();
    ga2_scores(M, norm, s_qk, s_m, s_part, s_Q, s_s, s_ga, s_sc);
    for (int i = tid; i < M; i += GA2_THREADS) ga[(size_t)b * M + i] = s_ga[i];
    float c = 0.f;
    for (int i = kq; i < M; i += 4) c = fmaf(s_ga[i], s_m[i] != 0.f ? s_qk[i * 256 + SCANN_D + col] : 0.f, c);
    s_part[kq * 128 + col] = c;
    __syncthreads();
    if (tid < 128) {
        c = ga2_comb(s_part, tid);
        s_ctx[tid] = c;
        if (ctx_out) ctx_out[(size_t)b * SCANN_D + tid] = c;
    }
    __syncthreads();
    float t = 0.f;
#pragma unroll
    for (int d = 0; d < 32; ++d) t = fmaf(s_ctx[kq * 32 + d], wb[d], t);
    s_part[kq * 128 + col] = t;
    __syncthreads();
    if (tid < 128) {
        t = bbc + ga2_comb(s_part, tid);
        if (tb_out) tb_out[(size_t)b * SCANN_D + tid] = t;
        const float v = warp_sum(swish_f(t) * wpc);
        if (lane == 0) s_sc[1 + warp] = v;
    }
    __syncthreads();
    if (tid == 0) {
        float yy = (s_sc[1] + s_sc[2] + s_sc[3] + s_sc[4]) + bp0;
        if (mrelu) yy = fmaxf(yy, 0.f);      // mrelu forward (custom_layers.py:15)
        y[b] = yy;
    }
}

template <bool DET>
__global__ void __launch_bounds__(GA2_THREADS, 1) ga_head_bwd_staged_kernel(
    const float* __restrict__ qk, const uint8_t* __restrict__ atom_mask, int M, int norm,
    const float* __restrict__ WbT, const float* __restrict__ wp, const float* __restrict__ tb,
    const float* __restrict__ dy, float* __restrict__ d_qk, float* __restrict__ d_tb, float* __restrict__ dwp,
    float* __restrict__ dbp) {
    extern __shared__ __align__(16) float sm[];
    const int Mp = (M + 3) & ~3;
    float* s_qk = sm;                          // M x 256
    float* s_part = s_qk + (size_t)M * 256;    // 4 x 128
    float* s_Q = s_part + 512;                 // 128
    float* s_dctx = s_Q + SCANN_D;             // 128
    float* s_dtb = s_dctx + SCANN_D;           // 128
    float* s_s = s_dtb + SCANN_D;              // Mp  normalised scores
    float* s_ga = s_s + Mp;                    // Mp
    float* s_ds = s_ga + Mp;                   // Mp  d_ga -> d_t -> d_s
    float* s_m = s_ds + Mp;                    // Mp
    float* s_sc = s_m + Mp;                    // 8
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, col = tid & 127, kq = tid >> 7;
    float wt[32];                              // d_ctx[col] = sum_n d_tb[n] WbT[n][col]: this quarter's 32 n
#pragma unroll
    for (int n = 0; n < 32; ++n) wt[n] = __ldg(WbT + (size_t)(kq * 32 + n) * SCANN_D + col);
    const float wpc = wp[col];
    pdl_wait();
    pdl_trigger();      // only after the own wait: at most one kernel ahead becomes resident early
    ga2_stage(qk + (size_t)b * M * 2 * SCANN_D, atom_mask + (size_t)b * M, M, s_qk, s_m);
    const float g = dy[b];
    if (tid < 128) {                           // head
        const float t = tb[(size_t)b * SCANN_D + tid];
        if constexpr (DET) {
            dwp[(size_t)b * SCANN_D + tid] = g * swish_f(t);
            if (tid == 0) dbp[b] = g;
        } else {
            atomicAdd(dwp + tid, g * swish_f(t));
            if (tid == 0) atomicAdd(dbp, g);
        }
        const float dt = g * wpc * swish_grad_f(t);
        s_dtb[tid] = dt;
        d_tb[(size_t)b * SCANN_D + tid] = dt;
    }
    __syncthreads();
    {
        float dc = 0.f;
#pragma unroll
        for (int n = 0; n < 32; ++n) dc = fmaf(s_dtb[kq * 32 + n], wt[n], dc);
        s_part[kq * 128 + col] = dc;
    }
    __syncthreads();
    if (tid < 128) s_dctx[tid] = ga2_comb(s_part, tid);
    __syncthreads();                           // s_part is rewritten by the score pass
    const float nrm = ga2_scores(M, norm, s_qk, s_m, s_part, s_Q, s_s, s_ga, s_sc);
    {                                          // d_ga_i = m_i <d_ctx, k_i>
        const float4 dc4 = ld4(s_dctx + lane * 4);
        for (int i = warp; i < M; i += GA2_THREADS / 32) {
            const float4 k = ld4(s_qk + i * 256 + SCANN_D + lane * 4);
            float v = k.x * dc4.x + k.y * dc4.y + k.z * dc4.z + k.w * dc4.w;
            v = warp_sum(s_m[i] != 0.f ? v : 0.f);
            if (lane == 0) s_ds[i] = v;
        }
    }
    __syncthreads();
    if (warp == 0) {                           // softmax / normalisation backward over the M-vector
        float p = 0.f;
        for (int i = lane; i < M; i += 32) p = fmaf(s_ga[i], s_ds[i], p);
        const float dot = warp_sum(p);
        float q = 0.f;
        for (int i = lane; i < M; i += 32) {
            const float dt = s_ga[i] * (s_ds[i] - dot);
            s_ds[i] = dt;
            q = fmaf(s_s[i], dt, q);
        }
        if (norm) {
            const float sd = warp_sum(q);
            for (int i = lane; i < M; i += 32) s_ds[i] = (s_ds[i] - s_s[i] * sd) / nrm;
        }
        for (int i = lane; i < M; i += 32)
            if (s_m[i] == 0.f) s_ds[i] = 0.f;
    }
    __syncthreads();
    {                                          // d_Q[col] = sum_i d_s_i m_i k_i[col]
        float a = 0.f;
        for (int i = kq; i < M; i += 4) a = fmaf(s_ds[i], s_m[i] != 0.f ? s_qk[i * 256 + SCANN_D + col] : 0.f, a);
        s_part[kq * 128 + col] = a;
    }
    __syncthreads();
    const float dQ = ga2_comb(s_part, col), Q = s_Q[col], dctx = s_dctx[col];
    float* dqkb = d_qk + (size_t)b * M * 2 * SCANN_D;
    for (int i = kq; i < M; i += 4) {
        const float q = s_qk[i * 256 + col], k = s_qk[i * 256 + SCANN_D + col];
        float dq = 0.f, dk = 0.f;
        if (s_m[i] != 0.f) {
            dk = s_ga[i] * dctx + s_ds[i] * (Q - q);
            dq = dQ - s_ds[i] * k;
        }
        dqkb[(size_t)i * 2 * SCANN_D + col] = dq;
        dqkb[(size_t)i * 2 * SCANN_D + SCANN_D + col] = dk;
    }
}

static inline size_t ga2_smem_bytes(int M, bool bwd) {
    const int Mp = (M + 3) & ~3;
    return ((size_t)M * 256 + 512 + (bwd ? 3 : 2) * SCANN_D + (bwd ? 4 : 3) * Mp + 8) * sizeof(float);
}
// the staged kernels need the opt-in shared-memory limit once per process
static bool ga2_ready() {
    static int state = 0;                      // 0 unknown, 1 ok, -1 failed (fall back to the unstaged kernels)
    if (state == 0) {
        cudaError_t e1 = cudaFuncSetAttribute(ga_head_fwd_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GA2_SMEM_MAX);
        cudaError_t e2 = cudaFuncSetAttribute(ga_head_bwd_staged_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, GA2_SMEM_MAX);
        cudaError_t e3 = cudaFuncSetAttribute(ga_head_bwd_staged_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, GA2_SMEM_MAX);
        state = (e1 == cudaSuccess && e2 == cudaSuccess && e3 == cudaSuccess) ? 1 : -1;
        if (state < 0) cudaGetLastError();
    }
    return state > 0;
}

// err_b = y_b - t_b ; dy_b = err_b (the 1/(B*RMSE) factor of d sqrt(mean err^2) is applied in the
// optimiser AFTER the gradient all-reduce, so data-parallel ranks need one collective only);
// sse[0] += sum err^2, abs_err[0] += sum |err|.
// DET (deterministic mode, launched as ONE CTA): the sums are stored, not added.
template <bool DET>
__global__ void __launch_bounds__(256) rmse_prepare_kernel(const float* __restrict__ y, const float* __restrict__ target,
                                                           int B, float* __restrict__ dy, float* __restrict__ sse) {
    __shared__ float s_a[8], s_b[8];
    pdl_wait();
    pdl_trigger();      // only after the own wait: at most one kernel ahead becomes resident early
    float a = 0.f, c = 0.f;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B; i += gridDim.x * blockDim.x) {
        float e = y[i] - target[i];
        dy[i] = e;
        a = fmaf(e, e, a);
        c += fabsf(e);
    }
    a = warp_sum(a);
    c = warp_sum(c);
    if ((threadIdx.x & 31) == 0) { s_a[threadIdx.x >> 5] = a; s_b[threadIdx.x >> 5] = c; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float ta = 0.f, tc = 0.f;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { ta += s_a[w]; tc += s_b[w]; }
        if constexpr (DET) {
            sse[0] = ta;
            sse[1] = tc;
        } else {
            atomicAdd(sse, ta);
            atomicAdd(sse + 1, tc);
        }
    }
}

extern "C" int scann_ga_head_forward(const float* qk, const uint8_t* atom_mask, int B, int M, int norm,
                                     const float* Wb, const float* bb, const float* wp, const float* bp, int mrelu,
                                     float* ga, float* y, float* ctx_out, float* tb_out, void* stream) {
    if (B <= 0) return 0;
    if (ga2_smem_bytes(M, false) <= GA2_SMEM_MAX && ga2_ready()) {
        scann_launch(ga_head_fwd_staged_kernel, dim3(B), dim3(GA2_THREADS), ga2_smem_bytes(M, false), stream, qk, atom_mask, M,
                     norm, Wb, bb, wp, bp, mrelu, ga, y, ctx_out, tb_out);
        return scann_check_launch("scann_ga_head_forward");
    }
    size_t smem = (size_t)(2 * SCANN_D + 4 + 2 * M) * sizeof(float);
    if (smem > 48 * 1024) { scann_set_error("ga_head_forward: M=%d too large", M); return 1; }
    scann_launch(ga_head_fwd_kernel, dim3(B), dim3(GA_THREADS), smem, stream, qk, atom_mask, M, norm, Wb, bb, wp, bp, mrelu,
                 ga, y, ctx_out, tb_out);
    return scann_check_launch("scann_ga_head_forward");
}

template <bool DET>
static int ga_head_backward_launch(const float* qk, const uint8_t* atom_mask, int B, int M, int norm, const float* WbT,
                                   const float* wp, const float* tb, const float* dy, float* d_qk, float* d_tb, float* dwp,
                                   float* dbp, void* stream) {
    if (B <= 0) return 0;
    if (ga2_smem_bytes(M, true) <= GA2_SMEM_MAX && ga2_ready()) {
        scann_launch(ga_head_bwd_staged_kernel<DET>, dim3(B), dim3(GA2_THREADS), ga2_smem_bytes(M, true), stream, qk, atom_mask, M,
                     norm, WbT, wp, tb, dy, d_qk, d_tb, dwp, dbp);
        return scann_check_launch("scann_ga_head_backward");
    }
    size_t smem = (size_t)(3 * SCANN_D + 4 + 3 * M) * sizeof(float);
    if (smem > 48 * 1024) { scann_set_error("ga_head_backward: M=%d too large", M); return 1; }
    scann_launch(ga_head_bwd_kernel<DET>, dim3(B), dim3(GA_THREADS), smem, stream, qk, atom_mask, M, norm, WbT, wp, tb, dy, d_qk,
                 d_tb, dwp, dbp);
    return scann_check_launch("scann_ga_head_backward");
}

extern "C" int scann_ga_head_backward(const float* qk, const uint8_t* atom_mask, int B, int M, int norm,
                                      const float* WbT, const float* wp, const float* tb, const float* dy,
                                      float* d_qk, float* d_tb, float* dwp, float* dbp, void* stream) {
    return ga_head_backward_launch<false>(qk, atom_mask, B, M, norm, WbT, wp, tb, dy, d_qk, d_tb, dwp, dbp, stream);
}

// Deterministic form: dwp_slots [B][128] and dbp_slots [B] receive the head gradient of each structure (scann_slot_reduce
// adds them up in structure order).
extern "C" int scann_ga_head_backward_det(const float* qk, const uint8_t* atom_mask, int B, int M, int norm,
                                          const float* WbT, const float* wp, const float* tb, const float* dy,
                                          float* d_qk, float* d_tb, float* dwp_slots, float* dbp_slots, void* stream) {
    return ga_head_backward_launch<true>(qk, atom_mask, B, M, norm, WbT, wp, tb, dy, d_qk, d_tb, dwp_slots, dbp_slots, stream);
}

extern "C" int scann_rmse_prepare(const float* y, const float* target, int B, float* dy, float* sse, void* stream) {
    if (B <= 0) return 0;
    int grid = (B + 255) / 256;
    if (grid > 64) grid = 64;
    scann_launch(rmse_prepare_kernel<false>, dim3(grid), dim3(256), 0, stream, y, target, B, dy, sse);
    return scann_check_launch("scann_rmse_prepare");
}

// Deterministic form: one CTA walks the whole batch and stores the sums into sse[0..1] in a fixed order.
extern "C" int scann_rmse_prepare_det(const float* y, const float* target, int B, float* dy, float* sse, void* stream) {
    if (B <= 0) return 0;
    scann_launch(rmse_prepare_kernel<true>, dim3(1), dim3(256), 0, stream, y, target, B, dy, sse);
    return scann_check_launch("scann_rmse_prepare_det");
}
