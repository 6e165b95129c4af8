// Optimiser step over the flat parameter arena: Keras-2.10 Adam(lr, decay=1e-5)
// (scann/models/scann_model.py:212) fused with the loss-gradient scaling and the l2
// regulariser gradient (kernel_regularizer=l2(1e-4): attention.py:27-28,95,97,108,260,262;
// scann_model.py:428,441).
//
// Backward kernels produce  G = sum_b err_b * d y_b / d theta  (err_b = y_b - t_b).
// loss = sqrt(SSE / B) + 1e-4 * sum_{l2 kernels} W^2   (scann/layers/losses.py:5-6), hence
//   d loss / d theta = G / (B * sqrt(SSE / B)) + 2e-4 * W * [theta is an l2 kernel]
// SSE sits right behind the gradients in the same arena so one all-reduce covers both.
#include "common.cuh"

struct AdamScalars {      // filled by the host every step (device copy)
    float alpha;          // lr_t * sqrt(1 - b2^t) / (1 - b1^t)
    float b1, b2, eps;
    float l2;             // 1e-4
    float batch;          // global batch size B
};

// DET (deterministic mode): the l2 sum of a CTA is combined in warp order and stored into reg_slots[blockIdx.x];
// adam_reg_sum_kernel adds the slots up in CTA order.
template <bool DET>
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                   float* __restrict__ m, float* __restrict__ v,
                                                   const float* __restrict__ l2mask, int n,
                                                   float* __restrict__ sse_rw, const AdamScalars* __restrict__ hs,
                                                   float* __restrict__ grad_out, int apply, float* __restrict__ reg_slots) {
    const float* sse = sse_rw;
    const AdamScalars h = *hs;
    const float rmse = sqrtf(sse[0] / h.batch);
    const float scale = 1.0f / (h.batch * rmse);
    float reg = 0.f;
    auto one = [&](float w, float gi, float lm, float& mi, float& vi, float& gr) -> float {
        reg = fmaf(lm * w, w, reg);                  // l2 penalty of the weights the loss was evaluated with
        gr = fmaf(gi, scale, 2.0f * h.l2 * lm * w);
        if (!apply) return w;
        mi = h.b1 * mi + (1.0f - h.b1) * gr;
        vi = h.b2 * vi + (1.0f - h.b2) * gr * gr;
        return w - h.alpha * mi / (sqrtf(vi) + h.eps);
    };
    // 16-byte accesses over the aligned body of the arena (seven streams of n floats), scalar tail
    const bool al16 = (((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v | (uintptr_t)l2mask | (uintptr_t)grad_out) & 15) == 0;
    const int n4 = al16 ? n >> 2 : 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
        const float4 w = reinterpret_cast<const float4*>(p)[i], gi = reinterpret_cast<const float4*>(g)[i],
                     lm = reinterpret_cast<const float4*>(l2mask)[i];
        float4 mi = make_float4(0.f, 0.f, 0.f, 0.f), vi = mi, gr, o;
        if (apply) { mi = reinterpret_cast<const float4*>(m)[i]; vi = reinterpret_cast<const float4*>(v)[i]; }
        o.x = one(w.x, gi.x, lm.x, mi.x, vi.x, gr.x); o.y = one(w.y, gi.y, lm.y, mi.y, vi.y, gr.y);
        o.z = one(w.z, gi.z, lm.z, mi.z, vi.z, gr.z); o.w = one(w.w, gi.w, lm.w, mi.w, vi.w, gr.w);
        if (grad_out) reinterpret_cast<float4*>(grad_out)[i] = gr;
        if (apply) {
            reinterpret_cast<float4*>(m)[i] = mi;
            reinterpret_cast<float4*>(v)[i] = vi;
            reinterpret_cast<float4*>(p)[i] = o;
        }
    }
    for (int i = 4 * n4 + blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float mi = apply ? m[i] : 0.f, vi = apply ? v[i] : 0.f, gr;
        const float o = one(p[i], g[i], l2mask[i], mi, vi, gr);
        if (grad_out) grad_out[i] = gr;
        if (apply) { m[i] = mi; v[i] = vi; p[i] = o; }
    }
    reg = warp_sum(reg);
    if constexpr (DET) {
        __shared__ float s_reg[8];
        if ((threadIdx.x & 31) == 0) s_reg[threadIdx.x >> 5] = reg;
        __syncthreads();
        if (threadIdx.x == 0) {
            float t = 0.f;
            for (int w = 0; w < 8; ++w) t += s_reg[w];
            reg_slots[blockIdx.x] = t;
        }
    } else {
        if ((threadIdx.x & 31) == 0) atomicAdd(sse_rw + 2, reg);
    }
}

// one CTA: thread i adds slots i, i + 256, ... in order, then the 256 partials are added in thread order
__global__ void __launch_bounds__(256) adam_reg_sum_kernel(const float* __restrict__ reg_slots, int nslots,
                                                           float* __restrict__ sse_rw) {
    __shared__ float s_t[256];
    float t = 0.f;
    for (int k = threadIdx.x; k < nslots; k += 256) t += reg_slots[k];
    s_t[threadIdx.x] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
        float a = 0.f;
        for (int i = 0; i < 256; ++i) a += s_t[i];
        sse_rw[2] += a;
    }
}

// out[0] = sqrt(SSE/B) + l2 * sum(mask * p^2) ; out[1] = sqrt(SSE/B) ; out[2] = sum|err| / B.
// sse[0] = SSE, sse[1] = sum |err| (scann_rmse_prepare), sse[2] = sum(mask * p^2) (scann_adam_step).
__global__ void loss_value_kernel(const float* __restrict__ sse, float batch, float l2, float* __restrict__ out) {
    float rmse = sqrtf(sse[0] / batch);
    out[0] = rmse + l2 * sse[2];
    out[1] = rmse;
    out[2] = sse[1] / batch;
}

extern "C" int scann_adam_step(float* params, const float* grads, float* m, float* v, const float* l2mask, int n,
                               float* sse, const void* scalars_dev, float* grad_out, int apply, void* stream) {
    if (n <= 0) return 0;
    int grid = (n / 4 + 255) / 256 + 1;
    if (grid > 1184) grid = 1184;
    adam_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(params, grads, m, v, l2mask, n, sse,
                                                               (const AdamScalars*)scalars_dev, grad_out, apply, nullptr);
    return scann_check_launch("scann_adam_step");
}

// Deterministic form: reg_slots = 1184 floats of workspace (the l2 sum per CTA).
extern "C" int scann_adam_step_det(float* params, const float* grads, float* m, float* v, const float* l2mask, int n,
                                   float* sse, const void* scalars_dev, float* grad_out, int apply, float* reg_slots,
                                   void* stream) {
    if (n <= 0) return 0;
    int grid = (n / 4 + 255) / 256 + 1;
    if (grid > 1184) grid = 1184;
    adam_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(params, grads, m, v, l2mask, n, sse,
                                                              (const AdamScalars*)scalars_dev, grad_out, apply, reg_slots);
    adam_reg_sum_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(reg_slots, grid, sse);
    return scann_check_launch("scann_adam_step_det");
}

extern "C" int scann_loss_value(const float* params, const float* l2mask, int n, const float* sse, float batch,
                                float l2, float* out3, void* stream) {
    (void)params; (void)l2mask; (void)n;
    loss_value_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(sse, batch, l2, out3);
    return scann_check_launch("scann_loss_value");
}
