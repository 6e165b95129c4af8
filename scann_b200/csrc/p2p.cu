// Data-parallel gradient exchange fused into the optimiser kernel, over NVLink peer memory.
//
// The reference trains on one device (keras fit, scann_model.py:232-241); here the batch is sharded over one
// process per GPU and every rank needs  G = sum_r G_r  (gradient arena + SSE, scann_b200/dist.py) before the Adam
// update.  With NCCL that is a launch + a latency-bound 3.6 MB all-reduce + the optimiser's own pass over the
// arena (55-85 us per 1.2 ms step).  Here every rank's gradient arena lives in a block that the other ranks map
// through CUDA IPC, and the optimiser kernel sums the peers' values itself while it updates: one pass, no
// collective launch.  Summation order is rank 0, 1, ... on EVERY rank, so the parameters stay bit-identical.
//
// Block of rank r (one cudaMalloc, one IPC handle):  [ arena: n + 4 floats, padded ] [ flags: 64 x u32 ]
//   flags[ 0.. 7]  ready[s]: rank s has finished its backward pass of step e   (written by rank s, value e)
//   flags[16..23]  done[s] : rank s has finished READING this rank's arena in step e
//   flags[32]      ticket of the optimiser kernel's CTAs ; flags[33] number of completed steps (epoch)
// Protocol per step e = epoch + 1 (all inside kernels, so it is captured into the step's CUDA graph):
//   scann_p2p_begin_step : wait until done[s] >= e - 1 for all s (the peers no longer read the arena that is
//                          about to be zeroed), zero the loss sums
//   ... zero arena, forward, backward ...
//   scann_adam_p2p_step  : block 0 publishes ready[r] = e to every peer; every CTA waits for ready[s] >= e; the
//                          kernel sums the arenas and updates; the last CTA publishes done[r] = e and advances
//                          the epoch.
// With four or more ranks the sum is TWO-SHOT (reading every peer's whole arena costs (W-1) x 3.6 MB per rank over
// NVLink: 36 us at 8 ranks, no better than NCCL): behind the flags the block carries a second arena-sized buffer;
// rank r first sums slice r of all arenas into its own buffer (reduce-scatter: (W-1)/W of one arena read remotely),
// publishes red[r] = e, and every rank then reads the W reduced slices from their owners (all-gather, again (W-1)/W of
// one arena) while it applies Adam.  Same summation order on every rank as before: parameters stay bit-identical.
#include <string.h>

#include "common.cuh"

#define P2P_MAX_RANKS 8
#define P2P_READY 0
#define P2P_DONE 16
#define P2P_TICKET 32
#define P2P_EPOCH 33
#define P2P_TICKET2 34                         // CTAs of this rank that have finished the reduce-scatter phase
#define P2P_RED 40                             // red[s]: rank s has written its reduced slice of step e
#define P2P_FLAG_WORDS 64
#define P2P_TWO_SHOT_MIN_RANKS 4

struct P2PBlock {
    const float* arena[P2P_MAX_RANKS];      // arena of every rank (own entry = local pointer)
    uint32_t* flags[P2P_MAX_RANKS];         // flag words of every rank
    int world, rank;
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// Spin until *p has reached `target` (wrap-safe) -- BOUNDED: a peer that died or a protocol error must not hang the
// GPU.  After ~2 s the wait gives up and marks sums[3] (the engine reports it); the step's result is then garbage.
__device__ __forceinline__ void p2p_wait_flag(const uint32_t* p, uint32_t target, float* sums) {
    const long long t0 = clock64();
    while ((int32_t)(ld_acquire_sys(p) - target) < 0) {
        if (clock64() - t0 > 4000000000LL) { if (sums) sums[3] = 1.0f; return; }
    }
}

struct AdamScalarsP {      // same block as AdamScalars in optim.cu
    float alpha, b1, b2, eps, l2, batch;
};

__global__ void __launch_bounds__(32) p2p_begin_step_kernel(const P2PBlock* __restrict__ blk, float* __restrict__ sums) {
    const P2PBlock b = *blk;
    const uint32_t* fl = b.flags[b.rank];
    const uint32_t e_prev = fl[P2P_EPOCH];
    const int s = threadIdx.x;
    if (s < 3) sums[s] = 0.f;                   // sums[3]: sticky "a flag wait gave up" marker
    if (s < b.world && s != b.rank) p2p_wait_flag(fl + P2P_DONE + s, e_prev, sums);
}

// sums[0] = global SSE, [1] = global sum |err|, [2] = l2 penalty sum (as sse[0..2] of adam_kernel / loss_value)
// DET (deterministic mode): the l2 sum of a CTA is combined in warp order and stored into reg_slots[blockIdx.x]; the
// last CTA of the rank (the ticket below) adds the slots in CTA order and stores sums[2].
template <bool DET>
__global__ void __launch_bounds__(256) adam_p2p_kernel(float* __restrict__ p, float* __restrict__ m, float* __restrict__ v,
                                                       const float* __restrict__ l2mask, int n,
                                                       const P2PBlock* __restrict__ blk, float* __restrict__ sums,
                                                       const AdamScalarsP* __restrict__ hs, float* __restrict__ grad_out,
                                                       int apply, float* __restrict__ reg_slots) {
    __shared__ P2PBlock b;
    if (threadIdx.x == 0) b = *blk;
    __syncthreads();
    uint32_t* fl = b.flags[b.rank];
    const uint32_t e = fl[P2P_EPOCH] + 1u;
    if (blockIdx.x == 0 && (int)threadIdx.x < b.world && (int)threadIdx.x != b.rank) {
        __threadfence_system();                 // this rank's gradients (earlier kernels of the stream) before the flag
        st_release_sys(b.flags[threadIdx.x] + P2P_READY + b.rank, e);
    }
    if ((int)threadIdx.x < b.world && (int)threadIdx.x != b.rank) p2p_wait_flag(fl + P2P_READY + threadIdx.x, e, sums);
    __syncthreads();
    const AdamScalarsP h = *hs;
    const int n4 = n >> 2;                      // every arena is 16-byte aligned (scann_p2p_alloc)
    const bool two_shot = b.world >= P2P_TWO_SHOT_MIN_RANKS;
    const int per = (n4 + b.world - 1) / b.world;                    // float4 elements per reduced slice
    if (two_shot) {
        // ---- reduce-scatter: this rank's slice of every arena -> its reduced buffer (behind its flag words)
        float4* red = reinterpret_cast<float4*>(fl + P2P_FLAG_WORDS);
        const int lo = b.rank * per, hi = min(n4, lo + per);
        for (int i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x) {
            // all remote loads first (a loop over a runtime rank count issues them one NVLink round trip after the other),
            // then the sum in rank order
            float4 t[P2P_MAX_RANKS];
#pragma unroll
            for (int r = 0; r < P2P_MAX_RANKS; ++r)
                t[r] = r < b.world ? reinterpret_cast<const float4*>(b.arena[r])[i] : make_float4(0.f, 0.f, 0.f, 0.f);
            float4 gi = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int r = 0; r < P2P_MAX_RANKS; ++r)
                if (r < b.world) { gi.x += t[r].x; gi.y += t[r].y; gi.z += t[r].z; gi.w += t[r].w; }
            red[i] = gi;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            const uint32_t t = atomicAdd(fl + P2P_TICKET2, 1u);
            if (t == gridDim.x - 1) {                                  // the last CTA of this rank: slice complete
                fl[P2P_TICKET2] = 0u;
                __threadfence_system();
                for (int r = 0; r < b.world; ++r) st_release_sys(b.flags[r] + P2P_RED + b.rank, e);
            }
        }
        if ((int)threadIdx.x < b.world) p2p_wait_flag(fl + P2P_RED + threadIdx.x, e, sums);
        __syncthreads();
    }
    float sse = 0.f, sabs = 0.f;
    {
        float s0[P2P_MAX_RANKS], s1[P2P_MAX_RANKS];
#pragma unroll
        for (int r = 0; r < P2P_MAX_RANKS; ++r) { s0[r] = r < b.world ? b.arena[r][n] : 0.f; s1[r] = r < b.world ? b.arena[r][n + 1] : 0.f; }
#pragma unroll
        for (int r = 0; r < P2P_MAX_RANKS; ++r) if (r < b.world) { sse += s0[r]; sabs += s1[r]; }
    }
    const float rmse = sqrtf(sse / h.batch);
    const float scale = 1.0f / (h.batch * rmse);
    if (blockIdx.x == 0 && threadIdx.x == 0) { sums[0] = sse; sums[1] = sabs; }
    float reg = 0.f;
    auto one = [&](float w, float gi, float lm, float& mi, float& vi, float& gr) -> float {
        reg = fmaf(lm * w, w, reg);
        gr = fmaf(gi, scale, 2.0f * h.l2 * lm * w);
        if (!apply) return w;
        mi = h.b1 * mi + (1.0f - h.b1) * gr;
        vi = h.b2 * vi + (1.0f - h.b2) * gr * gr;
        return w - h.alpha * mi / (sqrtf(vi) + h.eps);
    };
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
        float4 gi = make_float4(0.f, 0.f, 0.f, 0.f);
        if (two_shot) {                         // all-gather: the reduced slice of its owner
            gi = reinterpret_cast<const float4*>(b.flags[i / per] + P2P_FLAG_WORDS)[i];
        } else {
            float4 t[P2P_TWO_SHOT_MIN_RANKS - 1];                  // one-shot form: at most three ranks
#pragma unroll
            for (int r = 0; r < P2P_TWO_SHOT_MIN_RANKS - 1; ++r)
                t[r] = r < b.world ? reinterpret_cast<const float4*>(b.arena[r])[i] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int r = 0; r < P2P_TWO_SHOT_MIN_RANKS - 1; ++r)
                if (r < b.world) { gi.x += t[r].x; gi.y += t[r].y; gi.z += t[r].z; gi.w += t[r].w; }
        }
        const float4 w = reinterpret_cast<const float4*>(p)[i], lm = reinterpret_cast<const float4*>(l2mask)[i];
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
        float gi = 0.f;
        for (int r = 0; r < b.world; ++r) gi += b.arena[r][i];
        float mi = apply ? m[i] : 0.f, vi = apply ? v[i] : 0.f, gr;
        const float o = one(p[i], gi, l2mask[i], mi, vi, gr);
        if (grad_out) grad_out[i] = gr;
        if (apply) { m[i] = mi; v[i] = vi; p[i] = o; }
    }
    reg = warp_sum(reg);
    __shared__ float s_reg[8];
    if constexpr (DET) {
        if ((threadIdx.x & 31) == 0) s_reg[threadIdx.x >> 5] = reg;
    } else {
        if ((threadIdx.x & 31) == 0) atomicAdd(sums + 2, reg);
    }
    // the last CTA of this rank: every read of the peers' arenas is complete
    __syncthreads();
    if (threadIdx.x == 0) {
        if constexpr (DET) {
            float t = 0.f;
            for (int w = 0; w < 8; ++w) t += s_reg[w];
            reg_slots[blockIdx.x] = t;
        }
        __threadfence();
        const uint32_t t = atomicAdd(fl + P2P_TICKET, 1u);
        if (t == gridDim.x - 1) {
            if constexpr (DET) {
                __threadfence();
                const volatile float* rs = reg_slots;
                float a = 0.f;
                for (int c = 0; c < (int)gridDim.x; ++c) a += rs[c];
                sums[2] = a;
            }
            fl[P2P_TICKET] = 0u;
            fl[P2P_EPOCH] = e;
            __threadfence_system();
            for (int r = 0; r < b.world; ++r)
                if (r != b.rank) st_release_sys(b.flags[r] + P2P_DONE + b.rank, e);
        }
    }
}

// ---- host side ------------------------------------------------------------------------------------------
// One zeroed device allocation that other processes of the node can map (gradient arena + flag words).
extern "C" int scann_p2p_alloc(long long bytes, void** out_ptr) {
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, (size_t)bytes);
    if (e == cudaSuccess) e = cudaMemset(p, 0, (size_t)bytes);
    if (e != cudaSuccess) { scann_set_error("p2p_alloc: %s", cudaGetErrorString(e)); return 1; }
    *out_ptr = p;
    return 0;
}
extern "C" int scann_p2p_free(void* ptr) {
    cudaError_t e = cudaFree(ptr);
    if (e != cudaSuccess) { scann_set_error("p2p_free: %s", cudaGetErrorString(e)); return 1; }
    return 0;
}
// handle64: 64 bytes (cudaIpcMemHandle_t), to be sent to the other ranks of the node
extern "C" int scann_p2p_export(void* ptr, void* handle64) {
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, ptr);
    if (e != cudaSuccess) { scann_set_error("p2p_export: %s", cudaGetErrorString(e)); return 1; }
    memcpy(handle64, &h, sizeof(h));
    return 0;
}
extern "C" int scann_p2p_import(const void* handle64, void** out_ptr) {
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, sizeof(h));
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { scann_set_error("p2p_import: %s", cudaGetErrorString(e)); return 1; }
    *out_ptr = p;
    return 0;
}
extern "C" int scann_p2p_close(void* ptr) {
    cudaError_t e = cudaIpcCloseMemHandle(ptr);
    if (e != cudaSuccess) { scann_set_error("p2p_close: %s", cudaGetErrorString(e)); return 1; }
    return 0;
}

// block_dev: device copy of {arena[8], flags[8], world, rank} (ScannP2PBlock of include/scann_b200.h); sums: 4 floats.
extern "C" int scann_p2p_begin_step(const void* block_dev, float* sums, void* stream) {
    p2p_begin_step_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((const P2PBlock*)block_dev, sums);
    return scann_check_launch("scann_p2p_begin_step");
}

// scann_adam_step with the cross-rank sum folded in: the gradients are read from every rank's arena (block_dev)
// instead of one local, already reduced, array; sums[0..2] receive what scann_adam_step leaves in sse[0..2].
extern "C" int scann_adam_p2p_step(float* params, float* m, float* v, const float* l2mask, int n, const void* block_dev,
                                   float* sums, const void* scalars_dev, float* grad_out, int apply, void* stream) {
    if (n <= 0) return 0;
    if ((((uintptr_t)params | (uintptr_t)m | (uintptr_t)v | (uintptr_t)l2mask | (uintptr_t)grad_out) & 15) != 0) {
        scann_set_error("adam_p2p_step: arrays must be 16-byte aligned");
        return 1;
    }
    int grid = (n / 4 + 255) / 256 + 1;
    if (grid > 592) grid = 592;                  // all CTAs resident at once (they wait for the peers' flags)
    adam_p2p_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(params, m, v, l2mask, n, (const P2PBlock*)block_dev, sums,
                                                                  (const AdamScalarsP*)scalars_dev, grad_out, apply, nullptr);
    return scann_check_launch("scann_adam_p2p_step");
}

// Deterministic form: reg_slots = 592 floats of workspace (the l2 sum per CTA, added up in CTA order).  The cross-rank
// sum is already in rank order.
extern "C" int scann_adam_p2p_step_det(float* params, float* m, float* v, const float* l2mask, int n, const void* block_dev,
                                       float* sums, const void* scalars_dev, float* grad_out, int apply, float* reg_slots,
                                       void* stream) {
    if (n <= 0) return 0;
    if ((((uintptr_t)params | (uintptr_t)m | (uintptr_t)v | (uintptr_t)l2mask | (uintptr_t)grad_out) & 15) != 0) {
        scann_set_error("adam_p2p_step: arrays must be 16-byte aligned");
        return 1;
    }
    if (!reg_slots) { scann_set_error("adam_p2p_step_det: reg_slots is required"); return 1; }
    int grid = (n / 4 + 255) / 256 + 1;
    if (grid > 592) grid = 592;
    adam_p2p_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(params, m, v, l2mask, n, (const P2PBlock*)block_dev, sums,
                                                                 (const AdamScalarsP*)scalars_dev, grad_out, apply, reg_slots);
    return scann_check_launch("scann_adam_p2p_step_det");
}
