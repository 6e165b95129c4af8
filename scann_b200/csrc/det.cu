// Deterministic training mode (DESIGN.md section 4.7): the pieces that replace floating-point atomics by sums in an
// order fixed by the batch and the launch configuration.
//
//   scann_plan_inverse : for every atom row j, the pair rows whose neighbour is j, in ascending pair-row order (CSR)
//   scann_row_gather   : dst[j] = sum over that list of src[p], in list order (the gather_nd backward of the
//                        local-attention layers without scatter atomics)
//   scann_slot_reduce  : one launch over a table of per-CTA partial-sum arrays ("slots"): dst[i] += sum_s slot[s][i]
//                        in slot order
#include "common.cuh"

// ---- inverse neighbour CSR ----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) inv_count_kernel(const int32_t* __restrict__ ntiles, int stride,
                                                        const int32_t* __restrict__ pair_c,
                                                        const int32_t* __restrict__ pair_j, int R, int32_t* __restrict__ cnt) {
    const long long rows = (long long)*ntiles * stride;
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < rows; p += (long long)gridDim.x * blockDim.x) {
        if (pair_c[p] < 0) continue;
        const int j = pair_j[p];
        if (j >= 0 && j < R) atomicAdd(&cnt[j], 1);
    }
}

// exclusive scan of cnt[0..R) -> ptr[0..R]; cnt becomes the fill cursor (= ptr[j])
__global__ void __launch_bounds__(1024) inv_scan_kernel(int32_t* __restrict__ cnt, int R, int32_t* __restrict__ ptr) {
    __shared__ int32_t s_warp[32];
    __shared__ int32_t s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < R; base += 1024) {
        const int i = base + tid;
        const int v = i < R ? cnt[i] : 0;
        int x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) s_warp[warp] = x;
        __syncthreads();
        if (warp == 0) {
            int w = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += y;
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        const int excl = s_carry + (warp ? s_warp[warp - 1] : 0) + x - v;
        if (i < R) { ptr[i] = excl; cnt[i] = excl; }
        __syncthreads();
        if (tid == 1023) s_carry = excl + v;
        __syncthreads();
    }
    if (tid == 0) ptr[R] = s_carry;
}

// unordered fill (integer atomics: the order inside a segment depends on scheduling; inv_rank_kernel fixes it)
__global__ void __launch_bounds__(256) inv_fill_kernel(const int32_t* __restrict__ ntiles, int stride,
                                                       const int32_t* __restrict__ pair_c,
                                                       const int32_t* __restrict__ pair_j, int R,
                                                       int32_t* __restrict__ cursor, int32_t* __restrict__ tmp) {
    const long long rows = (long long)*ntiles * stride;
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < rows; p += (long long)gridDim.x * blockDim.x) {
        if (pair_c[p] < 0) continue;
        const int j = pair_j[p];
        if (j >= 0 && j < R) tmp[atomicAdd(&cursor[j], 1)] = (int32_t)p;
    }
}

// one warp per segment: every entry's position is the number of smaller entries (pair rows are distinct)
__global__ void __launch_bounds__(256) inv_rank_kernel(int R, const int32_t* __restrict__ ptr, const int32_t* __restrict__ tmp,
                                                       int32_t* __restrict__ idx) {
    const int lane = threadIdx.x & 31;
    const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (j >= R) return;
    const int b = ptr[j], n = ptr[j + 1] - b;
    for (int i = lane; i < n; i += 32) {
        const int v = tmp[b + i];
        int rank = 0;
        for (int k = 0; k < n; ++k) rank += tmp[b + k] < v;
        idx[b + rank] = v;
    }
}

extern "C" int scann_plan_inverse(const int32_t* ntiles, int tile_stride, long long rows, const int32_t* pair_c,
                                  const int32_t* pair_j, int R, int32_t* inv_ptr, int32_t* inv_idx, int32_t* cnt_ws,
                                  int32_t* tmp_ws, void* stream) {
    if (tile_stride != 32 && tile_stride != 64 && tile_stride != SCANN_TILE) { scann_set_error("plan_inverse: tile_stride must be 32, 64 or 128"); return 1; }
    if (R <= 0 || rows <= 0) { scann_set_error("plan_inverse: bad sizes R=%d rows=%lld", R, rows); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    cudaMemsetAsync(cnt_ws, 0, (size_t)R * sizeof(int32_t), st);
    long long g = (rows + 255) / 256;
    const int grid = (int)(g < 1184 ? g : 1184);
    inv_count_kernel<<<grid, 256, 0, st>>>(ntiles, tile_stride, pair_c, pair_j, R, cnt_ws);
    inv_scan_kernel<<<1, 1024, 0, st>>>(cnt_ws, R, inv_ptr);
    inv_fill_kernel<<<grid, 256, 0, st>>>(ntiles, tile_stride, pair_c, pair_j, R, cnt_ws, tmp_ws);
    inv_rank_kernel<<<(R + 7) / 8, 256, 0, st>>>(R, inv_ptr, tmp_ws, inv_idx);
    return scann_check_launch("scann_plan_inverse");
}

// ---- row gather ---------------------------------------------------------------------------------------------------
// one warp per atom row, lane l owns columns 4l..4l+3; the list is walked in order, eight indices at a time
__global__ void __launch_bounds__(256) row_gather_kernel(int R, const int32_t* __restrict__ ptr, const int32_t* __restrict__ idx,
                                                         const float* __restrict__ src0, float* __restrict__ dst0,
                                                         const float* __restrict__ src1, float* __restrict__ dst1) {
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (j < R) {
        const int b = ptr[j], e = ptr[j + 1];
        float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
        for (int k0 = b; k0 < e; k0 += 8) {
            int p[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) p[u] = k0 + u < e ? idx[k0 + u] : -1;
            float4 v0[8], v1[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                v0[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                v1[u] = v0[u];
                if (p[u] >= 0) {
                    v0[u] = ld4(src0 + (size_t)p[u] * SCANN_D + lane * 4);
                    if (src1) v1[u] = ld4(src1 + (size_t)p[u] * SCANN_D + lane * 4);
                }
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                if (p[u] < 0) break;
                a0 = make_float4(a0.x + v0[u].x, a0.y + v0[u].y, a0.z + v0[u].z, a0.w + v0[u].w);
                a1 = make_float4(a1.x + v1[u].x, a1.y + v1[u].y, a1.z + v1[u].z, a1.w + v1[u].w);
            }
        }
        st4(dst0 + (size_t)j * SCANN_D + lane * 4, a0);
        if (dst1) st4(dst1 + (size_t)j * SCANN_D + lane * 4, a1);
    }
    pdl_trigger();
}

extern "C" int scann_row_gather(int R, const int32_t* inv_ptr, const int32_t* inv_idx, const float* src0, float* dst0,
                                const float* src1, float* dst1, void* stream) {
    if (R <= 0) return 0;
    if (!src0 || !dst0 || (!src1 != !dst1)) { scann_set_error("row_gather: src / dst pairs must both be given"); return 1; }
    scann_launch(row_gather_kernel, dim3((R + 7) / 8), dim3(256), 0, stream, R, inv_ptr, inv_idx, src0, dst0, src1, dst1);
    return scann_check_launch("scann_row_gather");
}

// ---- slot reduction -----------------------------------------------------------------------------------------------
// Mirrors ScannSlotSum in include/scann_b200.h.
struct SlotSum {
    const float* slots;   // [nslots][ld]
    float* dst;           // [count] += sum over the slots, in slot order
    int nslots, count, ld, pad;
};

// A CTA covers 32 consecutive elements of one entry; its eight warps each add a contiguous eighth of the slots (in
// order), then the eight partials are added in warp order.  The split depends on nslots only: a fixed order.
__global__ void __launch_bounds__(256) slot_reduce_kernel(const SlotSum* __restrict__ table) {
    __shared__ float s_part[8][32];
    pdl_wait();
    const SlotSum e = table[blockIdx.y];
    const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + lane;
    if (blockIdx.x * 32 < e.count) {
        const int per = (e.nslots + 7) / 8, k0 = grp * per, k1 = min(e.nslots, k0 + per);
        float s = 0.f;
        if (i < e.count) {
            int k = k0;
            for (; k + 4 <= k1; k += 4) {               // four independent loads in flight, added in slot order
                const float v0 = e.slots[(size_t)k * e.ld + i], v1 = e.slots[(size_t)(k + 1) * e.ld + i];
                const float v2 = e.slots[(size_t)(k + 2) * e.ld + i], v3 = e.slots[(size_t)(k + 3) * e.ld + i];
                s += v0; s += v1; s += v2; s += v3;
            }
            for (; k < k1; ++k) s += e.slots[(size_t)k * e.ld + i];
        }
        s_part[grp][lane] = s;
        __syncthreads();
        if (grp == 0 && i < e.count) {
            float t = 0.f;
#pragma unroll
            for (int g = 0; g < 8; ++g) t += s_part[g][lane];
            e.dst[i] += t;
        }
    }
    pdl_trigger();
}

extern "C" int scann_slot_reduce(const void* table_dev, int nent, int max_count, void* stream) {
    if (nent <= 0 || max_count <= 0) return 0;
    if (nent > 65535) { scann_set_error("slot_reduce: at most 65535 table entries"); return 1; }
    scann_launch(slot_reduce_kernel, dim3((max_count + 31) / 32, nent), dim3(256), 0, stream, (const SlotSum*)table_dev);
    return scann_check_launch("scann_slot_reduce");
}
