// Chains of per-atom Dense layers in ONE kernel, WARP-SPECIALISED (round 2 form of chain_tc.cu).
//
// Same contract and arithmetic as dense_chain_kernel (chain_tc.cu: ResidualNorm + the next layer's x @ [W1|W3|Wq]
// projections in the forward pass, attention.py:25-40,141-161; their transposes with LayerNorm backward / swish' in
// the backward pass), but the 128x128 weight block no longer travels global -> registers -> hi/lo split ->
// tcgen05.st in every CTA at every GEMM step (1 700 of the ~7 800 cycles of a step there, serialised with the MMA
// issue and the epilogue).  Instead:
//
//   * weight_images_kernel writes, once per optimiser step, every 128x128 block of the parameter arena as the
//     ready-made tcgen05 operand: four K-blocks of [raw (tf32-truncated) | lo = w - raw] chunk blocks of
//     [128 rows x 128 B] in the 128-byte-swizzled K-major layout, in both orientations (W^T for the forward GEMMs,
//     W for the transposed ones) -- 128 KB per block and orientation;
//   * the PRODUCER warp streams these images with cp.async.bulk (32 KB per K-block) into a shared-memory ring,
//     as far ahead as the ring allows and before the programmatic-dependent-launch wait (parameters only);
//   * the MMA warp issues SS-mode tcgen05.mma (A = weight image, B = the TR-row activation image, both in shared
//     memory) into one of TWO accumulator sets, releases ring slots / activation images through tcgen05.commit;
//   * eight EPILOGUE warps load activation tiles, read the accumulators back (transposed through shared memory) and
//     run the row-wise epilogues of chain_tc.cu; the output of a step is written (raw + lo) as the operand image of
//     the next one.  Steps that share their input image (W1 | W3 | Wq) overlap: the tensor core works on the next
//     product while the epilogue of the previous one drains.
//
// Every mbarrier wait is bounded (pipe_common.cuh: pipe_wait): a protocol error ends with SCANN_ERR_PIPE_TIMEOUT and the wait
// site in the caller's status words (the engine raises on it), not with a hang.
#include <string.h>

#include "pipe_common.cuh"

#define C2_EPI_WARPS 16
#define C2_EPI_THREADS (C2_EPI_WARPS * 32)
#define C2_THREADS (C2_EPI_THREADS + 128)    // + producer warp (16) + three MMA warps (17..19)
#define C2_MAX_STEPS 6
#define C2_MAX_BLOCKS 18
#define C2_NSLOT 4                           // ring slots of one K-block: [raw 16 KB | lo 16 KB]
#define C2_SLOT_BYTES 32768u
#define C2_WIMG_FLOATS 32768                 // floats of one weight image (one block, one orientation)

extern "C" int scann_device_sm_count(void);

// phase timestamps of CTA 0 (development builds, -DSCANN_DEV_PROBES): [0][..] epilogue thread 0: start, then per step
// {operand images ready, accumulators ready, read-back done, row epilogue done}; [1][..] MMA thread: per block
// {image + accumulator available, last ring slot landed, committed}
#ifdef SCANN_DEV_PROBES
__device__ long long g_c2_clk[3][64];
#define C2CLK(role, i) do { if (blockIdx.x == 0 && (i) < 64) g_c2_clk[role][i] = clock64(); } while (0)
extern "C" int scann_debug_clocks_chain2(long long* host_out192) {
    cudaError_t e = cudaMemcpyFromSymbol(host_out192, g_c2_clk, sizeof(long long) * 192);
    if (e != cudaSuccess) { scann_set_error("debug_clocks_chain2: %s", cudaGetErrorString(e)); return 1; }
    return 0;
}
#else
#define C2CLK(role, i) do { } while (0)
#endif

// Same field order as ChainStep of chain_tc.cu / ScannChainStep of include/scann_b200.h; W[kb] points to a weight IMAGE.
struct C2Step {
    const float* A[3];
    const float* W[3];
    const float* bias;
    const float* resid;
    const float* pre_in;
    float* pre_out;
    const float* gamma;
    const float* beta;
    float* dgamma;
    float* dbeta;
    float* C;
    float* C2;
    const int32_t* cnt;
    float* np_ctx;
    float* np_out;
    const ScannDropCtl* drop;
    int lda, ldres, ldpre, ldc, ldc2;
    int kblk;
    int mode;
    int to_image;
    int drop_site;
    int pad;
};
#define C2_FRESH 1u      // the block's activation image is a new one: wait for it
#define C2_RELEASE 2u    // last block that reads the current image: hand the buffer back once the MMAs are done
#define C2_FIRST 4u      // first block of a step: accumulators start from zero
#define C2_LAST 8u       // last block of a step: accumulators complete -> epilogue
struct C2Block { const float* wimg; uint32_t flags; uint32_t pad; };
struct C2Args {
    int nsteps, R, nblocks, pad;
    int32_t* status;        // engine status words (nullable): a wait that gives up sets SCANN_ERR_PIPE_TIMEOUT + its site (41..47)
    C2Step s[C2_MAX_STEPS];
    C2Block b[C2_MAX_BLOCKS];
};

// ---------------------------------------------------------------------------------------------------------------
// weight images
// ---------------------------------------------------------------------------------------------------------------
// images[blk][orient][kb][part][128 rows x 128 B]: part 0 = raw (low 13 mantissa bits cleared), part 1 = lo.
// orient 0: A[m][k] = W[k][m] (the GEMM x @ W with W[in,out]); orient 1: A[m][k] = W[m][k] (x @ W^T).
__global__ void __launch_bounds__(256) weight_images_kernel(const float* __restrict__ params, const int32_t* __restrict__ offsets,
                                                            float* __restrict__ images) {
    const float* W = params + (size_t)offsets[blockIdx.x];
    const int orient = blockIdx.y;
    uint8_t* img = reinterpret_cast<uint8_t*>(images + ((size_t)blockIdx.x * 2 + orient) * C2_WIMG_FLOATS);
    for (int i = threadIdx.x; i < 4 * 1024; i += 256) {
        // thread -> (row m, physical chunk ip) so that the global READS are coalesced in either orientation
        const int kb = i >> 10, idx = i & 1023;
        const int m = orient ? idx >> 3 : idx & 127, ip = orient ? idx & 7 : idx >> 7;
        const int c4 = kb * 8 + (ip ^ (m & 7));              // logical 16-byte chunk stored at physical position ip
        float v[4];
        if (orient) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(W + (size_t)m * SCANN_D + c4 * 4));
            v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) v[q] = __ldg(W + (size_t)(c4 * 4 + q) * SCANN_D + m);
        }
        float4 h, l;
        tf32_split(v[0], h.x, l.x); tf32_split(v[1], h.y, l.y); tf32_split(v[2], h.z, l.z); tf32_split(v[3], h.w, l.w);
        uint8_t* dst = img + (size_t)kb * C2_SLOT_BYTES + (size_t)m * 128 + ip * 16;
        *reinterpret_cast<float4*>(dst) = h;
        *reinterpret_cast<float4*>(dst + 16384) = l;
    }
}

extern "C" int scann_weight_images(const float* params, const int32_t* offsets, int nblocks, float* images, void* stream) {
    if (nblocks <= 0) return 0;
    weight_images_kernel<<<dim3(nblocks, 2), 256, 0, (cudaStream_t)stream>>>(params, offsets, images);
    return scann_check_launch("scann_weight_images");
}

// ---------------------------------------------------------------------------------------------------------------
// the chain
// ---------------------------------------------------------------------------------------------------------------
template <int TR>
struct C2Cfg {
    static constexpr int NXBUF = TR == 32 ? 2 : 1;                   // activation image pairs (raw + lo)
    static constexpr uint32_t CB = TR * 128u;                        // one chunk block [TR rows x 128 B]
    static constexpr uint32_t IMG = 4u * CB;                         // one image [TR rows x 128 fp32]
    static constexpr uint32_t OFF_X = C2_NSLOT * C2_SLOT_BYTES;      // after the weight ring
    static constexpr uint32_t OFF_S = OFF_X + NXBUF * 2u * IMG;
    static constexpr uint32_t OFF_BAR = OFF_S + IMG;                 // w_full[4] w_empty[4] x_full[2] x_empty[2] acc_full[2] acc_empty[2]
    static constexpr uint32_t OFF_MISC = OFF_BAR + 16u * 8u;         // tmem slot, dead flag, copy of the kernel arguments
    static constexpr uint32_t SMEM = OFF_MISC + 16u + (uint32_t)sizeof(C2Args) + 1024u;   // + alignment slack
    static constexpr int RPW = TR / C2_EPI_WARPS;                    // rows per epilogue warp
    static constexpr int STEPS = RPW / 2;                            // 2-row passes per epilogue warp
    static constexpr int XIT = TR * 32 / C2_EPI_THREADS;             // 16-byte chunks per thread of one activation tile
    static constexpr uint32_t TCOLS = TR == 32 ? 256u : 512u;        // two accumulator sets of four x TR columns
};
template <int TR> __device__ __forceinline__ uint32_t c2_off4(int r, int c4) {
    return (uint32_t)(c4 >> 3) * C2Cfg<TR>::CB + (uint32_t)r * 128u + ((((uint32_t)c4 & 7u) ^ ((uint32_t)r & 7u)) << 4);
}
template <int TR> __device__ __forceinline__ uint32_t c2_off(int r, int c) { return c2_off4<TR>(r, c >> 2) + ((uint32_t)c & 3u) * 4u; }

__device__ __forceinline__ void c2_epi_sync() { asm volatile("bar.sync 1, %0;" ::"n"(C2_EPI_THREADS) : "memory"); }
__device__ __forceinline__ void hex_sum2(float& a, float& b) {      // sums over the 16 lanes of a row
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
}
__device__ __forceinline__ float4 c2_lo4(float4 v) {
    return make_float4(v.x - __uint_as_float(__float_as_uint(v.x) & 0xffffe000u), v.y - __uint_as_float(__float_as_uint(v.y) & 0xffffe000u),
                       v.z - __uint_as_float(__float_as_uint(v.z) & 0xffffe000u), v.w - __uint_as_float(__float_as_uint(v.w) & 0xffffe000u));
}
// drop_mult (common.cuh) on a control block that already sits in registers
__device__ __forceinline__ float c2_drop(const ScannDropCtl& c, uint32_t site, uint32_t idx) {
    return drop_hash(c.seed, site, idx) >= c.threshold ? __uint_as_float(c.scale_bits) : 0.0f;
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

// DET (deterministic mode, DESIGN.md section 4.7): the LayerNorm-backward column sums of a CTA are stored into its slot
// (dgamma / dbeta point to [grid][128] slot arrays) instead of being added into the gradient arena.
template <int TR, bool DET>
__global__ void __launch_bounds__(C2_THREADS, 1) dense_chain2_kernel(const __grid_constant__ C2Args ga) {
    typedef C2Cfg<TR> K;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* ring = smem;
    uint8_t* sX = smem + K::OFF_X;
    uint8_t* sS = smem + K::OFF_S;
    uint64_t* w_full = reinterpret_cast<uint64_t*>(smem + K::OFF_BAR);
    uint64_t *w_empty = w_full + 4, *x_full = w_full + 8, *x_empty = w_full + 10, *acc_full = w_full + 12, *acc_empty = w_full + 14;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + K::OFF_MISC);
    volatile int* dead = reinterpret_cast<volatile int*>(smem + K::OFF_MISC + 4);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int r0 = blockIdx.x * TR;
    // The step / block tables are read from a shared-memory copy: a step's fields indexed by the runtime step number
    // out of the constant bank cost a constant-cache miss (several hundred cycles) at every first touch, in the
    // middle of the row-wise epilogues
    const C2Args& a = *reinterpret_cast<const C2Args*>(smem + K::OFF_MISC + 16);
    {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(&ga);
        uint32_t* dst = reinterpret_cast<uint32_t*>(smem + K::OFF_MISC + 16);
        for (int i = tid; i < (int)(sizeof(C2Args) / 4); i += C2_THREADS) dst[i] = src[i];
    }
    if (warp == C2_EPI_WARPS) tmem_alloc(tmem_slot, K::TCOLS);
    if (tid == 0) {
        for (int i = 0; i < 4; ++i) { mbar_init(&w_full[i], 1); mbar_init(&w_empty[i], 3); }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&x_full[i], 1); mbar_init(&x_empty[i], 3); mbar_init(&acc_full[i], 3); mbar_init(&acc_empty[i], 1);
        }
        *dead = 0;
        mbar_fence_init();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == C2_EPI_WARPS) {
        // =========================================================== producer: weight images -> ring (slot = K-block)
        if (lane == 0) {
            for (int bi = 0; bi < a.nblocks; ++bi) {
                const uint8_t* src = reinterpret_cast<const uint8_t*>(a.b[bi].wimg);
#pragma unroll
                for (int kb = 0; kb < 4; ++kb) {
                    pipe_wait(&w_empty[kb], ((uint32_t)bi & 1u) ^ 1u, dead, a.status, 41, bi, kb);
                    mbar_expect_tx(&w_full[kb], C2_SLOT_BYTES);
                    bulk_load(ring + (size_t)kb * C2_SLOT_BYTES, src + (size_t)kb * C2_SLOT_BYTES, C2_SLOT_BYTES, &w_full[kb]);
                }
            }
        }
        __syncwarp();
        pdl_wait();
    } else if (warp > C2_EPI_WARPS) {
        // =========================================================== MMA issue: one product of 3xTF32 per warp
        // chain 0: W_lo X_raw, chain 1: W_raw X_lo, chain 2: W_raw X_raw -- each into its own accumulator columns
        const int chain = warp - C2_EPI_WARPS - 1;
        if (tc_elect_one()) {
            const uint32_t idesc = tc_idesc_tf32(128, TR, false, false);
            const uint32_t ring_a = smem_u32(ring) + (chain == 0 ? 16384u : 0u);
            int xi = -1, ai = 0;
            for (int bi = 0; bi < a.nblocks; ++bi) {
                const uint32_t fl = a.b[bi].flags;
                if (fl & C2_FRESH) {
                    ++xi;
                    pipe_wait(&x_full[xi % K::NXBUF], ((uint32_t)(xi / K::NXBUF)) & 1u, dead, a.status, 42, bi, xi);
                }
                if (fl & C2_FIRST) pipe_wait(&acc_empty[ai & 1], (((uint32_t)(ai >> 1)) & 1u) ^ 1u, dead, a.status, 43, bi, ai);
                if (chain == 2) C2CLK(1, bi * 3);
                // accumulator set: [W_lo X_raw | W_raw X_lo | main, K-blocks 0-1 | main, K-blocks 2-3].  The tensor core's
                // accumulate loses low-order bits of what it adds to a large accumulator (profiles/r01_tcgen05_probe.md);
                // two shorter main chains, added in fp32 by the epilogue, halve that loss
                const uint32_t t_acc = tmem + (uint32_t)(ai & 1) * 4u * TR + (uint32_t)chain * TR;
                const uint32_t ximg = smem_u32(sX + (size_t)(xi % K::NXBUF) * 2u * K::IMG) + (chain == 1 ? K::IMG : 0u);
#pragma unroll
                for (int kb = 0; kb < 4; ++kb) {
                    pipe_wait(&w_full[kb], (uint32_t)bi & 1u, dead, a.status, 44, bi, kb);
                    tc_fence_after();
                    if (kb == 3 && chain == 2) C2CLK(1, bi * 3 + 1);
                    const uint64_t da = pt_desc(ring_a + kb * C2_SLOT_BYTES), db = pt_desc(ximg + kb * K::CB);
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)
                        tc_mma_ss(t_acc + ((chain == 2 && kb >= 2) ? TR : 0), da + 2 * ks, db + 2 * ks, idesc,
                                  !((fl & C2_FIRST) && ks == 0 && (kb == 0 || (chain == 2 && kb == 2))));
                    tc_commit(&w_empty[kb]);
                }
                if (fl & C2_RELEASE) tc_commit(&x_empty[xi % K::NXBUF]);
                if (fl & C2_LAST) { tc_commit(&acc_full[ai & 1]); ++ai; }
                if (chain == 2) C2CLK(1, bi * 3 + 2);
            }
        }
        __syncwarp();
        pdl_wait();
    } else {
        // =========================================================== epilogue warps: 16 lanes per row, 8 columns per lane
        const int l16 = lane & 15, rsub = lane >> 4;
        const int q = warp & 3, part = warp >> 2;
        const uint32_t lane_base = (uint32_t)(q * 32) << 16;
        int xi = -1, ai = 0;
        pdl_wait();
        if (tid == 0) C2CLK(0, 0);
#pragma unroll 1
        for (int si = 0; si < a.nsteps; ++si) {
            const C2Step& st = a.s[si];
            // ---- activation tiles that come from global memory -> operand images (raw as loaded, lo = x - trunc(x))
#pragma unroll 1
            for (int kb = 0; kb < st.kblk; ++kb) {
                const float* A = st.A[kb];
                if (!A) break;
                ++xi;
                float4 xv[K::XIT];
#pragma unroll
                for (int it = 0; it < K::XIT; ++it) {
                    const int i = tid + it * C2_EPI_THREADS, r = i >> 5, c4 = i & 31;
                    xv[it] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (r0 + r < a.R) xv[it] = ld4(A + (size_t)(r0 + r) * st.lda + c4 * 4);
                }
                pipe_wait(&x_empty[xi % K::NXBUF], (((uint32_t)(xi / K::NXBUF)) & 1u) ^ 1u, dead, a.status, 45, si, xi);
                uint8_t* Xr = sX + (size_t)(xi % K::NXBUF) * 2u * K::IMG;
#pragma unroll
                for (int it = 0; it < K::XIT; ++it) {
                    const int i = tid + it * C2_EPI_THREADS, r = i >> 5, c4 = i & 31;
                    const uint32_t off = c2_off4<TR>(r, c4);
                    *reinterpret_cast<float4*>(Xr + off) = xv[it];
                    *reinterpret_cast<float4*>(Xr + K::IMG + off) = c2_lo4(xv[it]);
                }
                fence_async_smem();
                c2_epi_sync();
                if (tid == 0) mbar_arrive(&x_full[xi % K::NXBUF]);
            }
            if (tid == 0) C2CLK(0, 1 + si * 4);
            // ---- parameters and the first rows of the epilogue: in flight behind the MMA
            float4 bias[2], gam[2], bet[2];
#pragma unroll
            for (int it = 0; it < 2; ++it) {
                const int c0 = (l16 + 16 * it) * 4;
                bias[it] = st.bias ? ldg4(st.bias + c0) : make_float4(0.f, 0.f, 0.f, 0.f);
                gam[it] = st.gamma ? ldg4(st.gamma + c0) : bias[it];
                bet[it] = st.beta ? ldg4(st.beta + c0) : bias[it];
            }
            // dropout control block (device memory) and the neighbour count of the first row: fetched now, used after the MMA
            ScannDropCtl dctl = {0u, 0u, 0u, 0u};
            if (st.drop) dctl = *st.drop;
            int cnt0 = 1;
            if (st.cnt && r0 + warp * K::RPW + rsub < a.R) cnt0 = st.cnt[r0 + warp * K::RPW + rsub];
            float4 rv0[2], pv0[2];
            {
                const int r = r0 + warp * K::RPW + rsub;
#pragma unroll
                for (int it = 0; it < 2; ++it) {
                    rv0[it] = make_float4(0.f, 0.f, 0.f, 0.f);
                    pv0[it] = rv0[it];
                    if (r < a.R) {
                        if (st.resid) rv0[it] = ld4(st.resid + (size_t)r * st.ldres + (l16 + 16 * it) * 4);
                        if (st.mode == 2 || st.mode == 4) pv0[it] = ld4(st.pre_in + (size_t)r * st.ldpre + (l16 + 16 * it) * 4);
                    }
                }
            }
            pipe_wait(&acc_full[ai & 1], ((uint32_t)(ai >> 1)) & 1u, dead, a.status, 46, si, ai);
            tc_fence_after();
            if (tid == 0) C2CLK(0, 2 + si * 4);
            if (si == a.nsteps - 1) pdl_trigger();      // only the last epilogue is left
            // ---- epilogue 1: D^T (lane = feature, column = row) -> S[r][n]: the two correction products, then the main one
            {
                const int n = q * 32 + lane;
                const uint32_t t_acc = tmem + (uint32_t)(ai & 1) * 4u * TR + lane_base + (uint32_t)part * (TR / 4);
                if (TR == 32) {
                    float c0[8], c1[8], m0[8], m1[8];
                    tmem_ld8(t_acc, c0);
                    tmem_ld8(t_acc + TR, c1);
                    tmem_ld8(t_acc + 2 * TR, m0);
                    tmem_ld8(t_acc + 3 * TR, m1);
                    tmem_ld_wait();
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        *reinterpret_cast<float*>(sS + c2_off<TR>(part * 8 + k, n)) = (c0[k] + c1[k]) + (m0[k] + m1[k]);
                } else {
                    float c0[16], c1[16], m0[16], m1[16];
                    tmem_ld16(t_acc, c0);
                    tmem_ld16(t_acc + TR, c1);
                    tmem_ld16(t_acc + 2 * TR, m0);
                    tmem_ld16(t_acc + 3 * TR, m1);
                    tmem_ld_wait();
#pragma unroll
                    for (int k = 0; k < 16; ++k)
                        *reinterpret_cast<float*>(sS + c2_off<TR>(part * 16 + k, n)) = (c0[k] + c1[k]) + (m0[k] + m1[k]);
                }
            }
            tc_fence_before();
            c2_epi_sync();
            if (tid == 0) mbar_arrive(&acc_empty[ai & 1]);
            ++ai;
            if (tid == 0) C2CLK(0, 3 + si * 4);
            // ---- epilogue 2: row groups (16 lanes per row, 8 columns per lane) -- the arithmetic of chain_tc.cu
            const int mode = st.mode;
            const bool to_image = st.to_image != 0;
            uint8_t* Xn = nullptr;
            if (to_image) {
                ++xi;
                pipe_wait(&x_empty[xi % K::NXBUF], (((uint32_t)(xi / K::NXBUF)) & 1u) ^ 1u, dead, a.status, 47, si, xi);
                Xn = sX + (size_t)(xi % K::NXBUF) * 2u * K::IMG;
            }
            float dgam[2][4], dbet[2][4];
#pragma unroll
            for (int it = 0; it < 2; ++it)
#pragma unroll
                for (int k = 0; k < 4; ++k) { dgam[it][k] = 0.f; dbet[it][k] = 0.f; }
            if (tid == 0) C2CLK(2, si * 6);
#pragma unroll 1
            for (int step = 0; step < K::STEPS; ++step) {
                const int rr = warp * K::RPW + step * 2 + rsub, r = r0 + rr;
                const bool ok = r < a.R;
                float v[2][4];
#pragma unroll
                for (int it = 0; it < 2; ++it) {
                    const int c4 = l16 + 16 * it, c0 = c4 * 4;
                    const float4 acc = *reinterpret_cast<const float4*>(sS + c2_off4<TR>(rr, c4));
                    float4 rv = rv0[it];
                    if (step > 0) {
                        rv = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (st.resid && ok) rv = ld4(st.resid + (size_t)r * st.ldres + c0);
                    }
                    float d0 = 1.f, d1 = 1.f, d2 = 1.f, d3 = 1.f;
                    if (dctl.enabled && mode != 4) {
                        const uint32_t idx = (uint32_t)r * SCANN_D + c0;
                        d0 = c2_drop(dctl, st.drop_site, idx); d1 = c2_drop(dctl, st.drop_site, idx + 1);
                        d2 = c2_drop(dctl, st.drop_site, idx + 2); d3 = c2_drop(dctl, st.drop_site, idx + 3);
                    }
                    v[it][0] = (acc.x + bias[it].x) * d0 + rv.x; v[it][1] = (acc.y + bias[it].y) * d1 + rv.y;
                    v[it][2] = (acc.z + bias[it].z) * d2 + rv.z; v[it][3] = (acc.w + bias[it].w) * d3 + rv.w;
                }
                if (tid == 0) C2CLK(2, si * 6 + 1);
                if (mode == 1) {
#pragma unroll
                    for (int it = 0; it < 2; ++it) {
                        if (st.pre_out && ok)
                            st4(st.pre_out + (size_t)r * st.ldpre + (l16 + 16 * it) * 4,
                                make_float4(v[it][0], v[it][1], v[it][2], v[it][3]));
#pragma unroll
                        for (int k = 0; k < 4; ++k) v[it][k] = swish_fast(v[it][k]);
                    }
                } else if (mode == 2) {
#pragma unroll
                    for (int it = 0; it < 2; ++it) {
                        float4 p = pv0[it];
                        if (step > 0) {
                            p = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (ok) p = ld4(st.pre_in + (size_t)r * st.ldpre + (l16 + 16 * it) * 4);
                        }
                        v[it][0] *= swish_grad_fast(p.x); v[it][1] *= swish_grad_fast(p.y);
                        v[it][2] *= swish_grad_fast(p.z); v[it][3] *= swish_grad_fast(p.w);
                    }
                } else if (mode == 3) {
                    float s1 = 0.f;
#pragma unroll
                    for (int it = 0; it < 2; ++it) {
                        if (st.pre_out && ok)
                            st4(st.pre_out + (size_t)r * st.ldpre + (l16 + 16 * it) * 4,
                                make_float4(v[it][0], v[it][1], v[it][2], v[it][3]));
                        s1 += v[it][0] + v[it][1] + v[it][2] + v[it][3];
                    }
                    // shifted one-pass moments: shift = mean of the 8 columns of the row's first lane
                    const float sh = __shfl_sync(0xffffffffu, s1, lane & 16) * (1.0f / 8.0f);
                    float m1 = 0.f, m2 = 0.f;
#pragma unroll
                    for (int it = 0; it < 2; ++it)
#pragma unroll
                        for (int k = 0; k < 4; ++k) { v[it][k] -= sh; m1 += v[it][k]; m2 = fmaf(v[it][k], v[it][k], m2); }
                    hex_sum2(m1, m2);
                    m1 *= (1.0f / SCANN_D);
                    const float inv = rsqrtf(fmaxf(m2 * (1.0f / SCANN_D) - m1 * m1, 0.f) + SCANN_LN_EPS);
#pragma unroll
                    for (int it = 0; it < 2; ++it) {
                        v[it][0] = (v[it][0] - m1) * inv * gam[it].x + bet[it].x;
                        v[it][1] = (v[it][1] - m1) * inv * gam[it].y + bet[it].y;
                        v[it][2] = (v[it][2] - m1) * inv * gam[it].z + bet[it].z;
                        v[it][3] = (v[it][3] - m1) * inv * gam[it].w + bet[it].w;
                    }
                } else if (mode == 4) {
                    // LayerNorm backward: v = upstream gradient dy, pre_in = forward pre-LN value
                    float x[2][4];
                    float s1 = 0.f;
#pragma unroll
                    for (int it = 0; it < 2; ++it) {
                        float4 p = pv0[it];
                        if (step > 0) {
                            p = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (ok) p = ld4(st.pre_in + (size_t)r * st.ldpre + (l16 + 16 * it) * 4);
                        }
                        x[it][0] = p.x; x[it][1] = p.y; x[it][2] = p.z; x[it][3] = p.w;
                        s1 += p.x + p.y + p.z + p.w;
                    }
                    float d0 = 0.f;
                    hex_sum2(s1, d0);
                    const float mean = s1 * (1.0f / SCANN_D);
                    float var = 0.f, dummy = 0.f;
#pragma unroll
                    for (int it = 0; it < 2; ++it)
#pragma unroll
                        for (int k = 0; k < 4; ++k) { x[it][k] -= mean; var = fmaf(x[it][k], x[it][k], var); }
                    hex_sum2(var, dummy);
                    const float inv = rsqrtf(var * (1.0f / SCANN_D) + SCANN_LN_EPS);
                    const float g[2][4] = {{gam[0].x, gam[0].y, gam[0].z, gam[0].w}, {gam[1].x, gam[1].y, gam[1].z, gam[1].w}};
                    float t1 = 0.f, t2 = 0.f;
#pragma unroll
                    for (int it = 0; it < 2; ++it)
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            x[it][k] *= inv;                                    // x_hat
                            const float dy = ok ? v[it][k] : 0.f;
                            dgam[it][k] = fmaf(dy, x[it][k], dgam[it][k]);
                            dbet[it][k] += dy;
                            v[it][k] = dy * g[it][k];                           // d x_hat
                            t1 += v[it][k];
                            t2 = fmaf(v[it][k], x[it][k], t2);
                        }
                    hex_sum2(t1, t2);
                    t1 *= (1.0f / SCANN_D);
                    t2 *= (1.0f / SCANN_D);
#pragma unroll
                    for (int it = 0; it < 2; ++it)
#pragma unroll
                        for (int k = 0; k < 4; ++k) v[it][k] = inv * (v[it][k] - t1 - x[it][k] * t2);
                }
                if (tid == 0) C2CLK(2, si * 6 + 2);
                if (ok && st.C) {
#pragma unroll
                    for (int it = 0; it < 2; ++it)
                        st4(st.C + (size_t)r * st.ldc + (l16 + 16 * it) * 4, make_float4(v[it][0], v[it][1], v[it][2], v[it][3]));
                }
                if (mode == 4 && dctl.enabled) {
                    // gradient through the dropout that follows the Dense of the next (transposed) step
#pragma unroll
                    for (int it = 0; it < 2; ++it) {
                        const uint32_t idx = (uint32_t)r * SCANN_D + (l16 + 16 * it) * 4;
#pragma unroll
                        for (int k = 0; k < 4; ++k) v[it][k] *= c2_drop(dctl, st.drop_site, idx + k);
                    }
                }
                if (ok && st.C2) {
#pragma unroll
                    for (int it = 0; it < 2; ++it)
                        st4(st.C2 + (size_t)r * st.ldc2 + (l16 + 16 * it) * 4, make_float4(v[it][0], v[it][1], v[it][2], v[it][3]));
                }
                if (to_image) {
#pragma unroll
                    for (int it = 0; it < 2; ++it) {
                        const float4 o = make_float4(ok ? v[it][0] : 0.f, ok ? v[it][1] : 0.f, ok ? v[it][2] : 0.f, ok ? v[it][3] : 0.f);
                        const uint32_t off = c2_off4<TR>(rr, l16 + 16 * it);
                        *reinterpret_cast<float4*>(Xn + off) = o;
                        *reinterpret_cast<float4*>(Xn + K::IMG + off) = c2_lo4(o);
                    }
                }
                if (tid == 0) C2CLK(2, si * 6 + 3);
                if (st.cnt) {
                    // atoms without a valid neighbour: context = q, out = LayerNorm(q)   (attention.py:206-214)
                    const bool nop = ok && (step == 0 ? cnt0 : st.cnt[r]) == 0;
                    if (__any_sync(0xffffffffu, nop)) {
                        float m1 = 0.f, m2 = 0.f;
#pragma unroll
                        for (int it = 0; it < 2; ++it)
#pragma unroll
                            for (int k = 0; k < 4; ++k) m1 += v[it][k];
                        hex_sum2(m1, m2);
                        m1 *= (1.0f / SCANN_D);
                        float dd = 0.f;
#pragma unroll
                        for (int it = 0; it < 2; ++it)
#pragma unroll
                            for (int k = 0; k < 4; ++k) { const float d = v[it][k] - m1; m2 = fmaf(d, d, m2); }
                        hex_sum2(m2, dd);
                        const float inv = rsqrtf(m2 * (1.0f / SCANN_D) + SCANN_LN_EPS);
                        if (nop) {
#pragma unroll
                            for (int it = 0; it < 2; ++it) {
                                const int c0 = (l16 + 16 * it) * 4;
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
            if (tid == 0) C2CLK(2, si * 6 + 4);
            if (to_image) fence_async_smem();
            if (mode == 4) {
                // column sums over this CTA's rows without atomics: the two rows of a pass are added by a shuffle, every
                // warp leaves its 2 x 128 partial sums in the S bytes of its OWN rows (already consumed), then 256
                // threads add the 16 partials and issue one global reduction each
                __syncwarp();
#pragma unroll
                for (int it = 0; it < 2; ++it) {
                    float4 dg, db;
                    dg.x = dgam[it][0] + __shfl_xor_sync(0xffffffffu, dgam[it][0], 16); dg.y = dgam[it][1] + __shfl_xor_sync(0xffffffffu, dgam[it][1], 16);
                    dg.z = dgam[it][2] + __shfl_xor_sync(0xffffffffu, dgam[it][2], 16); dg.w = dgam[it][3] + __shfl_xor_sync(0xffffffffu, dgam[it][3], 16);
                    db.x = dbet[it][0] + __shfl_xor_sync(0xffffffffu, dbet[it][0], 16); db.y = dbet[it][1] + __shfl_xor_sync(0xffffffffu, dbet[it][1], 16);
                    db.z = dbet[it][2] + __shfl_xor_sync(0xffffffffu, dbet[it][2], 16); db.w = dbet[it][3] + __shfl_xor_sync(0xffffffffu, dbet[it][3], 16);
                    if (rsub == 0) {
                        uint8_t* base = sS + (size_t)warp * K::RPW * 128u + l16 * 16u;
                        *reinterpret_cast<float4*>(base + (size_t)it * K::CB) = dg;            // column p = 64 it + 4 l16
                        *reinterpret_cast<float4*>(base + (size_t)(2 + it) * K::CB) = db;
                    }
                }
                c2_epi_sync();
                if (tid < 2 * SCANN_D) {
                    const int p = tid & 127, which = tid >> 7;             // which: 0 dgamma, 1 dbeta
                    const uint8_t* base = sS + (size_t)(2 * which + (p >> 6)) * K::CB + (p & 63) * 4u;
                    float sum = 0.f;
#pragma unroll
                    for (int w = 0; w < C2_EPI_WARPS; ++w) sum += *reinterpret_cast<const float*>(base + (size_t)w * K::RPW * 128u);
                    if constexpr (DET) (which ? st.dbeta : st.dgamma)[(size_t)blockIdx.x * SCANN_D + p] = sum;
                    else atomicAdd((which ? st.dbeta : st.dgamma) + p, sum);
                }
            }
            if (tid == 0) C2CLK(2, si * 6 + 5);
            c2_epi_sync();        // S is rewritten by the next step; the new image is complete
            if (to_image && tid == 0) mbar_arrive(&x_full[xi % K::NXBUF]);
            if (tid == 0) C2CLK(0, 4 + si * 4);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == C2_EPI_WARPS) tmem_dealloc(tmem, K::TCOLS);
}

template <int TR, bool DET>
static int chain2_launch(const C2Args& a, void* stream) {
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(dense_chain2_kernel<TR, DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C2Cfg<TR>::SMEM);
        if (e != cudaSuccess) { scann_set_error("dense_chain2: smem opt-in failed: %s", cudaGetErrorString(e)); return 1; }
        configured = true;
    }
    scann_launch(dense_chain2_kernel<TR, DET>, dim3((a.R + TR - 1) / TR), dim3(C2_THREADS), (size_t)C2Cfg<TR>::SMEM, stream, a);
    return scann_check_launch("scann_dense_chain2");
}

// Rows that one wave of the warp-specialised form covers (one CTA per SM, 64-row tiles); more rows run in several waves.
extern "C" int scann_dense_chain2_max_rows(void) {
    static int sms = 0;
    if (sms == 0) sms = scann_device_sm_count();
    return sms * 64;
}

// Same contract as scann_dense_chain, except that W[kb] of every step points to the weight IMAGE of the block
// (scann_weight_images; orientation 0 for x @ W, 1 for x @ W^T).
template <bool DET>
static int chain2_run(const void* steps_host, int nsteps, int R, int32_t* status, void* stream) {
    if (nsteps < 1 || nsteps > C2_MAX_STEPS) { scann_set_error("dense_chain2: nsteps must be in 1..%d", C2_MAX_STEPS); return 1; }
    if (R <= 0) return 0;
    static_assert(sizeof(C2Args) <= 4096, "kernel parameter space");
    C2Args a;
    memset(&a, 0, sizeof(a));
    a.nsteps = nsteps;
    a.R = R;
    a.status = status;
    const C2Step* s = (const C2Step*)steps_host;
    int nb = 0;
    for (int i = 0; i < nsteps; ++i) {
        a.s[i] = s[i];
        C2Step& t = a.s[i];
        if (t.kblk < 1 || t.kblk > 3 || t.mode < 0 || t.mode > 4) { scann_set_error("dense_chain2: step %d: bad kblk/mode", i); return 1; }
        if (!t.A[0] && i == 0) { scann_set_error("dense_chain2: step 0 has no input"); return 1; }
        if (!t.A[0] && t.kblk != 1) { scann_set_error("dense_chain2: step %d: an image operand needs kblk == 1", i); return 1; }
        for (int kb = 0; kb < t.kblk; ++kb)
            if (!t.W[kb] || (kb > 0 && !t.A[kb])) { scann_set_error("dense_chain2: step %d: missing operand %d", i, kb); return 1; }
        if (((uintptr_t)t.W[0] | (uintptr_t)t.W[1] | (uintptr_t)t.W[2]) & 1023) { scann_set_error("dense_chain2: step %d: weight images must be 1024-byte aligned", i); return 1; }
        if ((t.mode == 2 || t.mode == 4) && !t.pre_in) { scann_set_error("dense_chain2: step %d: mode needs pre_in", i); return 1; }
        if ((t.mode == 3 || t.mode == 4) && !t.gamma) { scann_set_error("dense_chain2: step %d: mode needs gamma", i); return 1; }
        if (t.mode == 3 && !t.beta) { scann_set_error("dense_chain2: step %d: LayerNorm needs beta", i); return 1; }
        if (t.mode == 4 && (!t.dgamma || !t.dbeta)) { scann_set_error("dense_chain2: step %d: LayerNorm backward needs dgamma/dbeta", i); return 1; }
        if (t.cnt && (!t.np_out || !t.gamma || !t.beta)) { scann_set_error("dense_chain2: step %d: no-pair fix-up needs np_out/gamma/beta", i); return 1; }
        // an image is only produced for a consumer: the next step must read the resident image
        if (t.to_image && !(i + 1 < nsteps && !s[i + 1].A[0])) t.to_image = 0;
        for (int kb = 0; kb < t.kblk; ++kb, ++nb) {
            uint32_t fl = 0;
            if (t.A[kb] || (kb == 0 && i > 0 && a.s[i - 1].to_image)) fl |= C2_FRESH;
            if (kb == 0) fl |= C2_FIRST;
            if (kb == t.kblk - 1) fl |= C2_LAST;
            a.b[nb].wimg = t.W[kb];
            a.b[nb].flags = fl;
        }
    }
    // a block releases the current image when the next block brings a fresh one (or nothing follows)
    for (int i = 0; i < nb; ++i)
        if (i + 1 == nb || (a.b[i + 1].flags & C2_FRESH)) a.b[i].flags |= C2_RELEASE;
    a.nblocks = nb;
    static int sms = 0;
    if (sms == 0) sms = scann_device_sm_count();
    if ((R + 31) / 32 <= sms) return chain2_launch<32, DET>(a, stream);
    return chain2_launch<64, DET>(a, stream);
}

extern "C" int scann_dense_chain2(const void* steps_host, int nsteps, int R, int32_t* status, void* stream) {
    return chain2_run<false>(steps_host, nsteps, R, status, stream);
}

// Deterministic form: dgamma / dbeta of every mode-4 step are [scann_dense_chain2_grid(R)][128] slot arrays.
extern "C" int scann_dense_chain2_det(const void* steps_host, int nsteps, int R, int32_t* status, void* stream) {
    return chain2_run<true>(steps_host, nsteps, R, status, stream);
}

// CTAs of one scann_dense_chain2 launch over R rows (32-row tiles while they fit one wave, else 64-row tiles).
extern "C" int scann_dense_chain2_grid(int R) {
    static int sms = 0;
    if (sms == 0) sms = scann_device_sm_count();
    if (R <= 0) return 0;
    return (R + 31) / 32 <= sms ? (R + 31) / 32 : (R + 63) / 64;
}
