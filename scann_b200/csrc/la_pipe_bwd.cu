// Local attention backward (g_update = True) as two warp-specialised, TMA-fed pipelines per layer -- the backward
// counterpart of la_pipe.cu, same frame (pipe_frame.cuh), same arithmetic as la_tc_bwd.cu (SURVEY.md appendix A):
//
//   la_attn_bwd_pipe : softmax / context backward, d_k, d_q ; d_a = d_k @ Wk^T (3xTF32) ;
//                      d_nbr = d_a * g' scattered to dx[j] ; dg' (+)= d_a * x[j]
//   la_geom_bwd_pipe : LN_g backward, d_pre ; dg = d_z + d_pre @ W2^T (3xTF32) ; s_pre, t scatter
//
// A stage of the ring holds FOUR tile images (three stages per SM):
//   attention : keys k (TMA) -> d_k in place (hi operand, stored back over k for the weight-gradient launch) |
//               lo(d_k) -> transposed accumulator d_a | g' (TMA) | x[j] (cp.async gather) -> d_a * x[j] in place, which
//               leaves through a TMA store -- or a TMA reduce-add when the layer above already left its gradient in dg
//   geometry  : pre-activation (TMA) -> d_pre in place (hi operand, stored back over pre) | lo(d_pre) -> accumulator ->
//               dg in place | g (TMA) | dg' (TMA)
// Row mapping of the CUDA-core phases: warp w of a group owns rows w, w + 8, w + 16, w + 24 of the tile, lane l the
// 16-byte chunk l of the row (columns 4l..4l+3; an attention head = 4 adjacent lanes).
#include <string.h>

#include "pipe_frame.cuh"

#define PB_NS 3
typedef PipeFrame<PB_NS, 4> BwdFrame;
#define PB_STAGE (BwdFrame::STAGE)
#define PB_SMEM (BwdFrame::SMEM)

// phase timestamps of CTA 0, consumer group 0 (development builds: -DSCANN_DEV_PROBES): [kernel][tile ordinal][phase]
#ifdef SCANN_DEV_PROBES
__device__ long long g_pipe_clk_bwd[2][4][12];
#define BCLK(k, ph) do { if (blockIdx.x == 0 && tid == 0 && (i / PF_NG) < 4) g_pipe_clk_bwd[k][i / PF_NG][ph] = clock64(); } while (0)
extern "C" int scann_pipe_clocks_bwd(long long* host_out96) {
    cudaError_t e = cudaMemcpyFromSymbol(host_out96, g_pipe_clk_bwd, sizeof(long long) * 96);
    if (e != cudaSuccess) { scann_set_error("pipe_clocks_bwd: %s", cudaGetErrorString(e)); return 1; }
    return 0;
}
#else
#define BCLK(k, ph) do { } while (0)
#endif

__device__ __forceinline__ float dot4(float4 a, float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }

// =============================================================================================
// Attention backward
// =============================================================================================
struct PipeAttnBwdArgs {
    CUtensorMap tm_k, tm_g, tm_dg;
    const int32_t* ntiles; const int32_t* pair_c; const int32_t* pair_j;
    const float* x;          // [R,128]
    const float* proj;       // [R,384]; q = columns 256..383
    const float* WkT;        // transposed key kernel: WkT[n][ka] = Wk[ka][n]
    const float* d_ctx;      // [R,128]
    float* dq;               // [R,128] <- d_ctx + 0.25 sum_n de k   (atoms with pairs)
    float* dx_scatter;       // [R,128] += d_a * g' at the neighbour rows
    float* dbk;              // [128]   += column sums of d_k
    int dg_accum;            // dg already holds the gradient from the layer above: reduce-add instead of store
    const ScannDropCtl* drop; int drop_site;
    int32_t* status;
};

// Deterministic instantiations (DET = true, DESIGN.md section 4.7): d_a * g' is STORED at its pair row of dx_scatter
// (a [rows,128] per-pair buffer; scann_row_gather sums it per atom row afterwards) instead of being added at the
// neighbour row, and the column sums leave the CTA as one plain store per CTA slot (dbk: [grid][128]; dgamma_g /
// dbeta_g: [grid][256], gamma then beta) after the consumer warps have combined their partials in warp order.
// Geometry: t_scatter is not written at all -- d_pre stays per pair in the pre-activation buffer.
__device__ __forceinline__ void pb_consumer_sync() { asm volatile("bar.sync 14, %0;" ::"n"(PF_CW * 32) : "memory"); }

template <bool DET>
__global__ void __launch_bounds__(PF_THREADS, 1) la_attn_bwd_pipe_kernel(const __grid_constant__ PipeAttnBwdArgs a) {
    __shared__ float s_dbk[SCANN_D];
    if (threadIdx.x < SCANN_D) s_dbk[threadIdx.x] = 0.f;
    // stationary operand A[M = ka][K = n] = Wk[ka][n] (= transpose of WkT, loaded coalesced)
    PF_PROLOGUE(BwdFrame, PB_NS, a.WkT, 33)
    if (warp == PF_CW) {
        // ================= producer: k and g' tiles by TMA, x[j] rows by per-lane cp.async =================
        if (lane == 0) { tma_prefetch_desc(&a.tm_k); tma_prefetch_desc(&a.tm_g); }
        int i = 0;
        int jn = 0;
        if ((int)blockIdx.x < nt) {
            const int pcv = a.pair_c[(size_t)blockIdx.x * PT + lane];
            jn = pcv >= 0 ? a.pair_j[(size_t)blockIdx.x * PT + lane] : 0;
        }
        for (int t = blockIdx.x; t < nt; t += gridDim.x, ++i) {
            const int s = i % PB_NS;
            const uint32_t ph = (uint32_t)(i / PB_NS) & 1u;
            const int j = jn;
            const int tn = t + (int)gridDim.x;
            if (tn < nt) {
                const int pcv = a.pair_c[(size_t)tn * PT + lane];
                jn = pcv >= 0 ? a.pair_j[(size_t)tn * PT + lane] : 0;
            }
            pipe_wait(&c.empty[s], ph ^ 1u, c.dead, a.status, 21, t, s);
            __syncwarp();
            uint8_t* S0 = c.stages + (size_t)s * PB_STAGE;
            if (lane == 0) {
                mbar_expect_tx(&c.full[s], 2u * PT_IMG + 256u);
#pragma unroll
                for (int kb = 0; kb < 4; ++kb) tma_load_2d(S0 + kb * PT_CB, &a.tm_k, kb * 32, t * PT, &c.full[s]);
#pragma unroll
                for (int kb = 0; kb < 4; ++kb) tma_load_2d(S0 + 2 * PT_IMG + kb * PT_CB, &a.tm_g, kb * 32, t * PT, &c.full[s]);
                bulk_load(c.idx + s * 64, a.pair_c + (size_t)t * PT, 128u, &c.full[s]);
                bulk_load(c.idx + s * 64 + 32, a.pair_j + (size_t)t * PT, 128u, &c.full[s]);
                // the ring is only PB_NS tiles deep: pull the tile behind it into L2 now
                const int tp = t + PB_NS * (int)gridDim.x;
                if (tp < nt) {
#pragma unroll
                    for (int kb = 0; kb < 4; ++kb) { tma_prefetch_2d(&a.tm_k, kb * 32, tp * PT); tma_prefetch_2d(&a.tm_g, kb * 32, tp * PT); }
                }
            }
            const uint32_t X = smem_u32(S0 + 3 * PT_IMG);
#pragma unroll 8
            for (int rr = 0; rr < PT; ++rr) {
                const int jr = __shfl_sync(0xffffffffu, j, rr);
                cp_async16(X + pt_off4(rr, lane), a.x + (size_t)jr * SCANN_D + lane * 4);
            }
            cp_async_arrive(&c.full[s]);
        }
    } else if (warp > PF_CW) {
        if (lane == 0) tma_prefetch_desc(&a.tm_dg);
        PF_STORE_LOOP(PB_NS, PB_STAGE, 22,
            for (int kb = 0; kb < 4; ++kb) tma_store_2d(&a.tm_k, A + kb * PT_CB, kb * 32, t * PT);
            if (a.dg_accum) { for (int kb = 0; kb < 4; ++kb) tma_reduce_add_2d(&a.tm_dg, A + 3 * PT_IMG + kb * PT_CB, kb * 32, t * PT); }
            else { for (int kb = 0; kb < 4; ++kb) tma_store_2d(&a.tm_dg, A + 3 * PT_IMG + kb * PT_CB, kb * 32, t * PT); })
    } else {
        // ================= consumers =================
        const int grp = warp / PF_GW, wgl = warp % PF_GW, q = warp & 3, half = (warp >> 2) & 1, gtid = tid - grp * PF_GT;
        const uint32_t t_acc = t_acc0 + grp * 3 * PT;
        const int hl = lane >> 2;                                // head of this lane's columns
        float4 dbk = make_float4(0.f, 0.f, 0.f, 0.f);
        int i = grp;
        // The query and d_ctx rows of a tile's centre atoms come from global memory (L2): they are fetched one tile ahead
        // -- the indices at the start of the previous tile, the rows behind its MMA issue, into the registers that tile
        // no longer needs -- so that phase A does not start with an exposed L2 round trip
        float4 qv[4], dc[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int t0 = blockIdx.x + grp * gridDim.x;
            const int pn = t0 < nt ? a.pair_c[(size_t)t0 * PT + wgl + PF_GW * k] : -1;
            qv[k] = make_float4(0.f, 0.f, 0.f, 0.f);
            dc[k] = qv[k];
            if (pn >= 0) {
                qv[k] = ld4(a.proj + (size_t)pn * 3 * SCANN_D + 2 * SCANN_D + lane * 4);
                dc[k] = ld4(a.d_ctx + (size_t)pn * SCANN_D + lane * 4);
            }
        }
        for (int t = blockIdx.x + grp * gridDim.x; t < nt; t += PF_NG * gridDim.x, i += PF_NG) {
            const int s = i % PB_NS;
            const uint32_t ph = (uint32_t)(i / PB_NS) & 1u;
            const size_t rowbase = (size_t)t * PT;
            uint8_t* K = c.stages + (size_t)s * PB_STAGE;       // keys -> d_k (hi operand)
            uint8_t* Lo = K + PT_IMG;                           // lo(d_k) -> d_a
            uint8_t* G = K + 2 * PT_IMG;                        // g'
            uint8_t* X = K + 3 * PT_IMG;                        // x[j] -> d_a * x[j]
            const int32_t* sidx = c.idx + s * 64;
            float* Es = c.es + s * 2 * PT * 8;                  // [PT][8] e -> p
            float* Ds = Es + PT * 8;                            // [PT][8] dp -> de
            BCLK(0, 0);
            pipe_wait(&c.full[s], ph, c.dead, a.status, 23, t, s);
            BCLK(0, 1);
            int pc[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) pc[k] = sidx[wgl + PF_GW * k];
            // ---- phase A: e = 0.25 <q_h,k_h>, dp = <dctx_h,k_h> per (row, head)
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int r = wgl + PF_GW * k;
                if (pc[k] < 0) continue;                                // padding row (warp-uniform)
                const float4 kv = lds4(K + pt_off4(r, lane));
                const float e = quad_sum(dot4(kv, qv[k])) * 0.25f;
                const float d = quad_sum(dot4(kv, dc[k]));
                if ((lane & 3) == 0) { Es[r * 8 + hl] = e; Ds[r * 8 + hl] = d; }
            }
            pf_group_sync(grp);
            BCLK(0, 2);
            // ---- phase B1 (warp per HEAD, lane per row): softmax over an atom's rows and its backward.  The rows of an
            // atom are a contiguous run of lanes, so max / sums are segmented shuffle reductions: every warp is busy and
            // the cost does not depend on the neighbour count (first form: one warp per atom looped over its rows --
            // three or four of the eight warps worked, 24 % of the kernel's samples sat in the barrier behind them)
            const int myc = sidx[lane];
            const int prevc = __shfl_up_sync(0xffffffffu, myc, 1);
            const uint32_t vmask = __ballot_sync(0xffffffffu, myc >= 0);
            const uint32_t hmask = __ballot_sync(0xffffffffu, myc >= 0 && (lane == 0 || myc != prevc));
            const int nvalid = __popc(vmask), natoms = __popc(hmask);
            {
                const bool valid = myc >= 0;
                const uint32_t below = hmask & ((2u << lane) - 1u);              // run starts at or below this lane
                const uint32_t above = lane < 31 ? hmask & ~((2u << lane) - 1u) : 0u;
                const int lo = valid ? 31 - __clz(below) : lane;                 // first / last lane of this lane's run
                const int hi = valid ? (above ? __ffs(above) - 2 : nvalid - 1) : lane;
                const int h = wgl;
                const float e = valid ? Es[lane * 8 + h] : -INFINITY;
                float mx = e;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const float v = __shfl_down_sync(0xffffffffu, mx, o);
                    if (lane + o <= hi) mx = fmaxf(mx, v);
                }
                mx = __shfl_sync(0xffffffffu, mx, lo);
                const float p = valid ? __expf(e - mx) : 0.f;
                // gradient w.r.t. the softmax output = (gradient w.r.t. the dropped probabilities) * mask
                const float dm = valid ? drop_mult(a.drop, a.drop_site, (uint32_t)(rowbase + lane) * 8u + h) : 0.f;
                const float dp = valid ? Ds[lane * 8 + h] * dm : 0.f;
                float sm = p, dot = p * dp;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const float v1 = __shfl_down_sync(0xffffffffu, sm, o), v2 = __shfl_down_sync(0xffffffffu, dot, o);
                    if (lane + o <= hi) { sm += v1; dot += v2; }
                }
                sm = __shfl_sync(0xffffffffu, sm, lo);
                dot = __shfl_sync(0xffffffffu, dot, lo);
                if (valid) {
                    const float is = 1.0f / sm;
                    const float pn = p * is;
                    // d_k uses the dropped probabilities, the softmax backward the undropped ones
                    Es[lane * 8 + h] = pn * dm;
                    Ds[lane * 8 + h] = pn * (dp - dot * is);
                }
            }
            pf_group_sync(grp);
            BCLK(0, 3);
            // ---- phase B2: dq = d_ctx + 0.25 sum_n de k, by the warp that owns the atom's FIRST row (rows wgl + 8 k): its
            // d_ctx row already sits in that warp's registers (dc[k]), and the atoms spread over all eight warps.  The row
            // loop runs four rows per trip so that the shared-memory loads of a trip are in flight together.
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int r0 = wgl + PF_GW * k;
                if (!((hmask >> r0) & 1u)) continue;                      // (warp-uniform)
                const uint32_t nxt = r0 < 31 ? hmask & ~((2u << r0) - 1u) : 0u;
                const int n = (nxt ? __ffs(nxt) - 1 : nvalid) - r0;
                float c0 = 0.f, c1 = 0.f, c2 = 0.f, c3 = 0.f;
                for (int r = 0; r < n; r += 4) {
                    float de[4];
                    float4 kv[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int rr = r0 + (r + u < n ? r + u : 0);
                        de[u] = r + u < n ? Ds[rr * 8 + hl] : 0.f;
                        kv[u] = lds4(K + pt_off4(rr, lane));
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        c0 = fmaf(de[u], kv[u].x, c0); c1 = fmaf(de[u], kv[u].y, c1);
                        c2 = fmaf(de[u], kv[u].z, c2); c3 = fmaf(de[u], kv[u].w, c3);
                    }
                }
                st4(a.dq + (size_t)pc[k] * SCANN_D + lane * 4,
                    make_float4(dc[k].x + 0.25f * c0, dc[k].y + 0.25f * c1, dc[k].z + 0.25f * c2, dc[k].w + 0.25f * c3));
            }
            pf_group_sync(grp);
            BCLK(0, 4);
            // ---- phase C: dk = p d_ctx[c] + 0.25 de q[c] in place over k (hi operand), lo image, dbk
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int r = wgl + PF_GW * k;
                const uint32_t off = pt_off4(r, lane);
                float4 dk = make_float4(0.f, 0.f, 0.f, 0.f);
                if (pc[k] >= 0) {
                    const float p = Es[r * 8 + hl], de = 0.25f * Ds[r * 8 + hl];
                    dk = make_float4(fmaf(p, dc[k].x, de * qv[k].x), fmaf(p, dc[k].y, de * qv[k].y),
                                     fmaf(p, dc[k].z, de * qv[k].z), fmaf(p, dc[k].w, de * qv[k].w));
                }
                dbk = make_float4(dbk.x + dk.x, dbk.y + dk.y, dbk.z + dk.z, dbk.w + dk.w);
                sts4(K + off, dk);
                sts4(Lo + off, tf32_lo4(dk));
            }
            fence_async_smem();
            tc_fence_before();
            pf_group_sync(grp);
            BCLK(0, 5);
            if (wgl < 3) {                                      // d_a^T = Wk dk^T: one product chain per warp
                tc_fence_after();
                if (tc_elect_one()) pf_issue_chain(wgl, t_wraw, t_wlo, smem_u32(K), smem_u32(Lo), t_acc, &c.accf[s]);
                __syncwarp();
            }
            BCLK(0, 6);
            int jj[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) jj[k] = pc[k] >= 0 ? sidx[32 + wgl + PF_GW * k] : 0;
            // the next tile's query / d_ctx rows (its centre indices straight from global memory): in flight behind the
            // MMAs and phase D
            {
                const int tn = t + PF_NG * (int)gridDim.x;
                int pn[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) pn[k] = tn < nt ? a.pair_c[(size_t)tn * PT + wgl + PF_GW * k] : -1;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    qv[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                    dc[k] = qv[k];
                    if (pn[k] >= 0) {
                        qv[k] = ld4(a.proj + (size_t)pn[k] * 3 * SCANN_D + 2 * SCANN_D + lane * 4);
                        dc[k] = ld4(a.d_ctx + (size_t)pn[k] * SCANN_D + lane * 4);
                    }
                }
            }
            pipe_wait(&c.accf[s], ph, c.dead, a.status, 24, t, s);
            tc_fence_after();
            BCLK(0, 7);
            pf_acc_to_image(t_acc, Lo, nullptr, q, half, lane);
            tc_fence_before();
            pf_group_sync(grp);
            BCLK(0, 8);
            // ---- phase D: d_nbr = d_a * g' -> dx[j] ; d_a * x[j] in place over x[j] (-> dg through the store warp)
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int r = wgl + PF_GW * k;
                const uint32_t off = pt_off4(r, lane);
                float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
                if (pc[k] >= 0) {
                    const float4 da = lds4(Lo + off), gp = lds4(G + off), xj = lds4(X + off);
                    if constexpr (DET)
                        st4(a.dx_scatter + (rowbase + r) * SCANN_D + lane * 4,
                            make_float4(da.x * gp.x, da.y * gp.y, da.z * gp.z, da.w * gp.w));
                    else
                        red_add4(a.dx_scatter + (size_t)jj[k] * SCANN_D + lane * 4, da.x * gp.x, da.y * gp.y, da.z * gp.z, da.w * gp.w);
                    o = make_float4(da.x * xj.x, da.y * xj.y, da.z * xj.z, da.w * xj.w);
                }
                sts4(X + off, o);
            }
            fence_async_smem();
            pf_group_sync(grp);
            BCLK(0, 9);
            if (gtid == 0) mbar_arrive(&c.ready[s]);            // d_k and d_a * x[j]: over to the store warp
        }
        if constexpr (DET) {
            for (int w = 0; w < PF_CW; ++w) {
                if (warp == w) {
                    s_dbk[lane * 4 + 0] += dbk.x; s_dbk[lane * 4 + 1] += dbk.y;
                    s_dbk[lane * 4 + 2] += dbk.z; s_dbk[lane * 4 + 3] += dbk.w;
                }
                pb_consumer_sync();
            }
        } else {
            atomicAdd(&s_dbk[lane * 4 + 0], dbk.x); atomicAdd(&s_dbk[lane * 4 + 1], dbk.y);
            atomicAdd(&s_dbk[lane * 4 + 2], dbk.z); atomicAdd(&s_dbk[lane * 4 + 3], dbk.w);
        }
    }
    pdl_trigger();
    tc_fence_before();
    __syncthreads();
    if constexpr (DET) {
        if (tid < SCANN_D) a.dbk[(size_t)blockIdx.x * SCANN_D + tid] = s_dbk[tid];
    } else {
        if (tid < SCANN_D) atomicAdd(a.dbk + tid, s_dbk[tid]);
    }
    if (warp == PF_CW + 1) tmem_dealloc(tmem, 512);
}

// =============================================================================================
// Geometry backward
// =============================================================================================
struct PipeGeomBwdArgs {
    CUtensorMap tm_pre, tm_g, tm_dgt, tm_dgo;
    const int32_t* ntiles; const int32_t* pair_c; const int32_t* pair_j;
    const float* W2T;        // transposed block: W2T[n][k] = W2[k][n]
    const float* gamma_g;
    float* s_pre;            // [R,128]  <- sum_n d_pre (atoms with pairs)
    float* t_scatter;        // [R,128]  += d_pre at the neighbour rows
    float* dgamma_g; float* dbeta_g;
    int32_t* status;
};

template <bool DET>
__global__ void __launch_bounds__(PF_THREADS, 1) la_geom_bwd_pipe_kernel(const __grid_constant__ PipeGeomBwdArgs a) {
    __shared__ float s_acc[2 * SCANN_D];
    if (threadIdx.x < 2 * SCANN_D) s_acc[threadIdx.x] = 0.f;
    // stationary operand A[M = k][K = n] = W2[k][n]: (d_pre W2^T)^T = W2 d_pre^T
    // (Tried in round 2: phase A in the forward kernels' row-group mapping -- four rows of a warp at once, three-step
    // reductions, x_hat parked in the G image for a separate d_gamma / d_beta pass.  The phase itself got 30 % shorter
    // (4 300 -> 2 950 cycles) but the step 0.7 % SLOWER: the extra image traffic (4 STS.128 + 8 LDS.128 per lane and tile)
    // costs more than the shorter chain saves -- these kernels are bound by the shared-memory pipe, ~270 KB per tile.)
    PF_PROLOGUE(BwdFrame, PB_NS, a.W2T, 1)
    if (warp == PF_CW) {
        // ================= producer =================
        if (lane == 0) {
            tma_prefetch_desc(&a.tm_pre); tma_prefetch_desc(&a.tm_g); tma_prefetch_desc(&a.tm_dgt);
            int i = 0;
            for (int t = blockIdx.x; t < nt; t += gridDim.x, ++i) {
                const int s = i % PB_NS;
                const uint32_t ph = (uint32_t)(i / PB_NS) & 1u;
                pipe_wait(&c.empty[s], ph ^ 1u, c.dead, a.status, 31, t, s);
                uint8_t* S0 = c.stages + (size_t)s * PB_STAGE;
                mbar_expect_tx(&c.full[s], 3u * PT_IMG + 256u);
#pragma unroll
                for (int kb = 0; kb < 4; ++kb) tma_load_2d(S0 + kb * PT_CB, &a.tm_pre, kb * 32, t * PT, &c.full[s]);
#pragma unroll
                for (int kb = 0; kb < 4; ++kb) tma_load_2d(S0 + 2 * PT_IMG + kb * PT_CB, &a.tm_g, kb * 32, t * PT, &c.full[s]);
#pragma unroll
                for (int kb = 0; kb < 4; ++kb) tma_load_2d(S0 + 3 * PT_IMG + kb * PT_CB, &a.tm_dgt, kb * 32, t * PT, &c.full[s]);
                bulk_load(c.idx + s * 64, a.pair_c + (size_t)t * PT, 128u, &c.full[s]);
                bulk_load(c.idx + s * 64 + 32, a.pair_j + (size_t)t * PT, 128u, &c.full[s]);
                const int tp = t + PB_NS * (int)gridDim.x;            // L2 prefetch of the tile behind the ring
                if (tp < nt) {
#pragma unroll
                    for (int kb = 0; kb < 4; ++kb) {
                        tma_prefetch_2d(&a.tm_pre, kb * 32, tp * PT); tma_prefetch_2d(&a.tm_g, kb * 32, tp * PT);
                        tma_prefetch_2d(&a.tm_dgt, kb * 32, tp * PT);
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp > PF_CW) {
        if (lane == 0) tma_prefetch_desc(&a.tm_dgo);
        PF_STORE_LOOP(PB_NS, PB_STAGE, 32,
            for (int kb = 0; kb < 4; ++kb) tma_store_2d(&a.tm_pre, A + kb * PT_CB, kb * 32, t * PT);
            for (int kb = 0; kb < 4; ++kb) tma_store_2d(&a.tm_dgo, A + PT_IMG + kb * PT_CB, kb * 32, t * PT);)
    } else {
        // ================= consumers =================
        const int grp = warp / PF_GW, wgl = warp % PF_GW, q = warp & 3, half = (warp >> 2) & 1, gtid = tid - grp * PF_GT;
        const uint32_t t_acc = t_acc0 + grp * 3 * PT;
        const float4 gam = ldg4(a.gamma_g + lane * 4);
        float4 dgam = make_float4(0.f, 0.f, 0.f, 0.f), dbet = dgam;
        int i = grp;
        for (int t = blockIdx.x + grp * gridDim.x; t < nt; t += PF_NG * gridDim.x, i += PF_NG) {
            const int s = i % PB_NS;
            const uint32_t ph = (uint32_t)(i / PB_NS) & 1u;
            uint8_t* P = c.stages + (size_t)s * PB_STAGE;       // pre-activation -> d_pre (hi operand)
            uint8_t* Lo = P + PT_IMG;                           // lo(d_pre) -> d_pre @ W2^T -> dg
            uint8_t* G = P + 2 * PT_IMG;                        // layer input geometry g
            uint8_t* Dg = P + 3 * PT_IMG;                       // gradient w.r.t. g'
            const int32_t* sidx = c.idx + s * 64;
            BCLK(1, 0);
            pipe_wait(&c.full[s], ph, c.dead, a.status, 33, t, s);
            BCLK(1, 1);
            int pc[4];
            float4 dz[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) pc[k] = sidx[wgl + PF_GW * k];
            // ---- phase A: recompute z statistics, LN_g backward, d_pre
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int r = wgl + PF_GW * k;
                const uint32_t off = pt_off4(r, lane);
                if (pc[k] < 0) {                                         // padding row (warp-uniform)
                    dz[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                    sts4(P + off, dz[k]);
                    sts4(Lo + off, dz[k]);
                    continue;
                }
                const int jr = sidx[32 + r];
                const float4 pv = lds4(P + off), gv = lds4(G + off), dv = lds4(Dg + off);
                const float pre[4] = {pv.x, pv.y, pv.z, pv.w};
                const float g[4] = {gv.x, gv.y, gv.z, gv.w};
                const float dgt[4] = {dv.x, dv.y, dv.z, dv.w};
                const float gm[4] = {gam.x, gam.y, gam.z, gam.w};
                float z[4], sg[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) { sg[e] = sigmoid_fast(pre[e]); z[e] = pre[e] * sg[e] + g[e]; }
                const float s1 = z[0] + z[1] + z[2] + z[3];
                const float sh = __shfl_sync(0xffffffffu, s1, 0) * 0.25f;
                const float d[4] = {z[0] - sh, z[1] - sh, z[2] - sh, z[3] - sh};
                float m1 = d[0] + d[1] + d[2] + d[3], m2 = d[0] * d[0] + d[1] * d[1] + d[2] * d[2] + d[3] * d[3];
                warp_sum2(m1, m2);
                m1 *= (1.0f / SCANN_D);
                const float inv = rsqrtf(fmaxf(m2 * (1.0f / SCANN_D) - m1 * m1, 0.f) + SCANN_LN_EPS);
                float xh[4], dxh[4];
                float t1 = 0.f, t2 = 0.f;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    xh[e] = (d[e] - m1) * inv;
                    dxh[e] = dgt[e] * gm[e];
                    t1 += dxh[e];
                    t2 = fmaf(dxh[e], xh[e], t2);
                }
                warp_sum2(t1, t2);
                t1 *= (1.0f / SCANN_D);
                t2 *= (1.0f / SCANN_D);
                float dzv[4], dp[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    dzv[e] = inv * (dxh[e] - t1 - xh[e] * t2);
                    dp[e] = dzv[e] * sg[e] * (1.0f + pre[e] * (1.0f - sg[e]));        // swish'(pre)
                }
                dgam = make_float4(fmaf(dgt[0], xh[0], dgam.x), fmaf(dgt[1], xh[1], dgam.y), fmaf(dgt[2], xh[2], dgam.z),
                                   fmaf(dgt[3], xh[3], dgam.w));
                dbet = make_float4(dbet.x + dgt[0], dbet.y + dgt[1], dbet.z + dgt[2], dbet.w + dgt[3]);
                dz[k] = make_float4(dzv[0], dzv[1], dzv[2], dzv[3]);
                const float4 dpre = make_float4(dp[0], dp[1], dp[2], dp[3]);
                sts4(P + off, dpre);
                sts4(Lo + off, tf32_lo4(dpre));
                if constexpr (!DET) red_add4(a.t_scatter + (size_t)jr * SCANN_D + lane * 4, dp[0], dp[1], dp[2], dp[3]);
            }
            fence_async_smem();
            tc_fence_before();
            pf_group_sync(grp);
            BCLK(1, 2);
            if (wgl < 3) {                                      // W2 d_pre^T: one product chain per warp
                tc_fence_after();
                if (tc_elect_one()) pf_issue_chain(wgl, t_wraw, t_wlo, smem_u32(P), smem_u32(Lo), t_acc, &c.accf[s]);
                __syncwarp();
            }
            BCLK(1, 3);
            // ---- phase B (warp per atom, overlaps the MMAs): s_pre[c] = sum_n d_pre
            {
                const int myc = sidx[lane];
                const int prevc = __shfl_up_sync(0xffffffffu, myc, 1);
                const uint32_t vmask = __ballot_sync(0xffffffffu, myc >= 0);
                const uint32_t hmask = __ballot_sync(0xffffffffu, myc >= 0 && (lane == 0 || myc != prevc));
                const int nvalid = __popc(vmask), natoms = __popc(hmask);
                uint32_t m = hmask;
                for (int k = 0; k < wgl; ++k) m &= m - 1;
                for (int k = wgl; k < natoms; k += PF_GW) {
                    const int r0 = __ffs(m) - 1;
                    uint32_t mn = m;
                    mn &= mn - 1;
                    const int n = (mn ? __ffs(mn) - 1 : nvalid) - r0;
                    const int atom = sidx[r0];
                    float c0 = 0.f, c1 = 0.f, c2 = 0.f, c3 = 0.f;
                    for (int r = 0; r < n; ++r) {
                        const float4 v = lds4(P + pt_off4(r0 + r, lane));
                        c0 += v.x; c1 += v.y; c2 += v.z; c3 += v.w;
                    }
                    st4(a.s_pre + (size_t)atom * SCANN_D + lane * 4, make_float4(c0, c1, c2, c3));
                    for (int k2 = 0; k2 < PF_GW && m; ++k2) m &= m - 1;
                }
            }
            BCLK(1, 4);
            pipe_wait(&c.accf[s], ph, c.dead, a.status, 34, t, s);
            tc_fence_after();
            BCLK(1, 5);
            pf_acc_to_image(t_acc, Lo, nullptr, q, half, lane);
            tc_fence_before();
            pf_group_sync(grp);
            BCLK(1, 6);
            // ---- phase C: dg = d_z + d_pre @ W2^T (in place)
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t off = pt_off4(wgl + PF_GW * k, lane);
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (pc[k] >= 0) {
                    v = lds4(Lo + off);
                    v = make_float4(v.x + dz[k].x, v.y + dz[k].y, v.z + dz[k].z, v.w + dz[k].w);
                }
                sts4(Lo + off, v);
            }
            fence_async_smem();
            pf_group_sync(grp);
            BCLK(1, 7);
            if (gtid == 0) mbar_arrive(&c.ready[s]);            // d_pre and dg: over to the store warp
        }
        if constexpr (DET) {
            for (int w = 0; w < PF_CW; ++w) {
                if (warp == w) {
                    s_acc[lane * 4 + 0] += dgam.x; s_acc[lane * 4 + 1] += dgam.y;
                    s_acc[lane * 4 + 2] += dgam.z; s_acc[lane * 4 + 3] += dgam.w;
                    s_acc[SCANN_D + lane * 4 + 0] += dbet.x; s_acc[SCANN_D + lane * 4 + 1] += dbet.y;
                    s_acc[SCANN_D + lane * 4 + 2] += dbet.z; s_acc[SCANN_D + lane * 4 + 3] += dbet.w;
                }
                pb_consumer_sync();
            }
        } else {
            atomicAdd(&s_acc[lane * 4 + 0], dgam.x); atomicAdd(&s_acc[lane * 4 + 1], dgam.y);
            atomicAdd(&s_acc[lane * 4 + 2], dgam.z); atomicAdd(&s_acc[lane * 4 + 3], dgam.w);
            atomicAdd(&s_acc[SCANN_D + lane * 4 + 0], dbet.x); atomicAdd(&s_acc[SCANN_D + lane * 4 + 1], dbet.y);
            atomicAdd(&s_acc[SCANN_D + lane * 4 + 2], dbet.z); atomicAdd(&s_acc[SCANN_D + lane * 4 + 3], dbet.w);
        }
    }
    pdl_trigger();
    tc_fence_before();
    __syncthreads();
    if constexpr (DET) {
        if (tid < 2 * SCANN_D) a.dgamma_g[(size_t)blockIdx.x * 2 * SCANN_D + tid] = s_acc[tid];
    } else if (tid < SCANN_D) {
        atomicAdd(a.dgamma_g + tid, s_acc[tid]);
        atomicAdd(a.dbeta_g + tid, s_acc[SCANN_D + tid]);
    }
    if (warp == PF_CW + 1) tmem_dealloc(tmem, 512);
}

// ---- host ---------------------------------------------------------------------------------------------------
template <bool DET>
static int la_pipe_bwd_configure() {
    static bool configured = false;
    if (configured) return 0;
    cudaError_t e = cudaFuncSetAttribute(la_attn_bwd_pipe_kernel<DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PB_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(la_geom_bwd_pipe_kernel<DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PB_SMEM);
    if (e != cudaSuccess) { scann_set_error("la_backward_pipe: smem opt-in failed: %s", cudaGetErrorString(e)); return 1; }
    configured = true;
    return 0;
}

template <bool DET>
static int la_pipe_bwd_launch(int grid, long long rows, int which, const int32_t* ntiles, const int32_t* pair_c,
                              const int32_t* pair_j, const float* x, const float* proj, const float* g_in,
                              const float* g_new, float* kbuf, float* prebuf, const float* W2T, const float* WkT,
                              const float* gamma_g, const float* d_ctx, float* dg, int dg_has_up, float* dg_out,
                              float* dq, float* s_pre, float* t_scatter, float* dx_scatter, float* dgamma_g,
                              float* dbeta_g, float* dbk, const void* attn_drop, int drop_site, int32_t* status,
                              void* stream) {
    if (la_pipe_bwd_configure<DET>()) return 1;
    if (grid <= 0) return 0;
    if (which & 1) {
        PipeAttnBwdArgs ab;
        memset(&ab, 0, sizeof(ab));
        if (pipe_encode_tmap(&ab.tm_k, kbuf, rows) || pipe_encode_tmap(&ab.tm_g, g_new, rows) ||
            pipe_encode_tmap(&ab.tm_dg, dg, rows)) return 1;
        ab.ntiles = ntiles; ab.pair_c = pair_c; ab.pair_j = pair_j; ab.x = x; ab.proj = proj; ab.WkT = WkT; ab.d_ctx = d_ctx;
        ab.dq = dq; ab.dx_scatter = dx_scatter; ab.dbk = dbk; ab.dg_accum = dg_has_up ? 1 : 0;
        ab.drop = (const ScannDropCtl*)attn_drop; ab.drop_site = drop_site; ab.status = status;
        scann_launch(la_attn_bwd_pipe_kernel<DET>, dim3(grid), dim3(PF_THREADS), PB_SMEM, stream, ab);
    }
    if (which & 2) {
        PipeGeomBwdArgs gb;
        memset(&gb, 0, sizeof(gb));
        if (pipe_encode_tmap(&gb.tm_pre, prebuf, rows) || pipe_encode_tmap(&gb.tm_g, g_in, rows) ||
            pipe_encode_tmap(&gb.tm_dgt, dg, rows) || pipe_encode_tmap(&gb.tm_dgo, dg_out, rows)) return 1;
        gb.ntiles = ntiles; gb.pair_c = pair_c; gb.pair_j = pair_j; gb.W2T = W2T; gb.gamma_g = gamma_g; gb.s_pre = s_pre;
        gb.t_scatter = t_scatter; gb.dgamma_g = dgamma_g; gb.dbeta_g = dbeta_g; gb.status = status;
        scann_launch(la_geom_bwd_pipe_kernel<DET>, dim3(grid), dim3(PF_THREADS), PB_SMEM, stream, gb);
    }
    return scann_check_launch("scann_la_backward_pipe");
}

// Pipelined backward of LocalAttention (TF autodiff of attention.py:118-216 inside keras fit) for pair plans with
// tile_stride 32; same data contract as scann_la_backward_tc.  rows = tile_cap * 32.  which: bit 0 attention kernel,
// bit 1 geometry kernel.
extern "C" int scann_la_backward_pipe(int grid, long long rows, int which, const int32_t* ntiles, const int32_t* pair_c,
                                      const int32_t* pair_j, const float* x, const float* proj, const float* g_in,
                                      const float* g_new, float* kbuf, float* prebuf, const float* W2T, const float* WkT,
                                      const float* gamma_g, const float* d_ctx, float* dg, int dg_has_up, float* dg_out,
                                      float* dq, float* s_pre, float* t_scatter, float* dx_scatter, float* dgamma_g,
                                      float* dbeta_g, float* dbk, const void* attn_drop, int drop_site, int32_t* status,
                                      void* stream) {
    return la_pipe_bwd_launch<false>(grid, rows, which, ntiles, pair_c, pair_j, x, proj, g_in, g_new, kbuf, prebuf, W2T, WkT,
                                     gamma_g, d_ctx, dg, dg_has_up, dg_out, dq, s_pre, t_scatter, dx_scatter, dgamma_g,
                                     dbeta_g, dbk, attn_drop, drop_site, status, stream);
}

// Deterministic form (DESIGN.md section 4.7): same arguments, except
//   dx_scatter : [rows,128] per-pair buffer, d_a * g' stored at the pair row (scann_row_gather sums it per atom row)
//   t_scatter  : unused (d_pre is left per pair in prebuf)
//   dbk        : [grid][128] slots; dgamma_g : [grid][256] slots (gamma | beta); dbeta_g : unused
extern "C" int scann_la_backward_pipe_det(int grid, long long rows, int which, const int32_t* ntiles, const int32_t* pair_c,
                                          const int32_t* pair_j, const float* x, const float* proj, const float* g_in,
                                          const float* g_new, float* kbuf, float* prebuf, const float* W2T, const float* WkT,
                                          const float* gamma_g, const float* d_ctx, float* dg, int dg_has_up, float* dg_out,
                                          float* dq, float* s_pre, float* t_scatter, float* dx_scatter, float* dgamma_g,
                                          float* dbeta_g, float* dbk, const void* attn_drop, int drop_site, int32_t* status,
                                          void* stream) {
    return la_pipe_bwd_launch<true>(grid, rows, which, ntiles, pair_c, pair_j, x, proj, g_in, g_new, kbuf, prebuf, W2T, WkT,
                                    gamma_g, d_ctx, dg, dg_has_up, dg_out, dq, s_pre, t_scatter, dx_scatter, dgamma_g,
                                    dbeta_g, dbk, attn_drop, drop_site, status, stream);
}
