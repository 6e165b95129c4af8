/* scann_b200.h -- C ABI of libscann_b200.so (sm_100a only, no CPU fallback).
 *
 * Drop-in boundary for the SCANN attention hot path.  The reference has no FFI: the path sits
 * behind Keras Layer objects (scann/layers/attention.py, scann/layers/custom_layers.py) wired by
 * create_model (scann/models/scann_model.py:329-453).  Each entry point below names the reference
 * code it replaces.  Host code (Python, scann_b200/) binds these with ctypes and exchanges
 * tensors with the caller via DLPack; see INTEGRATION.md for the reference-side stub.
 *
 * Conventions
 *  - every function returns 0 on success; non-zero -> scann_last_error() holds a message;
 *  - all pointers are DEVICE pointers unless stated -- RAW pointers and sizes, not DLManagedTensor*: the DLPack
 *    hand-over (torch / tf.experimental.dlpack) happens on the host side, which passes data_ptr() of the
 *    imported tensor; arguments are borrowed, outputs are caller-allocated, nothing is allocated or freed inside
 *    the library (one explicit exception: scann_p2p_alloc / scann_p2p_free, whose block must be exportable through
 *    CUDA IPC);
 *  - `stream` is a cudaStream_t passed as void*; calls are asynchronous and re-entrant across
 *    streams; the only global state is the per-thread error string and two per-thread launch switches
 *    (scann_set_pdl, scann_set_la_groups4: scheduling choices, never numerics);
 *  - the data-parallel exchange is either an NCCL all-reduce of the gradient arena (scann_allreduce_*, NCCL bound at run
 *    time; torch.distributed's own all_reduce works as well) or the peer-memory form fused into the optimiser kernel
 *    (scann_p2p_*, scann_adam_p2p_step); the NCCL communicator is the one piece of process-wide state;
 *  - per-atom tensors are [R,128] fp32 row-major with R = B*M (row r = b*M + m);
 *    per-pair tensors use the tile-padded packed layout built by scann_plan_build:
 *    tile t owns rows [S t, S t + S) with S = tile_stride (32 for the pipelined local-attention kernels,
 *    64 / 128 for the round-1 kernels), rows with pair_c < 0 are padding;
 *  - weight blocks are [128,128] fp32 row-major (Keras Dense kernels, [in,out]);
 *  - `status` is a device int32 of SCANN_ERR_* bits set by kernels on malformed input.
 */
#ifndef SCANN_B200_H
#define SCANN_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCANN_ERR_TILE_OVERFLOW 1
#define SCANN_ERR_TOO_MANY_NBRS 2
#define SCANN_ERR_BAD_ATOMIC 4
#define SCANN_ERR_BAD_NEIGHBOR 8
#define SCANN_ERR_PIPE_TIMEOUT 16   /* a bounded mbarrier wait of a pipelined kernel gave up (status[1..4] say where) */

/* ---- library ---------------------------------------------------------------------------- */
const char* scann_last_error(void);
int scann_version(void);
/* SM count of the current device, -1 when no CUDA device is usable (callers must refuse to run). */
int scann_device_sm_count(void);
int scann_device_cc(void);
/* Programmatic dependent launch (per calling thread; returns the previous setting).  When on, the kernels of
 * the forward / backward chain are launched with programmatic stream serialisation so that a kernel's
 * prologue (tensor-memory allocation, weights -> tensor memory) overlaps the tail of its stream predecessor.
 * Switch it off for a launch whose stream predecessor is not a kernel of this library (memset, event join). */
int scann_set_pdl(int on);
/* Local-attention kernels with four warp groups per CTA (per calling thread; returns the previous mask).  Bit 0
 * geometry forward, 1 attention forward, 2 attention backward, 3 geometry backward: a set bit makes
 * scann_la_forward_tc / scann_la_backward_tc run that kernel with four tile streams per SM whenever the pair plan
 * has tile_stride 64 and mma_rows <= 48 (same results; a scheduling choice, not a numerical one). */
int scann_set_la_groups4(int mask);

/* ---- batch plan ---------------------------------------------------------------------------
 * Replaces the mask / index bookkeeping the reference does with dense padded tensors:
 * gather_shape (scann/layers/custom_layers.py:18-28), the (1-mask)*-1e9 additive mask and the
 * mask multiply of LocalAttention.call (scann/layers/attention.py:186-187, :206).  Inputs are the
 * padded arrays of DataIterator.__getitem__ (scann/utils/datagenerator.py:80-101):
 * neighbor_mask [B,M,N] uint8, neighbors [B,M,N] int32, dist/weight [B,M,N] fp32.
 * Outputs: cnt[R], rowptr[R], tile_a0/tile_a1[tile_cap] (atom range of each tile), ntiles[1],
 * pair_c/pair_j/pair_slot/pair_d/pair_w [tile_cap*tile_stride].  scratch: >= 4*ceil(R/128) int32 (2* without valid_rows).
 * With >= 6*ceil(R/128) + 6 int32, 8-byte aligned and ZEROED ONCE when allocated (never touched by the caller
 * afterwards), the plan is built by one launch (one CTA per 128 atom rows, decoupled look-back through the words
 * kept in scratch) instead of four; the result is identical.
 * tile_rows (<= tile_stride): greedy fill limit per tile, chosen by the caller to balance SM waves.
 * valid_rows, valid_j [tile_cap*tile_stride] / nvalid [1] (nullable): compact list of the valid pair rows in tile
 * order and the neighbour atom row of each, for
 * consumers that only reduce over pairs (scann_wgrad_batch_tc) and should not pay for padding rows. */
int scann_plan_build(const uint8_t* neighbor_mask, const int32_t* neighbors, const float* dist,
                     const float* weight, int B, int M, int N, int tile_cap, int tile_rows, int tile_stride,
                     int32_t* cnt, int32_t* rowptr,
                     int32_t* tile_a0, int32_t* tile_a1, int32_t* ntiles, int32_t* pair_c, int32_t* pair_j,
                     int32_t* pair_slot, float* pair_d, float* pair_w, int32_t* valid_rows, int32_t* valid_j,
                     int32_t* nvalid, int32_t* scratch, int scratch_len, int32_t* status, void* stream);

/* ---- ragged batch -> padded device buffers --------------------------------------------------------
 * DataIterator.__getitem__ (scann/utils/datagenerator.py:69-135) on the device: the batch arrives as CSR arrays in
 * one DEVICE blob (byte offsets off_*: struct_atom_off [B+1], atom_nbr_off [A+1], z [A], nbr_idx / nbr_w / nbr_d [P]
 * int32/float32, ring [A,2] int32 or off < 0, target [B] float32 or off < 0) and is expanded into the padded arrays
 * of the reference's input dict: neighbour value 1000 = padding marker (mask false, index 0), zero-padded weights
 * and distances, atom_mask = Z != 0. */
int scann_pack_batch(const void* csr, long long off_sa, long long off_an, long long off_z, long long off_idx,
                     long long off_w, long long off_d, long long off_ring, long long off_target, int B, int M, int N,
                     int32_t* atomic, uint8_t* atom_mask, int32_t* neighbors, uint8_t* neighbor_mask, float* weight,
                     float* dist, float* ring_out, float* target, void* stream);

/* ---- input embedding: Embedding + (extra_embed) + dense_embed swish -----------------------
 * scann/models/scann_model.py:361-374.  ring may be NULL (use_ring False). t0 (pre-activation,
 * saved for backward) may be NULL. */
int scann_embed_forward(const int32_t* atomic, const float* ring, int R, int E, int n_atoms, const float* emb,
                        const float* Wr, const float* br, const float* We, const float* be, float* t0, float* x0,
                        int32_t* status, const void* drop_ctl, const float* emb_rows, void* stream);
/* feature == "cgcnn" (scann_model.py:364-365): embed_atom is Dense(92 -> E) over per-atom feature vectors.
 * emb_rows [R,E] = atomic92 @ W + b is passed to scann_embed_forward (emb_rows != NULL replaces the lookup). */
int scann_cgcnn_embed_forward(const float* atomic92, const float* W, const float* b, int R, int F, int E,
                              float* emb_rows, void* stream);
int scann_cgcnn_embed_backward(const float* atomic92, const float* emb_rows, const float* ring, int R, int F, int E,
                               const float* Wr, const float* br, const float* We, const float* t0, const float* dx0,
                               float* d_cat_ws, float* dWemb, float* dbemb, float* dWr, float* dbr, float* dWe, float* dbe,
                               const void* drop_ctl, void* stream);
/* Gradients are ACCUMULATED into d_emb, dWr, dbr, dWe, dbe.  G_ws: (n_atoms+3)*128 floats. */
int scann_embed_backward(const int32_t* atomic, const float* ring, int R, int E, int n_atoms, const float* emb,
                         const float* Wr, const float* br, const float* We, const float* t0, const float* dx0,
                         float* G_ws, float* d_emb, float* dWr, float* dbr, float* dWe, float* dbe, const void* drop_ctl, void* stream);

/* ---- geometry initialisation: GaussianExpansion x2 + neighbor_d/neighbor_w Dense + Multiply --
 * scann/layers/custom_layers.py:55-65, scann/models/scann_model.py:378-389. */
int scann_geom_init_forward(const int32_t* ntiles, int grid, int tile_stride, const int32_t* pair_c, const float* pair_d,
                            const float* pair_w, const float* centers_d, const float* centers_w, const float* Wd,
                            const float* bd, const float* Ww, const float* bw, float* g0, void* stream);
int scann_geom_init_backward(const int32_t* ntiles, int grid, int tile_stride, const int32_t* pair_c, const float* pair_d,
                             const float* pair_w, const float* centers_d, const float* centers_w, const float* Wd,
                             const float* bd, const float* Ww, const float* bw, const float* dg0, float* dWd,
                             float* dbd, float* dWw, float* dbw, void* stream);

/* ---- per-atom Dense layers ------------------------------------------------------------------
 * C[r, nb*128+c] = epi(sum_kb A[kb][r,:] @ W[kb*nblk+nb] + bias[nb] (+ resid)); A/W/bias are HOST
 * arrays of device pointers.  mode: 0 none, 1 swish (pre_out <- pre-activation), 2 multiply by
 * swish'(pre_in), 3 LayerNorm(eps 1e-6) (pre_out <- pre-LN value).  Replaces keras Dense /
 * LayerNormalization calls of LocalAttention (attention.py:95-113,160), ResidualNorm (:25-40),
 * after_Lc and the GlobalAttention projections (scann_model.py:424-429, attention.py:269-272),
 * and, with transposed weight blocks, their input gradients. */
int scann_dense_forward(const float* const* A, int lda, const float* const* W, const float* const* bias, int kblk,
                        int nblk, int R, float* C, int ldc, int mode, const float* resid, int ldres,
                        const float* pre_in, float* pre_out, const float* gamma, const float* beta, void* stream);
/* Same contract on the tcgen05 tensor cores (3xTF32, weights stationary in tensor memory). */
int scann_dense_forward_tc(const float* const* A, int lda, const float* const* W, const float* const* bias,
                           int kblk, int nblk, int R, float* C, int ldc, int mode, const float* resid, int ldres,
                           const float* pre_in, float* pre_out, const float* gamma, const float* beta,
                           void* stream);
/* dW[kb*nblk+nb] += A[kb]^T @ G[nb] ; db[nb] += colsum(G[nb])  (TF autodiff of Dense). */
int scann_dense_wgrad(const float* const* A, int lda, const float* const* G, int ldg, int kblk, int nblk, int R,
                      float* const* dW, float* const* db, void* stream);
/* LayerNormalization backward; dv2 (row stride ld2) optionally receives a second copy of dv. */
int scann_layernorm_backward(const float* dy, const float* v, const float* gamma, int R, float* dv, float* dv2,
                             int ld2, float* dgamma, float* dbeta, void* stream);
/* Atoms with no valid neighbour: context = q, out = LN(q) (attention.py:206-214). */
int scann_la_nopair_forward(const int32_t* cnt, const float* proj, int R, const float* gamma, const float* beta,
                            float* ctx_pre, float* out, void* stream);
/* dst[off..] = transpose(src[off..]) for each listed 128x128 block (offsets: device int32). */
int scann_transpose_blocks(const float* src, float* dst, const int32_t* offsets, int nblocks, void* stream);

/* ---- chains of per-atom Dense layers in one kernel ----------------------------------------------
 * Rows (atoms) are independent in every per-atom layer, so the kernels between two local-attention layers
 * are fused: ResidualNorm (attention.py:25-40) + the next layer's x @ [W1|W3|Wq] projections
 * (attention.py:141-161) + "context = q" for atoms without neighbours (attention.py:206-214) in the forward
 * pass, and their transposes with LayerNorm backward / swish' in the backward pass.  A CTA carries its rows
 * through up to 6 steps; step i computes
 *     V = sum_kb A[kb] @ W[kb] + bias (+ resid)
 *     mode 0: out = V | 1: pre_out <- V, out = swish(V) | 2: out = V * swish'(pre_in)
 *          3: pre_out <- V, out = LayerNorm(V; gamma, beta, eps 1e-6)
 *          4: out = LayerNorm-backward(dy = V; forward value pre_in, gamma); dgamma, dbeta accumulated
 *     C, C2 <- out (nullable);  to_image: out is the A operand of step i+1 (that step has A[0] = NULL, kblk 1;
 *     an operand loaded from global memory also stays resident for later steps with A[0] = NULL).
 *     cnt != NULL: rows with cnt[r] == 0 additionally get np_ctx[r] = V, np_out[r] = LayerNorm(V; gamma, beta).
 *     drop != NULL (training-mode keras Dropout, attention.py:29, rate 0.1): modes 0-3 multiply (sum + bias) by the
 *     site's mask before the residual is added; mode 4 writes out to C and out * mask to C2 and the image.
 *     The mask is a hash of (seed, site, row * 128 + column) kept/scaled per the DEVICE control block
 *     ScannDropCtl {uint32 seed, threshold = rate * 2^32, float bits of 1/(1-rate), enabled}.
 * `steps` is a HOST array of nsteps structs holding device pointers. */
typedef struct ScannChainStep {
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
    const void* drop;      /* ScannDropCtl* (device) or NULL: training-mode Dropout of site drop_site, see below */
    int lda, ldres, ldpre, ldc, ldc2;
    int kblk;
    int mode;
    int to_image;
    int drop_site;
    int pad;
} ScannChainStep;
int scann_dense_chain(const ScannChainStep* steps, int nsteps, int R, void* stream);

/* Warp-specialised form of scann_dense_chain (chain2_tc.cu): same steps, same arithmetic, same reference lines
 * (attention.py:25-40,141-161,206-214; scann_model.py:424-429), but W[kb] of every step points to the WEIGHT IMAGE of
 * the 128x128 block instead of the block itself.  scann_weight_images writes the images of `nblocks` blocks of the
 * parameter arena (offsets[b] = element offset of block b, row-major [in,out]) into `images`
 * ([nblocks][2][32768] floats, 1024-byte aligned): orientation 0 is the operand of x @ W, orientation 1 of x @ W^T
 * (what the backward pass multiplies with) -- four K-blocks of [tf32-truncated | remainder] chunk blocks in the
 * 128-byte-swizzled K-major tcgen05 layout, streamed into shared memory with cp.async.bulk.  Call it after every change
 * of the parameters.  scann_dense_chain2_max_rows() = the rows one wave covers (64 per SM); more rows run in several waves.
 * status (nullable): 8 device ints; a bounded wait that gives up ORs 16 into word 0 and leaves {site 41..47, CTA, step / block,
 * buffer} in words 1..4, as the pipelined local-attention kernels do. */
int scann_weight_images(const float* params, const int32_t* offsets, int nblocks, float* images, void* stream);
int scann_dense_chain2(const ScannChainStep* steps, int nsteps, int R, int32_t* status, void* stream);
int scann_dense_chain2_max_rows(void);

/* ---- local attention (the hot kernel) ---------------------------------------------------------
 * LocalAttention.call, g_update=True, v_proj=False, kq_proj=True (scann/layers/attention.py:118-216).
 * proj = [x@W1+bf | x@W3 | x@Wq+bq] ([R,384]); W2 = rows 128..255 of filter_geo/kernel.
 * Outputs: g_out (geometry'), out = LN(context) [R,128], ctx_pre (nullable, pre-LN context),
 * attn (nullable) [rows,8] softmax weights.  grid: number of CTAs (<= SM count is sensible). */
int scann_la_forward(int grid, const int32_t* ntiles, const int32_t* tile_a0, const int32_t* tile_a1,
                     const int32_t* cnt, const int32_t* rowptr, const int32_t* pair_c, const int32_t* pair_j,
                     const float* x, const float* proj, const float* g_in, const float* W2, const float* Wk,
                     const float* bk, const float* gamma_g, const float* beta_g, const float* gamma,
                     const float* beta, float* g_out, float* ctx_pre, float* out, float* attn, void* stream);
/* Same forward on the tcgen05 tensor cores (3xTF32; two kernels: geometry update, attention).
 * pre_out / k_out ([rows,128], nullable) save the filter_geo pre-activation and the keys. */
int scann_la_forward_tc(int grid, int tile_stride, int mma_rows, const int32_t* ntiles, const int32_t* tile_a0, const int32_t* tile_a1,
                        const int32_t* cnt, const int32_t* rowptr, const int32_t* pair_c, const int32_t* pair_j,
                        const float* x, const float* proj, const float* g_in, const float* W2, const float* Wk,
                        const float* bk, const float* gamma_g, const float* beta_g, const float* gamma,
                        const float* beta, float* g_out, float* ctx_pre, float* out, float* attn, float* pre_out,
                        float* k_out, const void* attn_drop, int drop_site, void* stream);
/* The same forward as two warp-specialised, TMA-fed pipelines (la_pipe.cu) for pair plans with tile_stride 32
 * (at most 32 valid neighbours per atom): a producer warp streams the tiles of g through a six-stage shared-memory
 * ring with cp.async.bulk.tensor (and gathers the neighbour rows x[j] with cp.async), two consumer groups of eight
 * warps split each tile into its hi / lo operand images, issue its three tcgen05.mma product chains and run the
 * row-wise epilogue in place, and a store warp writes the finished tiles back with TMA.
 * rows = tile_cap * 32 (row count of every per-pair tensor; per-pair tensors must be 128-byte aligned).
 * which: bit 0 = geometry kernel, bit 1 = attention kernel.  status: the engine's int32[8] status buffer (word 0:
 * flag bits, SCANN_ERR_PIPE_TIMEOUT = 16 when a bounded mbarrier wait gave up; words 1..4: where). */
int scann_la_forward_pipe(int grid, long long rows, int which, const int32_t* ntiles, const int32_t* pair_c,
                          const int32_t* pair_j, const float* x, const float* proj, const float* g_in,
                          const float* W2, const float* Wk, const float* bk, const float* gamma_g,
                          const float* beta_g, const float* gamma, const float* beta, float* g_out, float* ctx_pre,
                          float* out, float* attn, float* pre_out, float* k_out, const void* attn_drop,
                          int drop_site, int32_t* status, void* stream);
/* attn_drop (ScannDropCtl*, device, nullable) / drop_site: training-mode Dropout(0.05) on the attention
 * probabilities of use_drop models (attention.py:115-116,191-192); mask index = pair row * 8 + head. */
/* LocalAttention.call with g_update=False (attention.py:155): geometry' = swish(rbf(d) @ Wf + bf) * w is
 * recomputed per layer from pair_d / pair_w; proj needs only its query block.  Inference only. */
int scann_la_forward_noupdate_tc(int grid, int tile_stride, int mma_rows, const int32_t* ntiles, const int32_t* tile_a0, const int32_t* tile_a1,
                                 const int32_t* cnt, const int32_t* rowptr, const int32_t* pair_c,
                                 const int32_t* pair_j, const float* x, const float* proj, const float* pair_d,
                                 const float* pair_w, const float* centers, const float* Wf, const float* bf,
                                 const float* Wk, const float* bk, const float* gamma, const float* beta,
                                 float* ctx_pre, float* out, float* attn, float* g_save, float* k_out, const void* attn_drop, int drop_site, void* stream);
/* Backward of the g_update=False layer: attention part (g_new / kbuf = g' / keys saved by the forward; kbuf <- d_k,
 * dg <- gradient w.r.t. g', dq / dx_scatter as in scann_la_backward_tc) ... */
int scann_la_backward_noupdate_tc(int grid, int tile_stride, int mma_rows, const int32_t* ntiles, const int32_t* tile_a0,
                                  const int32_t* tile_a1, const int32_t* cnt, const int32_t* rowptr, const int32_t* pair_c,
                                  const int32_t* pair_j, const float* x, const float* proj, const float* g_new,
                                  float* kbuf, const float* WkT, const float* d_ctx, float* dg, float* dq,
                                  float* dx_scatter, float* dbk, const void* attn_drop, int drop_site, void* stream);
/* g' = swish(rbf(d) @ Wf + bf) * w of a g_update=False layer (attention.py:155) written out as a
 * [tile_cap * tile_stride, 128] tensor (padding rows zero): the geometry operand of scann_la_forward_pipe (which = 2)
 * and scann_la_backward_pipe (which = 1) when such a layer runs on the pipelined attention kernels. */
int scann_noupdate_geom_forward(const int32_t* ntiles, int grid, int tile_stride, const int32_t* pair_c,
                                const float* pair_d, const float* pair_w, const float* centers_d, const float* Wf,
                                const float* bf, float* g_out, void* stream);
/* ... and the gradient of its geometry filter g' = swish(rbf(d) @ Wf + bf) * w: dWf [20,128], dbf accumulated. */
int scann_noupdate_geom_backward(const int32_t* ntiles, int grid, int tile_stride, const int32_t* pair_c,
                                 const float* pair_d, const float* pair_w, const float* centers_d, const float* Wf,
                                 const float* bf, const float* dg, float* dWf, float* dbf, void* stream);
/* Reverse-mode of the above (TF autodiff inside keras fit, scann_model.py:232-241).  d_ctx is the
 * gradient w.r.t. the pre-LN context; dq/s_pre are written for atoms with pairs, t_scatter /
 * dx_scatter are accumulated with atomics (pre-zero them); wpart: grid*2*128*128 floats. */
int scann_la_backward(int grid, const int32_t* ntiles, const int32_t* tile_a0, const int32_t* tile_a1,
                      const int32_t* cnt, const int32_t* rowptr, const int32_t* pair_c, const int32_t* pair_j,
                      const float* x, const float* proj, const float* g_in, const float* W2, const float* Wk,
                      const float* W2T, const float* WkT, const float* bk, const float* gamma_g,
                      const float* beta_g, const float* d_ctx, const float* dg_up, float* dg_out, float* dq,
                      float* s_pre, float* t_scatter, float* dx_scatter, float* wpart, float* dgamma_g,
                      float* dbeta_g, float* dbk, void* stream);
/* Same backward on the tcgen05 tensor cores (three kernels: attention, geometry, pair weight gradients).
 * kbuf / prebuf: in = keys / filter_geo pre-activation saved by scann_la_forward_tc, out = d_k / d_pre.
 * dg: gradient w.r.t. g' from the next layer (dg_has_up != 0, updated in place) or scratch.
 * Two kernels (attention, geometry); the pair weight gradients are scann_la_wgrad_tc. */
int scann_la_backward_tc(int grid, int tile_stride, int mma_rows, const int32_t* ntiles, const int32_t* tile_a0, const int32_t* tile_a1,
                         const int32_t* cnt, const int32_t* rowptr, const int32_t* pair_c, const int32_t* pair_j,
                         const float* x, const float* proj, const float* g_in, const float* g_new, float* kbuf,
                         float* prebuf, const float* W2T, const float* WkT, const float* gamma_g, const float* d_ctx,
                         float* dg, int dg_has_up, float* dg_out, float* dq, float* s_pre, float* t_scatter,
                         float* dx_scatter, float* wpart, float* dgamma_g, float* dbeta_g, float* dbk, const void* attn_drop, int drop_site, void* stream);
/* One half of scann_la_backward_tc: which bit 0 = attention kernel, bit 1 = geometry kernel. */
int scann_la_backward_tc_part(int which, int grid, int tile_stride, int mma_rows, const int32_t* ntiles, const int32_t* tile_a0, const int32_t* tile_a1,
                         const int32_t* cnt, const int32_t* rowptr, const int32_t* pair_c, const int32_t* pair_j,
                         const float* x, const float* proj, const float* g_in, const float* g_new, float* kbuf,
                         float* prebuf, const float* W2T, const float* WkT, const float* gamma_g, const float* d_ctx,
                         float* dg, int dg_has_up, float* dg_out, float* dq, float* s_pre, float* t_scatter,
                         float* dx_scatter, float* wpart, float* dgamma_g, float* dbeta_g, float* dbk, const void* attn_drop, int drop_site, void* stream);
/* The same backward as two warp-specialised, TMA-fed pipelines (la_pipe_bwd.cu) for pair plans with tile_stride 32
 * (see scann_la_forward_pipe): the tiles of k / g' / pre / g / dg' arrive by TMA, x[j] by cp.async, d_k / d_pre / dg
 * leave by TMA stores (dg by a TMA reduce-add when dg_has_up).  rows = tile_cap * 32; which: bit 0 attention kernel,
 * bit 1 geometry kernel. */
int scann_la_backward_pipe(int grid, long long rows, int which, const int32_t* ntiles, const int32_t* pair_c,
                           const int32_t* pair_j, const float* x, const float* proj, const float* g_in,
                           const float* g_new, float* kbuf, float* prebuf, const float* W2T, const float* WkT,
                           const float* gamma_g, const float* d_ctx, float* dg, int dg_has_up, float* dg_out, float* dq,
                           float* s_pre, float* t_scatter, float* dx_scatter, float* dgamma_g, float* dbeta_g,
                           float* dbk, const void* attn_drop, int drop_site, int32_t* status, void* stream);
/* Pair weight gradients of one layer (3xTF32, MN-major operands) into wpart[grid][2][128][128]:
 * slot 0 = (x[j]*g')^T d_k (key/kernel), slot 1 = g^T d_pre (filter_geo rows 128..255).  Needs the d_k /
 * d_pre that scann_la_backward_tc left in kbuf / prebuf; off the critical path (side stream). */
int scann_la_wgrad_tc(int grid, int tile_stride, const int32_t* ntiles, const int32_t* pair_c, const int32_t* pair_j, const float* x,
                      const float* g_in, const float* g_new, const float* dk, const float* dpre, float* wpart,
                      void* stream);
/* dWk += sum_cta wpart[cta][0] ; dW2 += sum_cta wpart[cta][1]  (per-CTA partial weight gradients). */
int scann_la_wpart_reduce(const float* wpart, const int32_t* ntiles, int grid, int tile_stride, float* dWk, float* dW2,
                          void* stream);

/* ---- all weight-gradient GEMMs of a train step in one persistent launch ---------------------------
 * dW += X^T Y for a list of problems (TF autodiff of every Dense / einsum kernel of the graph inside keras fit:
 * scann/layers/attention.py:118-216,25-40, scann/models/scann_model.py:424-447).  rows >= 0: per-atom problem
 * over that many rows; rows < 0: per-pair problem over the tile-padded pair rows (ntiles * tile_stride rows, rows
 * with pair_c < 0 skipped; or, when the plan's compact list valid_rows / nvalid is given, exactly the valid rows),
 * with X rows multiplied by xg[pair_j[row]] when xg != NULL.  db (nullable) += column
 * sums of Y (bias gradient).  `problems` is a DEVICE array; results are accumulated with atomics. */
typedef struct ScannWgradProblem {
    const float* X;
    const float* Y;
    const float* xg;
    float* dW;
    float* db;
    int ldx, ldy;
    int rows;
    int pad;
} ScannWgradProblem;
int scann_wgrad_batch_tc(int grid, const ScannWgradProblem* problems, int nprob, const int32_t* ntiles, int tile_stride,
                         const int32_t* pair_c, const int32_t* pair_j, const int32_t* valid_rows, const int32_t* valid_j,
                         const int32_t* nvalid, void* stream);

/* ---- global attention + property head ---------------------------------------------------------
 * GlobalAttention.call (scann/layers/attention.py:267-318) + bf_property / predict_property / mrelu
 * (scann/models/scann_model.py:437-447, scann/layers/custom_layers.py:6-15).  qk = [q | k] [R,256].
 * Outputs ga [R] (ga_score), y [B]; ctx_out / tb_out [B,128] nullable (saved for backward). */
int scann_ga_head_forward(const float* qk, const uint8_t* atom_mask, int B, int M, int norm, const float* Wb,
                          const float* bb, const float* wp, const float* bp, int mrelu, float* ga, float* y,
                          float* ctx_out, float* tb_out, void* stream);
int scann_ga_head_backward(const float* qk, const uint8_t* atom_mask, int B, int M, int norm, const float* WbT,
                           const float* wp, const float* tb, const float* dy, float* d_qk, float* d_tb, float* dwp,
                           float* dbp, void* stream);

/* ---- loss and optimiser -----------------------------------------------------------------------
 * root_mean_squared_error (scann/layers/losses.py:5-6): dy_b = y_b - t_b, sse[0] += sum err^2,
 * sse[1] += sum |err|; the 1/(B*RMSE) factor is applied in scann_adam_step after the gradient
 * all-reduce; scann_adam_step also accumulates sse[2] += sum(l2mask * w^2) for scann_loss_value.  Adam(lr, decay=1e-5) + l2(1e-4) regulariser gradient (scann_model.py:212). */
int scann_rmse_prepare(const float* y, const float* target, int B, float* dy, float* sse, void* stream);
int scann_adam_step(float* params, const float* grads, float* m, float* v, const float* l2mask, int n,
                    float* sse, const void* scalars_dev, float* grad_out, int apply, void* stream);
int scann_loss_value(const float* params, const float* l2mask, int n, const float* sse, float batch, float l2,
                     float* out3, void* stream);

/* ---- Voronoi neighbour lists (the model's input) -------------------------------------------------------------
 * compute_voronoi_neighbor (scann/utils/voronoi_neighbor.py:11-61): pymatgen VoronoiNN(weight="solid_angle", tol=0)
 * .get_voronoi_polyhedra + _extract_nn_info for every listed centre, in fp64, one warp per centre (voronoi.cu).
 * Structures: lattice [S,9] (rows = lattice vectors), coords [A,3] Cartesian, struct_atom_off [S+1] int32.
 * Centres: centre_atom [C] (global atom row), centre_struct [C], cutoff [C] (Angstrom; the point set is every image
 * within it).  allow_pathological: emit the finite facets of a cell that also has unbounded ones (otherwise such a
 * centre emits nothing and carries flag 1: pymatgen's caller widens its cutoff and runs it again).
 * slots: C * cap records of scratch (cap <= 64), slot_count [C] int32.  The result goes to `blob` (device):
 *   int32 off[C+1] (CSR), int32 flags[C] (1 = unbounded facet, plus the SCANN_ERR_VORONOI_* bits of that centre),
 *   zero padding to a multiple of 32 bytes, then ScannVoronoiFacet records (centre c: off[c] .. off[c+1]);
 *   blob bytes >= round_up(4 * (2C + 1), 32) + 32 * C * cap.
 * Records of a centre: its finite facets with solid angle > 0, in no particular order.  host_blob (nullable, host,
 * pinned for an asynchronous copy) receives the whole blob with one cudaMemcpyAsync on `stream`.
 * status [0] |= SCANN_ERR_VORONOI_*: two points of a cell closer than 1e-8 Angstrom, a capacity of the kernel
 * exceeded (64 facets, 32 vertices per facet, 128 points of one distance shell, |image| <= 511), a centre without a
 * finite facet, a cut whose facet boundary is not one cycle (numerically inconsistent input). */
#define SCANN_ERR_VORONOI_COINCIDENT 32
#define SCANN_ERR_VORONOI_CAPACITY 64
#define SCANN_ERR_VORONOI_NO_FACET 128
#define SCANN_ERR_VORONOI_TOPOLOGY 256
typedef struct ScannVoronoiFacet {
    double solid_angle;   /* pymatgen's fan formula over the facet's vertices, seen from the centre */
    double normalized;    /* solid_angle / the largest solid angle of the centre's cell */
    double distance;      /* |x_j + n L - x_i| */
    int32_t site;         /* j, index within the structure */
    int32_t image;        /* n packed as (n0 + 512) | (n1 + 512) << 10 | (n2 + 512) << 20 */
} ScannVoronoiFacet;
int scann_voronoi_neighbors(const double* lattice, const double* coords, const int32_t* struct_atom_off,
                            const int32_t* centre_atom, const int32_t* centre_struct, const double* cutoff,
                            int n_centres, int allow_pathological, int cap, void* slots, int32_t* slot_count,
                            void* blob, void* host_blob, int32_t* status, void* stream);

/* ---- NCCL gradient all-reduce (SURVEY.md 8b / 8e) ---------------------------------------------------------------
 * One process per GPU, one communicator per process.  Rank 0: scann_allreduce_unique_id(out128) -> 128 HOST bytes
 * (ncclUniqueId) that the caller sends to the other ranks; every rank, with its device current:
 * scann_allreduce_init(id128, rank, world) (collective); per step scann_allreduce_sum(arena, n + 4, stream) between the
 * backward pass and scann_adam_step (in place, asynchronous, capturable into the step's CUDA graph);
 * scann_allreduce_destroy at the end.  libnccl.so.2 is dlopen'ed on first use (the copy already loaded in the process,
 * e.g. PyTorch's, else the system one): the library itself does not link against NCCL. */
int scann_allreduce_unique_id(void* out128);
int scann_allreduce_init(const void* id128, int rank, int world);
int scann_allreduce_sum(float* buf, long long count, void* stream);
int scann_allreduce_world(void);
int scann_allreduce_destroy(void);

/* ---- gradient exchange over NVLink peer memory, fused into the optimiser -------------------------------------
 * Data-parallel training (one process per GPU; the reference trains on one device, scann_model.py:232-241): instead of
 * an NCCL all-reduce followed by scann_adam_step, every rank keeps its gradient arena in a block that the other ranks
 * of the node map through CUDA IPC, and the optimiser kernel sums the peers' arenas itself (fixed rank order, so
 * the parameters stay bit-identical on all ranks).  Block = [n + 4 floats, padded to 64] [64 x uint32 flag words];
 * scann_p2p_alloc returns it zeroed.  ScannP2PBlock (device copy passed as block_dev):
 *   const float* arena[8]; uint32_t* flags[8]; int world, rank;      (entry `rank` = the local block)
 * Per step: scann_p2p_begin_step (waits until no peer still reads the local arena, zeroes sums[0..3]) -> zero the
 * arena, forward, backward -> scann_adam_p2p_step (publishes / waits for "backward finished" flags, sums, updates,
 * publishes "finished reading").  sums[0..2] = what scann_adam_step leaves in sse[0..2] (pass it to scann_loss_value).
 * All waiting happens inside the kernels, so the sequence can be captured into a CUDA graph. */
int scann_p2p_alloc(long long bytes, void** out_ptr);
int scann_p2p_free(void* ptr);
int scann_p2p_export(void* ptr, void* handle64);
int scann_p2p_import(const void* handle64, void** out_ptr);
int scann_p2p_close(void* ptr);
int scann_p2p_begin_step(const void* block_dev, float* sums, void* stream);
int scann_adam_p2p_step(float* params, float* m, float* v, const float* l2mask, int n, const void* block_dev,
                        float* sums, const void* scalars_dev, float* grad_out, int apply, void* stream);

/* ---- development probes ------------------------------------------------------------------------
 * Exported only by development builds (nvcc -DSCANN_DEV_PROBES; the production library carries neither these entry
 * points nor the timestamp stores inside its kernels).
 * scann_tc_probe: one 128x128x128 tile product on the tcgen05 tensor cores (self-test of descriptors / layouts).
 * layout 0: A@W, 1: A^T@W, 2: A@W^T, 3: A@W with A in tensor memory; nprod 1 (TF32) or 3 (3xTF32).
 * scann_tc_time: out[0] = cycles per tcgen05.mma (128 x ncols x 8, tf32) in a chain of nmma accumulating MMAs; mode
 * bit 0: A from tensor memory, bit 1: core-matrix stride 128 B, bit 4: round-robin over (mode >> 8) accumulators.
 * scann_debug_clocks*: phase timestamps (clock64) of CTA 0 of the last la_geom_fwd_tc / dense_tc / dense_chain launch;
 * scann_pipe_clocks: of consumer group 0 of the last la_geom_fwd_pipe launch (96 int64, HOST). */
#ifdef SCANN_DEV_PROBES
int scann_tc_probe(const float* A, const float* W, float* D, int layout, int nprod, void* stream);
int scann_tc_time(float* out, int mode, int nmma, int ncols, void* stream);
int scann_debug_clocks(long long* host_out32);
int scann_debug_clocks_dense(long long* host_out16);
int scann_debug_clocks_chain(long long* host_out64);
int scann_debug_clocks_chain2(long long* host_out192);
int scann_pipe_clocks(long long* host_out96);
int scann_pipe_clocks_bwd(long long* host_out96);
#endif

#ifdef __cplusplus
}
#endif
#endif
