/*
 * vcr_b200 -- C ABI of the B200-native (sm_100a) VCR-Net registration inference path.
 *
 * The reference (qiaozhijian/VCR-Net) is pure Python/PyTorch and has no FFI or operator
 * registry: its hot path reaches the GPU only through ATen calls inside the functions cited
 * below.  Each entry point here replaces the ATen call sequence of one such call site.  The
 * host side stays Python (vcr_net_b200/, same class / function names as the reference) and
 * binds this header through ctypes (vcr_net_b200/_lib.py parses THIS file for the signatures).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer (fp32 unless stated), caller-allocated, never retained;
 *   - no hidden allocation and no synchronisation; calls are thread-safe and asynchronous on `stream` of the
 *     CURRENT device (nn.DataParallel's per-device threads).  The only process-wide state is (a) the launch
 *     counter, (b) three atomic TUNING knobs that select between bit-identical kernel variants
 *     (vcr_set_gemm_pair, vcr_set_flash_warps, vcr_set_knn3_direct) and (c) per-device caches of idempotent
 *     device queries, published with release/acquire atomics -- nothing a result depends on;
 *   - workspace comes from the caller; query its size with the matching *_workspace_bytes();
 *   - return value: 0 = VCR_OK, < 0 = error (the Python wrapper raises RuntimeError):
 *       -1 invalid argument / alignment, -2 unsupported shape, -3 launch failure, -4 workspace;
 *   - "token-major" = [B, N, C] row-major (a point's channels contiguous); "channel-major" =
 *     the reference's [B, C, N].
 * Reference citations are relative to the reference repository root.
 */
#ifndef VCR_B200_H
#define VCR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __CUDA_RUNTIME_H__
typedef struct CUstream_st* cudaStream_t;
#endif

/* ---- bookkeeping --------------------------------------------------------------------------------
 * vcr_launch_count: kernels launched by this library in this process so far (bench.py gpu_launches). */
long long vcr_launch_count(void);
int vcr_abi_version(void);

/* ---- kNN graph: util/util.py:143-160 knn(x,k) -------------------------------------------------
 * pd_ij = (-xx_j - (-2 x_i.x_j)) - xx_i, neighbours = ranks 1..k of the descending order (rank 0
 * dropped exactly like `topk(k+1)[..., 1:]`), ties -> lower index.  x: [B,D,N] (token_major=0) or
 * [B,N,D] (token_major=1); any D (fast paths for 3 and 64); 1<=k<=31; idx32 / idx64: [B,N,k], either may be NULL. */
size_t vcr_knn_workspace_bytes(int B, int N);
int vcr_knn_topk(const float* x, int B, int D, int N, int k, int token_major, int32_t* idx32,
                 int64_t* idx64, void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* D == 3 route of vcr_knn_topk: 1 (default) = distances evaluated on the fly from x|y|z|xx rows in shared memory
 * (4 CTAs per SM), 0 = the generic distance-tile kernel.  Bit-identical indices; returns the previous setting. */
int vcr_set_knn3_direct(int on);
/* Selection of the tensor-core route (vcr_knn_topk_tc): 0 = warp-per-query from a shared-memory distance tile, 1 =
 * thread-per-query straight from TMEM (queries on the M side of the MMA, register sorting networks; csrc/knn_tpq.cuh),
 * 2 (default) = thread-per-query from N >= 8192, where it measured faster.  Bit-identical indices; returns the
 * previous setting. */
int vcr_set_knn_tc_tpq(int on);

/* Tensor-core variant of the same function for feature-space kNN (16 <= D <= 128, k <= 30, token-major only):
 * tcgen05 distance tiles from the operand-format copy of x ([2 planes][B*N][ld] fp16 hi / lo*2^11, vcr_to_operand)
 * prefilter ranks 0..k+8, the survivors are re-ranked with the canonical fp32 chain and certified per query
 * (error bound eps on the approximate distances); uncertified 32-query groups are recomputed by the exact kernel in
 * the same launch sequence.  Output bit-identical to vcr_knn_topk on every input.  The last 4 bytes of the workspace
 * hold the number of queries that needed the exact kernel (telemetry). */
size_t vcr_knn_tc_workspace_bytes(int B, int N);
int vcr_knn_topk_tc(const float* x, const void* xop, int ld, long long plane_stride, int B, int D, int N, int k,
                    int32_t* idx32, int64_t* idx64, void* workspace, size_t workspace_bytes, cudaStream_t stream);
/* Ragged batches of both: item b holds n[b] real points (int32, device; clamped to [k+1, N]) in its N rows, the rest is
 * padding of any value.  Candidates j >= n[b] are never ranked, the tensor-core certificate's max |x|^2 is taken over the
 * real points, and the indices of a real query equal those of vcr_knn_topk / vcr_knn_topk_tc on the item alone.  A padded
 * query (n[b] <= q < N) gets its own index q in all k slots, so EdgeConv / gather-max over the graph stay in bounds.  The
 * lengths are read on the device only (no host sync): a captured graph can be replayed with new lengths.  Same workspace
 * sizes and the same vcr_set_knn3_direct / vcr_set_knn_tc_tpq routes. */
int vcr_knn_topk_ragged(const float* x, const int* n, int B, int D, int N, int k, int token_major, int32_t* idx32,
                        int64_t* idx64, void* workspace, size_t workspace_bytes, cudaStream_t stream);
int vcr_knn_topk_tc_ragged(const float* x, const void* xop, int ld, long long plane_stride, const int* n, int B, int D,
                           int N, int k, int32_t* idx32, int64_t* idx64, void* workspace, size_t workspace_bytes,
                           cudaStream_t stream);

/* ---- get_graph_feature: util/util.py:176-199 ---------------------------------------------------
 * xt token-major [B,N,D]; idx [B,N,k]; out [B,2D,N,k] contiguous = concat(x[idx], x centre). */
int vcr_graph_feature(const float* xt, int B, int D, int N, int k, const int* idx, float* out,
                      cudaStream_t stream);

/* ---- FPS: util/util.py:107-140 farthest_point_sample (== util/fps.py:10-49) ---------------------
 * xyz [B,3,N] -> idx [B,npoint]; N <= 229 376 (one CTA per cloud up to 14 336 points, beyond that one thread-block
 * cluster of 2, 4, 8 or 16 CTAs per cloud; -2 above 229 376 or when the device cannot co-schedule the cluster). */
int vcr_fps(const float* xyz, int B, int N, int npoint, int32_t* idx32, int64_t* idx64, cudaStream_t stream);

/* ---- generic fp32 GEMM with fused epilogue -------------------------------------------------------
 * Replaces nn.Conv1d/Conv2d(kernel 1)/nn.Linear (model/lpdnet_model.py:111-135,
 * model/transformer.py:210-224,238) and the torch.matmul calls of attention
 * (model/transformer.py:30,55) and of the VCP head (model/vcrnet_model.py:337).
 * C[z] = act(alpha * A[z](MxK) * op(B[z]) + bias[n]) + residual[z][m,n];  b_layout 0: B is [N,K],
 * 1: B is [K,N]; z = outer*nb_inner + inner with element strides s?o / s?i; act 0 none, 1 LeakyReLU. */
int vcr_gemm_f32(const float* A, int lda, long long sAo, long long sAi,
                 const float* B, int ldb, long long sBo, long long sBi, int b_layout,
                 float* C, int ldc, long long sCo, long long sCi,
                 const float* bias, const float* residual, int ldr, long long sRo, long long sRi,
                 int M, int N, int K, int nb_outer, int nb_inner,
                 float alpha, int act, float slope, cudaStream_t stream);

/* ---- tensor-core GEMM (tcgen05 + TMEM + TMA) --------------------------------------------------------
 * Same call sites as vcr_gemm_f32, on "operand-format" inputs: 16-bit K-major buffers laid out
 * [planes][rows][ld]; plane 0 = hi = fp16(x), plane 1 = lo = fp16((x-hi)*2^11) (mode 0, the fp32-parity
 * 3-term split); modes 1 / 2 = single-plane fp16 / bf16 (throughput modes).  Per batch z = (zo, zi) the A rows
 * start at zo*a_row_o + zi*a_row_i and the K range at column zo*a_col_o + zi*a_col_i (same for B), which
 * addresses attention heads inside fused projection buffers without copies.  Outputs, each optional:
 * C fp32 (+ residual R); H operand-format row-major for columns < h_split; HT operand-format transposed
 * ([plane][col - h_split][row]) for columns >= h_split.  vcr_to_operand converts fp32 -> operand format. */
int vcr_gemm_tc(const void* A, int lda, long long a_rows_total, int a_cols_total, long long a_plane,
                long long a_row_o, long long a_row_i, int a_col_o, int a_col_i,
                const void* B, int ldb, long long b_rows_total, int b_cols_total, long long b_plane,
                long long b_row_o, long long b_row_i, int b_col_o, int b_col_i,
                int M, int N, int K, int nb_outer, int nb_inner, int mode,
                float alpha, const float* bias, int act, float slope,
                float* C, int ldc, long long c_so, long long c_si,
                const float* R, int ldr, long long r_so, long long r_si,
                void* H, int ldh, long long h_plane, long long h_so, long long h_si, int h_split,
                void* HT, int ldt, long long t_plane, long long t_so, long long t_si,
                int out_planes, cudaStream_t stream);
/* Flash-style multi-head attention (model/transformer.py:13-55) on tcgen05/TMEM: softmax(Q K^T scale) V, d_k = 128,
 * scores and probabilities never leave the SM.  Q [planes][B*Nq][ldq] (head hh = columns hh*128..), K likewise
 * with B*Nk rows, VT [planes][B*H*128][ldv] (row (b*H+hh)*128+d, Nk key columns), O like Q.  keep: optional
 * uint8 [B,Nk] key mask (masked keys get -1e9, :51-52); lse: optional [B,H,Nq] log2-domain log-sum-exp. */
int vcr_flash_attn_tc(const void* Q, int ldq, long long q_plane, const void* K, int ldk, long long k_plane,
                      const void* VT, int ldv, long long v_plane, int B, int H, int Nq, int Nk, int dk,
                      int mode, float scale, const uint8_t* keep, void* O, int ldo, long long o_plane,
                      float* lse, cudaStream_t stream);
/* Ragged batch: item b has nq[b] queries and nk[b] keys (int32, device; clamped to [1, Nq] / [1, Nk]) in its Nq / Nk
 * rows.  Key tiles past nk[b] are not loaded, keys past nk[b] in the last tile get -inf whatever their score (the tail
 * treatment of a call with Nk = nk[b]), and a 128-query tile wholly past nq[b] is written as zeros after one key tile.
 * Output rows of real queries equal vcr_flash_attn_tc on the item alone bit for bit, provided the padded V columns of the
 * item's last key tile are finite (their probabilities are exactly 0).  Runs organisation 3 whatever vcr_set_flash_warps
 * says (2 gives the same bits); no key mask, no lse. */
int vcr_flash_attn_tc_ragged(const void* Q, int ldq, long long q_plane, const void* K, int ldk, long long k_plane,
                             const void* VT, int ldv, long long v_plane, const int* nq, const int* nk, int B, int H,
                             int Nq, int Nk, int dk, int mode, float scale, void* O, int ldo, long long o_plane,
                             cudaStream_t stream);
/* vcr_flash_attn_tc_ragged with the partial-overlap key mask keep [B, Nk] (uint8, row stride Nk): a key of item b with
 * keep == 0 gets -1e9 (:51-52), a key past nk[b] gets -inf whatever keep holds.  Rows of real queries equal
 * vcr_flash_attn_tc with keep = the item's first nk[b] mask bytes on the item alone, bit for bit (same finiteness condition). */
int vcr_flash_attn_tc_ragged_keep(const void* Q, int ldq, long long q_plane, const void* K, int ldk, long long k_plane,
                                  const void* VT, int ldv, long long v_plane, const int* nq, const int* nk,
                                  const uint8_t* keep, int B, int H, int Nq, int Nk, int dk, int mode, float scale, void* O,
                                  int ldo, long long o_plane, cudaStream_t stream);
/* Organisation of vcr_flash_attn_tc: 3 (default) = Q and P in tensor memory (tcgen05.mma with the A operand in TMEM; P is
 * written over the S tile it came from), 8 softmax warps; 2 = every operand in shared memory, 8 warps on every key tile
 * (same bits as 3); 4 = 16 warps; 1 = two groups of 4 warps alternating key tiles.  Process-wide tuning knob; returns the
 * previous setting. */
int vcr_set_flash_warps(int nwq);
/* Process-wide policy for the mode-0 GEMMs on CTA pairs (tcgen05 cta_group::2, 256 x 128 tile per pair of SMs, each
 * CTA staging half of the B tile): 0 never, 1 always, 2 auto (default: pairs except for the residual epilogue at
 * K < 1024).  Same results bit for bit; returns the previous setting. */
int vcr_set_gemm_pair(int on);
/* Policy 3: clusters of two pairs working on the same 256 rows, the A tile multicast between them.  This returns how many
 * such 4-CTA clusters the device co-schedules (0: unsupported; policy 3 then behaves like 1). */
int vcr_gemm_quad_clusters(void);
int vcr_to_operand(const float* x, int ld, long long rows, int cols, void* out, int ldo, long long plane_stride,
                   int planes, int bf16, cudaStream_t stream);

/* ---- LPDNet pieces: model/lpdnet_model.py:103-137 ------------------------------------------------
 * conv1_lpd (:111): xyz [B,3,N] -> token-major out[B*N, ldo] = LeakyReLU(W[Cout,3] p + bias). */
int vcr_conv3_act(const float* xyz, const float* w, const float* bias, int B, int N, int Cout, float slope,
                  float* out, int ldo, cudaStream_t stream);
/* convDG1 + max + convDG2 + max (:122-126) from PQ = [P | Q] (P = W_a f, Q = W_b f + bias, both 128
 * wide): x1 = max_k act(P[j]+Q[i]), x2 = act(max_k W2 e1 + b2).  k must be 20; idx is per-cloud local. */
int vcr_edgeconv_dg(const float* PQ, int ldpq, const int* idx, int k, int N, long long total_pts,
                    const float* W2, const float* b2, float slope, float* x1, int ld1, float* x2, int ld2,
                    cudaStream_t stream);
/* Tensor-core (tcgen05/TMEM) flavour of vcr_edgeconv_dg, same contract: the DG2 GEMM runs transposed
 * (D[out-channel][edge]) so max-over-k is an in-thread reduction.  mode: 0 = fp16 3-term split (fp32 parity),
 * 1 = fp16, 2 = bf16.  ldpq, ld1 multiples of 4, slope >= 0.  z (optional, NULL to skip): the per-edge convDG2
 * pre-activations W2 e1 + b2, [total_pts * 20][128] -- the values x2 is the activated max of, which the LPDNet backward
 * routes g_x2 by. */
int vcr_edgeconv_dg_tc(const float* PQ, int ldpq, const int* idx, int k, int N, long long total_pts,
                       const float* W2, const float* b2, float slope, int mode, float* x1, int ld1,
                       float* x2, int ld2, void* op1, void* op2, int ldop, long long op_plane, float* z,
                       cudaStream_t stream);
/* convSN1 + max (:130-132): out = act(max_k P[idx] + Q), C in {128,256,384,512}. */
int vcr_gather_max(const float* P, int ldp, const float* Q, int ldq, const int* idx, int k, int N,
                   long long total_pts, int C, float slope, float* out, int ldo, void* op, int ldop,
                   long long op_plane, cudaStream_t stream);
/* op1 / op2 / op above (optional, NULL to skip): the same output rows also in "h3" operand format ([2 planes][rows][ldop]
 * fp16 hi, lo * 2^11) for the GEMM that consumes them -- no separate vcr_to_operand pass over the LPDNet activations.
 * vcr_lpd_point_mlp: conv1_lpd + conv2_lpd of model/lpdnet_model.py:111-112 in one kernel (bit-identical to vcr_conv3_act +
 * vcr_gemm_f32), h1 optional, h2 fp32 + optional operand copy. */
int vcr_lpd_point_mlp(const float* xyz, const float* w1, const float* b1, const float* w2, const float* b2, int B, int N,
                      float slope, float* h1, float* h2, void* op, int ldop, long long op_plane, cudaStream_t stream);

/* ---- Transformer pieces: model/transformer.py -----------------------------------------------------
 * LayerNorm (:134-144): a*(x-mean)/(std_unbiased+eps)+b (+ residual if not NULL). D%128==0, D<=1024. */
int vcr_layernorm(const float* x, int ldx, const float* a, const float* b, float eps, long long M, int D,
                  const float* residual, int ldr, float* out, int ldo, cudaStream_t stream);
/* the same, additionally writing the operand-format copy [2 planes][M][ldop] (fp16 hi, lo * 2^11) and the squared row
 * norms sq[M] of `out` (what the VCP head, model/vcrnet_model.py:337-339, derives from the Transformer output). */
int vcr_layernorm_head(const float* x, int ldx, const float* a, const float* b, float eps, long long M, int D,
                       const float* residual, int ldr, float* out, int ldo, void* op, int ldop,
                       long long plane_stride, float* sq, cudaStream_t stream);
/* softmax over the last dim, in place (:34); keep[batch,n]==0 keys are set to -1e9 first (:51-52). */
int vcr_softmax_rows(float* S, int ld, long long rows, int n, const uint8_t* keep, long long rows_per_batch,
                     cudaStream_t stream);
/* column sums of probabilities over heads and queries (:39) / over sources (vcrnet_model.py:222). */
size_t vcr_colsum_workspace_bytes(int B, int n);
int vcr_colsum(const float* P, int ld, int B, long long rows_per_batch, int n, float* out, void* workspace,
               size_t workspace_bytes, cudaStream_t stream);
/* The materialised selectCom passes of a ragged batch (vcr_select_stats_ragged computes the other pairs): pd [B][Ns][ld]
 * from vcr_negdist over the padded block, pair b's ns[b] x nt[b] corner in use (int32, device; clamped to [0, Ns] /
 * [0, Nt]).  Only the pairs with nt[b] > 1024 -- those a pair alone routes to the materialised passes -- are touched, each
 * equal to its entry point on the pair alone over the pair's rows / columns, bit for bit.
 * vcr_softmax_rows_ragged: the pair's rows over its columns, in place.  vcr_colsum_ragged: out [B, Nt] column sums of the
 * pair's rows, columns past nt[b] written as 0 (workspace as vcr_colsum).  vcr_rowsum_colsoftmax_ragged: below. */
int vcr_softmax_rows_ragged(float* S, int ld, const int* ns, const int* nt, int B, int Ns, int Nt, cudaStream_t stream);
int vcr_colsum_ragged(const float* P, int ld, const int* ns, const int* nt, int B, int Ns, int Nt, float* out,
                      void* workspace, size_t workspace_bytes, cudaStream_t stream);
/* operand-format producers for vcr_gemm_tc: LayerNorm output / softmax probabilities written directly as
 * 16-bit hi(/lo) planes; row log-sum-exp statistics and the column sums of softmax(S) without
 * materialising the probabilities (partial-overlap key selection, model/transformer.py:39). */
int vcr_layernorm_operand(const float* x, int ldx, const float* a, const float* b, float eps, long long M, int D,
                          void* out, int ldo, long long plane_stride, int planes, int bf16, cudaStream_t stream);
int vcr_row_lse(const float* S, int ld, long long rows, int n, const uint8_t* keep, long long rows_per_batch,
                float* rmax, float* rsum, cudaStream_t stream);
int vcr_softmax_operand(const float* S, int ld, long long rows, int n, const uint8_t* keep,
                        long long rows_per_batch, void* out, int ldo, long long plane_stride, int planes,
                        int bf16, cudaStream_t stream);
/* The same statistic straight from the operand-format Q / K projections (model/transformer.py:33-39), nothing of size
 * Nq x Nk in HBM: per (batch, head, 128-query tile) two tcgen05 sweeps over the key tiles (row max / sum, then the
 * normalised probabilities summed over the tile's rows), partials reduced in a fixed order.  Q: [2 planes][B*Nq][ldq]
 * with head hh in columns [hh*128, +128), K likewise; d_k = 128; out [B, Nk]. */
size_t vcr_attn_colsum_workspace_bytes(int B, int H, int Nq, int Nk);
int vcr_attn_colsum_tc(const void* Q, int ldq, long long q_plane, const void* K, int ldk, long long k_plane,
                       int B, int H, int Nq, int Nk, int dk, float scale, float* out, void* workspace,
                       size_t workspace_bytes, cudaStream_t stream);
/* Ragged batch: item b has nq[b] queries and nk[b] keys (int32, device; clamped to [0, Nq] / [0, Nk]) in its Nq / Nk rows.
 * Keys past nk[b] are -inf in the row maxima and sums and their tiles are not loaded, query tiles past nq[b] are skipped,
 * and item b's partials are added in the order of the item alone ((hh * nqt_b + qt) * 4 + quarter, nqt_b = ceil(nq_b/128)).
 * out [B, Nk]: columns < nk[b] equal vcr_attn_colsum_tc on the item alone, bit for bit; the rest are 0.  Workspace as
 * vcr_attn_colsum_tc. */
int vcr_attn_colsum_tc_ragged(const void* Q, int ldq, long long q_plane, const void* K, int ldk, long long k_plane,
                              const int* nq, const int* nk, int B, int H, int Nq, int Nk, int dk, float scale, float* out,
                              void* workspace, size_t workspace_bytes, cudaStream_t stream);
/* fused, single-read form of vcr_row_lse + vcr_colsum_softmax (unmasked): out[B,n] = column sums of softmax rows */
size_t vcr_softmax_colsum_workspace_bytes(int B, long long rows_per_batch, int ld, int n);
int vcr_softmax_colsum(const float* S, int ld, int B, long long rows_per_batch, int n, float* out,
                       void* workspace, size_t workspace_bytes, cudaStream_t stream);
/* The same over a ragged batch of scaled scores S [B][H][Nq][ld] (fp32, ld >= Nk, ld % 4 == 0, 16-byte aligned): item b has
 * nq[b] queries and nk[b] keys (int32, device; clamped to [0, Nq] / [0, Nk]).  Its compact rows hh * nq_b + q are slabbed by
 * the rows-per-CTA of its own ld_b = ceil(nk_b / 4) * 4, as vcr_softmax_colsum slabs the item alone, so out [B, Nk] columns
 * < nk[b] equal vcr_softmax_colsum on S_b [H * nq_b, ld_b] bit for bit; the rest are 0. */
size_t vcr_softmax_colsum_ragged_workspace_bytes(int B, int H, int Nq, int Nk);
int vcr_softmax_colsum_ragged(const float* S, int ld, const int* nq, const int* nk, int B, int H, int Nq, int Nk,
                              float* out, void* workspace, size_t workspace_bytes, cudaStream_t stream);
int vcr_colsum_softmax(const float* S, int ld, int B, long long rows_per_batch, int n, const float* rmax,
                       const float* rsum, float* out, void* workspace, size_t workspace_bytes, cudaStream_t stream);
int vcr_rowsum(const float* P, int ld, long long rows, int n, float* out, cudaStream_t stream);
/* top-K (value desc, ties -> lower index, -0 == +0): sorted indices and/or a uint8 membership mask (:41-47).
 * n <= 262 144: one CTA per row up to 16 384, beyond that one thread-block cluster of 2, 4, 8 or 16 CTAs per row (16 384
 * keys each); -2 above 262 144 or when the device cannot co-schedule the cluster.  No workspace, no host sync. */
int vcr_topk_select(const float* vals, int B, int n, int K, int* idx_out, uint8_t* mask_out, cudaStream_t stream);
/* Ragged rows: row b of vals [B, n] holds n_len[b] values (clamped to [0, n]) and selects k_len[b] of them (clamped to
 * [0, min(K, n_len[b])]); both int32 on the device.  idx_out [B, K]: the indices vcr_topk_select gives on the row alone,
 * then 0; mask_out [B, n]: 1 on the selected keys, 0 elsewhere (past n_len[b] too).  n <= 16 384 (-2 above). */
int vcr_topk_select_ragged(const float* vals, const int* n_len, const int* k_len, int B, int n, int K, int* idx_out,
                           uint8_t* mask_out, cudaStream_t stream);

/* ---- VcpTopK head: model/vcrnet_model.py:162-347 ---------------------------------------------------
 * Row pass over dot[B,Ns,ld] = s_i.t_j: pd = (-xx_i + 2 dot) - yy_j, softmax over j, then
 * mode 0 (:344-345) corr[B,3,Ns] = sum_j P_ij tgt[B,3,Nt];  mode 1 (:221) P in place;
 * mode 2 (:295-299) best_idx = argmax_j, best_val = max_j P_ij. */
int vcr_sqnorm_rows(const float* X, int ld, long long rows, int D, float* out, cudaStream_t stream);
int vcr_softcorr_rows(float* dot, int ld, int B, int Ns, int Nt, const float* xx, const float* yy,
                      const float* tgt, int mode, float* corr, int* best_idx, float* best_val, cudaStream_t stream);
int vcr_negdist(float* dot, int ld, int B, int Ns, int Nt, const float* xx, const float* yy, cudaStream_t stream);
/* getCopairALL (:334-347) fused on tensor cores: S / T operand-format ("h3", 2 planes) embeddings [2][B*Ns][lds] /
 * [2][B*Nt][ldt], xx / yy their fp32 squared row norms, tgt [B,3,Nt] -> corr [B,3,Ns] = softmax_j(pd_ij) tgt_j with the
 * reference's pd operation order; the [Ns,Nt] score matrix never reaches HBM (online softmax in the GEMM epilogue). */
int vcr_softcorr_tc(const void* S, int lds, long long s_plane, const void* T, int ldt, long long t_plane,
                    const float* xx, const float* yy, const float* tgt, int B, int Ns, int Nt, int D,
                    float* corr, cudaStream_t stream);
/* Ragged batch: pair b has ns[b] sources and nt[b] targets (int32, device; clamped to [1, Ns] / [1, Nt]) in its Ns / Nt
 * rows.  128-source tiles past ns[b] and target tiles past nt[b] are skipped, targets past nt[b] in the last tile get the
 * tail treatment of a call with Nt = nt[b], the online softmax visits the tiles in the same order, and corr columns >= ns[b]
 * are written as 0: columns < ns[b] equal vcr_softcorr_tc on the pair alone, bit for bit. */
int vcr_softcorr_tc_ragged(const void* S, int lds, long long s_plane, const void* T, int ldt, long long t_plane,
                           const float* xx, const float* yy, const float* tgt, const int* ns, const int* nt, int B,
                           int Ns, int Nt, int D, float* corr, cudaStream_t stream);
/* getCopair (:264-332) through the same fused kernel: best_idx[B,Ns] = argmax_j pd_ij (ties -> lower j),
 * best_val[B,Ns] = max_j softmax_j(pd_ij) -- the hard correspondences of the partial path. */
int vcr_softcorr_best_tc(const void* S, int lds, long long s_plane, const void* T, int ldt, long long t_plane,
                         const float* xx, const float* yy, int B, int Ns, int Nt, int D,
                         int* best_idx, float* best_val, cudaStream_t stream);
/* Ragged batch, with the tile walk of vcr_softcorr_tc_ragged: rows < ns[b] equal vcr_softcorr_best_tc on the pair alone,
 * bit for bit; rows past ns[b] get best_idx = 0 and best_val = 0. */
int vcr_softcorr_best_tc_ragged(const void* S, int lds, long long s_plane, const void* T, int ldt, long long t_plane,
                                const float* xx, const float* yy, const int* ns, const int* nt, int B, int Ns, int Nt,
                                int D, int* best_idx, float* best_val, cudaStream_t stream);
/* selectCom's statistics (as vcr_select_stats) straight from the operands, on tensor cores, with no [Ns,Nt] buffer:
 * S / T, xx / yy as vcr_softcorr_best_tc takes them -> row_stat [B,Ns], col_stat [B,Nt].  Four launches of the fused
 * kernel (row max / sum over targets, the same over sources, then the two weighted sums), each row owned by one thread
 * pair: deterministic.  workspace: 2*(B*Ns + B*Nt) floats (the per-row and per-column max and 1/sum). */
size_t vcr_select_stats_tc_workspace_bytes(int B, int Ns, int Nt);
int vcr_select_stats_tc(const void* S, int lds, long long s_plane, const void* T, int ldt, long long t_plane,
                        const float* xx, const float* yy, int B, int Ns, int Nt, int D, float* row_stat, float* col_stat,
                        void* workspace, size_t workspace_bytes, cudaStream_t stream);
/* row sums of the softmax taken over sources (dim=1) (:243-244); workspace from the size query. */
size_t vcr_rowsum_colsoftmax_workspace_bytes(int B, int Nt);
int vcr_rowsum_colsoftmax(const float* pd, int ld, int B, int Ns, int Nt, float* out, void* workspace,
                          size_t workspace_bytes, cudaStream_t stream);
/* Ragged batch (see vcr_softmax_rows_ragged): out [B, Ns], rows past ns[b] written as 0; workspace as
 * vcr_rowsum_colsoftmax. */
int vcr_rowsum_colsoftmax_ragged(const float* pd, int ld, const int* ns, const int* nt, int B, int Ns, int Nt, float* out,
                                 void* workspace, size_t workspace_bytes, cudaStream_t stream);
/* selectCom (model/vcrnet_model.py:213-222, 243-244) selection statistics in two reads of the score products:
 * pd_ij = (-xx_i - (-2 dot_ij)) - yy_j is formed on the fly (dot [B,Ns,ld] is left untouched); row_stat [B,Ns] = row sums of
 * the column softmax, col_stat [B,Nt] = column sums of the row softmax.  Deterministic (fixed slab order). */
size_t vcr_select_stats_workspace_bytes(int B, int Ns, int Nt);
int vcr_select_stats(const float* dot, int ld, int B, int Ns, int Nt, const float* xx, const float* yy,
                     float* row_stat, float* col_stat, void* workspace, size_t workspace_bytes, cudaStream_t stream);
/* Ragged batch: pair b has ns[b] sources and nt[b] targets (int32, device; clamped to [0, Ns] / [0, Nt]) in dot [B][Ns][ld],
 * xx [B, Ns], yy [B, Nt].  Only the pairs with nt[b] <= 1024 -- those a pair alone sends to vcr_select_stats -- are computed:
 * row_stat rows < ns[b] and col_stat columns < nt[b] equal vcr_select_stats on the pair alone, bit for bit, and the rest of
 * their rows are 0.  The other pairs are left to the materialised passes (vcr_negdist in place, then
 * vcr_rowsum_colsoftmax_ragged, vcr_softmax_rows_ragged, vcr_colsum_ragged), which must run after this call.  Any Nt;
 * workspace: vcr_select_stats_workspace_bytes(B, Ns, Nt). */
int vcr_select_stats_ragged(const float* dot, int ld, const int* ns, const int* nt, int B, int Ns, int Nt, const float* xx,
                            const float* yy, float* row_stat, float* col_stat, void* workspace, size_t workspace_bytes,
                            cudaStream_t stream);
/* Rows idx[b,:] of an operand-format buffer ([2 planes][B*Nin][ld_in], 16-bit) and of its squared row norms: what getCopair
 * (model/vcrnet_model.py:264-332) needs of the points selectCom kept, without going back through fp32. */
int vcr_gather_operand_rows(const void* in, int ld_in, long long plane_in, int B, int Nin, const int* idx, int K,
                            int C, void* out, int ld_out, long long plane_out, const float* sq_in, float* sq_out,
                            cudaStream_t stream);
int vcr_gather_rows(const float* in, int ld_in, int B, int Nin, const int* idx, int K, int C, float* out,
                    int ld_out, cudaStream_t stream);
int vcr_gather_cols(const float* in, int B, int C, int Nin, const int* idx, int K, float* out, cudaStream_t stream);
/* getCopair's output gathers (:300-331, tgtK==1): src_out[b,:,r] = src[b,:,keep[b,r]],
 * corr_out[b,:,r] = tgt[b,:,best_idx[b,keep[b,r]]];  src [B,3,Ns], tgt [B,3,Nt], outputs [B,3,K]. */
int vcr_copair_gather(const float* src, const float* tgt, int B, int Ns, int Nt, const int* keep,
                      const int* best_idx, int K, float* src_out, float* corr_out, cudaStream_t stream);

/* ---- SVD head + pose algebra: model/vcrnet_model.py:350-399, :515-516, :21-43; util/util.py:91-96 --
 * src, corr [B,3,M] -> R_ab [B,3,3], t_ab [B,3]; optional R_ba = R^T, t_ba = -R^T t, H (covariance). */
int vcr_svd_head(const float* src, const float* corr, int B, int M, float* R_ab, float* t_ab,
                 float* R_ba, float* t_ba, float* H_out, cudaStream_t stream);
/* Ragged batch: pair b has m[b] points (int32, device; clamped to [1, M]) in its M columns; the fp64 means and covariance
 * run over exactly those points in the order of a call on the pair alone, so the outputs equal it bit for bit. */
int vcr_svd_head_ragged(const float* src, const float* corr, const int* m, int B, int M, float* R_ab, float* t_ab,
                        float* R_ba, float* t_ba, float* H_out, cudaStream_t stream);
/* out [B,C,N] = x with columns n >= len[b] (len clamped to [lo, N]) set to 0: the padding of a ragged batch made finite and
 * independent of what the caller left there.  out may be x. */
int vcr_zero_padding(const float* x, const int* len, int B, int C, int N, int lo, float* out, cudaStream_t stream);
int vcr_rigid_apply(const float* pc, const float* R, const float* t, int B, int N, float* out, cudaStream_t stream);
int vcr_pose_compose(const float* R_i, const float* t_i, float* R_f, float* t_f, int B, cudaStream_t stream);
int vcr_pose_inverse(const float* R, const float* t, float* R_inv, float* t_inv, int B, cudaStream_t stream);
/* host-side entry to the same 3x3 Jacobi SVD routine the kernel uses (unit tests; no GPU needed). */
int vcr_host_svd3(const double* H, double* U, double* S, double* V);

/* ---- layout / elementwise helpers -------------------------------------------------------------------
 * in [nb,R,C] (row stride ld_in) -> out [nb,C,R]: the .transpose(2,1).contiguous() of the reference. */
int vcr_transpose(const float* in, float* out, int nb, int R, int C, int ld_in, int ld_out,
                  long long stride_in, long long stride_out, cudaStream_t stream);
int vcr_add(const float* a, const float* b, float* out, long long n, cudaStream_t stream);

/* ---- data step + evaluation metrics on the device (SURVEY 8f row 2) ------------------------------------
 * vcr_make_pairs: util/data.py:247-309 minus the random draws (host draws pose + permutations like the reference):
 *   src[p,:,n] = base[p, idx_src[p,n]], tgt[p,:,n] = R_p base[p, idx_tgt[p,n]] + t_p in float64 (:289-291), outputs as
 *   fp64 [P,3,N] (input of the crop) and / or fp32.  pose [P,12] fp64 = row-major R then t.
 * vcr_crop_nearest: util/data.py:320-329: the `keep` points nearest to the last point, nearest first -> fp32 [P,3,keep].
 *   pc64 fp64 [P,3,N]; squared distances in fp64, ties -> lower index.  One CTA per cloud ranks by counting in shared
 *   memory: N <= 25 600 (-2 above).
 * vcr_crop_nearest_sort: the same crop for any N (P >= 1, 1 <= keep <= N, P*N <= 2^31 - 1, else -2): a stable LSD radix sort
 *   of the distances' fp64 bit patterns (8 passes of 8-bit digits, segmented per cloud) in `workspace` of at least
 *   vcr_crop_nearest_workspace_bytes(P, N) bytes (-4 if smaller), then a gather of the first `keep`.  Where both apply
 *   and no distance is NaN, the output equals vcr_crop_nearest's bit for bit; NaN distances go last in index order (as in
 *   numpy's stable argsort), and all `keep` columns are written for any input.
 *   No host sync, no allocation: the call can be captured in a CUDA graph.
 * vcr_eval_metrics: model/vcrnet_model.py:583-630 per-batch metrics accumulated into device double acc[8] =
 *   {pose loss, cycle loss, mse_ab, mae_ab, mse_ba, mae_ba, examples, -}, each weighted by the batch size. */
int vcr_make_pairs(const float* base, int P, int Nb, const int* idx_src, const int* idx_tgt, const double* pose,
                   int N, double* src64, double* tgt64, float* src, float* tgt, cudaStream_t stream);
int vcr_crop_nearest(const double* pc64, int P, int N, int keep, float* out, cudaStream_t stream);
size_t vcr_crop_nearest_workspace_bytes(int P, int N);
int vcr_crop_nearest_sort(const double* pc64, int P, int N, int keep, float* out, void* workspace, size_t workspace_bytes,
                          cudaStream_t stream);
int vcr_eval_metrics(const float* src, const float* tgt, int N, const float* srcK, const float* corrK, int M,
                     const float* R_gt, const float* t_gt, const float* R_ab, const float* t_ab,
                     const float* R_ba, const float* t_ba, int B, double* acc, cudaStream_t stream);
/* Ragged batches of the data step (int32 per-item lengths on the device, read there only and clamped into range; no host
 * sync, no allocation, so each call can be captured in a CUDA graph and replayed with new lengths):
 * vcr_make_pairs_ragged: vcr_make_pairs with item p at n[p] points (clamped to [0, N_max]) of N_max columns; idx_src /
 *   idx_tgt are [P, N_max] and are read below n[p] only.  Columns at or past n[p] are written as 0 in every output given.
 *   P in [1, 65535], Nb >= 1, N_max >= 1, else -2.
 * vcr_crop_nearest_ragged: the one-CTA crop of cloud p's first n[p] points (clamped to [1, N_max]) to the keep[p] (clamped
 *   to [0, min(keep_max, n[p])]) nearest to its point n[p] - 1 -> out [P,3,keep_max], columns past keep[p] written as 0.
 *   1 <= keep_max <= N_max <= 25 600 and P >= 1, else -2.
 * vcr_crop_nearest_sort_ragged: the same by the radix sort for any N_max (limits and -2 as vcr_crop_nearest_sort); the
 *   workspace is vcr_crop_nearest_workspace_bytes(P, N_max) bytes (-4 if smaller).  Keys past n[p] sort after every
 *   point of the cloud, NaN distances included.  Where both apply and no distance is NaN, the two ragged crops, and the
 *   uniform crop of each cloud alone, give the same bits.
 * vcr_eval_metrics_ragged: vcr_eval_metrics with pair b over its n[b] points of src / tgt [B,3,N_max] and its m[b]
 *   columns of srcK / corrK [B,3,M_max] (both clamped to [1, *]): each pair's sums are divided by its own denominators,
 *   and pair b adds what vcr_eval_metrics on it alone adds (up to the order of the fp64 sums).  B in [1, 65535]. */
int vcr_make_pairs_ragged(const float* base, int P, int Nb, const int* idx_src, const int* idx_tgt, const double* pose,
                          const int* n, int N_max, double* src64, double* tgt64, float* src, float* tgt,
                          cudaStream_t stream);
int vcr_crop_nearest_ragged(const double* pc64, const int* n, const int* keep, int P, int N_max, int keep_max,
                            float* out, cudaStream_t stream);
int vcr_crop_nearest_sort_ragged(const double* pc64, const int* n, const int* keep, int P, int N_max, int keep_max,
                                 float* out, void* workspace, size_t workspace_bytes, cudaStream_t stream);
int vcr_eval_metrics_ragged(const float* src, const float* tgt, const int* n, int N_max, const float* srcK,
                            const float* corrK, const int* m, int M_max, const float* R_gt, const float* t_gt,
                            const float* R_ab, const float* t_ab, const float* R_ba, const float* t_ba, int B,
                            double* acc, cudaStream_t stream);

/* ---- ICP refinement (--iter=0): model/icp_model.py:26-108 ICP.forward, model/vcrnet_model.py:46-62 -----------
 * vcr_icp_nearest = nearest_neighbor (:52-75): corr [B,3,Ns] = nearest dst point per src point under
 * pd = (-xx - (-2 s.d)) - yy (ties -> lower index); *err_sum (double, caller-zeroed) += sum of the best pd.
 * vcr_icp_advance = loop tail (:36-40) with the convergence test on the device: if the state's done flag is clear,
 * src <- R src + t, mean = *err_sum / (B*Ns), done = |prev - mean| < tolerance, prev = mean.  state is
 * vcr_icp_state_bytes() bytes {int done; int iters; double prev_error}, zeroed before the first iteration.
 * The rigid fit between the two calls is vcr_svd_head (best_fit_transform :77-108 == SVDHead arithmetic). */
size_t vcr_icp_state_bytes(void);
int vcr_icp_nearest(const float* src, const float* dst, int B, int Ns, int Nt, float* corr, int* nn_idx,
                    double* err_sum, cudaStream_t stream);
int vcr_icp_advance(float* src, const float* R, const float* t, int B, int Ns, const double* err_sum,
                    float tolerance, void* state, cudaStream_t stream);

/* ---- DGCNN / PointNet embeddings (--emb_nn dgcnn | pointnet, model/vcrnet_model.py:66-123) ----------
 * The per-edge 1x1 conv stack runs as GEMMs over a materialised [T*k, C] edge tensor (vcr_edge_gather_act builds
 * layer 1 from the split first conv, vcr_gemm_* the rest with eval-mode BatchNorm folded into weight and bias);
 * vcr_edge_max is x.max(dim=-1): out[pt, c] = max_kk E[pt, kk, c]. */
int vcr_edge_max(const float* E, int k, long long total_pts, int C, float* out, int ldo, cudaStream_t stream);

/* ---- LPDNet backward (BASELINE config 3: LPD pre-training forward + backward) ------------------------
 * The reference differentiates model/lpdnet_model.py:103-137 with autograd (loss at :149-229, optimiser step in
 * train_one_epoch :232-276).  These are the gradient kernels of the factored forward (csrc/train.cu); the dense
 * data-gradient products reuse vcr_gemm_f32 with b_layout = 1.
 * vcr_wgrad_f32: dW[N,K] += G[M,N]^T X[M,K], db[N] += column sums of G (db may be NULL); caller zero-initialises. */
int vcr_wgrad_f32(const float* G, int ldg, const float* X, int ldx, long long M, int N, int K, float* dW,
                  int lddw, float* db, cudaStream_t stream);
/* gz = gy * LeakyReLU'(z) from the saved post-activation y (F.leaky_relu backward).  scale_bits (may be NULL): the
 * output of vcr_absmax_bits for gy; gy is then also multiplied by 2^-floor(log2 max|gy|) (exponent clamped to
 * [-126, 126]), which brings max|gy| into [1, 2) so that the "h3" data-gradient products see normal fp16 operands. */
int vcr_act_bwd(const float* gy, int ldg, const float* y, int ldy, long long rows, int cols, float slope,
                const int* scale_bits, float* gz, int ldz, cudaStream_t stream);
/* bits = max(bits, bit pattern of max|x[i]|) over n contiguous floats; the caller zero-initialises bits. */
int vcr_absmax_bits(const float* x, long long n, int* bits, cudaStream_t stream);
/* out[0] = 2^floor(log2 m) for m the float whose bit pattern is bits[0] (same clamp): the inverse of vcr_act_bwd's scale. */
int vcr_pow2_inverse(const int* bits, float* out, cudaStream_t stream);
/* backward of vcr_gather_max (convSN1 + max over k, :130-132): gQ written, gP accumulated (zero-initialised). */
int vcr_gather_max_bwd(const float* P, int ldp, const float* Q, int ldq, const int* idx, int k, int N,
                       long long total_pts, int C, float slope, const float* gout, int ldgo, float* gP,
                       int ldgp, float* gQ, int ldgq, cudaStream_t stream);
/* e1[pt,kk,:] = act(P[nbr] + Q[pt]) with PQ = [P | Q] rows of 2C floats (convDG1 output, :123), E is [T*k, C]. */
int vcr_edge_gather_act(const float* PQ, int ldpq, const int* idx, int k, int N, long long total_pts, int C,
                        float slope, float* E, cudaStream_t stream);
/* Z [T,k,C] = convDG2 pre-activations in, g_Z out: g_x2 routed to the arg-max edge per (point, channel) (:125-126). */
int vcr_edge_max_bwd(float* Z, const float* gx, int ldgx, int k, long long total_pts, int C, float slope,
                     cudaStream_t stream);
/* g_e1 (+ g_x1 on the arg-max edge, :124) -> gPQ = [gP | gQ] rows of 2C floats (gP accumulated, zero-initialised). */
int vcr_edge_bwd_scatter(const float* E, const float* gE, const float* gx1, int ldgx, const int* idx, int k,
                         int N, long long total_pts, int C, float slope, float* gPQ, int ldg,
                         cudaStream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* VCR_B200_H */
