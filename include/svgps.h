/*
 * libsvgps — C-ABI of the tensor-core (tcgen05) kernels of the GPS object encoder and attention stack.
 * Raw device pointers + sizes + cudaStream_t (void*), int status (codes in svpointops.h), no
 * allocation, no synchronisation.  bf16 tensors are passed as void* (device, 2-byte elements).
 */
#ifndef SVGPS_H
#define SVGPS_H
#include "svpointops.h"

#ifdef __cplusplus
extern "C" {
#endif

/* bookkeeping of this library (separate counters from libsvpointops) */
unsigned long long svgps_launch_count(void);
int svgps_last_cuda_error(void);
const char *svgps_last_cuda_error_string(void);

/* Conformance probe of the tcgen05 conventions (tests only): D[128,N] f32 = A[128,K] bf16 x B[N,K]^T bf16,
 * one CTA, one TMEM accumulator; mode 0 = the descriptor convention used by the library. */
int sv_tc05_selftest(const void *A, const void *B, float *D, int N, int K, int mode, void *stream);

/* ---- PointNet++ set-abstraction MLP (inference form: eval-mode BatchNorm folded), tcgen05 ------------------
 * Replaces QueryAndGroup + SharedMLP(3 x Conv2d1x1+BN+ReLU) + max_pool2d of one PointnetSAModule
 * (reference: pointnet2_modules.py:34-75, pointnet2_utils.py:314-373, pytorch_utils.py:11-36).
 * `params` = packed device buffer of sv_sa_mlp_param_bytes(level) bytes built by
 * sceneverse_b200.modules.pointnet.pack_sa_params: [W1|W2|W3] bf16 in UMMA K-major layout with the BN
 * scale folded in, then shift1|shift2|shift3 (f32).  Outputs are point-major bf16 (B,npoint,C). */
int sv_sa_mlp_param_bytes(int level);
/* level 1: pts (B,P,6) f32 [xyz rgb], new_xyz (B,32,3), ball_idx (B,32,nsample) -> out (B,32,128) bf16
 * (mlp 6->64->64->128) */
int sv_sa1_mlp_bf16(const float *pts, const float *new_xyz, const int *ball_idx, const void *params, int B, int P,
                    int nsample, void *out_feat, void *stream);
/* level 2: xyz (B,P,3) f32, feat (B,P,128) bf16, new_xyz (B,16,3), ball_idx (B,16,nsample) -> out (B,16,256) bf16
 * (mlp 131->128->128->256) */
int sv_sa2_mlp_bf16(const float *xyz, const void *feat, const float *new_xyz, const int *ball_idx, const void *params,
                    int B, int P, int nsample, void *out_feat, void *stream);

/* ---- dense contraction with fused epilogue (tcgen05, TMA, persistent) --------------------------------------------
 * out[M,N] = epilogue(A[M,K] x B[N,K]^T): A, B bf16 row-major with leading dimensions lda, ldb (elements, % 8 == 0,
 * K % 8 == 0, 16-byte aligned) — B is the nn.Linear weight layout, so this replaces F.linear / 1x1 Conv2d
 * (reference call sites: SURVEY.md §2.3).  epilogue: + bias[N] (f32, may be NULL) -> act (0 none, 1 relu, 2 gelu-erf)
 * -> + residual[M,N] (same dtype / ld as out, may be NULL) -> store bf16 (out_f32 = 0) or f32 (1).
 * rowmax = 16: instead store max over each group of 16 consecutive rows into out[M/16,N] (PointNet++ SA3 max-pool). */
int sv_gemm_bf16(const void *A, int lda, const void *B, int ldb, int M, int N, int K, const float *bias, int act,
                 const void *residual, void *out, int ldo, int out_f32, int rowmax, void *stream);
/* Same GEMM with either operand given TRANSPOSED in memory (the two backward GEMMs of a linear layer without any copy):
 * a_transposed = 1: A is stored (K, M) row-major, lda >= M;  b_transposed = 1: B is stored (K, N) row-major, ldb >= N.
 * The staged tiles are then read by the tensor core as MN-major operands.  dgrad of y = x W^T: dx = g . W  ->
 * sv_gemm_bf16_ex(g, N, 0, W, Kin, 1, M, Kin, N, ...);  wgrad: dW = g^T . x -> sv_gemm_bf16_ex(g, N, 1, x, Kin, 1, N, Kin, M,
 * ..., out_f32 = 1).  (reference: autograd of every nn.Linear of the stack, e.g. modules/layers/transformers.py:122-134) */
int sv_gemm_bf16_ex(const void *A, int lda, int a_transposed, const void *B, int ldb, int b_transposed, int M, int N, int K,
                    const float *bias, int act, const void *residual, void *out, int ldo, int out_f32, int rowmax,
                    void *stream);

/* Micro-benchmark (profiling only): SM cycles for `iters` x 4 tcgen05.mma (M = 128, N, K = 16 each) issued back to back on
 * shared-memory-resident operands, per block, by operand layout (a_mn / b_mn = 1: MN-major, transposed operand).
 * cycles_out: 2 x `blocks` int64 on the device — SM cycles, then nanoseconds (globaltimer) of each block's issue loop.
 * Bits 1.. of a_mn are profiling flags: 1 = random operand bits instead of zeros, 2 = commit every four MMAs to a ring of
 * four barriers and wait for the group issued four groups earlier (the GEMM main loop's stage hand-shake). */
int sv_mma_bench(int N, int a_mn, int b_mn, int iters, int blocks, long long *cycles_out, void *stream);

/* Kernel selection of the GEMM family (tests / benchmarks): 0 = heuristic (default), 1 = single-CTA tiles (M = 128 per MMA),
 * 2 = CTA pairs (cta_group::2, M = 256 per MMA, each CTA stages half of the B tile) wherever M > 128, 4 = CTA pairs in
 * clusters of two that share the B tile through TMA multicast (forward / dgrad, 256-wide tiles; an experiment: only 33 clusters
 * of four CTAs are co-resident on a B200, so it is not selected by the heuristic).
 * Bits 8.. are profiling switches that make the RESULT GARBAGE (timing only): 1 = the epilogue skips its body,
 * 2 = the producer skips its TMA loads. */
int sv_gemm_force_ctas(int ctas);

/* Profiling: while `buf` (device, [grid][16] int64) is non-null every GEMM launch writes, per CTA, the MMA-issuing thread's
 * {loop cycles, cycles waiting for operands, cycles waiting for a free accumulator, k-steps issued, clock at start, at end,
 * loop nanoseconds (globaltimer)}, and from slot 8 two epilogue warps' {cycles at the bias barrier, waiting for the accumulator,
 * in the epilogue body, tiles}. */
int sv_gemm_profile(long long *buf);

/* ---- the three GEMMs of a linear layer y = x W^T + b with their fused epilogues (same tcgen05 kernel family) ------
 * Replace F.linear and its autograd (AddmmBackward: mm, mm, sum) for every nn.Linear of the attention stack, BERT and the
 * heads (reference: modules/layers/transformers.py:115-154,188-192,285-316; modules/language/bert.py:21-26).
 * x (M,K) bf16 ld ldx; w (N,K) bf16 ld ldw (nn.Linear layout); all leading dimensions % 8 == 0, 16-byte aligned bases.
 * forward:  out = dropout_p(act(x w^T + bias)) -> (M,N) bf16 | f32, ld ldo; act 0 none / 1 relu / 2 gelu(erf);
 *           pre_out (bf16, ld ldo, may be NULL) receives x w^T + bias before the activation (saved for the gelu backward);
 *           the dropout mask is the counter hash of csrc/attn_common.cuh keyed by (seed, row, column): nothing is stored. */
int sv_linear_fwd_bf16(const void *x, int ldx, const void *w, int ldw, int M, int N, int K, const float *bias, int act,
                       float dropout_p, unsigned long long seed, void *out, int ldo, int out_f32, void *pre_out,
                       void *stream);
/* dgrad:    dx (M,Kin) = (gy (M,N) . w (N,Kin)) x f, the weight read as a transposed (MN-major) operand, no copy.
 *           dact 0: f = 1.  dact 1: aux = the forward OUTPUT of a relu(+dropout) layer of shape (M,Kin): f = aux > 0 ? 1/(1-p) : 0.
 *           dact 2: aux = the saved PRE-activation of a gelu(+dropout) layer: f = gelu'(aux) x mask(seed,row,col)/(1-p).
 *           (the activation sits on the INPUT side of this linear: h = dropout(act(pre)), y = h w^T) */
int sv_linear_dgrad_bf16(const void *gy, int ldg, const void *w, int ldw, int M, int N, int Kin, int dact, const void *aux,
                         int ld_aux, float dropout_p, unsigned long long seed, void *dx, int ldx, int out_f32, void *stream);
/* wgrad:    dw (N,Kin) f32 (ld ld_dw) (+)= gy^T . x and db (N) f32 (+)= column sums of gy (db may be NULL), contraction over
 *           the M tokens split across the grid, results reduced with red.global.add — accumulate = 1 adds straight into an
 *           existing gradient buffer (the flat fp32 buffer the data-parallel all-reduce runs on), 0 overwrites.  The bias
 *           gradient costs one extra N = 16 MMA per K step against a tile of ones in the same main loop. */
int sv_linear_wgrad_bf16(const void *gy, int ldg, const void *x, int ldx, int M, int N, int Kin, float *dw, int ld_dw,
                         float *db, int accumulate, void *stream);

/* ---- fused attention forward (tcgen05): O = softmax(Q K^T * scale + spatial gate + key mask) V, head dim 64 ---------
 * q (B,Lq,*), k/v (B,Lk,*) bf16 with batch strides *_bs and row strides *_rs (elements, % 8 == 0); head h uses columns
 * [64h, 64h+64).  key_padding_mask (B,Lk) bytes, 1 = ignore (may be NULL).  spatial_w (B,Lq,spatial_heads*6) f32 =
 * [bias, w1..w5] per head and pairwise_locs (B,Lq,Lk,5) f32 enable the MultiHeadAttentionSpatial 'cond' gate
 * log(clamp(sigmoid(w . loc + b), 1e-6)) (reference: modules/layers/transformers.py:206-232); NULL = plain attention
 * (nn.MultiheadAttention core).  Lk <= 384.  out (B,Lq,H*64) bf16. */
int sv_attention_fwd_bf16(const void *q, long long q_bs, int q_rs, const void *k, long long k_bs, int k_rs,
                          const void *v, long long v_bs, int v_rs, void *out, long long o_bs, int o_rs,
                          const unsigned char *key_padding_mask, const float *spatial_w, int spatial_heads,
                          const float *pairwise_locs, int B, int H, int Lq, int Lk, float scale, void *stream);

/* same as sv_attention_fwd_bf16, additionally storing lse (B,H,Lq) f32 = log-sum-exp of each query's logits (needed by
 * sv_attention_bwd_bf16) */
int sv_attention_fwd_lse_bf16(const void *q, long long q_bs, int q_rs, const void *k, long long k_bs, int k_rs,
                              const void *v, long long v_bs, int v_rs, void *out, long long o_bs, int o_rs,
                              const unsigned char *key_padding_mask, const float *spatial_w, int spatial_heads,
                              const float *pairwise_locs, int B, int H, int Lq, int Lk, float scale, float *lse,
                              void *stream);
/* Backward of the fused attention; P is recomputed from Q, K, the gate and lse.  Without the gate ONE tcgen05 kernel (tile
 * rows == keys) computes P and dS once per (query, key) pair and produces dQ, dK and dV; keys past the last unmasked one
 * are skipped (their dK / dV rows are written as zeros).  With the gate two launches: dQ + gate-weight gradients with tile
 * rows == queries, dK/dV with tile rows == keys.  q/k/v as in the forward; o, d_o (B,Lq,H*64) bf16 contiguous; dq
 * (B,Lq,H*64), dk, dv (B,Lk,H*64) bf16 contiguous; d_spatial_w (B,Lq,H*6) f32 (NULL without gate; gate requires
 * spatial_heads == H); dvec: f32 scratch of sv_attention_bwd_scratch_floats(B, H, Lq, Lk) floats ((B,H,Lq) up to 128
 * keys, (B,H,Lq,64) beyond: the dQ partial sums over the key tiles).  Lq, Lk <= 384. */
int sv_attention_bwd_scratch_floats(int B, int H, int Lq, int Lk);
int sv_attention_bwd_bf16(const void *q, long long q_bs, int q_rs, const void *k, long long k_bs, int k_rs,
                          const void *v, long long v_bs, int v_rs, const void *o, const void *d_o,
                          const unsigned char *key_padding_mask, const float *spatial_w, const float *pairwise_locs,
                          const float *lse, int B, int H, int Lq, int Lk, float scale, void *dq, void *dk, void *dv,
                          float *d_spatial_w, float *dvec, void *stream);

/* Dropout variants (nn.MultiheadAttention applies dropout to the attention weights in training, reference
 * transformers.py:22-24,69-74,118-120): weight (b,h,i,j) is kept iff its 16-bit counter-based uniform (csrc/attn_common.cuh:
 * one 64-bit mix per (b,h,i) row, one 32-bit mix per key pair) >= round(p * 65536), and scaled by 1/(1-p); the backward
 * regenerates the same mask from (dropout_p, seed).  Not combinable with the spatial gate (the reference's spatial
 * attention has no weight dropout). */
int sv_attention_fwd_dropout_bf16(const void *q, long long q_bs, int q_rs, const void *k, long long k_bs, int k_rs,
                                  const void *v, long long v_bs, int v_rs, void *out, long long o_bs, int o_rs,
                                  const unsigned char *key_padding_mask, const float *spatial_w, int spatial_heads,
                                  const float *pairwise_locs, int B, int H, int Lq, int Lk, float scale, float *lse,
                                  float dropout_p, unsigned long long seed, void *stream);
int sv_attention_bwd_dropout_bf16(const void *q, long long q_bs, int q_rs, const void *k, long long k_bs, int k_rs,
                                  const void *v, long long v_bs, int v_rs, const void *o, const void *d_o,
                                  const unsigned char *key_padding_mask, const float *spatial_w,
                                  const float *pairwise_locs, const float *lse, int B, int H, int Lq, int Lk, float scale,
                                  void *dq, void *dk, void *dv, float *d_spatial_w, float *dvec, float dropout_p,
                                  unsigned long long seed, void *stream);

/* same backward with strided gradient outputs: rows of dq / dk / dv are d_rs elements apart (scene stride L * d_rs), so the
 * three can be the column slices [0,E) [E,2E) [2E,3E) of ONE packed (B,L,3E) buffer — the gradient of a packed QKV
 * projection, consumed by a single dgrad / wgrad GEMM (requires Lq == Lk for a shared packed buffer) */
int sv_attention_bwd_strided_bf16(const void *q, long long q_bs, int q_rs, const void *k, long long k_bs, int k_rs,
                                  const void *v, long long v_bs, int v_rs, const void *o, const void *d_o,
                                  const unsigned char *key_padding_mask, const float *spatial_w,
                                  const float *pairwise_locs, const float *lse, int B, int H, int Lq, int Lk, float scale,
                                  void *dq, void *dk, void *dv, int d_rs, float *d_spatial_w, float *dvec, float dropout_p,
                                  unsigned long long seed, void *stream);

/* Fused dropout + residual add + LayerNorm:  y = LayerNorm(residual + dropout(x)) * gamma + beta  (reference: the post-norm
 * blocks of modules/layers/transformers.py:145-154,311-315; plain LayerNorm of modules/utils.py:18-25 with residual = NULL,
 * dropout_p = 0).  x, residual, y, s: (R,D) contiguous, bf16 (io_bf16 = 1) or f32; D % 8 == 0, D <= 1024; gamma, beta (D)
 * f32; s receives the pre-norm sum (required when residual != NULL or dropout_p > 0; the backward's input — with neither,
 * pass x itself to the backward); mean, rstd (R) f32.  The dropout mask is the counter hash of csrc/attn_common.cuh keyed
 * by (seed, row, column): nothing is stored, the backward regenerates it. */
int sv_layer_norm_fwd(const void *x, const void *residual, int io_bf16, int R, int D, const float *gamma, const float *beta,
                      float eps, float dropout_p, unsigned long long seed, void *y, void *s, float *mean, float *rstd,
                      void *stream);
/* Backward: g = dL/dy (R,D) same dtype; ds = dL/d(residual) (= dL/dx without dropout); dx = ds o mask / (1 - p) (required
 * iff dropout_p > 0); dgamma, dbeta (D) f32; scratch: sv_layer_norm_scratch_floats(D) floats (per-CTA partial sums, reduced
 * in a fixed order by a second small kernel). */
int sv_layer_norm_bwd(const void *g, const void *s, int io_bf16, int R, int D, const float *gamma, const float *mean,
                      const float *rstd, float dropout_p, unsigned long long seed, void *ds, void *dx, float *dgamma,
                      float *dbeta, float *scratch, void *stream);
/* same; accumulate = 1 adds dgamma / dbeta into the given buffers (the flat gradient buffer) instead of overwriting them */
int sv_layer_norm_bwd_acc(const void *g, const void *s, int io_bf16, int R, int D, const float *gamma, const float *mean,
                          const float *rstd, float dropout_p, unsigned long long seed, void *ds, void *dx, float *dgamma,
                          float *dbeta, int accumulate, float *scratch, void *stream);

/* Row-wise L2 normalisation y = x / max(||x||_2, eps) over the last dimension and its backward
 * dx = (g - y (y . g)) / ||x|| (rows with ||x|| < eps: g / eps) — F.normalize(x, dim=-1, p=2) of the contrastive heads
 * (optim/loss/contra_loss.py:29-30, 59-60, 86-87 in the reference) and its autograd in one kernel per direction.
 * x / y / g / dx: (R, D) bf16 (io_bf16 = 1) or fp32, 16-byte aligned, D % 8 == 0, 8 <= D <= 1024; norm: (R) fp32. */
int sv_l2norm_fwd(const void *x, int io_bf16, int R, int D, float eps, void *y, float *norm, void *stream);
int sv_l2norm_bwd(const void *g, const void *y, const float *norm, int io_bf16, int R, int D, float eps, void *dx,
                  void *stream);
int sv_layer_norm_scratch_floats(int D);

/* Every in-kernel dropout mask (attention weights, fused LayerNorm) is a pure function of (seed, indices).  A captured
 * CUDA graph freezes the by-value seed, so a process may register ONE device counter: each dropout launch then uses
 * seed + *device_counter * odd_constant, read on the device at run time — increment the counter once per step (inside the
 * graph) and every replay draws fresh masks while forward and backward of the same step still agree.  NULL unregisters. */
int sv_dropout_seed_offset(const unsigned long long *device_counter);

/* Column sums out[c] = sum_r x[r][c] of a row-major (R, N) bf16 / f32 matrix (rows row_stride elements apart, N % 8 == 0),
 * fp32 accumulation, deterministic: the bias gradient of a linear layer (reference: autograd of every nn.Linear of the
 * stack, e.g. modules/layers/transformers.py:122-134).  scratch: sv_colsum_scratch_floats(N) floats. */
int sv_colsum(const void *x, long long row_stride, int is_bf16, int R, int N, float *out, float *scratch, void *stream);
int sv_colsum_scratch_floats(int N);

/* calc_pairwise_locs, 'center' relation (reference: modules/utils.py:38-87): centers (B,O,*) f32 with row stride
 * row_stride (>= 3 floats; xyz first) -> out (B,O,O,5) f32 = [dist/max_dist, dz/dist, dist2d/dist, dy/dist2d, dx/dist2d];
 * dist_norm = 0 keeps the raw distance in slot 0.  eps sits inside the square roots (1e-10 in the reference). */
int sv_pairwise_locs_f32(const float *centers, int row_stride, int B, int O, float eps, int dist_norm, float *out,
                         void *stream);

/* Fused softmax cross-entropy, forward + gradient (reference: optim/loss/loss.py:8-9,56-61 — F.cross_entropy with
 * ignore_index): logits (R,V) bf16 (is_bf16 = 1) or f32, rows row_stride elements apart; labels (R) int64.
 * loss_rows[r] = logsumexp(row) - row[label] (0 for ignored rows); grad_logits (R,V, contiguous, same dtype, may be NULL)
 * = softmax(row) - onehot(label) (zero rows for ignored labels).  The caller divides by the number of valid rows. */
int sv_cross_entropy_fwd_bwd(const void *logits, long long row_stride, int is_bf16, const long long *labels, int R, int V,
                             long long ignore_index, float *loss_rows, void *grad_logits, void *stream);
/* same, with gradient rows grad_row_stride (>= V) elements apart; columns [V, grad_row_stride) are written as zeros — the
 * gradient of a vocabulary padded to 16-byte rows (BERT LM head, V = 30522 -> 30528) feeds the backward GEMMs directly */
int sv_cross_entropy_fwd_bwd_strided(const void *logits, long long row_stride, int is_bf16, const long long *labels, int R,
                                     int V, long long ignore_index, float *loss_rows, void *grad_logits,
                                     long long grad_row_stride, void *stream);

/* Backward of a stand-alone activation behind a linear layer (the FFN form fuses this into sv_linear_dgrad_bf16):
 * out = g x act'(.), (M,N) bf16, N % 8 == 0.  mode 1: relu, aux = forward output; mode 2: gelu(erf), aux = pre-activation. */
int sv_act_bwd_bf16(const void *g, int ldg, const void *aux, int ld_aux, int mode, int M, int N, void *out, int ldo,
                    void *stream);

/* x[0..n) *= *scale (device scalar) in place, bf16 | f32, n % (8 | 4) == 0, 16-byte aligned: the 1/count scaling of the fused
 * cross-entropy gradient without a second (R, V) tensor. */
int sv_scale_inplace(void *x, long long n, int is_bf16, const float *scale, void *stream);

/* Gradient of an embedding lookup: dw[ids[t]][:] += grad_out[t][:] (fp32 red.add; rows with ids == padding_idx skipped).
 * grad_out (ntok, D) bf16 | f32 with row stride ldg; dw (vocab, D) f32 contiguous, NOT zeroed here (accumulates).
 * (reference: autograd of the three nn.Embedding tables of HF BertEmbeddings, modules/language/bert.py:21-26) */
int sv_embedding_bwd(const void *grad_out, long long ldg, int is_bf16, const long long *ids, int ntok, int D, long long vocab,
                     long long padding_idx, float *dw, void *stream);

/* clip_grad_norm_ + AdamW + bf16 shadow refresh over FLAT buffers in two launches (squared-norm partials, then the update;
 * reference: trainer/build.py:135-145, optim/utils.py:1-18).  params / exp_avg / exp_avg_sq / grads: n f32, 16-byte aligned;
 * shadow_bf16: n bf16 (may be NULL).  segments: DEVICE array of nseg records {long long begin, end; float lr_scale,
 * weight_decay} (element ranges, multiples of 4) — lr of a segment = base_lr * lr_scale * *lr_factor.  step: device 1-based
 * step counter (bias correction).  scratch: sv_adamw_scratch_floats() floats.  norm_out (may be NULL) receives ||g||.
 * max_norm <= 0 disables clipping. */
int sv_adamw_scratch_floats(void);
int sv_adamw_flat(float *params, float *exp_avg, float *exp_avg_sq, const float *grads, void *shadow_bf16, long long n,
                  const void *segments, int nseg, float max_norm, const float *lr_factor, const long long *step, float base_lr,
                  float beta1, float beta2, float eps, float *scratch, float *norm_out, void *stream);

/* ---- train-mode PointNet++ set abstraction in channels-last form (config C2: ObjCls pre-training with a trainable backbone) ----
 * A grouped tensor is the row matrix X[(b, centre, sample)][channel] in bf16: the 1x1 convolutions are sv_linear_*_bf16 (no bias),
 * BatchNorm2d with BATCH statistics is a column statistic over the rows, the neighbourhood max is a max over ns consecutive rows.
 * Reference: pointnet2_utils.py:291-373 (QueryAndGroup / GroupAll), pytorch_utils.py:11-36,67-120 (SharedMLP: Conv2d + BatchNorm2d +
 * ReLU), pointnet2_modules.py:70-73 (max_pool2d over nsample).
 * group_rows: X (B*np*ns, Cp) bf16, Cp % 8 == 0, Cp >= 3 + C: [xyz[idx] - centre | feat[idx] | 0]; centre NULL = raw xyz (GroupAll);
 * idx (B,np,ns) i32 or NULL (GroupAll: every point in order, np = 1, ns = N); feat (B,N,C) point-major f32 | bf16.
 * group_rows_grad: dfeat (B,N,C) f32 (zeroed here) += dX[:, 3:3+C] scattered by idx. */
int sv_pn_group_rows(const float *xyz, const float *centre, const void *feat, int feat_bf16, const int *idx, int B, int N, int C,
                     int np, int ns, int Cp, void *X, void *stream);
int sv_pn_group_rows_grad(const void *dX, const int *idx, int B, int N, int C, int np, int ns, int Cp, float *dfeat, void *stream);
/* BatchNorm (batch statistics over the R rows, biased variance) + ReLU: y, out (R,C) bf16; mean, rstd (C) f32 out; var_unbiased (C)
 * f32 out (may be NULL; for the running estimate); scratch: sv_pn_scratch_floats(C).  Backward: dy = d(out)/d(y) applied to dout,
 * dgamma / dbeta (C) f32 overwritten or accumulated. */
int sv_pn_scratch_floats(int C);
int sv_pn_bn_relu_fwd(const void *y, long long R, int C, const float *gamma, const float *beta, float eps, float *mean, float *rstd,
                      float *var_unbiased, void *out, float *scratch, void *stream);
int sv_pn_bn_relu_bwd(const void *y, const void *dout, long long R, int C, const float *gamma, const float *beta, const float *mean,
                      const float *rstd, void *dy, float *dgamma, float *dbeta, int accumulate, float *scratch, void *stream);
/* out[g][c] = max over the ns rows of group g, arg = index of the first maximum (bytes, ns <= 255); grad: gx[g*ns+s][c] = gout[g][c]
 * where s == arg, else 0. */
int sv_pn_rowgroup_max(const void *x, long long G, int ns, int C, void *out, unsigned char *arg, void *stream);
int sv_pn_rowgroup_max_grad(const void *gout, const unsigned char *arg, long long G, int ns, int C, void *gx, void *stream);

/* L2-normalise + all-gather fused over NVLink peer memory (reference: contra_loss.py:58-64,86-91 + dist_utils.py:131-149).
 * a, b: local (n,D) f32.  peer_bufs[world] / peer_signals[world]: DEVICE arrays of device pointers into a symmetric
 * allocation mapped on every rank: buffer = [2 parities][2 tensors][world*n][D] f32, signal = >= world uint32 words
 * (zero-initialised).  epoch must start at 1 and increase by 1 per call on every rank.  When the kernel completes the
 * local buffer holds, for parity epoch&1, normalize(a) and normalize(b) of all ranks in rank-major order. */
int sv_normalize_allgather_f32(const float *a, const float *b, int n, int D, void *const *peer_bufs,
                               void *const *peer_signals, unsigned *done_counter, int world, int rank, unsigned epoch,
                               void *stream);
/* same exchange with the epoch kept in device memory (*epoch_dev, zero-initialised, one word per exchange object): the
 * launch uses *epoch_dev + 1 and stores it back on completion, so a captured CUDA graph (frozen arguments) can replay it */
int sv_normalize_allgather_dev_f32(const float *a, const float *b, int n, int D, void *const *peer_bufs,
                                   void *const *peer_signals, unsigned *done_counter, int world, int rank,
                                   unsigned *epoch_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SVGPS_H */
