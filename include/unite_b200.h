/*
 * unite_b200 — C ABI of the B200-native UNITE training-step hot path.
 *
 * The reference (reddyav1/unite) is pure Python/PyTorch and has NO FFI layer (SURVEY.md §8(b)); its
 * boundary is the Python API (model factories, forward signatures, state_dict keys, train_one_epoch).
 * These entry points sit *behind* that Python surface: each one replaces the library call sequence the
 * reference issues at the cited file:line.  Conventions (all functions):
 *   - plain pointers and sizes; every buffer is device memory owned by the caller (PyTorch's allocator),
 *     borrowed for the call; nothing is allocated, freed or retained by the library;
 *   - stream-ordered on `stream` (a cudaStream_t passed as void*), no host synchronisation;
 *   - returns 0 when the work was enqueued, non-zero on argument / launch error with a thread-local
 *     message available from ub_last_error();
 *   - bf16 = raw 16-bit brain-float, row-major, leading dimensions in ELEMENTS.
 */
#ifndef UNITE_B200_H
#define UNITE_B200_H
#include <stdint.h>
#if defined(__GNUC__)
#define UB_API __attribute__((visibility("default")))
#else
#define UB_API
#endif
#ifdef __cplusplus
extern "C" {
#endif

UB_API int ub_version(void);
UB_API const char* ub_last_error(void);
UB_API int ub_sm_count(void);
/* Size every persistent grid of the library for n SMs instead of the whole device (0 = whole device); returns the count now in
 * effect.  Data-parallel runs leave a few SMs to the NCCL all-reduce that overlaps backward (unite_b200/ddp.py): a persistent
 * kernel whose static schedule assumes 148 resident CTAs stalls for the whole collective if 4 of them cannot be placed. */
UB_API int ub_set_sm_limit(int n);

/* ------------------------------------------------------------------------------------------------
 * GEMM (tcgen05/TMEM/TMA):  C[M,N] = epilogue( A[M,K] * B[N,K]^T )      bf16 x bf16 -> fp32 accumulate
 * Replaces every nn.Linear / F.linear / Conv3d(stride==kernel) / `x @ proj` on the path:
 *   teacher  clip.py:55-64 (in_proj, out_proj, c_fc, c_proj), clip.py:146 (conv1), clip.py:170 (x @ proj)
 *   student  modeling_finetune.py:108 (qkv), :117 (proj), :67-71 (fc1/fc2), :174 (PatchEmbed.proj),
 *            modeling_adaptation.py:204 (Linear_Decoder.head), and their autograd backward (dgrad / wgrad).
 * ---------------------------------------------------------------------------------------------- */
enum { UB_ACT_NONE = 0, UB_ACT_QUICKGELU = 1, UB_ACT_GELU = 2, UB_ACT_DGELU = 3, UB_ACT_DOT_AUX = 4 };

typedef struct ub_gemm_epilogue {
  const float* bias;      /* [N] added to the accumulator, or NULL                                         */
  const float* residual;  /* fp32 [M, ldr] added last, or NULL (may alias C when C is fp32)                 */
  const float* row_scale; /* per-sample scale (DropPath keep/(1-p)), indexed row / rows_per_scale, or NULL */
  const void* aux_in;     /* bf16 [M, ld_aux]: UB_ACT_DGELU multiplies by gelu'(aux_in)                    */
  void* aux_out;          /* bf16 [M, ld_aux]: UB_ACT_GELU also stores the pre-activation here, or NULL    */
  int64_t ldr;
  int64_t ld_aux;
  int32_t rows_per_scale;
  int32_t act;      /* UB_ACT_*                                                                           */
  int32_t out_fp32; /* 0: C is bf16, 1: C is fp32                                                         */
  int32_t accumulate; /* 1: C (fp32) += result with red.add (required when split_k > 1)                   */
  int32_t tile_ctas;  /* scheduling hint: 0 = cost model, 1 / 2 / 4 = CTAs per work item (4 = two pairs + B multicast) */
  int32_t max_ctas;   /* scheduling hint: 0 = whole device, > 0 = cap on the persistent grid (a GEMM run beside another),
                       * < 0 = non-persistent: one CTA (pair) per work item, for off-critical-path GEMMs on a low-priority stream */
  int32_t residual_f16; /* 1: `residual` is fp16 [M, ldr] and C is fp16 too (out_fp32 must be 0): the teacher's residual stream */
  int32_t ab_f16;       /* 1: A and B hold fp16 (not bf16) values                                                          */
  /* LayerNorm folded into the GEMM (frozen teacher): with A = the raw residual stream x (fp16), B = gamma o W, ln_c[n] =
   * sum_k B[n,k] and bias = beta W^T + b, the result rstd_m * (acc - mu_m * ln_c[n]) + bias[n] equals Linear(LN(x)).
   * ln_stats = fp32 [M,2] row (sum, sum of squares) of x, produced by the kernel that wrote x (stats_out below, or
   * ub_teacher_embed_ln); mu = sum * ln_inv_d, var = sumsq * ln_inv_d - mu^2.  All three NULL / 0 when unused.            */
  const float* ln_stats;
  const float* ln_c;
  float* stats_out;     /* residual_f16 epilogue only: += row (sum, sumsq) of the fp16 values written to C (must be zeroed)  */
  float ln_inv_d;
  float ln_eps;
  float* colsum_out;    /* DGELU epilogue only: += column sums over the M rows of the values written to C — the bias gradient of
                         * the Linear whose pre-activation is aux_in (saves the separate pass over C)                          */
  /* Grouped GEMM: several independent products of the same shape in ONE launch (the K alignment decoders of
   * modeling_adaptation.py:203-213, 322-325: y_k = z_k W_k^T + b_k, their dgrad and wgrad) — one wave-quantisation loss and one
   * launch instead of K.  C is the groups' outputs stacked along M (M = total rows, group_rows rows each, a multiple of 256);
   * the tile whose first row is m0 belongs to group g = m0 / group_rows and reads its operands at
   *   A: k + g * group_a_k, m - g * group_a_m        B: k + g * group_b_k, n + g * group_b_n        bias[n + g * group_bias]
   * (offsets in elements of the respective dimension; K is the per-group contraction length).  All 0 = ordinary GEMM.          */
  int32_t group_rows, group_a_k, group_a_m, group_b_k, group_b_n, group_bias;
  /* UB_ACT_DOT_AUX (bf16 out, N a multiple of 64): C = acc as usual, and in the same pass
   *   dot_out[((m / dot_seq_len) * (N / 64) + n / 64) * dot_seq_len + m % dot_seq_len] = sum over the 64 columns of head n / 64 of
   *   bf16(C[m, n]) * aux_in[m, n]
   * With C = dO (the attention-output gradient, produced by the proj dgrad GEMM) and aux_in = O this is D = rowsum(dO o O) in the
   * [n_seq, H, S] layout ub_attn_bwd wants (modeling_finetune.py:110-117 under autograd): the separate pass over O and dO goes away. */
  float* dot_out;
  int32_t dot_seq_len;
  int32_t reserved0;
} ub_gemm_epilogue;

/* a_mn_major / b_mn_major = 1: the operand is stored transposed, i.e. A is [K, lda>=M] / B is [K, ldb>=N]
 * row-major (used by weight-gradient GEMMs, where the contraction runs over tokens).                      */
UB_API int ub_gemm_bf16(const void* A, int64_t lda, int a_mn_major, const void* B, int64_t ldb, int b_mn_major,
                 void* C, int64_t ldc, int M, int N, int K, const ub_gemm_epilogue* ep, int split_k,
                 void* stream);

/* Several weight gradients over the same tokens in one launch — the four Linear layers of a transformer block
 * (modeling_finetune.py:56-119 under autograd: qkv, proj, fc1, fc2):  C_i[M_i, N_i] (fp32) += A_i^T B_i  with A_i = the bf16 output
 * gradient stored [K tokens, lda >= M_i] and B_i = the bf16 layer input stored [K tokens, ldb >= N_i]; up to 4 problems, any M_i /
 * N_i (multiples of 8), split_k ways along the tokens (fp32 reduce-add into C_i, which must hold the running gradient). */
typedef struct ub_gemm_problem {
  const void* A; int64_t lda;
  const void* B; int64_t ldb;
  float* C; int64_t ldc;
  int32_t M, N;
} ub_gemm_problem;
UB_API int ub_gemm_wgrad_multi(const ub_gemm_problem* problems, int n_problems, int K, int split_k, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused multi-head self-attention, head_dim 64 (flash-style: the S x S scores never reach HBM).
 *   qkv bf16 [n_seq*S, 3*H*64] (per row q|k|v, H heads x 64), o bf16 [n_seq*S, H*64], lse fp32 [n_seq,H,S].
 * Replaces modeling_finetune.py:110-116 (student Attention core) and clip.py:40-52 (nn.MultiheadAttention core);
 * ub_attn_bwd is their autograd backward (D_ws: fp32 [n_seq,H,S] scratch); ub_cls_attn is clip.py:95-96,183:
 * out[n_seq, S-1] = head-averaged softmax row of the CLS query (token 0) over the patch keys.
 * Every S runs on tcgen05 / TMEM kernels: S <= 240 without lse (the teacher's 197-token frames) and S <= 320 with lse / backward
 * (the student's visible tokens) keep the whole (sequence, head) item resident; longer sequences (the all-token passes of stage
 * 2 / 3, S = 1568: modeling_finetune.py:356-383, run_stage3.py:475-483) stream K / V (or Q / dO) chunks past 128-row tiles with an
 * online softmax forward and a two-pass backward (csrc/attention_long_tc.cu).
 * ---------------------------------------------------------------------------------------------- */
/* diagnostic: how many 4-CTA clusters of the GEMM kernel the device can hold at once (0 = cluster-of-4 tiles are not used) */
UB_API int ub_gemm_cluster4_capacity(void);

UB_API int ub_attn_fwd(const void* qkv, void* o, float* lse /* may be NULL */, int n_seq, int S, int H, float scale,
                       void* stream);
/* dbias (may be NULL): fp32 [3*H*64], += the column sums over all rows of the dq and dv thirds of dqkv — the q_bias / v_bias
 * gradients of modeling_finetune.py:104-108 (the key third has no bias and is left untouched) — accumulated by the kernels as they
 * store dqkv, which saves the separate pass over it.
 * o may be NULL when D_ws already holds D = rowsum(dO o O) in its [n_seq, H, S] layout (written by the GEMM that produced dO:
 * ub_gemm_epilogue.dot_out); otherwise D is computed here from o and d_o first. */
UB_API int ub_attn_bwd(const void* qkv, const void* o, const void* d_o, const float* lse, float* D_ws, void* dqkv, float* dbias,
                       int n_seq, int S, int H, float scale, void* stream);
UB_API int ub_cls_attn(const void* qkv, float* out, int n_seq, int S, int H, float scale, void* stream);

/* ------------------------------------------------------------------------------------------------
 * LayerNorm family (one warp per row, fp32 statistics; D multiple of 128, <= 1024).
 *   ub_layernorm_fwd   out[r] = LN(x[src_rows ? src_rows[r] : r]) * gamma + beta (+ post_add[post_idx[r]]); bf16 or fp32 out.
 *                      student norm1/norm2 (modeling_finetune.py:143-150), encoder.norm + gathered clip_pos_embed
 *                      (modeling_adaptation.py:168,318-320), teacher ln_1/ln_2 (clip.py:55-64), ln_post on gathered
 *                      visible tokens (clip.py:168 + run_stage1.py:393).
 *   ub_teacher_embed_ln  CLS/pos assembly + ln_pre (clip.py:150-152): E fp32 [frames*P, D] -> out fp32 [frames*(P+1), D].
 *   ub_layernorm_bwd   autograd backward of the student LNs fused with the residual-gradient add and the bf16 cast
 *                      (x DropPath scale) the following GEMMs consume; dgamma/dbeta are ACCUMULATED (red.add).
 *   ub_dec_tail_fwd/bwd  Linear_Decoder tail (modeling_adaptation.py:205-211): LN(C) then L2 normalise; fwd optionally
 *                      accumulates the alignment loss sum(2 - 2<out,tgt>) * loss_scale (run_stage1.py:431);
 *                      bwd takes the upstream gradient as go_scale * go.
 *   ub_l2norm_rows     x /= ||x|| per row (clip.py:173).
 * ---------------------------------------------------------------------------------------------- */
/* x: fp32 rows, or fp16 rows when x_f16 != 0 (the frozen teacher keeps its residual stream in fp16, as the reference's
 * autocast does; statistics are fp32 either way) */
UB_API int ub_layernorm_fwd(const void* x, int x_f16, const int* src_rows, const float* gamma, const float* beta, float eps,
                            const float* post_add, const int* post_idx, void* out, int out_fp32, int rows, int D,
                            void* stream);
/* out: fp32, or fp16 when out_f16 != 0; stats (may be NULL): fp32 [rows,2] = row (sum, sumsq) of the values written */
UB_API int ub_teacher_embed_ln(const float* E, const float* cls, const float* pos, const float* gamma, const float* beta,
                               float eps, void* out, int out_f16, float* stats, int frames, int P, int D, void* stream);
UB_API int ub_layernorm_bwd(const void* dy, const float* x, const float* gamma, float eps, const float* dx_in,
                            float* dx_out, void* dxs_out, const float* row_scale, int rows_per_scale, float* dgamma,
                            float* dbeta, float* dsum /* optional: += column sums of dxs (fp32) */, int rows, int D,
                            void* stream);
/* [loss_row_lo, loss_row_hi) / [go_row_lo, go_row_hi): the rows that take part in the loss and receive the upstream gradient — all
 * rows for clip_loss_data 'mixed', the first B_s clips for 'source', the rest for 'target' (run_stage1.py:418-423); rows outside
 * the range are still normalised and written by fwd, and get a zero gradient from bwd. */
UB_API int ub_dec_tail_fwd(const float* y, const float* gamma, const float* beta, float eps, float* out, const float* tgt,
                           float* loss_acc, float loss_scale, int loss_row_lo, int loss_row_hi, int rows, int D, void* stream);
UB_API int ub_dec_tail_bwd(const float* y, const float* gamma, const float* beta, float eps, const float* go,
                           float go_scale, int go_row_lo, int go_row_hi, void* dy_out, float* dgamma, float* dbeta, int rows, int D,
                           void* stream);
UB_API int ub_l2norm_rows(float* x, int rows, int D, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Token movement and the mask sampler.
 *   ub_patchify     fp32 clip [B,3,T,H,W] -> bf16 im2col rows [B*(T/tub)*(H/16)*(W/16), 3*tub*256]
 *                   (Conv3d stride==kernel as a GEMM: clip.py:123-128,146; modeling_finetune.py:165-174).
 *   ub_mask_select  run_stage1.py:379-387 (q != NULL: multinomial w/o replacement == top-n_vis of attn/q, q~Exp(1)
 *                   supplied by the caller) and utils.py:89-120 get_greedy_masks (q == NULL, k members).  Bit-exact.
 *                   mask uint8 [k, frames*P] (1 = masked), vis_idx / tea_rows int32 [k, frames/T, T*n_vis].
 *   ub_gather_rows  out[i,:] = in[(i / rows_per_group) * group_stride_rows + idx[i], :]  (rows_per_group == 0: no base)
 *                   — the `x[~mask]` gathers of modeling_adaptation.py:153,319 and run_stage1.py:393.
 *   ub_colsum_bf16  out[n] += sum_m x[m,n]  (bias gradients).
 *   ub_cast_scale_bf16  out = bf16(x * row_scale[row / rows_per_scale]).
 * ---------------------------------------------------------------------------------------------- */
UB_API int ub_patchify(const float* x, void* out, int B, int T, int H, int W, int tubelet, void* stream);
/* the same rows of the clip mixed as timm's batch-mode Mixup mixes it (stage-2 mixup_fn, engine_for_finetuning.py:86-87); x is
 * not written.  mix: DEVICE fp32 {apply, lam, 1 - lam, use_cutmix, t0, t1, h0, h1, w0, w1} (1 - lam computed in double, then
 * rounded).  apply == 0: ub_patchify.  cutmix: clip b takes clip B-1-b's values inside the half-open box [t0,t1) x [h0,h1) x
 * [w0,w1) of the T, H, W axes.  mixup: lam * x_b + (1 - lam) * x_{B-1-b}, both products and the sum rounded on their own in fp32
 * (bit-identical to torch's in-place mix).  B must be even. */
UB_API int ub_patchify_mix(const float* x, void* out, const float* mix, int B, int T, int H, int W, int tubelet, void* stream);
/* decoded uint8 frames [B,T,H,W,3] -> the same rows, with ToTensor + tensor_normalize(mean, std) applied on the way
 * (src/datasets/kinetics_sparse.py:236-243, 434-451); mean3 / std3 are HOST pointers to 3 floats.                     */
UB_API int ub_patchify_u8(const uint8_t* x, void* out, const float* mean3, const float* std3, int B, int T, int H, int W,
                          int tubelet, void* stream);
/* ub_patchify_mix of the frames ub_patchify_u8 reads: every byte normalised exactly as there, then mixed exactly as ub_patchify_mix
 * mixes (mix: the same DEVICE draw), so the rows equal ub_patchify of the torch-mixed normalised clip.  x is not written;
 * B even, H and W multiples of 16, x 16-byte aligned; mean3 / std3 are HOST pointers to 3 floats. */
UB_API int ub_patchify_mix_u8(const uint8_t* x, void* out, const float* mix, const float* mean3, const float* std3, int B, int T, int H,
                              int W, int tubelet, void* stream);
/* resize + patchify for the teacher: fp32 clip [B,3,T,H,W] (x_is_u8 = 0) or decoded uint8 frames [B,T,H,W,3] (x_is_u8 = 1,
 * normalised with the HOST mean3 / std3 as ub_patchify_u8 does, before the resize) -> bicubic resize of every (c, t) plane to
 * R x R (torch interpolate mode="bicubic", align_corners=False, antialias=False; no resize when R == H == W) -> bf16 im2col rows
 * [B*(T/tubelet)*(R/patch)^2, ld_out] in ub_patchify's token / feature order, for any even patch size.  ld_out >= 3*tubelet*patch^2,
 * a multiple of 8; the padding columns are written as zeros (a GEMM may contract over the padded K against zero weights). */
UB_API int ub_resize_patchify(const void* x, int x_is_u8, const float* mean3, const float* std3, void* out, int64_t ld_out, int B,
                              int T, int H, int W, int R, int patch, int tubelet, void* stream);
UB_API int ub_mask_select(const float* attn, const float* q, uint8_t* mask, int* vis_idx, int* tea_rows, int frames,
                          int P, int T, int k, int n_vis, void* stream);
UB_API int ub_gather_rows(const void* in, const int* idx, void* out, int64_t n_rows, int64_t row_bytes,
                          int rows_per_group, int64_t group_stride_rows, void* stream);
/* columns [skip_lo, skip_hi) are not accumulated (pass 0, 0 for none): the key third of the q|k|v bias has no gradient */
UB_API int ub_colsum_bf16(const void* x, int64_t ld, float* out, int M, int N, int skip_lo, int skip_hi, void* stream);
UB_API int ub_cast_scale_bf16(const float* x, void* out, const float* row_scale, int rows_per_scale, int64_t rows, int D,
                              void* stream);

/* ------------------------------------------------------------------------------------------------
 * Optimizer over the flat parameter arena [decay | no-decay]  (src/optim_factory.py:76-118,162-163; src/utils.py:631-643).
 * ---------------------------------------------------------------------------------------------- */
UB_API int ub_sumsq(const float* g, int64_t n, float* out /* accumulated */, void* stream);
UB_API int ub_adamw(float* p, const float* g, float* m, float* v, void* w_bf16 /* may be NULL */, int64_t n,
                    int64_t n_decay, float lr, float wd, float beta1, float beta2, float eps, int step, float grad_scale,
                    void* stream);
/* same update, per-step scalars in device memory: hyper[8] = lr, wd, beta1, beta2, eps, 1-beta1^t, sqrt(1-beta2^t), grad_scale
 * (lets the launch sit in a CUDA graph replayed every step).  gnorm_sq (may be NULL): += sum g^2 of the raw gradients read
 * by this very pass — the global gradient norm of utils.py:631-643 without a second sweep over the arena. */
UB_API int ub_adamw_dev(float* p, const float* g, float* m, float* v, void* w_bf16 /* may be NULL */, int64_t n,
                        int64_t n_decay, const float* hyper, float* gnorm_sq /* may be NULL */, void* stream);
/* Segmented form — the parameter groups of src/optim_factory.py:76-118 with a LayerDecayValueAssigner (run_stage2.py:616-617,
 * configs/stage2_config.yaml layer_decay 0.65): the arena is n_seg (<= 128) contiguous groups, seg_end4[s] (device int32) = end of
 * group s in units of 4 elements (ascending, last == n/4); hyper (device) = [-, -, beta1, beta2, eps, 1-beta1^t, sqrt(1-beta2^t),
 * grad_scale, lr[n_seg], wd[n_seg]] with lr[s] = schedule value * lr_scale of the group (engine_for_finetuning.py:76-81).
 * wd[s] < 0 marks a frozen group (requires_grad=False: left out of every group at optim_factory.py:83-84): untouched, and not
 * part of the gradient norm.  ub_sumsq_seg is the matching norm for clip_grad (frozen groups skipped). */
UB_API int ub_adamw_seg(float* p, const float* g, float* m, float* v, void* w_bf16 /* may be NULL */, int64_t n,
                        const int32_t* seg_end4, int n_seg, const float* hyper, float* gnorm_sq /* may be NULL */, void* stream);
UB_API int ub_sumsq_seg(const float* g, int64_t n, const int32_t* seg_end4, int n_seg, const float* hyper, float* out,
                        void* stream);
UB_API int ub_cast_bf16(const float* x, void* out, int64_t n, void* stream);
/* Model EMA of the stage-2 loop (timm 0.4.12 ModelEma.update, called after every optimizer update at
 * engine_for_finetuning.py:126-127): for every element of the fp32 arena, ema = fl(fl(ema * decay) + fl(p * one_minus_decay)),
 * the two products and the sum rounded on their own (no FMA: bit-identical to torch's `ema_v * decay + (1. - decay) * model_v`
 * in fp32), and ema_w16 = bf16 of the new ema, rounded as ub_cast_bf16 rounds.  The caller passes (float)decay and
 * (float)(1.0 - decay), 1 - decay computed in double.  n: a positive multiple of 4.  p is only read. */
UB_API int ub_ema_update(float* ema, void* ema_w16, const float* p, int64_t n, float decay, float one_minus_decay, void* stream);

/* DropPath factors for one step (src/models/modeling_finetune.py:42-50 via timm drop_path; rates = linspace(0, drop_path, depth),
 * :311): out fp32 [depth, 2, B] = floor(keep_l + u) / keep_l, u ~ U[0,1) from Philox4x32-10 keyed by `seed` with counter
 * (element / 4, 0, *step); the kernel then advances the DEVICE counter *step by one, so a captured launch draws fresh factors on
 * every CUDA-graph replay.  rates: device fp32 [depth].  Consumed as ub_gemm_epilogue.row_scale (forward) and as the row_scale of
 * ub_layernorm_bwd / ub_cast_scale_bf16 (backward). */
UB_API int ub_drop_path_draw(const float* rates, float* out, int depth, int B, uint64_t seed, uint64_t* step, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Data-parallel optimizer step fused with its collective (replaces DistributedDataParallel's bucketed all-reduce,
 * run_stage1.py:809 / run_stage2.py:641 / run_stage3.py:1246, + utils.py:608-622 + optim_factory.py:162-163):
 * reduce-scatter of the gradient arena inside the NVSwitch (multimem.ld_reduce), AdamW on the rank's slice of the decay
 * segment, all-gather of the refreshed bf16 shadow (multimem.st) — one kernel, no NCCL call.  `g_mc`, `w16_mc`,
 * `gnorm_sq_mc`, `flags_mc` are MULTICAST addresses of symmetric allocations (same size and offset on every rank);
 * `w16`, `flags` the rank's own mappings of the same memory.  p / m / v are local; their decay segment is updated on the
 * owning rank only (ZeRO-1), the no-decay segment on every rank.  flags: ub_nvls_slots() zero-initialised uint32 (symmetric),
 * epoch: ub_nvls_slots()/2 zero-initialised uint32 (local), err: one zero-initialised int32 (local; 1 / 2 / 3 = a peer never
 * reached the entry / exit / mid barrier within UB_NVLS_SPIN_S seconds (default 120).  The error is STICKY: the CTA that gave up
 * applies no update, and every later launch returns immediately without touching p / m / v or the shadows, so a stalled rank
 * can never train on partial gradient sums; the host polls err at its log points and raises on every rank).  hyper[8] as for ub_adamw_dev with
 * grad_scale = 1/world.  Every rank must launch it the same number of times.
 * g_peers / w16_peers (host arrays of `world` device pointers, by rank: every rank's mapping of the gradient arena / shadow,
 * own rank included): when given and world is 2, 4 or 8 the gradients are read with plain NVLink peer loads and summed in
 * rank order (bitwise reproducible) and the shadow is written with one store per peer, instead of multimem.ld_reduce /
 * multimem.st; the barriers and the gradient norm always use the multicast mapping.
 * stage_peers (every rank's mapping of a symmetric staging buffer of world * ceil(n_decay/8/world) * 8 floats): selects the
 * PUSH form — each rank first writes its gradients of every peer's slice into slot[rank] of that peer's staging buffer
 * (posted NVLink writes), a grid-wide cross-GPU counter follows, then the owner sums local copies in rank order.
 * prepushed != 0 (push form only): the caller has ALREADY filled the staging buffers — slot[rank] of every peer holds this rank's
 * gradients of that peer's slice — with peer-to-peer copies issued during backward and stream-ordered before this launch (the
 * overlap DistributedDataParallel gets from bucketed all-reduces); the kernel then skips its scatter phase and the mid barrier.
 * ---------------------------------------------------------------------------------------------- */
UB_API int ub_nvls_slots(void);
UB_API int ub_adamw_nvls(float* p, const float* g_mc, float* m, float* v, void* w16, void* w16_mc, int64_t n, int64_t n_decay,
                         int rank, int world, const float* hyper, float* gnorm_sq_mc /* may be NULL */, uint32_t* flags,
                         uint32_t* flags_mc, uint32_t* epoch, int32_t* err, const void* const* g_peers /* host array [world] or NULL */,
                         void* const* w16_peers /* host array [world] or NULL */,
                         void* const* stage_peers /* host array [world] or NULL */, int prepushed, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Classification heads and stage-3 pseudo-label fusion (fp32, small).
 *   ub_meanpool_fwd/bwd      x.mean(1): modeling_finetune.py:374-376 (stage 2), run_stage3.py:333-338 pool_outputs
 *   ub_linear_small_fwd/bwd  few-output Linear: `head` (modeling_finetune.py:382), `src_classifier` (run_stage3.py:1193);
 *                            bwd ACCUMULATES dW / db, dx optional
 *   ub_softmax_ce            loss_acc += scale * sum_b w_b CE(logits_b, y_b); dlogits = its gradient
 *                            (engine_for_finetuning.py:39; run_stage3.py:486, 606-615)
 *   ub_clip_zero_shot        utils.py:62-68: per-frame softmax(100 * cosine) averaged over the T frames of a clip
 *   ub_pseudo_label_fusion   run_stage3.py:489-490,556-587 ('clip_matchORconf'): msp / argmax of the student, selection
 *                            mask, pseudo labels (= student argmax, :576) and per-sample loss weights
 * ---------------------------------------------------------------------------------------------- */
UB_API int ub_meanpool_fwd(const float* x, float* out, int B, int N, int D, void* stream);
UB_API int ub_meanpool_bwd(const float* g, float* dx, int B, int N, int D, void* stream);
UB_API int ub_linear_small_fwd(const float* x, const float* W, const float* bias, float* out, int B, int C, int D,
                               void* stream);
UB_API int ub_linear_small_bwd(const float* x, const float* W, const float* dout, float* dx, float* dW, float* db, int B,
                               int C, int D, void* stream);
UB_API int ub_softmax_ce(const float* logits, const int* labels, const float* weights, float scale, float* loss_acc,
                         float* dlogits, int B, int C, void* stream);
/* soft-target CE of batch-mode mixup with label smoothing (timm SoftTargetCrossEntropy of mixup_target, run_stage2.py:702):
 * t_bc = lam (c == y_b ? on : off) + (1 - lam) (c == y_{B-1-b} ? on : off), off = s / C, on = 1 - s + off; mix: DEVICE fp32
 * {lam, on, off}.  loss_acc += scale * sum_b sum_c -t_bc log_softmax_c;  dlogits = scale * (softmax * sum_c t_bc - t).
 * lam = 1: label smoothing alone (LabelSmoothingCrossEntropy(s), CrossEntropyLoss(label_smoothing=s)). */
UB_API int ub_soft_target_ce(const float* logits, const int* labels, const float* mix, float scale, float* loss_acc,
                             float* dlogits, int B, int C, void* stream);
UB_API int ub_clip_zero_shot(const float* img_feat, const float* text_feat, float* probs, int B, int T, int C, int D,
                             void* stream);
UB_API int ub_pseudo_label_fusion(const float* logits_full, const float* clip_probs, float threshold, int conf_weighted,
                                  float* msp, int* pseudo, uint8_t* sel, float* weight, int B, int C, void* stream);

#ifdef __cplusplus
}
#endif
#endif
