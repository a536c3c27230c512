// Classification heads and the stage-3 pseudo-label fusion (small, latency-bound kernels; everything is fp32).
//
//   ub_meanpool_fwd/bwd      x.mean(1) over tokens: stage-2 `x.mean(1)` before fc_norm (modeling_finetune.py:374-376),
//                            stage-3 pool_outputs (run_stage3.py:333-338)
//   ub_linear_small_fwd/bwd  Linear with a handful of outputs: stage-2 `head` (modeling_finetune.py:382),
//                            stage-3 `src_classifier = nn.Linear(768, C)` (run_stage3.py:1193)
//   ub_softmax_ce            (weighted) cross-entropy forward + gradient: engine_for_finetuning.py:39,
//                            run_stage3.py:486 (source CE), :606-615 (confidence-weighted target CE)
//   ub_soft_target_ce        stage-2 mixup / label-smoothing loss + gradient (run_stage2.py:702), target built on the fly
//   ub_clip_zero_shot        utils.clip_infer after encode_image (utils.py:62-68): per-frame softmax(100 cos) mean over frames
//   ub_pseudo_label_fusion   selection_strategy 'clip_matchORconf' (run_stage3.py:489-490, 556-587): argmax / max-softmax of
//                            the student, match-or-exactly-one-confident selection, per-sample loss weights
#include "common.cuh"
#include "../../include/unite_b200.h"

namespace ub {

// out[b, d] = mean_n x[b, n, d];  grid (D/128, B), 128 threads, each thread one column, rows strided by 8 sub-rows
__global__ void __launch_bounds__(256) meanpool_fwd_kernel(const float* __restrict__ x, float* __restrict__ out, int N, int D) {
  __shared__ float s_part[8][32];
  const int b = blockIdx.y, d = blockIdx.x * 32 + (threadIdx.x & 31), rg = threadIdx.x >> 5;
  float acc = 0.f;
  if (d < D) {
    const float* p = x + ((int64_t)b * N) * D + d;
    for (int n = rg; n < N; n += 8) acc += p[(int64_t)n * D];
  }
  s_part[rg][threadIdx.x & 31] = acc;
  __syncthreads();
  if (rg == 0 && d < D) {
    float s = 0.f;
#pragma unroll
    for (int g = 0; g < 8; ++g) s += s_part[g][threadIdx.x];
    out[(int64_t)b * D + d] = s / (float)N;
  }
}

// dx[b, n, :] = g[b, :] / N   (fp32, 128-bit stores)
__global__ void __launch_bounds__(256) meanpool_bwd_kernel(const float4* __restrict__ g, float4* __restrict__ dx, int N, int D4,
                                                           long total4, float invN) {
  for (long id = (long)blockIdx.x * blockDim.x + threadIdx.x; id < total4; id += (long)gridDim.x * blockDim.x) {
    const int d4 = (int)(id % D4);
    const long b = id / ((long)N * D4);
    float4 v = g[b * D4 + d4];
    v.x *= invN; v.y *= invN; v.z *= invN; v.w *= invN;
    dx[id] = v;
  }
}

// out[b, c] = <x[b,:], W[c,:]> + bias[c];  one warp per (b, c)
__global__ void __launch_bounds__(256) linear_small_fwd_kernel(const float* __restrict__ x, const float* __restrict__ W,
                                                               const float* __restrict__ bias, float* __restrict__ out, int B,
                                                               int C, int D) {
  const int w = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (w >= B * C) return;
  const int b = w / C, c = w % C;
  float acc = 0.f;
  for (int d = lane; d < D; d += 32) acc += x[(int64_t)b * D + d] * W[(int64_t)c * D + d];
  acc = warp_sum(acc);
  if (lane == 0) out[w] = acc + (bias ? bias[c] : 0.f);
}

// dx[b, d] = sum_c dout[b,c] W[c,d] (optional);  dW[c,d] += sum_b dout[b,c] x[b,d];  db[c] += sum_b dout[b,c]
__global__ void __launch_bounds__(256) linear_small_bwd_kernel(const float* __restrict__ x, const float* __restrict__ W,
                                                               const float* __restrict__ dout, float* __restrict__ dx,
                                                               float* __restrict__ dW, float* __restrict__ db, int B, int C, int D) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d < D) {
    if (dx != nullptr) {
      for (int b = 0; b < B; ++b) {
        float a = 0.f;
        for (int c = 0; c < C; ++c) a += dout[b * C + c] * W[(int64_t)c * D + d];
        dx[(int64_t)b * D + d] = a;
      }
    }
    if (dW != nullptr) {
      for (int c = 0; c < C; ++c) {
        float a = 0.f;
        for (int b = 0; b < B; ++b) a += dout[b * C + c] * x[(int64_t)b * D + d];
        dW[(int64_t)c * D + d] += a;
      }
    }
  }
  if (db != nullptr && blockIdx.x == 0 && threadIdx.x < C) {
    float a = 0.f;
    for (int b = 0; b < B; ++b) a += dout[b * C + threadIdx.x];
    db[threadIdx.x] += a;
  }
}

// loss_acc += scale * sum_b w_b * CE(logits[b], label[b]);  dlogits[b,c] = scale * w_b * (softmax(logits[b])[c] - [c == label[b]])
// one warp per sample, C <= 1024
__global__ void __launch_bounds__(256) softmax_ce_kernel(const float* __restrict__ logits, const int* __restrict__ labels,
                                                         const float* __restrict__ weights, float scale, float* __restrict__ loss_acc,
                                                         float* __restrict__ dlogits, int B, int C) {
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  const float* l = logits + (int64_t)b * C;
  float mx = -INFINITY;
  for (int c = lane; c < C; c += 32) mx = fmaxf(mx, l[c]);
  mx = warp_max(mx);
  float se = 0.f;
  for (int c = lane; c < C; c += 32) se += expf(l[c] - mx);
  se = warp_sum(se);
  const int y = labels[b];
  const float w = (weights ? weights[b] : 1.0f) * scale;
  const float lse = mx + logf(se);
  if (lane == 0 && loss_acc != nullptr) atomicAdd(loss_acc, w * (lse - l[y]));
  if (dlogits != nullptr)
    for (int c = lane; c < C; c += 32) dlogits[(int64_t)b * C + c] = w * (expf(l[c] - lse) - (c == y ? 1.0f : 0.0f));
}

// Soft-target cross-entropy of batch-mode mixup (timm SoftTargetCrossEntropy(mixup_target(...)), run_stage2.py:702 with mixup):
//   t_bc = lam * (c == y_b ? on : off) + (1 - lam) * (c == y_{B-1-b} ? on : off)      mix (device fp32) = {lam, on, off}
//   loss_acc += scale * sum_b sum_c -t_bc * log_softmax(logits_b)_c;  dlogits[b,c] = scale * (softmax_bc * sum_c t_bc - t_bc)
// The [B,C] target is never stored.  lam = 1 is label smoothing alone (LabelSmoothingCrossEntropy, CrossEntropyLoss(label_smoothing)).
// One warp per sample, like softmax_ce.
__global__ void __launch_bounds__(256) soft_target_ce_kernel(const float* __restrict__ logits, const int* __restrict__ labels,
                                                             const float* __restrict__ mix, float scale, float* __restrict__ loss_acc,
                                                             float* __restrict__ dlogits, int B, int C) {
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  const float lam = mix[0], on = mix[1], off = mix[2], lam1 = 1.0f - lam;
  const int y = labels[b], y2 = labels[B - 1 - b];
  const float* l = logits + (int64_t)b * C;
  float mx = -INFINITY;
  for (int c = lane; c < C; c += 32) mx = fmaxf(mx, l[c]);
  mx = warp_max(mx);
  float se = 0.f, st = 0.f;
  for (int c = lane; c < C; c += 32) {
    se += expf(l[c] - mx);
    st += lam * (c == y ? on : off) + lam1 * (c == y2 ? on : off);
  }
  se = warp_sum(se);
  st = warp_sum(st);
  const float lse = mx + logf(se);
  float loss = 0.f;
  for (int c = lane; c < C; c += 32) {
    const float t = lam * (c == y ? on : off) + lam1 * (c == y2 ? on : off);
    loss += t * (lse - l[c]);
    if (dlogits != nullptr) dlogits[(int64_t)b * C + c] = scale * (expf(l[c] - lse) * st - t);
  }
  loss = warp_sum(loss);
  if (lane == 0 && loss_acc != nullptr) atomicAdd(loss_acc, scale * loss);
}

// probs[b, c] = mean_t softmax_c(100 * <img[b*T+t]/|.|, txt[c]/|.|>)   one block per clip, one warp per frame, C <= 32*? (loop)
__global__ void __launch_bounds__(256) clip_zero_shot_kernel(const float* __restrict__ img, const float* __restrict__ txt,
                                                             float* __restrict__ probs, int T, int C, int D) {
  extern __shared__ float s_acc[];   // [C] accumulated probabilities, then [warps][C] similarities
  const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  float* sim = s_acc + C + warp * C;
  for (int c = threadIdx.x; c < C; c += blockDim.x) s_acc[c] = 0.f;
  __syncthreads();
  for (int t = warp; t < T; t += nw) {
    const float* f = img + ((int64_t)b * T + t) * D;
    float nf = 0.f;
    for (int d = lane; d < D; d += 32) nf += f[d] * f[d];
    nf = rsqrtf(warp_sum(nf));
    float mx = -INFINITY;
    for (int c = 0; c < C; ++c) {
      const float* g = txt + (int64_t)c * D;
      float dot = 0.f, ng = 0.f;
      for (int d = lane; d < D; d += 32) { dot += f[d] * g[d]; ng += g[d] * g[d]; }
      dot = warp_sum(dot);
      ng = warp_sum(ng);
      const float s = 100.0f * dot * nf * rsqrtf(ng);
      if (lane == 0) sim[c] = s;
      mx = fmaxf(mx, s);
    }
    __syncwarp();
    float se = 0.f;
    for (int c = lane; c < C; c += 32) se += expf(sim[c] - mx);
    se = warp_sum(se);
    for (int c = lane; c < C; c += 32) atomicAdd(&s_acc[c], expf(sim[c] - mx) / se);
    __syncwarp();
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) probs[(int64_t)b * C + c] = s_acc[c] / (float)T;
}

// one warp per sample:  probs = softmax(logits_full), (msp, pred) = max/argmax (first maximum, like torch.max),
// (clip_msp, clip_pred) likewise;  match = clip_pred == pred;  conf = (msp >= thr) xor (clip_msp >= thr), and not match;
// sel = match | conf;  pseudo = pred;  weight = sel ? (conf_weighted ? msp : 1) : 0
__global__ void __launch_bounds__(256) pseudo_label_fusion_kernel(const float* __restrict__ logits, const float* __restrict__ clip_probs,
                                                                  float thr, int conf_weighted, float* __restrict__ msp_out,
                                                                  int* __restrict__ pseudo, uint8_t* __restrict__ sel,
                                                                  float* __restrict__ weight, int B, int C) {
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  const float* l = logits + (int64_t)b * C;
  const float* q = clip_probs + (int64_t)b * C;
  float mx = -INFINITY, cmx = -INFINITY;
  int am = 0x7fffffff, cam = 0x7fffffff;
  for (int c = lane; c < C; c += 32) {
    if (l[c] > mx) { mx = l[c]; am = c; }
    if (q[c] > cmx) { cmx = q[c]; cam = c; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, mx, o); const int a2 = __shfl_xor_sync(0xffffffffu, am, o);
    if (m2 > mx || (m2 == mx && a2 < am)) { mx = m2; am = a2; }
    const float c2 = __shfl_xor_sync(0xffffffffu, cmx, o); const int ca2 = __shfl_xor_sync(0xffffffffu, cam, o);
    if (c2 > cmx || (c2 == cmx && ca2 < cam)) { cmx = c2; cam = ca2; }
  }
  float se = 0.f;
  for (int c = lane; c < C; c += 32) se += expf(l[c] - mx);
  se = warp_sum(se);
  const float msp = 1.0f / se;             // softmax value of the arg-max class
  if (lane == 0) {
    const bool match = cam == am;
    const bool conf = ((msp >= thr) != (cmx >= thr)) && !match;
    const bool s = match || conf;
    msp_out[b] = msp;
    pseudo[b] = am;
    sel[b] = s ? 1 : 0;
    weight[b] = s ? (conf_weighted ? msp : 1.0f) : 0.0f;
  }
}

}  // namespace ub

using namespace ub;

extern "C" int ub_meanpool_fwd(const float* x, float* out, int B, int N, int D, void* stream) {
  UB_REQUIRE(x && out && B > 0 && N > 0 && D > 0, "meanpool_fwd: bad arguments");
  dim3 grid((D + 31) / 32, B);
  UB_LAUNCH(meanpool_fwd_kernel, grid, 256, 0, (cudaStream_t)stream, x, out, N, D);
  return check_launch("meanpool_fwd_kernel");
}

extern "C" int ub_meanpool_bwd(const float* g, float* dx, int B, int N, int D, void* stream) {
  UB_REQUIRE(g && dx && B > 0 && N > 0 && D > 0 && D % 4 == 0, "meanpool_bwd: bad arguments");
  const long total4 = (long)B * N * (D / 4);
  long blocks = (total4 + 255) / 256;
  const long cap = (long)sm_count() * 16;
  UB_LAUNCH(meanpool_bwd_kernel, (int)(blocks < cap ? blocks : cap), 256, 0, (cudaStream_t)stream, (const float4*)g, (float4*)dx, N, D / 4, total4,
                                                                                           1.0f / (float)N);
  return check_launch("meanpool_bwd_kernel");
}

extern "C" int ub_linear_small_fwd(const float* x, const float* W, const float* bias, float* out, int B, int C, int D, void* stream) {
  UB_REQUIRE(x && W && out && B > 0 && C > 0 && D > 0, "linear_small_fwd: bad arguments");
  UB_LAUNCH(linear_small_fwd_kernel, (B * C + 7) / 8, 256, 0, (cudaStream_t)stream, x, W, bias, out, B, C, D);
  return check_launch("linear_small_fwd_kernel");
}

extern "C" int ub_linear_small_bwd(const float* x, const float* W, const float* dout, float* dx, float* dW, float* db, int B, int C,
                                   int D, void* stream) {
  UB_REQUIRE(x && W && dout && B > 0 && C > 0 && C <= 256 && D > 0, "linear_small_bwd: bad arguments (C <= 256)");
  UB_LAUNCH(linear_small_bwd_kernel, (D + 255) / 256, 256, 0, (cudaStream_t)stream, x, W, dout, dx, dW, db, B, C, D);
  return check_launch("linear_small_bwd_kernel");
}

extern "C" int ub_softmax_ce(const float* logits, const int* labels, const float* weights, float scale, float* loss_acc,
                             float* dlogits, int B, int C, void* stream) {
  UB_REQUIRE(logits && labels && B > 0 && C > 0, "softmax_ce: bad arguments");
  UB_LAUNCH(softmax_ce_kernel, (B + 7) / 8, 256, 0, (cudaStream_t)stream, logits, labels, weights, scale, loss_acc, dlogits, B, C);
  return check_launch("softmax_ce_kernel");
}

extern "C" int ub_soft_target_ce(const float* logits, const int* labels, const float* mix, float scale, float* loss_acc, float* dlogits,
                                 int B, int C, void* stream) {
  UB_REQUIRE(logits && labels && mix && B > 0 && C > 0, "soft_target_ce: bad arguments");
  UB_LAUNCH(soft_target_ce_kernel, (B + 7) / 8, 256, 0, (cudaStream_t)stream, logits, labels, mix, scale, loss_acc, dlogits, B, C);
  return check_launch("soft_target_ce_kernel");
}

extern "C" int ub_clip_zero_shot(const float* img_feat, const float* text_feat, float* probs, int B, int T, int C, int D,
                                 void* stream) {
  UB_REQUIRE(img_feat && text_feat && probs && B > 0 && T > 0 && C > 0 && D > 0, "clip_zero_shot: bad arguments");
  const size_t smem = (size_t)(C + 8 * C) * sizeof(float);
  UB_REQUIRE(smem <= 48 * 1024, "clip_zero_shot: too many classes (C=%d)", C);
  UB_LAUNCH(clip_zero_shot_kernel, B, 256, smem, (cudaStream_t)stream, img_feat, text_feat, probs, T, C, D);
  return check_launch("clip_zero_shot_kernel");
}

extern "C" int ub_pseudo_label_fusion(const float* logits_full, const float* clip_probs, float threshold, int conf_weighted,
                                      float* msp, int* pseudo, uint8_t* sel, float* weight, int B, int C, void* stream) {
  UB_REQUIRE(logits_full && clip_probs && msp && pseudo && sel && weight && B > 0 && C > 0, "pseudo_label_fusion: bad arguments");
  UB_LAUNCH(pseudo_label_fusion_kernel, (B + 7) / 8, 256, 0, (cudaStream_t)stream, logits_full, clip_probs, threshold, conf_weighted, msp,
                                                                            pseudo, sel, weight, B, C);
  return check_launch("pseudo_label_fusion_kernel");
}
