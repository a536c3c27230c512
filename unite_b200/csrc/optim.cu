// Fused multi-tensor AdamW over the flat parameter arena (+ global grad-norm, + bf16 weight refresh).
//
// Replaces   src/optim_factory.py:162-163 (torch.optim.AdamW over two param groups: decay / no-decay,
//            optim_factory.py:76-118), src/utils.py:631-643 (get_grad_norm_: ~150 per-tensor norm kernels) and
//            the bf16 re-cast of the weights every GEMM of the next step consumes.
// All student parameters live in ONE fp32 buffer laid out [decay params | no-decay params]; gradients,
// exp_avg, exp_avg_sq are parallel buffers; `w_bf16` is the bf16 shadow the GEMMs read.
#include "common.cuh"
#include "../../include/unite_b200.h"

namespace ub {

// sum of squares of a flat fp32 buffer, accumulated into out[0] with one red.add per block
__global__ void __launch_bounds__(256) sumsq_kernel(const float4* __restrict__ g, long n4, float* __restrict__ out) {
  __shared__ float s_part[8];
  float acc = 0.f;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const float4 v = g[i];
    acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += s_part[w];
    atomicAdd(out, s);
  }
}

// torch.optim.AdamW semantics (decoupled decay):  p *= 1 - lr*wd;  m,v EMA;  p -= lr/bc1 * m / (sqrt(v)/sqrt(bc2) + eps)
// g is multiplied by grad_scale first (1/world_size when the all-reduce summed, or a clip coefficient).
__global__ void __launch_bounds__(256) adamw_kernel(float4* __restrict__ p, const float4* __restrict__ g, float4* __restrict__ m,
                                                    float4* __restrict__ v, uint2* __restrict__ w_bf16, long n4, long n4_decay,
                                                    float lr, float wd, float beta1, float beta2, float eps, float bc1,
                                                    float bc2_sqrt, float grad_scale) {
  const float step_size = lr / bc1;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    float4 pp = p[i], gg = g[i], mm = m[i], vv = v[i];
    const float decay = (i < n4_decay) ? (1.0f - lr * wd) : 1.0f;
#define UB_ADAM_ONE(c)                                               \
  {                                                                  \
    const float gr = gg.c * grad_scale;                              \
    pp.c *= decay;                                                   \
    mm.c = beta1 * mm.c + (1.0f - beta1) * gr;                       \
    vv.c = beta2 * vv.c + (1.0f - beta2) * gr * gr;                  \
    pp.c -= step_size * (mm.c / (sqrtf(vv.c) / bc2_sqrt + eps));     \
  }
    UB_ADAM_ONE(x) UB_ADAM_ONE(y) UB_ADAM_ONE(z) UB_ADAM_ONE(w)
#undef UB_ADAM_ONE
    p[i] = pp; m[i] = mm; v[i] = vv;
    if (w_bf16) {
      uint2 o;
      o.x = pack_bf16x2(pp.x, pp.y);
      o.y = pack_bf16x2(pp.z, pp.w);
      w_bf16[i] = o;
    }
  }
}

// Same update with the per-step scalars read from DEVICE memory (hyper[8] = lr, wd, beta1, beta2, eps, bc1, sqrt(bc2),
// grad_scale), so the launch can live inside a CUDA graph that is replayed every step while the host only refreshes
// those 32 bytes.
__global__ void __launch_bounds__(256) adamw_dev_kernel(float4* __restrict__ p, const float4* __restrict__ g, float4* __restrict__ m,
                                                        float4* __restrict__ v, uint2* __restrict__ w_bf16, long n4, long n4_decay,
                                                        const float* __restrict__ hyper, float* __restrict__ gnorm_sq) {
  __shared__ float s_part[8];
  float gacc = 0.f;                    // sum of squares of the raw gradients this thread reads (utils.py:631-643 for free)
  const float lr = hyper[0], wd = hyper[1], beta1 = hyper[2], beta2 = hyper[3], eps = hyper[4], bc1 = hyper[5], bc2_sqrt = hyper[6],
              grad_scale = hyper[7];
  const float step_size = lr / bc1;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    float4 pp = p[i], gg = g[i], mm = m[i], vv = v[i];
    gacc += gg.x * gg.x + gg.y * gg.y + gg.z * gg.z + gg.w * gg.w;
    const float decay = (i < n4_decay) ? (1.0f - lr * wd) : 1.0f;
#define UB_ADAM_ONE(c)                                               \
  {                                                                  \
    const float gr = gg.c * grad_scale;                              \
    pp.c *= decay;                                                   \
    mm.c = beta1 * mm.c + (1.0f - beta1) * gr;                       \
    vv.c = beta2 * vv.c + (1.0f - beta2) * gr * gr;                  \
    pp.c -= step_size * (mm.c / (sqrtf(vv.c) / bc2_sqrt + eps));     \
  }
    UB_ADAM_ONE(x) UB_ADAM_ONE(y) UB_ADAM_ONE(z) UB_ADAM_ONE(w)
#undef UB_ADAM_ONE
    p[i] = pp; m[i] = mm; v[i] = vv;
    if (w_bf16) {
      uint2 o;
      o.x = pack_bf16x2(pp.x, pp.y);
      o.y = pack_bf16x2(pp.z, pp.w);
      w_bf16[i] = o;
    }
  }
  if (gnorm_sq != nullptr) {
    gacc = warp_sum(gacc);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = gacc;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += s_part[w];
      atomicAdd(gnorm_sq, t);
    }
  }
}

// Segmented form: the arena is a sequence of n_seg contiguous parameter groups (src/optim_factory.py:76-118 with a
// LayerDecayValueAssigner: one group per (layer id, decay / no-decay), each with its own lr = schedule * lr_scale and weight
// decay, run_stage2.py:616-617 / engine_for_finetuning.py:76-81).  seg_end4[s] = end of group s in float4 units (ascending,
// last == n4); hyper = [-, -, beta1, beta2, eps, 1-beta1^t, sqrt(1-beta2^t), grad_scale, lr[n_seg], wd[n_seg]] in device
// memory (refreshed by one small async copy per step, so the launch can sit in a CUDA graph).  wd[s] < 0 marks a FROZEN
// group (requires_grad=False: optim_factory.py:83-84 leaves it out of every param group): p, m, v stay untouched and its
// gradient does not enter the norm.  Every thread walks the groups with a cursor — its indices only grow.
constexpr int kMaxSeg = 128;
__global__ void __launch_bounds__(256) adamw_seg_kernel(float4* __restrict__ p, const float4* __restrict__ g, float4* __restrict__ m,
                                                        float4* __restrict__ v, uint2* __restrict__ w_bf16, long n4,
                                                        const int* __restrict__ seg_end4, int n_seg, const float* __restrict__ hyper,
                                                        float* __restrict__ gnorm_sq) {
  __shared__ float s_part[8];
  __shared__ float s_lr[kMaxSeg], s_wd[kMaxSeg];
  __shared__ int s_end[kMaxSeg];
  for (int s = threadIdx.x; s < n_seg; s += blockDim.x) {
    s_end[s] = seg_end4[s];
    s_lr[s] = hyper[8 + s];
    s_wd[s] = hyper[8 + n_seg + s];
  }
  __syncthreads();
  float gacc = 0.f;
  const float beta1 = hyper[2], beta2 = hyper[3], eps = hyper[4], bc1 = hyper[5], bc2_sqrt = hyper[6], grad_scale = hyper[7];
  int seg = 0;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    while (seg < n_seg - 1 && i >= (long)s_end[seg]) ++seg;
    const float lr = s_lr[seg], wd = s_wd[seg];
    if (wd < 0.f) continue;                                   // frozen group
    float4 pp = p[i], gg = g[i], mm = m[i], vv = v[i];
    gacc += gg.x * gg.x + gg.y * gg.y + gg.z * gg.z + gg.w * gg.w;
    const float decay = 1.0f - lr * wd;
    const float step_size = lr / bc1;
#define UB_ADAM_ONE(c)                                               \
  {                                                                  \
    const float gr = gg.c * grad_scale;                              \
    pp.c *= decay;                                                   \
    mm.c = beta1 * mm.c + (1.0f - beta1) * gr;                       \
    vv.c = beta2 * vv.c + (1.0f - beta2) * gr * gr;                  \
    pp.c -= step_size * (mm.c / (sqrtf(vv.c) / bc2_sqrt + eps));     \
  }
    UB_ADAM_ONE(x) UB_ADAM_ONE(y) UB_ADAM_ONE(z) UB_ADAM_ONE(w)
#undef UB_ADAM_ONE
    p[i] = pp; m[i] = mm; v[i] = vv;
    if (w_bf16) {
      uint2 o;
      o.x = pack_bf16x2(pp.x, pp.y);
      o.y = pack_bf16x2(pp.z, pp.w);
      w_bf16[i] = o;
    }
  }
  if (gnorm_sq != nullptr) {
    gacc = warp_sum(gacc);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = gacc;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += s_part[w];
      atomicAdd(gnorm_sq, t);
    }
  }
}

// sum of squares over the non-frozen groups only (clip_grad needs the norm before the update)
__global__ void __launch_bounds__(256) sumsq_seg_kernel(const float4* __restrict__ g, long n4, const int* __restrict__ seg_end4, int n_seg,
                                                        const float* __restrict__ hyper, float* __restrict__ out) {
  __shared__ float s_part[8];
  __shared__ float s_wd[kMaxSeg];
  __shared__ int s_end[kMaxSeg];
  for (int s = threadIdx.x; s < n_seg; s += blockDim.x) {
    s_end[s] = seg_end4[s];
    s_wd[s] = hyper[8 + n_seg + s];
  }
  __syncthreads();
  float acc = 0.f;
  int seg = 0;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    while (seg < n_seg - 1 && i >= (long)s_end[seg]) ++seg;
    if (s_wd[seg] < 0.f) continue;
    const float4 v = g[i];
    acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += s_part[w];
    atomicAdd(out, s);
  }
}

__global__ void __launch_bounds__(256) cast_bf16_kernel(const float4* __restrict__ x, uint2* __restrict__ out, long n4) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const float4 v = x[i];
    uint2 o;
    o.x = pack_bf16x2(v.x, v.y);
    o.y = pack_bf16x2(v.z, v.w);
    out[i] = o;
  }
}

// Model EMA (timm 0.4.12 ModelEma.update): ema = fl(fl(ema * decay) + fl(p * one_minus_decay)), each product and the sum rounded
// on its own (no FMA), as torch evaluates `ema_v * decay + (1. - decay) * model_v` in fp32; the bf16 shadow of the new value is
// written in the same pass, so the EMA model can be evaluated at any time without a cast pass.
__global__ void __launch_bounds__(256) ema_update_kernel(float4* __restrict__ ema, uint2* __restrict__ ema_w16, const float4* __restrict__ p,
                                                         long n4, float decay, float one_minus_decay) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    float4 e = ema[i];
    const float4 q = p[i];
    e.x = __fadd_rn(__fmul_rn(e.x, decay), __fmul_rn(q.x, one_minus_decay));
    e.y = __fadd_rn(__fmul_rn(e.y, decay), __fmul_rn(q.y, one_minus_decay));
    e.z = __fadd_rn(__fmul_rn(e.z, decay), __fmul_rn(q.z, one_minus_decay));
    e.w = __fadd_rn(__fmul_rn(e.w, decay), __fmul_rn(q.w, one_minus_decay));
    ema[i] = e;
    uint2 o;
    o.x = pack_bf16x2(e.x, e.y);
    o.y = pack_bf16x2(e.z, e.w);
    ema_w16[i] = o;
  }
}

static int flat_grid4(long n4) {
  long want = (n4 + 255) / 256;
  const long cap = (long)sm_count() * 8;
  return (int)(want < cap ? (want < 1 ? 1 : want) : cap);
}

}  // namespace ub

using namespace ub;

extern "C" int ub_sumsq(const float* g, int64_t n, float* out, void* stream) {
  UB_REQUIRE(g && out && n > 0 && n % 4 == 0, "sumsq: n=%lld must be a positive multiple of 4", (long long)n);
  UB_LAUNCH(sumsq_kernel, flat_grid4(n / 4), 256, 0, (cudaStream_t)stream, (const float4*)g, n / 4, out);
  return check_launch("sumsq_kernel");
}

extern "C" int ub_adamw(float* p, const float* g, float* m, float* v, void* w_bf16, int64_t n, int64_t n_decay, float lr,
                        float wd, float beta1, float beta2, float eps, int step, float grad_scale, void* stream) {
  UB_REQUIRE(p && g && m && v, "adamw: null pointer");
  UB_REQUIRE(n > 0 && n % 4 == 0 && n_decay % 4 == 0 && n_decay >= 0 && n_decay <= n,
             "adamw: n=%lld and n_decay=%lld must be multiples of 4", (long long)n, (long long)n_decay);
  UB_REQUIRE(step >= 1, "adamw: step must be >= 1");
  const float bc1 = 1.0f - powf(beta1, (float)step);
  const float bc2 = 1.0f - powf(beta2, (float)step);
  UB_LAUNCH(adamw_kernel, flat_grid4(n / 4), 256, 0, (cudaStream_t)stream, (float4*)p, (const float4*)g, (float4*)m, (float4*)v,
                                                                   (uint2*)w_bf16, n / 4, n_decay / 4, lr, wd, beta1, beta2, eps,
                                                                   bc1, sqrtf(bc2), grad_scale);
  return check_launch("adamw_kernel");
}

extern "C" int ub_adamw_dev(float* p, const float* g, float* m, float* v, void* w_bf16, int64_t n, int64_t n_decay,
                            const float* hyper, float* gnorm_sq, void* stream) {
  UB_REQUIRE(p && g && m && v && hyper, "adamw_dev: null pointer");
  UB_REQUIRE(n > 0 && n % 4 == 0 && n_decay % 4 == 0 && n_decay >= 0 && n_decay <= n,
             "adamw_dev: n=%lld and n_decay=%lld must be multiples of 4", (long long)n, (long long)n_decay);
  UB_LAUNCH(adamw_dev_kernel, flat_grid4(n / 4), 256, 0, (cudaStream_t)stream, (float4*)p, (const float4*)g, (float4*)m, (float4*)v,
                                                                       (uint2*)w_bf16, n / 4, n_decay / 4, hyper, gnorm_sq);
  return check_launch("adamw_dev_kernel");
}

extern "C" int ub_adamw_seg(float* p, const float* g, float* m, float* v, void* w_bf16, int64_t n, const int32_t* seg_end4, int n_seg,
                            const float* hyper, float* gnorm_sq, void* stream) {
  UB_REQUIRE(p && g && m && v && hyper && seg_end4, "adamw_seg: null pointer");
  UB_REQUIRE(n > 0 && n % 4 == 0, "adamw_seg: n=%lld must be a positive multiple of 4", (long long)n);
  UB_REQUIRE(n_seg >= 1 && n_seg <= kMaxSeg, "adamw_seg: %d parameter groups (1..%d supported)", n_seg, kMaxSeg);
  UB_LAUNCH(adamw_seg_kernel, flat_grid4(n / 4), 256, 0, (cudaStream_t)stream, (float4*)p, (const float4*)g, (float4*)m, (float4*)v,
            (uint2*)w_bf16, n / 4, (const int*)seg_end4, n_seg, hyper, gnorm_sq);
  return check_launch("adamw_seg_kernel");
}

extern "C" int ub_sumsq_seg(const float* g, int64_t n, const int32_t* seg_end4, int n_seg, const float* hyper, float* out, void* stream) {
  UB_REQUIRE(g && out && hyper && seg_end4 && n > 0 && n % 4 == 0, "sumsq_seg: bad arguments");
  UB_REQUIRE(n_seg >= 1 && n_seg <= kMaxSeg, "sumsq_seg: %d parameter groups (1..%d supported)", n_seg, kMaxSeg);
  UB_LAUNCH(sumsq_seg_kernel, flat_grid4(n / 4), 256, 0, (cudaStream_t)stream, (const float4*)g, n / 4, (const int*)seg_end4, n_seg, hyper, out);
  return check_launch("sumsq_seg_kernel");
}

extern "C" int ub_cast_bf16(const float* x, void* out, int64_t n, void* stream) {
  UB_REQUIRE(x && out && n > 0 && n % 4 == 0, "cast_bf16: n=%lld must be a positive multiple of 4", (long long)n);
  UB_LAUNCH(cast_bf16_kernel, flat_grid4(n / 4), 256, 0, (cudaStream_t)stream, (const float4*)x, (uint2*)out, n / 4);
  return check_launch("cast_bf16_kernel");
}

extern "C" int ub_ema_update(float* ema, void* ema_w16, const float* p, int64_t n, float decay, float one_minus_decay, void* stream) {
  UB_REQUIRE(ema && ema_w16 && p, "ema_update: null pointer");
  UB_REQUIRE(n > 0 && n % 4 == 0, "ema_update: n=%lld must be a positive multiple of 4", (long long)n);
  UB_LAUNCH(ema_update_kernel, flat_grid4(n / 4), 256, 0, (cudaStream_t)stream, (float4*)ema, (uint2*)ema_w16, (const float4*)p, n / 4,
            decay, one_minus_decay);
  return check_launch("ema_update_kernel");
}
