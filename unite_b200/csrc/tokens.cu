// Token-level data movement and the mask sampler (HBM / latency bound).
//
//   ub_patchify      fp32 clip -> bf16 im2col rows (the A operand of the stride==kernel Conv3d as a GEMM)
//                    clip.py:123-128,146 (teacher conv1), modeling_finetune.py:165-174 (student PatchEmbed.proj)
//   ub_patchify_mix  the same rows of the batch-mode mixup / cutmix of the clip (stage-2 mixup_fn), x left untouched
//   ub_patchify_u8 / ub_patchify_mix_u8   the same two from decoded uint8 frames, normalised on the way
//   ub_mask_select   attention-guided visible-token selection, bit-exact
//                    run_stage1.py:379-387 (multinomial == top-N_vis of attn/q, q ~ Exp(1) supplied by the caller)
//                    utils.py:89-120 get_greedy_masks (k committee members take ranks i, i+k, ...; q == NULL)
//   ub_gather_rows   out[i,:] = in[idx[i],:]  — replaces the boolean-mask gathers `x[~mask]`
//                    (modeling_adaptation.py:153,319; run_stage1.py:393) without their nonzero() host syncs
//   ub_colsum_bf16   bias gradients: out[n] += sum_m dY[m,n]
#include "common.cuh"
#include "../../include/unite_b200.h"

namespace ub {

// ------------------------------------------------------------------------------------------------
// patchify: x fp32 [B,3,T,H,W] -> out bf16 [B*(T/tub)*(H/p)*(W/p), 3*tub*p*p], p == 16
// token order (t,h,w); feature order (c,kt,kh,kw) == flattened Conv3d weight [D,3,tub,16,16].
// One thread moves one (token, c, kt, kh) run of 16 contiguous pixels: 64 B read, 32 B written; consecutive
// threads take consecutive runs of the same token so the bf16 writes of a warp are one contiguous 1 KB span.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) patchify_kernel(const float* __restrict__ x, bf16* __restrict__ out, int B, int T,
                                                       int H, int W, int tub, long total_runs) {
  const int gh = H / 16, gw = W / 16, Tp = T / tub;
  const int runs_per_tok = 3 * tub * 16;
  for (long id = (long)blockIdx.x * blockDim.x + threadIdx.x; id < total_runs; id += (long)gridDim.x * blockDim.x) {
    const int run = (int)(id % runs_per_tok);
    const long tok = id / runs_per_tok;
    const int kh = run % 16, kt = (run / 16) % tub, c = run / (16 * tub);
    const int pw = (int)(tok % gw), ph = (int)((tok / gw) % gh), tp = (int)((tok / ((long)gw * gh)) % Tp);
    const int b = (int)(tok / ((long)gw * gh * Tp));
    const float* src = x + ((((long)b * 3 + c) * T + (tp * tub + kt)) * H + (ph * 16 + kh)) * W + pw * 16;
    const float4 f0 = *reinterpret_cast<const float4*>(src), f1 = *reinterpret_cast<const float4*>(src + 4),
                 f2 = *reinterpret_cast<const float4*>(src + 8), f3 = *reinterpret_cast<const float4*>(src + 12);
    uint4 o0, o1;
    o0.x = pack_bf16x2(f0.x, f0.y); o0.y = pack_bf16x2(f0.z, f0.w); o0.z = pack_bf16x2(f1.x, f1.y); o0.w = pack_bf16x2(f1.z, f1.w);
    o1.x = pack_bf16x2(f2.x, f2.y); o1.y = pack_bf16x2(f2.z, f2.w); o1.z = pack_bf16x2(f3.x, f3.y); o1.w = pack_bf16x2(f3.z, f3.w);
    bf16* dst = out + tok * (long)(runs_per_tok * 16) + run * 16;
    stg_v4(dst, o0);
    stg_v4(dst + 8, o1);
  }
}

// ------------------------------------------------------------------------------------------------
// patchify_mix: ub_patchify of the clip mixed as timm's batch-mode Mixup._mix_batch mixes it (run_stage2.py's mixup_fn,
// engine_for_finetuning.py:86-87), in one pass that never writes x — so a graph replayed over a resident input buffer mixes the
// clip afresh on every replay instead of mixing its own output again.
//   mix (device fp32) = {apply, lam, 1 - lam, use_cutmix, t0, t1, h0, h1, w0, w1}
//   apply == 0: copy.  cutmix: inside the half-open box [t0,t1) x [h0,h1) x [w0,w1) of the (T, H, W) axes, clip b takes clip
//   B-1-b's value.  mixup: lam * x_b + (1 - lam) * x_{B-1-b} with each product and the sum rounded on their own (no FMA) — what
//   x.mul_(lam).add_(x.flip(0).mul_(1 - lam)) computes in fp32, so the rows are bit-identical to patchify(torch-mixed clip).
// One thread moves the same (token, c, kt, kh) run of clips b and B-1-b (b < B/2, B even): every input byte is read once.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) patchify_mix_kernel(const float* __restrict__ x, bf16* __restrict__ out,
                                                           const float* __restrict__ mix, int B, int T, int H, int W, int tub,
                                                           long total_runs) {
  const bool apply = mix[0] != 0.f, cut = mix[3] != 0.f;
  const float lam = mix[1], lam1 = mix[2];
  const int t0 = (int)mix[4], t1 = (int)mix[5], h0 = (int)mix[6], h1 = (int)mix[7], w0 = (int)mix[8], w1 = (int)mix[9];
  const int gh = H / 16, gw = W / 16, Tp = T / tub;
  const int runs_per_tok = 3 * tub * 16;
  const long toks_per_clip = (long)Tp * gh * gw;
  const long clip_elems = 3L * T * H * W;
  for (long id = (long)blockIdx.x * blockDim.x + threadIdx.x; id < total_runs; id += (long)gridDim.x * blockDim.x) {
    const int run = (int)(id % runs_per_tok);
    const long tok = id / runs_per_tok;                       // token of the first half of the batch
    const int kh = run % 16, kt = (run / 16) % tub, c = run / (16 * tub);
    const int pw = (int)(tok % gw), ph = (int)((tok / gw) % gh), tp = (int)((tok / ((long)gw * gh)) % Tp);
    const int b = (int)(tok / toks_per_clip);
    const int t = tp * tub + kt, h = ph * 16 + kh;
    const long mirror = (long)(B - 1 - 2 * b);                // clip B-1-b is `mirror` clips further on
    const float* sa = x + ((((long)b * 3 + c) * T + t) * H + h) * W + pw * 16;
    const float* sb = sa + mirror * clip_elems;
    float a[16], m[16];
#pragma unroll
    for (int i = 0; i < 16; i += 4) {
      *reinterpret_cast<float4*>(&a[i]) = *reinterpret_cast<const float4*>(sa + i);
      *reinterpret_cast<float4*>(&m[i]) = *reinterpret_cast<const float4*>(sb + i);
    }
    if (apply) {
      if (cut) {
        if (t >= t0 && t < t1 && h >= h0 && h < h1) {
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const int w = pw * 16 + i;
            if (w >= w0 && w < w1) { const float s = a[i]; a[i] = m[i]; m[i] = s; }
          }
        }
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float va = a[i], vm = m[i];
          a[i] = __fadd_rn(__fmul_rn(va, lam), __fmul_rn(vm, lam1));
          m[i] = __fadd_rn(__fmul_rn(vm, lam), __fmul_rn(va, lam1));
        }
      }
    }
    uint4 o[4];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      o[i].x = pack_bf16x2(a[8 * i], a[8 * i + 1]); o[i].y = pack_bf16x2(a[8 * i + 2], a[8 * i + 3]);
      o[i].z = pack_bf16x2(a[8 * i + 4], a[8 * i + 5]); o[i].w = pack_bf16x2(a[8 * i + 6], a[8 * i + 7]);
      o[2 + i].x = pack_bf16x2(m[8 * i], m[8 * i + 1]); o[2 + i].y = pack_bf16x2(m[8 * i + 2], m[8 * i + 3]);
      o[2 + i].z = pack_bf16x2(m[8 * i + 4], m[8 * i + 5]); o[2 + i].w = pack_bf16x2(m[8 * i + 6], m[8 * i + 7]);
    }
    bf16* da = out + tok * (long)(runs_per_tok * 16) + run * 16;
    bf16* db = da + mirror * toks_per_clip * (long)(runs_per_tok * 16);
    stg_v4(da, o[0]);
    stg_v4(da + 8, o[1]);
    stg_v4(db, o[2]);
    stg_v4(db + 8, o[3]);
  }
}

// ------------------------------------------------------------------------------------------------
// patchify_u8: decoded frames uint8 [B,T,H,W,3] (decord / NVDEC layout) -> ImageNet-normalised bf16 im2col rows, i.e.
// ToTensor + tensor_normalize (kinetics_sparse.py:236-243, :434-451) + the THWC->CTHW permute + patchify in one pass:
//   v = (u / 255 - mean[c]) / std[c]   in fp32 with IEEE divides (bit-identical to the torch CPU pipeline), then bf16.
// One thread = one (token, kt, kh) run of 16 pixels: 48 contiguous bytes in, three 32-byte runs out (one per channel).
// The step then needs 38.5 MB of H2D per 32-clip batch instead of the 154 MB fp32 clip.
// ------------------------------------------------------------------------------------------------
// One run of the THWC frames: clip b, frame t, pixel row h, the 16 pixels from column w, of token `tok` at (kt, kh).
struct U8Run {
  long tok;
  int b, t, h, w, kt, kh;
};

UB_DEVINL U8Run u8_run(long id, int T, int H, int W, int tub) {
  const int gh = H / 16, gw = W / 16, Tp = T / tub;
  const int runs_per_tok = tub * 16;          // (kt, kh)
  U8Run r;
  const int run = (int)(id % runs_per_tok);
  r.tok = id / runs_per_tok;
  r.kh = run % 16;
  r.kt = run / 16;
  const int pw = (int)(r.tok % gw), ph = (int)((r.tok / gw) % gh), tp = (int)((r.tok / ((long)gw * gh)) % Tp);
  r.b = (int)(r.tok / ((long)gw * gh * Tp));
  r.t = tp * tub + r.kt;
  r.h = ph * 16 + r.kh;
  r.w = pw * 16;
  return r;
}

// byte offset of the run's first pixel in x, and element offset of its channel-0 segment in the im2col rows
UB_DEVINL long u8_src(const U8Run& r, int T, int H, int W) { return ((((long)r.b * T + r.t) * H + r.h) * W + r.w) * 3; }
UB_DEVINL long u8_dst(const U8Run& r, int tub) { return r.tok * (long)(3 * tub * 256) + r.kt * 256 + r.kh * 16; }

// the run's 48 bytes (16 pixels x RGB), one 16-byte load per third
UB_DEVINL void u8_load(const uint8_t* src, uint32_t* w) {
  *reinterpret_cast<uint4*>(&w[0]) = ldg_nc_v4(src);
  *reinterpret_cast<uint4*>(&w[4]) = ldg_nc_v4(src + 16);
  *reinterpret_cast<uint4*>(&w[8]) = ldg_nc_v4(src + 32);
}

// ToTensor + tensor_normalize of one byte: (u / 255 - mean) / std, each step an IEEE-rounded fp32 operation
UB_DEVINL float u8_norm(uint8_t u, float mean, float sd) { return __fdiv_rn(__fsub_rn(__fdiv_rn((float)u, 255.0f), mean), sd); }

__global__ void __launch_bounds__(256) patchify_u8_kernel(const uint8_t* __restrict__ x, bf16* __restrict__ out, float m0, float m1,
                                                          float m2, float s0, float s1, float s2, int B, int T, int H, int W, int tub,
                                                          long total_runs) {
  const float mean[3] = {m0, m1, m2}, sd[3] = {s0, s1, s2};
  for (long id = (long)blockIdx.x * blockDim.x + threadIdx.x; id < total_runs; id += (long)gridDim.x * blockDim.x) {
    const U8Run r = u8_run(id, T, H, W, tub);
    uint32_t w[12];
    u8_load(x + u8_src(r, T, H, W), w);
    const uint8_t* by = reinterpret_cast<const uint8_t*>(w);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      uint32_t o[8];
#pragma unroll
      for (int i = 0; i < 8; ++i)
        o[i] = pack_bf16x2(u8_norm(by[(2 * i) * 3 + c], mean[c], sd[c]), u8_norm(by[(2 * i + 1) * 3 + c], mean[c], sd[c]));
      bf16* dst = out + u8_dst(r, tub) + (long)c * (tub * 256);
      stg_v4(dst, make_uint4(o[0], o[1], o[2], o[3]));
      stg_v4(dst + 8, make_uint4(o[4], o[5], o[6], o[7]));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// patchify_mix_u8: ub_patchify_mix of the frames ub_patchify_u8 normalises — every byte normalised as there, then mixed as there
// (mixup and cutmix act on normalised values, as the reference's mixup_fn runs after its loader's tensor_normalize).
// One thread takes the same (token, kt, kh) run of clips b and B-1-b (b < B/2): 2 x 48 bytes in, 6 x 32 bytes out.
// A byte has 256 values per channel: each CTA normalises them once into a shared table (u8_norm, so every entry is bit-identical
// to ub_patchify_u8's value) and looks the pixels up, instead of two IEEE divides per pixel.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) patchify_mix_u8_kernel(const uint8_t* __restrict__ x, bf16* __restrict__ out,
                                                              const float* __restrict__ mix, float m0, float m1, float m2, float s0,
                                                              float s1, float s2, int B, int T, int H, int W, int tub, long total_runs) {
  __shared__ float lut[3][256];
  for (int i = threadIdx.x; i < 3 * 256; i += blockDim.x) {
    const int c = i / 256;
    lut[c][i % 256] = u8_norm((uint8_t)(i % 256), c == 0 ? m0 : (c == 1 ? m1 : m2), c == 0 ? s0 : (c == 1 ? s1 : s2));
  }
  __syncthreads();
  const bool apply = mix[0] != 0.f, cut = mix[3] != 0.f;
  const float lam = mix[1], lam1 = mix[2];
  const int t0 = (int)mix[4], t1 = (int)mix[5], h0 = (int)mix[6], h1 = (int)mix[7], w0 = (int)mix[8], w1 = (int)mix[9];
  const long clip_bytes = 3L * T * H * W;
  const long clip_rows = (long)(T / tub) * (H / 16) * (W / 16) * (3 * tub * 256);
  for (long id = (long)blockIdx.x * blockDim.x + threadIdx.x; id < total_runs; id += (long)gridDim.x * blockDim.x) {
    const U8Run r = u8_run(id, T, H, W, tub);                 // a run of the first half of the batch
    const long mirror = (long)(B - 1 - 2 * r.b);              // clip B-1-b is `mirror` clips further on
    const uint8_t* sa = x + u8_src(r, T, H, W);
    uint32_t wa[12], wm[12];
    u8_load(sa, wa);
    u8_load(sa + mirror * clip_bytes, wm);
    const uint8_t* ba = reinterpret_cast<const uint8_t*>(wa);
    const uint8_t* bm = reinterpret_cast<const uint8_t*>(wm);
    const bool in_box = apply && cut && r.t >= t0 && r.t < t1 && r.h >= h0 && r.h < h1;
    bf16* da = out + u8_dst(r, tub);
    bf16* db = da + mirror * clip_rows;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float a[16], m[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        a[i] = lut[c][ba[i * 3 + c]];
        m[i] = lut[c][bm[i * 3 + c]];
      }
      if (in_box) {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int w = r.w + i;
          if (w >= w0 && w < w1) { const float s = a[i]; a[i] = m[i]; m[i] = s; }
        }
      } else if (apply && !cut) {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float va = a[i], vm = m[i];
          a[i] = __fadd_rn(__fmul_rn(va, lam), __fmul_rn(vm, lam1));
          m[i] = __fadd_rn(__fmul_rn(vm, lam), __fmul_rn(va, lam1));
        }
      }
      uint32_t oa[8], om[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        oa[i] = pack_bf16x2(a[2 * i], a[2 * i + 1]);
        om[i] = pack_bf16x2(m[2 * i], m[2 * i + 1]);
      }
      const long co = (long)c * (tub * 256);
      stg_v4(da + co, make_uint4(oa[0], oa[1], oa[2], oa[3]));
      stg_v4(da + co + 8, make_uint4(oa[4], oa[5], oa[6], oa[7]));
      stg_v4(db + co, make_uint4(om[0], om[1], om[2], om[3]));
      stg_v4(db + co + 8, make_uint4(om[4], om[5], om[6], om[7]));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// resize_patchify: fp32 clip [B,3,T,H,W] or uint8 frames [B,T,H,W,3] -> (bicubic resize to R x R) -> bf16 im2col rows
// [B*(T/tub)*(R/p)^2, ld] for any even patch size p; feature order (c,kt,kh,kw) as ub_patchify, columns [3*tub*p*p, ld) zero.
// The resize is torch.nn.functional.interpolate(mode="bicubic", align_corners=False, antialias=False) per (c, t) plane:
//   src = scale * (dst + 0.5) - 0.5, scale = in / out;  i0 = min(floor(src), in - 1), f = clamp(src - i0, 0, 1);
//   taps i0-1 .. i0+2 clamped to the border, cubic-convolution weights with A = -0.75 computed in fp32;
//   out = sum_j wy_j * (sum_i wx_i * x[y_j, x_i]), summed in that order (ATen's separable upsample kernel).
// uint8 input is normalised first (same IEEE divides as patchify_u8), as the reference's loader normalises and its engine
// then resizes.  One CTA = one (clip, output frame, kt, patch row): the source rows that band of p output rows reads are
// staged [3][rows][W] fp32 in shared memory (each source pixel leaves HBM once, up to the 3-4 rows two bands share), then
// consecutive threads write consecutive bf16 pairs of one token's row.
// ------------------------------------------------------------------------------------------------
UB_DEVINL float cubic_near(float x, float A) { return ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f; }          // |x| <= 1
UB_DEVINL float cubic_far(float x, float A) { return ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A; }     // 1 < |x| < 2

// source tap indices (clamped to [0, n)) and weights of output coordinate `dst`
UB_DEVINL void bicubic_taps(int dst, float scale, int n, int* idx, float* w) {
  const float src = __fsub_rn(__fmul_rn(scale, __fadd_rn((float)dst, 0.5f)), 0.5f);
  const int i0 = min((int)floorf(src), n - 1);
  const float f = fminf(fmaxf(src - (float)i0, 0.f), 1.f);
  const float A = -0.75f;
  w[0] = cubic_far(f + 1.f, A);
  w[1] = cubic_near(f, A);
  w[2] = cubic_near(1.f - f, A);
  w[3] = cubic_far((1.f - f) + 1.f, A);
#pragma unroll
  for (int j = 0; j < 4; ++j) idx[j] = min(max(i0 - 1 + j, 0), n - 1);
}

template <bool U8>
__global__ void __launch_bounds__(256) resize_patchify_kernel(const void* __restrict__ xin, bf16* __restrict__ out, long ld, float m0,
                                                              float m1, float m2, float s0, float s1, float s2, int T, int H, int W,
                                                              int R, int p, int tub, int rows_max, float sy, float sx, int identity) {
  extern __shared__ float rp_smem[];
  const int gr = R / p, Tp = T / tub;
  int blk = blockIdx.x;
  const int ph = blk % gr; blk /= gr;
  const int kt = blk % tub; blk /= tub;
  const int tp = blk % Tp;
  const int b = blk / Tp;
  const int t = tp * tub + kt;
  float* pix = rp_smem;                                      // [3][rows_max][W]
  float* wx = pix + 3 * rows_max * W;                        // [R][4]
  int* ix = reinterpret_cast<int*>(wx + 4 * R);              // [R][4]
  float* wy = reinterpret_cast<float*>(ix + 4 * R);          // [p][4]
  int* iy = reinterpret_cast<int*>(wy + 4 * p);              // [p][4], relative to y_lo
  const int oy0 = ph * p;
  int y_lo = oy0, nrows = p;
  if (!identity) {
    int i[4];
    float w[4];
    bicubic_taps(oy0, sy, H, i, w);
    y_lo = i[0];
    bicubic_taps(oy0 + p - 1, sy, H, i, w);
    nrows = i[3] - y_lo + 1;
    for (int o = threadIdx.x; o < R + p; o += blockDim.x) {
      if (o < R) {
        bicubic_taps(o, sx, W, ix + 4 * o, wx + 4 * o);
      } else {
        const int r = o - R;
        bicubic_taps(oy0 + r, sy, H, iy + 4 * r, wy + 4 * r);
#pragma unroll
        for (int j = 0; j < 4; ++j) iy[4 * r + j] -= y_lo;
      }
    }
  }
  // ---- stage the band's source rows ----
  const long plane = (long)H * W;
  if constexpr (U8) {
    const uint8_t* src = static_cast<const uint8_t*>(xin) + (((long)b * T + t) * H + y_lo) * (long)W * 3;
    const int n = nrows * W * 3;
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
      const int c = e % 3, px = e / 3;
      const float mean = c == 0 ? m0 : (c == 1 ? m1 : m2), sd = c == 0 ? s0 : (c == 1 ? s1 : s2);
      const float v = __fdiv_rn(__fsub_rn(__fdiv_rn((float)src[e], 255.0f), mean), sd);
      pix[(c * rows_max + px / W) * W + px % W] = v;
    }
  } else {
    const float* x = static_cast<const float*>(xin);
    const int n = nrows * W;
    for (int c = 0; c < 3; ++c) {
      const float* src = x + (((long)b * 3 + c) * T + t) * plane + (long)y_lo * W;
      float* dst = pix + c * rows_max * W;
      if ((W & 3) == 0) {
        for (int e = threadIdx.x; e < n / 4; e += blockDim.x)
          reinterpret_cast<float4*>(dst)[e] = __ldg(reinterpret_cast<const float4*>(src) + e);
      } else {
        for (int e = threadIdx.x; e < n; e += blockDim.x) dst[e] = __ldg(src + e);
      }
    }
  }
  __syncthreads();
  // ---- resample + write: item = (pw, c, kh, kw pair), kw pair fastest ----
  const int hp = p / 2, pp = p * p, feat = 3 * tub * pp;
  const long tok0 = (((long)b * Tp + tp) * gr + ph) * gr;
  const int n_items = gr * 3 * p * hp;
  for (int e = threadIdx.x; e < n_items; e += blockDim.x) {
    const int kwp = e % hp;
    int r = e / hp;
    const int kh = r % p; r /= p;
    const int c = r % 3;
    const int pw = r / 3;
    const int ox = pw * p + 2 * kwp;
    const float* pc = pix + c * rows_max * W;
    float v[2];
    if (identity) {
      v[0] = pc[kh * W + ox];
      v[1] = pc[kh * W + ox + 1];
    } else {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int* xi = ix + 4 * (ox + h);
        const float* xw = wx + 4 * (ox + h);
        float acc = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float* row = pc + iy[4 * kh + j] * W;
          float s = row[xi[0]] * xw[0];
          s += row[xi[1]] * xw[1];
          s += row[xi[2]] * xw[2];
          s += row[xi[3]] * xw[3];
          acc = j == 0 ? s * wy[4 * kh] : acc + s * wy[4 * kh + j];
        }
        v[h] = acc;
      }
    }
    bf16* dst = out + (tok0 + pw) * ld + c * (tub * pp) + kt * pp + kh * p + 2 * kwp;
    *reinterpret_cast<uint32_t*>(dst) = pack_bf16x2(v[0], v[1]);
  }
  // ---- zero the row padding of this band's tokens (once per token: the kt == 0 CTA) ----
  if (kt == 0 && ld > feat) {
    const int hpad = (int)(ld - feat) / 2;
    for (int e = threadIdx.x; e < gr * hpad; e += blockDim.x)
      *reinterpret_cast<uint32_t*>(out + (tok0 + e / hpad) * ld + feat + 2 * (e % hpad)) = 0u;
  }
}

// ------------------------------------------------------------------------------------------------
// mask selection.  One warp per frame (row of attn): score = attn / q (IEEE fp32 divide, same as torch),
// rank_i = #{j : s_j > s_i or (s_j == s_i and j < i)};  member = rank % k, visible for that member iff rank / k < n_vis.
// Outputs (all per member m):
//   mask     uint8 [k, frames*P]        1 = masked (viewed as bool [k, B, T*P])
//   vis_idx  int32 [k, B, T*n_vis]      ascending token index inside the clip (t*P + p)
//   tea_rows int32 [k, B, T*n_vis]      row of that token in the teacher stream: (b*T + t)*(P+1) + 1 + p   (optional)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) mask_select_kernel(const float* __restrict__ attn, const float* __restrict__ q,
                                                          uint8_t* __restrict__ mask, int* __restrict__ vis_idx,
                                                          int* __restrict__ tea_rows, int frames, int P, int T, int k,
                                                          int n_vis) {
  extern __shared__ float s_scores[];  // [warps][P] scores, then ranks as int
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int f = blockIdx.x * (blockDim.x >> 5) + warp;
  if (f >= frames) return;
  float* sc = s_scores + warp * 2 * P;
  int* rk = reinterpret_cast<int*>(sc + P);
  for (int i = lane; i < P; i += 32) {
    const float a = attn[(long)f * P + i];
    sc[i] = q ? a / q[(long)f * P + i] : a;
  }
  __syncwarp();
  for (int i = lane; i < P; i += 32) {
    const float si = sc[i];
    int r = 0;
    for (int j = 0; j < P; ++j) {
      const float sj = sc[j];
      r += (sj > si) || (sj == si && j < i);
    }
    rk[i] = r;
  }
  __syncwarp();
  const int b = f / T, t = f % T;
  const long total = (long)frames * P;
  for (int m = 0; m < k; ++m) {
    int count = 0;
    for (int i0 = 0; i0 < P; i0 += 32) {
      const int i = i0 + lane;
      bool vis = false;
      if (i < P) {
        const int r = rk[i];
        vis = (r % k == m) && (r / k < n_vis);
        mask[(long)m * total + (long)f * P + i] = vis ? 0 : 1;
      }
      const unsigned bal = __ballot_sync(0xffffffffu, vis);
      if (vis) {
        const int slot = count + __popc(bal & ((1u << lane) - 1u));
        const long o = ((long)m * (frames / T) + b) * ((long)T * n_vis) + (long)t * n_vis + slot;
        vis_idx[o] = t * P + i;
        if (tea_rows) tea_rows[o] = (b * T + t) * (P + 1) + 1 + i;
      }
      count += __popc(bal);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// gather rows: out[i, :] = in[(base(i) +) idx[i], :], rows of `row_bytes` (multiple of 16) bytes
//   rows_per_group > 0: idx is relative to a group base:  src = (i / rows_per_group) * group_stride + idx[i]
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gather_rows_kernel(const uint4* __restrict__ in, const int* __restrict__ idx,
                                                          uint4* __restrict__ out, long n_rows, int chunks_per_row,
                                                          int rows_per_group, long group_stride) {
  const long total = n_rows * chunks_per_row;
  for (long id = (long)blockIdx.x * blockDim.x + threadIdx.x; id < total; id += (long)gridDim.x * blockDim.x) {
    const long r = id / chunks_per_row;
    const int c = (int)(id % chunks_per_row);
    long src = idx[r];
    if (rows_per_group > 0) src += (r / rows_per_group) * group_stride;
    out[id] = in[src * chunks_per_row + c];
  }
}

// ------------------------------------------------------------------------------------------------
// column sums of a bf16 matrix (bias gradients), accumulated into fp32 with red.add.
// CTA = 256 threads = 8 row-groups x 32 lanes; a lane owns 8 columns (one 16-byte load per row), the CTA covers
// 256 columns x ROWS_PER_CTA rows with 4 independent loads in flight per thread, then reduces the 8 row-groups
// through smem and issues one red.add per column.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) colsum_bf16_kernel(const bf16* __restrict__ x, int64_t ld, float* __restrict__ out,
                                                          int M, int N, int CS_ROWS, int skip_lo, int skip_hi) {
  __shared__ float s_part[8][256];
  const int lane = threadIdx.x & 31, rg = threadIdx.x >> 5;
  const int col = blockIdx.x * 256 + lane * 8;
  const int r0 = blockIdx.y * CS_ROWS;
  const int r1 = min(M, r0 + CS_ROWS);
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  if (col < N) {
    for (int r = r0 + rg; r < r1; r += 32) {
      uint4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        v[u] = (r + u * 8 < r1) ? ldg_nc_v4(x + (int64_t)(r + u * 8) * ld + col) : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float2 f;
        f = unpack_bf16x2(v[u].x); acc[0] += f.x; acc[1] += f.y;
        f = unpack_bf16x2(v[u].y); acc[2] += f.x; acc[3] += f.y;
        f = unpack_bf16x2(v[u].z); acc[4] += f.x; acc[5] += f.y;
        f = unpack_bf16x2(v[u].w); acc[6] += f.x; acc[7] += f.y;
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) s_part[rg][lane * 8 + i] = acc[i];
  __syncthreads();
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c < N && !(c >= skip_lo && c < skip_hi)) {      // skipped columns (the structurally zero key bias) are left untouched
    float s = 0.f;
#pragma unroll
    for (int g = 0; g < 8; ++g) s += s_part[g][threadIdx.x];
    atomicAdd(out + c, s);
  }
}

// out_bf16 = bf16(x * row_scale[row / rows_per_scale])   (fp32 -> bf16 cast of the residual-stream gradient)
__global__ void __launch_bounds__(256) cast_scale_bf16_kernel(const float4* __restrict__ x, uint2* __restrict__ out,
                                                              const float* __restrict__ row_scale, int rows_per_scale,
                                                              long n4, int d4) {
  for (long id = (long)blockIdx.x * blockDim.x + threadIdx.x; id < n4; id += (long)gridDim.x * blockDim.x) {
    float4 v = x[id];
    if (row_scale) {
      const float s = __ldg(row_scale + (id / d4) / rows_per_scale);
      v.x *= s; v.y *= s; v.z *= s; v.w *= s;
    }
    uint2 o;
    o.x = pack_bf16x2(v.x, v.y);
    o.y = pack_bf16x2(v.z, v.w);
    out[id] = o;
  }
}

static int flat_grid(long n_items, int block) {
  long want = (n_items + block - 1) / block;
  const long cap = (long)sm_count() * 16;
  return (int)(want < cap ? (want < 1 ? 1 : want) : cap);
}

}  // namespace ub

using namespace ub;

extern "C" int ub_patchify(const float* x, void* out, int B, int T, int H, int W, int tubelet, void* stream) {
  UB_REQUIRE(x && out, "patchify: null pointer");
  UB_REQUIRE(B > 0 && T > 0 && tubelet > 0 && T % tubelet == 0, "patchify: bad temporal shape T=%d tubelet=%d", T, tubelet);
  UB_REQUIRE(H % 16 == 0 && W % 16 == 0 && H > 0 && W > 0, "patchify: H, W must be multiples of the 16-pixel patch (H=%d W=%d)", H, W);
  const long tokens = (long)B * (T / tubelet) * (H / 16) * (W / 16);
  const long runs = tokens * 3 * tubelet * 16;
  UB_LAUNCH(patchify_kernel, flat_grid(runs, 256), 256, 0, (cudaStream_t)stream, x, (bf16*)out, B, T, H, W, tubelet, runs);
  return check_launch("patchify_kernel");
}

extern "C" int ub_patchify_mix(const float* x, void* out, const float* mix, int B, int T, int H, int W, int tubelet, void* stream) {
  UB_REQUIRE(x && out && mix, "patchify_mix: null pointer");
  UB_REQUIRE(B > 0 && B % 2 == 0, "patchify_mix: the batch must be even to pair clip b with clip B-1-b (B=%d)", B);
  UB_REQUIRE(T > 0 && tubelet > 0 && T % tubelet == 0, "patchify_mix: bad temporal shape T=%d tubelet=%d", T, tubelet);
  UB_REQUIRE(H % 16 == 0 && W % 16 == 0 && H > 0 && W > 0, "patchify_mix: H, W must be multiples of the 16-pixel patch (H=%d W=%d)", H, W);
  const long runs = (long)(B / 2) * (T / tubelet) * (H / 16) * (W / 16) * 3 * tubelet * 16;
  UB_LAUNCH(patchify_mix_kernel, flat_grid(runs, 256), 256, 0, (cudaStream_t)stream, x, (bf16*)out, mix, B, T, H, W, tubelet, runs);
  return check_launch("patchify_mix_kernel");
}

extern "C" int ub_patchify_u8(const uint8_t* x, void* out, const float* mean3, const float* std3, int B, int T, int H, int W,
                              int tubelet, void* stream) {
  UB_REQUIRE(x && out && mean3 && std3, "patchify_u8: null pointer");
  UB_REQUIRE(B > 0 && T > 0 && tubelet > 0 && T % tubelet == 0 && H % 16 == 0 && W % 16 == 0, "patchify_u8: bad shape B=%d T=%d H=%d W=%d tub=%d", B,
             T, H, W, tubelet);
  UB_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0, "patchify_u8: input must be 16-byte aligned");
  UB_REQUIRE(std3[0] != 0.f && std3[1] != 0.f && std3[2] != 0.f, "patchify_u8: zero std");
  const long runs = (long)B * (T / tubelet) * (H / 16) * (W / 16) * tubelet * 16;
  UB_LAUNCH(patchify_u8_kernel, flat_grid(runs, 256), 256, 0, (cudaStream_t)stream, x, (bf16*)out, mean3[0], mean3[1], mean3[2], std3[0],
            std3[1], std3[2], B, T, H, W, tubelet, runs);
  return check_launch("patchify_u8_kernel");
}

extern "C" int ub_patchify_mix_u8(const uint8_t* x, void* out, const float* mix, const float* mean3, const float* std3, int B, int T, int H,
                                  int W, int tubelet, void* stream) {
  UB_REQUIRE(x && out && mix && mean3 && std3, "patchify_mix_u8: null pointer");
  UB_REQUIRE(B > 0 && B % 2 == 0, "patchify_mix_u8: the batch must be even to pair clip b with clip B-1-b (B=%d)", B);
  UB_REQUIRE(T > 0 && tubelet > 0 && T % tubelet == 0 && H > 0 && W > 0 && H % 16 == 0 && W % 16 == 0,
             "patchify_mix_u8: bad shape B=%d T=%d H=%d W=%d tub=%d", B, T, H, W, tubelet);
  UB_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0, "patchify_mix_u8: input must be 16-byte aligned");
  UB_REQUIRE(std3[0] != 0.f && std3[1] != 0.f && std3[2] != 0.f, "patchify_mix_u8: zero std");
  const long runs = (long)(B / 2) * (T / tubelet) * (H / 16) * (W / 16) * tubelet * 16;
  UB_LAUNCH(patchify_mix_u8_kernel, flat_grid(runs, 256), 256, 0, (cudaStream_t)stream, x, (bf16*)out, mix, mean3[0], mean3[1], mean3[2],
            std3[0], std3[1], std3[2], B, T, H, W, tubelet, runs);
  return check_launch("patchify_mix_u8_kernel");
}

extern "C" int ub_resize_patchify(const void* x, int x_is_u8, const float* mean3, const float* std3, void* out, int64_t ld_out, int B,
                                  int T, int H, int W, int R, int patch, int tubelet, void* stream) {
  UB_REQUIRE(x && out, "resize_patchify: null pointer");
  UB_REQUIRE(B > 0 && T > 0 && tubelet > 0 && T % tubelet == 0, "resize_patchify: bad temporal shape T=%d tubelet=%d", T, tubelet);
  UB_REQUIRE(patch >= 2 && patch <= 32 && patch % 2 == 0, "resize_patchify: patch size %d must be even (2..32)", patch);
  UB_REQUIRE(H > 0 && W > 0 && R > 0 && R % patch == 0, "resize_patchify: output resolution R=%d must be a multiple of the patch size %d",
             R, patch);
  const int feat = 3 * tubelet * patch * patch;
  UB_REQUIRE(ld_out >= feat && ld_out % 8 == 0, "resize_patchify: row pitch %lld must be >= %d and a multiple of 8", (long long)ld_out, feat);
  UB_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0,
             "resize_patchify: input and output must be 16-byte aligned");
  UB_REQUIRE(!x_is_u8 || (mean3 && std3 && std3[0] != 0.f && std3[1] != 0.f && std3[2] != 0.f), "resize_patchify: uint8 input needs mean / std");
  const int identity = (R == H && R == W) ? 1 : 0;
  const float sy = (float)H / (float)R, sx = (float)W / (float)R;           // ATen area_pixel_compute_scale (align_corners=False)
  int rows_max = identity ? patch : (int)ceilf((patch - 1) * sy) + 6;      // source rows one band of `patch` output rows reads
  if (rows_max > H) rows_max = H;
  const size_t smem = ((size_t)3 * rows_max * W + (identity ? 0 : (size_t)8 * (R + patch))) * sizeof(float);
  UB_REQUIRE(smem <= 220 * 1024, "resize_patchify: a band of %d source rows x W=%d does not fit in shared memory", rows_max, W);
  const long ctas = (long)B * (T / tubelet) * tubelet * (R / patch);
  UB_REQUIRE(ctas < (1L << 31), "resize_patchify: too many tokens");
  float m[3] = {0.f, 0.f, 0.f}, s[3] = {1.f, 1.f, 1.f};
  if (x_is_u8) {
    for (int i = 0; i < 3; ++i) { m[i] = mean3[i]; s[i] = std3[i]; }
  }
  auto kern = x_is_u8 ? resize_patchify_kernel<true> : resize_patchify_kernel<false>;
  static size_t smem_set[2] = {48 * 1024, 48 * 1024};
  if (smem > smem_set[x_is_u8 ? 1 : 0]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    UB_REQUIRE(e == cudaSuccess, "cudaFuncSetAttribute(resize_patchify smem=%zu): %s", smem, cudaGetErrorString(e));
    smem_set[x_is_u8 ? 1 : 0] = smem;
  }
  UB_LAUNCH(kern, (int)ctas, 256, smem, (cudaStream_t)stream, x, (bf16*)out, (long)ld_out, m[0], m[1], m[2], s[0], s[1], s[2], T, H, W, R,
            patch, tubelet, rows_max, sy, sx, identity);
  return check_launch("resize_patchify_kernel");
}

extern "C" int ub_mask_select(const float* attn, const float* q, uint8_t* mask, int* vis_idx, int* tea_rows, int frames,
                              int P, int T, int k, int n_vis, void* stream) {
  UB_REQUIRE(attn && mask && vis_idx, "mask_select: null pointer");
  UB_REQUIRE(frames > 0 && P > 0 && T > 0 && frames % T == 0, "mask_select: frames=%d must be a multiple of T=%d", frames, T);
  UB_REQUIRE(k >= 1 && n_vis >= 1 && (long)k * n_vis <= P, "mask_select: k=%d x n_vis=%d exceeds P=%d", k, n_vis, P);
  const int warps = 4;
  const size_t smem = (size_t)warps * 2 * P * sizeof(float);
  UB_REQUIRE(smem <= 48 * 1024, "mask_select: P=%d too large", P);
  UB_LAUNCH(mask_select_kernel, (frames + warps - 1) / warps, warps * 32, smem, (cudaStream_t)stream, attn, q, mask, vis_idx, tea_rows,
                                                                                               frames, P, T, k, n_vis);
  return check_launch("mask_select_kernel");
}

extern "C" int ub_gather_rows(const void* in, const int* idx, void* out, int64_t n_rows, int64_t row_bytes,
                              int rows_per_group, int64_t group_stride_rows, void* stream) {
  UB_REQUIRE(in && idx && out, "gather_rows: null pointer");
  UB_REQUIRE(n_rows > 0 && row_bytes > 0 && row_bytes % 16 == 0, "gather_rows: row_bytes=%lld must be a positive multiple of 16",
             (long long)row_bytes);
  const int cpr = (int)(row_bytes / 16);
  UB_LAUNCH(gather_rows_kernel, flat_grid(n_rows * cpr, 256), 256, 0, (cudaStream_t)stream, (const uint4*)in, idx, (uint4*)out, n_rows,
                                                                                    cpr, rows_per_group, group_stride_rows);
  return check_launch("gather_rows_kernel");
}

extern "C" int ub_colsum_bf16(const void* x, int64_t ld, float* out, int M, int N, int skip_lo, int skip_hi, void* stream) {
  UB_REQUIRE(x && out && M > 0 && N > 0 && N % 8 == 0 && ld % 8 == 0, "colsum_bf16: N and ld must be multiples of 8 (M=%d N=%d)", M, N);
  UB_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0, "colsum_bf16: x must be 16-byte aligned");
  // rows per CTA (multiple of 32): small enough that the grid keeps ~6 CTAs per SM in flight — this is a latency-bound pass
  // over a few tens of MB, so bytes in flight per SM matter more than the number of atomics at the end
  const int gx = (N + 255) / 256;
  const int want_y = (6 * sm_count() + gx - 1) / gx;
  int rows = ((M + want_y - 1) / want_y + 31) / 32 * 32;
  rows = rows < 32 ? 32 : (rows > 128 ? 128 : rows);
  dim3 grid(gx, (M + rows - 1) / rows);
  UB_LAUNCH(colsum_bf16_kernel, grid, 256, 0, (cudaStream_t)stream, (const bf16*)x, ld, out, M, N, rows, skip_lo, skip_hi);
  return check_launch("colsum_bf16_kernel");
}

extern "C" int ub_cast_scale_bf16(const float* x, void* out, const float* row_scale, int rows_per_scale, int64_t rows, int D,
                                  void* stream) {
  UB_REQUIRE(x && out && rows > 0 && D > 0 && D % 4 == 0, "cast_scale_bf16: bad arguments");
  UB_REQUIRE(row_scale == nullptr || rows_per_scale > 0, "cast_scale_bf16: rows_per_scale must be > 0");
  const long n4 = rows * (D / 4);
  UB_LAUNCH(cast_scale_bf16_kernel, flat_grid(n4, 256), 256, 0, (cudaStream_t)stream, (const float4*)x, (uint2*)out, row_scale,
                                                                              rows_per_scale, n4, D / 4);
  return check_launch("cast_scale_bf16_kernel");
}
