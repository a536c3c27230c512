// LayerNorm family (HBM-bound): one warp per row, the row lives in registers, 128-bit coalesced access.
//
// Replaces   student  nn.LayerNorm(eps=1e-6): modeling_finetune.py:143-150 (norm1/norm2), modeling_adaptation.py:168
//                     (shared encoder.norm on the K tapped layers) + :318-320 (gathered clip_pos_embed add),
//                     Linear_Decoder.norm + L2 normalise (modeling_adaptation.py:203-213), fc_norm (modeling_finetune.py:376)
//            teacher  fp32 LayerNorm subclass (clip.py:20-26): ln_pre with CLS/pos assembly (:150-152), ln_1/ln_2 (:55-64),
//                     ln_post on gathered visible tokens (:168)
// and the autograd backward of the student ones.  Statistics are always fp32; the residual stream is fp32;
// outputs that feed a GEMM are bf16.  D must be a multiple of 128 and <= 1024.
#include "common.cuh"
#include <cuda_fp16.h>
#include <cstdlib>
#include "../../include/unite_b200.h"

namespace ub {

constexpr int LN_MAXV = 8;  // float4 per lane -> D <= 1024

// One row distributed over a warp: lane holds float4 chunks i*32+lane, i < NV (NV = D/128 is a template
// parameter so the row occupies exactly NV*4 registers and every loop is fully unrolled without predicates).
template <int NV>
struct RowT {
  float4 v[NV];
};

template <int NV>
UB_DEVINL void row_load_f32(RowT<NV>& r, const float* p, int nv, int lane) {
#pragma unroll
  for (int i = 0; i < NV; ++i)
    if (i < nv) r.v[i] = *reinterpret_cast<const float4*>(p + (i * 32 + lane) * 4);
}
template <int NV>
UB_DEVINL void row_load_bf16(RowT<NV>& r, const bf16* p, int nv, int lane) {
#pragma unroll
  for (int i = 0; i < NV; ++i)
    if (i < nv) {
      const uint2 u = *reinterpret_cast<const uint2*>(p + (i * 32 + lane) * 4);
      const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y);
      r.v[i] = make_float4(a.x, a.y, b.x, b.y);
    }
}
template <int NV>
UB_DEVINL void row_store_f32(const RowT<NV>& r, float* p, int nv, int lane) {
#pragma unroll
  for (int i = 0; i < NV; ++i)
    if (i < nv) *reinterpret_cast<float4*>(p + (i * 32 + lane) * 4) = r.v[i];
}
template <int NV>
UB_DEVINL void row_store_bf16(const RowT<NV>& r, bf16* p, int nv, int lane) {
#pragma unroll
  for (int i = 0; i < NV; ++i)
    if (i < nv) {
      uint2 u;
      u.x = pack_bf16x2(r.v[i].x, r.v[i].y);
      u.y = pack_bf16x2(r.v[i].z, r.v[i].w);
      *reinterpret_cast<uint2*>(p + (i * 32 + lane) * 4) = u;
    }
}
// fp16 rows: the frozen teacher keeps its residual stream in fp16 (what the reference's autocast does, clip.py under
// torch.cuda.amp.autocast); statistics and arithmetic stay fp32
template <int NV>
UB_DEVINL void row_load_f16(RowT<NV>& r, const __half* p, int nv, int lane) {
#pragma unroll
  for (int i = 0; i < NV; ++i)
    if (i < nv) {
      const uint2 u = *reinterpret_cast<const uint2*>(p + (i * 32 + lane) * 4);
      const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
      r.v[i] = make_float4(a.x, a.y, b.x, b.y);
    }
}
template <int NV>
UB_DEVINL void row_store_f16(const RowT<NV>& r, __half* p, int nv, int lane) {
#pragma unroll
  for (int i = 0; i < NV; ++i)
    if (i < nv) {
      uint2 u;
      const __half2 a = __floats2half2_rn(r.v[i].x, r.v[i].y), b = __floats2half2_rn(r.v[i].z, r.v[i].w);
      u.x = *reinterpret_cast<const uint32_t*>(&a);
      u.y = *reinterpret_cast<const uint32_t*>(&b);
      *reinterpret_cast<uint2*>(p + (i * 32 + lane) * 4) = u;
    }
}
template <int NV>
UB_DEVINL float row_sum(const RowT<NV>& r, int nv) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i)
    if (i < nv) s += (r.v[i].x + r.v[i].y) + (r.v[i].z + r.v[i].w);
  return warp_sum(s);
}
template <int NV>
UB_DEVINL float row_dot(const RowT<NV>& a, const RowT<NV>& b, int nv) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i)
    if (i < nv) s += a.v[i].x * b.v[i].x + a.v[i].y * b.v[i].y + a.v[i].z * b.v[i].z + a.v[i].w * b.v[i].w;
  return warp_sum(s);
}
// two-pass mean / rstd (matches torch's fp32 layer_norm to round-off); leaves x centred: x <- x - mean
template <int NV>
UB_DEVINL float row_center_rstd(RowT<NV>& x, int nv, int D, float eps) {
  const float mean = row_sum(x, nv) / (float)D;
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i)
    if (i < nv) {
      x.v[i].x -= mean; x.v[i].y -= mean; x.v[i].z -= mean; x.v[i].w -= mean;
      s += x.v[i].x * x.v[i].x + x.v[i].y * x.v[i].y + x.v[i].z * x.v[i].z + x.v[i].w * x.v[i].w;
    }
  s = warp_sum(s);
  return rsqrtf(s / (float)D + eps);
}
#define UB_ROW_FOREACH(i, nv) _Pragma("unroll") for (int i = 0; i < NV; ++i) if (i < nv)

// ------------------------------------------------------------------------------------------------
// forward:  out[r] = LN(x[src(r)]) * gamma + beta  (+ post_add[post_idx[r]])
// ------------------------------------------------------------------------------------------------
struct LnFwdArgs {
  const void* x;          // fp32, or fp16 when x_f16
  const int* src_rows;    // optional gather of input rows
  const float* gamma;
  const float* beta;
  const float* post_add;  // optional fp32 table [*, D]
  const int* post_idx;    // row of post_add per output row
  void* out;
  int out_fp32;
  int rows, D;
  float eps;
  int x_f16;
};

template <int NV>
__global__ void __launch_bounds__(256) ln_fwd_kernel(const LnFwdArgs a) {
  const int lane = threadIdx.x & 31;
  constexpr int nv = NV;
  const int wpb = blockDim.x >> 5;
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < a.rows; row += gridDim.x * wpb) {
    const int64_t src = a.src_rows ? a.src_rows[row] : row;
    RowT<NV> x;
    if (a.x_f16) row_load_f16(x, reinterpret_cast<const __half*>(a.x) + src * a.D, nv, lane);
    else row_load_f32(x, reinterpret_cast<const float*>(a.x) + src * a.D, nv, lane);
    const float rstd = row_center_rstd(x, nv, a.D, a.eps);
    UB_ROW_FOREACH(i, nv) {   // gamma / beta come from L1 every row: keeps the kernel at ~40 registers -> full occupancy
      float4 g, b;
      asm volatile("ld.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(g.x), "=f"(g.y), "=f"(g.z), "=f"(g.w) : "l"(a.gamma + (i * 32 + lane) * 4));
      asm volatile("ld.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "l"(a.beta + (i * 32 + lane) * 4));
      x.v[i].x = x.v[i].x * rstd * g.x + b.x;
      x.v[i].y = x.v[i].y * rstd * g.y + b.y;
      x.v[i].z = x.v[i].z * rstd * g.z + b.z;
      x.v[i].w = x.v[i].w * rstd * g.w + b.w;
    }
    if (a.post_add) {
      RowT<NV> pa;
      row_load_f32(pa, a.post_add + (int64_t)a.post_idx[row] * a.D, nv, lane);
      UB_ROW_FOREACH(i, nv) {
        x.v[i].x += pa.v[i].x; x.v[i].y += pa.v[i].y; x.v[i].z += pa.v[i].z; x.v[i].w += pa.v[i].w;
      }
    }
    if (a.out_fp32) row_store_f32(x, reinterpret_cast<float*>(a.out) + (int64_t)row * a.D, nv, lane);
    else row_store_bf16(x, reinterpret_cast<bf16*>(a.out) + (int64_t)row * a.D, nv, lane);
  }
}

// ------------------------------------------------------------------------------------------------
// teacher token assembly + ln_pre (clip.py:150-152): row (f, tok):  tok==0 ? cls : E[f*P + tok-1], + pos[tok], LN
// ------------------------------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(256) teacher_embed_ln_kernel(const float* __restrict__ E, const float* __restrict__ cls,
                                                               const float* __restrict__ pos, const float* __restrict__ gamma,
                                                               const float* __restrict__ beta, void* __restrict__ out,
                                                               int frames, int P, int D, float eps, int out_f16,
                                                               float* __restrict__ stats) {
  const int lane = threadIdx.x & 31;
  constexpr int nv = NV;
  const int wpb = blockDim.x >> 5;
  const int rows = frames * (P + 1);
  RowT<NV> g, b;
  row_load_f32(g, gamma, nv, lane);
  row_load_f32(b, beta, nv, lane);
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < rows; row += gridDim.x * wpb) {
    const int f = row / (P + 1), tok = row % (P + 1);
    RowT<NV> x, pe;
    if (tok == 0) row_load_f32(x, cls, nv, lane);
    else row_load_f32(x, E + ((int64_t)f * P + tok - 1) * D, nv, lane);
    row_load_f32(pe, pos + (int64_t)tok * D, nv, lane);
    UB_ROW_FOREACH(i, nv) {
      x.v[i].x += pe.v[i].x; x.v[i].y += pe.v[i].y; x.v[i].z += pe.v[i].z; x.v[i].w += pe.v[i].w;
    }
    const float rstd = row_center_rstd(x, nv, D, eps);
    UB_ROW_FOREACH(i, nv) {
      x.v[i].x = x.v[i].x * rstd * g.v[i].x + b.v[i].x;
      x.v[i].y = x.v[i].y * rstd * g.v[i].y + b.v[i].y;
      x.v[i].z = x.v[i].z * rstd * g.v[i].z + b.v[i].z;
      x.v[i].w = x.v[i].w * rstd * g.v[i].w + b.v[i].w;
    }
    if (out_f16) row_store_f16(x, reinterpret_cast<__half*>(out) + (int64_t)row * D, nv, lane);
    else row_store_f32(x, reinterpret_cast<float*>(out) + (int64_t)row * D, nv, lane);
    if (stats != nullptr) {
      // row (sum, sum of squares) of the values as STORED: the next GEMM folds the following LayerNorm into its epilogue
      if (out_f16) {
        UB_ROW_FOREACH(i, nv) {
          x.v[i].x = __half2float(__float2half_rn(x.v[i].x)); x.v[i].y = __half2float(__float2half_rn(x.v[i].y));
          x.v[i].z = __half2float(__float2half_rn(x.v[i].z)); x.v[i].w = __half2float(__float2half_rn(x.v[i].w));
        }
      }
      const float s1 = row_sum(x, nv), s2 = row_dot(x, x, nv);
      if (lane == 0) {
        stats[2 * (int64_t)row] = s1;
        stats[2 * (int64_t)row + 1] = s2;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// backward of y = LN(x)*gamma + beta, fused with the residual-stream gradient:
//   dx_out = (dx_in or 0) + rstd * (g*dy - mean(g*dy) - xhat * mean(g*dy*xhat))
//   dxs_out (bf16, optional) = bf16(dx_out * row_scale)          -- operand of the next dgrad / wgrad GEMMs
//   dgamma += sum_rows dy*xhat,  dbeta += sum_rows dy            -- red.add into fp32 [D]
// ------------------------------------------------------------------------------------------------
struct LnBwdArgs {
  const bf16* dy;
  const float* x;
  const float* gamma;
  const float* dx_in;       // optional
  float* dx_out;
  bf16* dxs_out;            // optional
  const float* row_scale;   // optional, indexed row / rows_per_scale
  int rows_per_scale;
  float* dgamma;
  float* dbeta;
  float* dsum;              // optional: += sum_rows dx_out * row_scale  (bias gradient of the Linear that consumes dxs)
  int rows, D;
  float eps;
};

// block-wide reduction of per-warp column partials, then one red.add per column per block
template <int NV>
UB_DEVINL void block_col_reduce_atomic(const RowT<NV>& part, float* s_buf, float* gdst, int nv, int D) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  row_store_f32(part, s_buf + warp * D, nv, lane);
  __syncthreads();
  for (int c = threadIdx.x; c < D; c += blockDim.x) {
    float s = 0.f;
    for (int w = 0; w < nw; ++w) s += s_buf[w * D + c];
    atomicAdd(gdst + c, s);
  }
}

// The per-column partial sums (dgamma, dbeta, dsum) live in SHARED memory, one private [3][D] strip per warp that the warp
// read-modify-writes once per row (lane l owns float4 slots i*32+l: conflict-free, no atomics), not in registers: the row pass
// then needs ~100 registers instead of 168 and 4 CTAs (16 warps, ~120 KB of loads in flight) fit per SM instead of 3.  ncu on the
// register version (profiles/ncu_step_dram_r02.json, round 1 VERDICT): 27.6 us for 110 MB = 0.65 of the HBM peak at 18 % active
// warps.
template <int NV>
__global__ void __launch_bounds__(128, 4) ln_bwd_kernel(const LnBwdArgs a) {
  extern __shared__ float s_red[];  // [warps][3][D]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int nv = NV;
  const int wpb = blockDim.x >> 5;
  float4* acc_g = reinterpret_cast<float4*>(s_red + (size_t)(warp * 3) * a.D);
  float4* acc_b = acc_g + a.D / 4;
  float4* acc_s = acc_b + a.D / 4;
  UB_ROW_FOREACH(i, nv) {
    acc_g[i * 32 + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
    acc_b[i * 32 + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
    acc_s[i * 32 + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const float invD = 1.f / (float)a.D;
  for (int row = blockIdx.x * wpb + warp; row < a.rows; row += gridDim.x * wpb) {
    // all three inputs of the row are requested before the first reduction: one memory latency per row instead of two
    RowT<NV> x, dy, dx;
    row_load_f32(x, a.x + (int64_t)row * a.D, nv, lane);
    row_load_bf16(dy, a.dy + (int64_t)row * a.D, nv, lane);
    if (a.dx_in) row_load_f32(dx, a.dx_in + (int64_t)row * a.D, nv, lane);
    const float rstd = row_center_rstd(x, nv, a.D, a.eps);
    float s1 = 0.f, s2 = 0.f;
    UB_ROW_FOREACH(i, nv) {
      // x <- xhat ; accumulate dgamma/dbeta ; dy <- g*dy
      x.v[i].x *= rstd; x.v[i].y *= rstd; x.v[i].z *= rstd; x.v[i].w *= rstd;
      float4 ag = acc_g[i * 32 + lane], ab = acc_b[i * 32 + lane];
      ag.x += dy.v[i].x * x.v[i].x; ag.y += dy.v[i].y * x.v[i].y; ag.z += dy.v[i].z * x.v[i].z; ag.w += dy.v[i].w * x.v[i].w;
      ab.x += dy.v[i].x; ab.y += dy.v[i].y; ab.z += dy.v[i].z; ab.w += dy.v[i].w;
      acc_g[i * 32 + lane] = ag;
      acc_b[i * 32 + lane] = ab;
      float4 g;   // gamma from L1 per row
      asm volatile("ld.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(g.x), "=f"(g.y), "=f"(g.z), "=f"(g.w) : "l"(a.gamma + (i * 32 + lane) * 4));
      dy.v[i].x *= g.x; dy.v[i].y *= g.y; dy.v[i].z *= g.z; dy.v[i].w *= g.w;
      s1 += (dy.v[i].x + dy.v[i].y) + (dy.v[i].z + dy.v[i].w);
      s2 += dy.v[i].x * x.v[i].x + dy.v[i].y * x.v[i].y + dy.v[i].z * x.v[i].z + dy.v[i].w * x.v[i].w;
    }
    s1 = warp_sum(s1) * invD;
    s2 = warp_sum(s2) * invD;
    UB_ROW_FOREACH(i, nv) {
      if (!a.dx_in) dx.v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      dx.v[i].x += rstd * (dy.v[i].x - s1 - x.v[i].x * s2);
      dx.v[i].y += rstd * (dy.v[i].y - s1 - x.v[i].y * s2);
      dx.v[i].z += rstd * (dy.v[i].z - s1 - x.v[i].z * s2);
      dx.v[i].w += rstd * (dy.v[i].w - s1 - x.v[i].w * s2);
    }
    row_store_f32(dx, a.dx_out + (int64_t)row * a.D, nv, lane);
    if (a.dxs_out) {
      const float sc = a.row_scale ? __ldg(a.row_scale + row / a.rows_per_scale) : 1.0f;
      UB_ROW_FOREACH(i, nv) {
        dx.v[i].x *= sc; dx.v[i].y *= sc; dx.v[i].z *= sc; dx.v[i].w *= sc;
        if (a.dsum != nullptr) {
          float4 as = acc_s[i * 32 + lane];
          as.x += dx.v[i].x; as.y += dx.v[i].y; as.z += dx.v[i].z; as.w += dx.v[i].w;
          acc_s[i * 32 + lane] = as;
        }
      }
      row_store_bf16(dx, a.dxs_out + (int64_t)row * a.D, nv, lane);
    }
  }
  // block-wide: one red.add per column and output per CTA
  __syncthreads();
  const int n_out = a.dsum != nullptr ? 3 : 2;
  for (int c = threadIdx.x; c < n_out * a.D; c += blockDim.x) {
    const int which = c / a.D, col = c - which * a.D;
    float t = 0.f;
    for (int w = 0; w < wpb; ++w) t += s_red[(size_t)(w * 3 + which) * a.D + col];
    float* dst = which == 0 ? a.dgamma : (which == 1 ? a.dbeta : a.dsum);
    atomicAdd(dst + col, t);
  }
}

// ------------------------------------------------------------------------------------------------
// The same backward with the rows STAGED THROUGH SHARED MEMORY by bulk copies (cp.async.bulk, one elected thread): a persistent
// CTA per SM, 8 warps (one row each per block of 8 rows; thread 0 also issues the copies) and a ring of row blocks that keeps 1-2 whole blocks (61 KB each
// at D = 768: x fp32, dx fp32, dy bf16) in flight per SM whatever the consumers are doing.  The register version above has at
// most 12-16 warps x one row in flight and only while those warps sit in their load phase (ncu: 40 % of the DRAM peak, 70 % of
// the issue slots without an eligible warp); here the memory system always has >= 60 KB per SM outstanding.  The column partials
// (dgamma, dbeta, dsum) stay in registers — with one CTA per SM there is no occupancy to protect.
// ------------------------------------------------------------------------------------------------
constexpr int LNB_ROWS = 8;          // rows per block = consumer warps
template <int NV>
__global__ void __launch_bounds__(256, 1) ln_bwd_staged_kernel(const LnBwdArgs a, int n_stages) {
  extern __shared__ __align__(128) uint8_t lnb_smem[];
  constexpr int D = NV * 128;
  constexpr int X_BYTES = LNB_ROWS * D * 4, DY_BYTES = LNB_ROWS * D * 2;
  constexpr int STAGE = 2 * X_BYTES + DY_BYTES;                       // x | dx | dy
  uint64_t* full = reinterpret_cast<uint64_t*>(lnb_smem + (size_t)n_stages * STAGE);
  uint64_t* empty = full + n_stages;
  float* s_red = reinterpret_cast<float*>(lnb_smem);                 // reused after the main loop: [8 warps][D]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int nv = NV;
  if (threadIdx.x == 0) {
    for (int i = 0; i < n_stages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], LNB_ROWS);
    }
    fence_mbar_init();
  }
  __syncthreads();
  const int n_blocks = (a.rows + LNB_ROWS - 1) / LNB_ROWS;
  // thread 0 doubles as the producer: before it consumes block `it` it requests block it + n_stages - 1 (bulk copies are
  // asynchronous, so this costs it a few instructions per block)
  auto request = [&](int j) {                       // j-th block of this CTA
    const int blk = blockIdx.x + j * gridDim.x;
    if (blk >= n_blocks) return;
    const int st = j % n_stages;
    mbar_wait(&empty[st], (uint32_t)((j / n_stages) & 1) ^ 1u);
    const int row0 = blk * LNB_ROWS, nr = min(LNB_ROWS, a.rows - row0);
    uint8_t* dst = lnb_smem + (size_t)st * STAGE;
    const uint32_t xb = (uint32_t)nr * D * 4, yb = (uint32_t)nr * D * 2;
    mbar_expect_tx(&full[st], xb + yb + (a.dx_in ? xb : 0u));
    bulk_load_1d(dst, a.x + (int64_t)row0 * D, xb, &full[st]);
    if (a.dx_in) bulk_load_1d(dst + X_BYTES, a.dx_in + (int64_t)row0 * D, xb, &full[st]);
    bulk_load_1d(dst + 2 * X_BYTES, a.dy + (int64_t)row0 * D, yb, &full[st]);
  };
  if (threadIdx.x == 0)
    for (int j = 0; j < n_stages - 1; ++j) request(j);
  // ------------------------------------------------------------------ consumers: warp w owns row w of every block
  RowT<NV> dgam, dbet, dsm;
  UB_ROW_FOREACH(i, nv) {
    dgam.v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    dbet.v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    dsm.v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const float invD = 1.f / (float)D;
  int it = 0;
  for (int blk = blockIdx.x; blk < n_blocks; blk += gridDim.x, ++it) {
    const int st = it % n_stages;
    const int row = blk * LNB_ROWS + warp;
    if (threadIdx.x == 0) request(it + n_stages - 1);
    __syncwarp();
    mbar_wait(&full[st], (uint32_t)((it / n_stages) & 1));
    if (row < a.rows) {
      const uint8_t* src = lnb_smem + (size_t)st * STAGE;
      RowT<NV> x, dy, dx;
      row_load_f32(x, reinterpret_cast<const float*>(src) + warp * D, nv, lane);
      row_load_bf16(dy, reinterpret_cast<const bf16*>(src + 2 * X_BYTES) + warp * D, nv, lane);
      if (a.dx_in) row_load_f32(dx, reinterpret_cast<const float*>(src + X_BYTES) + warp * D, nv, lane);
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[st]);          // the row is in registers: the slot may be refilled
      const float rstd = row_center_rstd(x, nv, D, a.eps);
      float s1 = 0.f, s2 = 0.f;
      UB_ROW_FOREACH(i, nv) {
        x.v[i].x *= rstd; x.v[i].y *= rstd; x.v[i].z *= rstd; x.v[i].w *= rstd;
        dgam.v[i].x += dy.v[i].x * x.v[i].x; dgam.v[i].y += dy.v[i].y * x.v[i].y;
        dgam.v[i].z += dy.v[i].z * x.v[i].z; dgam.v[i].w += dy.v[i].w * x.v[i].w;
        dbet.v[i].x += dy.v[i].x; dbet.v[i].y += dy.v[i].y; dbet.v[i].z += dy.v[i].z; dbet.v[i].w += dy.v[i].w;
        float4 g;   // gamma from L1 per row
        asm volatile("ld.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(g.x), "=f"(g.y), "=f"(g.z), "=f"(g.w) : "l"(a.gamma + (i * 32 + lane) * 4));
        dy.v[i].x *= g.x; dy.v[i].y *= g.y; dy.v[i].z *= g.z; dy.v[i].w *= g.w;
        s1 += (dy.v[i].x + dy.v[i].y) + (dy.v[i].z + dy.v[i].w);
        s2 += dy.v[i].x * x.v[i].x + dy.v[i].y * x.v[i].y + dy.v[i].z * x.v[i].z + dy.v[i].w * x.v[i].w;
      }
      s1 = warp_sum(s1) * invD;
      s2 = warp_sum(s2) * invD;
      UB_ROW_FOREACH(i, nv) {
        if (!a.dx_in) dx.v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        dx.v[i].x += rstd * (dy.v[i].x - s1 - x.v[i].x * s2);
        dx.v[i].y += rstd * (dy.v[i].y - s1 - x.v[i].y * s2);
        dx.v[i].z += rstd * (dy.v[i].z - s1 - x.v[i].z * s2);
        dx.v[i].w += rstd * (dy.v[i].w - s1 - x.v[i].w * s2);
      }
      row_store_f32(dx, a.dx_out + (int64_t)row * D, nv, lane);
      if (a.dxs_out) {
        const float sc = a.row_scale ? __ldg(a.row_scale + row / a.rows_per_scale) : 1.0f;
        UB_ROW_FOREACH(i, nv) {
          dx.v[i].x *= sc; dx.v[i].y *= sc; dx.v[i].z *= sc; dx.v[i].w *= sc;
          dsm.v[i].x += dx.v[i].x; dsm.v[i].y += dx.v[i].y; dsm.v[i].z += dx.v[i].z; dsm.v[i].w += dx.v[i].w;
        }
        row_store_bf16(dx, a.dxs_out + (int64_t)row * D, nv, lane);
      }
    } else {
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[st]);
    }
  }
  // ---- column partials of the 8 warps -> one red.add per column and CTA (the ring is idle by now: its smem is reused)
  auto reduce_out = [&](const RowT<NV>& part, float* gdst) {
    __syncthreads();
    row_store_f32(part, s_red + warp * D, nv, lane);
    __syncthreads();
    for (int c = threadIdx.x; c < D; c += 256) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < LNB_ROWS; ++w) t += s_red[w * D + c];
      atomicAdd(gdst + c, t);
    }
  };
  reduce_out(dgam, a.dgamma);
  reduce_out(dbet, a.dbeta);
  if (a.dsum != nullptr) reduce_out(dsm, a.dsum);
}

// ------------------------------------------------------------------------------------------------
// decoder tail (modeling_adaptation.py:203-213): out = u / ||u||,  u = LN(y)*gamma + beta        (fp32 in/out)
// optionally also accumulates the alignment loss  sum_rows (2 - 2 <out, tgt>) * loss_scale  (run_stage1.py:431)
// ------------------------------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(256) dec_tail_fwd_kernel(const float* __restrict__ y, const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, float* __restrict__ out,
                                                           const float* __restrict__ tgt, float* __restrict__ loss_acc,
                                                           float loss_scale, int rows, int D, float eps, int loss_lo,
                                                           int loss_hi) {
  __shared__ float s_loss[8];
  const int lane = threadIdx.x & 31;
  constexpr int nv = NV;
  const int wpb = blockDim.x >> 5;
  RowT<NV> g, b;
  row_load_f32(g, gamma, nv, lane);
  row_load_f32(b, beta, nv, lane);
  float lacc = 0.f;
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < rows; row += gridDim.x * wpb) {
    RowT<NV> x;
    row_load_f32(x, y + (int64_t)row * D, nv, lane);
    const float rstd = row_center_rstd(x, nv, D, eps);
    UB_ROW_FOREACH(i, nv) {
      x.v[i].x = x.v[i].x * rstd * g.v[i].x + b.v[i].x;
      x.v[i].y = x.v[i].y * rstd * g.v[i].y + b.v[i].y;
      x.v[i].z = x.v[i].z * rstd * g.v[i].z + b.v[i].z;
      x.v[i].w = x.v[i].w * rstd * g.v[i].w + b.v[i].w;
    }
    const float inv = 1.0f / sqrtf(row_dot(x, x, nv));
    UB_ROW_FOREACH(i, nv) { x.v[i].x *= inv; x.v[i].y *= inv; x.v[i].z *= inv; x.v[i].w *= inv; }
    row_store_f32(x, out + (int64_t)row * D, nv, lane);
    if (tgt && row >= loss_lo && row < loss_hi) {      // rows outside [loss_lo, loss_hi) do not enter the loss (clip_loss_data)
      RowT<NV> t;
      row_load_f32(t, tgt + (int64_t)row * D, nv, lane);
      lacc += 2.0f - 2.0f * row_dot(x, t, nv);
    }
  }
  if (tgt) {
    if (lane == 0) s_loss[threadIdx.x >> 5] = lacc;
    __syncthreads();
    if (threadIdx.x == 0) {
      float s = 0.f;
      for (int w = 0; w < wpb; ++w) s += s_loss[w];
      atomicAdd(loss_acc, s * loss_scale);
    }
  }
}

// backward of the decoder tail.  Upstream gradient wrt `out` is  go_scale * go[row]  (the engine passes
// go = targets, go_scale = -2/rows_total for the l2 alignment loss; autograd passes grad_output, 1).
//   du = (go - out*<out,go>) / ||u|| ;  dy = LNbwd(du)  -> bf16 ;  dgamma/dbeta accumulated.
template <int NV>
__global__ void __launch_bounds__(256) dec_tail_bwd_kernel(const float* __restrict__ y, const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, const float* __restrict__ go,
                                                           float go_scale, bf16* __restrict__ dy_out, float* __restrict__ dgamma,
                                                           float* __restrict__ dbeta, int rows, int D, float eps, int go_lo,
                                                           int go_hi) {
  extern __shared__ float s_red[];
  const int lane = threadIdx.x & 31;
  constexpr int nv = NV;
  const int wpb = blockDim.x >> 5;
  RowT<NV> g, b, dgam, dbet;
  row_load_f32(g, gamma, nv, lane);
  row_load_f32(b, beta, nv, lane);
  UB_ROW_FOREACH(i, nv) {
    dgam.v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    dbet.v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const float invD = 1.f / (float)D;
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < rows; row += gridDim.x * wpb) {
    RowT<NV> x, u, du;
    row_load_f32(x, y + (int64_t)row * D, nv, lane);
    row_load_f32(du, go + (int64_t)row * D, nv, lane);
    const float rstd = row_center_rstd(x, nv, D, eps);
    UB_ROW_FOREACH(i, nv) {
      x.v[i].x *= rstd; x.v[i].y *= rstd; x.v[i].z *= rstd; x.v[i].w *= rstd;   // xhat
      u.v[i].x = x.v[i].x * g.v[i].x + b.v[i].x; u.v[i].y = x.v[i].y * g.v[i].y + b.v[i].y;
      u.v[i].z = x.v[i].z * g.v[i].z + b.v[i].z; u.v[i].w = x.v[i].w * g.v[i].w + b.v[i].w;
    }
    const float inv = 1.0f / sqrtf(row_dot(u, u, nv));
    const float ug = row_dot(u, du, nv) * inv * inv;     // <out, go> / ||u||  (still unscaled by go_scale)
    const float k = (row >= go_lo && row < go_hi) ? go_scale * inv : 0.f;   // rows outside the range received no gradient
    float s1 = 0.f, s2 = 0.f;
    UB_ROW_FOREACH(i, nv) {
      // du <- go_scale * (go - out*<out,go>) / ||u||
      du.v[i].x = k * (du.v[i].x - u.v[i].x * ug); du.v[i].y = k * (du.v[i].y - u.v[i].y * ug);
      du.v[i].z = k * (du.v[i].z - u.v[i].z * ug); du.v[i].w = k * (du.v[i].w - u.v[i].w * ug);
      dgam.v[i].x += du.v[i].x * x.v[i].x; dgam.v[i].y += du.v[i].y * x.v[i].y;
      dgam.v[i].z += du.v[i].z * x.v[i].z; dgam.v[i].w += du.v[i].w * x.v[i].w;
      dbet.v[i].x += du.v[i].x; dbet.v[i].y += du.v[i].y; dbet.v[i].z += du.v[i].z; dbet.v[i].w += du.v[i].w;
      du.v[i].x *= g.v[i].x; du.v[i].y *= g.v[i].y; du.v[i].z *= g.v[i].z; du.v[i].w *= g.v[i].w;
      s1 += (du.v[i].x + du.v[i].y) + (du.v[i].z + du.v[i].w);
      s2 += du.v[i].x * x.v[i].x + du.v[i].y * x.v[i].y + du.v[i].z * x.v[i].z + du.v[i].w * x.v[i].w;
    }
    s1 = warp_sum(s1) * invD;
    s2 = warp_sum(s2) * invD;
    UB_ROW_FOREACH(i, nv) {
      du.v[i].x = rstd * (du.v[i].x - s1 - x.v[i].x * s2); du.v[i].y = rstd * (du.v[i].y - s1 - x.v[i].y * s2);
      du.v[i].z = rstd * (du.v[i].z - s1 - x.v[i].z * s2); du.v[i].w = rstd * (du.v[i].w - s1 - x.v[i].w * s2);
    }
    row_store_bf16(du, dy_out + (int64_t)row * D, nv, lane);
  }
  block_col_reduce_atomic(dgam, s_red, dgamma, nv, D);
  block_col_reduce_atomic(dbet, s_red, dbeta, nv, D);
}

// x[row] /= ||x[row]||   (teacher targets, clip.py:173)
template <int NV>
__global__ void __launch_bounds__(256) l2norm_rows_kernel(float* __restrict__ x, int rows, int D) {
  const int lane = threadIdx.x & 31;
  constexpr int nv = NV;
  const int wpb = blockDim.x >> 5;
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < rows; row += gridDim.x * wpb) {
    RowT<NV> v;
    row_load_f32(v, x + (int64_t)row * D, nv, lane);
    const float inv = 1.0f / sqrtf(row_dot(v, v, nv));
    UB_ROW_FOREACH(i, nv) { v.v[i].x *= inv; v.v[i].y *= inv; v.v[i].z *= inv; v.v[i].w *= inv; }
    row_store_f32(v, x + (int64_t)row * D, nv, lane);
  }
}

#define UB_LN_DISPATCH(D, KERNEL, GRID, SMEM, STREAM, ...)                                   \
  switch ((D) >> 7) {                                                                         \
    case 1: UB_LAUNCH(KERNEL<1>, GRID, 256, SMEM, STREAM, __VA_ARGS__); break;                       \
    case 2: UB_LAUNCH(KERNEL<2>, GRID, 256, SMEM, STREAM, __VA_ARGS__); break;                       \
    case 4: UB_LAUNCH(KERNEL<4>, GRID, 256, SMEM, STREAM, __VA_ARGS__); break;                       \
    case 6: UB_LAUNCH(KERNEL<6>, GRID, 256, SMEM, STREAM, __VA_ARGS__); break;                       \
    case 8: UB_LAUNCH(KERNEL<8>, GRID, 256, SMEM, STREAM, __VA_ARGS__); break;                       \
    default: break;                                                                           \
  }

static int ln_grid(int rows) {
  const int want = (rows + 7) / 8;
  const int cap = sm_count() * 8;
  return want < cap ? want : cap;
}
static int ln_bwd_grid(int rows) {
  const int want = (rows + 7) / 8;
  const int cap = sm_count() * 2;
  return want < cap ? want : cap;
}
static int check_D(int D, const char* who) {
  UB_REQUIRE(D == 128 || D == 256 || D == 512 || D == 768 || D == 1024, "%s: feature dim must be one of 128/256/512/768/1024 (D=%d)", who, D);
  return 0;
}

}  // namespace ub

using namespace ub;

extern "C" int ub_layernorm_fwd(const void* x, int x_f16, const int* src_rows, const float* gamma, const float* beta, float eps,
                                const float* post_add, const int* post_idx, void* out, int out_fp32, int rows, int D,
                                void* stream) {
  UB_REQUIRE(x && gamma && beta && out, "layernorm_fwd: null pointer");
  UB_REQUIRE(rows > 0, "layernorm_fwd: rows=%d", rows);
  UB_REQUIRE((post_add == nullptr) == (post_idx == nullptr), "layernorm_fwd: post_add and post_idx go together");
  if (check_D(D, "layernorm_fwd")) return 1;
  LnFwdArgs a{x, src_rows, gamma, beta, post_add, post_idx, out, out_fp32, rows, D, eps, x_f16};
  // (a bulk-copy-staged forward like ln_bwd_staged_kernel was measured and dropped: 0.58-0.72 ms per step against 0.51-0.58 ms for
  // this kernel — a 10 us launch over 47 MB does not amortise the ring's set-up)
  UB_LN_DISPATCH(D, ln_fwd_kernel, ln_grid(rows), 0, (cudaStream_t)stream, a)
  return check_launch("ln_fwd_kernel");
}

extern "C" int ub_teacher_embed_ln(const float* E, const float* cls, const float* pos, const float* gamma,
                                   const float* beta, float eps, void* out, int out_f16, float* stats, int frames, int P, int D,
                                   void* stream) {
  UB_REQUIRE(E && cls && pos && gamma && beta && out, "teacher_embed_ln: null pointer");
  if (check_D(D, "teacher_embed_ln")) return 1;
  UB_LN_DISPATCH(D, teacher_embed_ln_kernel, ln_grid(frames * (P + 1)), 0, (cudaStream_t)stream, E, cls, pos, gamma, beta, out, frames, P, D, eps, out_f16, stats)
  return check_launch("teacher_embed_ln_kernel");
}

extern "C" int ub_layernorm_bwd(const void* dy, const float* x, const float* gamma, float eps, const float* dx_in,
                                float* dx_out, void* dxs_out, const float* row_scale, int rows_per_scale, float* dgamma,
                                float* dbeta, float* dsum, int rows, int D, void* stream) {
  UB_REQUIRE(dy && x && gamma && dx_out && dgamma && dbeta, "layernorm_bwd: null pointer");
  UB_REQUIRE(row_scale == nullptr || rows_per_scale > 0, "layernorm_bwd: rows_per_scale must be > 0");
  UB_REQUIRE(dsum == nullptr || dxs_out != nullptr, "layernorm_bwd: dsum is the column sum of dxs_out");
  if (check_D(D, "layernorm_bwd")) return 1;
  LnBwdArgs a{(const bf16*)dy, x, gamma, dx_in, dx_out, (bf16*)dxs_out, row_scale, rows_per_scale, dgamma, dbeta, dsum, rows, D, eps};
  // large inputs: the bulk-copy-staged persistent kernel; small ones (the [B, D] fc_norm backward of stage 2) the plain one
  static int use_staged = -1;
  if (use_staged < 0) {
    const char* e = getenv("UB_LN_BWD_STAGED");
    use_staged = e ? atoi(e) : 1;
  }
  if (use_staged && rows >= 4 * LNB_ROWS * sm_count() && D >= 256) {
    const int n_stages = D <= 768 ? 3 : 2;
    const size_t smem = (size_t)n_stages * (LNB_ROWS * (size_t)D * 10) + 2 * n_stages * sizeof(uint64_t) + 16;
    const int n_blocks = (rows + LNB_ROWS - 1) / LNB_ROWS;
    const int grid = n_blocks < sm_count() ? n_blocks : sm_count();
    cudaStream_t st = (cudaStream_t)stream;
#define UB_LNB_CASE(NVV)                                                                                                     \
  case NVV: {                                                                                                                \
    static bool cfg = false;                                                                                                 \
    if (!cfg) {                                                                                                              \
      cudaError_t e = cudaFuncSetAttribute(ln_bwd_staged_kernel<NVV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
      UB_REQUIRE(e == cudaSuccess, "cudaFuncSetAttribute(ln_bwd_staged smem=%d): %s", (int)smem, cudaGetErrorString(e));      \
      cfg = true;                                                                                                            \
    }                                                                                                                        \
    UB_LAUNCH(ln_bwd_staged_kernel<NVV>, grid, 256, smem, st, a, n_stages);                                                  \
  } break;
    switch (D >> 7) {
      UB_LNB_CASE(2) UB_LNB_CASE(4) UB_LNB_CASE(6) UB_LNB_CASE(8)
      default: break;
    }
#undef UB_LNB_CASE
    return check_launch("ln_bwd_staged_kernel");
  }
  {
    const int want = (rows + 3) / 4, cap = sm_count() * 4;          // 4 warps per CTA, 4 CTAs per SM
    const int grid = want < cap ? want : cap;
    const size_t smem = 4 * 3 * (size_t)D * sizeof(float);         // [warps][dgamma | dbeta | dsum][D]
    cudaStream_t st = (cudaStream_t)stream;
    switch (D >> 7) {
      case 1: UB_LAUNCH(ln_bwd_kernel<1>, grid, 128, smem, st, a); break;
      case 2: UB_LAUNCH(ln_bwd_kernel<2>, grid, 128, smem, st, a); break;
      case 4: UB_LAUNCH(ln_bwd_kernel<4>, grid, 128, smem, st, a); break;
      case 6: UB_LAUNCH(ln_bwd_kernel<6>, grid, 128, smem, st, a); break;
      case 8: UB_LAUNCH(ln_bwd_kernel<8>, grid, 128, smem, st, a); break;
      default: break;
    }
  }
  return check_launch("ln_bwd_kernel");
}

extern "C" int ub_dec_tail_fwd(const float* y, const float* gamma, const float* beta, float eps, float* out,
                               const float* tgt, float* loss_acc, float loss_scale, int loss_row_lo, int loss_row_hi, int rows, int D,
                               void* stream) {
  UB_REQUIRE(y && gamma && beta && out, "dec_tail_fwd: null pointer");
  UB_REQUIRE((tgt == nullptr) || (loss_acc != nullptr), "dec_tail_fwd: tgt needs loss_acc");
  UB_REQUIRE(loss_row_lo >= 0 && loss_row_lo <= loss_row_hi && loss_row_hi <= rows, "dec_tail_fwd: loss rows [%d, %d) of %d", loss_row_lo,
             loss_row_hi, rows);
  if (check_D(D, "dec_tail_fwd")) return 1;
  UB_LN_DISPATCH(D, dec_tail_fwd_kernel, ln_grid(rows), 0, (cudaStream_t)stream, y, gamma, beta, out, tgt, loss_acc, loss_scale, rows, D, eps,
                 loss_row_lo, loss_row_hi)
  return check_launch("dec_tail_fwd_kernel");
}

extern "C" int ub_dec_tail_bwd(const float* y, const float* gamma, const float* beta, float eps, const float* go,
                               float go_scale, int go_row_lo, int go_row_hi, void* dy_out, float* dgamma, float* dbeta, int rows,
                               int D, void* stream) {
  UB_REQUIRE(y && gamma && beta && go && dy_out && dgamma && dbeta, "dec_tail_bwd: null pointer");
  UB_REQUIRE(go_row_lo >= 0 && go_row_lo <= go_row_hi && go_row_hi <= rows, "dec_tail_bwd: gradient rows [%d, %d) of %d", go_row_lo,
             go_row_hi, rows);
  if (check_D(D, "dec_tail_bwd")) return 1;
  UB_LN_DISPATCH(D, dec_tail_bwd_kernel, ln_bwd_grid(rows), 8 * D * sizeof(float), (cudaStream_t)stream, y, gamma, beta, go, go_scale,
                 (bf16*)dy_out, dgamma, dbeta, rows, D, eps, go_row_lo, go_row_hi)
  return check_launch("dec_tail_bwd_kernel");
}

extern "C" int ub_l2norm_rows(float* x, int rows, int D, void* stream) {
  UB_REQUIRE(x != nullptr && rows > 0, "l2norm_rows: bad arguments");
  if (check_D(D, "l2norm_rows")) return 1;
  UB_LN_DISPATCH(D, l2norm_rows_kernel, ln_grid(rows), 0, (cudaStream_t)stream, x, rows, D)
  return check_launch("l2norm_rows_kernel");
}
