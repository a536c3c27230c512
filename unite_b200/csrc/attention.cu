// Multi-head self-attention (head_dim 64, non-causal, no dropout): the C-ABI entry points, the backward's D pre-pass and
// the teacher's last-layer CLS-row attention map.
//
// Replaces   student  modeling_finetune.py:110-116 (q*scale, q@k^T, softmax, @v) and its autograd backward,
//            teacher  clip.py:40-52 (nn.MultiheadAttention core), clip.py:95-96,183 (head-averaged CLS row).
// Layout     qkv bf16 [n_seq*S, 3*H*64]: per token row q|k|v, each H heads x 64 (what both the packed in_proj
//            of nn.MultiheadAttention and `qkv.reshape(B,N,3,H,-1)` produce); o bf16 [n_seq*S, H*64].
// ub_attn_fwd / ub_attn_bwd pick one of four tcgen05 / TMEM kernels by S and by whether an LSE is kept: attention_tc.cu,
// attention_fwd_lse_tc.cu and attention_bwd_tc.cu for short sequences, attention_long_tc.cu for every longer one.  None of
// them writes the S x S score matrix to HBM: the forward keeps only the per-row log-sum-exp, the backward recomputes P.
#include "common.cuh"
#include "../../include/unite_b200.h"

namespace ub {

constexpr int HD = 64;          // head dim

// ------------------------------------------------------------------------------------------------
// backward pre-pass:  D[seq,h,row] = sum_d dO * O
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) attn_bwd_prep_kernel(const bf16* __restrict__ o, const bf16* __restrict__ d_o,
                                                            float* __restrict__ D, long n_chunks, int S, int H) {
  // one thread = 8 consecutive channels (16 B of o and of d_o); 8 threads = one (row, head); 3 shuffles finish the dot product
  const long id = (long)blockIdx.x * blockDim.x + threadIdx.x;
  float v = 0.f;
  if (id < n_chunks) {
    const uint4 a = ldg_nc_v4(o + id * 8), b = ldg_nc_v4(d_o + id * 8);
    float2 x, y;
    x = unpack_bf16x2(a.x); y = unpack_bf16x2(b.x); v = x.x * y.x + x.y * y.y;
    x = unpack_bf16x2(a.y); y = unpack_bf16x2(b.y); v += x.x * y.x + x.y * y.y;
    x = unpack_bf16x2(a.z); y = unpack_bf16x2(b.z); v += x.x * y.x + x.y * y.y;
    x = unpack_bf16x2(a.w); y = unpack_bf16x2(b.w); v += x.x * y.x + x.y * y.y;
  }
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  if (id < n_chunks && (threadIdx.x & 7) == 0) {
    const long rh = id >> 3;                       // row * H + head
    const long row = rh / H;
    const int h = (int)(rh % H);
    const long seq = row / S;
    const int r = (int)(row % S);
    D[(seq * H + h) * S + r] = v;
  }
}

// ------------------------------------------------------------------------------------------------
// teacher: head-averaged softmax row of the CLS query over the patch keys (clip.py:95-96,183)
//   out[seq, j] = 1/H * sum_h softmax_k(q_cls . k / sqrt(d))[j+1],   j in [0, S-1)
// ------------------------------------------------------------------------------------------------
__global__ void cls_attn_kernel(const bf16* __restrict__ qkv, float* __restrict__ out, int S, int H, float scale) {
  extern __shared__ float s_probs[];  // [H][S]
  const int seq = blockIdx.x, h = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t ld = 3 * (int64_t)H * HD;
  const bf16* base = qkv + (int64_t)seq * S * ld;
  // q_cls for this head, all 64 values in registers of every lane (read as 8 x 16 B, L1-broadcast)
  float q[HD];
  {
    const uint4* pq = reinterpret_cast<const uint4*>(base + h * HD);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const uint4 v = pq[i];
      float2 f;
      f = unpack_bf16x2(v.x); q[i * 8 + 0] = f.x; q[i * 8 + 1] = f.y;
      f = unpack_bf16x2(v.y); q[i * 8 + 2] = f.x; q[i * 8 + 3] = f.y;
      f = unpack_bf16x2(v.z); q[i * 8 + 4] = f.x; q[i * 8 + 5] = f.y;
      f = unpack_bf16x2(v.w); q[i * 8 + 6] = f.x; q[i * 8 + 7] = f.y;
    }
  }
  float* P = s_probs + h * S;
  float mx = -INFINITY;
  for (int j = lane; j < S; j += 32) {
    const uint4* pk = reinterpret_cast<const uint4*>(base + (int64_t)j * ld + (H + h) * HD);
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const uint4 v = pk[i];
      float2 f;
      f = unpack_bf16x2(v.x); acc += q[i * 8 + 0] * f.x + q[i * 8 + 1] * f.y;
      f = unpack_bf16x2(v.y); acc += q[i * 8 + 2] * f.x + q[i * 8 + 3] * f.y;
      f = unpack_bf16x2(v.z); acc += q[i * 8 + 4] * f.x + q[i * 8 + 5] * f.y;
      f = unpack_bf16x2(v.w); acc += q[i * 8 + 6] * f.x + q[i * 8 + 7] * f.y;
    }
    acc *= scale;
    P[j] = acc;
    mx = fmaxf(mx, acc);
  }
  mx = warp_max(mx);
  float sum = 0.f;
  for (int j = lane; j < S; j += 32) {
    const float e = __expf(P[j] - mx);
    P[j] = e;
    sum += e;
  }
  sum = warp_sum(sum);
  const float inv = 1.f / sum;
  for (int j = lane; j < S; j += 32) P[j] *= inv;
  __syncthreads();
  const float invH = 1.f / (float)H;
  for (int j = threadIdx.x; j < S - 1; j += blockDim.x) {
    float a = 0.f;
    for (int hh = 0; hh < H; ++hh) a += s_probs[hh * S + j + 1];
    out[(int64_t)seq * (S - 1) + j] = a * invH;
  }
}

}  // namespace ub

namespace ub {
int launch_attn_fwd_tc(const void* qkv, void* o, int n_seq, int S, int H, float scale, cudaStream_t stream);
int launch_attn_fwd_lse_tc(const void* qkv, void* o, float* lse, int n_seq, int S, int H, float scale, cudaStream_t stream);
int launch_attn_bwd_tc(const void* qkv, const void* d_o, const float* lse, const float* Dv, void* dqkv, float* dbias, int n_seq, int S,
                       int H, float scale, cudaStream_t stream);
int launch_attn_fwd_long_tc(const void* qkv, void* o, float* lse, int n_seq, int S, int H, float scale, cudaStream_t stream);
int launch_attn_bwd_long_tc(const void* qkv, const void* d_o, const float* lse, const float* Dv, void* dqkv, float* dbias, int n_seq, int S,
                            int H, float scale, cudaStream_t stream);
}
using namespace ub;

extern "C" int ub_attn_fwd(const void* qkv, void* o, float* lse, int n_seq, int S, int H, float scale, void* stream) {
  UB_REQUIRE(qkv && o, "attn_fwd: null pointer");
  UB_REQUIRE(n_seq > 0 && S > 0 && H > 0, "attn_fwd: bad shape n_seq=%d S=%d H=%d", n_seq, S, H);
  UB_REQUIRE(n_seq <= 65535 && H <= 65535, "attn_fwd: grid too large");
  // inference over short sequences (the teacher's 197-token frames): tcgen05 / TMEM kernel
  if (lse == nullptr && S <= 240) return   // (K and V for NK <= 240 padded keys fit the 227 KB smem budget twice)
    launch_attn_fwd_tc(qkv, o, n_seq, S, H, scale, (cudaStream_t)stream);
  // training forward (LSE kept for the backward) over the student's <= 320 visible tokens: two-chunk tcgen05 kernel
  if (lse != nullptr && S <= 320) return launch_attn_fwd_lse_tc(qkv, o, lse, n_seq, S, H, scale, (cudaStream_t)stream);
  // everything longer (stage-2 / stage-3 all-token passes, S = 1568): streamed-KV tcgen05 kernel, with or without LSE
  return launch_attn_fwd_long_tc(qkv, o, lse, n_seq, S, H, scale, (cudaStream_t)stream);
}

extern "C" int ub_attn_bwd(const void* qkv, const void* o, const void* d_o, const float* lse, float* D_ws, void* dqkv, float* dbias,
                           int n_seq, int S, int H, float scale, void* stream) {
  UB_REQUIRE(qkv && d_o && lse && D_ws && dqkv, "attn_bwd: null pointer");
  UB_REQUIRE(n_seq > 0 && S > 0 && H > 0, "attn_bwd: bad shape n_seq=%d S=%d H=%d", n_seq, S, H);
  cudaStream_t st = (cudaStream_t)stream;
  const int n_rows = n_seq * S;
  const long n_chunks = (long)n_rows * H * 8;
  if (o != nullptr) {        // o == NULL: D_ws already holds rowsum(dO o O) (the GEMM that produced dO wrote it: ub_gemm_epilogue.dot_out)
    UB_LAUNCH(attn_bwd_prep_kernel, (unsigned)((n_chunks + 255) / 256), 256, 0, st, (const bf16*)o, (const bf16*)d_o, D_ws, n_chunks, S, H);
    if (check_launch("attn_bwd_prep_kernel")) return 1;
  }
  // short sequences (the student's <= 320 visible tokens): single-pass tcgen05 / TMEM kernel
  if (S <= 320) return launch_attn_bwd_tc(qkv, d_o, lse, D_ws, dqkv, dbias, n_seq, S, H, scale, st);
  return launch_attn_bwd_long_tc(qkv, d_o, lse, D_ws, dqkv, dbias, n_seq, S, H, scale, st);
}

extern "C" int ub_cls_attn(const void* qkv, float* out, int n_seq, int S, int H, float scale, void* stream) {
  UB_REQUIRE(qkv && out, "cls_attn: null pointer");
  UB_REQUIRE(H >= 1 && H <= 32 && S >= 2, "cls_attn: unsupported H=%d S=%d", H, S);
  const size_t smem = (size_t)H * S * sizeof(float);
  UB_REQUIRE(smem <= 48 * 1024, "cls_attn: sequence too long for the CLS-row kernel (S=%d)", S);
  UB_LAUNCH(cls_attn_kernel, n_seq, H * 32, smem, (cudaStream_t)stream, (const bf16*)qkv, out, S, H, scale);
  return check_launch("cls_attn_kernel");
}
