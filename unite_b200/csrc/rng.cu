// Device-side DropPath draws (stochastic depth), replayable inside a CUDA graph.
//
// Replaces   timm.models.layers.drop_path as called by DropPath.forward (src/models/modeling_finetune.py:42-50) from
//            Block.forward (:143-150): per sample b and residual branch, x * floor(keep + u) / keep with u ~ U[0,1),
//            keep = 1 - p_l, p_l = linspace(0, drop_path, depth)[l] (:311, modeling_adaptation.py:92).
// The reference draws u with torch.rand inside every block (24 tiny launches per forward).  Here ONE launch per step
// writes all depth x 2 x B factors; the GEMM epilogues consume them as `row_scale` (forward) and the LayerNorm backward /
// cast kernels as their gradient scale.  The generator is counter-based (Philox4x32-10, Salmon et al. SC'11: key = seed,
// counter = (element/4, 0, step)), and the step number lives in DEVICE memory and is advanced by the kernel itself, so a
// captured launch produces fresh draws on every graph replay without any host involvement.  oracle/philox.py restates the
// same stream on the host, which makes the draws of step s reproducible for parity tests.
#include "common.cuh"
#include "../../include/unite_b200.h"

namespace ub {

UB_DEVINL void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// out[(l*2 + branch)*B + b] = floor(keep_l + u) / keep_l; one block, every thread reads the step before thread 0 bumps it
__global__ void __launch_bounds__(256) drop_path_draw_kernel(const float* __restrict__ rates, float* __restrict__ out, int depth, int B,
                                                             uint32_t seed_lo, uint32_t seed_hi, unsigned long long* __restrict__ step) {
  const unsigned long long s = *step;
  __syncthreads();
  const int n = depth * 2 * B;
  for (int q = threadIdx.x; 4 * q < n; q += blockDim.x) {
    uint32_t r[4];
    philox4x32_10((uint32_t)q, 0u, (uint32_t)s, (uint32_t)(s >> 32), seed_lo, seed_hi, r);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int e = 4 * q + j;
      if (e < n) {
        const float keep = 1.0f - rates[e / (2 * B)];
        const float u = (float)(r[j] >> 8) * 5.9604644775390625e-8f;      // 24 random bits -> [0, 1)
        out[e] = floorf(keep + u) / keep;
      }
    }
  }
  if (threadIdx.x == 0) *step = s + 1ull;
}

}  // namespace ub

using namespace ub;

extern "C" int ub_drop_path_draw(const float* rates, float* out, int depth, int B, uint64_t seed, uint64_t* step, void* stream) {
  UB_REQUIRE(rates && out && step && depth > 0 && B > 0, "drop_path_draw: null pointer or empty shape");
  UB_LAUNCH(drop_path_draw_kernel, 1, 256, 0, (cudaStream_t)stream, rates, out, depth, B, (uint32_t)seed, (uint32_t)(seed >> 32),
            (unsigned long long*)step);
  return check_launch("drop_path_draw_kernel");
}
