// Shared device helpers for the unite_b200 kernels (sm_100a only).
// PTX wrappers: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld), fences.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>

#define UB_DEVINL __device__ __forceinline__

namespace ub {

typedef __nv_bfloat16 bf16;

// ----------------------------------------------------------------------------------------------
// error plumbing (thread-local message, returned through ub_last_error())
// ----------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int check_launch(const char* what);

#define UB_REQUIRE(cond, ...)                 \
  do {                                        \
    if (!(cond)) {                            \
      ub::set_error(__VA_ARGS__);             \
      return 1;                               \
    }                                         \
  } while (0)

int sm_count();

// Every kernel launch of the library goes through here: each argument is static_cast to the kernel's parameter type, so
// that, for example, a void* may be passed for a float* parameter.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
#define UB_LAUNCH(kern, grid, block, smem, stream, ...) \
  (void)ub::launch_kernel(kern, dim3(grid), dim3(block), (size_t)(smem), (cudaStream_t)(stream), __VA_ARGS__)

// ----------------------------------------------------------------------------------------------
// small math / packing
// ----------------------------------------------------------------------------------------------
UB_DEVINL uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
UB_DEVINL float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}
UB_DEVINL float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
UB_DEVINL float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// GELU of the student MLP (modeling_finetune.py:56, nn.GELU = x * Phi(x)) and its derivative.
// B200's 3-operand FP32 pipe issues at half rate (~64 lane-ops/clk/SM), so a K=768 GEMM epilogue can afford about a
// dozen FP32 ops per output element before it, not the tensor pipe, sets the tile time.  Default evaluation:
//     Phi(x) = 0.5 * (1 + tanh(u)),  u = x * (0.7978845608 + 0.0356774081 x^2)        (MUFU.TANH, 5 FP ops)
// which differs from the erf form by <= 4.7e-4 absolute (<= 2.2e-4 of the value for |x| >= 1) — an order of
// magnitude below the bf16 resolution (3.9e-3 relative) of the tensors these values are stored in.  Compile with
// -DUB_GELU_ERF for the Abramowitz-Stegun 7.1.26 erf (|err| <= 1.5e-7; one ex2 + one rcp + 10 FP ops).
#ifdef UB_GELU_ERF
UB_DEVINL void gelu_cdf_pdf(float x, float& cdf, float& e) {
  const float z = fabsf(x) * 0.70710678118654752f;
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.0f)));
  e = __expf(-z * z);                                     // exp(-x^2/2)
  float poly = fmaf(1.061405429f, t, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  const float half_erfc = 0.5f * poly * t * e;            // 0.5*(1 - erf(z)), z >= 0
  cdf = x >= 0.f ? 1.0f - half_erfc : half_erfc;
}
UB_DEVINL float gelu_erf(float x) {
  float cdf, e;
  gelu_cdf_pdf(x, cdf, e);
  return x * cdf;
}
UB_DEVINL float gelu_erf_grad(float x) {
  float cdf, e;
  gelu_cdf_pdf(x, cdf, e);
  return fmaf(x * 0.3989422804014327f, e, cdf);
}
#else
UB_DEVINL float gelu_erf(float x) {
  const float x2 = x * x;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(x * fmaf(x2, 0.0356774081f, 0.7978845608f)));
  const float hx = 0.5f * x;
  return fmaf(hx, t, hx);
}
UB_DEVINL float gelu_erf_grad(float x) {
  const float x2 = x * x;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(x * fmaf(x2, 0.0356774081f, 0.7978845608f)));
  const float dudx = fmaf(x2, 0.1070322243f, 0.7978845608f);
  const float sech2 = fmaf(-t, t, 1.0f);
  return fmaf(0.5f * x * sech2, dudx, fmaf(0.5f, t, 0.5f));
}
#endif
// Two elements at a time on the packed fp32x2 pipe (FMUL2 / FFMA2): the K = 768 GELU epilogues are bound by FP32 issue
// slots, and the packed forms halve every instruction except the two MUFU.TANH.
#ifndef UB_GELU_ERF
UB_DEVINL float2 gelu_erf2(float2 x) {
  const float2 x2 = __fmul2_rn(x, x);
  const float2 in = __ffma2_rn(x2, make_float2(0.0356774081f, 0.0356774081f), make_float2(0.7978845608f, 0.7978845608f));
  const float2 u = __fmul2_rn(x, in);
  float2 t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t.x) : "f"(u.x));
  asm("tanh.approx.f32 %0, %1;" : "=f"(t.y) : "f"(u.y));
  const float2 hx = __fmul2_rn(x, make_float2(0.5f, 0.5f));
  return __ffma2_rn(hx, t, hx);
}
UB_DEVINL float2 gelu_erf_grad2(float2 x) {
  const float2 x2 = __fmul2_rn(x, x);
  const float2 in = __ffma2_rn(x2, make_float2(0.0356774081f, 0.0356774081f), make_float2(0.7978845608f, 0.7978845608f));
  const float2 u = __fmul2_rn(x, in);
  float2 t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t.x) : "f"(u.x));
  asm("tanh.approx.f32 %0, %1;" : "=f"(t.y) : "f"(u.y));
  const float2 dudx = __ffma2_rn(x2, make_float2(0.1070322243f, 0.1070322243f), make_float2(0.7978845608f, 0.7978845608f));
  const float2 sech2 = __ffma2_rn(make_float2(-t.x, -t.y), t, make_float2(1.0f, 1.0f));
  const float2 hxs = __fmul2_rn(__fmul2_rn(x, make_float2(0.5f, 0.5f)), sech2);
  return __ffma2_rn(hxs, dudx, __ffma2_rn(t, make_float2(0.5f, 0.5f), make_float2(0.5f, 0.5f)));
}
#else
UB_DEVINL float2 gelu_erf2(float2 x) { return make_float2(gelu_erf(x.x), gelu_erf(x.y)); }
UB_DEVINL float2 gelu_erf_grad2(float2 x) { return make_float2(gelu_erf_grad(x.x), gelu_erf_grad(x.y)); }
#endif
// QuickGELU (teacher, clip.py:29): x * sigmoid(1.702 x) = 0.5x * (1 + tanh(0.851 x)); one MUFU op
UB_DEVINL float quick_gelu(float x) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.851f * x));
  const float hx = 0.5f * x;
  return fmaf(hx, t, hx);
}

UB_DEVINL uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
UB_DEVINL void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
UB_DEVINL void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
UB_DEVINL void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
UB_DEVINL void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
UB_DEVINL void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
UB_DEVINL bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
#ifdef UB_MBAR_SUSPEND_HINT
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
#else
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
#endif
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
#ifdef UB_MBAR_SUSPEND_HINT
        , "r"((uint32_t)UB_MBAR_SUSPEND_HINT)
#endif
      : "memory");
  return ok != 0;
}
UB_DEVINL void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ----------------------------------------------------------------------------------------------
// TMA
// ----------------------------------------------------------------------------------------------
UB_DEVINL void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2D tile load global -> shared, completes `bytes` on the mbarrier
UB_DEVINL void tma_load_2d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
UB_DEVINL void tma_load_3d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// 1-D bulk copy global -> shared (no tensor map): `bytes` must be a multiple of 16, both addresses 16-byte aligned
UB_DEVINL void bulk_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// L2 prefetch of a tile (no smem, no completion tracking)
UB_DEVINL void tma_prefetch_2d(const CUtensorMap* m, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(m)), "r"(c0), "r"(c1)
               : "memory");
}

// smem -> global tile store / fp32 reduce-add (bulk async group completion), clipped at the tensor bounds
UB_DEVINL void tma_store_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
UB_DEVINL void tma_reduce_add_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
UB_DEVINL void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
UB_DEVINL void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

// ----------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ----------------------------------------------------------------------------------------------
UB_DEVINL void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
}
UB_DEVINL void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
UB_DEVINL void tmem_dealloc(uint32_t addr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols) : "memory");
}
UB_DEVINL void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
UB_DEVINL void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]; bf16 inputs, fp32 accumulate.  Issued by ONE thread.
UB_DEVINL void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
UB_DEVINL void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns (thread i <- lane i)
UB_DEVINL void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
UB_DEVINL void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor, K-major operand, 128-byte swizzle, rows 128 B apart
// (the layout a TMA box {64 bf16, rows} with CU_TENSOR_MAP_SWIZZLE_128B produces).
//   start address >> 4 | LBO (ignored for swizzled K-major, set 1) | SBO = 1024 B (8 rows) | version 1 | SW128
UB_DEVINL uint64_t umma_desc_kmajor_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// MN-major operand, 128-byte swizzle: smem holds [k][64 mn-elements] rows of 128 B (TMA box {64 mn, k-rows}),
// successive 64-wide mn chunks `lbo_bytes` apart, successive 8-k groups 1024 B apart.
UB_DEVINL uint64_t umma_desc_mnmajor_sw128(uint32_t saddr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor: kind::f16, A/B bf16, D fp32.
UB_DEVINL constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ----------------------------------------------------------------------------------------------
// CTA pairs (cluster of 2): cta_group::2 variants.  Both CTAs use identical smem layouts; the leader (rank 0)
// issues the MMAs, both issue their own TMA loads which complete_tx on the LEADER's mbarrier.
// ----------------------------------------------------------------------------------------------
UB_DEVINL uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
UB_DEVINL void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of the same smem offset in CTA `rank` of the cluster (shared::cluster window)
UB_DEVINL uint32_t mapa_u32(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
// relaxed: the arrive only orders TMEM reads (tcgen05.wait::ld + fence::before_thread_sync), no global-memory release
// is needed — a release.cluster arrive costs an ERRBAR that drains every outstanding store of the warp.
UB_DEVINL void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
UB_DEVINL void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (ok == 0);
}
UB_DEVINL void tma_load_2d_cg2(const CUtensorMap* m, uint32_t leader_bar_cluster_addr, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(leader_bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
// same, multicast: the box lands at this smem offset in every CTA of `mask`; each destination's bytes are counted on the
// barrier at this offset in the leader of THAT destination's pair
UB_DEVINL void tma_load_2d_cg2_mc(const CUtensorMap* m, uint32_t leader_bar_cluster_addr, void* dst, int c0, int c1, uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(leader_bar_cluster_addr), "r"(c0), "r"(c1), "h"(mask)
      : "memory");
}
UB_DEVINL void tmem_alloc_cg2(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
}
UB_DEVINL void tmem_relinquish_cg2() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
UB_DEVINL void tmem_dealloc_cg2(uint32_t addr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols) : "memory");
}
UB_DEVINL void umma_bf16_cg2(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (once) on the barrier at this smem offset in BOTH CTAs of the pair when the issued MMAs complete
UB_DEVINL void umma_commit_cg2(uint64_t* bar, uint16_t mask = 3) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(mask)
               : "memory");
}

// ----------------------------------------------------------------------------------------------
// attention kernels: A operand from TMEM (TS form), narrow TMEM loads / stores, 3-D TMA store, ex2
// ----------------------------------------------------------------------------------------------
UB_DEVINL void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// one elected lane of a converged warp (the compiler keeps the guarded region's operands in uniform registers)
UB_DEVINL bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred != 0;
}
// tcgen05.mma with descriptors given as {low word (address >> 4 | LBO << 16), constant high word}
UB_DEVINL void umma_ss_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"((uint32_t)accumulate)
      : "memory");
}
UB_DEVINL void umma_ts_lo(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"((uint32_t)accumulate)
      : "memory");
}
UB_DEVINL void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
UB_DEVINL void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
UB_DEVINL void tmem_st_32x8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
UB_DEVINL void tmem_ld_32x1(uint32_t taddr, uint32_t& r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(taddr) : "memory");
}
UB_DEVINL void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
UB_DEVINL void tma_store_3d(const CUtensorMap* m, const void* src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
UB_DEVINL float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ----------------------------------------------------------------------------------------------
// 128-bit streaming global access
// ----------------------------------------------------------------------------------------------
UB_DEVINL uint4 ldg_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
UB_DEVINL void stg_v4(void* p, uint4 v) {
  asm volatile("st.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}

}  // namespace ub
