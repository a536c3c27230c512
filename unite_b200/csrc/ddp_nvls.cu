// Data-parallel optimizer step fused with its collective over NVLink 5 / NVSwitch multicast (NVLS):
//     reduce-scatter of the gradient arena  +  AdamW on the owned shard  +  all-gather of the bf16 weight shadow
// in ONE kernel, no NCCL call on the step.
//
// Replaces   run_stage1.py:809 (DistributedDataParallel's bucketed all-reduce of 352 MB of fp32 gradients) followed by
//            src/utils.py:608-622 + src/optim_factory.py:162-163 (grad-norm, AdamW) and the bf16 re-cast of the weights.
//
// Every rank maps the SAME gradient arena and bf16 shadow through a multicast address (symmetric memory, one allocation
// per rank bound to one multicast object).  Rank r owns the r-th contiguous slice of the decay segment (the matrices):
//   g   = multimem.ld_reduce.add.v4.f32 [grads_mc + i]      the switch sums the N ranks' gradients on the way in
//   p,m,v (local fp32, owner only)  <- AdamW(g / N)
//   multimem.st.v4 [w16_mc + i]     <- bf16(p)              the switch writes the refreshed weights into all N shadows
// so each gradient element crosses NVLink once in each direction, 2 bytes per parameter come back instead of 4, the
// optimizer's own HBM traffic (28 B / param) is divided by N, and the gradient sum never lands in HBM at all.  The
// no-decay segment (biases / LayerNorm, ~0.1 % of the arena, read in fp32 by the kernels) is reduced and updated by every
// rank, so it stays replicated.  fp32 master weights and Adam moments of the decay segment are SHARDED (ZeRO-1): the
// host gathers them when a state_dict is taken (unite_b200/ddp.py: NvlsShardedStep.consolidate).
//
// Cross-GPU ordering: CTA b of every rank signals slot b on all ranks (multimem.red.release.sys) and spins on its own
// copy (ld.acquire.sys) — once on entry (every peer's backward has finished, nobody still reads the old shadow) and once
// before exit (every peer's loads of my gradients and stores into my shadow are done).  Slots are monotone counters, the
// per-CTA epoch lives in local device memory, so the launch is replayable inside a CUDA graph.  Spins are bounded: a
// peer that never arrives sets `err` and lets the kernel finish instead of hanging the GPU.
#include <cstdlib>
#include "common.cuh"
#include "../../include/unite_b200.h"

namespace ub {

UB_DEVINL float4 mc_ld_reduce_add_f32x4(const float* mc) {
  float4 r;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(mc) : "memory");
  return r;
}
UB_DEVINL void mc_st_b32x4(void* mc, uint4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};"
               :: "l"(mc), "f"(__uint_as_float(v.x)), "f"(__uint_as_float(v.y)), "f"(__uint_as_float(v.z)), "f"(__uint_as_float(v.w))
               : "memory");
}
UB_DEVINL float4 ld_sys_f32x4(const float4* p) {          // peer memory over NVLink: no L1, one pass
  float4 r;
#ifdef UB_NVLS_STRONG_LOADS
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p) : "memory");
#else
  // weak load: the data was published by the peer's release before the entry barrier's acquire, every address is read once
  asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p) : "memory");
#endif
  return r;
}
UB_DEVINL void mc_red_add_f32(float* mc, float v) {
  asm volatile("multimem.red.relaxed.sys.global.add.f32 [%0], %1;" :: "l"(mc), "f"(v) : "memory");
}
UB_DEVINL void mc_signal(uint32_t* mc_slot) {
  asm volatile("multimem.red.release.sys.global.add.u32 [%0], %1;" :: "l"(mc_slot), "r"(1u) : "memory");
}
UB_DEVINL uint32_t ld_acquire_sys_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// spin until *slot >= target (wrap-safe); gives up after `limit` clocks, records the failure in *err (sticky: every later
// launch returns at once, see nvls_dead) and returns false — the caller must then NOT touch parameters or optimizer state
UB_DEVINL bool wait_ge(const uint32_t* slot, uint32_t target, long long limit, int* err, int code) {
  const long long t0 = clock64();
  while ((int32_t)(ld_acquire_sys_u32(slot) - target) < 0) {
    if (clock64() - t0 > limit || *reinterpret_cast<volatile int*>(err) != 0) {
      atomicCAS(err, 0, code);
      return false;
    }
    __nanosleep(32);
  }
  return true;
}
// a previous launch (or another CTA of this one) gave up on a barrier: the step is void, nothing may be updated any more
UB_DEVINL bool nvls_dead(const int* err) { return *reinterpret_cast<const volatile int*>(err) != 0; }

struct NvlsStep {
  float* p; const float* g_mc; float* m; float* v;
  uint4* w16; uint4* w16_mc;
  long n8, n8_decay;
  int rank, world;
  const float* hyper;
  float* gnorm_mc;
  uint32_t* flags; uint32_t* flags_mc; uint32_t* epoch;
  int* err;
  long long spin_limit;
  const float* g_peer[8];        // every rank's mapping of the gradient arena, by rank (P2P mode)
  uint4* w16_peer[8];            // every rank's mapping of the bf16 shadow, by rank
  int mc_store;                  // 1: shadow written through the multicast address, 0: one plain store per peer
  float* stage_peer[8];          // push mode: every rank's mapping of the staging buffer [world][shard] (slot s = rank s's gradients)
  uint32_t* mid; uint32_t* mid_mc;   // push mode: grid-wide cross-GPU counter between the scatter and the update phase
  int prepushed;                     // push mode: the staging buffers were already filled by copy-engine pushes during backward
};

template <int kW, bool kDecay, bool kBroadcast, bool kNorm>
UB_DEVINL void nvls_update8(const NvlsStep& a, long i, const float4 g0, const float4 g1, float lr, float wd, float beta1, float beta2,
                            float eps, float step_size, float bc2_sqrt, float grad_scale, float& gacc) {
  float4* p4 = reinterpret_cast<float4*>(a.p) + 2 * i;
  float4* m4 = reinterpret_cast<float4*>(a.m) + 2 * i;
  float4* v4 = reinterpret_cast<float4*>(a.v) + 2 * i;
  float4 pp[2] = {p4[0], p4[1]}, mm[2] = {m4[0], m4[1]}, vv[2] = {v4[0], v4[1]};
  const float4 gg[2] = {g0, g1};
  const float decay = kDecay ? (1.0f - lr * wd) : 1.0f;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    if (kNorm) gacc += gg[h].x * gg[h].x + gg[h].y * gg[h].y + gg[h].z * gg[h].z + gg[h].w * gg[h].w;
#define UB_ADAM_ONE(c)                                                        \
  {                                                                           \
    const float gr = gg[h].c * grad_scale;                                    \
    pp[h].c *= decay;                                                         \
    mm[h].c = beta1 * mm[h].c + (1.0f - beta1) * gr;                          \
    vv[h].c = beta2 * vv[h].c + (1.0f - beta2) * gr * gr;                     \
    pp[h].c -= step_size * (mm[h].c / (sqrtf(vv[h].c) / bc2_sqrt + eps));     \
  }
    UB_ADAM_ONE(x) UB_ADAM_ONE(y) UB_ADAM_ONE(z) UB_ADAM_ONE(w)
#undef UB_ADAM_ONE
  }
  p4[0] = pp[0]; p4[1] = pp[1];
  m4[0] = mm[0]; m4[1] = mm[1];
  v4[0] = vv[0]; v4[1] = vv[1];
  uint4 o;
  o.x = pack_bf16x2(pp[0].x, pp[0].y); o.y = pack_bf16x2(pp[0].z, pp[0].w);
  o.z = pack_bf16x2(pp[1].x, pp[1].y); o.w = pack_bf16x2(pp[1].z, pp[1].w);
  if (!kBroadcast) {
    a.w16[i] = o;
  } else if (kW == 0 || a.mc_store) {
    mc_st_b32x4(a.w16_mc + i, o);
  } else {
#pragma unroll
    for (int r = 0; r < (kW > 0 ? kW : 1); ++r) a.w16_peer[r][i] = o;
  }
}

// one segment [lo, hi) of 8-element units, kU units per thread in flight: every load of a round is issued before the first is
// consumed (an NVLink round trip is microseconds; the queue depth is what buys bandwidth).
//   kW == 0   gradients summed inside the switch: multimem.ld_reduce on the multicast address
//   kW == N   gradients read from each of the N ranks' mappings (plain NVLink P2P loads) and summed in rank order — the
//             same order on every rank and every run, so the result is bitwise reproducible
template <int kU, int kW, bool kDecay, bool kBroadcast, bool kNorm>
UB_DEVINL void nvls_segment(const NvlsStep& a, long lo, long hi, long tid, long stride, float lr, float wd, float beta1, float beta2,
                            float eps, float step_size, float bc2_sqrt, float grad_scale, float& gacc) {
  constexpr int kSrc = kW > 0 ? kW : 1;
  for (long base = lo + tid; base < hi; base += stride * kU) {
    float4 g[kU][kSrc][2];
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      const long i = base + u * stride;
      if (i < hi) {
        if (kW == 0) {
          g[u][0][0] = mc_ld_reduce_add_f32x4(a.g_mc + 8 * i);
          g[u][0][1] = mc_ld_reduce_add_f32x4(a.g_mc + 8 * i + 4);
        } else {
#pragma unroll
          for (int r = 0; r < kSrc; ++r) {
            const float4* src = reinterpret_cast<const float4*>(a.g_peer[r]) + 2 * i;
            g[u][r][0] = ld_sys_f32x4(src);
            g[u][r][1] = ld_sys_f32x4(src + 1);
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      const long i = base + u * stride;
      if (i < hi) {
        float4 g0 = g[u][0][0], g1 = g[u][0][1];
#pragma unroll
        for (int r = 1; r < kSrc; ++r) {
          g0.x += g[u][r][0].x; g0.y += g[u][r][0].y; g0.z += g[u][r][0].z; g0.w += g[u][r][0].w;
          g1.x += g[u][r][1].x; g1.y += g[u][r][1].y; g1.z += g[u][r][1].z; g1.w += g[u][r][1].w;
        }
        nvls_update8<kW, kDecay, kBroadcast, kNorm>(a, i, g0, g1, lr, wd, beta1, beta2, eps, step_size, bc2_sqrt, grad_scale, gacc);
      }
    }
  }
}

template <int kU, int kW>
__global__ void __launch_bounds__(256) adamw_nvls_kernel(const NvlsStep a) {
  __shared__ float s_part[8];
  __shared__ uint32_t s_epoch;
  __shared__ int s_abort;
  const int b = blockIdx.x, nb = gridDim.x;
  // ---- entry barrier: every rank's backward is complete, no rank still reads the previous shadow ----
  if (threadIdx.x == 0) {
    s_abort = 0;
    if (nvls_dead(a.err)) {
      s_abort = 1;
    } else {
      const uint32_t e = a.epoch[b];
      s_epoch = e;
      mc_signal(a.flags_mc + b);
      if (!wait_ge(a.flags + b, (e + 1u) * (uint32_t)a.world, a.spin_limit, a.err, 1)) s_abort = 1;
    }
  }
  __syncthreads();
  if (s_abort) return;                   // a peer never arrived: applying AdamW to partial sums would silently diverge the ranks
  const float lr = a.hyper[0], wd = a.hyper[1], beta1 = a.hyper[2], beta2 = a.hyper[3], eps = a.hyper[4], bc1 = a.hyper[5],
              bc2_sqrt = a.hyper[6], grad_scale = a.hyper[7];
  const float step_size = lr / bc1;
  float gacc = 0.f;
  const long tid = (long)b * blockDim.x + threadIdx.x, stride = (long)nb * blockDim.x;
  // ---- owned slice of the decay segment: reduce in the switch, update, broadcast the bf16 shadow ----
  const long shard = (a.n8_decay + a.world - 1) / a.world;
  const long lo = min((long)a.rank * shard, a.n8_decay), hi = min(lo + shard, a.n8_decay);
  nvls_segment<kU, kW, true, true, true>(a, lo, hi, tid, stride, lr, wd, beta1, beta2, eps, step_size, bc2_sqrt, grad_scale, gacc);
  // ---- no-decay segment: replicated (every rank reduces and updates all of it); rank 0 counts it in the norm ----
  if (a.rank == 0)
    nvls_segment<1, kW, false, false, true>(a, a.n8_decay, a.n8, tid, stride, lr, wd, beta1, beta2, eps, step_size, bc2_sqrt, grad_scale, gacc);
  else
    nvls_segment<1, kW, false, false, false>(a, a.n8_decay, a.n8, tid, stride, lr, wd, beta1, beta2, eps, step_size, bc2_sqrt, grad_scale, gacc);
  // ---- global gradient norm (utils.py:631-643): every rank's partial lands in every rank's accumulator ----
  gacc = warp_sum(gacc);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = gacc;
  __syncthreads();                       // also: every thread of the CTA has issued its multimem stores
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += s_part[w];
    if (a.gnorm_mc != nullptr) mc_red_add_f32(a.gnorm_mc, t);
    // ---- exit barrier: my loads of the peers' gradients and my stores into their shadows are done, and theirs into mine ----
    __threadfence_system();
    const uint32_t e = s_epoch;
    mc_signal(a.flags_mc + nb + b);
    wait_ge(a.flags + nb + b, (e + 1u) * (uint32_t)a.world, a.spin_limit, a.err, 2);
    a.epoch[b] = e + 1u;
  }
}

// ---- push variant -------------------------------------------------------------------------------------------------------
// NVLink moves posted writes at nearly twice the rate of read round trips (measured here: the pull kernel saturates at
// ~350 GB/s per direction whatever the queue depth, NCCL's write-based rings reach 520-670 GB/s).  So the reduce-scatter is
// done by PUSHING: phase A writes my gradients of every peer's slice into slot[my rank] of that peer's staging buffer; a
// grid-wide cross-GPU counter separates it from phase B, where the owner sums its own gradients and the N-1 staged copies
// (all local HBM reads, rank order => bitwise reproducible), runs AdamW and stores the bf16 shadow to every rank.
template <int kW>
__global__ void __launch_bounds__(256) adamw_push_kernel(const NvlsStep a) {
  __shared__ float s_part[8];
  __shared__ uint32_t s_epoch;
  __shared__ int s_abort;
  const int b = blockIdx.x, nb = gridDim.x;
  if (threadIdx.x == 0) {
    s_abort = 0;
    if (nvls_dead(a.err)) {
      s_abort = 1;
    } else {
      const uint32_t e = a.epoch[b];
      s_epoch = e;
      mc_signal(a.flags_mc + b);
      if (!wait_ge(a.flags + b, (e + 1u) * (uint32_t)kW, a.spin_limit, a.err, 1)) s_abort = 1;
    }
  }
  __syncthreads();
  if (s_abort) return;                   // void step: no scatter, no update (see wait_ge)
  const long tid = (long)b * blockDim.x + threadIdx.x, stride = (long)nb * blockDim.x;
  const long shard = (a.n8_decay + kW - 1) / kW;
  const float4* g_local = reinterpret_cast<const float4*>(a.g_peer[a.rank]);
  // ---- phase A: scatter my gradients to their owners (staggered start so that the N ranks hit N different peers) ----
  // prepushed: every rank's slices already sit in the owners' staging buffers — peer-to-peer copies on the copy engines, issued
  // range by range while backward was still running (ddp.NvlsShardedStep.range_ready) and stream-ordered before this launch, so
  // once the entry barrier has seen every rank's kernel start, every push has landed: no scatter, no mid barrier.
#pragma unroll 1
  for (int j = 1; j < (a.prepushed ? 1 : kW); ++j) {
    const int q = (a.rank + j) % kW;
    const long qlo = min((long)q * shard, a.n8_decay), qhi = min(qlo + shard, a.n8_decay);
    const float4* src = g_local + 2 * qlo;
    float4* dst = reinterpret_cast<float4*>(a.stage_peer[q]) + 2 * ((long)a.rank * shard);
    const long cnt = 2 * (qhi - qlo);
    for (long i = tid; i < cnt; i += 4 * stride) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (i + u * stride < cnt) v[u] = __ldcs(src + i + u * stride);
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (i + u * stride < cnt) dst[i + u * stride] = v[u];
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();
    mc_signal(a.mid_mc);               // always counted (the counter is monotone over launches), only waited for after a scatter
    if (!a.prepushed && !wait_ge(a.mid, (s_epoch + 1u) * (uint32_t)(kW * nb), a.spin_limit, a.err, 3)) s_abort = 1;
  }
  __syncthreads();
  if (s_abort) return;                   // some rank's gradients never arrived: leave p / m / v and the shadows alone
  // ---- phase B: reduce (local reads), AdamW on my slice, shadow to every rank ----
  const float lr = a.hyper[0], wd = a.hyper[1], beta1 = a.hyper[2], beta2 = a.hyper[3], eps = a.hyper[4], bc1 = a.hyper[5],
              bc2_sqrt = a.hyper[6], grad_scale = a.hyper[7];
  const float step_size = lr / bc1;
  float gacc = 0.f;
  const long lo = min((long)a.rank * shard, a.n8_decay), hi = min(lo + shard, a.n8_decay);
  const float4* stage = reinterpret_cast<const float4*>(a.stage_peer[a.rank]);
  for (long i = lo + tid; i < hi; i += stride) {
    float4 x[kW][2];
#pragma unroll
    for (int s = 0; s < kW; ++s) {
      const float4* src = (s == a.rank) ? g_local + 2 * i : stage + 2 * ((long)s * shard + (i - lo));
      x[s][0] = __ldcs(src);
      x[s][1] = __ldcs(src + 1);
    }
    float4 g0 = x[0][0], g1 = x[0][1];
#pragma unroll
    for (int s = 1; s < kW; ++s) {
      g0.x += x[s][0].x; g0.y += x[s][0].y; g0.z += x[s][0].z; g0.w += x[s][0].w;
      g1.x += x[s][1].x; g1.y += x[s][1].y; g1.z += x[s][1].z; g1.w += x[s][1].w;
    }
    nvls_update8<kW, true, true, true>(a, i, g0, g1, lr, wd, beta1, beta2, eps, step_size, bc2_sqrt, grad_scale, gacc);
  }
  // no-decay segment (tiny, replicated): pulled straight from the peers' gradient arenas
  if (a.rank == 0)
    nvls_segment<1, kW, false, false, true>(a, a.n8_decay, a.n8, tid, stride, lr, wd, beta1, beta2, eps, step_size, bc2_sqrt, grad_scale, gacc);
  else
    nvls_segment<1, kW, false, false, false>(a, a.n8_decay, a.n8, tid, stride, lr, wd, beta1, beta2, eps, step_size, bc2_sqrt, grad_scale, gacc);
  gacc = warp_sum(gacc);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = gacc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += s_part[w];
    if (a.gnorm_mc != nullptr) mc_red_add_f32(a.gnorm_mc, t);
    __threadfence_system();
    const uint32_t e = s_epoch;
    mc_signal(a.flags_mc + nb + b);
    wait_ge(a.flags + nb + b, (e + 1u) * (uint32_t)kW, a.spin_limit, a.err, 2);
    a.epoch[b] = e + 1u;
  }
}

// tuning knobs (read once): UB_NVLS_UNROLL = 8-gradient units per thread in flight (0 = pick: 4 multicast, 8/world P2P),
// UB_NVLS_CTAS = CTAs per SM, UB_NVLS_MODE = p2p | mc (gradient loads), UB_NVLS_MCST = 1: shadow stores through multicast
static int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e && *e ? atoi(e) : dflt;
}
static int nvls_unroll() { static int u = env_int("UB_NVLS_UNROLL", 0); return u; }
static int nvls_ctas_per_sm() { static int c = env_int("UB_NVLS_CTAS", 2); return c < 1 ? 1 : (c > 8 ? 8 : c); }
// UB_NVLS_MODE: push (default) | p2p (pull with peer loads) | mc (pull with multimem.ld_reduce)
static int nvls_mode() { static int m = [] { const char* e = getenv("UB_NVLS_MODE"); return !e || !*e ? 2 : (e[0] == 'm' ? 0 : (e[1] == '2' ? 1 : 2)); }(); return m; }
static bool nvls_mode_mc() { return nvls_mode() == 0; }
static int nvls_mc_store() { static int m = env_int("UB_NVLS_MCST", 0); return m; }   // measured equal at 8 GPUs, slower at 2
static int nvls_grid() { return sm_count() * nvls_ctas_per_sm(); }
constexpr int kNvlsMaxCtasPerSm = 8;

}  // namespace ub

using namespace ub;

extern "C" int ub_nvls_slots(void) { return 2 * sm_count() * kNvlsMaxCtasPerSm + 8; }   // entry | exit | mid counter (+pad)

extern "C" int ub_adamw_nvls(float* p, const float* g_mc, float* m, float* v, void* w16, void* w16_mc, int64_t n, int64_t n_decay,
                             int rank, int world, const float* hyper, float* gnorm_sq_mc, uint32_t* flags, uint32_t* flags_mc,
                             uint32_t* epoch, int32_t* err, const void* const* g_peers, void* const* w16_peers,
                             void* const* stage_peers, int prepushed, void* stream) {
  UB_REQUIRE(p && g_mc && m && v && w16 && w16_mc && hyper && flags && flags_mc && epoch && err, "adamw_nvls: null pointer");
  UB_REQUIRE(n > 0 && n % 8 == 0 && n_decay % 8 == 0 && n_decay >= 0 && n_decay <= n,
             "adamw_nvls: n=%lld and n_decay=%lld must be multiples of 8", (long long)n, (long long)n_decay);
  UB_REQUIRE(world >= 1 && rank >= 0 && rank < world, "adamw_nvls: rank %d of %d", rank, world);
  UB_REQUIRE((g_peers == nullptr) == (w16_peers == nullptr), "adamw_nvls: g_peers and w16_peers go together");
  NvlsStep a;
  a.p = p; a.g_mc = g_mc; a.m = m; a.v = v;
  a.w16 = (uint4*)w16; a.w16_mc = (uint4*)w16_mc;
  a.n8 = n / 8; a.n8_decay = n_decay / 8;
  a.rank = rank; a.world = world;
  a.hyper = hyper; a.gnorm_mc = gnorm_sq_mc;
  a.flags = flags; a.flags_mc = flags_mc; a.epoch = epoch; a.err = err;
  // UB_NVLS_SPIN_S (default 120 s of SM clocks at ~1.9 GHz): beyond any legitimate rank skew (a peer capturing its CUDA graph,
  // writing a checkpoint, a loader hiccup); past it the step is declared void on this rank (see wait_ge / nvls_dead)
  static const long long spin_clocks = (long long)(env_int("UB_NVLS_SPIN_S", 120) > 0 ? env_int("UB_NVLS_SPIN_S", 120) : 120) * 1900000000LL;
  a.spin_limit = spin_clocks;
  const bool p2p = g_peers != nullptr && !nvls_mode_mc() && (world == 2 || world == 4 || world == 8);
  for (int r = 0; r < 8; ++r) {
    a.g_peer[r] = p2p && r < world ? (const float*)g_peers[r] : nullptr;
    a.w16_peer[r] = p2p && r < world ? (uint4*)w16_peers[r] : nullptr;
    UB_REQUIRE(!p2p || r >= world || (a.g_peer[r] && a.w16_peer[r]), "adamw_nvls: null peer pointer for rank %d", r);
  }
  a.mc_store = nvls_mc_store();
  int grid = nvls_grid();
  cudaStream_t st = (cudaStream_t)stream;
  int u = nvls_unroll();
  const bool push = p2p && stage_peers != nullptr && nvls_mode() == 2;
  const int slots_half = sm_count() * kNvlsMaxCtasPerSm;
  for (int r = 0; r < 8; ++r) a.stage_peer[r] = push && r < world ? (float*)stage_peers[r] : nullptr;
  UB_REQUIRE(!prepushed || push, "adamw_nvls: prepushed needs the push form (stage_peers, world 2 / 4 / 8, UB_NVLS_MODE=push)");
  a.prepushed = prepushed ? 1 : 0;
  a.mid = flags + 2 * slots_half;                       // one counter right behind the entry / exit slots
  a.mid_mc = flags_mc + 2 * slots_half;
  if (push) {
    // the mid barrier is grid-wide: every CTA must be resident
    int occ = 0;
    const void* fn = world == 2 ? (const void*)adamw_push_kernel<2> : world == 4 ? (const void*)adamw_push_kernel<4> : (const void*)adamw_push_kernel<8>;
    UB_REQUIRE(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, 256, 0) == cudaSuccess && occ >= 1, "adamw_nvls: occupancy query failed");
    if (grid > occ * sm_count()) grid = occ * sm_count();
    if (world == 2) UB_LAUNCH((adamw_push_kernel<2>), grid, 256, 0, st, a);
    else if (world == 4) UB_LAUNCH((adamw_push_kernel<4>), grid, 256, 0, st, a);
    else UB_LAUNCH((adamw_push_kernel<8>), grid, 256, 0, st, a);
    return check_launch("adamw_push_kernel");
  }
  if (!p2p) {
    if (u == 1) UB_LAUNCH((adamw_nvls_kernel<1, 0>), grid, 256, 0, st, a);
    else if (u == 2) UB_LAUNCH((adamw_nvls_kernel<2, 0>), grid, 256, 0, st, a);
    else UB_LAUNCH((adamw_nvls_kernel<4, 0>), grid, 256, 0, st, a);
  } else if (world == 2) {
    if (u == 1) UB_LAUNCH((adamw_nvls_kernel<1, 2>), grid, 256, 0, st, a);
    else if (u == 2) UB_LAUNCH((adamw_nvls_kernel<2, 2>), grid, 256, 0, st, a);
    else UB_LAUNCH((adamw_nvls_kernel<4, 2>), grid, 256, 0, st, a);
  } else if (world == 4) {
    if (u == 1) UB_LAUNCH((adamw_nvls_kernel<1, 4>), grid, 256, 0, st, a);
    else UB_LAUNCH((adamw_nvls_kernel<2, 4>), grid, 256, 0, st, a);
  } else {
    if (u == 2) UB_LAUNCH((adamw_nvls_kernel<2, 8>), grid, 256, 0, st, a);
    else UB_LAUNCH((adamw_nvls_kernel<1, 8>), grid, 256, 0, st, a);
  }
  return check_launch("adamw_nvls_kernel");
}
