// tcgen05 / TMEM attention for LONG sequences (head_dim 64, any S): forward with log-sum-exp and a two-pass backward.
//
// Replaces   modeling_finetune.py:100-119 (Attention.forward and its autograd backward) on the ALL-TOKEN passes — stage 2
//            (S = 1568, engine_for_finetuning.py:37-40), the stage-3 full-token passes (run_stage3.py:475-483) and BASELINE
//            configs[4]'s attention-dominated sizing — where attention_fwd_lse_tc.cu / attention_bwd_tc.cu (S <= 320, whole
//            item resident in smem / TMEM) do not apply.  The mma.sync kernels of attention.cu remain only as a debug fallback.
//
// One kernel template, three modes.  A work unit is a PAIR of 128-row "stationary" tiles of one (sequence, head); warpgroup g owns
// tile 2*pair+g, and both warpgroups consume the same ring of "streamed" chunks, so every chunk is fetched once per pair:
//   FWD   stationary Q tile            streamed (K, V) chunks of 64 keys      S = Q K^T -> online softmax -> O += P V, l += P 1
//   DQ    stationary (Q, dO) tile      streamed (K, V) chunks of 32 keys      S = Q K^T, dP = dO V^T, dS = P o (dP - D) -> dQ += dS K
//   DKV   stationary (K, V) tile       streamed (Q, dO) chunks of 32 queries  S^T = K Q^T, dP^T = V dO^T -> dV += P^T dO, dK += dS^T Q
// Every warpgroup has TWO score sets in TMEM: the scores of chunk n+1 are computed while chunk n is in the softmax threads, so a
// warpgroup's cycle is load + exponentials + store only.  The stationary tiles are double-buffered too (the next unit's tiles
// land during the current unit), so units follow each other without a refill bubble.
// P / dS are written back to TMEM as bf16 over the scores and feed the second product as its A operand (tcgen05.mma TS form);
// accumulators stay in TMEM for the whole unit, so nothing but the streamed chunks moves during the inner loop.  The backward
// runs as two passes (DKV then DQ), each with a single writer per output element — a one-pass scheme would have to reduce dQ (or
// dK / dV) across CTAs with fp32 atomics, ~5 MB per (sequence, head) at S = 1568, which costs more than recomputing S and dP.
//   warp 0      TMA producer (stationary tiles, streamed ring)          warp 3   DKV: per-chunk log-sum-exp / D loader
//   warps 1, 2  tcgen05.mma issue streams of warpgroup 0 / 1            warps 4-7 / 8-11   softmax / gradient warpgroups 0 / 1
// TMEM (256 columns per warpgroup): two score sets at [0,64) and [64,128) — FWD: S|P (64 keys); DQ / DKV: S [0,32) | dP [32,64) with
//                                    P / dS written over their first 16 columns — then the accumulators: FWD O [128,192) l [192,208);
//                                    DQ dQ [128,192); DKV dV [128,192) dK [192,256).
// FWD softmax reference: the row maximum of the first chunk, moved only when a later chunk exceeds it by more than 2^40 (O and l
// are then rescaled in TMEM) — O / l is invariant under the common factor, so the result is exact and O is normally never touched.
#include "common.cuh"
#include <cstdlib>
#include "../../include/unite_b200.h"

namespace ub {

int make_tmap_3d_bf16(CUtensorMap* out, const void* base, int64_t d2, int64_t d1, int64_t d0, int64_t stride1_elems,
                      int64_t stride2_elems, int box0, int box1);

constexpr int AL_THREADS = 384;
enum { AL_FWD = 0, AL_DQ = 1, AL_DKV = 2 };

template <int MODE>
struct ALC {
  static constexpr int NC = MODE == AL_FWD ? 64 : 32;         // streamed rows per chunk
  static constexpr int NSTG = MODE == AL_FWD ? 5 : 6;         // ring depth
  static constexpr int STAGE_BYTES = 2 * NC * 128;            // two operands of [NC rows][64 bf16]
  static constexpr int STAT_OPS = MODE == AL_FWD ? 1 : 2;     // stationary operands per warpgroup
  static constexpr int STAT_WG = STAT_OPS * 16384;            // one stationary tile set
  static constexpr int STAT = 0;                               // [2 buffers][2 warpgroups][STAT_OPS][128 rows][64 bf16]
  static constexpr int RING = 4 * STAT_WG;
  static constexpr int OUT = RING + NSTG * STAGE_BYTES;        // 8 warps x 4 KB output staging
  static constexpr int ONES = OUT + 32768;                     // [16][64] bf16 ones (FWD row sums)
  static constexpr int LD = ONES + (MODE == AL_FWD ? 2048 : 0);   // [NSTG][L: NC | D: NC] fp32 (DKV)
  static constexpr int BAR = LD + (MODE == AL_DKV ? NSTG * 256 : 0);
  static constexpr int NBAR = 3 * NSTG + 22;
  static constexpr int SMEM = BAR + NBAR * 8 + 16;
  static_assert(SMEM <= 232448, "exceeds the 227 KB per-CTA shared memory limit");
};

struct AttnLongParams {
  float* lse_out;        // FWD: [n_seq, H, S] or null
  const float* lse;      // DQ / DKV
  const float* Dv;       // DQ / DKV: rowsum(dO o O)
  float* dbias;          // DQ / DKV, optional fp32 [3*H*64]: += column sums of the dq / dv written (q_bias / v_bias gradients)
  int n_seq, S, H;
  int ntile, npair, nchunk;
  float sl2, scale;
};

template <int MODE>
__global__ void __launch_bounds__(AL_THREADS, 1)
attn_long_tc_kernel(const __grid_constant__ CUtensorMap tmStat, const __grid_constant__ CUtensorMap tmStatDO,
                    const __grid_constant__ CUtensorMap tmStrm, const __grid_constant__ CUtensorMap tmStrmDO,
                    const __grid_constant__ CUtensorMap tmOut, const AttnLongParams p) {
  using C = ALC<MODE>;
  constexpr int NC = C::NC, NSTG = C::NSTG;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::BAR);
  uint64_t* ring_full = bars;                  // [NSTG]
  uint64_t* ring_empty = bars + NSTG;          // [NSTG] both warpgroups' products of the chunk have completed
  uint64_t* ld_full = bars + 2 * NSTG;         // [NSTG] DKV: log-sum-exp / D of the chunk's queries are in smem
  uint64_t* stat_full = bars + 3 * NSTG;       // [2 warpgroups][2 buffers]
  uint64_t* stat_empty = stat_full + 4;        // [2][2] every MMA of the unit has read the stationary tile
  uint64_t* s_full = stat_full + 8;            // [2 warpgroups][2 score sets] scores of the chunk are in TMEM
  uint64_t* p_ready = stat_full + 12;          // [2][2] P / dS written back (4 warps)
  uint64_t* acc_full = stat_full + 16;         // [2] accumulators of the unit are final
  uint64_t* acc_free = stat_full + 18;         // [2] ... and have been read out (4 warps)
  uint64_t* pv_done = stat_full + 20;          // [2] FWD: products of the chunk completed (slow path only)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(stat_full + 22);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    tma_prefetch_desc(&tmStat);
    tma_prefetch_desc(&tmStrm);
    tma_prefetch_desc(&tmOut);
    if (MODE != AL_FWD) {
      tma_prefetch_desc(&tmStatDO);
      tma_prefetch_desc(&tmStrmDO);
    }
    for (int i = 0; i < NSTG; ++i) {
      mbar_init(&ring_full[i], 1);
      mbar_init(&ring_empty[i], 2);
      mbar_init(&ld_full[i], 1);
    }
    for (int i = 0; i < 4; ++i) {
      mbar_init(&stat_full[i], 1);
      mbar_init(&stat_empty[i], 1);
      mbar_init(&s_full[i], 1);
      mbar_init(&p_ready[i], 4);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_free[i], 4);
      mbar_init(&pv_done[i], 1);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  if (MODE == AL_FWD) {
    for (int i = threadIdx.x; i < 2048 / 16; i += blockDim.x)
      reinterpret_cast<uint4*>(smem + C::ONES)[i] = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int n_units = p.n_seq * p.H * p.npair;
  const int nchunk = p.nchunk;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp == 0) {
      // ------------------------------------------------------------------------------------------ TMA producer
      if (lane == 0) {
        uint32_t ci = 0;
        int ui = 0;
        for (int u = blockIdx.x; u < n_units; u += gridDim.x, ++ui) {
          const int item = u / p.npair, pair = u % p.npair, seq = item / p.H, h = item % p.H;
          const int sb = ui & 1;                                     // stationary buffer of this unit (the next unit's tiles
          for (int g = 0; g < 2; ++g) {                              // land while this one is still being consumed)
            const int t = min(2 * pair + g, p.ntile - 1);          // an odd tile count: warpgroup 1 repeats the last tile (not stored)
            uint8_t* dst = smem + C::STAT + (sb * 2 + g) * C::STAT_WG;
            uint64_t* fb = &stat_full[g * 2 + sb];
            mbar_wait(&stat_empty[g * 2 + sb], (uint32_t)((ui >> 1) & 1) ^ 1u);
            mbar_expect_tx(fb, C::STAT_WG);
            if (MODE == AL_FWD) {
              tma_load_3d(&tmStat, fb, dst, h * 64, t * 128, seq);
            } else if (MODE == AL_DQ) {
              tma_load_3d(&tmStat, fb, dst, h * 64, t * 128, seq);
              tma_load_3d(&tmStatDO, fb, dst + 16384, h * 64, t * 128, seq);
            } else {
              tma_load_3d(&tmStat, fb, dst, (p.H + h) * 64, t * 128, seq);
              tma_load_3d(&tmStat, fb, dst + 16384, (2 * p.H + h) * 64, t * 128, seq);
            }
          }
          for (int c = 0; c < nchunk; ++c, ++ci) {
            const uint32_t stage = ci % NSTG, ph = (ci / NSTG) & 1u;
            uint8_t* dst = smem + C::RING + stage * C::STAGE_BYTES;
            mbar_wait(&ring_empty[stage], ph ^ 1u);
            mbar_expect_tx(&ring_full[stage], C::STAGE_BYTES);
            if (MODE == AL_DKV) {
              tma_load_3d(&tmStrm, &ring_full[stage], dst, h * 64, c * NC, seq);
              tma_load_3d(&tmStrmDO, &ring_full[stage], dst + NC * 128, h * 64, c * NC, seq);
            } else {
              tma_load_3d(&tmStrm, &ring_full[stage], dst, (p.H + h) * 64, c * NC, seq);
              tma_load_3d(&tmStrm, &ring_full[stage], dst + NC * 128, (2 * p.H + h) * 64, c * NC, seq);
            }
          }
        }
      }
    } else if (warp <= 2) {
      // ------------------------------------------------------------------------------------------ MMA issue stream of warpgroup g
      const uint32_t g = (uint32_t)(warp - 1);
      constexpr uint32_t IDESC_S = umma_idesc_bf16(128, NC, 0, 0);     // scores: both operands K-major
      constexpr uint32_t IDESC_T = umma_idesc_bf16(128, 64, 0, 1);     // second product: A in TMEM, B MN-major
      constexpr uint32_t IDESC_R = umma_idesc_bf16(128, 16, 0, 0);     // FWD row sums: B = ones, K-major
      constexpr uint32_t HI = (1024u >> 4) | (1u << 14) | (2u << 29);
      constexpr uint32_t LO_K = 1u << 16, LO_MN = (8192u >> 4) << 16;
      const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0) + g * 256u;
      const uint32_t aStat = (smem_u32(smem + C::STAT) & 0x3FFFFu) >> 4;
      const uint32_t aRing = (smem_u32(smem + C::RING) & 0x3FFFFu) >> 4, aOnes = (smem_u32(smem + C::ONES) & 0x3FFFFu) >> 4;
      uint32_t ci = 0;                         // chunks consumed by this warpgroup; chunk n uses score set n & 1
      uint32_t si = 0;                         // score MMAs issued (runs up to two chunks ahead of ci)
      int ui = 0;
      for (int u = blockIdx.x; u < n_units; u += gridDim.x, ++ui) {
        const uint32_t sb = (uint32_t)(ui & 1);
        const uint32_t aS0 = aStat + (sb * 2u + g) * (uint32_t)(C::STAT_WG >> 4), aS1 = aS0 + 1024u;
        mbar_wait(&stat_full[g * 2 + sb], (uint32_t)((ui >> 1) & 1));
        // scores of the next chunk into set (si & 1): S = stat0 x strm0^T (and dP = stat1 x strm1^T)
        auto issue_scores = [&]() {
          const uint32_t stage = si % NSTG, set = si & 1u;
          const uint32_t a0 = aRing + stage * (uint32_t)(C::STAGE_BYTES >> 4), a1 = a0 + (uint32_t)((NC * 128) >> 4);
          mbar_wait(&ring_full[stage], (si / NSTG) & 1u);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t d = tb + set * 64u;
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_ss_lo(d, aS0 + LO_K + k * 2, HI, a0 + LO_K + k * 2, HI, IDESC_S, k > 0);
            if (MODE != AL_FWD) {
#pragma unroll
              for (int k = 0; k < 4; ++k) umma_ss_lo(d + 32, aS1 + LO_K + k * 2, HI, a1 + LO_K + k * 2, HI, IDESC_S, k > 0);
            }
            umma_commit(&s_full[g * 2 + set]);
          }
          __syncwarp();
          ++si;
        };
        issue_scores();
        if (nchunk > 1) issue_scores();
        for (int c = 0; c < nchunk; ++c, ++ci) {
          const uint32_t stage = ci % NSTG, set = ci & 1u;
          const uint32_t a0 = aRing + stage * (uint32_t)(C::STAGE_BYTES >> 4), a1 = a0 + (uint32_t)((NC * 128) >> 4);
          mbar_wait(&p_ready[g * 2 + set], (ci >> 1) & 1u);
          if (c == 0) mbar_wait(&acc_free[g], (uint32_t)(ui & 1) ^ 1u);      // the previous unit's accumulators have been read out
          tc_fence_after();
          if (elect_one()) {
            const bool acc = c > 0;
            const uint32_t tS = tb + set * 64u;
            if (MODE == AL_FWD) {
#pragma unroll
              for (int k = 0; k < NC / 16; ++k) umma_ts_lo(tb + 128, tS + k * 8, a1 + LO_MN + k * 128, HI, IDESC_T, acc || k > 0);
#pragma unroll
              for (int k = 0; k < NC / 16; ++k) umma_ts_lo(tb + 192, tS + k * 8, aOnes + LO_K, HI, IDESC_R, acc || k > 0);
              umma_commit(&pv_done[g]);
            } else if (MODE == AL_DQ) {
#pragma unroll
              for (int k = 0; k < NC / 16; ++k) umma_ts_lo(tb + 128, tS + 32 + k * 8, a0 + LO_MN + k * 128, HI, IDESC_T, acc || k > 0);
            } else {
#pragma unroll
              for (int k = 0; k < NC / 16; ++k) umma_ts_lo(tb + 128, tS + k * 8, a1 + LO_MN + k * 128, HI, IDESC_T, acc || k > 0);
#pragma unroll
              for (int k = 0; k < NC / 16; ++k) umma_ts_lo(tb + 192, tS + 32 + k * 8, a0 + LO_MN + k * 128, HI, IDESC_T, acc || k > 0);
            }
            umma_commit(&ring_empty[stage]);
            if (c == nchunk - 1) {
              umma_commit(&acc_full[g]);
              umma_commit(&stat_empty[g * 2 + sb]);
            }
          }
          __syncwarp();
          if (c + 2 < nchunk) issue_scores();     // into the set whose P / dS the products above have just consumed (in issue order)
        }
      }
    } else if (MODE == AL_DKV) {
      // ------------------------------------------------------------------------------------------ log-sum-exp / D loader (warp 3)
      uint32_t ci = 0;
      for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
        const int item = u / p.npair;
        const float* gL = p.lse + (int64_t)item * p.S;
        const float* gD = p.Dv + (int64_t)item * p.S;
        for (int c = 0; c < nchunk; ++c, ++ci) {
          const uint32_t stage = ci % NSTG, ph = (ci / NSTG) & 1u;
          mbar_wait(&ring_empty[stage], ph ^ 1u);
          float* sL = reinterpret_cast<float*>(smem + C::LD + stage * 256);
          {
            const int q = c * NC + lane;                                           // NC == 32: one query per lane
            sL[lane] = q < p.S ? __ldg(gL + q) * 1.4426950408889634f : INFINITY;   // +inf -> P = 0 for padded queries
            sL[NC + lane] = q < p.S ? __ldg(gD + q) : 0.f;
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&ld_full[stage]);
        }
      }
    }
  } else {
    // ------------------------------------------------------------------------------------------ softmax / gradient warpgroups
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    const uint32_t g = (uint32_t)((warp - 4) >> 2);
    const int sp = warp & 3;
    const uint32_t t_row = tmem_base + ((uint32_t)(sp * 32) << 16) + g * 256u;
    uint8_t* stg = smem + C::OUT + (warp - 4) * 4096;
    const uint32_t stg_a = smem_u32(stg);
    const uint32_t sw = (uint32_t)(lane & 7);
    const float sl2 = p.sl2;
    // TMEM (32 rows x 64 fp32 columns at t_src) -> * mul -> bf16 -> swizzled slab -> TMA store at (col, row, seq)
    auto store_tile = [&](uint32_t t_src, float mul, int col, int row, int seq, bool active, float* bias_dst) {
      if (lane == 0) tma_store_wait_read<0>();
      __syncwarp();
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        uint32_t r[32];
        tmem_ld_32x32(t_src + hh * 32, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint32_t a = stg_a + (uint32_t)lane * 128u + ((((uint32_t)(hh * 4 + j)) ^ sw) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a),
                       "r"(pack_bf16x2(__uint_as_float(r[8 * j]) * mul, __uint_as_float(r[8 * j + 1]) * mul)),
                       "r"(pack_bf16x2(__uint_as_float(r[8 * j + 2]) * mul, __uint_as_float(r[8 * j + 3]) * mul)),
                       "r"(pack_bf16x2(__uint_as_float(r[8 * j + 4]) * mul, __uint_as_float(r[8 * j + 5]) * mul)),
                       "r"(pack_bf16x2(__uint_as_float(r[8 * j + 6]) * mul, __uint_as_float(r[8 * j + 7]) * mul))
                       : "memory");
        }
      }
      tc_fence_before();
      fence_proxy_async();
      __syncwarp();
      if (lane == 0 && active && row < p.S) {
        tma_store_3d(&tmOut, stg, col, row, seq);
        tma_store_commit();
      }
      if (bias_dst != nullptr && active) {
        // bias gradient of these 64 columns = column sums of the bf16 slab just written.  Rows past the sequence end are exact
        // zeros in the DKV pass (zero-filled K / V rows give zero dK / dV rows only if P^T is zero there: it is not — so those
        // rows are masked here) and in the DQ pass (zero Q / dO rows: dS row = P (0 - 0) = 0).
        float c0 = 0.f, c1 = 0.f;
        const uint32_t chunk = (uint32_t)(lane >> 2), within = (uint32_t)(lane & 3) * 4u;
        const int valid = min(32, p.S - row);
#pragma unroll 8
        for (int r = 0; r < 32; ++r) {
          uint32_t u;
          asm volatile("ld.shared.b32 %0, [%1];" : "=r"(u) : "r"(stg_a + (uint32_t)r * 128u + ((chunk ^ (uint32_t)(r & 7)) << 4) + within));
          const float2 f = unpack_bf16x2(u);
          if (r < valid) { c0 += f.x; c1 += f.y; }
        }
        atomicAdd(bias_dst + 2 * lane, c0);
        atomicAdd(bias_dst + 2 * lane + 1, c1);
      }
    };
    // The TMEM read port (64 B/clk/SM) bounds every mode (4 B of scores per (query, key) pair forward, 8 B backward); what
    // mattered was taking the score MMAs off each warpgroup's critical path (two score sets, issued one chunk ahead).
    uint32_t ci = 0;
    int ui = 0;
    for (int u = blockIdx.x; u < n_units; u += gridDim.x, ++ui) {
      const int item = u / p.npair, pair = u % p.npair, seq = item / p.H, h = item % p.H;
      const int t_raw = 2 * pair + (int)g;
      const bool active = t_raw < p.ntile;
      const int t = min(t_raw, p.ntile - 1);
      const int row = t * 128 + sp * 32 + lane;             // stationary row of this thread
      float ref = 0.f;                                      // FWD: reference maximum (raw score units)
      float l2 = 0.f, dd = 0.f;                             // DQ: log-sum-exp * log2e and D of this query row
      if (MODE == AL_DQ && row < p.S) {
        l2 = __ldg(p.lse + (int64_t)item * p.S + row) * 1.4426950408889634f;
        dd = __ldg(p.Dv + (int64_t)item * p.S + row);
      }
      for (int c = 0; c < nchunk; ++c, ++ci) {
        const uint32_t stage = ci % NSTG, set = ci & 1u;
        const uint32_t t_set = t_row + set * 64u;
        mbar_wait(&s_full[g * 2 + set], (ci >> 1) & 1u);
        tc_fence_after();
        if (MODE == AL_FWD) {
          const int kvalid = min(NC, p.S - c * NC);
          uint32_t sv[NC];
#pragma unroll
          for (int q = 0; q < NC / 32; ++q) tmem_ld_32x32(t_set + q * 32, *reinterpret_cast<uint32_t(*)[32]>(&sv[q * 32]));
          tmem_ld_wait();
          float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
          if (kvalid == NC) {
#pragma unroll
            for (int i = 0; i < NC; ++i) m4[i & 3] = fmaxf(m4[i & 3], __uint_as_float(sv[i]));
          } else {
#pragma unroll
            for (int i = 0; i < NC; ++i)
              if (i < kvalid) m4[i & 3] = fmaxf(m4[i & 3], __uint_as_float(sv[i]));
          }
          const float mx = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
          if (c == 0) {
            ref = mx;
          } else if (__any_sync(0xffffffffu, (mx - ref) * sl2 > 40.0f)) {
            // slow path: move the reference of this warp's rows; O and l of the earlier chunks sit in TMEM scaled by 2^(-ref)
            mbar_wait(&pv_done[g], (ci - 1u) & 1u);
            tc_fence_after();
            const float nref = fmaxf(ref, mx);
            const float alpha = fast_exp2((ref - nref) * sl2);
            uint32_t r[32];
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              tmem_ld_32x32(t_row + 128 + hh * 32, r);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * alpha);
              tmem_st_32x16(t_row + 128 + hh * 32, *reinterpret_cast<uint32_t(*)[16]>(&r[0]));
              tmem_st_32x16(t_row + 128 + hh * 32 + 16, *reinterpret_cast<uint32_t(*)[16]>(&r[16]));
            }
            uint32_t l16[16];
            tmem_ld_32x16(t_row + 192, l16);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) l16[i] = __float_as_uint(__uint_as_float(l16[i]) * alpha);
            tmem_st_32x16(t_row + 192, l16);
            tmem_st_wait();
            ref = nref;
          }
          const float mb = ref * sl2;
#pragma unroll
          for (int q = 0; q < NC / 32; ++q) {
            uint32_t pk[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int k0 = q * 32 + 2 * i;
              float p0 = fast_exp2(fmaf(__uint_as_float(sv[k0]), sl2, -mb));
              float p1 = fast_exp2(fmaf(__uint_as_float(sv[k0 + 1]), sl2, -mb));
              if (kvalid != NC) {
                if (k0 >= kvalid) p0 = 0.f;
                if (k0 + 1 >= kvalid) p1 = 0.f;
              }
              pk[i] = pack_bf16x2(p0, p1);
            }
            tmem_st_32x16(t_set + q * 16, pk);
          }
        } else {
          // set = {S [0,32) | dP [32,64)}; P / dS (bf16, 16 columns each) are written over the first half of S / dP
          uint32_t sv[32], dv[32];
          if (MODE == AL_DKV) mbar_wait(&ld_full[stage], (ci / NSTG) & 1u);
          tmem_ld_32x32(t_set, sv);
          tmem_ld_32x32(t_set + 32, dv);
          tmem_ld_wait();
          uint32_t pk[16], dk[16];
          if (MODE == AL_DQ) {
            const int kvalid = min(NC, p.S - c * NC);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float p0 = fast_exp2(fmaf(__uint_as_float(sv[2 * i]), sl2, -l2));
              const float p1 = fast_exp2(fmaf(__uint_as_float(sv[2 * i + 1]), sl2, -l2));
              float d0 = p0 * (__uint_as_float(dv[2 * i]) - dd), d1 = p1 * (__uint_as_float(dv[2 * i + 1]) - dd);
              if (kvalid != NC) {
                if (2 * i >= kvalid) d0 = 0.f;
                if (2 * i + 1 >= kvalid) d1 = 0.f;
              }
              dk[i] = pack_bf16x2(d0, d1);
            }
            tmem_st_32x16(t_set + 32, dk);
          } else {
            const float4* L4 = reinterpret_cast<const float4*>(smem + C::LD + stage * 256);
            const float4* D4 = L4 + NC / 4;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 l = L4[i], d = D4[i];
              const float p0 = fast_exp2(fmaf(__uint_as_float(sv[4 * i]), sl2, -l.x));
              const float p1 = fast_exp2(fmaf(__uint_as_float(sv[4 * i + 1]), sl2, -l.y));
              const float p2 = fast_exp2(fmaf(__uint_as_float(sv[4 * i + 2]), sl2, -l.z));
              const float p3 = fast_exp2(fmaf(__uint_as_float(sv[4 * i + 3]), sl2, -l.w));
              pk[2 * i] = pack_bf16x2(p0, p1);
              pk[2 * i + 1] = pack_bf16x2(p2, p3);
              dk[2 * i] = pack_bf16x2(p0 * (__uint_as_float(dv[4 * i]) - d.x), p1 * (__uint_as_float(dv[4 * i + 1]) - d.y));
              dk[2 * i + 1] = pack_bf16x2(p2 * (__uint_as_float(dv[4 * i + 2]) - d.z), p3 * (__uint_as_float(dv[4 * i + 3]) - d.w));
            }
            tmem_st_32x16(t_set, pk);
            tmem_st_32x16(t_set + 32, dk);
          }
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&p_ready[g * 2 + set]);
      }
      // ---- accumulators of the unit -> global
      mbar_wait(&acc_full[g], (uint32_t)(ui & 1));
      tc_fence_after();
      const int row0 = t * 128 + sp * 32;
      if (MODE == AL_FWD) {
        uint32_t lsum;
        tmem_ld_32x1(t_row + 192, lsum);
        tmem_ld_wait();
        const float l = __uint_as_float(lsum);
        if (p.lse_out != nullptr && active && row < p.S) p.lse_out[(int64_t)item * p.S + row] = ref * p.scale + __logf(l);
        store_tile(t_row + 128, 1.0f / l, h * 64, row0, seq, active, nullptr);
      } else if (MODE == AL_DQ) {
        store_tile(t_row + 128, p.scale, h * 64, row0, seq, active, p.dbias ? p.dbias + h * 64 : nullptr);
      } else {
        store_tile(t_row + 128, 1.0f, (2 * p.H + h) * 64, row0, seq, active, p.dbias ? p.dbias + (2 * p.H + h) * 64 : nullptr);
        store_tile(t_row + 192, p.scale, (p.H + h) * 64, row0, seq, active, nullptr);
      }
      if (lane == 0) mbar_arrive(&acc_free[g]);
    }
    if (lane == 0) tma_store_wait_read<0>();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <int MODE>
static int launch_attn_long(const void* qkv, const void* d_o, void* out, float* lse_out, const float* lse, const float* Dv, float* dbias,
                            int n_seq, int S, int H, float scale, cudaStream_t stream) {
  using C = ALC<MODE>;
  AttnLongParams p;
  p.lse_out = lse_out; p.lse = lse; p.Dv = Dv; p.dbias = dbias;
  p.n_seq = n_seq; p.S = S; p.H = H;
  p.ntile = (S + 127) / 128;
  p.npair = (p.ntile + 1) / 2;
  p.nchunk = (S + C::NC - 1) / C::NC;
  p.scale = scale;
  p.sl2 = scale * 1.4426950408889634f;
  CUtensorMap tstat, tstat_do, tstrm, tstrm_do, tout;
  const int64_t ld = 3 * (int64_t)H * 64, ldo = (int64_t)H * 64;
  if (make_tmap_3d_bf16(&tstat, qkv, n_seq, S, ld, ld, (int64_t)S * ld, 64, 128)) return 1;
  if (make_tmap_3d_bf16(&tstrm, qkv, n_seq, S, ld, ld, (int64_t)S * ld, 64, C::NC)) return 1;
  tstat_do = tstat;
  tstrm_do = tstrm;
  if (MODE != AL_FWD) {
    if (make_tmap_3d_bf16(&tstat_do, d_o, n_seq, S, ldo, ldo, (int64_t)S * ldo, 64, 128)) return 1;
    if (make_tmap_3d_bf16(&tstrm_do, d_o, n_seq, S, ldo, ldo, (int64_t)S * ldo, 64, C::NC)) return 1;
    if (make_tmap_3d_bf16(&tout, out, n_seq, S, ld, ld, (int64_t)S * ld, 64, 32)) return 1;
  } else {
    if (make_tmap_3d_bf16(&tout, out, n_seq, S, ldo, ldo, (int64_t)S * ldo, 64, 32)) return 1;
  }
  static bool configured = false;
  auto kern = attn_long_tc_kernel<MODE>;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM);
    UB_REQUIRE(e == cudaSuccess, "cudaFuncSetAttribute(attn_long_tc mode %d smem=%d): %s", MODE, C::SMEM, cudaGetErrorString(e));
    configured = true;
  }
  const long units = (long)n_seq * H * p.npair;
  const int grid = (int)(units < sm_count() ? units : sm_count());
  UB_LAUNCH(kern, grid, AL_THREADS, C::SMEM, stream, tstat, tstat_do, tstrm, tstrm_do, tout, p);
  return check_launch("attn_long_tc_kernel");
}

int launch_attn_fwd_long_tc(const void* qkv, void* o, float* lse, int n_seq, int S, int H, float scale, cudaStream_t stream) {
  return launch_attn_long<AL_FWD>(qkv, nullptr, o, lse, nullptr, nullptr, nullptr, n_seq, S, H, scale, stream);
}

// D = rowsum(dO o O) is produced by attn_bwd_prep_kernel (attention.cu) before this call
int launch_attn_bwd_long_tc(const void* qkv, const void* d_o, const float* lse, const float* Dv, void* dqkv, float* dbias, int n_seq, int S,
                            int H, float scale, cudaStream_t stream) {
  if (launch_attn_long<AL_DKV>(qkv, d_o, dqkv, nullptr, lse, Dv, dbias, n_seq, S, H, scale, stream)) return 1;
  return launch_attn_long<AL_DQ>(qkv, d_o, dqkv, nullptr, lse, Dv, dbias, n_seq, S, H, scale, stream);
}

}  // namespace ub
