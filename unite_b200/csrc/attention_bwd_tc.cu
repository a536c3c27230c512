// tcgen05 / TMEM attention BACKWARD for sequences of up to 320 tokens (head_dim 64): the student's visible-token
// attention (modeling_finetune.py:100-119 under autograd; 12 layers x 384 (clip, head) pairs per step at S = 320).
//
// One persistent CTA per SM walks (sequence, head) items.  Everything is computed in the TRANSPOSED orientation so that
// the per-key reductions (dK, dV) read their A operand straight from TMEM and nothing but dS^T ever touches smem:
//     S^T  = K  Q^T              (SS, M = 128 keys, N = 32 queries, K = 64)       -> TMEM
//     dP^T = V  dO^T             (SS, same shape)                                 -> TMEM
//     P^T  = exp2(S^T * scale*log2e - LSE[q]),  dS^T = P^T o (dP^T - D[q])        (one thread per KEY row)
//     dV  += P^T  dO             (TS: A = P^T bf16 in TMEM over S^T, B = dO MN-major)
//     dK  += dS^T Q              (TS: A = dS^T bf16 in TMEM over dP^T, B = Q MN-major)
//     dQ  += dS   K              (SS: A = dS^T staged in smem and read MN-major, B = K MN-major; M = 128 queries)
// S and dP are recomputed ONCE per (key, query) pair (the mma.sync fallback in attention.cu needs two passes), and the
// five products run on the tensor pipe while the two softmax warpgroups alternate on the TMEM read port, which is what
// bounds this kernel (8 bytes of fp32 scores per pair at ~64 B/clk/SM).
//   warp 0        TMA producer: Q and dO of the item (64-row boxes), K/V tiles in a 2-slot ring (prefetches the next item)
//   warp 1        tcgen05.mma issuer (one thread), S/dP of chunk n+2 issued behind the TS products of chunk n
//   warp 2        loads LSE * log2e and D = rowsum(dO o O) of the item into smem (double-buffered)
//   warps 4-7     warpgroup 0: even 32-query chunks; dV epilogue; dQ tiles 0, 2
//   warps 8-11    warpgroup 1: odd chunks; dK epilogue; dQ tile 1
// TMEM columns: three rotating chunk sets {S^T [0,32) | dP^T [32,64)} at 0, 64, 128 (chunk n uses set n % 3, so the S/dP
//               MMAs run three chunks ahead of the warpgroups) | [192,256) dV | [256,320) dK | [320,512) dQ, three 128-query
//               tiles.  P^T / dS^T overwrite the first 16 columns of S^T / dP^T in place.
#include "common.cuh"
#include <cstdlib>
#include "../../include/unite_b200.h"

namespace ub {

int make_tmap_3d_bf16(CUtensorMap* out, const void* base, int64_t d2, int64_t d1, int64_t d0, int64_t stride1_elems,
                      int64_t stride2_elems, int box0, int box1);

constexpr int ABT_THREADS = 384;
constexpr int ABT_MAX_S = 320;
// shared memory map (bytes)
constexpr int ABT_Q = 0;                         // Q of the item: up to 5 boxes of [64 rows][64 d]
constexpr int ABT_DO = 40960;                    // dO, same
constexpr int ABT_KV = 81920;                    // 2 slots x {K tile, V tile} of [128 keys][64 d]
constexpr int ABT_DS = ABT_KV + 65536;           // dS^T staging: 2 regions of [128 keys][64 queries]
constexpr int ABT_OUT = ABT_DS + 32768;          // 8 warps x 4 KB output staging
constexpr int ABT_LD = ABT_OUT + 32768;          // [2 buffers][L: 320 | D: 320] fp32
constexpr int ABT_BAR = ABT_LD + 2 * 2 * 320 * 4;
constexpr int ABT_NBAR = 24;
constexpr int ABT_SMEM = ABT_BAR + ABT_NBAR * 8 + 16;

struct AttnBwdTcParams {
  const float* lse;
  const float* Dv;
  float* dbias;             // optional fp32 [3*H*64]: += column sums of the dq and dv written (the q_bias / v_bias gradients)
  int n_seq, S, H;
  int nkt, nc, nb, ntile;   // key tiles (128), query chunks (32), Q/dO boxes (64 rows), query tiles (128)
  float sl2, scale;
};

__global__ void __launch_bounds__(ABT_THREADS, 1)
attn_bwd_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                   const __grid_constant__ CUtensorMap tmDO, const __grid_constant__ CUtensorMap tmOut,
                   const AttnBwdTcParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + ABT_BAR);
  uint64_t* q_full = bars;            // [3] Q + dO rows of query tile t have landed (per item)
  uint64_t* qdo_empty = bars + 3;     // every MMA of the item has read Q / dO
  uint64_t* kv_full = bars + 4;       // [2]
  uint64_t* kv_empty = bars + 6;      // [2] every MMA of the key tile has read the slot
  uint64_t* s_full = bars + 8;        // [3] S^T / dP^T of the chunk in TMEM set (n % 3) are complete
  uint64_t* p_ready = bars + 11;      // [3] P^T / dS^T of that set written (TMEM + smem staging)
  uint64_t* stage_free = bars + 14;   // the dQ MMAs that read the dS^T staging have completed
  uint64_t* dkv_full = bars + 15;     // dV / dK of the key tile are final
  uint64_t* dkv_free = bars + 16;     // ... and have been read out
  uint64_t* dq_full = bars + 17;
  uint64_t* dq_free = bars + 18;
  uint64_t* ld_full = bars + 19;      // [2]
  uint64_t* ld_empty = bars + 21;     // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + ABT_NBAR);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmKV);
    tma_prefetch_desc(&tmDO);
    tma_prefetch_desc(&tmOut);
    for (int i = 0; i < 3; ++i) mbar_init(&q_full[i], 1);
    mbar_init(qdo_empty, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 1);
      mbar_init(&ld_full[i], 1);
      mbar_init(&ld_empty[i], 8);
    }
    for (int i = 0; i < 3; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&p_ready[i], 4);
    }
    mbar_init(stage_free, 1);
    mbar_init(dkv_full, 1);
    mbar_init(dkv_free, 8);
    mbar_init(dq_full, 1);
    mbar_init(dq_free, 8);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int n_items = p.n_seq * p.H;
  const int nkt = p.nkt, nc = p.nc, total = p.nkt * p.nc;
  constexpr uint32_t TM_DV = 192, TM_DK = 256, TM_DQ = 320;

  if (warp == 0) {
    // ------------------------------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      auto load_kv = [&](int kvn, int item, int kt) {
        const int slot = kvn & 1, seq = item / p.H, h = item % p.H;
        mbar_wait(&kv_empty[slot], ((kvn >> 1) & 1) ^ 1);
        uint8_t* dst = smem + ABT_KV + slot * 32768;
        mbar_expect_tx(&kv_full[slot], 32768);
        tma_load_3d(&tmKV, &kv_full[slot], dst, (p.H + h) * 64, kt * 128, seq);
        tma_load_3d(&tmKV, &kv_full[slot], dst + 16384, (2 * p.H + h) * 64, kt * 128, seq);
      };
      int it = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
        const int seq = item / p.H, h = item % p.H;
        if (it == 0) load_kv(0, item, 0);
        mbar_wait(qdo_empty, (it & 1) ^ 1);
        for (int t = 0; t < p.ntile; ++t) {
          const int b0 = 2 * t, b1 = min(p.nb, 2 * t + 2);
          mbar_expect_tx(&q_full[t], (uint32_t)(b1 - b0) * 16384u);
          for (int b = b0; b < b1; ++b) {
            tma_load_3d(&tmQ, &q_full[t], smem + ABT_Q + b * 8192, h * 64, b * 64, seq);
            tma_load_3d(&tmDO, &q_full[t], smem + ABT_DO + b * 8192, h * 64, b * 64, seq);
          }
        }
        for (int kt = 1; kt < nkt; ++kt) load_kv(it * nkt + kt, item, kt);
        if (item + (int)gridDim.x < n_items) load_kv((it + 1) * nkt, item + gridDim.x, 0);
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------------------------------ MMA issuer
    // The whole warp runs this code with warp-uniform values (so descriptors live in uniform registers); only the
    // tcgen05 instructions themselves are predicated on one elected lane.  Descriptors: only the low word (address >> 4)
    // changes; the high words are compile-time constants.
    constexpr uint32_t IDESC_S = umma_idesc_bf16(128, 32, 0, 0);    // S^T / dP^T : both operands K-major
    constexpr uint32_t IDESC_KV = umma_idesc_bf16(128, 64, 0, 1);   // dV / dK    : A in TMEM, B MN-major
    constexpr uint32_t IDESC_DQ = umma_idesc_bf16(128, 64, 1, 1);   // dQ         : A (dS^T staging) and B (K) MN-major
    constexpr uint32_t HI_K = (1024u >> 4) | (1u << 14) | (2u << 29);            // SBO 1024 B, version 1, 128B swizzle
    constexpr uint32_t LO_K = 1u << 16;                                           // LBO field (ignored, K-major)
    constexpr uint32_t LO_MN8 = (8192u >> 4) << 16, LO_MN16 = (16384u >> 4) << 16;
    const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t aQ = (smem_u32(smem + ABT_Q) & 0x3FFFFu) >> 4, aDO = (smem_u32(smem + ABT_DO) & 0x3FFFFu) >> 4;
    const uint32_t aKV = (smem_u32(smem + ABT_KV) & 0x3FFFFu) >> 4, aDS = (smem_u32(smem + ABT_DS) & 0x3FFFFu) >> 4;
    uint32_t kvn = 0, set = 0, ph = 0;    // key tiles consumed so far; TMEM set (n % 3) and phase ((n / 3) & 1) of chunk n
    uint32_t la_kvn = 0, la_set = 0;      // look-ahead cursor: next S^T / dP^T chunk to issue (3 chunks ahead)
    int it = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
      int la_kt = 0, la_c = 0;
      auto issue_sdp = [&]() {
        const uint32_t slot = la_kvn & 1u;
        if (la_c == 0) mbar_wait(&kv_full[slot], (la_kvn >> 1) & 1u);
        if (la_kt == 0 && (la_c & 3) == 0) mbar_wait(&q_full[la_c >> 2], it & 1);
        tc_fence_after();
        const uint32_t kd = aKV + slot * 2048u + LO_K, vd = kd + 1024u;
        const uint32_t qd = aQ + (uint32_t)la_c * 256u + LO_K, dod = aDO + (uint32_t)la_c * 256u + LO_K;
        const uint32_t dS = tb + la_set * 64u;
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss_lo(dS, kd + k * 2, HI_K, qd + k * 2, HI_K, IDESC_S, k > 0);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_ss_lo(dS + 32, vd + k * 2, HI_K, dod + k * 2, HI_K, IDESC_S, k > 0);
          umma_commit(&s_full[la_set]);
        }
        __syncwarp();
        if (++la_set == 3) la_set = 0;
        if (++la_c == nc) { la_c = 0; ++la_kt; ++la_kvn; }
      };
      issue_sdp();
      if (total > 1) issue_sdp();
      if (total > 2) issue_sdp();
      for (int kt = 0; kt < nkt; ++kt, ++kvn) {
        const uint32_t slot = kvn & 1u;
        for (int c = 0; c < nc; ++c) {
          mbar_wait(&p_ready[set], ph);
          if (c == 0) mbar_wait(dkv_free, (kvn & 1u) ^ 1u);
          const bool tile_end = (c & 3) == 3 || c == nc - 1;
          if (tile_end && kt == 0 && c < 4) mbar_wait(dq_free, (it & 1) ^ 1);
          tc_fence_after();
          const uint32_t dod = aDO + (uint32_t)c * 256u + LO_MN8, qd = aQ + (uint32_t)c * 256u + LO_MN8;
          const uint32_t tP = tb + set * 64u;
          const bool first = c == 0;
          if (elect_one()) {
            umma_ts_lo(tb + TM_DV, tP, dod, HI_K, IDESC_KV, !first);
            umma_ts_lo(tb + TM_DV, tP + 8, dod + 128, HI_K, IDESC_KV, true);
            umma_ts_lo(tb + TM_DK, tP + 32, qd, HI_K, IDESC_KV, !first);
            umma_ts_lo(tb + TM_DK, tP + 40, qd + 128, HI_K, IDESC_KV, true);
            if (tile_end) {
              const uint32_t ad = aDS + LO_MN16, bd = aKV + slot * 2048u + LO_MN8;
              const uint32_t dq = tb + TM_DQ + (uint32_t)(c >> 2) * 64u;
              umma_ss_lo(dq, ad, HI_K, bd, HI_K, IDESC_DQ, kt > 0);
#pragma unroll
              for (int k = 1; k < 8; ++k) umma_ss_lo(dq, ad + k * 128, HI_K, bd + k * 128, HI_K, IDESC_DQ, true);
              umma_commit(stage_free);
            }
            if (c == nc - 1) {
              umma_commit(dkv_full);
              umma_commit(&kv_empty[slot]);
              if (kt == nkt - 1) {
                umma_commit(dq_full);
                umma_commit(qdo_empty);
              }
            }
          }
          __syncwarp();
          if (++set == 3) { set = 0; ph ^= 1u; }
          if (la_kt < nkt) issue_sdp();
        }
      }
    }
  } else if (warp == 2) {
    // ------------------------------------------------------------------------------------------ LSE / D loader
    int it = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
      const int b = it & 1;
      mbar_wait(&ld_empty[b], ((it >> 1) & 1) ^ 1);
      float* sL = reinterpret_cast<float*>(smem + ABT_LD) + b * 640;
      float* sD = sL + 320;
      const float* gL = p.lse + (int64_t)item * p.S;
      const float* gD = p.Dv + (int64_t)item * p.S;
      for (int i = lane; i < nc * 32; i += 32) {
        sL[i] = i < p.S ? __ldg(gL + i) * 1.4426950408889634f : INFINITY;   // +inf -> P = 0 for padded queries
        sD[i] = i < p.S ? __ldg(gD + i) : 0.f;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&ld_full[b]);
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------------------------------ softmax-gradient warpgroups
    const int g = (warp - 4) >> 2;         // warpgroup
    const int sp = warp & 3;               // TMEM sub-partition = 32-row group of the key tile
    const uint32_t t_lane = tmem_base + ((uint32_t)(sp * 32) << 16);
    const int krow = sp * 32 + lane;       // key row of this thread within the tile
    const uint32_t ds_row = smem_u32(smem + ABT_DS) + (uint32_t)krow * 128u;
    const uint32_t sw = (uint32_t)(lane & 7);
    uint8_t* stg = smem + ABT_OUT + (warp - 4) * 4096;
    const uint32_t stg_a = smem_u32(stg);
    const float sl2 = p.sl2;
    int it = 0;
    uint32_t m_seq = 0;                    // dS^T staging use counter (same sequence as the MMA issuer's)
    uint32_t set = 0, ph = 0, par = 0;     // TMEM set (n % 3), its phase ((n / 3) & 1) and owner warpgroup (n & 1) of chunk n
    uint32_t kvn = 0;
    // TMEM (32 rows x 64 fp32 columns at t_src) -> * mul -> bf16 -> swizzled slab -> TMA store at (col, row, seq)
    auto store_tile = [&](uint32_t t_src, float mul, int col, int row, int seq, float* bias_dst) {
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
      if (lane == 0 && row < p.S) {
        tma_store_3d(&tmOut, stg, col, row, seq);
        tma_store_commit();
      }
      if (bias_dst != nullptr && row < p.S) {
        // bias gradient of these 64 columns: column sums of the bf16 slab just written, rows of the sequence only (a dQ tile's
        // rows past the last query chunk are whatever the never-written part of the dS^T staging held); lane l owns columns
        // 2l, 2l+1 — every lane reads 4 B of the same swizzled 128-byte row: conflict-free
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
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
      const int seq = item / p.H, h = item % p.H;
      const float* sL = reinterpret_cast<const float*>(smem + ABT_LD) + (it & 1) * 640;
      const float* sD = sL + 320;
      mbar_wait(&ld_full[it & 1], (it >> 1) & 1);
      for (int kt = 0; kt < nkt; ++kt, ++kvn) {
      for (int c = 0; c < nc; ++c) {
        if (par == (uint32_t)g) {
          const bool key_ok = kt * 128 + krow < p.S;
          const uint32_t t_s = t_lane + set * 64u, t_dp = t_s + 32u;
          mbar_wait(&s_full[set], ph);
          tc_fence_after();
          uint32_t sv[32], dv[32];
          tmem_ld_32x32(t_s, sv);
          tmem_ld_32x32(t_dp, dv);
          tmem_ld_wait();
          uint32_t pk[16], dk[16];
          const float4* L4 = reinterpret_cast<const float4*>(sL + c * 32);
          const float4* D4 = reinterpret_cast<const float4*>(sD + c * 32);
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
          if (!key_ok) {
#pragma unroll
            for (int i = 0; i < 16; ++i) { pk[i] = 0u; dk[i] = 0u; }
          }
          tmem_st_32x16(t_s, pk);
          tmem_st_32x16(t_dp, dk);
          // dS^T row of this key: 32 queries = 4 x 16 B into the [128 keys][64 queries] region of this half-tile
          const uint32_t m_cur = m_seq;
          if ((c & 3) < 2) {
            // first chunk of this warpgroup in the query tile: the dQ MMAs of the previous tile must be done with the staging
            mbar_wait(stage_free, (m_cur & 1) ^ 1);
          }
          {
            const uint32_t reg = ds_row + (uint32_t)(((c & 3) >> 1) * 16384);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint32_t a = reg + ((((uint32_t)((c & 1) * 4 + j)) ^ sw) << 4);
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(dk[4 * j]), "r"(dk[4 * j + 1]), "r"(dk[4 * j + 2]),
                           "r"(dk[4 * j + 3])
                           : "memory");
            }
          }
          tmem_st_wait();
          tc_fence_before();
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(&p_ready[set]);
        }
        par ^= 1u;
        if (++set == 3) { set = 0; ph ^= 1u; }
        if ((c & 3) == 3 || c == nc - 1) ++m_seq;
        if (c == nc - 1) {
          // ---- dV (warpgroup 0) / dK (warpgroup 1) of this key tile
          mbar_wait(dkv_full, kvn & 1);
          tc_fence_after();
          const int row = kt * 128 + sp * 32;
          if (g == 0) store_tile(t_lane + TM_DV, 1.0f, (2 * p.H + h) * 64, row, seq, p.dbias ? p.dbias + (2 * p.H + h) * 64 : nullptr);
          else store_tile(t_lane + TM_DK, p.scale, (p.H + h) * 64, row, seq, nullptr);     // the key bias is structurally zero
          if (lane == 0) mbar_arrive(dkv_free);
        }
      }
      }
      // ---- dQ of the item
      mbar_wait(dq_full, it & 1);
      tc_fence_after();
      for (int t = g; t < p.ntile; t += 2)
        store_tile(t_lane + TM_DQ + t * 64, p.scale, h * 64, t * 128 + sp * 32, seq, p.dbias ? p.dbias + h * 64 : nullptr);
      if (lane == 0) {
        mbar_arrive(dq_free);
        mbar_arrive(&ld_empty[it & 1]);
      }
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

// D = rowsum(dO o O) is produced by attn_bwd_prep_kernel (attention.cu) before this launch.
int launch_attn_bwd_tc(const void* qkv, const void* d_o, const float* lse, const float* Dv, void* dqkv, float* dbias, int n_seq, int S,
                       int H, float scale, cudaStream_t stream) {
  UB_REQUIRE(S <= ABT_MAX_S, "attn_bwd_tc: S=%d exceeds %d", S, ABT_MAX_S);
  AttnBwdTcParams p;
  p.lse = lse; p.Dv = Dv; p.dbias = dbias;
  p.n_seq = n_seq; p.S = S; p.H = H;
  p.nkt = (S + 127) / 128;
  p.nc = (S + 31) / 32;
  p.nb = (S + 63) / 64;
  p.ntile = (S + 127) / 128;
  p.scale = scale;
  p.sl2 = scale * 1.4426950408889634f;
  CUtensorMap tq, tkv, tdo, tout;
  const int64_t ld = 3 * (int64_t)H * 64, ldo = (int64_t)H * 64;
  if (make_tmap_3d_bf16(&tq, qkv, n_seq, S, ld, ld, (int64_t)S * ld, 64, 64)) return 1;
  if (make_tmap_3d_bf16(&tkv, qkv, n_seq, S, ld, ld, (int64_t)S * ld, 64, 128)) return 1;
  if (make_tmap_3d_bf16(&tdo, d_o, n_seq, S, ldo, ldo, (int64_t)S * ldo, 64, 64)) return 1;
  if (make_tmap_3d_bf16(&tout, dqkv, n_seq, S, ld, ld, (int64_t)S * ld, 64, 32)) return 1;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(attn_bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ABT_SMEM);
    UB_REQUIRE(e == cudaSuccess, "cudaFuncSetAttribute(attn_bwd_tc smem=%d): %s", ABT_SMEM, cudaGetErrorString(e));
    configured = true;
  }
  const int items = n_seq * H;
  const int grid = items < sm_count() ? items : sm_count();
  UB_LAUNCH(attn_bwd_tc_kernel, grid, ABT_THREADS, ABT_SMEM, stream, tq, tkv, tdo, tout, p);
  return check_launch("attn_bwd_tc_kernel");
}

}  // namespace ub
