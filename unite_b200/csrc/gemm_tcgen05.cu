// tcgen05 / TMEM / TMA GEMM for sm_100a:   C[M,N] = epilogue(A[M,K] * B[N,K]^T), bf16 in, fp32 accumulate.
//
// Replaces every dense contraction of the UNITE step (see include/unite_b200.h for the reference
// call sites).  Design (B200-first, nothing like the reference's cuBLAS calls):
//   * persistent CTAs (one per SM), static round-robin over (m-tile, n-tile, k-split) work items;
//     wide tiles run as CTA PAIRS (cluster of 2, tcgen05 cta_group::2): 256 x 256 per pair, each CTA keeps its own
//     128 rows of A and half of B in smem;
//   * warp 0  : TMA producer  (cp.async.bulk.tensor, 128B-swizzled boxes, STAGES-deep mbarrier ring);
//   * warp 1  : single-thread tcgen05.mma issuer (leader CTA of a pair), accumulators in TMEM, two accumulator
//               stages (2*BN columns) so the epilogue of tile i overlaps the MMAs of tile i+1;
//   * warps 2-9: epilogue.  tcgen05.ld gives each lane one accumulator ROW; bias / activation / DropPath scale are
//               applied in registers, the 32-row slab is written to a 128B-swizzled smem staging buffer and leaves
//               through the TMA engine (bulk tensor store, or cp.reduce.async.bulk .add for split-K weight
//               gradients).  The fp32 residual and the bf16 GELU pre-activation ARRIVE through TMA too (loaded
//               one slab ahead into the same staging buffers and combined in place), so the epilogue issues no
//               per-thread global loads/stores, no address arithmetic and no bounds checks (TMA clips).
//   * operands may be K-major (activations, weights [out,in]) or MN-major (the same row-major tensors
//     contracted over their ROW index: dgrad uses W as B^T, wgrad contracts over tokens) — no transposes
//     are ever materialised.
#include "common.cuh"
#include <cuda_fp16.h>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <unordered_map>
#include "../../include/unite_b200.h"

namespace ub {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int GEMM_THREADS = 320;  // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue
constexpr int EPI_BYTES = 8 * 2 * 4096;   // 8 epilogue warps x 2 staging slabs of 32 rows x 128 B
// Dynamic shared memory of a GEMM CTA (the layout gemm_body carves out): the STAGES-deep A / B ring, the staging slabs, the bias
// tile [2][BN], the mbarriers (full / empty per stage, tfull / tempty x 2, two residual barriers per epilogue warp) and the TMEM slot.
constexpr int gemm_smem_bytes(int BN, int STAGES, int NCTA) {
  return STAGES * (BM * BK * 2 + (BN / (NCTA >= 2 ? 2 : 1)) * BK * 2) + EPI_BYTES + 2 * BN * 4 + (2 * STAGES + 4 + 16) * 8 + 16;
}

struct GemmParams {
  int M, N, K;
  int splits, kb_per_split;
  const float* bias;
  const float* row_scale;
  int rows_per_scale;
  int act;
  int accumulate;
  int has_aux_out;
  int ab_f16;               // operands are fp16 instead of bf16
  const float* ln_stats;    // LayerNorm fold: row (sum, sumsq) of A
  const float* ln_c;        //                 column sums of B
  float ln_inv_d, ln_eps;
  float* stats_out;         // EPI 3: row (sum, sumsq) of the fp16 output
  float* colsum_out;        // EPI 2: += column sums of the values written to C (the bias gradient of the Linear that produced aux)
  float* dot_out;           // EPI 2 with act == UB_ACT_DOT_AUX: per (row, 64-column head) dot product of the bf16 output with aux
  int dot_seq_len;
  // grouped GEMM (ub_gemm_epilogue.group_*): work item with first C row m0 belongs to group g = m0 / group_rows
  int group_rows;           // 0 = ungrouped
  int a_k_off, a_m_off;     // A coordinates: k += g * a_k_off, m -= g * a_m_off
  int b_k_off, b_n_off;     // B coordinates: k += g * b_k_off, n += g * b_n_off
  int bias_off;             // bias index += g * bias_off
  // multi-problem launch (ub_gemm_wgrad_multi): n_prob products of the same K and operand majors but different M x N and
  // buffers; tile t belongs to problem i with tile_off[i] <= t < tile_off[i + 1], which has ntile_n[i] tiles along N
  int n_prob;
  int tile_off[5];
  int ntile_n[4];
};

constexpr int GEMM_MAX_PROB = 4;
struct GemmMultiMaps {
  CUtensorMap a[GEMM_MAX_PROB], b[GEMM_MAX_PROB], c[GEMM_MAX_PROB];
};

// EPI : 0 = bias / activation (/ pre-activation copy), 1 = + fp32 residual (fp32 out), 2 = DGELU: * gelu'(aux) (bf16 out),
//       3 = + fp16 residual (fp16 out: the frozen teacher's residual stream), 4 = EPI 0 with the LayerNorm fold (its own
//       instantiation: the fold's column sums are 32 registers that the plain epilogues should not carry)
// OUT32: C is fp32 (32-column slabs) or bf16 (64-column slabs); both give 128-byte staging rows
// NCTA: 1 = one CTA per 128 x BN tile; 2 = CTA pair per 256 x BN tile; 4 = cluster of two pairs on a 512 x BN tile that
//       share B: each CTA fetches a quarter of the B tile and TMA-multicasts it to the CTA of the same rank in the other pair
//       (the mainloop is bound by L2 -> SM bytes: 24 KB instead of 32 KB per CTA and k-block)
template <int BN, int STAGES, bool A_MN, bool B_MN, int EPI, bool OUT32, int NCTA, bool MULTI>
UB_DEVINL void gemm_body(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const CUtensorMap& tmR,
                         const CUtensorMap& tmX, const GemmMultiMaps* mm, const GemmParams& p) {
  constexpr int CG = NCTA >= 2 ? 2 : 1;      // CTAs per MMA (tcgen05 cta_group)
  constexpr int NP = NCTA / CG;              // CTA pairs per cluster
  constexpr int BN_L = BN / CG;              // rows of B resident in this CTA
  constexpr int A_BYTES = BM * BK * 2;
  constexpr int B_BYTES = BN_L * BK * 2;
  constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr uint32_t TMEM_COLS = 2 * BN;  // 256 or 512: power of two
  constexpr uint32_t IDESC_BF16 = umma_idesc_bf16(BM * CG, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
  constexpr uint32_t FMT_BF16 = (1u << 7) | (1u << 10);          // a_format / b_format = BF16; 0 = F16
  const uint32_t IDESC = p.ab_f16 ? (IDESC_BF16 & ~FMT_BF16) : IDESC_BF16;
  constexpr int CW = OUT32 ? 32 : 64;        // columns per epilogue slab
  constexpr int SLABS = (BN / 2) / CW;       // slabs per warp per tile
  static_assert(EPI != 1 || OUT32, "residual epilogue writes fp32");
  static_assert(EPI != 2 || !OUT32, "DGELU epilogue writes bf16");
  static_assert(EPI != 3 || !OUT32, "the fp16-residual epilogue writes fp16");
  const uint32_t cta_rank = NCTA >= 2 ? cluster_ctarank() : 0u;
  const uint32_t pr = cta_rank & (CG - 1);          // rank inside the pair
  const uint32_t pp = cta_rank / CG;                // pair inside the cluster
  const uint32_t leader_rank = cta_rank - pr;
  const bool leader = pr == 0;

  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* epi_s = smem + STAGES * STAGE_BYTES;                       // [8 warps][2][4096], 1024-aligned
  float* bias_s = reinterpret_cast<float*>(epi_s + EPI_BYTES);         // [2][BN]
  uint64_t* full = reinterpret_cast<uint64_t*>(bias_s + 2 * BN);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint64_t* tempty = tfull + 2;
  uint64_t* rbar = tempty + 2;                                         // [8 warps][2] residual / aux slab arrived
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(rbar + 16);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    if ((smem_u32(smem) & 1023u) != 0) __trap();   // swizzled TMA / UMMA tiles need the 1024-byte alignment
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmC);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], NP);        // one commit per pair that reads (or multicasts into) the slot
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], 8 * CG);     // the leader's copy collects the epilogue warps of both CTAs
    }
    for (int i = 0; i < 16; ++i) mbar_init(&rbar[i], 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    if (NCTA >= 2) {
      tmem_alloc_cg2(tmem_slot, TMEM_COLS);
      tmem_relinquish_cg2();
    } else {
      tmem_alloc(tmem_slot, TMEM_COLS);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  if (NCTA >= 2) cluster_sync(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int m_tiles = (p.M + BM * NCTA - 1) / (BM * NCTA);
  const int n_tiles = (p.N + BN - 1) / BN;
  const int total_kb = (p.K + BK - 1) / BK;
  const int total_work = (MULTI ? p.tile_off[p.n_prob] : m_tiles * n_tiles) * p.splits;
  // (problem, tile row, tile column) of tile t: one problem unless MULTI
  auto decode = [&](int t, int& pi, int& tm, int& tn) {
    if (MULTI) {
      pi = 0;
#pragma unroll
      for (int i = 1; i < GEMM_MAX_PROB; ++i) pi += (i < p.n_prob && t >= p.tile_off[i]) ? 1 : 0;
      const int lt = t - p.tile_off[pi], ntn = p.ntile_n[pi];
      tm = lt / ntn;
      tn = lt - tm * ntn;
    } else {
      pi = 0;
      tm = t / n_tiles;
      tn = t - tm * n_tiles;
    }
  };
  const int w_first = blockIdx.x / NCTA, w_step = gridDim.x / NCTA;   // both CTAs of a pair walk the same work items

  // ---- this pair's list of work items: item i is work index w_first + i * w_step = (tile, k-split)
  const int n_items = w_first < total_work ? (total_work - w_first + w_step - 1) / w_step : 0;
  // item i -> (tile, k-block range)
  auto get_item = [&](int i, int& tile, int& kb0, int& kb1) {
    const int w = w_first + i * w_step, ks = w % p.splits;
    tile = w / p.splits;
    kb0 = ks * p.kb_per_split;
    kb1 = min(total_kb, kb0 + p.kb_per_split);
  };

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    int stage = 0;
    uint32_t phase = 0;
    for (int it = 0; it < n_items; ++it) {
      int tile, kb0, kb1;
      get_item(it, tile, kb0, kb1);
      int pi, tm, tn;
      decode(tile, pi, tm, tn);
      const CUtensorMap* pA = MULTI ? &mm->a[pi] : &tmA;
      const CUtensorMap* pB = MULTI ? &mm->b[pi] : &tmB;
      const int grp = p.group_rows ? (tm * (BM * NCTA)) / p.group_rows : 0;
      const int m0 = tm * (BM * NCTA) + (int)cta_rank * BM - grp * p.a_m_off;      // this CTA's rows of A
      const int n0 = tn * BN + (int)pr * BN_L + grp * p.b_n_off;                   // this CTA's rows of B
      const int ka = grp * p.a_k_off, kbo = grp * p.b_k_off;                                     // K offsets of the group
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&empty[stage], phase ^ 1);
        if (lane == 0) {
          uint8_t* sA = smem + stage * STAGE_BYTES;
          uint8_t* sB = sA + A_BYTES;
          if (NCTA >= 2) {
            // both CTAs' loads complete on the LEADER's full barrier, which expects the bytes of the whole pair
            const uint32_t lbar = mapa_u32(smem_u32(&full[stage]), leader_rank);
            if (leader) mbar_expect_tx(&full[stage], STAGE_BYTES * 2);
            if (A_MN) {
#pragma unroll
              for (int j = 0; j < BM / 64; ++j) tma_load_2d_cg2(pA, lbar, sA + j * 8192, m0 + j * 64, kb * BK + ka);
            } else {
              tma_load_2d_cg2(pA, lbar, sA, kb * BK + ka, m0);
            }
            if (NCTA == 4) {
              // this CTA's quarter of the B tile (64 rows / one 64-wide MN chunk = 8 KB) lands in both pairs
              const uint16_t mask = (uint16_t)((1u << pr) | (1u << (CG + pr)));
              if (B_MN) tma_load_2d_cg2_mc(pB, lbar, sB + pp * 8192, n0 + (int)pp * 64, kb * BK + kbo, mask);
              else tma_load_2d_cg2_mc(pB, lbar, sB + pp * 8192, kb * BK + kbo, n0 + (int)pp * 64, mask);
            } else if (B_MN) {
#pragma unroll
              for (int j = 0; j < BN_L / 64; ++j) tma_load_2d_cg2(pB, lbar, sB + j * 8192, n0 + j * 64, kb * BK + kbo);
            } else {
              tma_load_2d_cg2(pB, lbar, sB, kb * BK + kbo, n0);
            }
          } else {
            mbar_expect_tx(&full[stage], STAGE_BYTES);
            if (A_MN) {
#pragma unroll
              for (int j = 0; j < BM / 64; ++j) tma_load_2d(pA, &full[stage], sA + j * 8192, m0 + j * 64, kb * BK + ka);
            } else {
              tma_load_2d(pA, &full[stage], sA, kb * BK + ka, m0);
            }
            if (B_MN) {
#pragma unroll
              for (int j = 0; j < BN_L / 64; ++j) tma_load_2d(pB, &full[stage], sB + j * 8192, n0 + j * 64, kb * BK + kbo);
            } else {
              tma_load_2d(pB, &full[stage], sB, kb * BK + kbo, n0);
            }
          }
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1 && leader) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA of a pair only)
    int stage = 0;
    uint32_t phase = 0;
    int as = 0;
    uint32_t aphase = 0;
    for (int it = 0; it < n_items; ++it) {
      int tile, kb0, kb1;
      get_item(it, tile, kb0, kb1);
      if (NCTA >= 2) mbar_wait_cluster(&tempty[as], aphase ^ 1); else mbar_wait(&tempty[as], aphase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&full[stage], phase);
        tc_fence_after();
        if (lane == 0) {
          const uint32_t sA = smem_u32(smem + stage * STAGE_BYTES);
          const uint32_t sB = sA + A_BYTES;
          const uint64_t adesc = A_MN ? umma_desc_mnmajor_sw128(sA, 8192) : umma_desc_kmajor_sw128(sA);
          const uint64_t bdesc = B_MN ? umma_desc_mnmajor_sw128(sB, 8192) : umma_desc_kmajor_sw128(sB);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // advance along K by 16 elements: 32 B inside the swizzle atom (K-major) or two 8-row groups (MN-major)
            const uint64_t ad = adesc + (uint64_t)(A_MN ? (k * 2048) >> 4 : (k * 32) >> 4);
            const uint64_t bd = bdesc + (uint64_t)(B_MN ? (k * 2048) >> 4 : (k * 32) >> 4);
            if (NCTA >= 2) umma_bf16_cg2(d_tmem, ad, bd, IDESC, (kb > kb0 || k > 0) ? 1u : 0u);
            else umma_bf16(d_tmem, ad, bd, IDESC, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          // frees the smem slot (in both CTAs of a pair) once these MMAs have read it
          if (NCTA >= 2) umma_commit_cg2(&empty[stage], (uint16_t)((1u << NCTA) - 1)); else umma_commit(&empty[stage]);
          if (kb == kb1 - 1) {
            if (NCTA >= 2) umma_commit_cg2(&tfull[as], (uint16_t)(3u << leader_rank)); else umma_commit(&tfull[as]);
          }
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
      as ^= 1;
      if (as == 0) aphase ^= 1;
    }
  } else if (warp >= 2) {
    // ------------------------------------------------------------------ epilogue (warps 2..9)
    const int we = warp - 2;
    const int sp = warp & 3;            // TMEM sub-partition this warp may read
    const int half = we >> 2;           // which half of the BN columns
    const int etid = threadIdx.x - 64;  // 0..255
    uint8_t* const slab0 = epi_s + we * (2 * 4096);      // two 4 KB staging slabs: slab0 + (b << 12)
    const uint32_t slab0_a = smem_u32(slab0);
    uint64_t* rb = rbar + we * 2;
    const uint32_t sw = (uint32_t)(lane & 7);      // 16-byte chunk XOR of this lane's row (128B swizzle)
    const uint32_t rowoff = (uint32_t)lane * 128u;
    int as = 0;
    uint32_t aphase = 0;
    uint32_t cc = 0;                    // running slab counter of this warp: staging buffer = cc & 1
    // (row, col) of this warp's slab `c` of work item `i`
    auto item_tile = [&](int i) {
      int tile, kb0, kb1;
      get_item(i, tile, kb0, kb1);
      return tile;
    };
    auto slab_row = [&](int i) {
      int pi, tm, tn;
      decode(item_tile(i), pi, tm, tn);
      return tm * (BM * NCTA) + (int)cta_rank * BM + sp * 32;
    };
    auto slab_col = [&](int i, int c) {
      int pi, tm, tn;
      decode(item_tile(i), pi, tm, tn);
      return tn * BN + half * (BN / 2) + c * CW;
    };
    if (EPI != 0 && EPI != 4 && n_items > 0 && lane == 0) {
      // residual / pre-activation slab of the first (tile, slab) pair of this warp
      mbar_expect_tx(&rb[0], 4096);
      tma_load_2d(&tmR, &rb[0], slab0, slab_col(0, 0), slab_row(0));
    }
    for (int w = 0; w < n_items; ++w) {
      int w_pi, w_tm, w_tn;
      decode(item_tile(w), w_pi, w_tm, w_tn);
      const CUtensorMap* pC = MULTI ? &mm->c[w_pi] : &tmC;
      const int n0 = w_tn * BN;
      const int row0 = slab_row(w);
      float* bias_tile = bias_s + as * BN;
      if (p.bias != nullptr) {
        const int goff = p.group_rows ? ((w_tm * (BM * NCTA)) / p.group_rows) * p.bias_off : 0;
        if (etid < BN) bias_tile[etid] = (n0 + etid < p.N) ? __ldg(p.bias + goff + n0 + etid) : 0.0f;
        asm volatile("bar.sync 1, 256;" ::: "memory");
      }
      float rscale = 1.0f;
      if (p.row_scale != nullptr) {
        const int row = row0 + lane;
        rscale = row < p.M ? __ldg(p.row_scale + row / p.rows_per_scale) : 0.0f;
      }
      float ln_rstd = 1.0f, ln_rm = 0.0f;       // LayerNorm fold: acc -> rstd * acc - (rstd * mu) * c[n]
      if (EPI == 4) {
        const int row = row0 + lane;
        if (row < p.M) {
          const float2 st = __ldg(reinterpret_cast<const float2*>(p.ln_stats) + row);
          const float mu = st.x * p.ln_inv_d;
          ln_rstd = rsqrtf(fmaxf(st.y * p.ln_inv_d - mu * mu, 0.0f) + p.ln_eps);
          ln_rm = ln_rstd * mu;
        }
      }
      float st1 = 0.0f, st2 = 0.0f;             // EPI 3: row statistics of the fp16 values this thread writes
      mbar_wait(&tfull[as], aphase);
      tc_fence_after();
      const uint32_t t_row = tmem_base + ((uint32_t)(sp * 32) << 16) + (uint32_t)(as * BN + half * (BN / 2));
#pragma unroll 1
      for (int c = 0; c < SLABS; ++c, ++cc) {
        const int b = (int)(cc & 1u);
        const int col0 = slab_col(w, c);
        // ---- staging-buffer hand-over with the TMA engine
        if (EPI == 0 || EPI == 4) {
          // buffer b was last read by the store issued two slabs ago (one slab ago when a pre-activation copy uses b^1)
          if (lane == 0) {
            if (p.has_aux_out) tma_store_wait_read<0>(); else tma_store_wait_read<1>();
          }
          __syncwarp();
        } else {
          // the store of the previous slab read buffer b ^ 1: once done, the operand of the next slab is prefetched into it
          if (lane == 0) {
            tma_store_wait_read<0>();
            int nw = w, nc = c + 1;
            while (nc >= SLABS) { nc -= SLABS; ++nw; }
            if (nw < n_items) {
              const int nb = b ^ 1;
              mbar_expect_tx(&rb[nb], 4096);
              tma_load_2d(&tmR, &rb[nb], slab0 + (nb << 12), slab_col(nw, nc), slab_row(nw));
            }
          }
          __syncwarp();
          mbar_wait(&rb[b], (cc >> 1) & 1u);
        }
        // ---- accumulators -> registers -> epilogue math -> staging slab (row per lane, 128 B per row)
        float dsum = 0.0f;        // UB_ACT_DOT_AUX: this lane's row of the slab (64 columns = one head) dotted with aux
#pragma unroll
        for (int h = 0; h < CW / 32; ++h) {
          uint32_t r[32];
          tmem_ld_32x32(t_row + (uint32_t)(c * CW + h * 32), r);
          // LayerNorm fold: the column sums of B for these 32 columns are fetched (L1-resident, same address for every lane)
          // while the accumulator load is in flight
          float4 cc[EPI == 4 ? 8 : 1];
          if (EPI == 4) {
            const int gc = col0 + h * 32;
#pragma unroll
            for (int j = 0; j < 8; ++j)
              cc[EPI == 4 ? j : 0] = (gc + 4 * j < p.N) ? __ldg(reinterpret_cast<const float4*>(p.ln_c + gc + 4 * j)) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
          tmem_ld_wait();
          float v[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
          if (EPI == 4) {
            const float2 rs2 = make_float2(ln_rstd, ln_rstd), nrm2 = make_float2(-ln_rm, -ln_rm);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 q = cc[EPI == 4 ? j : 0];
              const float2 a = __ffma2_rn(nrm2, make_float2(q.x, q.y), __fmul2_rn(rs2, make_float2(v[4 * j], v[4 * j + 1])));
              const float2 b = __ffma2_rn(nrm2, make_float2(q.z, q.w), __fmul2_rn(rs2, make_float2(v[4 * j + 2], v[4 * j + 3])));
              v[4 * j] = a.x; v[4 * j + 1] = a.y; v[4 * j + 2] = b.x; v[4 * j + 3] = b.y;
            }
          }
          if (p.bias != nullptr) {
            const float* bt = bias_tile + half * (BN / 2) + c * CW + h * 32;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 bb = *reinterpret_cast<const float4*>(bt + j * 4);
              v[4 * j] += bb.x; v[4 * j + 1] += bb.y; v[4 * j + 2] += bb.z; v[4 * j + 3] += bb.w;
            }
          }
          if (EPI == 0 || EPI == 4) {
            if (p.act == UB_ACT_QUICKGELU) {
#pragma unroll
              for (int i = 0; i < 32; ++i) v[i] = quick_gelu(v[i]);
            } else if (p.act == UB_ACT_GELU) {
              if (p.has_aux_out) {
                // pre-activation copy (bf16) goes out through the other staging buffer
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  const uint32_t a = slab0_a + ((uint32_t)(b ^ 1) << 12) + rowoff + ((((uint32_t)(h * 4 + j)) ^ sw) << 4);
                  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(pack_bf16x2(v[8 * j], v[8 * j + 1])),
                               "r"(pack_bf16x2(v[8 * j + 2], v[8 * j + 3])), "r"(pack_bf16x2(v[8 * j + 4], v[8 * j + 5])),
                               "r"(pack_bf16x2(v[8 * j + 6], v[8 * j + 7]))
                               : "memory");
                }
              }
#pragma unroll
              for (int i = 0; i < 32; i += 2) {
                const float2 y = gelu_erf2(make_float2(v[i], v[i + 1]));
                v[i] = y.x; v[i + 1] = y.y;
              }
            }
          }
          if (EPI == 2 && p.act == UB_ACT_DOT_AUX) {
            // dot product of the bf16-rounded output with aux (the values the consumer of C and of dot_out will see)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint4 pk;
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                           : "=r"(pk.x), "=r"(pk.y), "=r"(pk.z), "=r"(pk.w)
                           : "r"(slab0_a + ((uint32_t)b << 12) + rowoff + ((((uint32_t)(h * 4 + j)) ^ sw) << 4)));
              const uint32_t ax[4] = {pk.x, pk.y, pk.z, pk.w};
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const float2 o2 = unpack_bf16x2(ax[q]);
                const float2 c2 = unpack_bf16x2(pack_bf16x2(v[8 * j + 2 * q], v[8 * j + 2 * q + 1]));
                dsum = fmaf(c2.x, o2.x, dsum);
                dsum = fmaf(c2.y, o2.y, dsum);
              }
            }
          } else if (EPI == 2) {
            // multiply by gelu'(pre-activation): bf16 slab row of this lane, chunks h*4 .. h*4+3
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint4 pk;
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                           : "=r"(pk.x), "=r"(pk.y), "=r"(pk.z), "=r"(pk.w)
                           : "r"(slab0_a + ((uint32_t)b << 12) + rowoff + ((((uint32_t)(h * 4 + j)) ^ sw) << 4)));
              const float2 g0 = gelu_erf_grad2(unpack_bf16x2(pk.x)), g1 = gelu_erf_grad2(unpack_bf16x2(pk.y));
              const float2 g2 = gelu_erf_grad2(unpack_bf16x2(pk.z)), g3 = gelu_erf_grad2(unpack_bf16x2(pk.w));
              v[8 * j] *= g0.x; v[8 * j + 1] *= g0.y;
              v[8 * j + 2] *= g1.x; v[8 * j + 3] *= g1.y;
              v[8 * j + 4] *= g2.x; v[8 * j + 5] *= g2.y;
              v[8 * j + 6] *= g3.x; v[8 * j + 7] *= g3.y;
            }
          }
          if (p.row_scale != nullptr) {
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] *= rscale;
          }
          if (EPI == 2 && p.colsum_out != nullptr) {
            // column sums over this warp's 32 rows (rows past M are exact zeros: A and the pre-activation are zero-filled by
            // TMA): recursive halving — at each step a lane keeps one half of its columns and hands the other half to its
            // partner — 31 shuffles, after which lane L holds the total of column L of this 32-column group
            float s[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) s[i] = v[i];
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) {
              const bool upper = (lane & off) != 0;
#pragma unroll
              for (int i = 0; i < off; ++i) {
                const float give = upper ? s[i] : s[i + off];
                const float keep = upper ? s[i + off] : s[i];
                s[i] = keep + __shfl_xor_sync(0xffffffffu, give, off);
              }
            }
            const int gcol = col0 + h * 32 + lane;
            if (gcol < p.N) atomicAdd(p.colsum_out + gcol, s[0]);
          }
          if (OUT32) {
            // fp32 slab: 8 chunks of 4 floats; EPI 1 adds the residual that TMA placed in the same slab
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const uint32_t a = slab0_a + ((uint32_t)b << 12) + rowoff + ((((uint32_t)j) ^ sw) << 4);
              if (EPI == 1) {
                float4 rr;
                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(rr.x), "=f"(rr.y), "=f"(rr.z), "=f"(rr.w) : "r"(a));
                v[4 * j] += rr.x; v[4 * j + 1] += rr.y; v[4 * j + 2] += rr.z; v[4 * j + 3] += rr.w;
              }
              asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v[4 * j]), "f"(v[4 * j + 1]), "f"(v[4 * j + 2]),
                           "f"(v[4 * j + 3])
                           : "memory");
            }
          } else if (EPI == 3) {
            // fp16 slab: the residual that TMA placed here is read, added in fp32 and replaced by the fp16 sum
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint32_t a = slab0_a + ((uint32_t)b << 12) + rowoff + ((((uint32_t)(h * 4 + j)) ^ sw) << 4);
              uint4 pk;
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(pk.x), "=r"(pk.y), "=r"(pk.z), "=r"(pk.w) : "r"(a));
              const float2 r0 = __half22float2(*reinterpret_cast<const __half2*>(&pk.x)), r1 = __half22float2(*reinterpret_cast<const __half2*>(&pk.y));
              const float2 r2 = __half22float2(*reinterpret_cast<const __half2*>(&pk.z)), r3 = __half22float2(*reinterpret_cast<const __half2*>(&pk.w));
              const __half2 o0 = __floats2half2_rn(v[8 * j] + r0.x, v[8 * j + 1] + r0.y), o1 = __floats2half2_rn(v[8 * j + 2] + r1.x, v[8 * j + 3] + r1.y);
              const __half2 o2 = __floats2half2_rn(v[8 * j + 4] + r2.x, v[8 * j + 5] + r2.y), o3 = __floats2half2_rn(v[8 * j + 6] + r3.x, v[8 * j + 7] + r3.y);
              if (p.stats_out != nullptr) {
                const float2 f0 = __half22float2(o0), f1 = __half22float2(o1), f2 = __half22float2(o2), f3 = __half22float2(o3);
                st1 += ((f0.x + f0.y) + (f1.x + f1.y)) + ((f2.x + f2.y) + (f3.x + f3.y));
                st2 += ((f0.x * f0.x + f0.y * f0.y) + (f1.x * f1.x + f1.y * f1.y)) + ((f2.x * f2.x + f2.y * f2.y) + (f3.x * f3.x + f3.y * f3.y));
              }
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(*reinterpret_cast<const uint32_t*>(&o0)),
                           "r"(*reinterpret_cast<const uint32_t*>(&o1)), "r"(*reinterpret_cast<const uint32_t*>(&o2)),
                           "r"(*reinterpret_cast<const uint32_t*>(&o3))
                           : "memory");
            }
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint32_t a = slab0_a + ((uint32_t)b << 12) + rowoff + ((((uint32_t)(h * 4 + j)) ^ sw) << 4);
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(pack_bf16x2(v[8 * j], v[8 * j + 1])),
                           "r"(pack_bf16x2(v[8 * j + 2], v[8 * j + 3])), "r"(pack_bf16x2(v[8 * j + 4], v[8 * j + 5])),
                           "r"(pack_bf16x2(v[8 * j + 6], v[8 * j + 7]))
                           : "memory");
            }
          }
        }
        if (EPI == 2 && p.act == UB_ACT_DOT_AUX) {
          const int row = row0 + lane;
          if (row < p.M && col0 < p.N) {
            const int seq = row / p.dot_seq_len, r = row - seq * p.dot_seq_len;
            p.dot_out[((size_t)seq * (p.N >> 6) + (col0 >> 6)) * p.dot_seq_len + r] = dsum;
          }
        }
        // ---- hand the slab to the TMA engine
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          if (p.accumulate) tma_reduce_add_2d(pC, slab0 + (b << 12), col0, row0);
          else tma_store_2d(pC, slab0 + (b << 12), col0, row0);
          if ((EPI == 0 || EPI == 4) && p.has_aux_out) tma_store_2d(&tmX, slab0 + ((b ^ 1) << 12), col0, row0);
          tma_store_commit();
        }
      }
      if (EPI == 3 && p.stats_out != nullptr && row0 + lane < p.M) {
        atomicAdd(p.stats_out + 2 * (size_t)(row0 + lane), st1);
        atomicAdd(p.stats_out + 2 * (size_t)(row0 + lane) + 1, st2);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (NCTA >= 2) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty[as]), leader_rank)); else mbar_arrive(&tempty[as]);
      }
      as ^= 1;
      if (as == 0) aphase ^= 1;
    }
    if (lane == 0) tma_store_wait_read<0>();   // staging smem must stay valid until the engine has read it
  }

  tc_fence_before();
  if (NCTA >= 2) cluster_sync(); else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if (NCTA >= 2) tmem_dealloc_cg2(tmem_base, TMEM_COLS); else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

template <int BN, int STAGES, bool A_MN, bool B_MN, int EPI, bool OUT32, int NCTA>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmR,
            const __grid_constant__ CUtensorMap tmX, const GemmParams p) {
  gemm_body<BN, STAGES, A_MN, B_MN, EPI, OUT32, NCTA, false>(tmA, tmB, tmC, tmR, tmX, nullptr, p);
}

// Several weight gradients of one backward block in ONE launch (TN, fp32 reduce-add, CTA pairs): dW_i += dY_i^T X_i for up to four
// (dY_i, X_i, dW_i) of different widths over the same tokens.  The four launches it replaces each paid their own prologue /
// pipeline fill / drain (~5 us) and their own wave quantisation on the 74 CTA pairs.
template <int STAGES>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_multi_kernel(const __grid_constant__ GemmMultiMaps mm, const GemmParams p) {
  gemm_body<256, STAGES, true, true, 0, true, 2, true>(mm.a[0], mm.b[0], mm.c[0], mm.c[0], mm.c[0], &mm, p);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  }
  return fn;
}

// 2D row-major tensor [rows, cols] of `esize`-byte elements (2: bf16, 4: fp32) with leading dimension ld (elements);
// box = {box_cols, box_rows}, 128-byte swizzle.  Descriptors are cached: the step re-uses the same buffers every iteration.
struct TmapKey {
  const void* base; int64_t rows, cols, ld; int box_cols, box_rows, esize;
  bool operator==(const TmapKey& o) const {
    return base == o.base && rows == o.rows && cols == o.cols && ld == o.ld && box_cols == o.box_cols && box_rows == o.box_rows &&
           esize == o.esize;
  }
};
struct TmapKeyHash {
  size_t operator()(const TmapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.base);
    auto mix = [&](size_t v) { h ^= v + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2); };
    mix((size_t)k.rows); mix((size_t)k.cols); mix((size_t)k.ld); mix((size_t)k.box_cols * 1024 + k.box_rows * 8 + k.esize);
    return h;
  }
};

int make_tmap_2d(CUtensorMap* out, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_cols, int box_rows,
                 int esize) {
  static std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash> cache;
  static std::mutex mu;
  const TmapKey key{base, rows, cols, ld, box_cols, box_rows, esize};
  {
    std::lock_guard<std::mutex> g(mu);
    auto it = cache.find(key);
    if (it != cache.end()) {
      *out = it->second;
      return 0;
    }
  }
  EncodeTiledFn enc = get_encode_fn();
  UB_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
  UB_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0, "TMA base pointer must be 16-byte aligned");
  UB_REQUIRE((ld * esize) % 16 == 0, "TMA row pitch must be a multiple of 16 bytes (ld=%lld, esize=%d)", (long long)ld, esize);
  UB_REQUIRE(box_cols * esize == 128, "internal: TMA box must span 128 bytes per row");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * esize};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, esize == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base),
                   dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  UB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld cols=%lld ld=%lld box=%dx%d)", (int)r,
             (long long)rows, (long long)cols, (long long)ld, box_cols, box_rows);
  std::lock_guard<std::mutex> g(mu);
  if (cache.size() > 65536) cache.clear();
  cache.emplace(key, *out);
  return 0;
}

struct GemmMaps {
  CUtensorMap a, b, c, r, x;
};

template <int BN, int STAGES, bool A_MN, bool B_MN, int EPI, bool OUT32, int NCTA>
static int launch_gemm_epi(const GemmMaps& m, const GemmParams& p, int grid, cudaStream_t stream) {
  constexpr int SMEM = gemm_smem_bytes(BN, STAGES, NCTA);
  static_assert(SMEM <= 232448, "exceeds the 227 KB per-CTA shared memory limit");
  static bool configured = false;
  auto kern = gemm_kernel<BN, STAGES, A_MN, B_MN, EPI, OUT32, NCTA>;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
    UB_REQUIRE(e == cudaSuccess, "cudaFuncSetAttribute(gemm smem=%d): %s", SMEM, cudaGetErrorString(e));
    configured = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = SMEM;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = NCTA;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, m.a, m.b, m.c, m.r, m.x, p);
  UB_REQUIRE(e == cudaSuccess, "gemm_kernel launch: %s", cudaGetErrorString(e));
  return check_launch("gemm_kernel");
}

// Clusters of 4 must sit inside one GPC: ask the driver how many fit at once (a persistent grid must be co-resident).
static int max_clusters4() {
  static int cached = -1;
  if (cached >= 0) return cached;
  auto kern = gemm_kernel<256, 5, false, false, 0, false, 4>;
  constexpr int SMEM = gemm_smem_bytes(256, 5, 4);
  int n = 0;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM) == cudaSuccess) {
    cudaLaunchConfig_t q{};
    q.gridDim = dim3(sm_count() / 4 * 4);
    q.blockDim = dim3(GEMM_THREADS);
    q.dynamicSmemBytes = SMEM;
    cudaLaunchAttribute qa[1];
    qa[0].id = cudaLaunchAttributeClusterDimension;
    qa[0].val.clusterDim.x = 4; qa[0].val.clusterDim.y = 1; qa[0].val.clusterDim.z = 1;
    q.attrs = qa; q.numAttrs = 1;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &q) != cudaSuccess) n = 0;
  }
  (void)cudaGetLastError();
  cached = n > 0 ? n : 0;
  return cached;
}

// epilogue variants actually used per operand-major combination (keeps the kernel count down):
//   NT   (activations x weights): every variant          NN (dgrad, B = W): bf16 out, plain or DGELU
//   TN   (wgrad, both MN-major) : fp32 out (accumulate)
template <int BN, int STAGES, bool A_MN, bool B_MN, int NCTA>
static int launch_gemm(const GemmMaps& m, const GemmParams& p, int epi, bool out32, int grid, cudaStream_t stream) {
  if constexpr (A_MN) {
    if (epi == 0 && out32) return launch_gemm_epi<BN, STAGES, A_MN, B_MN, 0, true, NCTA>(m, p, grid, stream);
  } else if constexpr (B_MN) {
    if (epi == 0 && !out32) return launch_gemm_epi<BN, STAGES, A_MN, B_MN, 0, false, NCTA>(m, p, grid, stream);
    if (epi == 2) return launch_gemm_epi<BN, STAGES, A_MN, B_MN, 2, false, NCTA>(m, p, grid, stream);
  } else {
    if (epi == 0 && out32) return launch_gemm_epi<BN, STAGES, A_MN, B_MN, 0, true, NCTA>(m, p, grid, stream);
    if (epi == 0 && !out32) return launch_gemm_epi<BN, STAGES, A_MN, B_MN, 0, false, NCTA>(m, p, grid, stream);
    if (epi == 4 && !out32) return launch_gemm_epi<BN, STAGES, A_MN, B_MN, 4, false, NCTA>(m, p, grid, stream);
    if (epi == 1) return launch_gemm_epi<BN, STAGES, A_MN, B_MN, 1, true, NCTA>(m, p, grid, stream);
    if (epi == 2) return launch_gemm_epi<BN, STAGES, A_MN, B_MN, 2, false, NCTA>(m, p, grid, stream);
    if (epi == 3) return launch_gemm_epi<BN, STAGES, A_MN, B_MN, 3, false, NCTA>(m, p, grid, stream);
  }
  set_error("gemm: epilogue variant (epi=%d, fp32 out=%d) is not instantiated for operand majors a_mn=%d b_mn=%d", epi, (int)out32,
            (int)A_MN, (int)B_MN);
  return 1;
}

}  // namespace ub

extern "C" int ub_gemm_cluster4_capacity(void) { return ub::max_clusters4(); }

extern "C" int ub_gemm_wgrad_multi(const ub_gemm_problem* pr, int n, int K, int split_k, void* stream) {
  using namespace ub;
  UB_REQUIRE(pr != nullptr && n >= 1 && n <= GEMM_MAX_PROB, "gemm_wgrad_multi: 1..%d problems expected (got %d)", GEMM_MAX_PROB, n);
  UB_REQUIRE(K > 0, "gemm_wgrad_multi: K=%d", K);
  GemmMultiMaps mm;
  memset(&mm, 0, sizeof(mm));
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.K = K;
  p.accumulate = 1;
  p.n_prob = n;
  int tiles = 0;
  for (int i = 0; i < n; ++i) {
    UB_REQUIRE(pr[i].A && pr[i].B && pr[i].C && pr[i].M > 0 && pr[i].N > 0 && pr[i].N % 8 == 0 && pr[i].M % 8 == 0,
               "gemm_wgrad_multi: problem %d: null operand or bad shape M=%d N=%d", i, pr[i].M, pr[i].N);
    if (make_tmap_2d(&mm.a[i], pr[i].A, K, pr[i].M, pr[i].lda, 64, 64, 2)) return 1;       // dY_i  [K tokens, M_i]  (MN-major A)
    if (make_tmap_2d(&mm.b[i], pr[i].B, K, pr[i].N, pr[i].ldb, 64, 64, 2)) return 1;       // X_i   [K tokens, N_i]  (MN-major B)
    if (make_tmap_2d(&mm.c[i], pr[i].C, pr[i].M, pr[i].N, pr[i].ldc, 32, 32, 4)) return 1;  // dW_i  [M_i, N_i] fp32
    p.tile_off[i] = tiles;
    p.ntile_n[i] = (pr[i].N + 255) / 256;
    tiles += ((pr[i].M + 2 * BM - 1) / (2 * BM)) * p.ntile_n[i];
  }
  for (int i = n; i <= GEMM_MAX_PROB; ++i) p.tile_off[i] = tiles;
  for (int i = n; i < GEMM_MAX_PROB; ++i) { mm.a[i] = mm.a[0]; mm.b[i] = mm.b[0]; mm.c[i] = mm.c[0]; p.ntile_n[i] = 1; }
  p.M = pr[0].M; p.N = pr[0].N;                    // unused by the multi-problem schedule (kept sane)
  const int total_kb = (K + BK - 1) / BK;
  if (split_k < 1) split_k = 1;
  if (split_k > total_kb) split_k = total_kb;
  p.kb_per_split = (total_kb + split_k - 1) / split_k;
  p.splits = (total_kb + p.kb_per_split - 1) / p.kb_per_split;
  const long total_work = (long)tiles * p.splits;
  const int units = sm_count() / 2;
  const int grid = (int)(total_work < units ? total_work : units) * 2;
  constexpr int STAGES = 5;
  constexpr int SMEM = gemm_smem_bytes(256, STAGES, 2);
  static_assert(SMEM <= 232448, "exceeds the 227 KB per-CTA shared memory limit");
  static bool configured = false;
  auto kern = gemm_multi_kernel<STAGES>;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
    UB_REQUIRE(e == cudaSuccess, "cudaFuncSetAttribute(gemm_multi smem=%d): %s", SMEM, cudaGetErrorString(e));
    configured = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = SMEM;
  cfg.stream = reinterpret_cast<cudaStream_t>(stream);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, mm, p);
  UB_REQUIRE(e == cudaSuccess, "gemm_multi_kernel launch: %s", cudaGetErrorString(e));
  return check_launch("gemm_multi_kernel");
}

extern "C" int ub_gemm_bf16(const void* A, int64_t lda, int a_mn_major, const void* B, int64_t ldb, int b_mn_major,
                            void* C, int64_t ldc, int M, int N, int K, const ub_gemm_epilogue* ep_in, int split_k,
                            void* stream) {
  using namespace ub;
  UB_REQUIRE(M > 0 && N > 0 && K > 0, "gemm: empty problem M=%d N=%d K=%d", M, N, K);
  UB_REQUIRE(N % 8 == 0, "gemm: N must be a multiple of 8 (N=%d)", N);
  UB_REQUIRE(A && B && C, "gemm: null operand");
  ub_gemm_epilogue ep;
  if (ep_in) ep = *ep_in; else { memset(&ep, 0, sizeof(ep)); }
  if (split_k < 1) split_k = 1;
  UB_REQUIRE(split_k == 1 || (ep.accumulate && ep.out_fp32), "gemm: split_k>1 needs fp32 accumulate output");
  UB_REQUIRE(!ep.accumulate || ep.out_fp32, "gemm: accumulate needs fp32 output");
  UB_REQUIRE(ep.row_scale == nullptr || ep.rows_per_scale > 0, "gemm: rows_per_scale must be > 0");
  UB_REQUIRE(ep.act != UB_ACT_DGELU || ep.aux_in != nullptr, "gemm: DGELU needs aux_in");
  UB_REQUIRE(ep.act != UB_ACT_DOT_AUX || (ep.aux_in != nullptr && ep.dot_out != nullptr && ep.dot_seq_len > 0 && !ep.out_fp32 && N % 64 == 0 &&
                                          M % ep.dot_seq_len == 0 && ep.residual == nullptr && !ep.accumulate && ep.row_scale == nullptr &&
                                          ep.colsum_out == nullptr && ep.group_rows == 0),
             "gemm: UB_ACT_DOT_AUX needs aux_in, dot_out, dot_seq_len dividing M, a bf16 output with N %% 64 == 0 and no other epilogue option");
  UB_REQUIRE(!(ep.act == UB_ACT_DGELU && ep.residual != nullptr), "gemm: DGELU with a residual is not supported");
  UB_REQUIRE(ep.residual == nullptr || ep.out_fp32 || ep.residual_f16, "gemm: the residual epilogue writes fp32 (or fp16 with residual_f16)");
  UB_REQUIRE(!ep.residual_f16 || (ep.residual != nullptr && !ep.out_fp32), "gemm: residual_f16 needs a residual and a 2-byte (fp16) output");
  UB_REQUIRE((ep.ln_stats == nullptr) == (ep.ln_c == nullptr), "gemm: ln_stats and ln_c go together");
  UB_REQUIRE(ep.ln_stats == nullptr || (ep.residual == nullptr && ep.act != UB_ACT_DGELU && ep.act != UB_ACT_DOT_AUX && !ep.accumulate &&
                                        ep.ln_inv_d > 0.f && N % 4 == 0 && !ep.out_fp32 && !a_mn_major && !b_mn_major),
             "gemm: the LayerNorm fold works with the bias / activation epilogue, K-major operands and a 2-byte output only");
  UB_REQUIRE(ep.stats_out == nullptr || ep.residual_f16, "gemm: stats_out belongs to the fp16-residual epilogue");
  UB_REQUIRE(ep.act != UB_ACT_DGELU || !ep.out_fp32, "gemm: the DGELU epilogue writes bf16");
  UB_REQUIRE(ep.colsum_out == nullptr || ep.act == UB_ACT_DGELU, "gemm: colsum_out belongs to the DGELU epilogue");
  UB_REQUIRE(ep.residual == nullptr || (ep.act == UB_ACT_NONE && !ep.accumulate),
             "gemm: residual cannot be combined with an activation / accumulate");
  UB_REQUIRE(ep.aux_out == nullptr || (ep.act == UB_ACT_GELU && !ep.out_fp32), "gemm: aux_out is the bf16 GELU pre-activation copy");

  const int G = ep.group_rows > 0 ? (M + ep.group_rows - 1) / ep.group_rows : 1;      // groups of a grouped GEMM
  UB_REQUIRE(ep.group_rows >= 0 && (ep.group_rows == 0 || (ep.group_rows % 256 == 0 && M % ep.group_rows == 0)),
             "gemm: group_rows=%d must be a multiple of 256 that divides M=%d", ep.group_rows, M);
  UB_REQUIRE(ep.group_rows > 0 || (ep.group_a_k | ep.group_a_m | ep.group_b_k | ep.group_b_n | ep.group_bias) == 0,
             "gemm: group offsets need group_rows");
  UB_REQUIRE(ep.group_rows == 0 || (ep.residual == nullptr && ep.aux_in == nullptr && ep.aux_out == nullptr && ep.row_scale == nullptr &&
                                    ep.ln_stats == nullptr && ep.stats_out == nullptr && ep.colsum_out == nullptr),
             "gemm: a grouped GEMM supports the bias / accumulate epilogues only");
  UB_REQUIRE(ep.group_rows == 0 || (ep.group_a_k % BK == 0 && ep.group_b_k % BK == 0 && K % BK == 0),
             "gemm: grouped K offsets and K must be multiples of %d", BK);
  const int total_kb = (K + BK - 1) / BK;
  if (split_k > total_kb) split_k = total_kb;
  int kb_per_split = (total_kb + split_k - 1) / split_k;
  split_k = (total_kb + kb_per_split - 1) / kb_per_split;  // no empty splits

  // tile choice: 256-wide tiles unless that costs a whole extra wave; CTA pairs (256 x 256 per pair) for the wide tiles
  const int sms = sm_count();
  static int force_ncta = -1;
  if (force_ncta < 0) {
    const char* e = getenv("UB_GEMM_NCTA");
    force_ncta = e ? atoi(e) : 0;
  }
  // estimated time ~ waves x per-SM tile area / efficiency of the configuration (measured on B200: the 256-wide CTA-pair
  // tile has twice the operand reuse of the 128-wide tile and sustains ~1.3 PF; 1-CTA 256-wide ~1.15 PF; 128-wide ~0.75 PF)
  auto cost = [&](int bm, int bn, int units, double eff) {
    if (eff <= 0.0) return 1e30;
    const long tiles = (long)((M + bm - 1) / bm) * ((N + bn - 1) / bn) * split_k;
    const long waves = (tiles + units - 1) / units;
    return (double)waves * (double)BM * bn / eff;
  };
  const double c128 = cost(BM, 128, sms, 0.58), c256 = cost(BM, 256, sms, 0.88);
  const double c256x2 = M > BM ? cost(2 * BM, 256, sms / 2, 1.0) : 1e30;
  int bn = 256, ncta = 1;
  if (N <= 128 || (c128 < c256 && c128 < c256x2)) bn = 128;
  else if (c256x2 <= c256) ncta = 2;
  // two pairs sharing B by multicast: fewer L2 -> SM bytes per flop, but 512-row work items and whole clusters of 4 SMs
  const int units4 = max_clusters4();
  if (ncta == 2 && M >= 4 * BM && units4 > 0) {
    static double eff4 = -1.0;
    if (eff4 < 0) {
      const char* e = getenv("UB_GEMM_EFF4");
      eff4 = e ? atof(e) : 0.0;
    }
    // measured on B200: 9 % more throughput per SM (25 % fewer L2 -> SM bytes), but only 33 clusters of 4 fit (132 of 148
    // SMs), a net loss of 3 % — so the cost model only picks it when told the per-SM gain (UB_GEMM_EFF4) outweighs that
    if (force_ncta == 4 || (force_ncta == 0 && cost(4 * BM, 256, units4, eff4) < c256x2)) ncta = 4;
  }
  if (force_ncta == 1) ncta = 1;
  if (force_ncta == 2 && bn == 256) ncta = 2;
  static int force_bn = -1;            // experiments: UB_GEMM_BN=128|256 overrides the tile width for every call
  if (force_bn < 0) {
    const char* e = getenv("UB_GEMM_BN");
    force_bn = e ? atoi(e) : 0;
  }
  if (force_bn == 128) { bn = 128; ncta = 1; }
  if (force_bn == 256 && N > 128) bn = 256;
  // per-call hint (beats the environment): used when two GEMMs are run side by side on disjoint sets of SMs
  if (ep.tile_ctas == 1) ncta = 1;
  if (ep.tile_ctas == 2 && bn == 256 && M > BM) ncta = 2;
  if (ep.tile_ctas == 4 && bn == 256 && M >= 4 * BM && units4 > 0) ncta = 4;

  const int epi = ep.residual != nullptr ? (ep.residual_f16 ? 3 : 1)
                                         : ((ep.act == UB_ACT_DGELU || ep.act == UB_ACT_DOT_AUX) ? 2 : (ep.ln_stats != nullptr ? 4 : 0));
  const bool out32 = ep.out_fp32 != 0;
  GemmMaps m;
  memset(&m, 0, sizeof(m));
  // operand extents (a grouped GEMM addresses all groups through one map: the group offsets widen the respective dimension)
  const int64_t a_k_ext = (int64_t)K + (int64_t)(G - 1) * ep.group_a_k, a_m_ext = ep.group_a_m > 0 ? ep.group_a_m : M;
  const int64_t b_k_ext = (int64_t)K + (int64_t)(G - 1) * ep.group_b_k, b_n_ext = (int64_t)N + (int64_t)(G - 1) * ep.group_b_n;
  if (a_mn_major) {
    if (make_tmap_2d(&m.a, A, a_k_ext, a_m_ext, lda, 64, 64, 2)) return 1;
  } else {
    if (make_tmap_2d(&m.a, A, a_m_ext, a_k_ext, lda, BK, BM, 2)) return 1;
  }
  if (b_mn_major) {
    if (make_tmap_2d(&m.b, B, b_k_ext, b_n_ext, ldb, 64, 64, 2)) return 1;
  } else {
    if (make_tmap_2d(&m.b, B, b_n_ext, b_k_ext, ldb, BK, bn / ncta, 2)) return 1;
  }
  if (make_tmap_2d(&m.c, C, M, N, ldc, out32 ? 32 : 64, 32, out32 ? 4 : 2)) return 1;
  m.r = m.c;
  m.x = m.c;
  if (epi == 1 && make_tmap_2d(&m.r, ep.residual, M, N, ep.ldr, 32, 32, 4)) return 1;
  if (epi == 3 && make_tmap_2d(&m.r, ep.residual, M, N, ep.ldr, 64, 32, 2)) return 1;
  if (epi == 2 && make_tmap_2d(&m.r, ep.aux_in, M, N, ep.ld_aux, 64, 32, 2)) return 1;
  if (ep.aux_out != nullptr && make_tmap_2d(&m.x, ep.aux_out, M, N, ep.ld_aux, 64, 32, 2)) return 1;

  GemmParams p;
  p.M = M; p.N = N; p.K = K;
  p.splits = split_k; p.kb_per_split = kb_per_split;
  p.bias = ep.bias; p.row_scale = ep.row_scale; p.rows_per_scale = ep.rows_per_scale;
  p.act = ep.act; p.accumulate = ep.accumulate; p.has_aux_out = ep.aux_out != nullptr;
  p.ab_f16 = ep.ab_f16;
  p.ln_stats = ep.ln_stats; p.ln_c = ep.ln_c; p.ln_inv_d = ep.ln_inv_d; p.ln_eps = ep.ln_eps;
  p.stats_out = ep.stats_out;
  p.colsum_out = ep.colsum_out;
  p.dot_out = ep.dot_out; p.dot_seq_len = ep.dot_seq_len;
  p.group_rows = ep.group_rows; p.a_k_off = ep.group_a_k; p.a_m_off = ep.group_a_m;
  p.b_k_off = ep.group_b_k; p.b_n_off = ep.group_b_n; p.bias_off = ep.group_bias;
  const long total_work = (long)((M + BM * ncta - 1) / (BM * ncta)) * ((N + bn - 1) / bn) * split_k;
  int units = ncta == 4 ? units4 : sms / ncta;
  if (ep.max_ctas > 0 && ep.max_ctas / ncta >= 1 && ep.max_ctas / ncta < units) units = ep.max_ctas / ncta;
  const int grid = (int)(total_work < units ? total_work : units) * ncta;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);

#define UB_GEMM_CASE(AMN, BMN)                                                                       \
  if ((a_mn_major != 0) == AMN && (b_mn_major != 0) == BMN) {                                         \
    if (bn == 256 && ncta == 4) return launch_gemm<256, 5, AMN, BMN, 4>(m, p, epi, out32, grid, st);  \
    if (bn == 256 && ncta == 2) return launch_gemm<256, 5, AMN, BMN, 2>(m, p, epi, out32, grid, st);  \
    return bn == 256 ? launch_gemm<256, 3, AMN, BMN, 1>(m, p, epi, out32, grid, st)                   \
                     : launch_gemm<128, 5, AMN, BMN, 1>(m, p, epi, out32, grid, st);                  \
  }
  UB_GEMM_CASE(false, false)
  UB_GEMM_CASE(false, true)
  UB_GEMM_CASE(true, true)
#undef UB_GEMM_CASE
  set_error("gemm: unsupported operand-major combination a_mn=%d b_mn=%d", a_mn_major, b_mn_major);
  return 1;
}
