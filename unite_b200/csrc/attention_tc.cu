// tcgen05 / TMEM fused attention forward for short sequences (S <= 240, head_dim 64, no LSE): the teacher's
// per-frame 197-token attention (clip.py:40-52, 12 layers x 3072 (frame, head) pairs per step).
//
// One persistent CTA per SM walks (sequence, head) items; per item the whole K and V of the head sit in smem
// (3-D TMA boxes that clip / zero-fill at the SEQUENCE boundary, so padded rows never read the next frame).
//   warp 0      TMA producer, 2-stage ring of {Q, K, V}
//   warp 1      tcgen05.mma issuer:  S_t = Q_t K^T  (128 x NK x 64, SS)  ->  TMEM;   O_t = P_t V (128 x 64 x NK, TS: the
//               A operand P is read straight from TMEM, it never touches smem)
//   warps 2-5   softmax + output of query tile A (rows 0..127), one thread per query row
//   warps 6-9   the same for query tile B (rows 128..255) — the two groups ping-pong on the tensor pipe
// TMEM map per tile (256 columns): S fp32 [0, NK)  ->  P bf16x2 [0, NK/2) overwrites S in place  ->  O fp32 [128, 192),
// row sums of P [192, 208) — produced by the tensor core too (P x ones, N = 16), so the softmax threads spend their
// FP32 issue slots on exactly one max, one FFMA and one ex2 per score.
#include "common.cuh"
#include <mutex>
#include <unordered_map>
#include "../../include/unite_b200.h"

namespace ub {

int make_tmap_3d_bf16(CUtensorMap* out, const void* base, int64_t d2, int64_t d1, int64_t d0, int64_t stride1_elems,
                      int64_t stride2_elems, int box0, int box1);

constexpr int ATC_THREADS = 320;

struct AttnTcParams {
  int n_seq, S, H, NK, n_qt, RB;
  float sl2;          // softmax scale * log2(e)
  uint32_t idesc_s, idesc_o, idesc_r;
};
constexpr int ONES_BYTES = 16 * 4 * 128;   // [16 rows (N)] x [256 keys (K)] bf16, K-major: 4 k-blocks of 16 x 128 B
// register-resident kernels (NKT > 0): the first ATC_NH0 32-key blocks of a score row are turned into P while the rest is still
// being read; their P lives in the tile's spare columns [NKT, NKT + 16 * ATC_NH0) instead of over the scores
constexpr int ATC_NH0(int nkt) { return (nkt / 32) / 2; }
// TMEM column (within the tile) of the bf16 P operand of key step k (16 keys = 8 columns)
UB_DEVINL constexpr uint32_t atc_p_col(int nkt, int k) { return nkt > 0 && k < 2 * ATC_NH0(nkt) ? (uint32_t)(nkt + k * 8) : (uint32_t)(k * 8); }

// NKT == 0: generic (runtime NK, two TMEM passes over S, 10 warps).
// NKT  > 0: NK == NKT at compile time; each softmax thread keeps its whole score row (NKT fp32) in REGISTERS, so S is read
//           from TMEM once (TMEM reads, ~64 B/clk/SM, are what bounds this kernel).  Needs 232 registers per softmax thread:
//           12 warps in warpgroup-aligned roles (WG0 = TMA + MMA (+2 idle warps), WG1 / WG2 = softmax of tile A / B) and
//           setmaxnreg to move registers from WG0 to the softmax warpgroups.
template <int NKT>
__global__ void __launch_bounds__(NKT ? 384 : ATC_THREADS, 1)
attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                   const __grid_constant__ CUtensorMap tmO, const AttnTcParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int q_bytes = p.RB * 128;                  // Q of a head: RB rows x 64 bf16 (both query tiles)
  const int kv_bytes = p.NK * 128;                 // K or V of a head: NK rows (keys padded to 16; multiple of 1 KB)
  const int stage_bytes = q_bytes + 2 * kv_bytes;
  uint8_t* o_stage = smem + 2 * stage_bytes;       // 8 warps x 4 KB
  uint8_t* ones_s = o_stage + 8 * 4096;            // constant B operand of the row-sum MMA
  uint64_t* kv_full = reinterpret_cast<uint64_t*>(ones_s + ONES_BYTES);
  uint64_t* kv_empty = kv_full + 2;
  uint64_t* s_full = kv_empty + 2;
  uint64_t* p_ready = s_full + 2;
  uint64_t* o_full = p_ready + 2;
  uint64_t* s_free = o_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_free + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmKV);
    tma_prefetch_desc(&tmO);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], NKT ? 2 : 1);   // one commit per MMA-issuer warp
      mbar_init(&s_full[i], 1);
      mbar_init(&p_ready[i], 4);
      mbar_init(&o_full[i], 1);
      mbar_init(&s_free[i], 4);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  // ones tile: every element 1.0 (bf16 0x3F80) — the swizzle is irrelevant for a constant
  for (int i = threadIdx.x; i < ONES_BYTES / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(ones_s)[i] = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int n_items = p.n_seq * p.H;
  constexpr int SM_WARP0 = NKT ? 4 : 2;    // first softmax warp

  if (warp < SM_WARP0) {
  if (NKT) asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");   // whole warpgroup 0 (TMA, MMA, 2 idle warps)
  if (warp == 0) {
    // ---------------------------------------------------------------- TMA producer
    int it = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
      const int st = it & 1, seq = item / p.H, h = item % p.H;
      mbar_wait(&kv_empty[st], ((it >> 1) & 1) ^ 1);
      if (lane == 0) {
        uint8_t* sQ = smem + st * stage_bytes;
        mbar_expect_tx(&kv_full[st], stage_bytes);
        tma_load_3d(&tmQ, &kv_full[st], sQ, h * 64, 0, seq);
        tma_load_3d(&tmKV, &kv_full[st], sQ + q_bytes, (p.H + h) * 64, 0, seq);
        tma_load_3d(&tmKV, &kv_full[st], sQ + q_bytes + kv_bytes, (2 * p.H + h) * 64, 0, seq);
      }
      __syncwarp();
    }
  } else if (warp == 1 || (NKT && warp == 2)) {
    // ---------------------------------------------------------------- MMA issuer(s): NKT kernels run one in-order
    // issue stream PER query tile (warp 1: tile A, warp 2: tile B) so a wait of one tile never blocks the other
    const int t_lo = NKT ? warp - 1 : 0, t_hi = NKT ? warp : p.n_qt;
    int it = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
      const int st = it & 1;
      const uint32_t sQ = smem_u32(smem + st * stage_bytes);
      const uint32_t sK = sQ + q_bytes, sV = sK + kv_bytes;
      const uint32_t sOnes = smem_u32(ones_s);
      mbar_wait(&kv_full[st], (it >> 1) & 1);
      tc_fence_after();
      for (int t = t_lo; t < t_hi; ++t) {
        mbar_wait(&s_free[t], (it & 1) ^ 1);
        tc_fence_after();
        if (lane == 0) {
          const uint64_t qd = umma_desc_kmajor_sw128(sQ + t * 16384), kd = umma_desc_kmajor_sw128(sK);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16(tmem_base + t * 256, qd + k * 2, kd + k * 2, p.idesc_s, k > 0 ? 1u : 0u);
          umma_commit(&s_full[t]);
        }
        __syncwarp();
      }
      for (int t = t_lo; t < t_hi; ++t) {
        mbar_wait(&p_ready[t], it & 1);
        tc_fence_after();
        if (lane == 0) {
          const uint64_t vd = umma_desc_mnmajor_sw128(sV, 8192);
          const int ksteps = (NKT ? NKT : p.NK) >> 4;
          for (int k = 0; k < ksteps; ++k)
            umma_bf16_ts(tmem_base + t * 256 + 128, tmem_base + t * 256 + atc_p_col(NKT, k), vd + (uint64_t)(k * 128), p.idesc_o, k > 0 ? 1u : 0u);
          // row sums of the bf16 P actually used above:  P (128 x NK) x ones (NK x 16)
          const uint64_t od = umma_desc_kmajor_sw128(sOnes);
          for (int k = 0; k < ksteps; ++k)
            umma_bf16_ts(tmem_base + t * 256 + 192, tmem_base + t * 256 + atc_p_col(NKT, k), od + (uint64_t)((k >> 2) * 128 + (k & 3) * 2), p.idesc_r,
                         k > 0 ? 1u : 0u);
          umma_commit(&o_full[t]);
          if (t == t_hi - 1) umma_commit(&kv_empty[st]);   // every MMA of this stream has read the item's smem
        }
        __syncwarp();
      }
    }
  }
  } else {
    // ---------------------------------------------------------------- softmax + output, one thread per query row
    if (NKT) asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    const int we = warp - SM_WARP0;
    const int t = we >> 2;                 // query tile of this warpgroup
    const int sp = warp & 3;               // TMEM sub-partition
    const uint32_t t_row = tmem_base + ((uint32_t)(sp * 32) << 16) + (uint32_t)(t * 256);
    uint8_t* stg = o_stage + we * 4096;
    const uint32_t stg_a = smem_u32(stg);
    const int row0 = t * 128 + sp * 32;    // first query row (within the sequence) of this warp
    const int S = p.S, NK = NKT ? NKT : p.NK;
    const float sl2 = p.sl2;
    if (t < p.n_qt) {
      int it = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
        const int seq = item / p.H, h = item % p.H;
        if (NKT && t == 1 && it == 0) asm volatile("bar.arrive 2, 256;" ::: "memory");   // warpgroup A goes first
        mbar_wait(&s_full[t], it & 1);
        tc_fence_after();
        if constexpr (NKT > 0) {
          // ---- single pass: every score is read from TMEM once (S > NKT - 16 by construction: only the last 16 need masks).
          // The row is fetched in two halves: the second half is in flight on the TMEM read port while the first half is in
          // the exponentials, which takes the load time of half a row out of the tile's QK^T -> softmax -> PV dependency chain
          // (that chain, not a throughput limit, is what bounds this kernel: profiles/ncu_attn_r01b_pingpong.txt).  The softmax
          // reference is the maximum of the FIRST half: O / l is invariant under the common factor, so the result is exact; only
          // if the second half exceeds it by more than 2^60 are the first half's exponentials redone against the true maximum.
          // P of the first half goes to the 48 spare columns [208, 256) of the tile, so its scores stay intact in TMEM for that
          // redo and their registers are free while the second half is processed.
          constexpr int NFULL = NKT / 32, TAIL = NKT % 32;
          constexpr int NH0 = ATC_NH0(NKT);                 // 32-column loads of the first half
          static_assert(TAIL == 0 || TAIL == 16, "NKT must be a multiple of 16");
          static_assert(NH0 * 32 <= NKT - 16 && NKT + NH0 * 16 <= 256, "first half: unmasked, and its P must fit the spare columns");
          float mb1;
          auto exp32 = [&](const uint32_t (&v)[32], int c) {         // keys [32 c, 32 c + 32) -> bf16 P
            uint32_t pk[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int k0 = c * 32 + 2 * i;
              float p0 = fast_exp2(fmaf(__uint_as_float(v[2 * i]), sl2, -mb1));
              float p1 = fast_exp2(fmaf(__uint_as_float(v[2 * i + 1]), sl2, -mb1));
              if (k0 >= NKT - 16) {
                if (k0 >= S) p0 = 0.f;
                if (k0 + 1 >= S) p1 = 0.f;
              }
              pk[i] = pack_bf16x2(p0, p1);
            }
            tmem_st_32x16(t_row + (c < NH0 ? NKT + c * 16 : c * 16), pk);
          };
          uint32_t s0[NH0][32], s1[NFULL - NH0][32], s1t[16];
#pragma unroll
          for (int c = 0; c < NH0; ++c) tmem_ld_32x32(t_row + c * 32, s0[c]);
          tmem_ld_wait();
#pragma unroll
          for (int c = NH0; c < NFULL; ++c) tmem_ld_32x32(t_row + c * 32, s1[c - NH0]);     // in flight during the exponentials below
          if constexpr (TAIL) tmem_ld_32x16(t_row + NFULL * 32, s1t);
          float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
          for (int c = 0; c < NH0; ++c)
#pragma unroll
            for (int i = 0; i < 32; ++i) m4[i & 3] = fmaxf(m4[i & 3], __uint_as_float(s0[c][i]));
          const float m0 = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
          mb1 = m0 * sl2;
          // ping-pong: the exp phases of the two warpgroups alternate (each gets the full MUFU rate while the other one
          // waits on / feeds the tensor pipe).  Named barriers 2 (A's turn) and 3 (B's turn), 256 threads each.
          if (t == 0) asm volatile("bar.sync 2, 256;" ::: "memory"); else asm volatile("bar.sync 3, 256;" ::: "memory");
#pragma unroll
          for (int c = 0; c < NH0; ++c) exp32(s0[c], c);
          tmem_ld_wait();                                   // the second half has landed
          float n4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
          for (int c = NH0; c < NFULL; ++c)
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              if (c * 32 + i < NKT - 16 || c * 32 + i < S) n4[i & 3] = fmaxf(n4[i & 3], __uint_as_float(s1[c - NH0][i]));
            }
          if constexpr (TAIL) {
#pragma unroll
            for (int i = 0; i < 16; ++i)
              if (NFULL * 32 + i < S) n4[i & 3] = fmaxf(n4[i & 3], __uint_as_float(s1t[i]));
          }
          const float m1 = fmaxf(fmaxf(n4[0], n4[1]), fmaxf(n4[2], n4[3]));
          if (__any_sync(0xffffffffu, (m1 - m0) * sl2 > 60.0f)) {
            // rare: redo the first half against the true maximum, one 32-key block at a time from its intact scores
            mb1 = fmaxf(m0, m1) * sl2;
#pragma unroll 1
            for (int c = 0; c < NH0; ++c) {
              uint32_t r[32], pk[16];
              tmem_ld_32x32(t_row + c * 32, r);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 16; ++i)
                pk[i] = pack_bf16x2(fast_exp2(fmaf(__uint_as_float(r[2 * i]), sl2, -mb1)), fast_exp2(fmaf(__uint_as_float(r[2 * i + 1]), sl2, -mb1)));
              tmem_st_32x16(t_row + NKT + c * 16, pk);
            }
          }
#pragma unroll
          for (int c = NH0; c < NFULL; ++c) exp32(s1[c - NH0], c);
          if constexpr (TAIL) {
            uint32_t pk[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int k0 = NFULL * 32 + 2 * i;
              const float p0 = (k0 < S) ? fast_exp2(fmaf(__uint_as_float(s1t[2 * i]), sl2, -mb1)) : 0.f;
              const float p1 = (k0 + 1 < S) ? fast_exp2(fmaf(__uint_as_float(s1t[2 * i + 1]), sl2, -mb1)) : 0.f;
              pk[i] = pack_bf16x2(p0, p1);
            }
            tmem_st_32x8(t_row + NFULL * 16, pk);
          }
          if (t == 0) asm volatile("bar.arrive 3, 256;" ::: "memory"); else asm volatile("bar.arrive 2, 256;" ::: "memory");
        } else {
        // ---- pass 1: row maximum over the valid keys (only the chunk that straddles S pays for masking)
        float mx = -INFINITY;
        for (int kb = 0; kb < NK; kb += 32) {
          if (kb + 32 <= NK) {
            uint32_t r[32];
            tmem_ld_32x32(t_row + kb, r);
            tmem_ld_wait();
            if (kb + 32 <= S) {
              float m4[4] = {mx, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
              for (int i = 0; i < 32; ++i) m4[i & 3] = fmaxf(m4[i & 3], __uint_as_float(r[i]));
              mx = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i)
                if (kb + i < S) mx = fmaxf(mx, __uint_as_float(r[i]));
            }
          } else {
            uint32_t r[16];
            tmem_ld_32x16(t_row + kb, r);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i)
              if (kb + i < S) mx = fmaxf(mx, __uint_as_float(r[i]));
          }
        }
        const float mb = mx * sl2;
        // ---- pass 2: P = exp2(s*sl2 - mb) -> bf16x2 back into TMEM (columns kb/2 ..); the row sum comes from the MMA
        for (int kb = 0; kb < NK; kb += 32) {
          if (kb + 32 <= NK) {
            uint32_t r[32], pk[16];
            tmem_ld_32x32(t_row + kb, r);
            tmem_ld_wait();
            if (kb + 32 <= S) {
#pragma unroll
              for (int i = 0; i < 16; ++i)
                pk[i] = pack_bf16x2(fast_exp2(fmaf(__uint_as_float(r[2 * i]), sl2, -mb)),
                                    fast_exp2(fmaf(__uint_as_float(r[2 * i + 1]), sl2, -mb)));
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float p0 = (kb + 2 * i < S) ? fast_exp2(fmaf(__uint_as_float(r[2 * i]), sl2, -mb)) : 0.f;
                const float p1 = (kb + 2 * i + 1 < S) ? fast_exp2(fmaf(__uint_as_float(r[2 * i + 1]), sl2, -mb)) : 0.f;
                pk[i] = pack_bf16x2(p0, p1);
              }
            }
            tmem_st_32x16(t_row + (kb >> 1), pk);
          } else {
            uint32_t r[16], pk[8];
            tmem_ld_32x16(t_row + kb, r);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float p0 = (kb + 2 * i < S) ? fast_exp2(fmaf(__uint_as_float(r[2 * i]), sl2, -mb)) : 0.f;
              const float p1 = (kb + 2 * i + 1 < S) ? fast_exp2(fmaf(__uint_as_float(r[2 * i + 1]), sl2, -mb)) : 0.f;
              pk[i] = pack_bf16x2(p0, p1);
            }
            tmem_st_32x8(t_row + (kb >> 1), pk);
          }
        }
        }   // generic two-pass path
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&p_ready[t]);
        // ---- O = (P V) / rowsum -> bf16 -> smem slab -> TMA store clipped at the sequence end
        if (lane == 0) tma_store_wait_read<0>();   // the slab of the previous item has been read
        __syncwarp();
        mbar_wait(&o_full[t], it & 1);
        tc_fence_after();
        // all of O (64 fp32 per row) and the row sum are taken out of TMEM first, so the tile's columns go back to the MMA warp
        // (next item's Q K^T) before the normalise / pack / staging work instead of after it
        uint32_t rsum, r0[32], r1[32];
        tmem_ld_32x1(t_row + 192, rsum);
        tmem_ld_32x32(t_row + 128, r0);
        tmem_ld_32x32(t_row + 160, r1);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&s_free[t]);            // S / P / O columns of this tile may be overwritten by the next item
        const float inv = 1.0f / __uint_as_float(rsum);
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const uint32_t* r = hh ? r1 : r0;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t a = stg_a + (uint32_t)lane * 128u + ((((uint32_t)(hh * 4 + j)) ^ (uint32_t)(lane & 7)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a),
                         "r"(pack_bf16x2(__uint_as_float(r[8 * j]) * inv, __uint_as_float(r[8 * j + 1]) * inv)),
                         "r"(pack_bf16x2(__uint_as_float(r[8 * j + 2]) * inv, __uint_as_float(r[8 * j + 3]) * inv)),
                         "r"(pack_bf16x2(__uint_as_float(r[8 * j + 4]) * inv, __uint_as_float(r[8 * j + 5]) * inv)),
                         "r"(pack_bf16x2(__uint_as_float(r[8 * j + 6]) * inv, __uint_as_float(r[8 * j + 7]) * inv))
                         : "memory");
          }
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0 && row0 < S) {
          tma_store_3d(&tmO, stg, h * 64, row0, seq);
          tma_store_commit();
        }
      }
      if (lane == 0) tma_store_wait_read<0>();
      // balance the ping-pong: B's last hand-over to A has no taker
      if (NKT && t == 0 && blockIdx.x < n_items) asm volatile("bar.sync 2, 256;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---- 3-D tensor maps (bf16, 128-byte swizzle), cached ---------------------------------------------------------
typedef CUresult (*EncodeTiledFn3)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
struct Key3 {
  const void* base; int64_t d2, d1, d0, s1, s2; int b0, b1;
  bool operator==(const Key3& o) const {
    return base == o.base && d2 == o.d2 && d1 == o.d1 && d0 == o.d0 && s1 == o.s1 && s2 == o.s2 && b0 == o.b0 && b1 == o.b1;
  }
};
struct Key3Hash {
  size_t operator()(const Key3& k) const {
    size_t h = reinterpret_cast<size_t>(k.base);
    auto mix = [&](size_t v) { h ^= v + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2); };
    mix((size_t)k.d2); mix((size_t)k.d1); mix((size_t)k.d0); mix((size_t)k.s1); mix((size_t)k.s2); mix((size_t)k.b0 * 4096 + k.b1);
    return h;
  }
};

// tensor [d2][d1][d0] (d0 contiguous), strides in elements; box {b0, b1, 1}
int make_tmap_3d_bf16(CUtensorMap* out, const void* base, int64_t d2, int64_t d1, int64_t d0, int64_t stride1_elems,
                      int64_t stride2_elems, int box0, int box1) {
  static std::unordered_map<Key3, CUtensorMap, Key3Hash> cache;
  static std::mutex mu;
  static EncodeTiledFn3 enc = nullptr;
  const Key3 key{base, d2, d1, d0, stride1_elems, stride2_elems, box0, box1};
  {
    std::lock_guard<std::mutex> g(mu);
    auto it = cache.find(key);
    if (it != cache.end()) {
      *out = it->second;
      return 0;
    }
  }
  if (enc == nullptr) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      enc = reinterpret_cast<EncodeTiledFn3>(sym);
  }
  UB_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is not available from the driver");
  UB_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0 && (stride1_elems * 2) % 16 == 0 && (stride2_elems * 2) % 16 == 0,
             "3-D TMA map: base and strides must be 16-byte aligned");
  cuuint64_t dims[3] = {(cuuint64_t)d0, (cuuint64_t)d1, (cuuint64_t)d2};
  cuuint64_t strides[2] = {(cuuint64_t)stride1_elems * 2, (cuuint64_t)stride2_elems * 2};
  cuuint32_t box[3] = {(cuuint32_t)box0, (cuuint32_t)box1, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  UB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (3-D) failed with CUresult %d", (int)r);
  std::lock_guard<std::mutex> g(mu);
  if (cache.size() > 65536) cache.clear();
  cache.emplace(key, *out);
  return 0;
}

// used by ub_attn_fwd (attention.cu) when S <= 240 and no LSE is requested
int launch_attn_fwd_tc(const void* qkv, void* o, int n_seq, int S, int H, float scale, cudaStream_t stream) {
  AttnTcParams p;
  p.n_seq = n_seq; p.S = S; p.H = H;
  p.NK = (S + 15) / 16 * 16;
  p.n_qt = (S + 127) / 128;
  p.RB = S > 128 ? 256 : 128;
  p.sl2 = scale * 1.4426950408889634f;
  p.idesc_s = umma_idesc_bf16(128, p.NK, 0, 0);
  p.idesc_o = umma_idesc_bf16(128, 64, 0, 1);
  p.idesc_r = umma_idesc_bf16(128, 16, 0, 0);
  CUtensorMap tq, tkv, to;
  const int64_t ld = 3 * (int64_t)H * 64, ldo = (int64_t)H * 64;
  if (make_tmap_3d_bf16(&tq, qkv, n_seq, S, ld, ld, (int64_t)S * ld, 64, p.RB)) return 1;
  if (make_tmap_3d_bf16(&tkv, qkv, n_seq, S, ld, ld, (int64_t)S * ld, 64, p.NK)) return 1;
  if (make_tmap_3d_bf16(&to, o, n_seq, S, ldo, ldo, (int64_t)S * ldo, 64, 32)) return 1;
  const int smem = 2 * (p.RB * 128 + 2 * p.NK * 128) + 8 * 4096 + ONES_BYTES + 12 * 8 + 16;
  const int items = n_seq * H;
  const int grid = items < sm_count() ? items : sm_count();
  if (p.NK == 208) {  // the teacher's 197-token frames (224^2 / 16^2 patches + CLS)
    static int configured208 = 0;
    if (configured208 < smem) {
      cudaError_t e = cudaFuncSetAttribute(attn_fwd_tc_kernel<208>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
      UB_REQUIRE(e == cudaSuccess, "cudaFuncSetAttribute(attn_fwd_tc<208> smem=%d): %s", smem, cudaGetErrorString(e));
      configured208 = smem;
    }
    UB_LAUNCH(attn_fwd_tc_kernel<208>, grid, 384, smem, stream, tq, tkv, to, p);
    return check_launch("attn_fwd_tc_kernel<208>");
  }
  static int configured = 0;
  if (configured < smem) {
    cudaError_t e = cudaFuncSetAttribute(attn_fwd_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    UB_REQUIRE(e == cudaSuccess, "cudaFuncSetAttribute(attn_fwd_tc smem=%d): %s", smem, cudaGetErrorString(e));
    configured = smem;
  }
  UB_LAUNCH(attn_fwd_tc_kernel<0>, grid, ATC_THREADS, smem, stream, tq, tkv, to, p);
  return check_launch("attn_fwd_tc_kernel");
}

}  // namespace ub
