// tcgen05 / TMEM attention FORWARD WITH LOG-SUM-EXP for sequences of up to 320 tokens (head_dim 64): the student's
// visible-token attention in training (modeling_finetune.py:100-119; 12 layers x 384 (clip, head) pairs x 3 query tiles).
//
// Persistent CTA per SM.  Query tiles (128 rows) of consecutive (sequence, head) items form one flat stream; tile n belongs
// to warpgroup n & 1, so the two warpgroups ping-pong on the tensor pipe / TMEM port / MUFU.  The keys of an item are taken in
// two chunks of 160 (S^T never needs more than 160 TMEM columns):
//     S_c = Q K_c^T              (SS, M = 128 queries, N = 160, K = 64)  ->  TMEM, read ONCE into registers (160 fp32 / thread)
//     P_c = exp2(S_c * scale*log2e - ref)   bf16 back into TMEM over S_c;   O (+)= P_c V_c,  l (+)= P_c 1   (TS MMAs)
// `ref` is the row maximum of the FIRST chunk.  The second chunk reuses it (mathematically exact: O / l is invariant under a
// common factor), so O is never rescaled in the common case; only if a row's second-chunk maximum exceeds ref by more than 2^64
// does the warp take the slow path (wait for P_a V_a, scale its O / l rows in TMEM by 2^(ref - new), move ref).
//   warp 0        TMA producer: K/V of the item (2-slot ring, next item prefetched), Q tile of each warpgroup
//   warps 1, 2    tcgen05.mma issue streams of warpgroup 0 / 1 (in-order per warpgroup, never blocking each other)
//   warps 4-7     warpgroup 0: softmax + output + LSE of its tiles, one thread per query row;   warps 8-11: warpgroup 1
// TMEM per warpgroup (256 columns): S / P [0,160) | O [160,224) | l [224,240).
// smem: K/V ring 2 x 80 KB | Q 2 x 16 KB | output staging 8 warps x 4 KB | ones tile 2 KB.
#include "common.cuh"
#include <cstdlib>
#include "../../include/unite_b200.h"

namespace ub {

int make_tmap_3d_bf16(CUtensorMap* out, const void* base, int64_t d2, int64_t d1, int64_t d0, int64_t stride1_elems,
                      int64_t stride2_elems, int box0, int box1);

constexpr int AFL_THREADS = 384;
constexpr int AFL_NKC = 160;                      // keys per chunk
constexpr int AFL_KV = 0;                         // 2 slots x {K [320][64], V [320][64]}
constexpr int AFL_Q = 163840;                     // 2 x [128][64]
constexpr int AFL_OUT = AFL_Q + 32768;            // 8 warps x 4 KB
constexpr int AFL_ONES = AFL_OUT + 32768;         // [16 rows][64] bf16 ones (B operand of the row-sum MMA, any k-step)
constexpr int AFL_BAR = AFL_ONES + 2048;
constexpr int AFL_NBAR = 20;
constexpr int AFL_SMEM = AFL_BAR + AFL_NBAR * 8 + 16;

struct AttnFwdLseParams {
  float* lse;
  int n_seq, S, H, nt, nch;      // nt query tiles per item, nch key chunks (1 or 2)
  float sl2, scale;
};

__global__ void __launch_bounds__(AFL_THREADS, 1)
attn_fwd_lse_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                       const __grid_constant__ CUtensorMap tmO, const AttnFwdLseParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + AFL_BAR);
  uint64_t* kv_full = bars;          // [2]
  uint64_t* kv_empty = bars + 2;     // [2] count nt: every tile's MMA stream has read the slot
  uint64_t* q_full = bars + 4;       // [2] per warpgroup
  uint64_t* q_empty = bars + 6;      // [2] the tile's S MMAs are done with Q
  uint64_t* s_full = bars + 8;       // [2] one completion per (tile, chunk)
  uint64_t* p_ready = bars + 10;     // [2]
  uint64_t* o_full = bars + 12;      // [2] per tile
  uint64_t* pv_done = bars + 14;     // [2] per tile: P_a V_a has completed (slow path only waits on it)
  uint64_t* s_free = bars + 16;      // [2] O / l of the tile have been read
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + AFL_NBAR);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmKV);
    tma_prefetch_desc(&tmO);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], p.nt);
      mbar_init(&q_full[i], 1);
      mbar_init(&q_empty[i], 1);        // commit behind the tile's last S MMA
      mbar_init(&s_full[i], 1);
      mbar_init(&p_ready[i], 4);
      mbar_init(&o_full[i], 1);
      mbar_init(&pv_done[i], 1);
      mbar_init(&s_free[i], 4);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < 2048 / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(smem + AFL_ONES)[i] = make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int n_items = p.n_seq * p.H;
  const int nt = p.nt, nch = p.nch;

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp == 0) {
      // ------------------------------------------------------------------------------------------ TMA producer
      if (lane == 0) {
        auto load_kv = [&](int it, int item) {
          const int slot = it & 1, seq = item / p.H, h = item % p.H;
          mbar_wait(&kv_empty[slot], ((it >> 1) & 1) ^ 1);
          uint8_t* dst = smem + AFL_KV + slot * 81920;
          mbar_expect_tx(&kv_full[slot], (uint32_t)nch * 40960u);
          for (int c = 0; c < nch; ++c) {
            tma_load_3d(&tmKV, &kv_full[slot], dst + c * 20480, (p.H + h) * 64, c * AFL_NKC, seq);
            tma_load_3d(&tmKV, &kv_full[slot], dst + 40960 + c * 20480, (2 * p.H + h) * 64, c * AFL_NKC, seq);
          }
        };
        int it = 0;
        uint32_t n = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
          const int seq = item / p.H, h = item % p.H;
          if (it == 0) load_kv(0, item);
          for (int t = 0; t < nt; ++t, ++n) {
            const uint32_t g = n & 1u, j = n >> 1;
            mbar_wait(&q_empty[g], (j & 1u) ^ 1u);
            mbar_expect_tx(&q_full[g], 16384);
            tma_load_3d(&tmQ, &q_full[g], smem + AFL_Q + g * 16384, h * 64, t * 128, seq);
            if (t == (nt > 1 ? 1 : 0) && item + (int)gridDim.x < n_items) load_kv(it + 1, item + gridDim.x);
          }
        }
      }
    } else if (warp <= 2) {
      // ------------------------------------------------------------------------------------------ MMA issue stream of warpgroup g
      const uint32_t g = (uint32_t)(warp - 1);
      constexpr uint32_t IDESC_S = umma_idesc_bf16(128, AFL_NKC, 0, 0);
      constexpr uint32_t IDESC_O = umma_idesc_bf16(128, 64, 0, 1);
      constexpr uint32_t IDESC_R = umma_idesc_bf16(128, 16, 0, 0);
      constexpr uint32_t HI = (1024u >> 4) | (1u << 14) | (2u << 29);
      constexpr uint32_t LO_K = 1u << 16, LO_MN = (8192u >> 4) << 16;
      const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0) + g * 256u;
      const uint32_t aQ = ((smem_u32(smem + AFL_Q) & 0x3FFFFu) >> 4) + g * 1024u;
      const uint32_t aKV = (smem_u32(smem + AFL_KV) & 0x3FFFFu) >> 4, aOnes = (smem_u32(smem + AFL_ONES) & 0x3FFFFu) >> 4;
      int it = 0;
      uint32_t n = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
        const uint32_t slot = it & 1u;
        const uint32_t aK = aKV + slot * 5120u, aV = aK + 2560u;
        for (int t = 0; t < nt; ++t, ++n) {
          if ((n & 1u) != g) continue;
          const uint32_t j = n >> 1;
          mbar_wait(&kv_full[slot], (it >> 1) & 1);
          mbar_wait(&q_full[g], j & 1u);
          mbar_wait(&s_free[g], (j & 1u) ^ 1u);
          tc_fence_after();
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_ss_lo(tb, aQ + LO_K + k * 2, HI, aK + LO_K + k * 2, HI, IDESC_S, k > 0);
            umma_commit(&s_full[g]);
            if (nch == 1) umma_commit(&q_empty[g]);
          }
          __syncwarp();
          for (int c = 0; c < nch; ++c) {
            mbar_wait(&p_ready[g], (j * (uint32_t)nch + (uint32_t)c) & 1u);
            tc_fence_after();
            if (elect_one()) {
              const uint32_t vd = aV + (uint32_t)c * 1280u + LO_MN;
#pragma unroll
              for (int k = 0; k < AFL_NKC / 16; ++k) umma_ts_lo(tb + 160, tb + k * 8, vd + k * 128, HI, IDESC_O, c > 0 || k > 0);
#pragma unroll
              for (int k = 0; k < AFL_NKC / 16; ++k) umma_ts_lo(tb + 224, tb + k * 8, aOnes + LO_K, HI, IDESC_R, c > 0 || k > 0);
              if (c + 1 < nch) {
                umma_commit(&pv_done[g]);
                const uint32_t kd = aK + 1280u + LO_K;
#pragma unroll
                for (int k = 0; k < 4; ++k) umma_ss_lo(tb, aQ + LO_K + k * 2, HI, kd + k * 2, HI, IDESC_S, k > 0);
                umma_commit(&s_full[g]);
                umma_commit(&q_empty[g]);
              } else {
                umma_commit(&o_full[g]);
                umma_commit(&kv_empty[slot]);
              }
            }
            __syncwarp();
          }
        }
      }
    }
  } else {
    // ------------------------------------------------------------------------------------------ softmax / output warpgroups
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    const uint32_t g = (uint32_t)((warp - 4) >> 2);
    const int sp = warp & 3;
    const uint32_t t_row = tmem_base + ((uint32_t)(sp * 32) << 16) + g * 256u;
    uint8_t* stg = smem + AFL_OUT + (warp - 4) * 4096;
    const uint32_t stg_a = smem_u32(stg);
    const uint32_t sw = (uint32_t)(lane & 7);
    const float sl2 = p.sl2;
    // ping-pong: the exp / P-store phases of the two warpgroups strictly alternate (named barriers 2 = A's turn, 3 = B's turn,
    // 256 threads each), so one warpgroup has the MUFU while the other one is on the TMEM read port / waits for the tensor pipe
    auto my_turn = [&]() {
      if (g == 0) asm volatile("bar.sync 2, 256;" ::: "memory"); else asm volatile("bar.sync 3, 256;" ::: "memory");
    };
    auto pass_turn = [&]() {
      if (g == 0) asm volatile("bar.arrive 3, 256;" ::: "memory"); else asm volatile("bar.arrive 2, 256;" ::: "memory");
    };
    if (g == 1) asm volatile("bar.arrive 2, 256;" ::: "memory");      // warpgroup A goes first
    int it = 0;
    uint32_t n = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
      const int seq = item / p.H, h = item % p.H;
      for (int t = 0; t < nt; ++t, ++n) {
        if ((n & 1u) != g) continue;
        const uint32_t j = n >> 1;
        float ref = 0.f;                 // reference maximum (raw score units) of this row
        for (int c = 0; c < nch; ++c) {
          const int kvalid = min(AFL_NKC, p.S - c * AFL_NKC);       // valid keys of this chunk (> 0 by construction)
          mbar_wait(&s_full[g], (j * (uint32_t)nch + (uint32_t)c) & 1u);
          tc_fence_after();
          uint32_t sv[AFL_NKC];
#pragma unroll
          for (int q = 0; q < AFL_NKC / 32; ++q) tmem_ld_32x32(t_row + q * 32, *reinterpret_cast<uint32_t(*)[32]>(&sv[q * 32]));
          tmem_ld_wait();
          float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
          if (kvalid == AFL_NKC) {
#pragma unroll
            for (int i = 0; i < AFL_NKC; ++i) m4[i & 3] = fmaxf(m4[i & 3], __uint_as_float(sv[i]));
          } else {
#pragma unroll
            for (int i = 0; i < AFL_NKC; ++i)
              if (i < kvalid) m4[i & 3] = fmaxf(m4[i & 3], __uint_as_float(sv[i]));
          }
          const float mx = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
          if (c == 0) {
            ref = mx;
          } else if (__any_sync(0xffffffffu, (mx - ref) * sl2 > 64.0f)) {
            // slow path: move the reference of this warp's rows (O and l of chunk a sit in TMEM, scaled by 2^(-ref))
            mbar_wait(&pv_done[g], j & 1u);
            tc_fence_after();
            const float nref = fmaxf(ref, mx);
            const float alpha = fast_exp2((ref - nref) * sl2);
            uint32_t r[32];
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              tmem_ld_32x32(t_row + 160 + hh * 32, r);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * alpha);
              tmem_st_32x16(t_row + 160 + hh * 32, *reinterpret_cast<uint32_t(*)[16]>(&r[0]));
              tmem_st_32x16(t_row + 160 + hh * 32 + 16, *reinterpret_cast<uint32_t(*)[16]>(&r[16]));
            }
            uint32_t l16[16];                      // the row-sum accumulator is 16 identical columns
            tmem_ld_32x16(t_row + 224, l16);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) l16[i] = __float_as_uint(__uint_as_float(l16[i]) * alpha);
            tmem_st_32x16(t_row + 224, l16);
            tmem_st_wait();
            ref = nref;
          }
          const float mb = ref * sl2;
          my_turn();
#pragma unroll
          for (int q = 0; q < AFL_NKC / 32; ++q) {
            uint32_t pk[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int k0 = q * 32 + 2 * i;
              float p0 = fast_exp2(fmaf(__uint_as_float(sv[k0]), sl2, -mb));
              float p1 = fast_exp2(fmaf(__uint_as_float(sv[k0 + 1]), sl2, -mb));
              if (kvalid != AFL_NKC) {
                if (k0 >= kvalid) p0 = 0.f;
                if (k0 + 1 >= kvalid) p1 = 0.f;
              }
              pk[i] = pack_bf16x2(p0, p1);
            }
            tmem_st_32x16(t_row + q * 16, pk);
          }
          pass_turn();
          tmem_st_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&p_ready[g]);
        }
        // ---- O / l -> bf16 rows (swizzled slab -> TMA store clipped at the sequence end) + log-sum-exp
        if (lane == 0) tma_store_wait_read<0>();   // the slab of this warp's previous tile has been read
        __syncwarp();
        mbar_wait(&o_full[g], j & 1u);
        tc_fence_after();
        uint32_t lsum;
        tmem_ld_32x1(t_row + 224, lsum);
        tmem_ld_wait();
        const float l = __uint_as_float(lsum);
        const float inv = 1.0f / l;
        const int row = t * 128 + sp * 32 + lane;
        if (row < p.S) p.lse[((int64_t)seq * p.H + h) * p.S + row] = ref * p.scale + __logf(l);
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          uint32_t r[32];
          tmem_ld_32x32(t_row + 160 + hh * 32, r);
          tmem_ld_wait();
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint32_t a = stg_a + (uint32_t)lane * 128u + ((((uint32_t)(hh * 4 + q)) ^ sw) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a),
                         "r"(pack_bf16x2(__uint_as_float(r[8 * q]) * inv, __uint_as_float(r[8 * q + 1]) * inv)),
                         "r"(pack_bf16x2(__uint_as_float(r[8 * q + 2]) * inv, __uint_as_float(r[8 * q + 3]) * inv)),
                         "r"(pack_bf16x2(__uint_as_float(r[8 * q + 4]) * inv, __uint_as_float(r[8 * q + 5]) * inv)),
                         "r"(pack_bf16x2(__uint_as_float(r[8 * q + 6]) * inv, __uint_as_float(r[8 * q + 7]) * inv))
                         : "memory");
          }
        }
        tc_fence_before();
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(&s_free[g]);              // S / P / O / l columns may be overwritten by this warpgroup's next tile
          if (t * 128 + sp * 32 < p.S) {
            tma_store_3d(&tmO, stg, h * 64, t * 128 + sp * 32, seq);
            tma_store_commit();
          }
        }
      }
    }
    if (lane == 0) tma_store_wait_read<0>();
    // balance the ping-pong: A owns ceil(T/2) of this CTA's T tiles, B floor(T/2); B plays dummy turns for the difference and
    // A takes B's last hand-over
    const int items_cta = (n_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int T = items_cta * nt;
    if (g == 1) {
      for (int i = 0; i < ((T + 1) / 2 - T / 2) * nch; ++i) { my_turn(); pass_turn(); }
    } else {
      my_turn();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

int launch_attn_fwd_lse_tc(const void* qkv, void* o, float* lse, int n_seq, int S, int H, float scale, cudaStream_t stream) {
  UB_REQUIRE(S >= 1 && S <= 2 * AFL_NKC, "attn_fwd_lse_tc: S=%d out of range", S);
  AttnFwdLseParams p;
  p.lse = lse;
  p.n_seq = n_seq; p.S = S; p.H = H;
  p.nt = (S + 127) / 128;
  p.nch = S > AFL_NKC ? 2 : 1;
  p.scale = scale;
  p.sl2 = scale * 1.4426950408889634f;
  CUtensorMap tq, tkv, to;
  const int64_t ld = 3 * (int64_t)H * 64, ldo = (int64_t)H * 64;
  if (make_tmap_3d_bf16(&tq, qkv, n_seq, S, ld, ld, (int64_t)S * ld, 64, 128)) return 1;
  if (make_tmap_3d_bf16(&tkv, qkv, n_seq, S, ld, ld, (int64_t)S * ld, 64, AFL_NKC)) return 1;
  if (make_tmap_3d_bf16(&to, o, n_seq, S, ldo, ldo, (int64_t)S * ldo, 64, 32)) return 1;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(attn_fwd_lse_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AFL_SMEM);
    UB_REQUIRE(e == cudaSuccess, "cudaFuncSetAttribute(attn_fwd_lse_tc smem=%d): %s", AFL_SMEM, cudaGetErrorString(e));
    configured = true;
  }
  const int items = n_seq * H;
  const int grid = items < sm_count() ? items : sm_count();
  UB_LAUNCH(attn_fwd_lse_tc_kernel, grid, AFL_THREADS, AFL_SMEM, stream, tq, tkv, to, p);
  return check_launch("attn_fwd_lse_tc_kernel");
}

}  // namespace ub
