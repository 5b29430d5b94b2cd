// vtk_attention.cu -- masked variable-length flash-style attention forward on tcgen05 (sm_100a).
//
// Replaces modules/attention.py:109-127 (flash_attn_func / F.scaled_dot_product_attention) of the
// reference: out = softmax(q k^T / sqrt(d)) v per (image, head), q/k already QK-normed + RoPE'd by the
// QKV GEMM epilogue.  The reference's sdpa backend masks keys with patch_mask (ae.py:173-187) by
// materialising a [B,1,N,N] bool mask; here the mask is a per-image key length (padded keys are never
// loaded -- whole kv tiles past kv_len[b] are skipped, padded query tiles exit at once).  Masked inference runs
// on the packed NaFlex layout, where every image's valid tokens form a prefix of its rows; the padded training
// step permutes tokens so that every mask is a prefix mask.  The flash backend's semantics (no mask) = kv_len null.
//
// One CTA per (256-query block, head, image) = two 128-query tiles A and B that share every K/V tile:
//   warps 0-3 : softmax warpgroup A   (one query row per thread, TMEM lane = row)
//   warps 4-7 : softmax warpgroup B
//   warp  8   : TMA producer (Q_a, Q_b once; K_j / V_j tiles of 128 keys through one smem ring)
//   warp  9   : MMA issuer: S_x = Q_x K_j^T (128x128xd) and O_x += P_x V_j (128xdx128), fp32 in TMEM
// Per tile a softmax thread pulls its 128 scores out of TMEM in one batch (so the MMA warp can start
// S(j+1) immediately), takes the row max, exponentiates with ex2.approx (log2 domain, scale folded into an
// FFMA), writes P as bf16 into 128B-swizzled shared memory (the A operand of the PV MMA) and rescales O in
// TMEM only when its running max moved by more than 2^8 (lazy rescale; the stale max cancels in O / l).
// While warpgroup A exponentiates, the tensor core works for B and vice versa.
// V is consumed as an MN-major B operand straight from its [key, d] layout (no transpose pass).
// Head dims: any d % 8 == 0 up to 128 runs on the kernel of the next tile width DH (d <= 64: the persistent d = 64 kernel, else the
// d = 128 one).  Q / K / V / O move through 3-D tensor maps {d, heads, rows}, so the tile columns d..DH-1 load as zeros (they add
// nothing to S or to P V) and only the head's d columns are stored.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>

#include "vtk_common.cuh"
#include "vtk_kernels.h"

namespace vtk {

static constexpr int ATT_BQ = 128;   // queries per softmax warpgroup
static constexpr int ATT_BKV = 128;  // keys per tile
static constexpr int BLK = 16384;    // one [128 x 64] bf16 swizzled block
static constexpr float RESCALE_THRESHOLD = 8.0f;  // log2 units

// NQ = query tiles per CTA.  NQ = 2 (one CTA per SM): two softmax warpgroups ping-pong on the tensor core and
// share every K/V tile.  NQ = 1 (the persistent d = 64 kernel): 112 KB of shared memory and 256 TMEM columns, so TWO CTAs are
// resident per SM and hide each other's load / MMA / store latencies -- the better shape for the short
// sequences of the 256 px configs (N = 256: two K/V tiles per CTA, latency-bound otherwise).
template <int DH, int NQ> struct AttnShape {
  static constexpr int NB = DH / 64;               // 64-column blocks per head
  static constexpr int TILE_BYTES = NB * BLK;      // one Q / K / V tile
  static constexpr int RK = 2;                     // K ring slots
  static constexpr int RV = (DH == 64) ? 2 : 1;    // V ring slots (227 KB smem budget at d = 128)
  static constexpr int P_BYTES = 2 * BLK;          // 128 x 128 bf16
  static constexpr int OFF_Q = 0;                  // Q_a (, Q_b)
  static constexpr int OFF_K = OFF_Q + NQ * TILE_BYTES;
  static constexpr int OFF_V = OFF_K + RK * TILE_BYTES;
  static constexpr int OFF_P = OFF_V + RV * TILE_BYTES;      // P_a (, P_b)
  static constexpr int OFF_BAR = OFF_P + NQ * P_BYTES;
  static constexpr int SMEM_BYTES = OFF_BAR + 256;           // the dynamic smem base is declared 1024-byte aligned
  static constexpr uint32_t TMEM_COLS = NQ == 2 ? 512 : 256; // S_q at [q*128, +128), O_q at [NQ*128 + q*DH, +DH)
  static constexpr int O_COL0 = NQ * 128;
  static constexpr int THREADS = 128 * NQ + 64;
  static constexpr int WARP_TMA = 4 * NQ, WARP_MMA = 4 * NQ + 1;
};

struct AttnParams {
  bf16* out; long long ld_out;
  const int* kv_len;
  int N, heads, d, zero_invalid, tma_out;   // d = the true head width (<= DH; columns d..DH-1 of a tile are TMA zero fill)
  int window;         // sliding window |i - j| <= window on the token index (flash backend, attention.py:113-116); < 0 = none
  float scale_log2;   // (1/sqrt(d)) * log2(e)
  unsigned long long* prof;   // perf experiments (env VTK_ATTN_PROF): clock64 accumulators, or null
  float* lse;                 // [rows, heads] log2-domain logsumexp of the scaled scores (training), or null; +inf for zero rows
  // packed NaFlex batches: image b owns packed rows [cu[b], cu[b+1]) and holds kv_len[b] valid tokens at the front; work group g
  // (128 query rows for the persistent kernel, NQ * 128 for the one-shot kernel) is the (g - cuq[img])-th group of image
  // img = grp_img[g]; cuq[B] (= *n_grp) groups exist; grp_order lists them longest image first
  const int* cu; const int* cuq; const int* grp_img; const int* grp_order; const int* n_grp;
};

__device__ __forceinline__ float max3f(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Set the masked scores of one 128-key tile to -inf.  The common case -- the tail tile of an image, no window -- is handled
// per 32-column chunk with warp-uniform branches: chunks entirely inside kvlen are skipped and only the chunks at / beyond
// the boundary pay a compare + select per column (the general per-element test costs ~12 instructions per score and
// made a masked tile 8x as expensive as an unmasked one).
template <int NCH>
__device__ __forceinline__ void mask_scores(uint32_t (&v)[NCH][32], int kv0, int kvlen, int W, int qi) {
  if (W < 0) {
    const int lim = kvlen - kv0;   // columns >= lim are masked
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      if (lim < (c + 1) * 32) {
        const int l = lim - c * 32;
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (i >= l) v[c][i] = 0xff800000u;   // -inf
      }
    }
    return;
  }
#pragma unroll
  for (int c = 0; c < NCH; ++c)
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const int kc = kv0 + c * 32 + i;
      const bool ok = kc < kvlen && abs(kc - qi) <= W;
      if (!ok) v[c][i] = 0xff800000u;   // -inf
    }
}

// Exponentiate one 128-key score tile held in registers (v = raw scores), accumulate the row sum and write P as
// bf16 into the row's 128B-swizzled shared-memory slots.  Software-pipelined by hand: all FFMA2 (scale, subtract
// max) first, then the exponential of pair i+DIST is issued before the FADD2 / F2FP / STS that consume pair i, so a
// warp never stalls on its own MUFU latency (ptxas otherwise places each consumer right behind its producer and
// the XU pipe idles ~55 % of the exponentiation phase with only two softmax warps per scheduler).
// (Exponentiating part of the pairs with a degree-3 polynomial on the FMA pipe, FlashAttention-4's trick, was measured
// 4-9 % SLOWER here -- the f32x2 FMA pipe is as loaded as the MUFU -- and was removed; profiles/README.md.)
__device__ __forceinline__ void softmax_exp_tile(uint32_t (&v)[4][32], uint64_t sc2, uint64_t nm2, uint8_t* prow, int r,
                                                 uint64_t& sum2a, uint64_t& sum2b) {
#pragma unroll
  for (int pr = 0; pr < 64; ++pr) {
    float e0, e1;
    f2_unpack(f2_fma(f2_pack(__uint_as_float(v[pr >> 4][2 * (pr & 15)]), __uint_as_float(v[pr >> 4][2 * (pr & 15) + 1])), sc2, nm2), e0, e1);
    v[pr >> 4][2 * (pr & 15)] = __float_as_uint(e0);
    v[pr >> 4][2 * (pr & 15) + 1] = __float_as_uint(e1);
  }
  constexpr int DIST = 3;
  uint32_t pk[4];
#pragma unroll
  for (int pr = 0; pr < 64 + DIST; ++pr) {
    if (pr < 64) {
      uint32_t& a = v[pr >> 4][2 * (pr & 15)];
      uint32_t& b = v[pr >> 4][2 * (pr & 15) + 1];
      asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+r"(a));
      asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+r"(b));
    }
    if (pr >= DIST) {
      const int q = pr - DIST;
      const float e0 = __uint_as_float(v[q >> 4][2 * (q & 15)]), e1 = __uint_as_float(v[q >> 4][2 * (q & 15) + 1]);
      if (q & 1) sum2b = f2_add(sum2b, f2_pack(e0, e1));
      else sum2a = f2_add(sum2a, f2_pack(e0, e1));
      pk[q & 3] = bf2_cvt(e0, e1);
      if ((q & 3) == 3) {
        const int gg = q >> 2;   // 16-byte chunk index 0..15 along the 128 keys; swizzle-128B: chunk' = chunk ^ (row & 7)
        const int blk = gg >> 3, ch = (gg & 7) ^ (r & 7);
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(smem_u32(prow + blk * BLK + (ch << 4))), "r"(pk[0]), "r"(pk[1]),
                     "r"(pk[2]), "r"(pk[3])
                     : "memory");
      }
    }
  }
}

// Same, but P goes to TENSOR MEMORY (columns [tP, tP + 64) of the thread's lane: key pair q -> 32-bit column q, low half =
// key 2q) as the A operand of a tcgen05.mma that reads A from TMEM: no 32 KB shared-memory write + read per tile.
__device__ __forceinline__ void softmax_exp_tile_tmem(uint32_t (&v)[4][32], uint64_t sc2, uint64_t nm2, uint32_t tP,
                                                      uint64_t& sum2a, uint64_t& sum2b) {
#pragma unroll
  for (int pr = 0; pr < 64; ++pr) {
    float e0, e1;
    f2_unpack(f2_fma(f2_pack(__uint_as_float(v[pr >> 4][2 * (pr & 15)]), __uint_as_float(v[pr >> 4][2 * (pr & 15) + 1])), sc2, nm2), e0, e1);
    v[pr >> 4][2 * (pr & 15)] = __float_as_uint(e0);
    v[pr >> 4][2 * (pr & 15) + 1] = __float_as_uint(e1);
  }
  constexpr int DIST = 3;
  uint32_t pk[8];
#pragma unroll
  for (int pr = 0; pr < 64 + DIST; ++pr) {
    if (pr < 64) {
      uint32_t& a = v[pr >> 4][2 * (pr & 15)];
      uint32_t& b = v[pr >> 4][2 * (pr & 15) + 1];
      asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+r"(a));
      asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+r"(b));
    }
    if (pr >= DIST) {
      const int q = pr - DIST;
      const float e0 = __uint_as_float(v[q >> 4][2 * (q & 15)]), e1 = __uint_as_float(v[q >> 4][2 * (q & 15) + 1]);
      if (q & 1) sum2b = f2_add(sum2b, f2_pack(e0, e1));
      else sum2a = f2_add(sum2a, f2_pack(e0, e1));
      pk[q & 7] = bf2_cvt(e0, e1);
      if ((q & 7) == 7) tmem_st8(tP + (q & ~7), pk[0], pk[1], pk[2], pk[3], pk[4], pk[5], pk[6], pk[7]);
    }
  }
}

template <int DH, int NQ>
__global__ void __launch_bounds__(128 * NQ + 64, NQ == 1 ? 2 : 1)
attn_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
            const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmO, const AttnParams p) {
  using S = AttnShape<DH, NQ>;
  pdl_wait();      // PDL: the work description below is read from global memory (pack plan, kv_len), so wait first
  pdl_trigger();
  const long long t_cta0 = p.prof ? clock64() : 0;
  const int head = blockIdx.y;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  int q0, img, N, kvlen;
  long long row0;
  if (p.cu) {
    // packed NaFlex layout: blockIdx.x = work group (NQ * 128 query rows of one image)
    if ((int)blockIdx.x >= __ldg(p.n_grp)) return;   // beyond the groups of this batch (whole CTA)
    const int grp = p.grp_order ? p.grp_order[blockIdx.x] : (int)blockIdx.x;   // CTAs are issued in index order: longest images first
    img = p.grp_img[grp];
    row0 = p.cu[img];
    q0 = (grp - p.cuq[img]) * (NQ * ATT_BQ);
    kvlen = p.kv_len[img];
    // rows stored: the valid ones, plus (zero_invalid: the training forward, which needs lse) the image's pad rows as 0 / +inf.
    // Rows past cu[img + 1] belong to the next image and are never stored.
    N = p.zero_invalid ? p.cu[img + 1] - (int)row0 : kvlen;
  } else {
    q0 = blockIdx.x * (NQ * ATT_BQ);
    img = blockIdx.z;
    N = p.N;
    kvlen = p.kv_len ? p.kv_len[img] : N;
    kvlen = kvlen < N ? kvlen : N;
    row0 = (long long)img * N;
  }
  const int T = (kvlen + ATT_BKV - 1) / ATT_BKV;
  const int qlimit = p.zero_invalid ? kvlen : N;           // query rows >= qlimit are padding
  const int nact = (T == 0 || q0 >= qlimit) ? 0 : ((NQ == 2 && q0 + ATT_BQ < qlimit) ? 2 : 1);

  // query tiles with nothing to attend to: define the output as 0 (uniform per warpgroup)
  if (warp < 4 * NQ) {
    const int wg = warp >> 2;
    if (wg >= nact) {
      const int qi = q0 + wg * ATT_BQ + (warp & 3) * 32 + lane;
      if (qi < N) {
        bf16* op = p.out + (row0 + qi) * p.ld_out + head * p.d;
        for (int c = 0; c < p.d; c += 8) st_global_v4(op + c, 0u, 0u, 0u, 0u);
        if (p.lse) p.lse[(row0 + qi) * p.heads + head] = INFINITY;
      }
    }
  }
  if (nact == 0) return;   // whole CTA
  // key tiles this CTA visits: all T, or only those intersecting the sliding window of its query rows
  const int W = p.window;
  int j_lo = 0, j_hi = T - 1;
  if (W >= 0) {
    const int q_last = min(q0 + nact * ATT_BQ, N) - 1;
    j_lo = max(0, q0 - W) / ATT_BKV;
    j_hi = min(T - 1, (int)min((long long)q_last + W, (long long)N - 1) / ATT_BKV);
  }
  const int Tn = j_hi - j_lo + 1;

  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sQ = smem + S::OFF_Q;
  uint8_t* sK = smem + S::OFF_K;
  uint8_t* sV = smem + S::OFF_V;
  uint8_t* sP = smem + S::OFF_P;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* q_full = bars + 0;
  uint64_t* k_full = bars + 1;               // [2]
  uint64_t* k_empty = bars + 3;              // [2]
  uint64_t* v_full = bars + 5;               // [2]
  uint64_t* v_empty = bars + 7;              // [2]
  uint64_t* s_full = bars + 9;               // [2]
  uint64_t* s_empty = s_full + 2;            // [2]
  uint64_t* p_full = s_full + 4;             // [2]
  uint64_t* pv_done = s_full + 6;            // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_full + 8);

  if (warp == S::WARP_TMA) {
    // 17 mbarriers, one lane each: [0] q_full | k_full[2] k_empty[2] v_full[2] v_empty[2] | s_full[2] s_empty[2] p_full[2] pv_done[2]
    if (lane < 17) {
      const bool wg_count = (lane >= 11 && lane <= 14);   // s_empty, p_full: all 128 softmax threads arrive
      mbar_init(&bars[lane], wg_count ? 128u : 1u);
    } else if (lane == 17) {
      tma_prefetch_desc(&tmQ);
    } else if (lane == 18) {
      tma_prefetch_desc(&tmK);
    } else if (lane == 19) {
      tma_prefetch_desc(&tmV);
    }
    fence_barrier_init();
    __syncwarp();
  }
  if (warp == S::WARP_MMA) {
    tmem_alloc(tmem_slot, S::TMEM_COLS);
    tmem_relinquish();
  }
  if (warp == S::WARP_TMA && lane == 0) {
    // Q tiles and K_0 go out before the CTA-wide sync: their latency overlaps the TMEM allocation
    mbar_expect_tx(q_full, (uint32_t)(nact * S::TILE_BYTES));
    for (int t = 0; t < nact; ++t)
      for (int nb = 0; nb < S::NB; ++nb)
        tma_load_3d(sQ + t * S::TILE_BYTES + nb * BLK, &tmQ, q_full, nb * 64, head, (int)(row0 + q0 + t * ATT_BQ));
    mbar_expect_tx(&k_full[0], S::TILE_BYTES);
    for (int nb = 0; nb < S::NB; ++nb)
      tma_load_3d(sK + nb * BLK, &tmK, &k_full[0], nb * 64, head, (int)(row0 + (long long)j_lo * ATT_BKV));
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const long long t_sync = p.prof ? clock64() : 0;

  if (warp == S::WARP_TMA) {
    if (lane == 0) {
      // ===== TMA producer ===== (Q and K_0 were issued before the sync)
      // issue order K_0, K_1, V_0, K_2, V_1, ...: K_{j+1} is needed (for S(j+1)) before V_j (for PV(j))
      auto load_k = [&](int jj) {   // jj = position in this CTA's tile sequence; key tile index = j_lo + jj
        const int slot = jj % S::RK;
        mbar_wait(&k_empty[slot], ((uint32_t)(jj / S::RK) & 1u) ^ 1u);
        mbar_expect_tx(&k_full[slot], S::TILE_BYTES);
        for (int nb = 0; nb < S::NB; ++nb)
          tma_load_3d(sK + slot * S::TILE_BYTES + nb * BLK, &tmK, &k_full[slot], nb * 64, head,
                      (int)(row0 + (long long)(j_lo + jj) * ATT_BKV));
      };
      for (int jj = 0; jj < Tn; ++jj) {
        if (jj + 1 < Tn) load_k(jj + 1);
        const int slot = jj % S::RV;
        mbar_wait(&v_empty[slot], ((uint32_t)(jj / S::RV) & 1u) ^ 1u);
        mbar_expect_tx(&v_full[slot], S::TILE_BYTES);
        for (int nb = 0; nb < S::NB; ++nb)
          tma_load_3d(sV + slot * S::TILE_BYTES + nb * BLK, &tmV, &v_full[slot], nb * 64, head,
                      (int)(row0 + (long long)(j_lo + jj) * ATT_BKV));
      }
    }
  } else if (warp == S::WARP_MMA) {
    if (lane == 0) {
      // ===== MMA issuer =====
      const uint32_t idesc_s = make_idesc_bf16(ATT_BQ, ATT_BKV, 0, 0);
      const uint32_t idesc_o = make_idesc_bf16(ATT_BQ, DH, 0, 1);   // B (= V) is MN-major
      auto k_wait = [&](int j) {
        mbar_wait(&k_full[j % S::RK], (uint32_t)(j / S::RK) & 1u);
        return smem_u32(sK + (j % S::RK) * S::TILE_BYTES);
      };
      auto v_wait = [&](int j) {
        mbar_wait(&v_full[j % S::RV], (uint32_t)(j / S::RV) & 1u);
        return smem_u32(sV + (j % S::RV) * S::TILE_BYTES);
      };
      auto issue_s = [&](int q, uint32_t ka) {
        const uint32_t qa = smem_u32(sQ + q * S::TILE_BYTES);
#pragma unroll
        for (int kk = 0; kk < DH / 16; ++kk) {
          const uint32_t off = (kk >> 2) * BLK + (kk & 3) * 32;
          umma_bf16_ss(tmem_base + q * 128, make_desc_kmajor_sw128(qa + off), make_desc_kmajor_sw128(ka + off), idesc_s,
                       kk != 0 ? 1u : 0u);
        }
        umma_commit(&s_full[q]);
      };
      auto issue_pv = [&](int q, int j, uint32_t va) {
        const uint32_t pa = smem_u32(sP + q * S::P_BYTES);
#pragma unroll
        for (int kk = 0; kk < ATT_BKV / 16; ++kk) {
          const uint64_t adesc = make_desc_kmajor_sw128(pa + (kk >> 2) * BLK + (kk & 3) * 32);
          // V tile: NB blocks of [128 keys x 64 d]; MN-major: LBO = block stride, SBO = 8-key group stride
          const uint64_t bdesc = make_smem_desc(va + kk * 2048, BLK, 1024, 2);
          umma_bf16_ss(tmem_base + S::O_COL0 + q * DH, adesc, bdesc, idesc_o, (j | kk) != 0 ? 1u : 0u);
        }
        umma_commit(&pv_done[q]);
      };
      mbar_wait(q_full, 0);
      {
        const uint32_t ka = k_wait(0);
        tc_fence_after();
        for (int q = 0; q < nact; ++q) issue_s(q, ka);
        umma_commit(&k_empty[0]);
      }
      for (int j = 0; j < Tn; ++j) {   // j = position in the tile sequence
        const uint32_t jp = (uint32_t)j & 1u;
        if (j + 1 < Tn) {   // S(j+1) as soon as the softmax threads have pulled S(j) into registers
          const uint32_t ka = k_wait(j + 1);
          for (int q = 0; q < nact; ++q) {
            mbar_wait(&s_empty[q], jp);
            tc_fence_after();
            issue_s(q, ka);
          }
          umma_commit(&k_empty[(j + 1) % S::RK]);
        }
        const uint32_t va = v_wait(j);
        for (int q = 0; q < nact; ++q) {
          mbar_wait(&p_full[q], jp);
          tc_fence_after();
          issue_pv(q, j, va);
        }
        umma_commit(&v_empty[j % S::RV]);
      }
    }
  } else if ((warp >> 2) < nact) {
    // ===== softmax warpgroups: thread <-> query row =====
    const int q = warp >> 2;
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    const uint32_t tS = tmem_base + lane_base + q * 128;
    const uint32_t tO = tmem_base + lane_base + S::O_COL0 + q * DH;
    uint8_t* prow = sP + q * S::P_BYTES + r * 128;
    const float sc = p.scale_log2;
    float m_run = -INFINITY, l_run = 0.f;
    long long w_s = 0, w_pv = 0, t_first = 0;
    const int qi = q0 + q * ATT_BQ + r;
    for (int j = 0; j < Tn; ++j) {   // j = position in the tile sequence
      const int kv0 = (j_lo + j) * ATT_BKV;
      const int qt0 = q0 + q * ATT_BQ;
      const bool win_mask = W >= 0 && (kv0 < qt0 + ATT_BQ - 1 - W || kv0 + ATT_BKV - 1 > qt0 + W);
      const bool need_mask = (kv0 + ATT_BKV > kvlen) || win_mask;
      const long long ta = p.prof ? clock64() : 0;
      mbar_wait(&s_full[q], (uint32_t)j & 1u);
      if (p.prof) { const long long tb = clock64(); if (j == 0) t_first = tb - t_sync; else w_s += tb - ta; }
      __syncwarp();
      tc_fence_after();
      uint32_t v[4][32];
      tmem_ld32(tS + 0, v[0]);
      tmem_ld32(tS + 32, v[1]);
      tmem_ld32(tS + 64, v[2]);
      tmem_ld32(tS + 96, v[3]);
      tmem_wait_ld();
      tc_fence_before();
      mbar_arrive(&s_empty[q]);   // S is in registers: the tensor core may overwrite it with S(j+1)
      if (need_mask) mask_scores(v, kv0, kvlen, W, qi);
      float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
      for (int i = 0; i < 32; i += 2) {   // FMNMX3: two elements per instruction
        mx0 = max3f(mx0, __uint_as_float(v[0][i]), __uint_as_float(v[0][i + 1]));
        mx1 = max3f(mx1, __uint_as_float(v[1][i]), __uint_as_float(v[1][i + 1]));
        mx2 = max3f(mx2, __uint_as_float(v[2][i]), __uint_as_float(v[2][i + 1]));
        mx3 = max3f(mx3, __uint_as_float(v[3][i]), __uint_as_float(v[3][i + 1]));
      }
      const float m_tile = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3)) * sc;
      // lazy rescale: keep the stale max unless it moved by more than 2^8
      float m_use = m_run, alpha = 1.f;
      if (m_tile > m_run + RESCALE_THRESHOLD || m_run == -INFINITY) {
        m_use = fmaxf(m_run, m_tile);
        alpha = (m_run == -INFINITY) ? 0.f : ex2_approx(m_run - m_use);
      }
      const float m_sub = (m_use == -INFINITY) ? 0.f : m_use;
      // packed pipeline per key pair: FFMA2 (scale, subtract max) -> 2 x MUFU.EX2 -> FADD2 (row sum) ->
      // F2FP.BF16.PACK_AB (P as bf16x2, round to nearest even): 2.5 issue slots per element, XU does ex2 only
      const uint64_t sc2 = f2_pack(sc, sc), nm2 = f2_pack(-m_sub, -m_sub);
      uint64_t sum2a = 0ull, sum2b = 0ull;
      // P buffer and O are free once PV(j-1) has completed (it was issued a whole softmax tile ago)
      if (j > 0) {
        const long long tc = p.prof ? clock64() : 0;
        mbar_wait(&pv_done[q], (uint32_t)(j - 1) & 1u);
        if (p.prof) w_pv += clock64() - tc;
        __syncwarp();
        tc_fence_after();
      }
      // 128 columns = 2 blocks x 8 chunks of 16 B; swizzle-128B: chunk' = chunk ^ (row & 7); each 16-byte chunk
      // (8 keys) is written as soon as it is exponentiated
      softmax_exp_tile(v, sc2, nm2, prow, r, sum2a, sum2b);
      float sum0, sum1;
      f2_unpack(f2_add(sum2a, sum2b), sum0, sum1);
      l_run = l_run * alpha + (sum0 + sum1);
      m_run = m_use;
      if (j > 0 && __any_sync(0xffffffffu, alpha != 1.f)) {
#pragma unroll
        for (int c = 0; c < DH; c += 32) {
          uint32_t o[32];
          tmem_ld32(tO + c, o);
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
          tmem_st32(tO + c, o);
        }
        tmem_wait_st();
      }
      fence_proxy_async_smem();   // P (generic-proxy smem writes) -> visible to the MMA (async proxy)
      tc_fence_before();
      mbar_arrive(&p_full[q]);
    }
    // epilogue: O / l
    const long long td = p.prof ? clock64() : 0;
    mbar_wait(&pv_done[q], (uint32_t)(Tn - 1) & 1u);
    const long long te = p.prof ? clock64() : 0;
    __syncwarp();
    tc_fence_after();
    const float inv = l_run > 0.f ? 1.f / l_run : 0.f;
    const bool zero_row = p.zero_invalid && qi >= kvlen;
    const float osc = zero_row ? 0.f : inv;
    if (p.lse && qi < N) p.lse[(row0 + qi) * p.heads + head] = (zero_row || !(l_run > 0.f)) ? INFINITY : m_run + log2f(l_run);
    bf16* op = p.out + (row0 + qi) * p.ld_out + head * p.d;
    uint32_t o[DH / 32][32];
#pragma unroll
    for (int c = 0; c < DH / 32; ++c) tmem_ld32(tO + c * 32, o[c]);
    tmem_wait_ld();
    if (p.tma_out && (p.cu == nullptr || q0 + (q + 1) * ATT_BQ <= N)) {
      // the tile does not straddle an image (N % 128 == 0, or a full tile of a packed image).  Stage this warp's 32 rows in the (now idle) Q buffer
      // in the 128B-swizzled layout and let one TMA store per 64-column block write full 128-byte row segments.
      uint8_t* srow = sQ + q * S::TILE_BYTES + r * 128;
#pragma unroll
      for (int c = 0; c < DH / 32; ++c)
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint32_t w[4];
#pragma unroll
          for (int i = 0; i < 4; ++i)
            w[i] = bf2_cvt(__uint_as_float(o[c][8 * g + 2 * i]) * osc, __uint_as_float(o[c][8 * g + 2 * i + 1]) * osc);
          const int col = c * 32 + 8 * g;   // column inside the head
          const int ch = ((col & 63) >> 3) ^ (r & 7);
          *reinterpret_cast<uint4*>(srow + (col >> 6) * BLK + (ch << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
        }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
#pragma unroll
        for (int nb = 0; nb < S::NB; ++nb)
          tma_store_3d(&tmO, sQ + q * S::TILE_BYTES + nb * BLK + quarter * 32 * 128, nb * 64, head,
                       (int)(row0 + q0 + q * ATT_BQ + quarter * 32));
        tma_store_commit();
        tma_store_wait_read();
      }
    } else if (qi < N) {
#pragma unroll
      for (int c = 0; c < DH / 32; ++c)
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          if (c * 32 + 8 * g >= p.d) break;   // the tile's zero columns past the head width
          uint32_t w[4];
#pragma unroll
          for (int i = 0; i < 4; ++i)
            w[i] = pack_bf16x2(__uint_as_float(o[c][8 * g + 2 * i]) * osc, __uint_as_float(o[c][8 * g + 2 * i + 1]) * osc);
          st_global_v4(op + c * 32 + 8 * g, w[0], w[1], w[2], w[3]);
        }
    }
    if (p.prof && warp == 0 && lane == 0) {
      const long long tf = clock64();
      atomicAdd(&p.prof[0], (unsigned long long)(t_sync - t_cta0));   // prologue up to the CTA-wide sync
      atomicAdd(&p.prof[1], (unsigned long long)t_first);             // sync -> first S ready (Q/K load + S MMA)
      atomicAdd(&p.prof[2], (unsigned long long)w_s);                 // later waits for S
      atomicAdd(&p.prof[3], (unsigned long long)w_pv);                // waits for PV(j-1) inside the loop
      atomicAdd(&p.prof[4], (unsigned long long)(te - td));           // wait for the last PV
      atomicAdd(&p.prof[5], (unsigned long long)(tf - te));           // O epilogue
      atomicAdd(&p.prof[6], (unsigned long long)(tf - t_cta0));       // whole CTA
      atomicAdd(&p.prof[7], 1ull);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == S::WARP_MMA) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem_base, S::TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------
// Persistent variant for d = 64 (one 128-query tile per work item, two CTAs resident per SM).
//
// The one-shot kernel above pays barrier init + TMEM allocation + the first Q/K load (~3.9 k of ~10.5 k cycles per CTA
// at N = 256, measured with VTK_ATTN_PROF) for every (image, head, query tile).  Here a CTA walks a strided list of work
// items and the three roles run ahead of each other ACROSS items: the TMA thread refills the Q buffer as soon as the
// last S MMA of the current item has been committed and the K/V rings as their slots drain, the MMA thread issues
// S(next item, tile 0) while the softmax warps are still on the previous item's last tile / epilogue, so in steady
// state the softmax warps never wait for a load.  O is staged in the (idle) P buffer and leaves through a TMA store
// whose completion is only awaited right before P is written again.
// Barrier phases are tracked with running counters (tiles / K loads / V loads / items seen by this CTA).
// ------------------------------------------------------------------------------------------------
struct AttnItem {
  int img, head, q0, kvlen, qlimit, j_lo, Tn, nrows;   // nrows = token rows of the image (row guard of the direct stores)
  long long row0;                                      // first row of the image in the q/k/v/out buffers
  bool active;
};

template <bool PACKED>
__device__ __forceinline__ AttnItem attn_item(const AttnParams& p, int w, int qtiles) {
  AttnItem it;
  if (PACKED) {   // packed layout: work item = (group of 128 query rows of one image, head); every group holds a valid query
    const int rank = w / p.heads;
    it.head = w - rank * p.heads;
    const int grp = p.grp_order[rank];       // longest images first (pack_plan_kernel)
    it.img = p.grp_img[grp];
    it.row0 = p.cu[it.img];
    it.q0 = (grp - p.cuq[it.img]) * ATT_BQ;
    it.kvlen = p.kv_len[it.img];
    // rows stored: the valid ones (+ the image's pad rows as 0 / +inf under zero_invalid); rows past cu[img + 1] belong to the next image
    it.nrows = p.zero_invalid ? p.cu[it.img + 1] - (int)it.row0 : it.kvlen;
  } else {
    const int per_img = qtiles * p.heads;
    it.img = w / per_img;
    const int r = w - it.img * per_img;
    it.head = r / qtiles;
    it.q0 = (r - it.head * qtiles) * ATT_BQ;
    int kvlen = p.kv_len ? p.kv_len[it.img] : p.N;
    it.kvlen = kvlen < p.N ? kvlen : p.N;
    it.nrows = p.N;
    it.row0 = (long long)it.img * p.N;
  }
  it.qlimit = p.zero_invalid ? it.kvlen : it.nrows;
  const int T = (it.kvlen + ATT_BKV - 1) / ATT_BKV;
  it.active = T > 0 && it.q0 < it.qlimit;
  it.j_lo = 0;
  int j_hi = T - 1;
  if (p.window >= 0) {
    const int q_last = min(it.q0 + ATT_BQ, it.nrows) - 1;
    it.j_lo = max(0, it.q0 - p.window) / ATT_BKV;
    j_hi = min(T - 1, (int)min((long long)q_last + p.window, (long long)it.nrows - 1) / ATT_BKV);
  }
  it.Tn = j_hi - it.j_lo + 1;
  return it;
}

// Item k of this CTA.  SNAKE = false: plain round-robin (w = blockIdx + k * grid).  SNAKE = true (packed batches, whose
// item list is sorted by cost -- pack_plan_kernel's grp_order): items are dealt boustrophedon-wise (0 .. G-1, then
// G-1 .. 0, ...), so every CTA ends up with nearly the same amount of work without a shared counter (c3: max/mean CTA
// load 1.03 instead of 1.19).  Returns false when the CTA is done; a SNAKE caller must skip w >= total.
template <bool SNAKE>
__device__ __forceinline__ bool item_at(int k, int total, int& w) {
  const int G = (int)gridDim.x, b = (int)blockIdx.x;
  if (!SNAKE) {
    w = b + k * G;
    return w < total;
  }
  const int base = (k >> 1) * 2 * G;
  w = base + ((k & 1) ? 2 * G - 1 - b : b);
  return base < total;
}

template <int DH, bool SNAKE>
__global__ void __launch_bounds__(192, 2)
attn_persist_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                    const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmO, const AttnParams p,
                    const int total_items_host, const int qtiles) {
  using S = AttnShape<DH, 1>;
  static_assert(DH == 64, "persistent attention: d = 64 only");
  constexpr uint32_t P_COL = S::O_COL0 + DH;   // P (bf16, 128 keys = 64 columns) after S [0,128) and O [128,192)
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int W = p.window;

  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sQ = smem + S::OFF_Q;
  uint8_t* sK = smem + S::OFF_K;
  uint8_t* sV = smem + S::OFF_V;
  uint8_t* sP = smem + S::OFF_P;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* q_full = bars + 0;
  uint64_t* k_full = bars + 1;               // [2]
  uint64_t* k_empty = bars + 3;              // [2]
  uint64_t* v_full = bars + 5;               // [2]
  uint64_t* v_empty = bars + 7;              // [2]
  uint64_t* s_full = bars + 9;
  uint64_t* s_empty = bars + 10;             // count 128
  uint64_t* p_full = bars + 11;              // count 128
  uint64_t* pv_done = bars + 12;
  uint64_t* q_empty = bars + 13;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);

  if (warp == 4) {
    if (lane < 14) mbar_init(&bars[lane], (lane == 10 || lane == 11) ? 128u : 1u);
    else if (lane == 17) tma_prefetch_desc(&tmQ);
    else if (lane == 18) tma_prefetch_desc(&tmK);
    else if (lane == 19) tma_prefetch_desc(&tmV);
    else if (lane == 20) tma_prefetch_desc(&tmO);
    fence_barrier_init();
    __syncwarp();
  }
  if (warp == 5) {
    tmem_alloc(tmem_slot, S::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // PDL: barrier init + TMEM allocation overlapped the previous kernel's tail; global memory only from here on
  pdl_trigger();
  pdl_wait();
  const int total_items = SNAKE ? min(total_items_host, __ldg(p.n_grp) * p.heads) : total_items_host;   // SNAKE <=> packed layout

  if (warp == 4) {
    if (lane == 0) {
      // ===== TMA producer =====
      uint32_t n_item = 0, n_k = 0, n_v = 0;   // active items / K tiles / V tiles issued so far by this CTA
      for (int k = 0, w; item_at<SNAKE>(k, total_items, w); ++k) {
        if (SNAKE && w >= total_items) continue;
        const AttnItem it = attn_item<SNAKE>(p, w, qtiles);
        if (!it.active) continue;
        const long long row0 = it.row0;
        if (n_item > 0) mbar_wait(q_empty, (n_item - 1) & 1u);     // last S MMA of the previous item has read Q
        mbar_expect_tx(q_full, S::TILE_BYTES);
        tma_load_3d(sQ, &tmQ, q_full, 0, it.head, (int)(row0 + it.q0));
        ++n_item;
        auto load_k = [&](int jj) {
          const uint32_t slot = n_k % S::RK;
          mbar_wait(&k_empty[slot], ((n_k / S::RK) & 1u) ^ 1u);
          mbar_expect_tx(&k_full[slot], S::TILE_BYTES);
          tma_load_3d(sK + slot * S::TILE_BYTES, &tmK, &k_full[slot], 0, it.head, (int)(row0 + (long long)(it.j_lo + jj) * ATT_BKV));
          ++n_k;
        };
        load_k(0);
        for (int jj = 0; jj < it.Tn; ++jj) {
          if (jj + 1 < it.Tn) load_k(jj + 1);
          const uint32_t slot = n_v % S::RV;
          mbar_wait(&v_empty[slot], ((n_v / S::RV) & 1u) ^ 1u);
          mbar_expect_tx(&v_full[slot], S::TILE_BYTES);
          tma_load_3d(sV + slot * S::TILE_BYTES, &tmV, &v_full[slot], 0, it.head, (int)(row0 + (long long)(it.j_lo + jj) * ATT_BKV));
          ++n_v;
        }
      }
    }
  } else if (warp == 5) {
    if (lane == 0) {
      // ===== MMA issuer =====
      const uint32_t idesc_s = make_idesc_bf16(ATT_BQ, ATT_BKV, 0, 0);
      const uint32_t idesc_o = make_idesc_bf16(ATT_BQ, DH, 0, 1);   // B (= V) is MN-major
      uint32_t n_item = 0, n_k = 0, n_v = 0, n_t = 0;   // n_t = key tiles whose S has been issued so far
      uint32_t n_pv = 0;                                 // key tiles whose PV has been issued so far
      const uint32_t qa = smem_u32(sQ);
      auto issue_s = [&]() {   // S(tile n_t) = Q K^T; waits for the K tile and for the S buffer
        const uint32_t slot = n_k % S::RK;
        mbar_wait(&k_full[slot], (n_k / S::RK) & 1u);
        if (n_t > 0) mbar_wait(s_empty, (n_t - 1) & 1u);
        tc_fence_after();
        const uint32_t ka = smem_u32(sK + slot * S::TILE_BYTES);
#pragma unroll
        for (int kk = 0; kk < DH / 16; ++kk)
          umma_bf16_ss(tmem_base, make_desc_kmajor_sw128(qa + kk * 32), make_desc_kmajor_sw128(ka + kk * 32), idesc_s, kk != 0 ? 1u : 0u);
        umma_commit(&k_empty[slot]);
        umma_commit(s_full);
        ++n_k;
        ++n_t;
      };
      for (int k = 0, w; item_at<SNAKE>(k, total_items, w); ++k) {
        if (SNAKE && w >= total_items) continue;
        const AttnItem it = attn_item<SNAKE>(p, w, qtiles);
        if (!it.active) continue;
        mbar_wait(q_full, n_item & 1u);
        ++n_item;
        issue_s();
        for (int jj = 0; jj < it.Tn; ++jj) {
          if (jj + 1 < it.Tn) issue_s();          // S(jj+1) as soon as the softmax threads have pulled S(jj)
          else umma_commit(q_empty);              // every S MMA of this item has been issued: Q may be refilled when they finish
          const uint32_t slot = n_v % S::RV;
          mbar_wait(&v_full[slot], (n_v / S::RV) & 1u);
          mbar_wait(p_full, n_pv & 1u);
          tc_fence_after();
          const uint32_t va = smem_u32(sV + slot * S::TILE_BYTES);
#pragma unroll
          for (int kk = 0; kk < ATT_BKV / 16; ++kk) {
            const uint64_t bdesc = make_smem_desc(va + kk * 2048, BLK, 1024, 2);
            // A = P from tensor memory: 16 keys = 8 packed 32-bit columns per MMA
            umma_bf16_ts(tmem_base + S::O_COL0, tmem_base + P_COL + kk * 8, bdesc, idesc_o, (jj | kk) != 0 ? 1u : 0u);
          }
          umma_commit(&v_empty[slot]);
          umma_commit(pv_done);
          ++n_v;
          ++n_pv;
        }
      }
    }
  } else {
    // ===== softmax warpgroup: thread <-> query row =====
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    const uint32_t tS = tmem_base + lane_base;
    const uint32_t tO = tmem_base + lane_base + S::O_COL0;
    const float sc = p.scale_log2;
    uint32_t n_t = 0;          // key tiles processed so far by this CTA (phase of s_full / p_full / pv_done)
    bool store_pending = false;
    const bool prof = p.prof != nullptr && warp == 0 && lane == 0;
    long long c_wait_s = 0, c_load = 0, c_max = 0, c_wait_pv = 0, c_exp = 0, c_tail = 0, c_epi_wait = 0, c_epi = 0;
    const long long c_begin = prof ? clock64() : 0;
#define PCLK() (prof ? clock64() : 0)
    for (int k = 0, w; item_at<SNAKE>(k, total_items, w); ++k) {
        if (SNAKE && w >= total_items) continue;
      const AttnItem it = attn_item<SNAKE>(p, w, qtiles);
      const long long row0 = it.row0;
      const int N = it.nrows;
      const int qi = it.q0 + r;
      if (!it.active) {   // nothing to attend to: the output rows are 0
        if (qi < N) {
          bf16* op = p.out + (row0 + qi) * p.ld_out + it.head * p.d;
          for (int c = 0; c < p.d; c += 8) st_global_v4(op + c, 0u, 0u, 0u, 0u);
          if (p.lse) p.lse[(row0 + qi) * p.heads + it.head] = INFINITY;
        }
        continue;
      }
      const int kvlen = it.kvlen;
      float m_run = -INFINITY, l_run = 0.f;
      for (int j = 0; j < it.Tn; ++j, ++n_t) {
        const int kv0 = (it.j_lo + j) * ATT_BKV;
        const bool win_mask = W >= 0 && (kv0 < it.q0 + ATT_BQ - 1 - W || kv0 + ATT_BKV - 1 > it.q0 + W);
        const bool need_mask = (kv0 + ATT_BKV > kvlen) || win_mask;
        const long long k0 = PCLK();
        mbar_wait(s_full, n_t & 1u);
        __syncwarp();
        tc_fence_after();
        const long long k1 = PCLK();
        uint32_t v[4][32];
        tmem_ld32(tS + 0, v[0]);
        tmem_ld32(tS + 32, v[1]);
        tmem_ld32(tS + 64, v[2]);
        tmem_ld32(tS + 96, v[3]);
        tmem_wait_ld();
        tc_fence_before();
        mbar_arrive(s_empty);   // S is in registers: the tensor core may overwrite it with the next tile's S
        const long long k2 = PCLK();
        if (need_mask) mask_scores(v, kv0, kvlen, W, qi);
        float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          mx0 = max3f(mx0, __uint_as_float(v[0][i]), __uint_as_float(v[0][i + 1]));
          mx1 = max3f(mx1, __uint_as_float(v[1][i]), __uint_as_float(v[1][i + 1]));
          mx2 = max3f(mx2, __uint_as_float(v[2][i]), __uint_as_float(v[2][i + 1]));
          mx3 = max3f(mx3, __uint_as_float(v[3][i]), __uint_as_float(v[3][i + 1]));
        }
        const float m_tile = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3)) * sc;
        float m_use = m_run, alpha = 1.f;
        if (m_tile > m_run + RESCALE_THRESHOLD || m_run == -INFINITY) {
          m_use = fmaxf(m_run, m_tile);
          alpha = (m_run == -INFINITY) ? 0.f : ex2_approx(m_run - m_use);
        }
        const float m_sub = (m_use == -INFINITY) ? 0.f : m_use;
        const uint64_t sc2 = f2_pack(sc, sc), nm2 = f2_pack(-m_sub, -m_sub);
        uint64_t sum2a = 0ull, sum2b = 0ull;
        // P's tensor-memory columns are free once the previous tile's PV (this item's or the previous item's last) has completed
        const long long k3 = PCLK();
        if (n_t > 0) {
          mbar_wait(pv_done, (n_t - 1) & 1u);
          __syncwarp();
          tc_fence_after();
        }
        const long long k4 = PCLK();
        softmax_exp_tile_tmem(v, sc2, nm2, tmem_base + lane_base + P_COL, sum2a, sum2b);
        tmem_wait_st();
        const long long k5 = PCLK();
        float sum0, sum1;
        f2_unpack(f2_add(sum2a, sum2b), sum0, sum1);
        l_run = l_run * alpha + (sum0 + sum1);
        m_run = m_use;
        if (j > 0 && __any_sync(0xffffffffu, alpha != 1.f)) {
#pragma unroll
          for (int c = 0; c < DH; c += 32) {
            uint32_t o[32];
            tmem_ld32(tO + c, o);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            tmem_st32(tO + c, o);
          }
          tmem_wait_st();
        }
        fence_proxy_async_smem();
        tc_fence_before();
        mbar_arrive(p_full);
        if (prof) {
          const long long k6 = clock64();
          c_wait_s += k1 - k0; c_load += k2 - k1; c_max += k3 - k2; c_wait_pv += k4 - k3; c_exp += k5 - k4; c_tail += k6 - k5;
        }
      }
      // epilogue of the item: O / l
      const long long e0 = PCLK();
      mbar_wait(pv_done, (n_t - 1) & 1u);
      __syncwarp();
      tc_fence_after();
      const long long e1 = PCLK();
      const float inv = l_run > 0.f ? 1.f / l_run : 0.f;
      const bool zero_row = p.zero_invalid && qi >= kvlen;
      const float osc = zero_row ? 0.f : inv;
      if (p.lse && qi < N) p.lse[(row0 + qi) * p.heads + it.head] = (zero_row || !(l_run > 0.f)) ? INFINITY : m_run + log2f(l_run);
      uint32_t o[DH / 32][32];
#pragma unroll
      for (int c = 0; c < DH / 32; ++c) tmem_ld32(tO + c * 32, o[c]);
      tmem_wait_ld();
      tc_fence_before();
      if (p.tma_out && (!SNAKE || it.q0 + ATT_BQ <= it.nrows)) {   // packed: only full tiles leave through TMA (a partial tile shares rows with the next image)
        if (store_pending) {   // the previous item's TMA store has read the staging rows
          if (lane == 0) tma_store_wait_read();
          __syncwarp();
          store_pending = false;
        }
        uint8_t* srow = sP + r * 128;   // (P lives in tensor memory: sP is only the O staging buffer here)
#pragma unroll
        for (int c = 0; c < DH / 32; ++c)
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            uint32_t wv[4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
              wv[i] = bf2_cvt(__uint_as_float(o[c][8 * g + 2 * i]) * osc, __uint_as_float(o[c][8 * g + 2 * i + 1]) * osc);
            const int col = c * 32 + 8 * g;
            const int ch = (col >> 3) ^ (r & 7);
            *reinterpret_cast<uint4*>(srow + (ch << 4)) = make_uint4(wv[0], wv[1], wv[2], wv[3]);
          }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_3d(&tmO, sP + quarter * 32 * 128, 0, it.head, (int)(row0 + it.q0 + quarter * 32));
          tma_store_commit();
        }
        store_pending = true;
      } else if (qi < N) {
        bf16* op = p.out + (row0 + qi) * p.ld_out + it.head * p.d;
#pragma unroll
        for (int c = 0; c < DH / 32; ++c)
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            uint32_t wv[4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
              wv[i] = bf2_cvt(__uint_as_float(o[c][8 * g + 2 * i]) * osc, __uint_as_float(o[c][8 * g + 2 * i + 1]) * osc);
            if (c * 32 + 8 * g < p.d) st_global_v4(op + c * 32 + 8 * g, wv[0], wv[1], wv[2], wv[3]);   // not the zero columns past d
          }
      }
      if (prof) { c_epi_wait += e1 - e0; c_epi += clock64() - e1; }
    }
    if (store_pending && lane == 0) tma_store_wait_read();
    if (prof) {
      const long long tot = clock64() - c_begin;
      atomicAdd(&p.prof[0], (unsigned long long)c_wait_s); atomicAdd(&p.prof[1], (unsigned long long)c_load);
      atomicAdd(&p.prof[2], (unsigned long long)c_max); atomicAdd(&p.prof[3], (unsigned long long)c_wait_pv);
      atomicAdd(&p.prof[4], (unsigned long long)c_exp); atomicAdd(&p.prof[5], (unsigned long long)c_tail);
      atomicAdd(&p.prof[6], (unsigned long long)c_epi_wait); atomicAdd(&p.prof[7], (unsigned long long)c_epi);
      atomicAdd(&p.prof[8], (unsigned long long)tot); atomicAdd(&p.prof[9], (unsigned long long)n_t);
    }
#undef PCLK
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem_base, S::TMEM_COLS);
  }
}

// Q / K / V / O of every kernel: one head per map coordinate, so a head narrower than the kernel's tile width (d < DH) loads its
// pad columns as zeros -- they add nothing to S = Q K^T or to P V -- and stores only its own d columns.
static int encode_attn_maps(const AttnArgs& a, long long Mrows, CUtensorMap* tmQ, CUtensorMap* tmK, CUtensorMap* tmV, CUtensorMap* tmO) {
  if (encode_tmap_heads(tmQ, a.q, a.d, a.heads, Mrows, a.ld_qkv, ATT_BQ)) return -1;
  if (encode_tmap_heads(tmK, a.k, a.d, a.heads, Mrows, a.ld_qkv, ATT_BKV)) return -1;
  if (encode_tmap_heads(tmV, a.v, a.d, a.heads, Mrows, a.ld_qkv, ATT_BKV)) return -1;
  return encode_tmap_heads(tmO, a.out, a.d, a.heads, Mrows, a.ld_out, 32);
}

static int launch_attention_persist(const AttnArgs& a, cudaStream_t stream) {
  using S = AttnShape<64, 1>;
  const bool packed = a.cu != nullptr;
  const long long Mrows = packed ? a.row_cap : (long long)a.B * a.N;
  if (packed && (!a.cuq || !a.grp_img || !a.grp_order || !a.kv_len || a.window >= 0 || a.row_cap <= 0 || a.grp_cap <= 0)) {
    set_error("attention: packed layout needs cu/cuq/grp_img/grp_order/kv_len, row and group capacities and no window");
    return -2;
  }
  CUtensorMap tmQ, tmK, tmV, tmO;
  if (encode_attn_maps(a, Mrows, &tmQ, &tmK, &tmV, &tmO)) return -1;
  AttnParams p;
  p.out = a.out; p.ld_out = a.ld_out;
  p.kv_len = a.kv_len;
  p.N = a.N; p.heads = a.heads; p.d = a.d; p.zero_invalid = a.zero_invalid_rows;
  p.tma_out = (packed || a.N % ATT_BQ == 0) ? 1 : 0;
  p.window = a.window;
  p.lse = a.lse;
  p.cu = a.cu; p.cuq = a.cuq; p.grp_img = a.grp_img; p.grp_order = a.grp_order; p.n_grp = a.cuq ? a.cuq + a.B : nullptr;
  p.prof = nullptr;
  static const int prof_mode = getenv("VTK_ATTN_PROF") ? atoi(getenv("VTK_ATTN_PROF")) : 0;
  static unsigned long long* d_prof = nullptr;
  if (prof_mode) {
    if (!d_prof) cudaMalloc(&d_prof, 16 * sizeof(unsigned long long));
    cudaMemsetAsync(d_prof, 0, 16 * sizeof(unsigned long long), stream);
    p.prof = d_prof;
  }
  p.scale_log2 = (float)((1.0 / sqrt((double)a.d)) * 1.4426950408889634);
  // P stays in tensor memory (A operand of the PV MMA read from TMEM, no 32 KB shared-memory round trip per tile): 3-4 % faster
  // than a shared-memory P buffer (43.9 vs 45.6 us at the c2 shape)
  auto kern = packed ? attn_persist_kernel<64, true> : attn_persist_kernel<64, false>;
  if (ensure_max_smem(reinterpret_cast<const void*>(kern), S::SMEM_BYTES, "cudaFuncSetAttribute(attn_persist)")) return -1;
  const int qtiles = (a.N + ATT_BQ - 1) / ATT_BQ;
  const long long total = packed ? (long long)a.grp_cap * a.heads : (long long)a.B * a.heads * qtiles;
  if (total >= (1ll << 31)) { set_error("attention: too many work items"); return -2; }
  const int grid = (int)std::min<long long>(total, 2ll * usable_sms());
  const cudaError_t lerr = launch_k(kern, dim3(grid), dim3(192), S::SMEM_BYTES, stream, tmQ, tmK, tmV, tmO, p, (int)total, qtiles);
  if (lerr != cudaSuccess) return check_cuda(lerr, "attention (persistent) launch");
  if (prof_mode) {
    unsigned long long h[16];
    cudaDeviceSynchronize();
    cudaMemcpy(h, d_prof, sizeof(h), cudaMemcpyDeviceToHost);
    const double nt = h[9] ? (double)h[9] : 1.0;
    fprintf(stderr, "[attn prof] persistent N=%d grid=%d: cycles per key tile (softmax warp 0): wait S %.0f | tmem load %.0f | mask+max %.0f | "
            "wait PV/store %.0f | exp+P %.0f | tail %.0f || per tile amortised: epilogue wait %.0f, epilogue %.0f, total %.0f\n",
            a.N, grid, h[0] / nt, h[1] / nt, h[2] / nt, h[3] / nt, h[4] / nt, h[5] / nt, h[6] / nt, h[7] / nt, h[8] / nt);
  }
  return check_cuda(cudaGetLastError(), "attention (persistent) launch");
}

template <int DH, int NQ>
static int launch_attention_t(const AttnArgs& a, cudaStream_t stream) {
  using S = AttnShape<DH, NQ>;
  const bool packed = a.cu != nullptr;
  if (packed && (!a.cuq || !a.grp_img || !a.kv_len || a.window >= 0 || a.row_cap <= 0 || a.grp_cap <= 0)) {
    set_error("attention: packed layout needs cu/cuq/grp_img/kv_len, row and group capacities and no window");
    return -2;
  }
  const long long Mrows = packed ? a.row_cap : (long long)a.B * a.N;
  CUtensorMap tmQ, tmK, tmV, tmO;
  if (encode_attn_maps(a, Mrows, &tmQ, &tmK, &tmV, &tmO)) return -1;
  AttnParams p;
  p.out = a.out; p.ld_out = a.ld_out;
  p.kv_len = a.kv_len;
  p.N = a.N; p.heads = a.heads; p.d = a.d; p.zero_invalid = a.zero_invalid_rows;
  p.tma_out = (packed || a.N % ATT_BQ == 0) ? 1 : 0;
  p.window = a.window;
  p.lse = a.lse;
  p.cu = a.cu; p.cuq = a.cuq; p.grp_img = a.grp_img; p.grp_order = a.grp_order; p.n_grp = a.cuq ? a.cuq + a.B : nullptr;
  p.scale_log2 = (float)((1.0 / sqrt((double)a.d)) * 1.4426950408889634);
  static const int prof_mode = getenv("VTK_ATTN_PROF") ? atoi(getenv("VTK_ATTN_PROF")) : 0;
  static unsigned long long* d_prof = nullptr;
  p.prof = nullptr;
  if (prof_mode) {
    if (!d_prof) cudaMalloc(&d_prof, 8 * sizeof(unsigned long long));
    cudaMemsetAsync(d_prof, 0, 8 * sizeof(unsigned long long), stream);
    p.prof = d_prof;
  }
  auto kern = attn_kernel<DH, NQ>;
  if (ensure_max_smem(reinterpret_cast<const void*>(kern), S::SMEM_BYTES, "cudaFuncSetAttribute(attn)")) return -1;
  dim3 grid((a.N + NQ * ATT_BQ - 1) / (NQ * ATT_BQ), a.heads, a.B);
  if (packed) grid = dim3((unsigned)a.grp_cap, a.heads, 1);
  const cudaError_t lerr = launch_k(kern, grid, dim3(S::THREADS), S::SMEM_BYTES, stream, tmQ, tmK, tmV, tmO, p);
  if (lerr != cudaSuccess) return check_cuda(lerr, "attention launch");
  if (prof_mode) {
    unsigned long long h[8];
    cudaDeviceSynchronize();
    cudaMemcpy(h, d_prof, sizeof(h), cudaMemcpyDeviceToHost);
    const double n = h[7] ? (double)h[7] : 1.0;
    fprintf(stderr, "[attn prof] d=%d NQ=%d N=%d: per CTA cycles: prologue %.0f | first S ready %.0f | wait S %.0f | wait PV in loop %.0f | "
            "wait last PV %.0f | epilogue %.0f | total %.0f (softmax+rest %.0f)\n", DH, NQ, a.N, h[0] / n, h[1] / n, h[2] / n, h[3] / n,
            h[4] / n, h[5] / n, h[6] / n, (h[6] - h[0] - h[1] - h[2] - h[3] - h[4] - h[5]) / n);
  }
  return check_cuda(cudaGetLastError(), "attention launch");
}

int launch_attention(const AttnArgs& a, cudaStream_t stream) {
  if (a.B <= 0 || a.N <= 0 || a.heads <= 0) { set_error("attention: empty problem"); return -2; }
  if ((a.ld_qkv % 8) || (a.ld_out % 8)) { set_error("attention: row strides must be multiples of 8"); return -2; }
  if (!head_dim_supported(a.d)) {
    set_error("attention: head_dim %d unsupported (supported: multiples of 8 from 8 to 128)", a.d);
    return -3;
  }
  if (head_tile(a.d) == 64) return launch_attention_persist(a, stream);
  return launch_attention_t<128, 2>(a, stream);
}

}  // namespace vtk
