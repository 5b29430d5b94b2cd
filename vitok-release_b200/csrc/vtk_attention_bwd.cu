// vtk_attention_bwd.cu -- attention backward on tcgen05 (training step, BASELINE config 5).
//
// Autograd of modules/attention.py:109-127 (flash_attn_func / scaled_dot_product_attention): given q, k, v
// (QK-normed, roped), dO, the forward's log2-domain logsumexp and delta = rowsum(dO * O):
//     P  = exp2(S * scale*log2e - lse)          S = q k^T
//     dV = P^T dO        dP = dO v^T        dS = P * (dP - delta) * scale
//     dQ = dS k          dK = dS^T q
// Two passes, each one CTA per 128-row tile, so that no accumulator is shared between CTAs (no atomics):
//   MODE 0 (dK/dV): CTA = key tile j (K_j, V_j resident in smem); loops over query tiles i; accumulates dV_j, dK_j in TMEM
//   MODE 1 (dQ)   : CTA = query tile i (Q_i, dO_i resident);      loops over key tiles j;   accumulates dQ_i in TMEM
// Every step runs S and dP on the tensor core (both K-major), 128 threads (thread <-> query row, the TMEM lane)
// turn them into P and dS as bf16 in 128B-swizzled shared memory, and the second group of MMAs consumes them:
//   dV += P^T dO, dK += dS^T Q : A = the [query x key] tile read MN-major (transposed by the descriptor),
//                                B = dO / Q read MN-major straight from their [row, d] layout
//   dQ += dS K                 : A = dS K-major, B = K_j MN-major
// The step loop itself is serial (S / dP -> P / dS -> second MMA group), but the TMA thread fetches ahead: both streamed tiles
// of the next step in MODE 1, Q_i in MODE 0 (see the buffer comment in the kernel).  S/dP recomputation makes it 7 MMAs per
// tile pair instead of the minimal 5.  Attention is ~5 % of the step's FLOPs at config 5.
// Two compute warpgroups (warps 0-3 and 8-11) split every [128 x 128] S / dP tile by columns (64 keys each; a warp may
// only read the TMEM lanes of its quarter, so both groups own the same rows), which halves the P / dS latency that
// sits between the two MMA groups; tiles that need no masking skip the per-element key test.
// Packed NaFlex layout (vtk_attention_bwd_packed_bf16, the training step with AE.train_token_packing): the same two passes over
// 128-row tiles of one image, image b at packed rows [cu[b], cu[b] + n_valid[b]); the grid is the plan's compact work list of
// (128-row group, head) instead of (tiles, heads, B).  Stores stay inside [cu[b], cu[b+1]) (zeros for the image's pad rows), and MODE 0
// masks query rows >= n_valid[b] explicitly: after a partial last tile they are the next image's rows, whose dO is not 0.
#include <math.h>
#include <stdio.h>

#include "vtk_common.cuh"
#include "vtk_kernels.h"

namespace vtk {

static constexpr int BWD_T = 128;      // tile edge (queries and keys)
static constexpr int BWD_BLK = 16384;  // one [128 x 64] bf16 swizzled block

template <int DH> struct BwdShape {
  static constexpr int NB = DH / 64;
  static constexpr int TILE = NB * BWD_BLK;
  static constexpr int OFF_R0 = 0;                 // resident tile 0 (MODE 0: K_j, MODE 1: Q_i)
  static constexpr int OFF_R1 = TILE;              // resident tile 1 (MODE 0: V_j, MODE 1: dO_i)
  static constexpr int OFF_S0 = 2 * TILE;          // streamed tile 0 (MODE 0: Q_i, MODE 1: K_j)
  static constexpr int OFF_S1 = 3 * TILE;          // streamed tile 1 (MODE 0: dO_i, MODE 1: V_j)
  static constexpr int OFF_P = 4 * TILE;           // P  [128 q x 128 k] bf16 (2 blocks)
  static constexpr int OFF_DS = OFF_P + 2 * BWD_BLK;
  static constexpr int OFF_X = OFF_DS + 2 * BWD_BLK;   // one extra tile: MODE 0 second Q_i buffer; MODE 1 second V_j buffer (its second K_j
                                                       // buffer is the P region, which MODE 1 does not write)
  static constexpr int OFF_BAR = OFF_X + TILE;
  static constexpr int SMEM_BYTES = OFF_BAR + 128;     // d = 128: 229 504 bytes (limit 232 448)
  // TMEM columns: S [0,128) dP [128,256) acc0 [256, 256+DH) acc1 [256+DH, 256+2DH)
};

static __device__ __forceinline__ float ex2_approx_bwd(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

struct BwdParams {
  const float* lse; const float* delta;
  bf16* dq; bf16* dk; bf16* dv; long long ld_d;
  const int* kv_len;
  int N, heads, d, zero_invalid, window;   // d = the true head width (<= DH; columns d..DH-1 of a tile are TMA zero fill)
  float scale, scale_log2;
  // packed layout (PACKED kernels): image b = rows [cu[b], cu[b+1]), kv_len[b] valid tokens in front; 128-row group g is the
  // (g - cuq[img])-th tile of img = grp_img[g]; *n_grp groups exist, grp_order lists them longest image first
  const int* cu; const int* cuq; const int* grp_img; const int* grp_order; const int* n_grp;
};

// P and dS of one 32-key chunk of a row: P = exp2(S * scale*log2e - lse), dS = P * (dP - delta) * scale, written as bf16
// into the row's 128B-swizzled slots.  MASKED = false: every key of the chunk is live (no per-element test).  qlive = false
// (packed MODE 0: a query row past the image end, which belongs to the next image): P and dS of the whole row are 0.
template <int MODE, bool MASKED>
__device__ __forceinline__ void bwd_chunk(const uint32_t (&sv)[32], const uint32_t (&dv)[32], float lse_r, float delta_r,
                                          float scale_log2, float scale, int kc0, int kvlen, int W, int qi, bool qlive, uint8_t* prow,
                                          uint8_t* dsrow, int c, int r) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    uint32_t pp[4], dd[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float pv[2], dsv[2];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int col = 8 * g + 2 * i + e;
        float pe = ex2_approx_bwd(fmaf(__uint_as_float(sv[col]), scale_log2, -lse_r));
        if (MASKED) {
          const int kc = kc0 + col;
          const bool ok = qlive && kc < kvlen && (W < 0 || abs(kc - qi) <= W);
          pe = ok ? pe : 0.f;
        }
        pv[e] = pe;
        dsv[e] = pe * (__uint_as_float(dv[col]) - delta_r) * scale;
        if (MASKED) dsv[e] = qlive ? dsv[e] : 0.f;   // the next image's dP may be anything: no 0 * inf
      }
      pp[i] = bf2_cvt(pv[0], pv[1]);
      dd[i] = bf2_cvt(dsv[0], dsv[1]);
    }
    const int gg = c * 4 + g;   // 16-byte chunk index along the 128 keys
    const int blk = gg >> 3, ch = (gg & 7) ^ (r & 7);
    if (MODE == 0) *reinterpret_cast<uint4*>(prow + blk * BWD_BLK + (ch << 4)) = make_uint4(pp[0], pp[1], pp[2], pp[3]);
    *reinterpret_cast<uint4*>(dsrow + blk * BWD_BLK + (ch << 4)) = make_uint4(dd[0], dd[1], dd[2], dd[3]);
  }
}

// PACKED: the packed NaFlex layout.  One CTA per (128-row group of one image, head) from the plan's work list instead of a
// (tiles, heads, B) grid; N becomes the image's packed row count (valid rows, then its pad rows, which get zero gradients), and
// MODE 0 masks query rows >= kv_len explicitly: in the padded layout those rows are the image's own padding (dO = 0, lse = +inf),
// here the rows after a partial last query tile belong to the next image.
template <int DH, int MODE, bool PACKED>
__global__ void __launch_bounds__(384, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmDO, const BwdParams p) {
  using S = BwdShape<DH>;
  int tile0, head, img, N, kvlen;   // tile0 = MODE 0: first key of this CTA; MODE 1: first query
  long long row0;
  if (PACKED) {
    const int rank = blockIdx.x / p.heads;
    if (rank >= __ldg(p.n_grp)) return;   // beyond the groups of this batch (whole CTA)
    head = blockIdx.x - rank * p.heads;
    const int grp = p.grp_order[rank];
    img = p.grp_img[grp];
    row0 = p.cu[img];
    N = p.cu[img + 1] - (int)row0;
    kvlen = p.kv_len[img];
    tile0 = (grp - p.cuq[img]) * BWD_T;
  } else {
    tile0 = blockIdx.x * BWD_T;
    head = blockIdx.y;
    img = blockIdx.z;
    N = p.N;
    kvlen = p.kv_len ? p.kv_len[img] : N;
    kvlen = kvlen < N ? kvlen : N;
    row0 = (long long)img * N;
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qlimit = p.zero_invalid ? kvlen : N;
  const int W = p.window;

  // the range of the OTHER dimension's tiles this CTA visits
  int t_lo = 0, t_hi;
  if (MODE == 0) {
    t_hi = (qlimit + BWD_T - 1) / BWD_T - 1;                 // query tiles with at least one live row
    if (W >= 0) {
      t_lo = max(0, tile0 - W) / BWD_T;
      t_hi = min(t_hi, (min(tile0 + BWD_T - 1, N - 1) + W) / BWD_T);
    }
  } else {
    t_hi = (kvlen + BWD_T - 1) / BWD_T - 1;
    if (W >= 0) {
      t_lo = max(0, tile0 - W) / BWD_T;
      t_hi = min(t_hi, (min(tile0 + BWD_T - 1, N - 1) + W) / BWD_T);
    }
  }
  const bool dead = (MODE == 0) ? (tile0 >= kvlen) : (tile0 >= qlimit);
  const int steps = dead ? 0 : (t_hi - t_lo + 1);

  if (steps <= 0) {   // nothing contributes: the gradient rows of this tile are 0
    if (warp < 4) {
      const int ri = tile0 + warp * 32 + lane;
      if (ri < N) {
        if (MODE == 0) {
          bf16* a = p.dk + (row0 + ri) * p.ld_d + head * p.d;
          bf16* b = p.dv + (row0 + ri) * p.ld_d + head * p.d;
          for (int c = 0; c < p.d; c += 8) { st_global_v4(a + c, 0u, 0u, 0u, 0u); st_global_v4(b + c, 0u, 0u, 0u, 0u); }
        } else {
          bf16* a = p.dq + (row0 + ri) * p.ld_d + head * p.d;
          for (int c = 0; c < p.d; c += 8) st_global_v4(a + c, 0u, 0u, 0u, 0u);
        }
      }
    }
    return;
  }

  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sR0 = smem + S::OFF_R0;
  uint8_t* sR1 = smem + S::OFF_R1;
  uint8_t* sS0 = smem + S::OFF_S0;
  uint8_t* sS1 = smem + S::OFF_S1;
  uint8_t* sP = smem + S::OFF_P;
  uint8_t* sDS = smem + S::OFF_DS;
  // The step loop is serial (load -> S / dP -> P / dS -> second MMA group), so whatever the TMA thread cannot fetch ahead is exposed:
  // ~2 300 of the ~8 000 cycles of a step were the 64 KB of streamed tiles.  MODE 1 (dQ) does not write P, which leaves room for a
  // SECOND pair of streamed tiles (K_j in the P region, V_j in the extra tile X): its loads run one step ahead.  MODE 0 needs K, V, Q, dO,
  // P, dS = 192 KB at d = 128; the extra tile double-buffers Q_i only, so the S MMAs of the next step start at once and only the dO load
  // (half the bytes, partly under those MMAs) stays exposed.  Each streamed tile has its own full / free barriers.
  constexpr int NB0 = 2, NB1 = MODE == 1 ? 2 : 1;          // buffers of stream tile 0 / 1
  uint8_t* sSb0[2] = {sS0, smem + (MODE == 1 ? S::OFF_P : S::OFF_X)};
  uint8_t* sSb1[2] = {sS1, smem + S::OFF_X};               // (second entry used by MODE 1 only)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* res_full = bars + 0;   // resident tiles landed
  uint64_t* s0_full = bars + 1;    // [2] stream tile 0 of a step landed (buffer = step % NB0)
  uint64_t* s0_free = bars + 3;    // [2] the second MMA group of that step has read it
  uint64_t* s1_full = bars + 5;    // [2] stream tile 1 (buffer = step % NB1)
  uint64_t* s1_free = bars + 7;    // [2]
  uint64_t* sdp_full = bars + 9;   // S and dP of this step are in TMEM
  uint64_t* sdp_free = bars + 10;  // count 256: threads have pulled S / dP into registers
  uint64_t* pds_full = bars + 11;  // count 256: P and dS of this step are in smem
  uint64_t* acc_done = bars + 12;  // all MMAs finished (epilogue)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 14);

  if (warp == 4) {
    if (lane < 13) mbar_init(&bars[lane], (lane == 10 || lane == 11) ? 256u : 1u);
    else if (lane == 16) tma_prefetch_desc(&tmQ);
    else if (lane == 17) tma_prefetch_desc(&tmK);
    else if (lane == 18) tma_prefetch_desc(&tmV);
    else if (lane == 19) tma_prefetch_desc(&tmDO);
    fence_barrier_init();
    __syncwarp();
  }
  if (warp == 5) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    if (lane == 0) {
      // ===== TMA producer =====
      const CUtensorMap* mR0 = MODE == 0 ? &tmK : &tmQ;
      const CUtensorMap* mR1 = MODE == 0 ? &tmV : &tmDO;
      const CUtensorMap* mS0 = MODE == 0 ? &tmQ : &tmK;
      const CUtensorMap* mS1 = MODE == 0 ? &tmDO : &tmV;
      mbar_expect_tx(res_full, 2 * S::TILE);
      for (int nb = 0; nb < S::NB; ++nb) {
        tma_load_3d(sR0 + nb * BWD_BLK, mR0, res_full, nb * 64, head, (int)(row0 + tile0));
        tma_load_3d(sR1 + nb * BWD_BLK, mR1, res_full, nb * 64, head, (int)(row0 + tile0));
      }
      // issue order: tile 0 of step t, then tile 1 of step t -- with NB1 = 1 the wait for tile 1's buffer (the previous step's second MMA
      // group) comes AFTER tile 0 of this step has been requested, so tile 0 always runs a step ahead
      for (int t = 0; t < steps; ++t) {
        const int other0 = (t_lo + t) * BWD_T;
        const int b0 = t % NB0, b1 = t % NB1;
        if (t >= NB0) mbar_wait(&s0_free[b0], (uint32_t)(t / NB0 - 1) & 1u);   // the step that used this buffer last is done with it
        mbar_expect_tx(&s0_full[b0], S::TILE);
        for (int nb = 0; nb < S::NB; ++nb) tma_load_3d(sSb0[b0] + nb * BWD_BLK, mS0, &s0_full[b0], nb * 64, head, (int)(row0 + other0));
        if (t >= NB1) mbar_wait(&s1_free[b1], (uint32_t)(t / NB1 - 1) & 1u);
        mbar_expect_tx(&s1_full[b1], S::TILE);
        for (int nb = 0; nb < S::NB; ++nb) tma_load_3d(sSb1[b1] + nb * BWD_BLK, mS1, &s1_full[b1], nb * 64, head, (int)(row0 + other0));
      }
    }
  } else if (warp == 5) {
    if (lane == 0) {
      // ===== MMA issuer =====
      const uint32_t idesc_s = make_idesc_bf16(BWD_T, BWD_T, 0, 0);      // S, dP: both operands K-major
      const uint32_t idesc_tt = make_idesc_bf16(BWD_T, DH, 1, 1);        // dV, dK: A and B MN-major
      const uint32_t idesc_q = make_idesc_bf16(BWD_T, DH, 0, 1);         // dQ: A K-major, B MN-major
      const uint32_t aP = smem_u32(sP), aDS = smem_u32(sDS);
      mbar_wait(res_full, 0);
      for (int t = 0; t < steps; ++t) {
        const int b0 = t % NB0, b1 = t % NB1;
        // operands by role
        const uint32_t aQ = smem_u32(MODE == 0 ? sSb0[b0] : sR0), aK = smem_u32(MODE == 0 ? sR0 : sSb0[b0]);
        const uint32_t aDO = smem_u32(MODE == 0 ? sSb1[b1] : sR1), aV = smem_u32(MODE == 0 ? sR1 : sSb1[b1]);
        mbar_wait(&s0_full[b0], (uint32_t)(t / NB0) & 1u);
        if (t > 0) mbar_wait(sdp_free, (uint32_t)(t - 1) & 1u);
        tc_fence_after();
#pragma unroll
        for (int kk = 0; kk < DH / 16; ++kk) {
          const uint32_t off = (kk >> 2) * BWD_BLK + (kk & 3) * 32;
          umma_bf16_ss(tmem_base + 0, make_desc_kmajor_sw128(aQ + off), make_desc_kmajor_sw128(aK + off), idesc_s, kk != 0);
        }
        mbar_wait(&s1_full[b1], (uint32_t)(t / NB1) & 1u);
        tc_fence_after();
#pragma unroll
        for (int kk = 0; kk < DH / 16; ++kk) {
          const uint32_t off = (kk >> 2) * BWD_BLK + (kk & 3) * 32;
          umma_bf16_ss(tmem_base + 128, make_desc_kmajor_sw128(aDO + off), make_desc_kmajor_sw128(aV + off), idesc_s, kk != 0);
        }
        umma_commit(sdp_full);
        mbar_wait(pds_full, (uint32_t)t & 1u);
        tc_fence_after();
        if (MODE == 0) {
#pragma unroll
          for (int kk = 0; kk < BWD_T / 16; ++kk) {   // contraction over the 128 queries, 16 per MMA
            // A: [query x key] tile, MN-major (M = keys): LBO = stride between the two 64-key blocks, SBO = 8-query group
            const uint64_t aPt = make_smem_desc(aP + kk * 2048, BWD_BLK, 1024, 2);
            const uint64_t aDSt = make_smem_desc(aDS + kk * 2048, BWD_BLK, 1024, 2);
            // B: [query x d] tile, MN-major (N = d)
            const uint64_t bDO = make_smem_desc(aDO + kk * 2048, BWD_BLK, 1024, 2);
            const uint64_t bQ = make_smem_desc(aQ + kk * 2048, BWD_BLK, 1024, 2);
            umma_bf16_ss(tmem_base + 256, aPt, bDO, idesc_tt, (t | kk) != 0);          // dV += P^T dO
            umma_bf16_ss(tmem_base + 256 + DH, aDSt, bQ, idesc_tt, (t | kk) != 0);    // dK += dS^T Q
          }
        } else {
#pragma unroll
          for (int kk = 0; kk < BWD_T / 16; ++kk) {   // contraction over the 128 keys
            const uint64_t aD = make_desc_kmajor_sw128(aDS + (kk >> 2) * BWD_BLK + (kk & 3) * 32);
            const uint64_t bK = make_smem_desc(aK + kk * 2048, BWD_BLK, 1024, 2);
            umma_bf16_ss(tmem_base + 256, aD, bK, idesc_q, (t | kk) != 0);            // dQ += dS K
          }
        }
        umma_commit(&s0_free[b0]);
        umma_commit(&s1_free[b1]);
      }
      umma_commit(acc_done);
    }
  } else if (warp < 4 || warp >= 8) {
    // ===== compute warps: thread <-> query row of the current query tile; column half = warpgroup =====
    const int half = warp >> 3;   // 0: keys [0, 64) of the tile, 1: keys [64, 128)
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    uint8_t* prow = sP + r * 128;
    uint8_t* dsrow = sDS + r * 128;
    float lse_r = INFINITY, delta_r = 0.f;
    int qi = 0;
    if (MODE == 1) {
      qi = tile0 + r;
      if (qi < qlimit) {
        lse_r = p.lse[(row0 + qi) * p.heads + head];
        delta_r = p.delta[(row0 + qi) * p.heads + head];
      }
    }
    for (int t = 0; t < steps; ++t) {
      const int other0 = (t_lo + t) * BWD_T;
      const int k0 = MODE == 0 ? tile0 : other0;    // first key of the tile pair
      if (MODE == 0) {
        qi = other0 + r;
        lse_r = INFINITY;
        delta_r = 0.f;
        if (qi < qlimit) {
          lse_r = p.lse[(row0 + qi) * p.heads + head];
          delta_r = p.delta[(row0 + qi) * p.heads + head];
        }
      }
      mbar_wait(sdp_full, (uint32_t)t & 1u);
      __syncwarp();
      tc_fence_after();
      if (t > 0) {   // P / dS buffers are free once the previous step's second MMA group has completed
        mbar_wait(&s1_free[(t - 1) % NB1], (uint32_t)((t - 1) / NB1) & 1u);
        __syncwarp();
      }
      // warp-uniform; packed MODE 0 also masks the query rows of an image's partial last query tile
      const bool row_mask = PACKED && MODE == 0 && other0 + BWD_T > qlimit;
      const bool need_mask = (k0 + BWD_T > kvlen) || W >= 0 || row_mask;
      const bool qlive = !row_mask || qi < qlimit;
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const int c = 2 * half + cc;
        uint32_t sv[32], dv[32];
        tmem_ld32(tmem_base + lane_base + c * 32, sv);
        tmem_ld32(tmem_base + lane_base + 128 + c * 32, dv);
        tmem_wait_ld();
        if (need_mask) bwd_chunk<MODE, true>(sv, dv, lse_r, delta_r, p.scale_log2, p.scale, k0 + c * 32, kvlen, W, qi, qlive, prow, dsrow, c, r);
        else bwd_chunk<MODE, false>(sv, dv, lse_r, delta_r, p.scale_log2, p.scale, k0 + c * 32, kvlen, W, qi, true, prow, dsrow, c, r);
      }
      tc_fence_before();
      mbar_arrive(sdp_free);
      fence_proxy_async_smem();
      mbar_arrive(pds_full);
    }
    // epilogue: accumulators -> bf16 rows of dK/dV (MODE 0: TMEM lane = key) or dQ (MODE 1: lane = query)
    mbar_wait(acc_done, 0);
    __syncwarp();
    tc_fence_after();
    const int ri = tile0 + r;
#pragma unroll
    for (int a = 0; a < (MODE == 0 ? 2 : 1); ++a) {
      bf16* base = MODE == 0 ? (a == 0 ? p.dv : p.dk) : p.dq;
      bf16* op = base + (row0 + ri) * p.ld_d + head * p.d;
      const bool live = MODE == 0 ? (ri < kvlen) : (ri < qlimit);
#pragma unroll
      for (int c = half * (DH / 2); c < (half + 1) * (DH / 2); c += 32) {
        uint32_t o[32];
        tmem_ld32(tmem_base + lane_base + 256 + a * DH + c, o);
        tmem_wait_ld();
        if (ri < N) {
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            if (c + 8 * g >= p.d) break;   // the tile's columns past the head width
            uint32_t w[4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
              w[i] = live ? bf2_cvt(__uint_as_float(o[8 * g + 2 * i]), __uint_as_float(o[8 * g + 2 * i + 1])) : 0u;
            st_global_v4(op + c + 8 * g, w[0], w[1], w[2], w[3]);
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <int DH, bool PACKED>
static int launch_bwd_t(const AttnBwdArgs& a, cudaStream_t stream) {
  using S = BwdShape<DH>;
  const long long Mrows = PACKED ? a.row_cap : (long long)a.B * a.N;
  // one head per map coordinate: at d < DH the pad columns of Q, K, V and dO load as zeros (dP = dO V^T needs them in dO too)
  CUtensorMap tmQ, tmK, tmV, tmDO;
  if (encode_tmap_heads(&tmQ, a.q, a.d, a.heads, Mrows, a.ld_qkv, BWD_T)) return -1;
  if (encode_tmap_heads(&tmK, a.k, a.d, a.heads, Mrows, a.ld_qkv, BWD_T)) return -1;
  if (encode_tmap_heads(&tmV, a.v, a.d, a.heads, Mrows, a.ld_qkv, BWD_T)) return -1;
  if (encode_tmap_heads(&tmDO, a.dout, a.d, a.heads, Mrows, a.ld_do, BWD_T)) return -1;
  BwdParams p;
  p.lse = a.lse; p.delta = a.delta; p.dq = a.dq; p.dk = a.dk; p.dv = a.dv; p.ld_d = a.ld_d; p.kv_len = a.kv_len;
  p.N = a.N; p.heads = a.heads; p.d = a.d; p.zero_invalid = PACKED ? 1 : a.zero_invalid_rows; p.window = PACKED ? -1 : a.window;
  p.scale = (float)(1.0 / sqrt((double)a.d));
  p.scale_log2 = (float)((1.0 / sqrt((double)a.d)) * 1.4426950408889634);
  p.cu = a.cu; p.cuq = a.cuq; p.grp_img = a.grp_img; p.grp_order = a.grp_order; p.n_grp = a.cuq ? a.cuq + a.B : nullptr;
  auto k0 = attn_bwd_kernel<DH, 0, PACKED>;
  auto k1 = attn_bwd_kernel<DH, 1, PACKED>;
  if (ensure_max_smem(reinterpret_cast<const void*>(k0), S::SMEM_BYTES, "attr(attn_bwd0)")) return -1;
  if (ensure_max_smem(reinterpret_cast<const void*>(k1), S::SMEM_BYTES, "attr(attn_bwd1)")) return -1;
  dim3 grid((a.N + BWD_T - 1) / BWD_T, a.heads, a.B);
  if (PACKED) grid = dim3((unsigned)((long long)a.grp_cap * a.heads));
  k0<<<grid, 384, S::SMEM_BYTES, stream>>>(tmQ, tmK, tmV, tmDO, p);
  if (check_cuda(cudaGetLastError(), "attention bwd (dK/dV) launch")) return -1;
  k1<<<grid, 384, S::SMEM_BYTES, stream>>>(tmQ, tmK, tmV, tmDO, p);
  return check_cuda(cudaGetLastError(), "attention bwd (dQ) launch");
}

int launch_attention_bwd(const AttnBwdArgs& a, cudaStream_t stream) {
  const bool packed = a.cu != nullptr;   // (N is not used by the packed layout)
  if (a.B <= 0 || (!packed && a.N <= 0) || a.heads <= 0) { set_error("attention_bwd: empty problem"); return -2; }
  if ((a.ld_qkv % 8) || (a.ld_do % 8) || (a.ld_d % 8)) { set_error("attention_bwd: row strides must be multiples of 8"); return -2; }
  if (packed && (!a.cuq || !a.grp_img || !a.grp_order || !a.kv_len || a.row_cap <= 0 || a.grp_cap <= 0 ||
                 (long long)a.grp_cap * a.heads >= (1ll << 31))) {
    set_error("attention_bwd: packed layout needs cu/cuq/grp_img/grp_order/kv_len and positive row and group capacities");
    return -2;
  }
  if (!head_dim_supported(a.d)) {
    set_error("attention_bwd: head_dim %d unsupported (supported: multiples of 8 from 8 to 128)", a.d);
    return -3;
  }
  if (head_tile(a.d) == 64) return packed ? launch_bwd_t<64, true>(a, stream) : launch_bwd_t<64, false>(a, stream);
  return packed ? launch_bwd_t<128, true>(a, stream) : launch_bwd_t<128, false>(a, stream);
}

}  // namespace vtk
