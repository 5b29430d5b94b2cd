// vtk_gemm.cu -- persistent, warp-specialised tcgen05 GEMM for sm_100a with fused epilogues.
//
//   out = epilogue( A[M,K] (bf16, K-major) x B[N,K]^T (bf16, K-major) ), fp32 accumulation in TMEM.
//
// Roles (one CTA per SM, 128 + 32*NEPI threads):
//   warp 0   : TMA producer  -- cp.async.bulk.tensor 128B-swizzled boxes into a smem ring
//   warp 1   : MMA issuer    -- one lane issues tcgen05.mma (128 x {256|128} x 16), commits to mbarriers
//   warp 2   : TMEM allocator (2 accumulator buffers so the epilogue of tile i overlaps the MMAs of tile i+1)
//   warp 3   : idle
//   warps 4..: epilogue      -- 8 or 16 warps; tcgen05.ld (32x32b: one accumulator row per thread), fused math,
//                               16-byte stores
//
// Tile scheduler: static persistent, m fastest (concurrent CTAs share the same weight rows in L2).  When the
// last wave would be less than half full, its tiles are split into half-width tiles (UMMA N = BN/2) so the
// tail costs half a wave instead of a full one.
//
// Fused epilogues replace these reference call sites (/root/reference):
//   EPI_BIAS        nn.Linear + bias                      vitok/models/ae.py:191,220,242
//   EPI_BIAS_LN     to_code + LayerNorm(no affine)        vitok/models/ae.py:207, modules/norm.py:28-39
//   EPI_QKV_SWIGLU  qkv_proj -> norm_q/norm_k -> RoPE     modules/attention.py:95-107, rotary_embedding.py:102-129
//                   fc1 -> chunk -> silu(g) * v           modules/mlp.py:21-22
//   EPI_RESID       out_proj + fc2 -> LayerScale -> +x    vitok/models/ae.py:62-65, modules/layerscale.py:23
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>

#include "vtk_common.cuh"
#include "vtk_kernels.h"

namespace vtk {

static constexpr int BM = 128;
static constexpr int BK = 64;                        // 64 bf16 = one 128-byte swizzle atom
static constexpr int A_STAGE_BYTES = BM * BK * 2;    // 16 KB
static constexpr int SMEM_BUDGET = 192 * 1024;

static constexpr int OUT_GRANULE_BYTES = 2048;       // [32 rows x 32 cols] bf16 staging block (two per epilogue warp)

template <int BN> struct GemmShape {
  static constexpr int B_STAGE_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  static constexpr int STAGES = SMEM_BUDGET / STAGE_BYTES;
  static constexpr int TMEM_COLS = (2 * BN < 32) ? 32 : 2 * BN;
  // ring | per-warp output staging (TMA-store epilogues only) | barriers | fp32 q/k norm weights | alignment slack
  static constexpr int smem_bytes(int out_warps) { return STAGES * STAGE_BYTES + out_warps * 2 * OUT_GRANULE_BYTES + 256 + 1024 + 1024; }
};

// Per-warp staging block for the TMA-store epilogues: 32 rows (this warp's TMEM lanes) x 32 bf16 columns,
// 64-byte rows, SWIZZLE_64B (16-byte chunk index ^= (row >> 1) & 3) so that the 32 lanes' 16-byte writes
// are bank-conflict free and the block can be written to global memory as full 64-byte row segments by
// one cp.async.bulk.tensor store (clipped at the tensor bounds) instead of 32 row-strided 16-byte stores.
struct OutStage {
  uint8_t* base;     // two granule buffers per warp: the TMA store of one drains while the next is filled
  int lane, row0, cur;
  __device__ __forceinline__ void begin() {
    cur ^= 1;
    if (lane == 0) tma_store_wait_read_le1();   // the store issued from this buffer two granules ago has read it
    __syncwarp();
  }
  __device__ __forceinline__ void put(int chunk, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    *reinterpret_cast<uint4*>(base + cur * OUT_GRANULE_BYTES + lane * 64 + ((chunk ^ ((lane >> 1) & 3)) << 4)) =
        make_uint4(a, b, c, d);
  }
  __device__ __forceinline__ void flush(const CUtensorMap* tm, int col) {
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) {
      tma_store_2d(tm, base + cur * OUT_GRANULE_BYTES, col, row0);
      tma_store_commit();
    }
  }
};

struct TileSched {
  int num_m, num_n, gm, full_tiles, total_tiles, bn, bm;
  int workers;  // persistent workers (CTAs or CTA pairs) the schedule was built for = the launch grid
  int gm_cap;   // band height limit (tile rows) chosen on the host from the A-panel size
  int split;    // 1: a short last wave may be split into half-width tiles
  // Tile counts for M rows on `units` persistent workers (CTAs or CTA pairs).  Shared by the host launcher and by the
  // kernels that read M from device memory (NaFlex token packing: the packed row count is only known on the device).
  __host__ __device__ void setup(int M, int units) {
    num_m = (M + bm - 1) / bm;
    gm = gm_cap < num_m ? gm_cap : num_m;
    if (gm < 1) gm = 1;
    const int big = num_m * num_n;
    workers = big < units ? big : units;
    const int rem = workers > 0 ? big % workers : 0;
    full_tiles = big;
    total_tiles = big;
    if (split && rem > 0 && 2 * rem <= workers) {   // short last wave: half-width tiles
      full_tiles = big - rem;
      total_tiles = full_tiles + 2 * rem;
    }
    // Small problems (the per-GPU shards of a strong-scaled batch: M = 2048 rows x N = 1024 is 32 pair tiles for 74 pairs):
    // when cutting EVERY tile in half shortens the schedule -- cost in full-tile times: waves of full tiles (+ 1/2 for a
    // split last wave) against half-waves of half tiles -- all tiles are half-width, so twice as many workers are busy.
    if (split == 1 && workers > 0) {
      const int cur2 = 2 * ((full_tiles + workers - 1) / workers) + (total_tiles > full_tiles ? 1 : 0);   // in half-tile times
      const int hw = 2 * big < units ? 2 * big : units;
      const int half2 = (2 * big + hw - 1) / hw;
      if (half2 < cur2) {
        full_tiles = 0;
        total_tiles = 2 * big;
        workers = hw;
      }
    }
  }
  // Big tiles are visited in bands of `gm` row-tiles: inside a band m is fastest and n sweeps all column
  // tiles, so the band's A panel (gm x 128 x K) stays L2-resident while the weights stream through once
  // per band.  full_tiles big tiles, then (total_tiles - full_tiles) half-width tiles.
  __device__ __forceinline__ void big(int t, int& mi, int& ni) const {
    const int band_tiles = gm * num_n;
    const int band = t / band_tiles;
    const int r = t - band * band_tiles;
    const int rows = min(gm, num_m - band * gm);   // the last band may be short
    ni = r / rows;
    mi = band * gm + (r - ni * rows);
  }
  __device__ __forceinline__ void decode(int t, int& m0, int& n0, int& width) const {
    int mi, ni;
    if (t < full_tiles) {
      big(t, mi, ni);
      m0 = mi * bm;
      n0 = ni * bn;
      width = bn;
    } else {
      const int u = t - full_tiles;
      big(full_tiles + (u >> 1), mi, ni);
      m0 = mi * bm;
      n0 = ni * bn + (u & 1) * (bn >> 1);
      width = bn >> 1;
    }
  }
};

// ------------------------------------------------------------------------------------------------
// epilogue bodies.  One accumulator row per thread; work is done in 16-column chunks so that 16 epilogue
// warps (96 registers/thread) fit next to the 4 control warps.  Global operands (bias, gamma, RoPE table,
// norm weights, residual) are requested BEFORE the TMEM load so both latencies overlap.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void load_bf16x8(const bf16* p, float (&f)[8]) {
  uint4 v = ld_global_nc_v4(p);
  f[0] = bf16_lo(v.x); f[1] = bf16_hi(v.x); f[2] = bf16_lo(v.y); f[3] = bf16_hi(v.y);
  f[4] = bf16_lo(v.z); f[5] = bf16_hi(v.z); f[6] = bf16_lo(v.w); f[7] = bf16_hi(v.w);
}
__device__ __forceinline__ float u4_lo(const uint4& v, int i) {   // element 2i of 8 packed bf16
  const uint32_t w = i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w;
  return bf16_lo(w);
}
__device__ __forceinline__ float u4_hi(const uint4& v, int i) {   // element 2i+1
  const uint32_t w = i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w;
  return bf16_hi(w);
}

// GEMM output element pair as bf16: bf16(acc * rs) with rs = the row's fused-norm1 scale (1.0 when norm1 is not fused)
__device__ __forceinline__ uint32_t cvt_acc2(uint32_t lo_bits, uint32_t hi_bits, uint64_t rs2) {
  float a, b;
  f2_unpack(f2_mul(f2_pack(__uint_as_float(lo_bits), __uint_as_float(hi_bits)), rs2), a, b);
  return bf2_cvt(a, b);
}

// out = bf16(acc + bias)
__device__ __forceinline__ void epi_bias_unit(const EpiParams& p, uint32_t taddr, int row, bool row_ok, int n, int N,
                                              int ucols) {
  uint64_t ss2 = 0ull;   // sum of squares of this unit's bf16 outputs (fused norm1, see EpiParams::ss_out)
  for (int cc = 0; cc < ucols; cc += 16) {
    const int col = n + cc;
    if (col >= N) break;  // warp-uniform
    uint4 b0 = make_uint4(0, 0, 0, 0), b1 = make_uint4(0, 0, 0, 0);
    const bool second = col + 8 < N;
    if (p.bias) {
      b0 = ld_global_nc_v4(p.bias + col);
      if (second) b1 = ld_global_nc_v4(p.bias + col + 8);
    }
    uint4 a0 = make_uint4(0, 0, 0, 0), a1 = make_uint4(0, 0, 0, 0);   // accumulate: what `out` already holds
    if (p.accumulate && row_ok) {
      const bf16* ap = p.out + (long long)row * p.ldo + col;
      a0 = ld_global_v4(ap);
      if (second) a1 = ld_global_v4(ap + 8);
    }
    uint32_t r[16];
    tmem_ld16(taddr + cc, r);
    tmem_wait_ld();
    if (row_ok) {
      uint32_t o[8];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        o[i] = pack_bf16x2(__uint_as_float(r[2 * i]) + u4_lo(b0, i) + u4_lo(a0, i), __uint_as_float(r[2 * i + 1]) + u4_hi(b0, i) + u4_hi(a0, i));
        o[4 + i] = pack_bf16x2(__uint_as_float(r[8 + 2 * i]) + u4_lo(b1, i) + u4_lo(a1, i),
                               __uint_as_float(r[8 + 2 * i + 1]) + u4_hi(b1, i) + u4_hi(a1, i));
      }
      bf16* op = p.out + (long long)row * p.ldo + col;
      st_global_v4(op, o[0], o[1], o[2], o[3]);
      if (second) st_global_v4(op + 8, o[4], o[5], o[6], o[7]);
      if (p.ss_out) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (i >= 4 && !second) break;
          const uint64_t t = bf2_to_f2(o[i]);
          ss2 = f2_fma(t, t, ss2);
        }
      }
    }
  }
  if (p.ss_out && row_ok && n < N) {
    float s0, s1;
    f2_unpack(ss2, s0, s1);
    p.ss_out[(long long)row * p.ss_ld + (n >> 6)] = s0 + s1;
  }
}

// x = bf16(x + bf16(bf16(acc) * gamma)), in place; 32-column granules leave through the staging block.
// Packed bf16x2 arithmetic: bf2_mul(bf16(acc), gamma) and bf2_add(x, .) round exactly where the reference's
// eager bf16 ops do (layerscale.py:23, ae.py:64-65), at 1.5 instructions per element.
// partial (split-K, gemm2_kernel<..., SK>): the OTHER K-half's fp32 accumulator in shared memory, as [32 rows x 32 columns] blocks of
// 4 KB (128-byte rows, 16-byte chunks XOR-swizzled by row & 7; block = warp quarter * 8 + column / 32); the pointer addresses this
// thread's row in column block 0 of its quarter.  Added to the TMEM accumulator first; tcol = column of taddr inside the tile.
__device__ __forceinline__ void epi_resid_unit(const EpiParams& p, uint32_t taddr, int row, bool row_ok, int n, int N,
                                               int ucols, OutStage& st, const CUtensorMap* tmX, uint64_t rs2,
                                               const uint8_t* partial = nullptr, int tcol = 0) {
  uint64_t ss2 = 0ull;   // sum of squares of the new x over this 64-column unit (fused norm1 of the next block)
  for (int cc = 0; cc < ucols; cc += 32) {
    const int col = n + cc;
    if (col >= N) break;
    const int nch = min(4, (N - col) >> 3);   // 16-byte chunks of this granule inside the tensor (N % 8 == 0)
    const bf16* xp = p.out + (long long)row * p.ldo + col;
    uint4 xv[4], gv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      xv[j] = make_uint4(0, 0, 0, 0);
      gv[j] = make_uint4(0, 0, 0, 0);
      if (j < nch) {
        if (row_ok) xv[j] = ld_global_v4(xp + 8 * j);
        gv[j] = ld_global_nc_v4(p.gamma + col + 8 * j);
      }
    }
    uint32_t r[32];
    tmem_ld32(taddr + cc, r);
    tmem_wait_ld();
    if (partial) {
      const uint8_t* prow = partial + ((tcol + cc) >> 5) * 4096;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 pv = *reinterpret_cast<const float4*>(prow + ((j ^ (st.lane & 7)) << 4));
        r[4 * j + 0] = __float_as_uint(__uint_as_float(r[4 * j + 0]) + pv.x);
        r[4 * j + 1] = __float_as_uint(__uint_as_float(r[4 * j + 1]) + pv.y);
        r[4 * j + 2] = __float_as_uint(__uint_as_float(r[4 * j + 2]) + pv.z);
        r[4 * j + 3] = __float_as_uint(__uint_as_float(r[4 * j + 3]) + pv.w);
      }
    }
    st.begin();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t xs[4] = {xv[j].x, xv[j].y, xv[j].z, xv[j].w};
      const uint32_t gs[4] = {gv[j].x, gv[j].y, gv[j].z, gv[j].w};
      uint32_t o[4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
        o[i] = bf2_add(xs[i], bf2_mul(cvt_acc2(r[8 * j + 2 * i], r[8 * j + 2 * i + 1], rs2), gs[i]));   // rs2 = 1 unless FP8
      st.put(j, o[0], o[1], o[2], o[3]);
      if (p.ss_out && j < nch) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint64_t t = bf2_to_f2(o[i]);
          ss2 = f2_fma(t, t, ss2);
        }
      }
    }
    st.flush(tmX, col);
  }
  if (p.ss_out && row_ok && n < N) {
    float s0, s1;
    f2_unpack(ss2, s0, s1);
    p.ss_out[(long long)row * p.ss_ld + (n >> 6)] = s0 + s1;
  }
}

// bias[c, c + 16) as fp32; a last group of 8 columns (N % 16 == 8) reads zeros for the 8 past N
__device__ __forceinline__ void load_bias16(const bf16* bias, int c, int N, float (&b)[16]) {
  load_bf16x8(bias + c, *reinterpret_cast<float(*)[8]>(&b[0]));
  if (c + 8 < N) load_bf16x8(bias + c + 8, *reinterpret_cast<float(*)[8]>(&b[8]));
  else
#pragma unroll
    for (int i = 8; i < 16; ++i) b[i] = 0.f;
}

// LayerNorm without affine over all N (= C, a multiple of 8) columns of the row; the reference rounds the Linear output to
// bf16 first (nn.Linear in bf16), normalises in fp32 and rounds again (norm.py:39).
__device__ __forceinline__ void epi_bias_ln_row(const EpiParams& p, uint32_t taddr, int row, bool row_ok, int N) {
  float sum = 0.f;
  for (int c = 0; c < N; c += 16) {
    float b[16];
    load_bias16(p.bias, c, N, b);
    uint32_t r[16];
    tmem_ld16(taddr + c, r);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (i < 8 || c + 8 < N) sum += bf16r(__uint_as_float(r[i]) + b[i]);
  }
  const float mean = sum / (float)N;
  float var = 0.f;
  for (int c = 0; c < N; c += 16) {
    float b[16];
    load_bias16(p.bias, c, N, b);
    uint32_t r[16];
    tmem_ld16(taddr + c, r);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      float dv = bf16r(__uint_as_float(r[i]) + b[i]) - mean;
      if (i < 8 || c + 8 < N) var += dv * dv;
    }
  }
  const float rstd = rsqrtf(var / (float)N + p.eps);
  for (int c = 0; c < N; c += 16) {
    float b[16];
    load_bias16(p.bias, c, N, b);
    uint32_t r[16];
    tmem_ld16(taddr + c, r);
    tmem_wait_ld();
    uint32_t o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float v0 = (bf16r(__uint_as_float(r[2 * i]) + b[2 * i]) - mean) * rstd;
      float v1 = (bf16r(__uint_as_float(r[2 * i + 1]) + b[2 * i + 1]) - mean) * rstd;
      o[i] = pack_bf16x2(v0, v1);
    }
    if (row_ok) {
      bf16* op = p.out + (long long)row * p.ldo + c;
      st_global_v4(op, o[0], o[1], o[2], o[3]);
      if (c + 8 < N) st_global_v4(op + 8, o[4], o[5], o[6], o[7]);
    }
  }
}

// RoPE table layout ("pair-expanded, chunk-major", written by rope_table_kernel): per token row 2d bf16 =
//   C2[d] = (c_0, c_0, c_1, c_1, ...)  |  S2[d] = (-s_0, +s_0, -s_1, +s_1, ...)
// stored in 16-byte chunks so that the 32 rows of one epilogue warp are contiguous per chunk:
//   byte offset(row m, chunk c) = ((m >> 5) * (2d / 8) + c) * 512 + (m & 31) * 16
// -> a warp-wide 16-byte load touches 4 cache lines instead of 32, and the pair (c,c) / (-s,s) words feed
// HMUL2.BF16 directly:  out = Y * C2 + swap(Y) * S2   (rotary_embedding.py:121-124, bf16 rounding per op).
__device__ __forceinline__ const uint4* rope_row_ptr(const EpiParams& p, int rrow) {
  const long long grp = rrow >> 5;
  return reinterpret_cast<const uint4*>(p.rope) + (grp * (p.d >> 2)) * 32 + (rrow & 31);
}

// One q or k head: per-head RMSNorm over d (fp32, eps inside rsqrt; attention.py:103, norm.py:22-25) then
// interleaved-pair 2D RoPE.  w_s = this head kind's norm weight as fp32 in shared memory.
__device__ __forceinline__ void epi_qk_head(const EpiParams& p, uint32_t taddr, const uint4* rope_row, int ncol,
                                            const float* w_s, OutStage& st, const CUtensorMap* tmQKV, uint64_t rs2) {
  const int d = p.d;
  uint64_t ss2 = 0ull;
  for (int cc = 0; cc < d; cc += 32) {
    uint32_t r[32];
    tmem_ld32(taddr + cc, r);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const uint64_t t = bf2_to_f2(cvt_acc2(r[2 * i], r[2 * i + 1], rs2));   // q as the bf16 GEMM output
      ss2 = f2_fma(t, t, ss2);
    }
  }
  float s0, s1;
  f2_unpack(ss2, s0, s1);
  const float rstd = rsqrtf((s0 + s1) / (float)d + p.eps);
  const uint64_t rstd2 = f2_pack(rstd, rstd);
  const int s2_chunk0 = d >> 3;   // first chunk of the S2 half
  for (int cc = 0; cc < d; cc += 32) {
    uint4 c2[4], s2[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      c2[j] = ld_global_nc_v4(rope_row + ((cc >> 3) + j) * 32);
      s2[j] = ld_global_nc_v4(rope_row + (s2_chunk0 + (cc >> 3) + j) * 32);
    }
    uint32_t r[32];
    tmem_ld32(taddr + cc, r);
    tmem_wait_ld();
    st.begin();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 wa = *reinterpret_cast<const float4*>(w_s + cc + 8 * j);
      const float4 wb = *reinterpret_cast<const float4*>(w_s + cc + 8 * j + 4);
      const uint64_t w2[4] = {f2_pack(wa.x, wa.y), f2_pack(wa.z, wa.w), f2_pack(wb.x, wb.y), f2_pack(wb.z, wb.w)};
      const uint32_t cw[4] = {c2[j].x, c2[j].y, c2[j].z, c2[j].w};
      const uint32_t sw[4] = {s2[j].x, s2[j].y, s2[j].z, s2[j].w};
      uint32_t o[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint64_t t = bf2_to_f2(cvt_acc2(r[8 * j + 2 * i], r[8 * j + 2 * i + 1], rs2));
        float y0, y1;
        f2_unpack(f2_mul(f2_mul(t, rstd2), w2[i]), y0, y1);
        const uint32_t Y = bf2_cvt(y0, y1);
        o[i] = bf2_add(bf2_mul(Y, cw[i]), bf2_mul(bf2_swap(Y), sw[i]));
      }
      st.put(j, o[0], o[1], o[2], o[3]);
    }
    st.flush(tmQKV, ncol + cc);
  }
}

// d = 64 specialisation: the head's 64 accumulator columns are read from TMEM once, kept as 32 packed bf16x2
// registers (that IS the reference's bf16 q/k), and both the sum of squares and the normalise+rotate pass run
// from those registers -- one TMEM round trip instead of two on the epilogue's critical path.
__device__ __forceinline__ void epi_qk_head64(const EpiParams& p, uint32_t taddr, const uint4* rope_row, int ncol,
                                              const float* w_s, OutStage& st, const CUtensorMap* tmQKV, uint64_t rs2) {
  uint32_t P[32];
  uint64_t ss2 = 0ull;
  {
    uint32_t r0[32], r1[32];
    tmem_ld32(taddr, r0);
    tmem_ld32(taddr + 32, r1);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      P[i] = cvt_acc2(r0[2 * i], r0[2 * i + 1], rs2);
      P[16 + i] = cvt_acc2(r1[2 * i], r1[2 * i + 1], rs2);
    }
  }
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const uint64_t t = bf2_to_f2(P[i]);
    ss2 = f2_fma(t, t, ss2);
  }
  float s0, s1;
  f2_unpack(ss2, s0, s1);
  const float rstd = rsqrtf((s0 + s1) * (1.f / 64.f) + p.eps);
  const uint64_t rstd2 = f2_pack(rstd, rstd);
#pragma unroll
  for (int cc = 0; cc < 64; cc += 32) {
    uint4 c2[4], s2[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      c2[j] = ld_global_nc_v4(rope_row + ((cc >> 3) + j) * 32);
      s2[j] = ld_global_nc_v4(rope_row + (8 + (cc >> 3) + j) * 32);
    }
    st.begin();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 wa = *reinterpret_cast<const float4*>(w_s + cc + 8 * j);
      const float4 wb = *reinterpret_cast<const float4*>(w_s + cc + 8 * j + 4);
      const uint64_t w2[4] = {f2_pack(wa.x, wa.y), f2_pack(wa.z, wa.w), f2_pack(wb.x, wb.y), f2_pack(wb.z, wb.w)};
      const uint32_t cw[4] = {c2[j].x, c2[j].y, c2[j].z, c2[j].w};
      const uint32_t sw[4] = {s2[j].x, s2[j].y, s2[j].z, s2[j].w};
      uint32_t o[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float y0, y1;
        f2_unpack(f2_mul(f2_mul(bf2_to_f2(P[(cc >> 1) + 4 * j + i]), rstd2), w2[i]), y0, y1);
        const uint32_t Y = bf2_cvt(y0, y1);
        o[i] = bf2_add(bf2_mul(Y, cw[i]), bf2_mul(bf2_swap(Y), sw[i]));
      }
      st.put(j, o[0], o[1], o[2], o[3]);
    }
    st.flush(tmQKV, ncol + cc);
  }
}

__device__ __forceinline__ void epi_qkv_swiglu_unit(const EpiParams& p, uint32_t taddr, int rrow, int n, int ucols,
                                                    const float* normw_s, OutStage& st, const CUtensorMap* tmQKV,
                                                    const CUtensorMap* tmACT, uint64_t rs2) {
  if (n < p.qp) {
    const int threeD = 3 * p.D;
    // plain bf16 copy of 32 columns (V; q and k too at the head dims whose QK-norm + RoPE run after the GEMM)
    auto copy32 = [&](uint32_t ta, int col) {
      uint32_t r[32];
      tmem_ld32(ta, r);
      tmem_wait_ld();
      st.begin();
#pragma unroll
      for (int j = 0; j < 4; ++j)
        st.put(j, cvt_acc2(r[8 * j], r[8 * j + 1], rs2), cvt_acc2(r[8 * j + 2], r[8 * j + 3], rs2),
               cvt_acc2(r[8 * j + 4], r[8 * j + 5], rs2), cvt_acc2(r[8 * j + 6], r[8 * j + 7], rs2));
      st.flush(tmQKV, col);
    };
    if (!qk_norm_fused(p.d)) {   // a head may straddle two units here: copy the unit, columns past 3D are clipped by the store
      for (int cc = 0; cc < ucols && n + cc < threeD; cc += 32) copy32(taddr + cc, n + cc);
      return;
    }
    const uint4* rope_row = rope_row_ptr(p, rrow);
    for (int hc = 0; hc < ucols; hc += p.d) {
      const int ncol = n + hc;
      if (ncol >= threeD) break;  // zero-padded columns between 3D and qp
      const int seg = ncol / p.D;
      if (seg == 2) {  // V: plain bf16 copy
        for (int cc = 0; cc < p.d; cc += 32) copy32(taddr + hc + cc, ncol + cc);
      } else {
        if (p.d == 64) epi_qk_head64(p, taddr + hc, rope_row, ncol, normw_s + seg * 128, st, tmQKV, rs2);
        else epi_qk_head(p, taddr + hc, rope_row, ncol, normw_s + seg * 128, st, tmQKV, rs2);
      }
    }
  } else {
    // SwiGLU: 32 packed columns = [v(16) | g(16)] -> 16 outputs; mlp.py:21-22 with bf16 rounding of
    // fc1's output, of silu(g) and of the product (bf2_mul).  64 packed columns fill one 32-column output
    // granule; columns at or beyond Hf come from zero weight rows and are clipped by the TMA store.
    const uint64_t nlog2e = f2_pack(-1.4426950408889634f, -1.4426950408889634f);
    const uint64_t one2 = f2_pack(1.f, 1.f);
    for (int cc = 0; cc < ucols; cc += 64) {
      const int j0 = (n + cc - p.qp) >> 5;      // first of the two 32-column groups of this granule
      if (16 * j0 >= p.Hf) break;               // whole granule out of range (warp-uniform)
      uint32_t ra[32], rb[32];
      tmem_ld32(taddr + cc, ra);
      tmem_ld32(taddr + cc + 32, rb);
      tmem_wait_ld();
      st.begin();
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const uint32_t (&r)[32] = half ? rb : ra;
        uint32_t o[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const uint32_t Vp = cvt_acc2(r[2 * i], r[2 * i + 1], rs2);
          const uint64_t g2 = bf2_to_f2(cvt_acc2(r[16 + 2 * i], r[16 + 2 * i + 1], rs2));
          float e0, e1, g0, g1;
          f2_unpack(f2_mul(g2, nlog2e), e0, e1);
          asm("ex2.approx.ftz.f32 %0, %0;" : "+f"(e0));
          asm("ex2.approx.ftz.f32 %0, %0;" : "+f"(e1));
          f2_unpack(f2_add(f2_pack(e0, e1), one2), e0, e1);   // 1 + exp(-g)  (>= 1, or +inf -> rcp = 0)
          asm("rcp.approx.ftz.f32 %0, %0;" : "+f"(e0));
          asm("rcp.approx.ftz.f32 %0, %0;" : "+f"(e1));
          f2_unpack(f2_mul(g2, f2_pack(e0, e1)), g0, g1);     // silu(g) = g * sigmoid(g)
          o[i] = bf2_mul(bf2_cvt(g0, g1), Vp);
        }
        st.put(2 * half, o[0], o[1], o[2], o[3]);
        st.put(2 * half + 1, o[4], o[5], o[6], o[7]);
      }
      st.flush(tmACT, 16 * j0);
    }
  }
}

// fused norm1: the row's scale rsqrt(mean(x^2) + eps) from the producer's per-unit sums of squares (fixed order)
__device__ __forceinline__ uint64_t row_scale2(const EpiParams& p, int rrow) {
  float rs = 1.f;
  if (p.ss_in) {
    const float4* sp = reinterpret_cast<const float4*>(p.ss_in + (long long)rrow * p.ss_units);
    float ss = 0.f;
    for (int u = 0; u < (p.ss_units >> 2); ++u) {
      const float4 v = __ldg(sp + u);
      ss += (v.x + v.y) + (v.z + v.w);
    }
    rs = rsqrtf(ss * p.ss_inv_d + p.eps);
  }
  if (p.a_scale) rs *= __ldg(p.a_scale + rrow) * p.w_scale;   // FP8 operands: dynamic per-row activation scale x weight scale
  return f2_pack(rs, rs);
}

// ------------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------------
template <int BN, int EPI, int NEPI>
__global__ void __launch_bounds__(128 + 32 * NEPI, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmO0, const __grid_constant__ CUtensorMap tmO1, const int M_cap, const int N,
            const int K, const TileSched sched_host, const EpiParams epi) {
  using S = GemmShape<BN>;
  int M = M_cap;
  TileSched sched = sched_host;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + S::STAGES * A_STAGE_BYTES;
  constexpr bool kStaged = (EPI == EPI_QKV_SWIGLU || EPI == EPI_RESID);
  uint8_t* sOut = smem + S::STAGES * S::STAGE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sOut + (kStaged ? NEPI * 2 * OUT_GRANULE_BYTES : 0));
  uint64_t* full = bars;
  uint64_t* empty = bars + S::STAGES;
  uint64_t* tfull = bars + 2 * S::STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  float* normw_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 256);   // [2][128] fp32: norm_q | norm_k

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_k = (K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < S::STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], NEPI);
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, S::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // PDL: everything above overlapped the previous kernel's tail; nothing below may run before it has completed
  pdl_trigger();
  pdl_wait();
  if (epi.m_dev) {   // packed NaFlex batches: the row count lives in device memory (M_cap = capacity the tensor maps were encoded for)
    M = min(__ldg(epi.m_dev), M_cap);
    sched.setup(M, (int)gridDim.x);
  }
  if (EPI == EPI_QKV_SWIGLU && warp >= 4) {
    for (int i = threadIdx.x - 128; i < 2 * epi.d; i += 32 * NEPI) {
      const int kind = i >= epi.d;
      normw_s[kind * 128 + (i - kind * epi.d)] = __bfloat162float((kind ? epi.normk : epi.normq)[i - kind * epi.d]);
    }
    named_bar_sync(1, 32 * NEPI);   // epilogue warps only
  }

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer =====
      int s = 0;
      uint32_t ph = 0;
      for (int t = blockIdx.x; t < sched.total_tiles; t += gridDim.x) {
        int m0, n0, width;
        sched.decode(t, m0, n0, width);
        const uint32_t tx = A_STAGE_BYTES + (uint32_t)width * BK * 2;
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(&empty[s], ph ^ 1);
          mbar_expect_tx(&full[s], tx);
          tma_load_2d(sA + s * A_STAGE_BYTES, &tmA, &full[s], kb * BK, m0);
          // B is fetched as 128-row boxes so that full and half-width tiles share one tensor map
          for (int nb = 0; nb < width; nb += 128)
            tma_load_2d(sB + s * S::B_STAGE_BYTES + nb * (BK * 2), &tmB, &full[s], kb * BK, n0 + nb);
          if (++s == S::STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===== MMA issuer =====
      int s = 0;
      uint32_t ph = 0;
      int acc = 0;
      uint32_t acc_ph = 0;
      for (int t = blockIdx.x; t < sched.total_tiles; t += gridDim.x) {
        int m0, n0, width;
        sched.decode(t, m0, n0, width);
        const uint32_t idesc = make_idesc_bf16(BM, width, 0, 0);
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        mbar_wait(&tempty[acc], acc_ph ^ 1);
        tc_fence_after();
        for (int kb = 0; kb < num_k; ++kb) {
          mbar_wait(&full[s], ph);
          tc_fence_after();
          const uint32_t a0 = smem_u32(sA + s * A_STAGE_BYTES);
          const uint32_t b0 = smem_u32(sB + s * S::B_STAGE_BYTES);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            umma_bf16_ss(d_tmem, make_desc_kmajor_sw128(a0 + k * 32), make_desc_kmajor_sw128(b0 + k * 32), idesc,
                         (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit(&empty[s]);  // smem slot reusable once these MMAs have read it
          if (++s == S::STAGES) { s = 0; ph ^= 1; }
        }
        umma_commit(&tfull[acc]);  // accumulator complete -> epilogue
        if (++acc == 2) { acc = 0; acc_ph ^= 1; }
      }
    }
  } else if (warp >= 4) {
    // ===== epilogue =====
    const int ew = warp - 4;
    const int quarter = warp & 3;           // TMEM lane quarter this warp may access
    const int half = ew >> 2;               // column group: 0 .. NEPI/4-1
    constexpr int NHALF = NEPI / 4;
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    OutStage st;
    st.base = sOut + ew * 2 * OUT_GRANULE_BYTES;
    st.lane = lane;
    st.row0 = 0;
    st.cur = 0;
    int acc = 0;
    uint32_t acc_ph = 0;
    for (int t = blockIdx.x; t < sched.total_tiles; t += gridDim.x) {
      int m0, n0, width;
      sched.decode(t, m0, n0, width);
      const int row = m0 + quarter * 32 + lane;
      const bool row_ok = row < M;
      st.row0 = m0 + quarter * 32;
      const int rrow = row_ok ? row : (M - 1);
      uint64_t rs2 = 0ull;
      if (EPI == EPI_QKV_SWIGLU) rs2 = row_scale2(epi, rrow);
      mbar_wait(&tfull[acc], acc_ph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + lane_base + (uint32_t)(acc * BN);
      if (EPI == EPI_BIAS_LN) {
        epi_bias_ln_row(epi, taddr, row, row_ok, N);
      } else {
        const int U = (EPI == EPI_QKV_SWIGLU && epi.d == 128) ? 128 : 64;   // a fused-norm unit holds whole heads
        for (int c0 = half * U; c0 < width; c0 += NHALF * U) {
          if (EPI == EPI_BIAS) epi_bias_unit(epi, taddr + c0, row, row_ok, n0 + c0, N, U);
          if (EPI == EPI_RESID) epi_resid_unit(epi, taddr + c0, row, row < M, n0 + c0, N, U, st, &tmO0, f2_pack(1.f, 1.f));
          if (EPI == EPI_QKV_SWIGLU) epi_qkv_swiglu_unit(epi, taddr + c0, rrow, n0 + c0, U, normw_s, st, &tmO0, &tmO1, rs2);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[acc]);
      if (++acc == 2) { acc = 0; acc_ph ^= 1; }
    }
    if (kStaged && lane == 0) tma_store_wait_read();   // smem must outlive the last bulk store's reads
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, S::TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
template <int BN, int EPI, int NEPI>
static int launch_gemm_t(const GemmArgs& a, bool allow_split, cudaStream_t stream) {
  using S = GemmShape<BN>;
  CUtensorMap tmA, tmB;
  if (encode_tmap_bf16_sw128(&tmA, a.A, (uint64_t)a.K, (uint64_t)a.M, (uint64_t)a.lda, BM)) return -1;
  if (encode_tmap_bf16_sw128(&tmB, a.B, (uint64_t)a.K, (uint64_t)a.b_rows, (uint64_t)a.ldb, BN < 128 ? BN : 128))
    return -1;
  TileSched sc;
  sc.bn = BN;
  sc.bm = BM;
  sc.num_n = (a.N + BN - 1) / BN;
  // band height: keep the A panel of a band (gm x 128 x K bf16) around 32 MB so it stays in the 126 MB L2
  // together with the weight tiles that are in flight
  {
    const long long panel = (long long)BM * a.K * 2;
    long long gm = (32ll << 20) / (panel > 0 ? panel : 1);
    sc.gm_cap = (int)(gm < 1 ? 1 : gm > (1 << 20) ? (1 << 20) : gm);
  }
  sc.split = (allow_split && BN >= 256) ? 1 : 0;
  const int sms = usable_sms();
  sc.setup(a.M, sms);   // a.M is the row capacity when a.m_dev is given (the kernel redoes this with the device value)
  const int grid = sc.workers;
  // output tensor maps for the TMA-store epilogues (box = 32 cols x 32 rows, SWIZZLE_64B)
  CUtensorMap tmO0 = tmA, tmO1 = tmA;
  constexpr bool kStaged = (EPI == EPI_QKV_SWIGLU || EPI == EPI_RESID);
  if (EPI == EPI_QKV_SWIGLU) {
    if (encode_tmap_bf16(&tmO0, a.epi.qkv, (uint64_t)3 * a.epi.D, (uint64_t)a.M, (uint64_t)a.epi.ld_qkv, 32, 32, 64)) return -1;
    if (encode_tmap_bf16(&tmO1, a.epi.act, (uint64_t)a.epi.Hf, (uint64_t)a.M, (uint64_t)a.epi.ld_act, 32, 32, 64)) return -1;
  } else if (EPI == EPI_RESID) {
    if (encode_tmap_bf16(&tmO0, a.epi.out, (uint64_t)a.N, (uint64_t)a.M, (uint64_t)a.epi.ldo, 32, 32, 64)) return -1;
  }
  const int smem_bytes = S::smem_bytes(kStaged ? NEPI : 0);
  auto kern = gemm_kernel<BN, EPI, NEPI>;
  if (ensure_max_smem(reinterpret_cast<const void*>(kern), smem_bytes, "cudaFuncSetAttribute(gemm)")) return -1;
  return check_cuda(launch_k(kern, dim3(grid), dim3(128 + 32 * NEPI), smem_bytes, stream, tmA, tmB, tmO0, tmO1, a.M, a.N, a.K, sc, a.epi),
                    "gemm launch");
}

// ------------------------------------------------------------------------------------------------
// CTA-pair kernel (cluster of 2, tcgen05 cta_group::2): one 256 x 256 output tile per pair.
//
// Each CTA owns 128 rows of the tile: it TMA-loads its own A rows and HALF of the B tile (the tensor core of
// both SMs reads the two B halves from both shared memories), so per k-block a CTA stages 16 KB + 16 KB
// instead of 16 KB + 32 KB: 2/3 of the L2->SM traffic, 2/3 of the shared-memory writes and reads, room for a
// 6-stage ring.  The leader CTA (cluster rank 0) issues every MMA (M = 256); tcgen05.commit multicasts the
// "slot free" and "accumulator ready" arrivals to both CTAs; all TMA loads of a stage complete on the
// leader's full barrier; the epilogue warps of both CTAs release an accumulator on the leader's barrier.
// The epilogue code is shared with the single-CTA kernel (each CTA finishes its own 128 x 256 half).
// ------------------------------------------------------------------------------------------------
static constexpr int G2_BN = 256;
static constexpr int G2_B_STAGE_BYTES = (G2_BN / 2) * BK * 2;                 // 16 KB: this CTA's half of B
static constexpr int G2_STAGE_BYTES = A_STAGE_BYTES + G2_B_STAGE_BYTES;       // 32 KB
static constexpr int g2_smem_bytes(int stages, int out_warps) {
  return stages * G2_STAGE_BYTES + out_warps * 2 * OUT_GRANULE_BYTES + 256 + 1024 + 1024;
}

template <bool P> __device__ __forceinline__ long long prof_clock() {
  if constexpr (P) return clock64();
  return 0;
}

// TRANS = true: both operands are given TRANSPOSED in memory ("TN" product, the weight gradient dW = dY^T X of the training
// step): A is [K, M] row-major and B is [K, N] row-major, so their tiles are staged as [64 k-rows x 64 columns] swizzled
// blocks and read by the tensor core MN-major (idesc a_major = b_major = 1, LBO = block stride 8 KB) -- no transpose pass.
// TRANS = 2: only B is given transposed ([K, N] row-major) -- the data gradient dX = dY W with W used as stored.
// CL = 4: a cluster of TWO CTA pairs working on vertically adjacent 256-row tiles of the same N-tile.  The B (weight) tile is
// the same for both pairs, so every CTA loads only half of its B share and TMA-multicasts it to its counterpart in the other pair
// (rank r <-> r ^ 2): 48 KB instead of 64 KB leave L2 per pair and k-block, which is what bounds the main loop (DESIGN 3.1).
// A stage slot is then written by two producers, so its "empty" barrier collects the MMA commits of both pairs.
// SK = true (CL = 4, EPI_RESID): SPLIT-K over the two pairs of the cluster -- both pairs compute the SAME 256 x 256 tile, pair p over
// k-blocks [p * ceil(num_k / 2), ...).  For the small per-GPU batches of a strong-scaled job (M = 2048 rows: 32 tiles for 74 pairs) the
// main loop is bound by what ONE SM can pull from L2 (~40 B/clk), so the only way to go faster is to put more SMs on the same bytes:
// 32 tiles x 2 K-halves keep 128 SMs busy (23.9 -> ~14 us per launch).  Pair 1 then ships its fp32 accumulator through distributed
// shared memory into the (now idle) stage ring of pair 0, whose epilogue adds it to its own accumulator and finishes the tile.
// ONE tile per cluster (the host launches exactly as many clusters as tiles): the ring is not reused after the reduction.
template <int EPI, int NEPI, int G2_STAGES, bool PROF, bool FP8 = false, int TRANS = 0, int CL = 2, bool SK = false>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(128 + 32 * NEPI, 1)
gemm2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
             const __grid_constant__ CUtensorMap tmO0, const __grid_constant__ CUtensorMap tmO1, const int M_cap, const int N,
             const int K, const TileSched sched_host, const EpiParams epi) {
  int M = M_cap;
  TileSched sched = sched_host;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + G2_STAGES * A_STAGE_BYTES;
  constexpr bool kStaged = (EPI == EPI_QKV_SWIGLU || EPI == EPI_RESID);
  uint8_t* sOut = smem + G2_STAGES * G2_STAGE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sOut + (kStaged ? NEPI * 2 * OUT_GRANULE_BYTES : 0));
  uint64_t* full = bars;                    // [STAGES]  used in the leader only (count 1: its arrive.expect_tx)
  uint64_t* empty = bars + G2_STAGES;       // [STAGES]  both CTAs (multicast commit)
  uint64_t* tfull = bars + 2 * G2_STAGES;   // [2]       both CTAs (multicast commit)
  uint64_t* tempty = tfull + 2;             // [2]       leader only: 2 * NEPI arrivals (epilogue warps of both CTAs)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  uint64_t* peer_done = tempty + 4;         // SK, pair 1: pair 0's MMAs have completed (its stage ring may be overwritten)
  uint64_t* part_full = tempty + 5;         // SK, pair 0: pair 1's accumulator has arrived in this CTA's ring (128 KB of bulk copies)
  float* normw_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 256);
  static_assert(!SK || (CL == 4 && EPI == EPI_RESID && TRANS == 0), "split-K: 4-CTA cluster, residual epilogue, K-major operands");
  static_assert(!SK || G2_STAGES * G2_STAGE_BYTES >= BM * G2_BN * 4, "split-K: the stage ring must hold a 128 x 256 fp32 accumulator");

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();   // rank in the cluster
  const uint32_t rank = crank & 1u;           // rank inside the CTA pair
  const uint32_t pair = crank >> 1;           // 0, or 0 / 1 with CL = 4
  const uint32_t lead = crank & ~1u;          // cluster rank of this pair's leader CTA
  const uint32_t rrank = SK ? rank : crank;   // which 128-row slice of the cluster's tile this CTA owns
  const int cluster_id = blockIdx.x / CL;
  const int num_clusters = gridDim.x / CL;
  constexpr int BKE = FP8 ? 2 * BK : BK;   // elements per k-block: one 128-byte swizzle row of bf16 (64) or e4m3 (128)
  const int num_k = (K + BKE - 1) / BKE;
  int kb0 = 0, kb1 = num_k;                // this pair's k-blocks
  if (SK) {
    const int kh = (num_k + 1) >> 1;
    kb0 = (int)pair * kh;
    kb1 = min(num_k, kb0 + kh);
  }

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (EPI == EPI_BIAS && epi.k_split > 0) tma_prefetch_desc(&tmO1);
    for (int s = 0; s < G2_STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], SK ? 1 : CL / 2);   // one MMA commit per pair that writes into this CTA's slot
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], 2 * NEPI);
    }
    if (SK) {
      mbar_init(peer_done, 1);
      mbar_init(part_full, 1);
    }
    fence_barrier_init();
    if (SK && pair == 0) mbar_expect_tx(part_full, BM * G2_BN * 4);   // the partner's 128 x 256 fp32 accumulator, by bulk copies
  }
  if (warp == 2) {
    tmem_alloc_2cta(tmem_slot, 512);
    tmem_relinquish_2cta();
  }
  tc_fence_before();
  cluster_sync_all();   // barriers of both CTAs initialised before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // PDL: the prologue above overlapped the previous kernel's tail; global memory is touched only from here on
  pdl_trigger();
  pdl_wait();
  if (epi.m_dev) {   // packed NaFlex batches: row count from device memory (see gemm_kernel)
    M = min(__ldg(epi.m_dev), M_cap);
    sched.setup(M, (int)(gridDim.x / CL));
  }
  if (EPI == EPI_QKV_SWIGLU && warp >= 4) {
    for (int i = threadIdx.x - 128; i < 2 * epi.d; i += 32 * NEPI) {
      const int kind = i >= epi.d;
      normw_s[kind * 128 + (i - kind * epi.d)] = __bfloat162float((kind ? epi.normk : epi.normq)[i - kind * epi.d]);
    }
    named_bar_sync(1, 32 * NEPI);   // epilogue warps only
  }

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer (both CTAs) =====
      int s = 0;
      uint32_t ph = 0;
      long long w_empty = 0;
      for (int t = cluster_id; t < sched.total_tiles; t += num_clusters) {
        int m0, n0, width;
        sched.decode(t, m0, n0, width);
        const int hw = width >> 1;                                      // B rows staged by this CTA
        const uint32_t tx = 2u * (A_STAGE_BYTES + (uint32_t)hw * BK * 2);   // both CTAs' bytes land on the leader's barrier
        for (int kb = kb0; kb < kb1; ++kb) {
          const long long c0 = prof_clock<PROF>();
          mbar_wait(&empty[s], ph ^ 1);
          w_empty += prof_clock<PROF>() - c0;
          const uint32_t fb = mapa_u32(smem_u32(&full[s]), lead);
          if (rank == 0) mbar_expect_tx(&full[s], tx);
          if (TRANS & 1) {   // boxes of [64 k-rows x 64 columns]: coordinates (column, k)
            for (int mb = 0; mb < BM; mb += 64)
              tma_load_2d_2cta(sA + s * A_STAGE_BYTES + mb * (BK * 2), &tmA, fb, m0 + (int)rrank * BM + mb, kb * BK);
          } else {
            tma_load_2d_2cta(sA + s * A_STAGE_BYTES, &tmA, fb, kb * BKE, m0 + (int)rrank * BM);
          }
          // second weight matrix for the k-blocks at / beyond k_split (EPI_BIAS only: its output tensor maps are unused, tmO1 carries B2)
          const bool second_b = EPI == EPI_BIAS && !TRANS && epi.k_split > 0 && kb * BKE >= epi.k_split;
          const CUtensorMap* tb = second_b ? &tmO1 : &tmB;
          const int kc = second_b ? kb * BKE - epi.k_split : kb * BKE;
          if (CL == 4 && !SK) {   // this CTA fetches half of its B share and multicasts it to its counterpart in the other pair
            const int nb = (int)pair * (hw >> 1);
            if (TRANS & 2) tma_load_2d_2cta_mc(sB + s * G2_B_STAGE_BYTES + nb * (BK * 2), &tmB, fb, n0 + (int)rank * hw + nb, kb * BK,
                                               (uint16_t)((1u << rank) | (1u << (rank + 2))));   // one [64 k-rows x 64 columns] box
            else tma_load_2d_2cta_mc(sB + s * G2_B_STAGE_BYTES + nb * (BK * 2), tb, fb, kc, n0 + (int)rank * hw + nb,
                                     (uint16_t)((1u << rank) | (1u << (rank + 2))));
          } else {
            for (int nb = 0; nb < hw; nb += 64) {
              if (TRANS & 2) tma_load_2d_2cta(sB + s * G2_B_STAGE_BYTES + nb * (BK * 2), &tmB, fb, n0 + (int)rank * hw + nb, kb * BK);
              else tma_load_2d_2cta(sB + s * G2_B_STAGE_BYTES + nb * (BK * 2), tb, fb, kc, n0 + (int)rank * hw + nb);
            }
          }
          if (++s == G2_STAGES) { s = 0; ph ^= 1; }
        }
      }
      if (PROF && epi.prof) atomicAdd(&epi.prof[5], (unsigned long long)w_empty);
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      // ===== MMA issuer (leader CTA only) =====
      int s = 0;
      uint32_t ph = 0;
      int acc = 0;
      uint32_t acc_ph = 0;
      long long w_full = 0, w_tempty = 0;
      const long long t_begin = prof_clock<PROF>();
      for (int t = cluster_id; t < sched.total_tiles; t += num_clusters) {
        int m0, n0, width;
        sched.decode(t, m0, n0, width);
        const uint32_t idesc = FP8 ? make_idesc_e4m3(2 * BM, width) : make_idesc_bf16(2 * BM, width, (TRANS & 1) ? 1 : 0, (TRANS & 2) ? 1 : 0);
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * G2_BN);
        long long c0 = prof_clock<PROF>();
        mbar_wait(&tempty[acc], acc_ph ^ 1);
        w_tempty += prof_clock<PROF>() - c0;
        tc_fence_after();
        for (int kb = kb0; kb < kb1; ++kb) {
          c0 = prof_clock<PROF>();
          mbar_wait(&full[s], ph);
          w_full += prof_clock<PROF>() - c0;
          tc_fence_after();
          const uint32_t a0 = smem_u32(sA + s * A_STAGE_BYTES);
          const uint32_t b0 = smem_u32(sB + s * G2_B_STAGE_BYTES);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            if (TRANS) umma_bf16_ss_2cta(d_tmem,   // MN-major: 16 k-rows = 2 KB inside a block, 8 KB between column blocks
                                         (TRANS & 1) ? make_smem_desc(a0 + k * 2048, 8192, 1024, 2) : make_desc_kmajor_sw128(a0 + k * 32),
                                         (TRANS & 2) ? make_smem_desc(b0 + k * 2048, 8192, 1024, 2) : make_desc_kmajor_sw128(b0 + k * 32),
                                         idesc, ((kb - kb0) | k) != 0 ? 1u : 0u);
            else if (FP8) umma_f8_ss_2cta(d_tmem, make_desc_kmajor_sw128(a0 + k * 32), make_desc_kmajor_sw128(b0 + k * 32), idesc,
                                     ((kb - kb0) | k) != 0 ? 1u : 0u);
            else umma_bf16_ss_2cta(d_tmem, make_desc_kmajor_sw128(a0 + k * 32), make_desc_kmajor_sw128(b0 + k * 32), idesc,
                                   ((kb - kb0) | k) != 0 ? 1u : 0u);
          }
          umma_commit_2cta(&empty[s], (CL == 4 && !SK) ? (uint16_t)0xF : (uint16_t)(3u << lead));   // slot reusable: told to every CTA that writes into it
          if (++s == G2_STAGES) { s = 0; ph ^= 1; }
        }
        umma_commit_2cta(&tfull[acc], (uint16_t)(3u << lead));   // accumulator complete -> epilogues of both CTAs of this pair
        if (SK && pair == 0) umma_commit_2cta(peer_done, (uint16_t)0xC);   // ... and pair 1 may overwrite this pair's stage ring
        if (++acc == 2) { acc = 0; acc_ph ^= 1; }
      }
      if (PROF && epi.prof) {
        atomicAdd(&epi.prof[0], (unsigned long long)w_full);
        atomicAdd(&epi.prof[1], (unsigned long long)w_tempty);
        atomicAdd(&epi.prof[2], (unsigned long long)(prof_clock<PROF>() - t_begin));
        atomicAdd(&epi.prof[7], 1ull);
      }
    }
  } else if (warp >= 4) {
    // ===== epilogue (both CTAs, each on its own 128 rows) =====
    const int ew = warp - 4;
    const int quarter = warp & 3;
    const int half = ew >> 2;
    constexpr int NHALF = NEPI / 4;
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    OutStage st;
    st.base = sOut + ew * 2 * OUT_GRANULE_BYTES;
    st.lane = lane;
    st.row0 = 0;
    st.cur = 0;
    int acc = 0;
    uint32_t acc_ph = 0;
    long long w_tfull = 0, w_work = 0;
    const long long t_begin = prof_clock<PROF>();
    for (int t = cluster_id; t < sched.total_tiles; t += num_clusters) {
      int m0, n0, width;
      sched.decode(t, m0, n0, width);
      m0 += (int)rrank * BM;
      const int row = m0 + quarter * 32 + lane;
      const bool row_ok = row < M;
      st.row0 = m0 + quarter * 32;
      const int rrow = row < M ? row : (M - 1);
      uint64_t rs2 = 0ull;
      if (EPI == EPI_QKV_SWIGLU || EPI == EPI_RESID) rs2 = row_scale2(epi, rrow);
      if (EPI == EPI_QKV_SWIGLU && n0 < 2 * epi.D) {
        // q/k tile: pull this warp's 32 RoPE-table rows (one contiguous 32 * 4d-byte block, thanks to the
        // chunk-major layout) into L1 while the accumulator is still being computed
        const uint8_t* blk = reinterpret_cast<const uint8_t*>(epi.rope) + (long long)((m0 + quarter * 32) >> 5) * (128ll * epi.d);
        if (m0 + quarter * 32 < M)
          for (int off = lane * 128; off < 128 * epi.d; off += 32 * 128)
            asm volatile("prefetch.global.L1 [%0];" ::"l"(blk + off));
      }
      if (EPI == EPI_RESID && row < M) {
        // the residual rows of this warp's units: one 128-byte line per lane and unit
        for (int c0 = half * 64; c0 < width; c0 += NHALF * 64)
          if (n0 + c0 < N) asm volatile("prefetch.global.L1 [%0];" ::"l"(epi.out + (long long)row * epi.ldo + n0 + c0));
      }
      const long long c0 = prof_clock<PROF>();
      mbar_wait(&tfull[acc], acc_ph);
      const long long c1 = prof_clock<PROF>();
      w_tfull += c1 - c0;
      tc_fence_after();
      const uint32_t taddr = tmem_base + lane_base + (uint32_t)(acc * G2_BN);
      const uint8_t* partial = nullptr;
      if (SK) {
        if (pair == 1) {
          // Ship this K-half's accumulator to the partner CTA (crank - 2: same rows, other K-half).  Every warp stages its
          // [32 rows x 32 columns] fp32 blocks (4 KB, 128-byte rows, 16-byte chunks XOR-swizzled by row & 7) in THIS CTA's idle
          // stage ring and sends each with one bulk shared->shared::cluster copy that completes on the partner's part_full.
          bool peer_ready = false;
          for (int c0 = half * 64; c0 < width; c0 += NHALF * 64)
            for (int cc = 0; cc < 64; cc += 32) {
              uint32_t r[32];
              tmem_ld32(taddr + c0 + cc, r);
              tmem_wait_ld();
              const uint32_t blk = (uint32_t)(quarter * 8 + ((c0 + cc) >> 5)) * 4096u;
              uint8_t* rowp = sA + blk + (uint32_t)lane * 128u;
#pragma unroll
              for (int j = 0; j < 8; ++j)
                *reinterpret_cast<uint4*>(rowp + ((j ^ (lane & 7)) << 4)) = make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
              fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0) {
                if (!peer_ready) { mbar_wait(peer_done, 0); peer_ready = true; }   // the partner pair's MMAs have read the last of its ring
                bulk_copy_to_cluster(mapa_u32(smem_u32(sA + blk), crank - 2u), sA + blk, 4096u, mapa_u32(smem_u32(part_full), crank - 2u));
              }
            }
          tc_fence_before();
          if (++acc == 2) { acc = 0; acc_ph ^= 1; }
          continue;
        }
        mbar_wait(part_full, 0);   // all 128 KB of the partner's accumulator have landed in this CTA's ring
        partial = sA + (uint32_t)(quarter * 8) * 4096u + (uint32_t)lane * 128u;
      }
      const int U = (EPI == EPI_QKV_SWIGLU && epi.d == 128) ? 128 : 64;   // a fused-norm unit holds whole heads
      for (int c0 = half * U; c0 < width; c0 += NHALF * U) {
        if (EPI == EPI_BIAS) epi_bias_unit(epi, taddr + c0, row, row_ok, n0 + c0, N, U);
        if (EPI == EPI_RESID) epi_resid_unit(epi, taddr + c0, row, row < M, n0 + c0, N, U, st, &tmO0, rs2, partial, c0);
        if (EPI == EPI_QKV_SWIGLU) epi_qkv_swiglu_unit(epi, taddr + c0, rrow, n0 + c0, U, normw_s, st, &tmO0, &tmO1, rs2);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty[acc]), lead));
      w_work += prof_clock<PROF>() - c1;
      if (++acc == 2) { acc = 0; acc_ph ^= 1; }
    }
    if (kStaged && lane == 0) tma_store_wait_read();
    if (PROF && epi.prof && lane == 0 && rank == 0) {   // per epilogue warp of the leader: slots 8.. = wait, 8+NEPI.. = work
      atomicAdd(&epi.prof[8 + ew], (unsigned long long)w_tfull);
      atomicAdd(&epi.prof[8 + NEPI + ew], (unsigned long long)w_work);
      if (ew == 0) atomicAdd(&epi.prof[6], (unsigned long long)(prof_clock<PROF>() - t_begin));
    }
  }

  tc_fence_before();
  cluster_sync_all();   // the peer's shared memory / barriers stay alive until every MMA and arrive has landed
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_2cta(tmem_base, 512);
  }
}

// 4-CTA-cluster launch (gemm2_kernel<..., CL = 4>, residual and plain epilogues): super-tiles of 512 x 256, no half-width tiles; the number of co-resident
// clusters is what the hardware can place (GPCs whose SM count is not a multiple of 4 leave SMs unused)
// split-K launch (gemm2_kernel<..., CL = 4, SK = true>): one 256 x 256 tile per 4-CTA cluster, K halved between its two pairs
template <int NEPI, int G2_STAGES>
static int launch_gemm2_sk(const GemmArgs& a, const CUtensorMap& tmA, const CUtensorMap& tmB, TileSched sc, cudaStream_t stream, bool& taken) {
  taken = false;
  sc.bm = 2 * BM;
  sc.split = 0;
  const int smem_bytes = g2_smem_bytes(G2_STAGES, NEPI);
  auto kern = gemm2_kernel<EPI_RESID, NEPI, G2_STAGES, false, false, 0, 4, true>;
  static int max_clusters_dev[64] = {0};
  int& max_clusters = max_clusters_dev[current_device() & 63];
  if (ensure_max_smem(reinterpret_cast<const void*>(kern), smem_bytes, "cudaFuncSetAttribute(gemm2 split-K)")) return -1;
  if (max_clusters == 0) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(4 * 64); cfg.blockDim = dim3(128 + 32 * NEPI); cfg.dynamicSmemBytes = smem_bytes;
    cudaLaunchAttribute at;
    at.id = cudaLaunchAttributeClusterDimension; at.val.clusterDim.x = 4; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
    cfg.attrs = &at; cfg.numAttrs = 1;
    int n = 0;
    if (check_cuda(cudaOccupancyMaxActiveClusters(&n, kern, &cfg), "cudaOccupancyMaxActiveClusters(gemm2 split-K)")) return -1;
    max_clusters = n > 0 ? n : -1;
  }
  sc.setup(a.M, 1 << 20);
  const int tiles = sc.num_m * sc.num_n;
  if (max_clusters < 0 || tiles > max_clusters) return 0;   // not every tile gets its own co-resident cluster: caller falls back
  CUtensorMap tmO0 = tmA, tmO1 = tmA;
  if (encode_tmap_bf16(&tmO0, a.epi.out, (uint64_t)a.N, (uint64_t)a.M, (uint64_t)a.epi.ldo, 32, 32, 64)) return -1;
  taken = true;
  return check_cuda(launch_k(kern, dim3(4 * tiles), dim3(128 + 32 * NEPI), smem_bytes, stream, tmA, tmB, tmO0, tmO1, a.M, a.N, a.K, sc, a.epi),
                    "gemm2 (split-K) launch");
}

template <int EPI, int NEPI, int G2_STAGES>
static int launch_gemm2_cl4(const GemmArgs& a, const CUtensorMap& tmA, const CUtensorMap& tmB, TileSched sc, cudaStream_t stream) {
  sc.bm = 4 * BM;
  sc.split = 0;
  sc.gm_cap = sc.gm_cap > 1 ? sc.gm_cap / 2 : 1;   // the band height was sized for 256-row tiles: keep the A panel of a band at ~32 MB
  const int smem_bytes = g2_smem_bytes(G2_STAGES, EPI == EPI_RESID ? NEPI : 0);
  auto kern = a.fp8 ? gemm2_kernel<EPI, NEPI, G2_STAGES, false, true, 0, 4> : gemm2_kernel<EPI, NEPI, G2_STAGES, false, false, 0, 4>;
  if constexpr (EPI == EPI_BIAS) {   // transposed-operand variants (the training step's data / weight gradients)
    if (a.trans == 3) kern = gemm2_kernel<EPI, NEPI, G2_STAGES, false, false, 3, 4>;
    else if (a.trans == 2) kern = gemm2_kernel<EPI, NEPI, G2_STAGES, false, false, 2, 4>;
  }
  static int max_clusters_dev[64][4] = {{0, 0, 0, 0}};
  int (&max_clusters)[4] = max_clusters_dev[current_device() & 63];
  const int vi = a.fp8 ? 1 : a.trans == 3 ? 3 : a.trans == 2 ? 2 : 0;
  if (ensure_max_smem(reinterpret_cast<const void*>(kern), smem_bytes, "cudaFuncSetAttribute(gemm2 cl4)")) return -1;
  if (max_clusters[vi] == 0) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(4 * 64); cfg.blockDim = dim3(128 + 32 * NEPI); cfg.dynamicSmemBytes = smem_bytes;
    cudaLaunchAttribute at;
    at.id = cudaLaunchAttributeClusterDimension; at.val.clusterDim.x = 4; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
    cfg.attrs = &at; cfg.numAttrs = 1;
    int n = 0;
    if (check_cuda(cudaOccupancyMaxActiveClusters(&n, kern, &cfg), "cudaOccupancyMaxActiveClusters(gemm2 cl4)")) return -1;
    if (n <= 0) { set_error("gemm2 cl4: no 4-CTA cluster fits on this device"); return -1; }
    max_clusters[vi] = n;
  }
  const int avail = std::min(max_clusters[vi], std::max(1, usable_sms() / 4));   // (reserve_sms: room for a concurrent collective)
  sc.setup(a.M, avail);
  const int big = sc.num_m * sc.num_n;
  const int clusters = big < avail ? big : avail;
  CUtensorMap tmO0 = tmA, tmO1 = tmA;
  if (EPI == EPI_RESID) {
    if (encode_tmap_bf16(&tmO0, a.epi.out, (uint64_t)a.N, (uint64_t)a.M, (uint64_t)a.epi.ldo, 32, 32, 64)) return -1;
  } else if (EPI == EPI_BIAS && a.epi.k_split > 0) {
    if (encode_tmap_bf16_sw128(&tmO1, a.B2, (uint64_t)(a.K - a.epi.k_split), (uint64_t)a.b_rows, (uint64_t)a.ldb2, 64)) return -1;
  }
  return check_cuda(launch_k(kern, dim3(4 * clusters), dim3(128 + 32 * NEPI), smem_bytes, stream, tmA, tmB, tmO0, tmO1, a.M, a.N, a.K, sc,
                             a.epi), "gemm2 (4-CTA cluster) launch");
}

template <int EPI, int NEPI, int G2_STAGES>
static int launch_gemm2_s(const GemmArgs& a, cudaStream_t stream) {
  CUtensorMap tmA, tmB;
  if (a.trans) {   // transposed operand(s) [K, columns] row-major: boxes of 64 columns x 64 k-rows
    if (a.trans & 1) { if (encode_tmap_bf16_sw128(&tmA, a.A, (uint64_t)a.M, (uint64_t)a.K, (uint64_t)a.lda, 64)) return -1; }
    else if (encode_tmap_bf16_sw128(&tmA, a.A, (uint64_t)a.K, (uint64_t)a.M, (uint64_t)a.lda, BM)) return -1;
    if (encode_tmap_bf16_sw128(&tmB, a.B, (uint64_t)a.b_rows, (uint64_t)a.K, (uint64_t)a.ldb, 64)) return -1;
  } else if (a.fp8) {
    if (encode_tmap_u8_sw128(&tmA, a.A, (uint64_t)a.K, (uint64_t)a.M, (uint64_t)a.lda, BM)) return -1;
    if (encode_tmap_u8_sw128(&tmB, a.B, (uint64_t)a.K, (uint64_t)a.b_rows, (uint64_t)a.ldb, 64)) return -1;
  } else {
    if (encode_tmap_bf16_sw128(&tmA, a.A, (uint64_t)a.K, (uint64_t)a.M, (uint64_t)a.lda, BM)) return -1;
    if (encode_tmap_bf16_sw128(&tmB, a.B, (uint64_t)(a.epi.k_split > 0 ? a.epi.k_split : a.K), (uint64_t)a.b_rows, (uint64_t)a.ldb, 64)) return -1;
  }
  TileSched sc;
  sc.bn = G2_BN;
  sc.bm = 2 * BM;
  sc.num_n = (a.N + G2_BN - 1) / G2_BN;
  {
    const long long panel = 2ll * BM * a.K * 2;
    long long gm = (32ll << 20) / (panel > 0 ? panel : 1);
    sc.gm_cap = (int)(gm < 1 ? 1 : gm > (1 << 20) ? (1 << 20) : gm);
  }
  sc.split = 1;
  // Split-K for the residual GEMM of small batches: at most pairs / 2 tiles (half of the SMs would idle) and a long K
  if constexpr (EPI == EPI_RESID) {
    const long long tiles2 = (long long)((a.M + 2 * BM - 1) / (2 * BM)) * sc.num_n;
    if (flag_gemm_splitk() && !a.fp8 && !a.trans && !a.epi.prof && a.M > BM && 2 * tiles2 <= num_sms() / 2 && a.K >= 16 * BK) {
      bool taken = false;
      const int r = launch_gemm2_sk<NEPI, G2_STAGES>(a, tmA, tmB, sc, stream, taken);
      if (r || taken) return r;
    }
  }
  // 4-CTA clusters (two pairs sharing the B tile by TMA multicast): bf16 / fp8 K-major operands, enough M for two 256-row tiles
  // Measured (B200, c2 / c4 in the bench pipeline): out_proj+fc2 residual GEMM 3.19 -> 3.11 ms / 21.5 -> 20.5 ms, but the QKV+fc1 GEMM
  // 6.99 -> 7.18 / 43.9 -> 45.2 ms -- only 33 clusters (132 of 148 SMs) are co-resident, which the epilogue-heavy kernel feels more than
  // it gains from the lighter L2 traffic.  So: the light epilogues only (residual, plain / bias; the 5B training step's forward GEMMs
  // gain 1 %), and the transposed-operand variants (data / weight gradients of the training step) included: alone wgrad 1333-1365 ->
  // 1414-1441 TF/s, dgrad 1395 -> 1439 TF/s, 5B step 302.8 -> 296.3 ms.
  if constexpr (EPI == EPI_RESID || EPI == EPI_BIAS) {
    // ... and only when the 512-row super tiles fill the ~33 co-resident clusters at least once: below that (the small per-GPU
    // batches of a strong-scaled job) the pair kernel with half-width tiles keeps more SMs busy
    const long long tiles4 = (long long)((a.M + 4 * BM - 1) / (4 * BM)) * sc.num_n;
    if (tiles4 >= num_sms() / 4 - 4 && !a.epi.prof && a.M > 2 * BM) return launch_gemm2_cl4<EPI, NEPI, G2_STAGES>(a, tmA, tmB, sc, stream);
  }
  const int pairs = usable_sms() / 2;
  sc.setup(a.M, pairs);
  const int clusters = sc.workers;
  CUtensorMap tmO0 = tmA, tmO1 = tmA;
  constexpr bool kStaged = (EPI == EPI_QKV_SWIGLU || EPI == EPI_RESID);
  if (EPI == EPI_QKV_SWIGLU) {
    if (encode_tmap_bf16(&tmO0, a.epi.qkv, (uint64_t)3 * a.epi.D, (uint64_t)a.M, (uint64_t)a.epi.ld_qkv, 32, 32, 64)) return -1;
    if (encode_tmap_bf16(&tmO1, a.epi.act, (uint64_t)a.epi.Hf, (uint64_t)a.M, (uint64_t)a.epi.ld_act, 32, 32, 64)) return -1;
  } else if (EPI == EPI_RESID) {
    if (encode_tmap_bf16(&tmO0, a.epi.out, (uint64_t)a.N, (uint64_t)a.M, (uint64_t)a.epi.ldo, 32, 32, 64)) return -1;
  } else if (EPI == EPI_BIAS && a.epi.k_split > 0) {
    if (encode_tmap_bf16_sw128(&tmO1, a.B2, (uint64_t)(a.K - a.epi.k_split), (uint64_t)a.b_rows, (uint64_t)a.ldb2, 64)) return -1;
  }
  const int smem_bytes = g2_smem_bytes(G2_STAGES, kStaged ? NEPI : 0);
  auto kern = a.fp8 ? gemm2_kernel<EPI, NEPI, G2_STAGES, false, true>
              : a.epi.prof ? gemm2_kernel<EPI, NEPI, G2_STAGES, true> : gemm2_kernel<EPI, NEPI, G2_STAGES, false>;
  if constexpr (EPI == EPI_BIAS) {   // transposed-operand variants (launch_gemm_inner accepts trans with this epilogue only)
    if (a.trans == 3) kern = a.epi.prof ? gemm2_kernel<EPI, NEPI, G2_STAGES, true, false, 3> : gemm2_kernel<EPI, NEPI, G2_STAGES, false, false, 3>;
    else if (a.trans == 2) kern = a.epi.prof ? gemm2_kernel<EPI, NEPI, G2_STAGES, true, false, 2> : gemm2_kernel<EPI, NEPI, G2_STAGES, false, false, 2>;
  }
  if (ensure_max_smem(reinterpret_cast<const void*>(kern), smem_bytes, "cudaFuncSetAttribute(gemm2)")) return -1;
  return check_cuda(launch_k(kern, dim3(2 * clusters), dim3(128 + 32 * NEPI), smem_bytes, stream, tmA, tmB, tmO0, tmO1, a.M, a.N, a.K, sc,
                             a.epi), "gemm2 launch");
}

int launch_gemm_inner(EpiKind kind, const GemmArgs& a, cudaStream_t stream);

static unsigned long long* g_prof = nullptr;

// VTK_GEMM_PROF=1: every pair-kernel launch is followed by a sync and a per-role cycle report on stderr.
static void prof_report(const char* what, int NEPI) {
  unsigned long long h[64];
  cudaDeviceSynchronize();
  cudaMemcpy(h, g_prof, sizeof(h), cudaMemcpyDeviceToHost);
  const double n = h[7] ? (double)h[7] : 1.0;
  fprintf(stderr, "[gemm prof] %s: per leader CTA: mma total %.0f cyc | mma wait full %.0f | mma wait tempty %.0f | producer wait empty %.0f | epi(w0) total %.0f\n",
          what, h[2] / n, h[0] / n, h[1] / n, h[5] / (2 * n), h[6] / n);
  fprintf(stderr, "[gemm prof]   epilogue warps wait-tfull / work (cycles per leader CTA):");
  for (int i = 0; i < NEPI; ++i) fprintf(stderr, " %.0f/%.0f", h[8 + i] / n, h[8 + NEPI + i] / n);
  fprintf(stderr, "\n");
}

int launch_gemm(EpiKind kind, const GemmArgs& a_in, cudaStream_t stream) {
  GemmArgs a = a_in;
  a.epi.prof = nullptr;
  static int prof_mode = -1;
  if (prof_mode < 0) { const char* e = getenv("VTK_GEMM_PROF"); prof_mode = e ? atoi(e) : 0; }
  if (prof_mode) {
    if (!g_prof) cudaMalloc(&g_prof, 64 * sizeof(unsigned long long));
    cudaMemsetAsync(g_prof, 0, 64 * sizeof(unsigned long long), stream);
    a.epi.prof = g_prof;
    const int r = launch_gemm_inner(kind, a, stream);
    if (r == 0) prof_report(kind == EPI_QKV_SWIGLU ? "qkv_swiglu" : kind == EPI_RESID ? "proj_resid" : "linear", 8);
    return r;
  }
  return launch_gemm_inner(kind, a, stream);
}

int launch_gemm_inner(EpiKind kind, const GemmArgs& a, cudaStream_t stream) {
  if (a.M <= 0 || a.N <= 0 || a.K <= 0) { set_error("gemm: empty problem M=%d N=%d K=%d", a.M, a.N, a.K); return -2; }
  if (!a.trans && ((a.K % 8) || (a.lda % 8) || (a.ldb % 8) || (a.N % 8))) {
    set_error("gemm: K, N and the row strides must be multiples of 8 (K=%d N=%d lda=%lld ldb=%lld)", a.K, a.N, a.lda, a.ldb);
    return -2;
  }
  if ((reinterpret_cast<uintptr_t>(a.A) | reinterpret_cast<uintptr_t>(a.B)) & 15) {
    set_error("gemm: operand pointers must be 16-byte aligned");
    return -2;
  }
  if (a.epi.k_split > 0) {   // two weight matrices, one accumulator: pair kernel only (the caller checks the shape)
    if (kind != EPI_BIAS || a.trans || a.fp8 || !a.B2 || (a.epi.k_split % BK) || a.epi.k_split >= a.K || (a.ldb2 % 8) || a.M <= BM || a.N <= 128 ||
        (reinterpret_cast<uintptr_t>(a.B2) & 15)) {
      set_error("gemm(k_split): needs the bf16 pair kernel (M > 128, N > 128), k_split %% 64 == 0 inside K, a 16-byte aligned second matrix");
      return -3;
    }
    return launch_gemm2_s<EPI_BIAS, 8, 6>(a, stream);
  }
  if (a.trans) {   // transposed operands (weight gradients): CTA-pair kernel, plain epilogue
    if (kind != EPI_BIAS || a.fp8 || (a.trans != 2 && a.trans != 3)) {
      set_error("gemm(trans): only the plain bf16 epilogue has transposed-operand variants (trans = 2: B, 3: A and B)");
      return -3;
    }
    if (((a.trans & 1) && (a.M % 8)) || (!(a.trans & 1) && (a.K % 8)) || (a.lda % 8) || (a.ldb % 8) || (a.N % 8)) {
      set_error("gemm(trans): the contiguous dimensions and the row strides must be multiples of 8");
      return -2;
    }
    return launch_gemm2_s<EPI_BIAS, 8, 6>(a, stream);
  }
  if (a.fp8) {   // e4m3 operands: CTA-pair kernel only (any M: rows beyond M are zero-filled by TMA and never stored)
    if ((a.K % 16) || (a.lda % 16) || (a.ldb % 16)) { set_error("gemm(fp8): K and the row strides must be multiples of 16 bytes"); return -2; }
    if (kind == EPI_QKV_SWIGLU) {
      if (!head_dim_supported(a.epi.d) || a.epi.qp % 256 || a.epi.D % a.epi.d || a.epi.Hf % 16) {
        set_error("gemm(fp8): unsupported attention geometry D=%d d=%d Hf=%d qp=%d", a.epi.D, a.epi.d, a.epi.Hf, a.epi.qp);
        return -3;
      }
      // (16 epilogue warps instead of 8 change nothing here: 4.82 vs 4.89 ms at c2 -- with e4m3 operands the pair tile needs
      // 128 B/clk/SM from L2, three times what the fabric delivers, so the FP8 GEMMs are L2-bandwidth-bound, not epilogue-bound)
      return launch_gemm2_s<EPI_QKV_SWIGLU, 8, 6>(a, stream);
    }
    if (kind == EPI_RESID) return launch_gemm2_s<EPI_RESID, 8, 6>(a, stream);
    if (kind == EPI_BIAS) return launch_gemm2_s<EPI_BIAS, 8, 6>(a, stream);
    set_error("gemm(fp8): epilogue %d has no FP8 variant", (int)kind);
    return -3;
  }
  switch (kind) {
    case EPI_BIAS:
      if (a.N <= 64) return launch_gemm_t<64, EPI_BIAS, 8>(a, false, stream);
      if (a.N <= 128) return launch_gemm_t<128, EPI_BIAS, 8>(a, false, stream);
      if (a.M > BM) return launch_gemm2_s<EPI_BIAS, 8, 6>(a, stream);
      return launch_gemm_t<256, EPI_BIAS, 16>(a, true, stream);
    case EPI_BIAS_LN:
      if (a.N % 8 || a.N > 256 || !a.epi.bias) { set_error("gemm: LN epilogue needs N%%8==0, N<=256 and a bias (N=%d)", a.N); return -2; }
      if (a.N <= 64) return launch_gemm_t<64, EPI_BIAS_LN, 4>(a, false, stream);
      if (a.N <= 128) return launch_gemm_t<128, EPI_BIAS_LN, 4>(a, false, stream);
      return launch_gemm_t<256, EPI_BIAS_LN, 4>(a, false, stream);
    case EPI_QKV_SWIGLU:
      if (!head_dim_supported(a.epi.d) || a.epi.qp % 256 || a.epi.D % a.epi.d || a.epi.Hf % 16) {
        set_error("gemm: unsupported attention geometry D=%d d=%d Hf=%d qp=%d (head_dim: multiples of 8 from 8 to 128)", a.epi.D,
                  a.epi.d, a.epi.Hf, a.epi.qp);
        return -3;
      }
      if (a.M > BM) return launch_gemm2_s<EPI_QKV_SWIGLU, 8, 6>(a, stream);
      return launch_gemm_t<256, EPI_QKV_SWIGLU, 8>(a, true, stream);
    case EPI_RESID:
      if (a.M > BM) return launch_gemm2_s<EPI_RESID, 8, 6>(a, stream);
      return launch_gemm_t<256, EPI_RESID, 8>(a, true, stream);
  }
  set_error("gemm: unknown epilogue %d", (int)kind);
  return -2;
}

// ------------------------------------------------------------------------------------------------
// descriptor probe: one CTA, one 128 x N tile, no pipelining.  Lets a test sweep the shared-memory
// descriptor fields (LBO / SBO / per-UMMA_K start-address step) for the MN-major B operand that the
// attention kernel uses for V, and sanity-check the K-major path in isolation.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128, 1)
umma_probe_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, float* D, int N,
                  int K, int b_mn_major, uint32_t lbo, uint32_t sbo, uint32_t kstep) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  // A: K/64 blocks of [128 x 64] (16 KB each).  B K-major: K/64 blocks of [N x 64]; B MN-major: N/64 blocks of [K x 64].
  uint8_t* sA = smem;
  uint8_t* sB = smem + (K / 64) * 16384;
  __shared__ uint64_t bar_load, bar_mma;
  __shared__ uint32_t tmem_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    mbar_init(&bar_load, 1);
    mbar_init(&bar_mma, 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(&tmem_slot, 256);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  if (threadIdx.x == 0) {
    uint32_t bytes = (uint32_t)(128 * K * 2 + N * K * 2);
    mbar_expect_tx(&bar_load, bytes);
    for (int kb = 0; kb < K / 64; ++kb) tma_load_2d(sA + kb * 16384, &tmA, &bar_load, kb * 64, 0);
    if (!b_mn_major) {
      for (int kb = 0; kb < K / 64; ++kb) tma_load_2d(sB + kb * (N * 128), &tmB, &bar_load, kb * 64, 0);
    } else {
      for (int nb = 0; nb < N / 64; ++nb) tma_load_2d(sB + nb * (K * 128), &tmB, &bar_load, nb * 64, 0);
    }
    mbar_wait(&bar_load, 0);
    tc_fence_after();
    const uint32_t idesc = make_idesc_bf16(128, N, 0, b_mn_major);
    for (int k = 0; k < K / 16; ++k) {
      const uint32_t aaddr = smem_u32(sA) + (k / 4) * 16384 + (k % 4) * 32;
      uint64_t bdesc;
      if (!b_mn_major) {
        bdesc = make_desc_kmajor_sw128(smem_u32(sB) + (k / 4) * (N * 128) + (k % 4) * 32);
      } else {
        bdesc = make_smem_desc(smem_u32(sB) + k * kstep, lbo, sbo, 2);
      }
      umma_bf16_ss(tmem_base, make_desc_kmajor_sw128(aaddr), bdesc, idesc, k != 0);
    }
    umma_commit(&bar_mma);
  }
  mbar_wait(&bar_mma, 0);
  tc_fence_after();
  const int row = warp * 32 + lane;
  for (int c = 0; c < N; c += 32) {
    uint32_t r[32];
    tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + c, r);
    tmem_wait_ld();
    for (int i = 0; i < 32; ++i) D[row * N + c + i] = __uint_as_float(r[i]);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 256);
}

int launch_umma_probe(const bf16* A, const bf16* B, float* D, int N, int K, int b_mn_major, uint32_t lbo_bytes,
                      uint32_t sbo_bytes, uint32_t kstep_bytes, cudaStream_t stream) {
  if (N % 64 || N > 256 || K % 64 || K > 256) { set_error("probe: N, K must be multiples of 64 and <= 256"); return -2; }
  CUtensorMap tmA, tmB;
  if (encode_tmap_bf16_sw128(&tmA, A, K, 128, K, 128)) return -1;
  if (!b_mn_major) {
    if (encode_tmap_bf16_sw128(&tmB, B, K, N, K, N)) return -1;   // B [N, K]
  } else {
    if (encode_tmap_bf16_sw128(&tmB, B, N, K, N, K)) return -1;   // B [K, N]: box = 64 (n) x K rows
  }
  const int smem = 128 * K * 2 + N * K * 2 + 1024;
  if (check_cuda(cudaFuncSetAttribute(umma_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem), "probe attr"))
    return -1;
  umma_probe_kernel<<<1, 128, smem, stream>>>(tmA, tmB, D, N, K, b_mn_major, lbo_bytes, sbo_bytes, kstep_bytes);
  return check_cuda(cudaGetLastError(), "probe launch");
}

}  // namespace vtk
