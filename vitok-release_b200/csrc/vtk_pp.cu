// vtk_pp.cu -- NaFlex patchify / unpatchify / index packing as coalesced, vectorised gather kernels.
//
//   patchify     vitok/pp/ops.py:217-285 + patch_collate_fn (vitok/data.py:77-94): writes straight into the
//                batched [B, T, 3p^2] buffers (no per-image dicts, no torch.stack), builds patch_mask /
//                row_idx / col_idx / time_idx / orig_height / orig_width / grid_rows / grid_cols.
//                Optional fused front end: uint8 HWC -> to_tensor | normalize(minus_one_to_one)
//                (ops.py:140-155) and bf16 output.
//   resize_patchify  vitok/pp/ops.py:169-214 + :217-285: over-budget images resized (antialiased bicubic, ATen's
//                _upsample_bicubic2d_aa) to the token budget and patchified in one launch sequence.
//   unpatchify   vitok/pp/ops.py:295-335: scatter + fold restated as a gather through a cell->token map,
//                with _convert_format (vitok/pp/io.py:91-121) optionally fused.
// All integer/byte work is bit-exact against the reference.
#include "vtk_common.cuh"
#include "vtk_kernels.h"

namespace vtk {

// ToTensor (u / 255, fp32 division) then Normalize(0.5, 0.5) ((t - 0.5) / 0.5 == (t - 0.5) * 2 exactly), ops.py:140-161
__device__ __forceinline__ float norm_u8(uint32_t u) {
  return __fmul_rn(__fsub_rn(__fdiv_rn((float)u, 255.0f), 0.5f), 2.0f);
}
// The same value without the division sequence and without a table: q0 = u * RN(1/255), one FMA residual + one FMA correction is the
// textbook correctly-rounded quotient, and for the 256 possible inputs it is bit-identical to __fdiv_rn (checked exhaustively against
// norm_u8 by patchify_selftest_kernel / tests/test_gpu_pp.py).  3 FMA-pipe instructions instead of a shared-memory lookup whose
// random bank conflicts bounded the uint8 front end at half of HBM bandwidth.
__device__ __forceinline__ float norm_u8_fast(uint32_t u) {
  // float(u) for u < 2^23 without the conversion pipe: 2^23 + u is exact in fp32, subtract 2^23 again
  const float uf = __fsub_rn(__uint_as_float(0x4B000000u | u), 8388608.0f), rcp = 0.0039215688593685627f;   // RN(1 / 255)
  const float q0 = __fmul_rn(uf, rcp);
  const float rem = __fmaf_rn(-q0, 255.0f, uf);
  const float q = __fmaf_rn(rem, rcp, q0);
  return __fmul_rn(__fsub_rn(q, 0.5f), 2.0f);
}
__global__ void patchify_selftest_kernel(int* mismatches) {
  const uint32_t u = threadIdx.x;
  if (__float_as_uint(norm_u8(u)) != __float_as_uint(norm_u8_fast(u))) atomicAdd(mismatches, 1);
}

template <typename OutT>
__device__ __forceinline__ void store4(OutT* dst, float4 v) {
  if (sizeof(OutT) == 4) *reinterpret_cast<float4*>(dst) = v;
  else *reinterpret_cast<uint2*>(dst) = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
}

// One warp per token: the token's 3p^2 output elements are written as contiguous 16-byte (fp32) / 8-byte (bf16) chunks,
// lane after lane (fully coalesced), and gathered from the image as 16-pixel row segments.  All per-token index work
// (image table, grid, row / col) is done once per token; PT = compile-time patch size (16 / 32; 0 = any multiple of 4)
// turns the per-chunk divisions into shifts -- the first version of this kernel spent its time in 64-bit div / mod
// (issue-bound at 1.9 TB/s).  uint8 HWC input: a lane reads the 12 contiguous bytes of 4 pixels (3 x 32-bit loads) and
// writes one chunk per channel; the 256-entry normalisation table lives in shared memory (bit-exact by construction).
template <typename OutT, int PT>
__global__ void __launch_bounds__(256) patchify_kernel(const PatchifyArgs a) {
  pdl_wait();      // PDL (vtk_common.cuh): this kernel may have been launched before its predecessor finished
  pdl_trigger();
  __shared__ float lut[256];
  if (a.in_dtype == 1) {
    lut[threadIdx.x] = norm_u8(threadIdx.x);
    __syncthreads();
  }
  const int p = PT ? PT : a.patch, T = a.max_tokens;
  const int pp = p * p, P = 3 * pp, p4 = p >> 2, chunks = pp >> 2;   // chunks = 4-pixel groups per channel
  const int lane = threadIdx.x & 31;
  const unsigned ntok = (unsigned)a.B * (unsigned)T;
  const unsigned nwarp = gridDim.x * (blockDim.x >> 5);
  for (unsigned bt = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); bt < ntok; bt += nwarp) {
    const int b = (int)(bt / (unsigned)T), t = (int)(bt - (unsigned)b * (unsigned)T);
    const long long off = a.img_table[3 * b + 0];
    const int H = (int)a.img_table[3 * b + 1], W = (int)a.img_table[3 * b + 2];
    const int gr = (H + p - 1) / p, gc = (W + p - 1) / p;
    const int n = gr * gc;
    const bool valid = t < n && n <= T;
    const int r = valid ? t / gc : 0, c = valid ? t - (t / gc) * gc : 0;
    OutT* dst = reinterpret_cast<OutT*>(a.patches) + (long long)bt * P;
    if (!valid) {
      for (int e4 = lane; e4 < 3 * chunks; e4 += 32) store4(dst + (e4 << 2), make_float4(0.f, 0.f, 0.f, 0.f));
    } else if (a.in_dtype == 0) {
      const float* img = reinterpret_cast<const float*>(a.images) + off;
      const bool al = ((reinterpret_cast<uintptr_t>(img) | ((uintptr_t)W << 2)) & 15) == 0;   // rows start 16-byte aligned
      if (PT && al && (r + 1) * p <= H && (c + 1) * p <= W) {
        // interior token of an aligned image (every token of the fixed-size configs): no bounds tests, and all of a lane's
        // 16-byte loads are issued before the first store -- this kernel is latency-bound otherwise (two loads in flight per
        // lane reached 3.3 TB/s), six to eight independent loads per lane keep enough bytes in flight for HBM
        constexpr int NIT = PT ? (3 * PT * PT / 4) / 32 : 1;    // 6 (p = 16) / 24 (p = 32) chunks per lane
        constexpr int UN = NIT % 8 == 0 ? 8 : 6;
        const float* base = img + (long long)(r * p) * W + c * p;
        const long long plane = (long long)H * W;
#pragma unroll 1
        for (int it0 = 0; it0 < NIT; it0 += UN) {
          float4 v[UN];
#pragma unroll
          for (int u = 0; u < UN; ++u) {
            const int e4 = lane + 32 * (it0 + u);
            const int ch = e4 / chunks, rem = e4 - ch * chunks;
            const int dy = rem / p4, dx = (rem - dy * p4) << 2;
            v[u] = __ldg(reinterpret_cast<const float4*>(base + ch * plane + (long long)dy * W + dx));
          }
#pragma unroll
          for (int u = 0; u < UN; ++u) store4(dst + ((lane + 32 * (it0 + u)) << 2), v[u]);
        }
      } else
#pragma unroll 2
      for (int e4 = lane; e4 < 3 * chunks; e4 += 32) {
        const int ch = e4 / chunks, rem = e4 - ch * chunks;
        const int dy = rem / p4, dx = (rem - dy * p4) << 2;
        const int y = r * p + dy, x = c * p + dx;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);      // zero padding to the patch boundary (ops.py:235-238)
        if (y < H) {
          const float* src = img + ((long long)ch * H + y) * W + x;
          if (al && x + 3 < W) {
            v = __ldg(reinterpret_cast<const float4*>(src));
          } else {
            if (x < W) v.x = __ldg(src);
            if (x + 1 < W) v.y = __ldg(src + 1);
            if (x + 2 < W) v.z = __ldg(src + 2);
            if (x + 3 < W) v.w = __ldg(src + 3);
          }
        }
        store4(dst + (e4 << 2), v);
      }
    } else {
      const uint8_t* img = reinterpret_cast<const uint8_t*>(a.images) + off;
      const bool al = (reinterpret_cast<uintptr_t>(img) & 3) == 0;
      if (PT && al && (W & 3) == 0 && (r + 1) * p <= H && (c + 1) * p <= W) {
        // interior token, 4-byte aligned rows: a lane's 12-byte pixel groups are loaded up front (see the fp32 path)
        constexpr int NQ = PT ? (PT * PT / 4) / 32 : 1;         // 2 (p = 16) / 8 (p = 32) 4-pixel groups per lane
        const uint8_t* base = img + ((long long)(r * p) * W + c * p) * 3;
#pragma unroll 1
        for (int q0 = 0; q0 < NQ; q0 += 4) {
          uint32_t w[4][3];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            if (q0 + u < NQ) {
              const int q = lane + 32 * (q0 + u);
              const int dy = q / p4, dx = (q - dy * p4) << 2;
              const uint32_t* s32 = reinterpret_cast<const uint32_t*>(base + ((long long)dy * W + dx) * 3);
              w[u][0] = __ldg(s32); w[u][1] = __ldg(s32 + 1); w[u][2] = __ldg(s32 + 2);
            }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            if (q0 + u < NQ) {
              const int q = lane + 32 * (q0 + u);
              const uint32_t w0 = w[u][0], w1 = w[u][1], w2 = w[u][2];
              store4(dst + (q << 2), make_float4(lut[w0 & 255], lut[w0 >> 24], lut[(w1 >> 16) & 255], lut[(w2 >> 8) & 255]));
              store4(dst + pp + (q << 2), make_float4(lut[(w0 >> 8) & 255], lut[w1 & 255], lut[w1 >> 24], lut[(w2 >> 16) & 255]));
              store4(dst + 2 * pp + (q << 2), make_float4(lut[(w0 >> 16) & 255], lut[(w1 >> 8) & 255], lut[w2 & 255], lut[w2 >> 24]));
            }
          }
        }
      } else
      for (int q = lane; q < chunks; q += 32) {
        const int dy = q / p4, dx = (q - dy * p4) << 2;
        const int y = r * p + dy, x = c * p + dx;
        float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0, v2 = v0;
        if (y < H && x < W) {
          const uint8_t* src = img + ((long long)y * W + x) * 3;    // 12 contiguous bytes: r g b r g b r g b r g b
          uint32_t w0 = 0, w1 = 0, w2 = 0;
          if (al && x + 3 < W && (((long long)y * W + x) & 3) == 0) {
            const uint32_t* s32 = reinterpret_cast<const uint32_t*>(src);
            w0 = __ldg(s32); w1 = __ldg(s32 + 1); w2 = __ldg(s32 + 2);
          } else {
            const int nb = min(4, W - x) * 3;
            for (int k = 0; k < nb; ++k) {
              const uint32_t u = src[k];
              if (k < 4) w0 |= u << (8 * k); else if (k < 8) w1 |= u << (8 * (k - 4)); else w2 |= u << (8 * (k - 8));
            }
          }
          const int np = min(4, W - x);   // pixels inside the image; the rest stay 0.0 (padding is applied AFTER normalize)
          v0.x = lut[w0 & 255]; v1.x = lut[(w0 >> 8) & 255]; v2.x = lut[(w0 >> 16) & 255];
          if (np > 1) { v0.y = lut[w0 >> 24]; v1.y = lut[w1 & 255]; v2.y = lut[(w1 >> 8) & 255]; }
          if (np > 2) { v0.z = lut[(w1 >> 16) & 255]; v1.z = lut[w1 >> 24]; v2.z = lut[w2 & 255]; }
          if (np > 3) { v0.w = lut[(w2 >> 8) & 255]; v1.w = lut[(w2 >> 16) & 255]; v2.w = lut[w2 >> 24]; }
        }
        store4(dst + (q << 2), v0);
        store4(dst + pp + (q << 2), v1);
        store4(dst + 2 * pp + (q << 2), v2);
      }
    }
    if (lane == 0) {  // index packing, one lane per token
      a.patch_mask[bt] = valid ? 1 : 0;
      a.row_idx[bt] = r;
      a.col_idx[bt] = c;
      a.time_idx[bt] = 0;
      if (t == 0) {
        a.meta[0 * a.B + b] = H;
        a.meta[1 * a.B + b] = W;
        a.meta[2 * a.B + b] = gr;
        a.meta[3 * a.B + b] = gc;
        if (n > T && a.status) atomicExch(a.status, 1);
      }
    }
  }
}

// uint8 HWC input, staged through shared memory (round 2, second rewrite).  A register-only row kernel reads coalesced but every one of its
// store instructions touches 32 different 128-byte lines (a lane owns one image row of one token = 16 elements of a plane, the next lane
// the next TOKEN), and the load/store unit needs one pass per line: ncu 1.8 TB/s, LSU wavefronts 71 % of peak.  Here a persistent CTA walks
// STRIPS = the PT image rows of one token row x up to 256 pixels:
//   phase 1: the strip's PT row segments (<= 768 contiguous bytes each) land in shared memory -- one cp.async.bulk per row, completing on
//            an mbarrier, when every segment is 16-byte aligned (all fixed-size configs); otherwise 16-byte loads from the aligned-down
//            address (edge vectors byte by byte, nothing outside [row start, row end) is ever read), the row's misalignment is kept;
//   phase 2: a lane produces 16 output bytes (8 bf16 / 4 fp32 consecutive pixels of one plane row); lanes are ordered along the token's
//            plane, so a warp-wide store writes 512 CONTIGUOUS bytes.  The 3 x PXT source bytes are read as 32-bit words (+ one funnel
//            shift per word for unaligned rows) and normalised through a 256-entry table that is replicated PER LANE
//            (lut[byte][lane]: every lane reads its own bank, so the random byte values cannot collide -- the single 1 KB table of the
//            first uint8 kernel was bounded by exactly those conflicts, and the arithmetic form costs 6 FMA-pipe instructions per byte,
//            which made a first version of this kernel issue-bound at 2.8 TB/s): shift + mask-or + LDS = 3 instructions per byte.
//            The table holds norm_u8 = the reference's own operation order (ops.py:140-161), bit-exact by construction.
// Pixels outside the image (patch padding) are 0.0, applied after normalisation as in the reference (ops.py:235-238).
static constexpr int STRIP_CW = 256;                       // pixels per strip
static constexpr int STRIP_ROW_BYTES = STRIP_CW * 3 + 16;  // 49 vectors: 768 bytes + up to 15 of misalignment
template <int PT>
static constexpr int strip_smem_bytes() { return 256 * 32 * 4 + PT * STRIP_ROW_BYTES + 16; }
template <typename OutT, int PT>
__global__ void __launch_bounds__(256) patchify_u8_strip_kernel(const PatchifyArgs a, const int max_gr, const int nchunk) {
  constexpr int p = PT, pp = p * p, P = 3 * pp;
  constexpr int PXT = 16 / (int)sizeof(OutT);            // pixels per lane
  constexpr int SEG = PT / PXT;                          // lanes per plane row
  constexpr int UPT = PT * SEG;                          // lanes (work units) per token: 32 .. 256, a multiple of 32
  constexpr int NW = (3 * PXT) / 4;                      // source words per unit: 6 / 3
  constexpr int NVEC = STRIP_ROW_BYTES / 16;             // 49
  extern __shared__ __align__(128) uint8_t strip_smem[];
  float* lut = reinterpret_cast<float*>(strip_smem);     // [256][32]
  uint8_t* strip = strip_smem + 256 * 32 * 4;
  __shared__ __align__(8) uint64_t bar;
  __shared__ int mis_s[PT];
  const int tid = threadIdx.x, lane = tid & 31;
  if (tid == 0) {
    mbar_init(&bar, 1);
    fence_barrier_init();
  }
  {
    const float v = norm_u8((uint32_t)tid);   // this warp's 32 entries, one per lane; every lane then writes its own column (bank)
#pragma unroll 8
    for (int j = 0; j < 32; ++j) lut[((tid & ~31) + j) * 32 + lane] = __shfl_sync(0xffffffffu, v, j);
  }
  __syncthreads();
  pdl_wait();
  pdl_trigger();
  const int T = a.max_tokens;
  uint32_t bar_ph = 0;
  const unsigned per_img = (unsigned)max_gr * (unsigned)nchunk;
  const unsigned items = (unsigned)a.B * per_img;
  const uint32_t lut_lane = smem_u32(lut) + (uint32_t)lane * 4u;   // shared-window address of this lane's table column
  for (unsigned it = blockIdx.x; it < items; it += gridDim.x) {
    const int b = (int)(it / per_img);
    const int rem = (int)(it - (unsigned)b * per_img);
    const int r = rem / nchunk, x0 = (rem - r * nchunk) * STRIP_CW;
    const int H = (int)a.img_table[3 * b + 1], W = (int)a.img_table[3 * b + 2];
    const int gr = (H + p - 1) / p, gc = (W + p - 1) / p;
    if (gr * gc > T || r >= gr || x0 >= gc * p) continue;                      // block-uniform
    const uint8_t* img = reinterpret_cast<const uint8_t*>(a.images) + a.img_table[3 * b];
    const int npx = min(STRIP_CW, W - x0);                                      // >= 1: x0 is a multiple of 256 below gc * p, hence below W
    const int nbytes = npx * 3;
    const int nrows = min(p, H - r * p);                                        // image rows in this strip (>= 1)
    const long long rowb = (long long)W * 3;
    const uint8_t* src0 = img + ((long long)(r * p) * W + x0) * 3;
    const bool bulk = ((reinterpret_cast<uintptr_t>(src0) | (uintptr_t)rowb | (uintptr_t)nbytes) & 15) == 0;
    if (bulk) {
      if (tid < 32) {
        fence_proxy_async_smem();   // this buffer was read / written through the generic proxy by the previous item
        if (tid == 0) mbar_expect_tx(&bar, (uint32_t)(nrows * nbytes));
        __syncwarp();
        for (int dy = tid; dy < nrows; dy += 32)
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                           smem_u32(strip + dy * STRIP_ROW_BYTES)),
                       "l"(src0 + dy * rowb), "r"((uint32_t)nbytes), "r"(smem_u32(&bar))
                       : "memory");
      }
      if (tid < PT) mis_s[tid] = 0;
      mbar_wait(&bar, bar_ph);
      bar_ph ^= 1;
      __syncthreads();   // mis_s
    } else {
      constexpr int NIT = (PT * NVEC + 255) / 256;
      uint4 v[NIT];
#pragma unroll
      for (int i = 0; i < NIT; ++i) {
        const int u = tid + 256 * i;
        const int dy = u / NVEC, k = u - dy * NVEC;
        v[i] = make_uint4(0u, 0u, 0u, 0u);
        if (dy < nrows) {
          const uint8_t* sp = src0 + dy * rowb;                                  // row segment [sp, sp + nbytes)
          const int mis = (int)(reinterpret_cast<uintptr_t>(sp) & 15);
          const int lo = 16 * k - mis;                                           // first byte of vector k relative to sp
          if (lo >= 0 && lo + 16 <= nbytes) {
            v[i] = __ldg(reinterpret_cast<const uint4*>(sp + lo));
          } else if (lo + 16 > 0 && lo < nbytes) {                               // edge vector: only the bytes inside the row
            uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll 1
            for (int j = max(0, -lo); j < min(16, nbytes - lo); ++j) {
              const uint32_t by = (uint32_t)__ldg(sp + lo + j) << (8 * (j & 3));
              if ((j >> 2) == 0) w[0] |= by; else if ((j >> 2) == 1) w[1] |= by; else if ((j >> 2) == 2) w[2] |= by; else w[3] |= by;
            }
            v[i] = make_uint4(w[0], w[1], w[2], w[3]);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < NIT; ++i) {
        const int u = tid + 256 * i;
        const int dy = u / NVEC, k = u - dy * NVEC;
        if (dy < PT) *reinterpret_cast<uint4*>(strip + dy * STRIP_ROW_BYTES + 16 * k) = v[i];
      }
      if (tid < PT) mis_s[tid] = (int)(reinterpret_cast<uintptr_t>(src0 + min(tid, nrows - 1) * rowb) & 15);
      __syncthreads();
    }
    // ---- phase 2: 256 / UPT tokens per pass; a thread keeps its (plane row, segment) and walks the tokens
    const int c0 = x0 / p, ntok = min(gc - c0, STRIP_CW / p);
    OutT* const dst_strip = reinterpret_cast<OutT*>(a.patches) + ((long long)b * T + r * gc + c0) * P;
    {
      constexpr int TPP = 256 / UPT;                                             // tokens per pass
      const int q = tid % UPT, dy = q / SEG, seg = q - dy * SEG;
      const int mis = mis_s[dy];
      const bool row_in = (r * p + dy) < H;
      const uint8_t* srow = strip + dy * STRIP_ROW_BYTES;
      for (int tok = tid / UPT; tok < ntok; tok += TPP) {
        const int xl = tok * p + seg * PXT;                                      // pixel offset inside the strip
        const int o = mis + xl * 3;
        const uint32_t* wp = reinterpret_cast<const uint32_t*>(srow + (o & ~3));
        uint32_t w[NW + 1];
#pragma unroll
        for (int k = 0; k <= NW; ++k) w[k] = wp[k];
        if (mis & 3) {                                                           // (block-uniform per row for the usual layouts)
          const uint32_t sh = (uint32_t)(o & 3) * 8u;
#pragma unroll
          for (int k = 0; k < NW; ++k) w[k] = __funnelshift_r(w[k], w[k + 1], sh);
        }
        const int nin = row_in ? min(PXT, W - (x0 + xl)) : 0;                    // pixels of this run inside the image (may be <= 0)
        OutT* dst = dst_strip + tok * P + dy * p + seg * PXT;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
          float f[PXT];
#pragma unroll
          for (int j = 0; j < PXT; ++j) {
            const int i = 3 * j + ch;
            // byte (i & 3) of the word alone in a register (PRMT), times one table row (32 lanes x 4 bytes) plus this lane's column:
            // one ALU-pipe and one FMA-pipe instruction per byte, then the conflict-free LDS
            const uint32_t by = __byte_perm(w[i >> 2], 0u, 0x4440u + (uint32_t)(i & 3));
            asm("ld.shared.f32 %0, [%1];" : "=f"(f[j]) : "r"(by * 128u + lut_lane));
          }
          if (nin < PXT) {
#pragma unroll
            for (int j = 0; j < PXT; ++j) f[j] = j < nin ? f[j] : 0.f;
          }
          if (sizeof(OutT) == 4) {
            *reinterpret_cast<float4*>(dst + ch * pp) = make_float4(f[0], f[1], f[2], f[3]);
          } else {
            *reinterpret_cast<uint4*>(dst + ch * pp) = make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]),
                                                                  pack_bf16x2(f[PXT > 4 ? 4 : 0], f[PXT > 4 ? 5 : 1]),
                                                                  pack_bf16x2(f[PXT > 4 ? 6 : 2], f[PXT > 4 ? 7 : 3]));
          }
        }
      }
    }
    __syncthreads();   // the strip buffer is reused by the next item
  }
  // ---- per token (one THREAD per token): index arrays and metadata; then the zero rows of padding tokens, which are one contiguous
  // range per image ([n_b, T), or all of it when the grid does not fit) written CTA-wide with 16-byte stores
  const unsigned ntokens = (unsigned)a.B * (unsigned)T;
  for (unsigned bt = blockIdx.x * 256u + (unsigned)tid; bt < ntokens; bt += gridDim.x * 256u) {
    const int b = (int)(bt / (unsigned)T), t = (int)(bt - (unsigned)b * (unsigned)T);
    const int H = (int)a.img_table[3 * b + 1], W = (int)a.img_table[3 * b + 2];
    const int gr = (H + p - 1) / p, gc = (W + p - 1) / p;
    const int n = gr * gc;
    const bool valid = t < n && n <= T;
    a.patch_mask[bt] = valid ? 1 : 0;
    a.row_idx[bt] = valid ? t / gc : 0;
    a.col_idx[bt] = valid ? t - (t / gc) * gc : 0;
    a.time_idx[bt] = 0;
    if (t == 0) {
      a.meta[0 * a.B + b] = H;
      a.meta[1 * a.B + b] = W;
      a.meta[2 * a.B + b] = gr;
      a.meta[3 * a.B + b] = gc;
      if (n > T && a.status) atomicExch(a.status, 1);
    }
  }
  for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
    const int H = (int)a.img_table[3 * b + 1], W = (int)a.img_table[3 * b + 2];
    const int n = ((H + p - 1) / p) * ((W + p - 1) / p);
    const int first = n <= T ? n : 0;                                            // first padding token of this image
    uint4* z = reinterpret_cast<uint4*>(reinterpret_cast<OutT*>(a.patches) + ((long long)b * T + first) * P);   // (P * sizeof(OutT) is a multiple of 16)
    const long long nv = (long long)(T - first) * P * (long long)sizeof(OutT) / 16;
    for (long long i = tid; i < nv; i += 256) z[i] = make_uint4(0u, 0u, 0u, 0u);
  }
}

template <typename OutT, int PT>
static int patchify_u8_strip_launch(const PatchifyArgs& a, cudaStream_t stream) {
  const int max_gr = (a.max_h + PT - 1) / PT;
  const int nchunk = ((a.max_w + PT - 1) / PT * PT + STRIP_CW - 1) / STRIP_CW;
  const long long items = (long long)a.B * max_gr * nchunk;
  if (items >= (1ll << 31)) { set_error("patchify: batch bounding box too large"); return -2; }
  auto kern = patchify_u8_strip_kernel<OutT, PT>;
  constexpr int smem = strip_smem_bytes<PT>();
  if (ensure_max_smem(reinterpret_cast<const void*>(kern), smem, "cudaFuncSetAttribute(patchify strips)")) return -1;
  // persistent CTAs (every one builds the 32 KB table once): 4 (p = 16: 45 KB) / 3 (p = 32: 57 KB) per SM
  long long blocks = (long long)num_sms() * (PT == 16 ? 4 : 3);
  if (blocks > items) blocks = items;
  if (blocks < 1) blocks = 1;
  (void)launch_k(kern, dim3((unsigned)blocks), dim3(256), smem, stream, a, max_gr, nchunk);
  return 0;
}

template <typename OutT>
static void patchify_dispatch(const PatchifyArgs& a, int blocks, cudaStream_t stream) {
  if (a.patch == 16) (void)launch_k(patchify_kernel<OutT, 16>, dim3(blocks), dim3(256), 0, stream, a);
  else if (a.patch == 32) (void)launch_k(patchify_kernel<OutT, 32>, dim3(blocks), dim3(256), 0, stream, a);
  else (void)launch_k(patchify_kernel<OutT, 0>, dim3(blocks), dim3(256), 0, stream, a);
}

int launch_patchify(const PatchifyArgs& a, cudaStream_t stream) {
  if (a.patch % 4 || a.patch <= 0) { set_error("patchify: patch size must be a positive multiple of 4 (got %d)", a.patch); return -2; }
  if (a.B <= 0 || a.max_tokens <= 0) return 0;
  const long long ntok = (long long)a.B * a.max_tokens;
  if (ntok >= (1ll << 31)) { set_error("patchify: B * max_tokens too large"); return -2; }
  if (a.in_dtype == 1 && (a.patch == 16 || a.patch == 32) && a.max_h > 0 && a.max_w > 0) {
    // uint8 HWC front end over the batch's bounding box (the caller knows every image size): the shared-memory-staged strip kernel
    int rc;
    if (a.out_dtype == 0) rc = a.patch == 16 ? patchify_u8_strip_launch<float, 16>(a, stream) : patchify_u8_strip_launch<float, 32>(a, stream);
    else rc = a.patch == 16 ? patchify_u8_strip_launch<bf16, 16>(a, stream) : patchify_u8_strip_launch<bf16, 32>(a, stream);
    if (rc) return rc;
    return check_cuda(cudaGetLastError(), "patchify (uint8 strips) launch");
  }
  long long blocks = (ntok + 7) / 8;                   // one warp per token, 8 warps per CTA: the block scheduler balances the tail
  const long long cap = (long long)num_sms() * 8 * 16;  // (a fixed grid of one wave left the last tokens to a few warps); warp-stride beyond
  if (blocks > cap) blocks = cap;
  if (a.out_dtype == 0) patchify_dispatch<float>(a, (int)blocks, stream);
  else patchify_dispatch<bf16>(a, (int)blocks, stream);
  return check_cuda(cudaGetLastError(), "patchify launch");
}

int launch_patchify_selftest(int* mismatches, cudaStream_t stream) {
  if (check_cuda(cudaMemsetAsync(mismatches, 0, sizeof(int), stream), "selftest memset")) return -1;
  patchify_selftest_kernel<<<1, 256, 0, stream>>>(mismatches);
  return check_cuda(cudaGetLastError(), "patchify selftest launch");
}

// ---------------------------------------------------------------------------------------------
// resize_to_token_budget + normalize + patchify (vitok/pp/ops.py:169-214, :217-285)
//
// The reference resizes an over-budget [3,H,W] fp32 image with TF.resize(BICUBIC, antialias=True), i.e. ATen's CPU
// _upsample_bicubic2d_aa (align_corners=False): separable, width pass first, an axis whose size is unchanged is not resampled.
// Here: (1) plan = prefix sums over the batch -> workspace header; (2) per-image resample tables; (3) width pass, one CTA per source
// row staged in shared memory, into an fp32 [3, H, w'] scratch image; (4) height pass fused with patchify, one warp per token.
// ---------------------------------------------------------------------------------------------
static constexpr int RS_ROW_CAP = 4096;   // source rows up to this width are staged in shared memory (3 x 4096 fp32 = 48 KB)

// ATen's cubic filter with a = -0.5 (antialiased bicubic) in fp32.  The CPU build contracts both polynomials into FMAs; so do we
// (the resulting weights equal torch's one-hot weight matrices exactly).
__device__ __forceinline__ float aa_cubic(float x) {
  x = fabsf(x);
  if (x < 1.f) return __fmaf_rn(__fmul_rn(__fmaf_rn(1.5f, x, -2.5f), x), x, 1.f);
  if (x < 2.f) return __fmaf_rn(__fmaf_rn(__fmaf_rn(-0.5f, x, 2.5f), x, -4.f), x, 2.f);
  return 0.f;
}

// Table column of output coordinate o (ATen _compute_indices_min_size_weights_aa, with its float / double mix), stored with stride
// n_out (tap-major, so that the lanes of a warp, which own consecutive outputs, read consecutive words): [0] = xmin and [1] = tap
// count as int bits, [2 ..] = the normalised weights, zero beyond the tap count.
__device__ void aa_entry(int n_in, int n_out, int o, int kt, float* e) {
  const int st = n_out;
  const float scale = __fdiv_rn((float)n_in, (float)n_out);
  const float support = scale >= 1.f ? __fmul_rn(2.f, scale) : 2.f;
  const int kmax = (int)ceilf(support) * 2 + 1;
  const float invscale = scale >= 1.f ? (float)(1.0 / (double)scale) : 1.f;
  const float center = (float)((double)scale * ((double)o + 0.5));
  const int xmin = max((int)((double)__fsub_rn(center, support) + 0.5), 0);
  int xs = min((int)((double)__fadd_rn(center, support) + 0.5), n_in) - xmin;
  xs = min(max(xs, 0), min(kmax, kt));
  float* w = e + 2 * st;
  float tot = 0.f;
  for (int j = 0; j < xs; ++j) {
    const float d = __fsub_rn((float)(j + xmin), center);
    w[j * st] = aa_cubic((float)(((double)d + 0.5) * (double)invscale));
    tot = __fadd_rn(tot, w[j * st]);
  }
  if (tot != 0.f)
    for (int j = 0; j < xs; ++j) w[j * st] = __fdiv_rn(w[j * st], tot);
  for (int j = xs; j < kt; ++j) w[j * st] = 0.f;
  e[0] = __int_as_float(xmin);
  e[st] = __int_as_float(xs);
}

// plan: one CTA.  Workspace = header, then one region per image: its resample tables (width, then height), then its width-pass
// scratch image.  hdr[0 .. B] = region offsets in floats from the end of the header, hdr[B+1 .. 2B+1] = width-pass row prefix,
// hdr[2B+2] = 1 when the batch is usable (every size >= 1 and the workspace large enough).
__global__ void __launch_bounds__(1024) resize_plan_kernel(const int64_t* __restrict__ tab, int B, long long ws_bytes, int64_t* hdr,
                                                           int* status) {
  pdl_wait();
  pdl_trigger();
  __shared__ long long sh[2][1024];
  __shared__ int bad;
  const int tid = threadIdx.x, nt = blockDim.x;
  if (tid == 0) bad = 0;
  const int per = (B + nt - 1) / nt, b0 = min(B, tid * per), b1 = min(B, b0 + per);
  long long s[2] = {0, 0};
  __syncthreads();
  for (int b = b0; b < b1; ++b) {
    const ResizeImage im = resize_image(tab, b);
    if (im.H < 1 || im.W < 1 || im.h < 1 || im.w < 1) bad = 1;
    s[0] += im.region_floats(); s[1] += im.width_rows();
  }
  sh[0][tid] = s[0]; sh[1][tid] = s[1];
  __syncthreads();
  for (int d = 1; d < nt; d <<= 1) {                 // inclusive scan of the per-thread sums
    const long long v0 = tid >= d ? sh[0][tid - d] : 0, v1 = tid >= d ? sh[1][tid - d] : 0;
    __syncthreads();
    sh[0][tid] += v0; sh[1][tid] += v1;
    __syncthreads();
  }
  long long r0 = sh[0][tid] - s[0], r1 = sh[1][tid] - s[1];
  for (int b = b0; b < b1; ++b) {
    const ResizeImage im = resize_image(tab, b);
    hdr[b] = r0; hdr[B + 1 + b] = r1;
    r0 += im.region_floats(); r1 += im.width_rows();
  }
  if (tid == nt - 1) {
    hdr[B] = sh[0][tid]; hdr[2 * B + 1] = sh[1][tid];
    const bool ok = !bad && sh[1][tid] < (1ll << 31) && resize_header_bytes(B) + 4 * (size_t)sh[0][tid] <= (size_t)ws_bytes;
    hdr[2 * B + 2] = ok ? 1 : 0;
    if (!ok && status) atomicExch(status, 2);
  }
}

__global__ void __launch_bounds__(256) resize_tables_kernel(const int64_t* __restrict__ tab, int B, const int64_t* __restrict__ hdr,
                                                            float* data) {
  pdl_wait();
  pdl_trigger();
  if (!hdr[2 * B + 2]) return;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    const ResizeImage im = resize_image(tab, b);
    float* t = data + hdr[b];
    if (im.w != im.W) {
      const int kt = resize_kt(im.W, im.w);
      for (int o = threadIdx.x; o < im.w; o += blockDim.x) aa_entry(im.W, im.w, o, kt, t + o);
      t += (long long)im.w * (kt + 2);
    }
    if (im.h != im.H) {
      const int kt = resize_kt(im.H, im.h);
      for (int o = threadIdx.x; o < im.h; o += blockDim.x) aa_entry(im.H, im.h, o, kt, t + o);
    }
  }
}

// source pixel (ch, y, x) as the reference's normalised fp32 tensor holds it (the uint8 value is what patchify's front end produces)
__device__ __forceinline__ float resize_src(const void* images, int in_dtype, long long off, int H, int W, int ch, int y, int x) {
  if (in_dtype == 1) return norm_u8_fast(__ldg(reinterpret_cast<const uint8_t*>(images) + off + ((long long)y * W + x) * 3 + ch));
  return __ldg(reinterpret_cast<const float*>(images) + off + ((long long)ch * H + y) * W + x);
}

// width pass: work item = one source row of an image whose width changes; the row (normalised fp32, 3 planes) is staged in shared
// memory when it is at most RS_ROW_CAP pixels wide.  Each output sums its taps in order in fp32, every product rounded before it is
// added (ATen's loop: out = x0 * w0; out += xj * wj).
__global__ void __launch_bounds__(256) resize_width_kernel(const void* __restrict__ images, int in_dtype, const int64_t* __restrict__ tab,
                                                           int B, const int64_t* __restrict__ hdr, float* data) {
  extern __shared__ float row_s[];
  pdl_wait();
  pdl_trigger();
  if (!hdr[2 * B + 2]) return;
  const int64_t* rows = hdr + B + 1;
  const int items = (int)rows[B];                    // sum of the heights of the images whose width changes
  for (int it = blockIdx.x; it < items; it += gridDim.x) {
    int lo = 0, hi = B - 1;                          // the image b with rows[b] <= it < rows[b + 1]
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (rows[mid] <= it) lo = mid; else hi = mid - 1;
    }
    const int b = lo, y = (int)(it - rows[b]);
    const ResizeImage im = resize_image(tab, b);
    const int W = im.W, w2 = im.w, kt = resize_kt(W, w2);
    const bool staged = W <= RS_ROW_CAP;
    if (staged) {
      if (in_dtype == 1) {
        const uint8_t* src = reinterpret_cast<const uint8_t*>(images) + im.off + (long long)y * W * 3;
        for (int i = threadIdx.x; i < 3 * W; i += blockDim.x) {
          const int px = i / 3, ch = i - px * 3;
          row_s[ch * W + px] = norm_u8_fast(__ldg(src + i));
        }
      } else {
        for (int i = threadIdx.x; i < 3 * W; i += blockDim.x) {
          const int ch = i / W, x = i - ch * W;
          row_s[i] = __ldg(reinterpret_cast<const float*>(images) + im.off + ((long long)ch * im.H + y) * W + x);
        }
      }
      __syncthreads();
    }
    const float* tw = data + hdr[b];
    float* dst = data + hdr[b] + im.table_floats() + (long long)y * w2;
    const long long plane = (long long)im.H * w2;
    for (int i = threadIdx.x; i < 3 * w2; i += blockDim.x) {
      const int ch = i / w2, o = i - ch * w2;
      const float* e = tw + o;                       // column o of the tap-major table (stride w2)
      const int xmin = __float_as_int(e[0]), xs = __float_as_int(e[w2]);
      const float* wt = e + 2 * w2;
      float acc = 0.f;
      if (staged) {
        const float* s = row_s + ch * W + xmin;
        if (xs > 0) acc = __fmul_rn(s[0], wt[0]);
        for (int j = 1; j < xs; ++j) acc = __fadd_rn(acc, __fmul_rn(s[j], wt[j * w2]));
      } else {
        if (xs > 0) acc = __fmul_rn(resize_src(images, in_dtype, im.off, im.H, W, ch, y, xmin), wt[0]);
        for (int j = 1; j < xs; ++j)
          acc = __fadd_rn(acc, __fmul_rn(resize_src(images, in_dtype, im.off, im.H, W, ch, y, xmin + j), wt[j * w2]));
      }
      dst[ch * plane + o] = acc;
    }
    __syncthreads();                                 // row_s is reused by the next item
  }
}

// height pass + patchify: one warp per output token, element order ch * p^2 + dy * p + dx.  Pixels come from the width pass's scratch
// image, or straight from the source when the width is unchanged; an image of unchanged size reads exactly what patchify reads.
template <typename OutT>
__global__ void __launch_bounds__(256) resize_patchify_kernel(const ResizePatchifyArgs a, const int64_t* __restrict__ hdr,
                                                              const float* __restrict__ data) {
  pdl_wait();
  pdl_trigger();
  const int p = a.patch, pp = p * p, P = 3 * pp, T = a.max_tokens, B = a.B;
  const bool ok = hdr[2 * B + 2] != 0;
  const int lane = threadIdx.x & 31;
  const unsigned ntok = (unsigned)B * (unsigned)T;
  const unsigned nwarp = gridDim.x * (blockDim.x >> 5);
  for (unsigned bt = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); bt < ntok; bt += nwarp) {
    const int b = (int)(bt / (unsigned)T), t = (int)(bt - (unsigned)b * (unsigned)T);
    const ResizeImage im = resize_image(a.img_table, b);
    const int h2 = im.h, w2 = im.w;
    const bool sized = h2 >= 1 && w2 >= 1;
    const int gr = sized ? (h2 + p - 1) / p : 0, gc = sized ? (w2 + p - 1) / p : 0, n = gr * gc;
    const bool rs_w = w2 != im.W, rs_h = h2 != im.H;
    const bool valid = t < n && n <= T;
    const bool data_ok = valid && (ok || (!rs_w && !rs_h));       // an unusable workspace leaves the resized images' patches zero
    const int r = valid ? t / gc : 0, c = valid ? t - (t / gc) * gc : 0;
    OutT* dst = reinterpret_cast<OutT*>(a.patches) + (long long)bt * P;
    const float* reg = data + (ok ? hdr[b] : 0);
    const float* scr = reg + (ok ? im.table_floats() : 0);
    const float* th = reg + (rs_w ? (long long)w2 * (resize_kt(im.W, w2) + 2) : 0);
    for (int e = lane; e < P; e += 32) {
      const int ch = e / pp, rem = e - ch * pp, dy = rem / p, dx = rem - dy * p;
      const int y = r * p + dy, x = c * p + dx;
      float v = 0.f;                                 // zero padding to the patch grid (ops.py:235-238)
      if (data_ok && y < h2 && x < w2) {
        if (rs_h) {
          const float* ey = th + y;                  // column y of the tap-major table (stride h2)
          const int ymin = __float_as_int(ey[0]), ys = __float_as_int(ey[h2]);
          for (int j = 0; j < ys; ++j) {
            const float s = rs_w ? scr[((long long)ch * im.H + ymin + j) * w2 + x]
                                 : resize_src(a.images, a.in_dtype, im.off, im.H, im.W, ch, ymin + j, x);
            const float wj = ey[(2 + j) * h2];
            v = j == 0 ? __fmul_rn(s, wj) : __fadd_rn(v, __fmul_rn(s, wj));
          }
        } else {
          v = rs_w ? scr[((long long)ch * im.H + y) * w2 + x] : resize_src(a.images, a.in_dtype, im.off, im.H, im.W, ch, y, x);
        }
      }
      if (sizeof(OutT) == 4) reinterpret_cast<float*>(dst)[e] = v;
      else reinterpret_cast<bf16*>(dst)[e] = __float2bfloat16_rn(v);
    }
    if (lane == 0) {
      a.patch_mask[bt] = valid ? 1 : 0;
      a.row_idx[bt] = r;
      a.col_idx[bt] = c;
      a.time_idx[bt] = 0;
      if (t == 0) {
        a.meta[0 * B + b] = h2;                      // the reference's patchify sees the resized tensor
        a.meta[1 * B + b] = w2;
        a.meta[2 * B + b] = gr;
        a.meta[3 * B + b] = gc;
        if (n > T && a.status) atomicExch(a.status, 1);
      }
    }
  }
}

int launch_resize_patchify(const ResizePatchifyArgs& a, cudaStream_t stream) {
  if (a.patch <= 0) { set_error("resize_patchify: patch size must be positive (got %d)", a.patch); return -2; }
  if (a.B <= 0 || a.max_tokens <= 0) return 0;
  const long long ntok = (long long)a.B * a.max_tokens;
  if (ntok >= (1ll << 31)) { set_error("resize_patchify: B * max_tokens too large"); return -2; }
  const size_t hb = resize_header_bytes(a.B);
  if (a.workspace_bytes < hb) {
    set_error("resize_patchify: workspace of %zu bytes is smaller than its %zu-byte header", a.workspace_bytes, hb);
    return -2;
  }
  int64_t* hdr = reinterpret_cast<int64_t*>(a.workspace);
  float* data = reinterpret_cast<float*>(reinterpret_cast<char*>(a.workspace) + hb);
  const int sms = num_sms();
  // the work sizes (rows to resample, table entries) are known only on the device: persistent grids that read them from the header
  (void)launch_k(resize_plan_kernel, dim3(1), dim3(1024), 0, stream, a.img_table, a.B, (long long)a.workspace_bytes, hdr, a.status);
  (void)launch_k(resize_tables_kernel, dim3((unsigned)min(a.B, 4 * sms)), dim3(256), 0, stream, a.img_table, a.B, (const int64_t*)hdr,
                 data);
  (void)launch_k(resize_width_kernel, dim3((unsigned)(8 * sms)), dim3(256), (size_t)(3 * RS_ROW_CAP * sizeof(float)), stream, a.images,
                 a.in_dtype, a.img_table, a.B, (const int64_t*)hdr, data);
  long long blocks = (ntok + 7) / 8;                 // one warp per token, 8 warps per CTA
  const long long cap = (long long)sms * 8 * 16;
  if (blocks > cap) blocks = cap;
  if (a.out_dtype == 0)
    (void)launch_k(resize_patchify_kernel<float>, dim3((unsigned)blocks), dim3(256), 0, stream, a, (const int64_t*)hdr, (const float*)data);
  else
    (void)launch_k(resize_patchify_kernel<bf16>, dim3((unsigned)blocks), dim3(256), 0, stream, a, (const int64_t*)hdr, (const float*)data);
  return check_cuda(cudaGetLastError(), "resize_patchify launch");
}

size_t resize_workspace_bytes(const int64_t* img_table_host, int B) {
  size_t floats = 0;
  for (int b = 0; b < B; ++b) floats += (size_t)resize_image(img_table_host, b).region_floats();
  return resize_header_bytes(B) + 4 * floats;
}

// ---------------------------------------------------------------------------------------------
// unpatchify
// ---------------------------------------------------------------------------------------------
__global__ void cellmap_kernel(const UnpatchifyArgs a) {
  pdl_wait();      // PDL (vtk_common.cuh): this kernel may have been launched before its predecessor finished
  pdl_trigger();
  const long long total = (long long)a.B * a.N;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    if (!a.patch_mask[i]) continue;
    const int b = (int)(i / a.N), t = (int)(i % a.N);
    const long long r = a.row_idx[i], c = a.col_idx[i];
    const long long cell = r * a.gx + c;   // flat_idx = row * max_x + col (ops.py:328)
    if (r < 0 || c < 0 || cell >= (long long)a.gy * a.gx) {
      if (a.status) atomicExch(a.status, 1);   // the reference's scatter raises an index error here
      continue;
    }
    atomicMax(&a.cell_map[(long long)b * a.gy * a.gx + cell], t);
  }
}

__device__ __forceinline__ float convert_px(float x, int fmt, bool bf16_math) {
  // vitok/pp/io.py:91-121 from "minus_one_to_one"; each eager op rounds to the tensor dtype.  Halving is exact in both
  // dtypes, so "/ 2" is a multiplication by 0.5 (no division sequence on the XU pipe)
  if (fmt == 1) {  // 0_255: ((clamp(x,-1,1) + 1) / 2 * 255).round()
    float t = fminf(fmaxf(x, -1.f), 1.f);
    if (bf16_math) { t = bf16r(t + 1.f); t = bf16r(t * 0.5f); t = bf16r(t * 255.f); }
    else { t = __fadd_rn(t, 1.f); t = __fmul_rn(t, 0.5f); t = __fmul_rn(t, 255.f); }
    return rintf(t);
  }
  if (fmt == 2) {  // zero_to_one: ((x + 1) / 2).clamp(0, 1)
    float t;
    if (bf16_math) { t = bf16r(x + 1.f); t = bf16r(t * 0.5f); }
    else { t = __fmul_rn(__fadd_rn(x, 1.f), 0.5f); }
    return fminf(fmaxf(t, 0.f), 1.f);
  }
  return x;
}

// Four pixels of the "0_255" conversion -> packed uchar4, with no conversion-pipe (XU) instruction: the bf16 roundings are packed
// cvt.rn.bf16x2.f32 (bf16(bf16(t * 0.5) * 255) == bf16(t * 127.5): halving is exact and an 8-bit x 8-bit significand product is exact
// in fp32, so both round the same real number once), and round() + the cast to uint8 are one FADD with 1.5 * 2^23 (round to nearest
// even in the low mantissa bits, what torch.round does) + a mask.  The first version (F2F / FRND / F2I per element) was XU-bound.
__device__ __forceinline__ uint32_t to_u8x4(const float (&v)[4], bool bf16_math) {
  float t[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) t[k] = fminf(fmaxf(v[k], -1.f), 1.f);
  if (bf16_math) {
    const uint32_t a01 = bf2_cvt(t[0] + 1.f, t[1] + 1.f), a23 = bf2_cvt(t[2] + 1.f, t[3] + 1.f);
    const uint32_t b01 = bf2_cvt(bf16_lo(a01) * 127.5f, bf16_hi(a01) * 127.5f), b23 = bf2_cvt(bf16_lo(a23) * 127.5f, bf16_hi(a23) * 127.5f);
    t[0] = bf16_lo(b01); t[1] = bf16_hi(b01); t[2] = bf16_lo(b23); t[3] = bf16_hi(b23);
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) t[k] = __fmul_rn(__fmul_rn(__fadd_rn(t[k], 1.f), 0.5f), 255.f);
  }
  uint32_t r = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) r |= (__float_as_uint(__fadd_rn(t[k], 12582912.f)) & 255u) << (8 * k);
  return r;
}

// One warp per canvas cell (b, r, c): the token that owns the cell is looked up once, its 3p^2 elements are read as
// contiguous 8 / 16-byte chunks (coalesced) and written as p-pixel row segments of the three channel planes.  Patch sizes
// other than 16 / 32 (any multiple of 4); those two have the row kernel below.
template <typename T>
__global__ void __launch_bounds__(256) unpatchify_kernel(const UnpatchifyArgs a) {
  pdl_wait();      // PDL (vtk_common.cuh): this kernel may have been launched before its predecessor finished
  pdl_trigger();
  const int p = a.patch, pp = p * p, P = 3 * pp, p4 = p >> 2, chunks = pp >> 2;
  const int Hc = a.gy * p, Wc = a.gx * p;
  const int cells_per_img = a.gy * a.gx;
  const unsigned ncell = (unsigned)a.B * (unsigned)cells_per_img;
  const bool bfm = sizeof(T) == 2;
  const int lane = threadIdx.x & 31;
  const unsigned nwarp = gridDim.x * (blockDim.x >> 5);
  for (unsigned bc = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); bc < ncell; bc += nwarp) {
    const int b = (int)(bc / (unsigned)cells_per_img), cell = (int)(bc - (unsigned)b * (unsigned)cells_per_img);
    const int r = cell / a.gx, c = cell - r * a.gx;
    // token 0 is re-scattered into cell 0 after the main scatter (ops.py:332-333)
    const int tok = (cell == 0) ? (a.patch_mask[(long long)b * a.N] ? 0 : -1) : a.cell_map[bc];
    const T* src = reinterpret_cast<const T*>(a.patches) + ((long long)b * a.N + (tok >= 0 ? tok : 0)) * P;
#pragma unroll 2
    for (int e4 = lane; e4 < 3 * chunks; e4 += 32) {
      const int ch = e4 / chunks, rem = e4 - ch * chunks;
      const int dy = rem / p4, dx = (rem - dy * p4) << 2;
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      if (tok >= 0) {
        if (sizeof(T) == 4) {
          const float4 f = __ldg(reinterpret_cast<const float4*>(src + (e4 << 2)));
          v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
        } else {
          const uint2 u = __ldg(reinterpret_cast<const uint2*>(src + (e4 << 2)));
          v[0] = bf16_lo(u.x); v[1] = bf16_hi(u.x); v[2] = bf16_lo(u.y); v[3] = bf16_hi(u.y);
        }
      }
      const long long o = (((long long)b * 3 + ch) * Hc + r * p + dy) * Wc + c * p + dx;
      if (a.out_format == 1) {
        *reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(a.out) + o) = to_u8x4(v, bfm);
      } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = convert_px(v[k], a.out_format, bfm);
        if (sizeof(T) == 4) {
          *reinterpret_cast<float4*>(reinterpret_cast<float*>(a.out) + o) = make_float4(v[0], v[1], v[2], v[3]);
        } else {
          *reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(a.out) + o) = make_uint2(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]));
        }
      }
    }
  }
}

// Row-coalesced variant (compile-time patch size): thread <-> PXT consecutive pixels of FOUR consecutive canvas rows of one channel
// plane, PXT chosen so that every store is 16 bytes (16 pixels of uint8, 8 of bf16, 4 of fp32).  A warp writes 512 contiguous bytes per
// row -- the cell-per-warp kernel above writes p-pixel pieces (16 bytes of uint8: half a sector) -- and reads the owning tokens'
// elements as 16-byte chunks.  The four rows lie in the same patch row, so one cell-map lookup serves all the loads, which are issued
// before the first store.
template <typename T, int PT, int PXT, bool U8OUT>
__global__ void __launch_bounds__(256) unpatchify_rows_kernel(const UnpatchifyArgs a) {
  pdl_wait();
  pdl_trigger();
  constexpr int p = PT, pp = p * p, P = 3 * pp;
  constexpr int LV = PXT * (int)sizeof(T) / 16;     // 16-byte loads per row
  static_assert(PT % PXT == 0 && LV >= 1, "unpatchify_rows: PXT must divide the patch size and fill a 16-byte load");
  const int Hc = a.gy * p, Wc = a.gx * p, WX = Wc / PXT, R4 = Hc >> 2;
  const int cells_per_img = a.gy * a.gx;
  const bool bfm = sizeof(T) == 2;
  const long long total = (long long)a.B * 3 * R4 * WX;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int xq = (int)(idx % WX);
    const long long t1 = idx / WX;
    const int yq = (int)(t1 % R4);
    const int t2 = (int)(t1 / R4);
    const int ch = t2 % 3, b = t2 / 3;
    const int y0 = yq << 2, x = xq * PXT;
    const int r = y0 / p, dy0 = y0 - r * p, c = x / p, dx = x - c * p;
    const int cell = r * a.gx + c;
    // token 0 is re-scattered into cell 0 after the main scatter (ops.py:332-333)
    const int tok = (cell == 0) ? (a.patch_mask[(long long)b * a.N] ? 0 : -1) : a.cell_map[(long long)b * cells_per_img + cell];
    uint4 raw[4][LV];
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int l = 0; l < LV; ++l) raw[k][l] = make_uint4(0u, 0u, 0u, 0u);     // (0.0 in both dtypes)
    if (tok >= 0) {
      const T* src = reinterpret_cast<const T*>(a.patches) + ((long long)b * a.N + tok) * P + ch * pp + dy0 * p + dx;
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int l = 0; l < LV; ++l) raw[k][l] = __ldg(reinterpret_cast<const uint4*>(src + k * p) + l);
    }
    const long long o = (((long long)b * 3 + ch) * Hc + y0) * Wc + x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float v[PXT];
#pragma unroll
      for (int l = 0; l < LV; ++l) {
        const uint32_t w[4] = {raw[k][l].x, raw[k][l].y, raw[k][l].z, raw[k][l].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          if (sizeof(T) == 4) v[4 * l + e] = __uint_as_float(w[e]);
          else { v[8 * l + 2 * e] = bf16_lo(w[e]); v[8 * l + 2 * e + 1] = bf16_hi(w[e]); }
        }
      }
      if (U8OUT) {
        uint32_t q[PXT / 4];
#pragma unroll
        for (int g = 0; g < PXT / 4; ++g) {
          const float f4[4] = {v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]};
          q[g] = to_u8x4(f4, bfm);
        }
        uint8_t* op = reinterpret_cast<uint8_t*>(a.out) + o + (long long)k * Wc;
        if (PXT == 16) *reinterpret_cast<uint4*>(op) = make_uint4(q[0], q[1], q[2 % (PXT / 4)], q[3 % (PXT / 4)]);
        else
#pragma unroll
          for (int g = 0; g < PXT / 4; ++g) *reinterpret_cast<uint32_t*>(op + 4 * g) = q[g];
      } else {
#pragma unroll
        for (int e = 0; e < PXT; ++e) v[e] = convert_px(v[e], a.out_format, bfm);
        if (sizeof(T) == 4) {
          float* op = reinterpret_cast<float*>(a.out) + o + (long long)k * Wc;
#pragma unroll
          for (int g = 0; g < PXT / 4; ++g) *reinterpret_cast<float4*>(op + 4 * g) = make_float4(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
        } else {
          bf16* op = reinterpret_cast<bf16*>(a.out) + o + (long long)k * Wc;
#pragma unroll
          for (int g = 0; g < PXT / 8; ++g)
            *reinterpret_cast<uint4*>(op + 8 * g) = make_uint4(pack_bf16x2(v[8 * g], v[8 * g + 1]), pack_bf16x2(v[8 * g + 2], v[8 * g + 3]),
                                                               pack_bf16x2(v[8 * g + 4], v[8 * g + 5]), pack_bf16x2(v[8 * g + 6], v[8 * g + 7]));
        }
      }
    }
  }
}

template <typename T, int PT>
static void unpatchify_rows_launch(const UnpatchifyArgs& a, cudaStream_t stream) {
  constexpr int PX_SAME = 16 / (int)sizeof(T);     // same-dtype output: 16-byte stores
  const bool u8 = a.out_format == 1;
  const int pxt = u8 ? 16 : PX_SAME;
  const long long total = (long long)a.B * 3 * (a.gy * PT / 4) * (a.gx * PT / pxt);
  long long rb = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 8 * 16;
  if (rb > cap) rb = cap;
  if (u8) (void)launch_k(unpatchify_rows_kernel<T, PT, 16, true>, dim3((unsigned)rb), dim3(256), 0, stream, a);
  else (void)launch_k(unpatchify_rows_kernel<T, PT, PX_SAME, false>, dim3((unsigned)rb), dim3(256), 0, stream, a);
}

template <typename T>
static void unpatchify_dispatch(const UnpatchifyArgs& a, int blocks, cudaStream_t stream) {
  if (a.patch == 16) unpatchify_rows_launch<T, 16>(a, stream);
  else if (a.patch == 32) unpatchify_rows_launch<T, 32>(a, stream);
  else (void)launch_k(unpatchify_kernel<T>, dim3(blocks), dim3(256), 0, stream, a);
}

int launch_cellmap(const UnpatchifyArgs& a, cudaStream_t stream) {
  const long long cells = (long long)a.B * a.gy * a.gx;
  if (check_cuda(cudaMemsetAsync(a.cell_map, 0xFF, cells * sizeof(int), stream), "cell_map memset")) return -1;
  const long long cap = (long long)num_sms() * 16;
  long long blocks = ((long long)a.B * a.N + 255) / 256;
  if (blocks > cap) blocks = cap;
  (void)launch_k(cellmap_kernel, dim3((int)blocks), dim3(256), 0, stream, a);
  return 0;
}

int launch_unpatchify(const UnpatchifyArgs& a, cudaStream_t stream) {
  if (a.patch % 4 || a.patch <= 0) { set_error("unpatchify: patch size must be a positive multiple of 4 (got %d)", a.patch); return -2; }
  if (a.gy <= 0 || a.gx <= 0) { set_error("unpatchify: empty canvas %dx%d", a.gy, a.gx); return -2; }
  if (a.B <= 0) return 0;
  if (int rc = launch_cellmap(a, stream)) return rc;
  const long long cells = (long long)a.B * a.gy * a.gx;
  if (cells >= (1ll << 31)) { set_error("unpatchify: canvas too large"); return -2; }
  long long blocks = (cells + 7) / 8;                    // one warp per cell, 8 warps per CTA
  const long long cap2 = (long long)num_sms() * 8 * 16;
  if (blocks > cap2) blocks = cap2;
  if (a.dtype == 0) unpatchify_dispatch<float>(a, (int)blocks, stream);
  else unpatchify_dispatch<bf16>(a, (int)blocks, stream);
  return check_cuda(cudaGetLastError(), "unpatchify launch");
}

// out2[0] = max(row)+1, out2[1] = max(col)+1 over valid tokens (ops.py:319-321); out2 must be zeroed.
__global__ void grid_extent_kernel(const uint8_t* __restrict__ mask, const int64_t* __restrict__ row,
                                   const int64_t* __restrict__ col, long long total, int* out2) {
  pdl_wait();      // PDL (vtk_common.cuh): this kernel may have been launched before its predecessor finished
  pdl_trigger();
  int my = 0, mx = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    if (mask[i]) {
      my = max(my, (int)row[i] + 1);
      mx = max(mx, (int)col[i] + 1);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    my = max(my, __shfl_xor_sync(0xffffffffu, my, o));
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMax(&out2[0], my);
    atomicMax(&out2[1], mx);
  }
}
int launch_grid_extent(const uint8_t* mask, const int64_t* row, const int64_t* col, int B, int N, int* out2,
                       cudaStream_t stream) {
  if (check_cuda(cudaMemsetAsync(out2, 0, 2 * sizeof(int), stream), "grid_extent memset")) return -1;
  const long long total = (long long)B * N;
  if (total <= 0) return 0;
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 4;
  if (blocks > cap) blocks = cap;
  (void)launch_k(grid_extent_kernel, dim3((int)blocks), dim3(256), 0, stream, mask, row, col, total, out2);
  return check_cuda(cudaGetLastError(), "grid_extent launch");
}

}  // namespace vtk
