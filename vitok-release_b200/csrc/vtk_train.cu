// vtk_train.cu -- HBM-bound kernels of the training step (BASELINE config 5): the un-fused forward pieces that
// keep what the backward pass needs, and the backward of every non-GEMM op of the AE block.
//
// Reference being restated (autograd of these eager ops; scripts/train_vae.py:304-320,371-372 drives them):
//   Block.forward            vitok/models/ae.py:55-65        x + gamma * (attn(h) + mlp(h)), h = RMSNorm(x)
//   RMSNorm                  modules/norm.py:17-25           fp32 math, eps inside rsqrt
//   QK-norm + 2D RoPE        modules/attention.py:103-107, modules/rotary_embedding.py:102-129
//   SwiGLU                   modules/mlp.py:20-23
//   LayerNorm (no affine)    modules/norm.py:28-39           the latent bottleneck's output_fn
//   Charbonnier loss         scripts/train_vae.py:314-320    sqrt(diff^2 + eps^2), masked per-image mean
//   AdamW (multi-tensor)     scripts/train_vae.py:185-208    torch.optim.AdamW semantics, fp32 master weights + fp32 moments
//
// GEMMs of the backward pass (dgrad / wgrad) run on the tcgen05 GEMM of vtk_gemm.cu with transposed-operand variants (the
// weights and activations are read MN-major as stored: no transposed copies).
#include <stdlib.h>

#include <algorithm>
#include <type_traits>

#include "vtk_common.cuh"
#include "vtk_kernels.h"

namespace vtk {

static __device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
static __device__ __forceinline__ void unpack8(const uint4& q, float (&f)[8]) {
  f[0] = bf16_lo(q.x); f[1] = bf16_hi(q.x); f[2] = bf16_lo(q.y); f[3] = bf16_hi(q.y);
  f[4] = bf16_lo(q.z); f[5] = bf16_hi(q.z); f[6] = bf16_lo(q.w); f[7] = bf16_hi(q.w);
}
static __device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  return make_uint4(bf2_cvt(f[0], f[1]), bf2_cvt(f[2], f[3]), bf2_cvt(f[4], f[5]), bf2_cvt(f[6], f[7]));
}
static int grid_for(long long work_items, int per_block, int waves = 16) {
  long long b = (work_items + per_block - 1) / per_block;
  const long long cap = (long long)num_sms() * waves;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

// ------------------------------------------------------------------------------------------------
// forward pieces (same rounding points and the same packed bf16 arithmetic as the fused GEMM epilogues, so the
// training forward is bit-identical to the inference forward)
// ------------------------------------------------------------------------------------------------

// zraw [M, >= 3D] (raw bf16 q | k | v of the QKV GEMM) -> qkv [M, 3D]: per-head RMSNorm(q), RMSNorm(k) over d,
// 2D RoPE from the pair-expanded chunk-major table, v copied.  One warp per (row, head slot), lane <-> pairs.
template <int DH>
__global__ void __launch_bounds__(256) qk_norm_rope_fwd_kernel(const bf16* __restrict__ zraw, long long ldz,
                                                               const bf16* __restrict__ wq, const bf16* __restrict__ wk,
                                                               const bf16* __restrict__ rope, bf16* __restrict__ qkv,
                                                               long long ldq, int M, int heads, float eps) {
  constexpr int PPL = DH / 64;   // pairs per lane
  const int lane = threadIdx.x & 31;
  const long long slots = (long long)M * 3 * heads;
  const int D = heads * DH;
  for (long long s = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); s < slots; s += (long long)gridDim.x * 8) {
    const int m = (int)(s / (3 * heads));
    const int hs = (int)(s - (long long)m * 3 * heads);
    const int seg = hs / heads, head = hs - seg * heads;
    const uint32_t* src = reinterpret_cast<const uint32_t*>(zraw + (long long)m * ldz + seg * D + head * DH);
    uint32_t* dst = reinterpret_cast<uint32_t*>(qkv + (long long)m * ldq + seg * D + head * DH);
    uint32_t t[PPL];
#pragma unroll
    for (int i = 0; i < PPL; ++i) t[i] = src[lane + 32 * i];
    if (seg == 2) {
#pragma unroll
      for (int i = 0; i < PPL; ++i) dst[lane + 32 * i] = t[i];
      continue;
    }
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < PPL; ++i) ss += bf16_lo(t[i]) * bf16_lo(t[i]) + bf16_hi(t[i]) * bf16_hi(t[i]);
    ss = warp_sum(ss);
    const float rstd = rsqrtf(ss / (float)DH + eps);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(seg == 0 ? wq : wk);
    // table: row group (m >> 5), chunk c (8 bf16 = 4 words), row-in-group (m & 31)
    const uint32_t* tw = reinterpret_cast<const uint32_t*>(rope) + ((long long)(m >> 5) * (DH >> 2)) * 128 + (m & 31) * 4;
#pragma unroll
    for (int i = 0; i < PPL; ++i) {
      const int pr = lane + 32 * i;   // pair index 0 .. DH/2-1
      const uint32_t wv = w[pr];
      const float y0 = bf16_lo(t[i]) * rstd * bf16_lo(wv), y1 = bf16_hi(t[i]) * rstd * bf16_hi(wv);
      const uint32_t Y = bf2_cvt(y0, y1);
      const uint32_t c2 = tw[(pr >> 2) * 128 + (pr & 3)];
      const uint32_t s2 = tw[(((DH >> 1) + pr) >> 2) * 128 + (pr & 3)];
      dst[pr] = bf2_add(bf2_mul(Y, c2), bf2_mul(bf2_swap(Y), s2));
    }
  }
}

// The same for any head dim d % 8 == 0, d <= 128 (pairs lane and lane + 32 of the head).  Also safe in place (zraw == qkv, ldz == ldq:
// the inference path of the head dims whose QK-norm + RoPE the QKV GEMM epilogue does not fuse): a thread reads every element it writes
// before writing it, and no other thread touches it.  nseg = 3 copies v as well, nseg = 2 (in place) leaves it.
__global__ void __launch_bounds__(256) qk_norm_rope_fwd_any_kernel(const bf16* zraw, long long ldz, const bf16* __restrict__ wq,
                                                                   const bf16* __restrict__ wk, const bf16* __restrict__ rope, bf16* qkv,
                                                                   long long ldq, int M, int heads, int d, int nseg, float eps) {
  const int lane = threadIdx.x & 31;
  const int np = d >> 1;   // pairs per head
  const long long slots = (long long)M * nseg * heads;
  const int D = heads * d;
  for (long long s = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); s < slots; s += (long long)gridDim.x * 8) {
    const int m = (int)(s / (nseg * heads));
    const int hs = (int)(s - (long long)m * nseg * heads);
    const int seg = hs / heads, head = hs - seg * heads;
    const uint32_t* src = reinterpret_cast<const uint32_t*>(zraw + (long long)m * ldz + seg * D + head * d);
    uint32_t* dst = reinterpret_cast<uint32_t*>(qkv + (long long)m * ldq + seg * D + head * d);
    uint32_t t[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) t[i] = lane + 32 * i < np ? src[lane + 32 * i] : 0u;
    if (seg == 2) {
#pragma unroll
      for (int i = 0; i < 2; ++i)
        if (lane + 32 * i < np) dst[lane + 32 * i] = t[i];
      continue;
    }
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < 2; ++i) ss += bf16_lo(t[i]) * bf16_lo(t[i]) + bf16_hi(t[i]) * bf16_hi(t[i]);
    ss = warp_sum(ss);
    const float rstd = rsqrtf(ss / (float)d + eps);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(seg == 0 ? wq : wk);
    const uint32_t* tw = reinterpret_cast<const uint32_t*>(rope) + ((long long)(m >> 5) * (d >> 2)) * 128 + (m & 31) * 4;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int pr = lane + 32 * i;
      if (pr >= np) break;
      const uint32_t wv = w[pr];
      const float y0 = bf16_lo(t[i]) * rstd * bf16_lo(wv), y1 = bf16_hi(t[i]) * rstd * bf16_hi(wv);
      const uint32_t Y = bf2_cvt(y0, y1);
      const uint32_t c2 = tw[(pr >> 2) * 128 + (pr & 3)];
      const uint32_t s2 = tw[((np + pr) >> 2) * 128 + (pr & 3)];
      dst[pr] = bf2_add(bf2_mul(Y, c2), bf2_mul(bf2_swap(Y), s2));
    }
  }
}

// zraw[:, qp:] -> act [M, Hf] = bf16(bf16(silu(g)) * v).  layout 0: 16-column groups (value16 | gate16) -- the packed
// w_in of the inference path; layout 1: [value Hf | gate Hf], fc1's own row order (training: no weight repack).
__device__ __forceinline__ void swiglu_cols(int o, int qp, int Hf, int layout, long long& voff, long long& goff) {
  if (layout == 0) { voff = qp + ((o >> 4) << 5) + (o & 8); goff = voff + 16; }
  else { voff = qp + o; goff = voff + Hf; }
}
template <typename IT>   // IT = unsigned when M * Hf / 8 < 2^32: a 32-bit division per vector instead of the 64-bit sequence
__global__ void __launch_bounds__(256) swiglu_fwd_kernel(const bf16* __restrict__ zraw, long long ldz, int qp,
                                                         bf16* __restrict__ act, long long lda, int M, int Hf, int layout) {
  const int vec_per_row = Hf >> 3;
  const IT total = (IT)M * (IT)vec_per_row;
  for (IT i = (IT)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (IT)gridDim.x * blockDim.x) {
    const int m = (int)(i / (IT)vec_per_row);
    const int o = (int)(i - (IT)m * (IT)vec_per_row) << 3;   // first of 8 output columns
    long long voff, goff;
    swiglu_cols(o, qp, Hf, layout, voff, goff);
    float v[8], g[8], r[8];
    unpack8(ld_global_nc_v4(zraw + (long long)m * ldz + voff), v);
    unpack8(ld_global_nc_v4(zraw + (long long)m * ldz + goff), g);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float s = bf16r(g[k] * (1.f / (1.f + __expf(-g[k]))));
      r[k] = s * v[k];
    }
    *reinterpret_cast<uint4*>(act + (long long)m * lda + o) = pack8(r);
  }
}

// x_out = bf16(x + bf16(y * gamma))   (in place on x allowed)
// Stochastic depth (drop_path, ae.py:15-30,65; decoder blocks in training): keep [B] holds the per-image 0/1 draw
// floor(keep_prob + U[0,1)); the LayerScale output is divided by keep_prob (rounded to bf16, x.div) and multiplied by the
// draw before it is added: x_out = x + bf16(bf16(y * gamma) / keep_prob) * keep[image].  keep == nullptr: no drop_path.
__device__ __forceinline__ uint32_t drop_scale2(uint32_t t, float inv_keep_num, float keep_prob, float kp) {
  // t = packed bf16x2 of the LayerScale output; returns bf16(t / keep_prob) * kp   (kp = 0 or 1)
  const float a = bf16r(bf16_lo(t) / keep_prob) * kp, b = bf16r(bf16_hi(t) / keep_prob) * kp;
  (void)inv_keep_num;
  return bf2_cvt(a, b);
}
__global__ void __launch_bounds__(256) resid_fwd_kernel(const bf16* __restrict__ x, const bf16* __restrict__ y,
                                                        const bf16* __restrict__ gamma, bf16* __restrict__ out, int M, int D,
                                                        const float* __restrict__ keep, int rows_per_img, float keep_prob) {
  const int vpr = D >> 3;
  const long long total = (long long)M * vpr;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % vpr) << 3;
    const uint4 xv = ld_global_v4(x + i * 8), yv = ld_global_nc_v4(y + i * 8), gv = ld_global_nc_v4(gamma + c);
    uint4 t;
    t.x = bf2_mul(yv.x, gv.x); t.y = bf2_mul(yv.y, gv.y); t.z = bf2_mul(yv.z, gv.z); t.w = bf2_mul(yv.w, gv.w);
    if (keep) {
      const float kp = __ldg(keep + (i / vpr) / rows_per_img);
      t.x = drop_scale2(t.x, 0.f, keep_prob, kp); t.y = drop_scale2(t.y, 0.f, keep_prob, kp);
      t.z = drop_scale2(t.z, 0.f, keep_prob, kp); t.w = drop_scale2(t.w, 0.f, keep_prob, kp);
    }
    uint4 o;
    o.x = bf2_add(xv.x, t.x); o.y = bf2_add(xv.y, t.y); o.z = bf2_add(xv.z, t.z); o.w = bf2_add(xv.w, t.w);
    *reinterpret_cast<uint4*>(out + i * 8) = o;
  }
}

// out = LN_noaffine(x) over C <= 256 columns (biased variance, fp32), one warp per row.  x already holds
// bf16(linear + bias).
__global__ void __launch_bounds__(256) ln_fwd_kernel(const bf16* __restrict__ x, bf16* __restrict__ out, int M, int C, float eps) {
  const int lane = threadIdx.x & 31;
  for (long long m = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); m < M; m += (long long)gridDim.x * 8) {
    float v[8];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int c = lane + 32 * k;
      v[k] = c < C ? __bfloat162float(x[m * C + c]) : 0.f;
      s += v[k];
    }
    const float mean = warp_sum(s) / (float)C;
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int c = lane + 32 * k;
      if (c < C) q += (v[k] - mean) * (v[k] - mean);
    }
    const float rstd = rsqrtf(warp_sum(q) / (float)C + eps);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int c = lane + 32 * k;
      if (c < C) out[m * C + c] = __float2bfloat16_rn((v[k] - mean) * rstd);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// backward pieces
// ------------------------------------------------------------------------------------------------

// dy = bf16(dx * gamma);  dgamma[c] += sum_rows dx * y   (fp32 atomics, one per column and block)
// block = 32 column groups (8 columns each) x 8 row lanes; grid = (ceil(D/256), row chunks)
// drop_path (keep != nullptr): the gradient of the LayerScale output is bf16(dx * keep[image] / keep_prob) (autograd of x.div and
// of the multiplication by the draw); dy and dgamma follow from it.
__global__ void __launch_bounds__(256) resid_bwd_kernel(const bf16* __restrict__ dx, const bf16* __restrict__ y,
                                                        const bf16* __restrict__ gamma, bf16* __restrict__ dy,
                                                        float* __restrict__ dgamma, int M, int D, const float* __restrict__ keep,
                                                        int rows_per_img, float keep_prob) {
  __shared__ float red[8][256 + 8];
  const int cg = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c = blockIdx.x * 256 + cg * 8;
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (c < D) {
    float g[8];
    unpack8(ld_global_nc_v4(gamma + c), g);
    for (long long m = (long long)blockIdx.y * 8 + rl; m < M; m += (long long)gridDim.y * 8) {
      float a[8], b[8], o[8];
      unpack8(ld_global_nc_v4(dx + m * D + c), a);
      unpack8(ld_global_nc_v4(y + m * D + c), b);
      if (keep) {
        const float kp = __ldg(keep + m / rows_per_img);
#pragma unroll
        for (int k = 0; k < 8; ++k) a[k] = bf16r(a[k] * kp / keep_prob);
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        acc[k] += a[k] * b[k];
        o[k] = a[k] * g[k];
      }
      *reinterpret_cast<uint4*>(dy + m * D + c) = pack8(o);
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) red[rl][cg * 8 + k] = acc[k];
  __syncthreads();
  const int col = threadIdx.x;
  float s = 0.f;
#pragma unroll
  for (int r = 0; r < 8; ++r) s += red[r][col];
  if (blockIdx.x * 256 + col < D) atomicAdd(&dgamma[blockIdx.x * 256 + col], s);
}

// plain column sums: out[c] += sum_rows in[r, c]   (bias gradients)
__global__ void __launch_bounds__(256) colsum_kernel(const bf16* __restrict__ in, long long ld, float* __restrict__ out, int M, int C) {
  __shared__ float red[8][256 + 8];
  const int cg = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c = blockIdx.x * 256 + cg * 8;
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (c < C) {
    for (long long m = (long long)blockIdx.y * 8 + rl; m < M; m += (long long)gridDim.y * 8) {
      float a[8];
      unpack8(ld_global_nc_v4(in + m * ld + c), a);
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] += a[k];
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) red[rl][cg * 8 + k] = acc[k];
  __syncthreads();
  const int col = threadIdx.x;
  float s = 0.f;
#pragma unroll
  for (int r = 0; r < 8; ++r) s += red[r][col];
  if (blockIdx.x * 256 + col < C) atomicAdd(&out[blockIdx.x * 256 + col], s);
}

// SwiGLU backward: d_act [M, Hf] (row stride ldd), zraw (value16 | gate16 groups at column qp) ->
// dz[:, qp:] in the same packed order:  d_val = d_act * silu(g),  d_gate = d_act * val * sig(g) * (1 + g * (1 - sig(g)))
template <typename IT>
__global__ void __launch_bounds__(256) swiglu_bwd_kernel(const bf16* __restrict__ dact, long long ldd,
                                                         const bf16* __restrict__ zraw, long long ldz, int qp,
                                                         bf16* __restrict__ dz, long long lddz, int M, int Hf, int layout) {
  const int vec_per_row = Hf >> 3;
  const IT total = (IT)M * (IT)vec_per_row;
  for (IT i = (IT)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (IT)gridDim.x * blockDim.x) {
    const int m = (int)(i / (IT)vec_per_row);
    const int o = (int)(i - (IT)m * (IT)vec_per_row) << 3;
    long long zoff, goff;
    swiglu_cols(o, qp, Hf, layout, zoff, goff);
    float v[8], g[8], d[8], dv[8], dg[8];
    unpack8(ld_global_nc_v4(zraw + (long long)m * ldz + zoff), v);
    unpack8(ld_global_nc_v4(zraw + (long long)m * ldz + goff), g);
    unpack8(ld_global_nc_v4(dact + (long long)m * ldd + o), d);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float sg = 1.f / (1.f + __expf(-g[k]));
      dv[k] = d[k] * (g[k] * sg);
      dg[k] = d[k] * v[k] * sg * (1.f + g[k] * (1.f - sg));
    }
    *reinterpret_cast<uint4*>(dz + (long long)m * lddz + zoff) = pack8(dv);
    *reinterpret_cast<uint4*>(dz + (long long)m * lddz + goff) = pack8(dg);
  }
}

// QK-norm + RoPE backward, in place on dz[:, 0:2D] (which holds dq | dk w.r.t. the roped, normed q/k):
//   un-rotate:  g = R^T dq           (pair i: g0 = c*d0 + s*d1, g1 = -s*d0 + c*d1)
//   RMSNorm:    xh = x * rstd, gw = g * w,  dx = rstd * (gw - xh * mean(gw * xh)),  dw += g * xh
// One warp per (row, q-or-k head); the lane <-> pair mapping is fixed, so dw accumulates in registers and is
// reduced once per block (shared memory) and once per grid (fp32 atomics).  dw = [2][DH] (q then k).
template <int DH>
__global__ void __launch_bounds__(256) qk_norm_rope_bwd_kernel(bf16* __restrict__ dz, long long lddz,
                                                               const bf16* __restrict__ zraw, long long ldz,
                                                               const bf16* __restrict__ wq, const bf16* __restrict__ wk,
                                                               const bf16* __restrict__ rope, float* __restrict__ dw,
                                                               int M, int heads, float eps) {
  constexpr int PPL = DH / 64;
  __shared__ float red[8][2][DH];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int D = heads * DH;
  float acc[2][PPL][2];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int i = 0; i < PPL; ++i) acc[a][i][0] = acc[a][i][1] = 0.f;
  const long long slots = (long long)M * 2 * heads;
  for (long long s = (long long)blockIdx.x * 8 + warp; s < slots; s += (long long)gridDim.x * 8) {
    const int m = (int)(s / (2 * heads));
    const int hs = (int)(s - (long long)m * 2 * heads);
    const int seg = hs / heads, head = hs - seg * heads;
    const uint32_t* xs = reinterpret_cast<const uint32_t*>(zraw + (long long)m * ldz + seg * D + head * DH);
    uint32_t* dp = reinterpret_cast<uint32_t*>(dz + (long long)m * lddz + seg * D + head * DH);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(seg == 0 ? wq : wk);
    const uint32_t* tw = reinterpret_cast<const uint32_t*>(rope) + ((long long)(m >> 5) * (DH >> 2)) * 128 + (m & 31) * 4;
    float x0[PPL], x1[PPL], g0[PPL], g1[PPL];
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < PPL; ++i) {
      const int pr = lane + 32 * i;
      const uint32_t xv = xs[pr], dv = dp[pr];
      x0[i] = bf16_lo(xv); x1[i] = bf16_hi(xv);
      ss += x0[i] * x0[i] + x1[i] * x1[i];
      const uint32_t c2 = tw[(pr >> 2) * 128 + (pr & 3)];
      const uint32_t s2 = tw[(((DH >> 1) + pr) >> 2) * 128 + (pr & 3)];
      const float c = bf16_lo(c2), sn = bf16_hi(s2);   // C2 = (c, c), S2 = (-s, +s)
      const float d0 = bf16_lo(dv), d1 = bf16_hi(dv);
      g0[i] = c * d0 + sn * d1;
      g1[i] = -sn * d0 + c * d1;
    }
    ss = warp_sum(ss);
    const float rstd = rsqrtf(ss / (float)DH + eps);
    float dot = 0.f;
    float gw0[PPL], gw1[PPL];
#pragma unroll
    for (int i = 0; i < PPL; ++i) {
      const int pr = lane + 32 * i;
      const uint32_t wv = w[pr];
      x0[i] *= rstd; x1[i] *= rstd;                       // xh
      const float isq = seg == 0 ? 1.f : 0.f;             // (no dynamic indexing of the register accumulators)
      acc[0][i][0] += isq * g0[i] * x0[i];
      acc[0][i][1] += isq * g1[i] * x1[i];
      acc[1][i][0] += (1.f - isq) * g0[i] * x0[i];
      acc[1][i][1] += (1.f - isq) * g1[i] * x1[i];
      gw0[i] = g0[i] * bf16_lo(wv); gw1[i] = g1[i] * bf16_hi(wv);
      dot += gw0[i] * x0[i] + gw1[i] * x1[i];
    }
    dot = warp_sum(dot) / (float)DH;
#pragma unroll
    for (int i = 0; i < PPL; ++i)
      dp[lane + 32 * i] = bf2_cvt(rstd * (gw0[i] - x0[i] * dot), rstd * (gw1[i] - x1[i] * dot));
  }
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int i = 0; i < PPL; ++i) {
      red[warp][a][2 * (lane + 32 * i)] = acc[a][i][0];
      red[warp][a][2 * (lane + 32 * i) + 1] = acc[a][i][1];
    }
  __syncthreads();
  for (int e = threadIdx.x; e < 2 * DH; e += blockDim.x) {
    float s = 0.f;
#pragma unroll
    for (int wp = 0; wp < 8; ++wp) s += red[wp][e / DH][e % DH];
    atomicAdd(&dw[e], s);
  }
}

// The same for any head dim d % 8 == 0, d <= 128 (pairs lane and lane + 32 of the head).  dw = [2][d].
__global__ void __launch_bounds__(256) qk_norm_rope_bwd_any_kernel(bf16* __restrict__ dz, long long lddz, const bf16* __restrict__ zraw,
                                                                   long long ldz, const bf16* __restrict__ wq, const bf16* __restrict__ wk,
                                                                   const bf16* __restrict__ rope, float* __restrict__ dw, int M, int heads,
                                                                   int d, float eps) {
  __shared__ float red[8][2][128];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int np = d >> 1;
  const int D = heads * d;
  float acc[2][2][2];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int i = 0; i < 2; ++i) acc[a][i][0] = acc[a][i][1] = 0.f;
  const long long slots = (long long)M * 2 * heads;
  for (long long s = (long long)blockIdx.x * 8 + warp; s < slots; s += (long long)gridDim.x * 8) {
    const int m = (int)(s / (2 * heads));
    const int hs = (int)(s - (long long)m * 2 * heads);
    const int seg = hs / heads, head = hs - seg * heads;
    const uint32_t* xs = reinterpret_cast<const uint32_t*>(zraw + (long long)m * ldz + seg * D + head * d);
    uint32_t* dp = reinterpret_cast<uint32_t*>(dz + (long long)m * lddz + seg * D + head * d);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(seg == 0 ? wq : wk);
    const uint32_t* tw = reinterpret_cast<const uint32_t*>(rope) + ((long long)(m >> 5) * (d >> 2)) * 128 + (m & 31) * 4;
    float x0[2], x1[2], g0[2], g1[2];
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int pr = lane + 32 * i;
      x0[i] = x1[i] = g0[i] = g1[i] = 0.f;
      if (pr < np) {
        const uint32_t xv = xs[pr], dv = dp[pr];
        x0[i] = bf16_lo(xv); x1[i] = bf16_hi(xv);
        const uint32_t c2 = tw[(pr >> 2) * 128 + (pr & 3)];
        const uint32_t s2 = tw[((np + pr) >> 2) * 128 + (pr & 3)];
        const float c = bf16_lo(c2), sn = bf16_hi(s2);   // C2 = (c, c), S2 = (-s, +s)
        const float d0 = bf16_lo(dv), d1 = bf16_hi(dv);
        g0[i] = c * d0 + sn * d1;
        g1[i] = -sn * d0 + c * d1;
      }
      ss += x0[i] * x0[i] + x1[i] * x1[i];
    }
    ss = warp_sum(ss);
    const float rstd = rsqrtf(ss / (float)d + eps);
    float dot = 0.f;
    float gw0[2], gw1[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int pr = lane + 32 * i;
      const uint32_t wv = pr < np ? w[pr] : 0u;
      x0[i] *= rstd; x1[i] *= rstd;                       // xh
      const float isq = seg == 0 ? 1.f : 0.f;             // (no dynamic indexing of the register accumulators)
      acc[0][i][0] += isq * g0[i] * x0[i];
      acc[0][i][1] += isq * g1[i] * x1[i];
      acc[1][i][0] += (1.f - isq) * g0[i] * x0[i];
      acc[1][i][1] += (1.f - isq) * g1[i] * x1[i];
      gw0[i] = g0[i] * bf16_lo(wv); gw1[i] = g1[i] * bf16_hi(wv);
      dot += gw0[i] * x0[i] + gw1[i] * x1[i];
    }
    dot = warp_sum(dot) / (float)d;
#pragma unroll
    for (int i = 0; i < 2; ++i)
      if (lane + 32 * i < np) dp[lane + 32 * i] = bf2_cvt(rstd * (gw0[i] - x0[i] * dot), rstd * (gw1[i] - x1[i] * dot));
  }
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      red[warp][a][2 * (lane + 32 * i)] = acc[a][i][0];
      red[warp][a][2 * (lane + 32 * i) + 1] = acc[a][i][1];
    }
  __syncthreads();
  for (int e = threadIdx.x; e < 2 * d; e += blockDim.x) {
    float sum = 0.f;
#pragma unroll
    for (int wp = 0; wp < 8; ++wp) sum += red[wp][e / d][e % d];
    atomicAdd(&dw[e], sum);
  }
}

// RMSNorm backward (norm1), one warp per row:  xh = x * rstd, gw = dh * w,
//   dx_out = dx_res + rstd * (gw - xh * mean(gw * xh))   (dx_res = gradient arriving through the residual path)
//   dw[c] += dh * xh.   Columns are lane-strided in 16-byte vectors, so each thread owns fixed columns.
template <int NV>
__global__ void __launch_bounds__(256) rmsnorm_bwd_kernel(const bf16* __restrict__ x, const bf16* __restrict__ dh,
                                                          const bf16* __restrict__ w, const bf16* __restrict__ dx_res,
                                                          bf16* __restrict__ dx_out, float* __restrict__ dw, int M, int D,
                                                          float eps) {
  extern __shared__ float red[];   // [8][D]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nvec = D >> 3;
  float acc[NV][8];
#pragma unroll
  for (int i = 0; i < NV; ++i)
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[i][k] = 0.f;
  for (long long m = (long long)blockIdx.x * 8 + warp; m < M; m += (long long)gridDim.x * 8) {
    // three passes over the row (the re-reads hit L1/L2); only the dw accumulators live across rows
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int v = lane + 32 * i;
      if (v < nvec) {
        float xv[8];
        unpack8(ld_global_nc_v4(x + m * D + 8 * v), xv);
#pragma unroll
        for (int k = 0; k < 8; ++k) ss += xv[k] * xv[k];
      }
    }
    ss = warp_sum(ss);
    const float rstd = rsqrtf(ss / (float)D + eps);
    float dot = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int v = lane + 32 * i;
      if (v < nvec) {
        float xv[8], d[8], wv[8];
        unpack8(ld_global_nc_v4(x + m * D + 8 * v), xv);
        unpack8(ld_global_nc_v4(dh + m * D + 8 * v), d);
        unpack8(ld_global_nc_v4(w + 8 * v), wv);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float xh = xv[k] * rstd;
          acc[i][k] += d[k] * xh;
          dot += d[k] * wv[k] * xh;
        }
      }
    }
    dot = warp_sum(dot) / (float)D;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int v = lane + 32 * i;
      if (v < nvec) {
        float xv[8], d[8], wv[8], r[8], o[8];
        unpack8(ld_global_nc_v4(x + m * D + 8 * v), xv);
        unpack8(ld_global_nc_v4(dh + m * D + 8 * v), d);
        unpack8(ld_global_nc_v4(w + 8 * v), wv);
        unpack8(ld_global_v4(dx_res + m * D + 8 * v), r);
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] = r[k] + rstd * (d[k] * wv[k] - xv[k] * rstd * dot);
        *reinterpret_cast<uint4*>(dx_out + m * D + 8 * v) = pack8(o);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int v = lane + 32 * i;
    if (v < nvec)
#pragma unroll
      for (int k = 0; k < 8; ++k) red[warp * D + 8 * v + k] = acc[i][k];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < D; c += blockDim.x) {
    float s = 0.f;
#pragma unroll
    for (int wp = 0; wp < 8; ++wp) s += red[wp * D + c];
    atomicAdd(&dw[c], s);
  }
}

// LayerNorm (no affine) backward over C <= 256 columns, one warp per row.  zlin = bf16(linear + bias) is the
// saved input: dx = rstd * (dz - mean(dz) - zh * mean(dz * zh)),  zh = (zlin - mean) * rstd
__global__ void __launch_bounds__(256) ln_bwd_kernel(const bf16* __restrict__ zlin, const bf16* __restrict__ dz,
                                                     bf16* __restrict__ dx, int M, int C, float eps) {
  const int lane = threadIdx.x & 31;
  for (long long m = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); m < M; m += (long long)gridDim.x * 8) {
    float v[8], g[8];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int c = lane + 32 * k;
      v[k] = c < C ? __bfloat162float(zlin[m * C + c]) : 0.f;
      g[k] = c < C ? __bfloat162float(dz[m * C + c]) : 0.f;
      s += v[k];
    }
    const float mean = warp_sum(s) / (float)C;
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int c = lane + 32 * k;
      if (c < C) q += (v[k] - mean) * (v[k] - mean);
    }
    const float rstd = rsqrtf(warp_sum(q) / (float)C + eps);
    float sg = 0.f, sgz = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int c = lane + 32 * k;
      v[k] = c < C ? (v[k] - mean) * rstd : 0.f;
      sg += g[k];
      sgz += g[k] * v[k];
    }
    sg = warp_sum(sg) / (float)C;
    sgz = warp_sum(sgz) / (float)C;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int c = lane + 32 * k;
      if (c < C) dx[m * C + c] = __float2bfloat16_rn(rstd * (g[k] - sg - v[k] * sgz));
    }
  }
}

// Charbonnier loss (scripts/train_vae.py:314-320): per token mean over P of sqrt(diff^2 + eps^2) with
// diff = float(pred) - float(target); per image mean over its valid tokens; batch mean.
//   loss_sum[b] += per-token means of image b (fp32 atomics);  n_valid[b] is computed by the caller
//   dpred = diff / sqrt(diff^2 + eps^2) / (P * n_valid[b] * B) on valid tokens, 0 elsewhere.
// One warp per token.
__global__ void __launch_bounds__(256) charbonnier_kernel(const bf16* __restrict__ pred, const bf16* __restrict__ target,
                                                          const uint8_t* __restrict__ mask, const int* __restrict__ n_valid,
                                                          float* __restrict__ loss_sum, bf16* __restrict__ dpred, int B, int N,
                                                          int P, float eps) {
  const int lane = threadIdx.x & 31;
  const int nvec = P >> 3;
  const long long tokens = (long long)B * N;
  for (long long tk = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); tk < tokens; tk += (long long)gridDim.x * 8) {
    const int b = (int)(tk / N);
    const bool valid = mask == nullptr || mask[tk] != 0;
    const int nv = mask == nullptr ? N : n_valid[b];
    const float gscale = valid && nv > 0 ? 1.f / ((float)P * (float)nv * (float)B) : 0.f;
    float s = 0.f;
    for (int v = lane; v < nvec; v += 32) {
      float a[8], t[8], g[8];
      unpack8(ld_global_nc_v4(pred + tk * P + 8 * v), a);
      unpack8(ld_global_nc_v4(target + tk * P + 8 * v), t);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float d = a[k] - t[k];
        const float r = sqrtf(d * d + eps * eps);
        s += r;
        g[k] = d / r * gscale;
      }
      if (dpred) *reinterpret_cast<uint4*>(dpred + tk * P + 8 * v) = pack8(g);
    }
    s = warp_sum(s);
    if (lane == 0 && valid && nv > 0) atomicAdd(&loss_sum[b], s / (float)P / (float)nv);
  }
}

// one AdamW element update in fp32 (torch.optim.AdamW semantics):
//   p *= 1 - lr * wd;  m = b1 m + (1 - b1) g;  v = b2 v + (1 - b2) g^2;  p -= lr / bc1 * m / (sqrt(v) / sqrt(bc2) + eps)
__device__ __forceinline__ void adamw_one(float& pf, float gf, float& mf, float& vf, float lr, float b1, float b2, float eps,
                                          float wd, float bc1, float bc2_sqrt) {
  pf *= 1.f - lr * wd;
  mf = b1 * mf + (1.f - b1) * gf;
  vf = b2 * vf + (1.f - b2) * gf * gf;
  const float denom = sqrtf(vf) / bc2_sqrt + eps;
  pf -= (lr / bc1) * (mf / denom);
}

// ema + w (master - ema) with torch.lerp's formula (ATen/native/Lerp.h), the fp32 arithmetic torch._foreach_lerp_(ema, master, w)
// runs: the two branches keep the result exact at w = 0 and w = 1
__device__ __forceinline__ float ema_lerp(float e, float m, float w) {
  return fabsf(w) < 0.5f ? e + w * (m - e) : m - (m - e) * (1.f - w);
}

// ------------------------------------------------------------------------------------------------
// Multi-tensor AdamW with the reference's optimizer precision (scripts/train_vae.py:200-208 keeps fp32 parameters and fp32
// Adam moments under autocast): per tensor an fp32 MASTER copy of the parameter and fp32 exp_avg / exp_avg_sq are updated
// in fp32 and the bf16 model parameter is re-emitted from the master in the same pass -- an update smaller than half a bf16
// ulp of the weight is therefore not lost (it accumulates in the master).  fp32 model parameters are their own master
// (p16 == nullptr).  Up to ADAMW_MAX_T tensors per launch travel in the kernel parameters; work is cut into chunks of
// ADAMW_CHUNK elements and dealt to the blocks round-robin, so one launch covers tensors of any size mix.
//   kClip: every gradient is multiplied by *coef (device memory: the clip coefficient of grad_norm_finish_kernel) after
//          grad_scale; coef == 1 leaves the step bit-identical to the unclipped one.
//   kEma:  the fp32 EMA of the master follows the new master value in the same pass, ema = lerp(ema, master, ema_w).
// HBM traffic per parameter: 4 + 4 + 4 (master, m, v) + 2 (bf16 grad) read, 4 + 4 + 4 + 2 written = 28 bytes; kEma adds the
// EMA's 4 read + 4 written = 36 bytes; kClip adds nothing here (one coefficient per launch).
// ------------------------------------------------------------------------------------------------
static constexpr int ADAMW_MAX_T = 64;
static constexpr int ADAMW_CHUNK = 8192;   // elements per (block, iteration): 256 threads x 4 vectors of 8
struct AdamwBatch {
  float* master[ADAMW_MAX_T];
  bf16* p16[ADAMW_MAX_T];
  const void* g[ADAMW_MAX_T];
  float* m[ADAMW_MAX_T];
  float* v[ADAMW_MAX_T];
  long long n[ADAMW_MAX_T];
  int chunk0[ADAMW_MAX_T + 1];   // first global chunk of every tensor
  float wd[ADAMW_MAX_T];
  unsigned char g_f32[ADAMW_MAX_T];
  int nt;
};
struct AdamwEmaBatch : AdamwBatch {
  float* ema[ADAMW_MAX_T];
};
template <bool kEma>
using AdamwBatchT = typename std::conditional<kEma, AdamwEmaBatch, AdamwBatch>::type;

// tensor of global chunk ch: binary search in chunk0 (nt <= 64)
__device__ __forceinline__ int chunk_tensor(const AdamwBatch& b, int ch) {
  int lo = 0, hi = b.nt;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (b.chunk0[mid] <= ch) lo = mid; else hi = mid;
  }
  return lo;
}

// gradient as the update sees it: times the host scale, then (clipping) times the device coefficient
template <bool kClip>
__device__ __forceinline__ float scaled(float grad_scale, float coef, float g) {
  float x = g * grad_scale;
  if constexpr (kClip) x *= coef;
  return x;
}

template <bool kClip, bool kEma>
__global__ void __launch_bounds__(256) adamw_multi_kernel(const __grid_constant__ AdamwBatchT<kEma> b, float lr, float b1, float b2,
                                                          float eps, float bc1, float bc2_sqrt, float grad_scale,
                                                          const float* __restrict__ coef, float ema_w) {
  const int total = b.chunk0[b.nt];
  float cf = 1.f;
  if constexpr (kClip) cf = __ldg(coef);
  for (int ch = blockIdx.x; ch < total; ch += gridDim.x) {
    const int t = chunk_tensor(b, ch);
    const long long e0 = (long long)(ch - b.chunk0[t]) * ADAMW_CHUNK;
    const long long n = b.n[t];
    const long long e1 = e0 + ADAMW_CHUNK < n ? e0 + ADAMW_CHUNK : n;
    float* __restrict__ mp = b.master[t];
    bf16* __restrict__ pp = b.p16[t];
    float* __restrict__ mm = b.m[t];
    float* __restrict__ vv = b.v[t];
    float* __restrict__ ee = nullptr;
    if constexpr (kEma) ee = b.ema[t];
    const float wd = b.wd[t];
    const bool gf32 = b.g_f32[t] != 0;
    const bool vec = ((reinterpret_cast<uintptr_t>(mp) | reinterpret_cast<uintptr_t>(mm) | reinterpret_cast<uintptr_t>(vv) |
                       reinterpret_cast<uintptr_t>(b.g[t]) | reinterpret_cast<uintptr_t>(ee)) & 15) == 0 &&
                     (pp == nullptr || (reinterpret_cast<uintptr_t>(pp) & 7) == 0);
    long long i = e0 + 4 * (long long)threadIdx.x;
    if (vec) {
      for (; i + 3 < e1; i += 4 * 256) {   // 4 elements per thread and iteration: 16-byte fp32 vectors, 8-byte bf16 vectors
        float4 pf = *reinterpret_cast<const float4*>(mp + i), mf = *reinterpret_cast<const float4*>(mm + i), vf = *reinterpret_cast<const float4*>(vv + i);
        float g4[4];
        if (gf32) {
          const float4 q = __ldg(reinterpret_cast<const float4*>(static_cast<const float*>(b.g[t]) + i));
          g4[0] = q.x; g4[1] = q.y; g4[2] = q.z; g4[3] = q.w;
        } else {
          const uint2 q = __ldg(reinterpret_cast<const uint2*>(static_cast<const bf16*>(b.g[t]) + i));
          g4[0] = bf16_lo(q.x); g4[1] = bf16_hi(q.x); g4[2] = bf16_lo(q.y); g4[3] = bf16_hi(q.y);
        }
        adamw_one(pf.x, scaled<kClip>(grad_scale, cf, g4[0]), mf.x, vf.x, lr, b1, b2, eps, wd, bc1, bc2_sqrt);
        adamw_one(pf.y, scaled<kClip>(grad_scale, cf, g4[1]), mf.y, vf.y, lr, b1, b2, eps, wd, bc1, bc2_sqrt);
        adamw_one(pf.z, scaled<kClip>(grad_scale, cf, g4[2]), mf.z, vf.z, lr, b1, b2, eps, wd, bc1, bc2_sqrt);
        adamw_one(pf.w, scaled<kClip>(grad_scale, cf, g4[3]), mf.w, vf.w, lr, b1, b2, eps, wd, bc1, bc2_sqrt);
        *reinterpret_cast<float4*>(mp + i) = pf;
        *reinterpret_cast<float4*>(mm + i) = mf;
        *reinterpret_cast<float4*>(vv + i) = vf;
        if (pp) *reinterpret_cast<uint2*>(pp + i) = make_uint2(bf2_cvt(pf.x, pf.y), bf2_cvt(pf.z, pf.w));
        if constexpr (kEma) {
          float4 ef = *reinterpret_cast<const float4*>(ee + i);
          ef.x = ema_lerp(ef.x, pf.x, ema_w); ef.y = ema_lerp(ef.y, pf.y, ema_w);
          ef.z = ema_lerp(ef.z, pf.z, ema_w); ef.w = ema_lerp(ef.w, pf.w, ema_w);
          *reinterpret_cast<float4*>(ee + i) = ef;
        }
      }
      // tail of the chunk (n % 4 elements of the last chunk)
      i = e0 + ((e1 - e0) & ~3LL) + threadIdx.x;
    } else {
      i = e0 + threadIdx.x;
    }
    for (; i < e1; i += vec ? 256 * 1024 : 256) {
      float pf = mp[i], mf = mm[i], vf = vv[i];
      const float gf = scaled<kClip>(grad_scale, cf, gf32 ? static_cast<const float*>(b.g[t])[i] : __bfloat162float(static_cast<const bf16*>(b.g[t])[i]));
      adamw_one(pf, gf, mf, vf, lr, b1, b2, eps, wd, bc1, bc2_sqrt);
      mp[i] = pf; mm[i] = mf; vv[i] = vf;
      if (pp) pp[i] = __float2bfloat16_rn(pf);
      if constexpr (kEma) ee[i] = ema_lerp(ee[i], pf, ema_w);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Global L2 gradient norm for clipping (torch.nn.utils.clip_grad_norm_), deterministic: grad_sumsq_kernel writes one fp32 sum of
// squares per ADAMW_CHUNK chunk to its own slot (thread-sequential, then a fixed shuffle tree: no atomics), and the one-CTA
// grad_norm_finish_kernel adds the slots in a fixed order in fp64.  A chunk's partial depends only on that chunk's gradient values,
// and its slot only on its position in the tensor table, so the norm does not depend on how the table is cut into launches.
// HBM traffic per parameter: the gradient read once, 2 bytes (bf16) or 4 (fp32).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) grad_sumsq_kernel(const __grid_constant__ AdamwBatch b, float* __restrict__ partials) {
  __shared__ float red[8];
  const int total = b.chunk0[b.nt];
  for (int ch = blockIdx.x; ch < total; ch += gridDim.x) {
    const int t = chunk_tensor(b, ch);
    const long long e0 = (long long)(ch - b.chunk0[t]) * ADAMW_CHUNK;
    const long long n = b.n[t];
    const long long e1 = e0 + ADAMW_CHUNK < n ? e0 + ADAMW_CHUNK : n;
    const bool gf32 = b.g_f32[t] != 0;
    const char* gp = static_cast<const char*>(b.g[t]);
    const int esz = gf32 ? 4 : 2;
    float s = 0.f;
    long long i = e0 + threadIdx.x;
    if ((reinterpret_cast<uintptr_t>(gp) & 15) == 0) {   // 16-byte loads: 8 bf16 or 4 fp32 values; 32 values per thread and chunk
      const int per = 16 / esz;
      const long long nvec = (e1 - e0) / per;
      for (long long v = threadIdx.x; v < nvec; v += 256) {
        const uint4 q = ld_global_nc_v4(gp + (e0 + v * per) * esz);
        if (gf32) {
          const float f0 = __uint_as_float(q.x), f1 = __uint_as_float(q.y), f2 = __uint_as_float(q.z), f3 = __uint_as_float(q.w);
          s = fmaf(f0, f0, s); s = fmaf(f1, f1, s); s = fmaf(f2, f2, s); s = fmaf(f3, f3, s);
        } else {
          float f[8];
          unpack8(q, f);
#pragma unroll
          for (int k = 0; k < 8; ++k) s = fmaf(f[k], f[k], s);
        }
      }
      i = e0 + nvec * per + threadIdx.x;                 // the last chunk's n % per values
    }
    for (; i < e1; i += 256) {
      const float x = gf32 ? reinterpret_cast<const float*>(gp)[i] : __bfloat162float(reinterpret_cast<const bf16*>(gp)[i]);
      s = fmaf(x, x, s);
    }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
      float r = threadIdx.x < 8 ? red[threadIdx.x] : 0.f;
      r = warp_sum(r);
      if (threadIdx.x == 0) partials[ch] = r;
    }
    __syncthreads();
  }
}

// norm_coef[0] = sqrt(sum of the partials), norm_coef[1] = clamp(max_norm / (norm + 1e-6), max = 1) -- evaluated as torch evaluates
// it for an fp32 norm (Tensor.__rtruediv__: reciprocal, then times max_norm; clamp keeps NaN), so inf and NaN norms give torch's
// coefficient (an inf norm: 0; a NaN norm: NaN).
__global__ void __launch_bounds__(256) grad_norm_finish_kernel(const float* __restrict__ partials, long long n_slots, float max_norm,
                                                               float* __restrict__ norm_coef) {
  __shared__ double red[256];
  double s = 0.0;
  for (long long i = threadIdx.x; i < n_slots; i += 256) s += (double)partials[i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const float norm = (float)sqrt(red[0]);
    const float c = (1.f / (norm + 1e-6f)) * max_norm;
    norm_coef[0] = norm;
    norm_coef[1] = c > 1.f ? 1.f : c;
  }
}

// x *= *scale (bf16 tensor, fp32 device scalar): the Charbonnier gradient times the incoming loss gradient
__global__ void __launch_bounds__(256) scale_by_dev_kernel(bf16* __restrict__ x, const float* __restrict__ scale, long long n) {
  const float s = __ldg(scale);
  if (s == 1.f) return;
  const long long nvec = n >> 3, stride = (long long)gridDim.x * blockDim.x, tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (long long i = tid; i < nvec; i += stride) {
    float f[8];
    unpack8(ld_global_v4(x + 8 * i), f);
#pragma unroll
    for (int k = 0; k < 8; ++k) f[k] *= s;
    *reinterpret_cast<uint4*>(x + 8 * i) = pack8(f);
  }
  for (long long i = (nvec << 3) + tid; i < n; i += stride) x[i] = __float2bfloat16_rn(__bfloat162float(x[i]) * s);
}

// per attention row and head: delta = sum_d dO * O   (the softmax-backward row term), fp32 [M, heads]; lane <-> pairs lane, lane + 32
__global__ void __launch_bounds__(256) attn_delta_kernel(const bf16* __restrict__ o, long long ldo, const bf16* __restrict__ dob,
                                                         long long lddo, float* __restrict__ delta, int M, int heads, int d) {
  const int lane = threadIdx.x & 31;
  const long long slots = (long long)M * heads;
  for (long long s = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); s < slots; s += (long long)gridDim.x * 8) {
    const long long m = s / heads;
    const int head = (int)(s - m * heads);
    const uint32_t* a = reinterpret_cast<const uint32_t*>(o + m * ldo + head * d);
    const uint32_t* b = reinterpret_cast<const uint32_t*>(dob + m * lddo + head * d);
    float acc = 0.f;
    for (int pr = lane; pr < (d >> 1); pr += 32) {
      const uint32_t x = a[pr], y = b[pr];
      acc += bf16_lo(x) * bf16_lo(y) + bf16_hi(x) * bf16_hi(y);
    }
    acc = warp_sum(acc);
    if (lane == 0) delta[s] = acc;
  }
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// round 2: 16-byte versions of the three kernels that sat furthest below the HBM roofline in the 5B step
// (torch.profiler, 44 blocks: qk_norm_rope_fwd 132 us, qk_norm_rope_bwd 177 us, rmsnorm_bwd 207 us per launch for
// 302 / 300 / 200 MB, i.e. 2.3 / 1.7 / 1.0 TB/s).  The versions above moved 4 bytes per lane and instruction with a
// warp-wide reduction per 256 bytes (qk), or re-read every row three times with 128 accumulator registers (rmsnorm).
// ------------------------------------------------------------------------------------------------

// sum over the LPH (8 or 16) consecutive lanes that share a head
template <int LPH>
static __device__ __forceinline__ float head_sum(float v) {
#pragma unroll
  for (int o = LPH / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// RoPE table chunks of row m for the lane's 8 columns (chunk j of C2, chunk DH/8 + j of S2); layout: vtk_gemm.cu rope_row_ptr
template <int DH>
static __device__ __forceinline__ void rope_chunks(const bf16* rope, int m, int j, uint4& c2, uint4& s2) {
  const uint4* t = reinterpret_cast<const uint4*>(rope) + ((long long)(m >> 5) * (DH >> 2)) * 32 + (m & 31);
  c2 = ld_global_nc_v4(reinterpret_cast<const bf16*>(t + j * 32));
  s2 = ld_global_nc_v4(reinterpret_cast<const bf16*>(t + ((DH >> 3) + j) * 32));
}

// Forward: a lane owns 8 consecutive columns (4 RoPE pairs) of one head, LPH = DH / 8 lanes share a head, a warp covers 256 consecutive
// columns of [q | k | v] per pass (heads % (32 / LPH) == 0, so a pass never straddles q / k / v) and UN passes are in flight.
template <int DH, int UN>
__global__ void __launch_bounds__(256) qk_norm_rope_fwd16_kernel(const bf16* __restrict__ zraw, long long ldz,
                                                                 const bf16* __restrict__ wq, const bf16* __restrict__ wk,
                                                                 const bf16* __restrict__ rope, bf16* __restrict__ qkv,
                                                                 long long ldq, int M, int heads, float eps) {
  constexpr int LPH = DH / 8, HPW = 32 / LPH;
  const int lane = threadIdx.x & 31, sub = lane / LPH, j = lane - sub * LPH;
  const unsigned upr = (unsigned)(3 * heads / HPW);                 // 256-column units per row
  const unsigned total = (unsigned)M * upr;
  const unsigned nwarps = gridDim.x * 8u;
  float wqf[8], wkf[8];
  unpack8(ld_global_nc_v4(wq + 8 * j), wqf);
  unpack8(ld_global_nc_v4(wk + 8 * j), wkf);
  for (unsigned u0 = (blockIdx.x * 8u + (threadIdx.x >> 5)) * UN; u0 < total; u0 += nwarps * UN) {
    uint4 t[UN];
    int mrow[UN], g[UN];
#pragma unroll
    for (int k = 0; k < UN; ++k) {
      const unsigned u = u0 + k;
      t[k] = make_uint4(0u, 0u, 0u, 0u);
      mrow[k] = -1;
      if (u < total) {
        mrow[k] = (int)(u / upr);
        g[k] = (int)(u - (unsigned)mrow[k] * upr);
        t[k] = ld_global_nc_v4(zraw + (long long)mrow[k] * ldz + g[k] * 256 + lane * 8);
      }
    }
#pragma unroll
    for (int k = 0; k < UN; ++k) {
      if (mrow[k] < 0) continue;
      const int m = mrow[k];
      bf16* dst = qkv + (long long)m * ldq + g[k] * 256 + lane * 8;
      const int seg = (g[k] * HPW) / heads;                         // warp-uniform
      if (seg == 2) {                                               // v: copy
        *reinterpret_cast<uint4*>(dst) = t[k];
        continue;
      }
      uint4 c2, s2;
      rope_chunks<DH>(rope, m, j, c2, s2);
      float x[8];
      unpack8(t[k], x);
      float ss = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) ss += x[i] * x[i];
      ss = head_sum<LPH>(ss);
      const float rstd = rsqrtf(ss / (float)DH + eps);
      const float* w = seg == 0 ? wqf : wkf;
      const uint32_t cw[4] = {c2.x, c2.y, c2.z, c2.w}, sw[4] = {s2.x, s2.y, s2.z, s2.w};
      uint32_t o[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint32_t Y = bf2_cvt(x[2 * i] * rstd * w[2 * i], x[2 * i + 1] * rstd * w[2 * i + 1]);
        o[i] = bf2_add(bf2_mul(Y, cw[i]), bf2_mul(bf2_swap(Y), sw[i]));
      }
      *reinterpret_cast<uint4*>(dst) = make_uint4(o[0], o[1], o[2], o[3]);
    }
  }
}

// Backward, in place on dz[:, 0:2D]: same lane <-> column mapping; the lane's dw accumulators (8 columns x {q, k}) are
// reduced over the lanes that own the same columns, then per block and per grid.
template <int DH, int UN>
__global__ void __launch_bounds__(256) qk_norm_rope_bwd16_kernel(bf16* __restrict__ dz, long long lddz,
                                                                 const bf16* __restrict__ zraw, long long ldz,
                                                                 const bf16* __restrict__ wq, const bf16* __restrict__ wk,
                                                                 const bf16* __restrict__ rope, float* __restrict__ dw,
                                                                 int M, int heads, float eps) {
  constexpr int LPH = DH / 8, HPW = 32 / LPH;
  __shared__ float red[8][2][DH];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, sub = lane / LPH, j = lane - sub * LPH;
  const unsigned upr = (unsigned)(2 * heads / HPW);
  const unsigned total = (unsigned)M * upr;
  const unsigned nwarps = gridDim.x * 8u;
  float wqf[8], wkf[8], accq[8], acck[8];
  unpack8(ld_global_nc_v4(wq + 8 * j), wqf);
  unpack8(ld_global_nc_v4(wk + 8 * j), wkf);
#pragma unroll
  for (int i = 0; i < 8; ++i) accq[i] = acck[i] = 0.f;
  for (unsigned u0 = (blockIdx.x * 8u + (unsigned)warp) * UN; u0 < total; u0 += nwarps * UN) {
    uint4 tx[UN], td[UN];
    int mrow[UN], g[UN];
#pragma unroll
    for (int k = 0; k < UN; ++k) {
      const unsigned u = u0 + k;
      mrow[k] = -1;
      tx[k] = td[k] = make_uint4(0u, 0u, 0u, 0u);
      if (u < total) {
        mrow[k] = (int)(u / upr);
        g[k] = (int)(u - (unsigned)mrow[k] * upr);
        tx[k] = ld_global_nc_v4(zraw + (long long)mrow[k] * ldz + g[k] * 256 + lane * 8);
        td[k] = ld_global_v4(dz + (long long)mrow[k] * lddz + g[k] * 256 + lane * 8);
      }
    }
#pragma unroll
    for (int k = 0; k < UN; ++k) {
      if (mrow[k] < 0) continue;
      const int m = mrow[k];
      const int seg = (g[k] * HPW) / heads;                         // 0 = q, 1 = k (warp-uniform)
      uint4 c2, s2;
      rope_chunks<DH>(rope, m, j, c2, s2);
      float x[8], d[8], gr[8];
      unpack8(tx[k], x);
      unpack8(td[k], d);
      const uint32_t cw[4] = {c2.x, c2.y, c2.z, c2.w}, sw[4] = {s2.x, s2.y, s2.z, s2.w};
      float ss = 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float c = bf16_lo(cw[i]), sn = bf16_hi(sw[i]);        // C2 = (c, c), S2 = (-s, +s)
        gr[2 * i] = c * d[2 * i] + sn * d[2 * i + 1];               // un-rotate
        gr[2 * i + 1] = -sn * d[2 * i] + c * d[2 * i + 1];
        ss += x[2 * i] * x[2 * i] + x[2 * i + 1] * x[2 * i + 1];
      }
      ss = head_sum<LPH>(ss);
      const float rstd = rsqrtf(ss / (float)DH + eps);
      const float* w = seg == 0 ? wqf : wkf;
      float gw[8], dot = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        x[i] *= rstd;                                               // xh
        gw[i] = gr[i] * w[i];
        dot += gw[i] * x[i];
      }
      if (seg == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) accq[i] += gr[i] * x[i];
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) acck[i] += gr[i] * x[i];
      }
      dot = head_sum<LPH>(dot) / (float)DH;
      float o[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = rstd * (gw[i] - x[i] * dot);
      *reinterpret_cast<uint4*>(dz + (long long)m * lddz + g[k] * 256 + lane * 8) = pack8(o);
    }
  }
  // lanes sub = 0 .. HPW-1 own the same columns: fold them, then warps, then the grid
#pragma unroll
  for (int i = 0; i < 8; ++i) {
#pragma unroll
    for (int o = LPH; o < 32; o <<= 1) {
      accq[i] += __shfl_xor_sync(0xffffffffu, accq[i], o);
      acck[i] += __shfl_xor_sync(0xffffffffu, acck[i], o);
    }
  }
  if (sub == 0) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      red[warp][0][8 * j + i] = accq[i];
      red[warp][1][8 * j + i] = acck[i];
    }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < 2 * DH; e += blockDim.x) {
    float sum = 0.f;
#pragma unroll
    for (int wp = 0; wp < 8; ++wp) sum += red[wp][e / DH][e % DH];
    atomicAdd(&dw[e], sum);
  }
}

// RMSNorm backward with column-owning threads: CTA = D / 8 threads (rounded up to whole warps), a thread keeps 8 fixed columns, so
// dw needs 8 accumulators (not 128) and every operand is read ONCE: RB rows per pass, all 3 x RB 16-byte loads of a thread issued up
// front, ONE block-wide reduction per pass for both row statistics -- sum x^2 and sum dh w x (mean(gw * xh) = rstd * that / D, so it
// does not have to wait for rstd) --, through ping-pong shared-memory slots (one __syncthreads per pass).
template <int RB, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB) rmsnorm_bwd_cols_kernel(const bf16* __restrict__ x, const bf16* __restrict__ dh,
                                                                const bf16* __restrict__ w, const bf16* __restrict__ dx_res,
                                                                bf16* __restrict__ dx_out, float* __restrict__ dw, int M, int D,
                                                                float eps) {
  __shared__ __align__(16) float red[2][32][2 * RB];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  const bool active = tid < (D >> 3);
  const int c = tid * 8;
  float wv[8], acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) wv[i] = acc[i] = 0.f;
  if (active) unpack8(ld_global_nc_v4(w + c), wv);
  const float inv_d = 1.f / (float)D;
  int buf = 0;
  for (long long m0 = (long long)blockIdx.x * RB; m0 < M; m0 += (long long)gridDim.x * RB) {
    uint4 xr[RB], dr[RB], rr[RB];
#pragma unroll
    for (int r = 0; r < RB; ++r) {
      xr[r] = dr[r] = rr[r] = make_uint4(0u, 0u, 0u, 0u);
      if (active && m0 + r < M) {
        const long long off = (m0 + r) * D + c;
        xr[r] = ld_global_nc_v4(x + off);
        dr[r] = ld_global_nc_v4(dh + off);
        rr[r] = ld_global_v4(dx_res + off);
      }
    }
    float part[2 * RB];
#pragma unroll
    for (int r = 0; r < RB; ++r) {
      float xv[8], dv[8];
      unpack8(xr[r], xv);
      unpack8(dr[r], dv);
      float ss = 0.f, s2 = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        ss += xv[i] * xv[i];
        s2 += dv[i] * wv[i] * xv[i];
      }
      part[r] = warp_sum(ss);
      part[RB + r] = warp_sum(s2);
    }
    if (lane == 0) {
#pragma unroll
      for (int q = 0; q < 2 * RB; ++q) red[buf][warp][q] = part[q];
    }
    __syncthreads();
    float tot[2 * RB];
#pragma unroll
    for (int q = 0; q < 2 * RB; ++q) tot[q] = 0.f;
    for (int wp = 0; wp < nw; ++wp) {
#pragma unroll
      for (int q = 0; q < 2 * RB; q += 4) {
        const float4 v = *reinterpret_cast<const float4*>(&red[buf][wp][q]);
        tot[q] += v.x; tot[q + 1] += v.y; tot[q + 2] += v.z; tot[q + 3] += v.w;
      }
    }
    buf ^= 1;
    if (active) {
#pragma unroll
      for (int r = 0; r < RB; ++r) {
        if (m0 + r >= M) break;
        const float rstd = rsqrtf(tot[r] * inv_d + eps);
        const float dot = rstd * tot[RB + r] * inv_d;               // mean(gw * xh)
        float xv[8], dv[8], rv[8], o[8];
        unpack8(xr[r], xv);
        unpack8(dr[r], dv);
        unpack8(rr[r], rv);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float xh = xv[i] * rstd;
          acc[i] += dv[i] * xh;
          o[i] = rv[i] + rstd * (dv[i] * wv[i] - xh * dot);
        }
        *reinterpret_cast<uint4*>(dx_out + (m0 + r) * D + c) = pack8(o);
      }
    }
  }
  if (active) {
#pragma unroll
    for (int i = 0; i < 8; ++i) atomicAdd(&dw[c + i], acc[i]);
  }
}


#define VTK_TRAIN_CHECK(cond, ...) \
  do {                             \
    if (!(cond)) {                 \
      set_error(__VA_ARGS__);      \
      return -2;                   \
    }                              \
  } while (0)

int launch_qk_norm_rope_fwd(const bf16* zraw, long long ldz, const bf16* wq, const bf16* wk, const bf16* rope, bf16* qkv,
                            long long ldq, int M, int heads, int d, float eps, cudaStream_t st) {
  VTK_TRAIN_CHECK(head_dim_supported(d), "qk_norm_rope: head_dim %d unsupported (supported: multiples of 8 from 8 to 128)", d);
  if (M <= 0) return 0;
  const bool in_place = zraw == qkv;
  VTK_TRAIN_CHECK(!in_place || ldz == ldq, "qk_norm_rope: in place needs ldz == ldq");
  if (in_place || (d != 64 && d != 128)) {
    const int nseg = in_place ? 2 : 3;
    qk_norm_rope_fwd_any_kernel<<<grid_for((long long)M * nseg * heads, 8), 256, 0, st>>>(zraw, ldz, wq, wk, rope, qkv, ldq, M, heads, d,
                                                                                           nseg, eps);
    return check_cuda(cudaGetLastError(), "qk_norm_rope_fwd (any d) launch");
  }
  const int hpw = 32 / (d / 8);
  if (heads % hpw == 0 && ldz % 8 == 0 && ldq % 8 == 0 && (long long)M * (3 * heads / hpw) < (1ll << 31) &&
      ((reinterpret_cast<uintptr_t>(zraw) | reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(wq) | reinterpret_cast<uintptr_t>(wk) |
        reinterpret_cast<uintptr_t>(rope)) & 15) == 0) {
    const int g16 = grid_for(((long long)M * (3 * heads / hpw) + 3) / 4, 8, 8);
    if (d == 64) qk_norm_rope_fwd16_kernel<64, 4><<<g16, 256, 0, st>>>(zraw, ldz, wq, wk, rope, qkv, ldq, M, heads, eps);
    else qk_norm_rope_fwd16_kernel<128, 4><<<g16, 256, 0, st>>>(zraw, ldz, wq, wk, rope, qkv, ldq, M, heads, eps);
    return check_cuda(cudaGetLastError(), "qk_norm_rope_fwd16 launch");
  }
  const int grid = grid_for((long long)M * 3 * heads, 8);
  if (d == 64) qk_norm_rope_fwd_kernel<64><<<grid, 256, 0, st>>>(zraw, ldz, wq, wk, rope, qkv, ldq, M, heads, eps);
  else qk_norm_rope_fwd_kernel<128><<<grid, 256, 0, st>>>(zraw, ldz, wq, wk, rope, qkv, ldq, M, heads, eps);
  return check_cuda(cudaGetLastError(), "qk_norm_rope_fwd launch");
}
int launch_swiglu_fwd(const bf16* zraw, long long ldz, int qp, bf16* act, long long lda, int M, int Hf, int layout, cudaStream_t st) {
  VTK_TRAIN_CHECK(Hf % 16 == 0 && lda % 8 == 0 && ldz % 8 == 0, "swiglu: Hf %% 16 and strides %% 8 required");
  if (M <= 0) return 0;
  if ((long long)M * (Hf / 8) + (long long)num_sms() * 16 * 256 < (1ll << 32))
    swiglu_fwd_kernel<unsigned><<<grid_for((long long)M * (Hf / 8), 256), 256, 0, st>>>(zraw, ldz, qp, act, lda, M, Hf, layout);
  else swiglu_fwd_kernel<long long><<<grid_for((long long)M * (Hf / 8), 256), 256, 0, st>>>(zraw, ldz, qp, act, lda, M, Hf, layout);
  return check_cuda(cudaGetLastError(), "swiglu_fwd launch");
}
int launch_resid_fwd(const bf16* x, const bf16* y, const bf16* gamma, bf16* out, int M, int D, cudaStream_t st, const float* keep,
                     int rows_per_img, float keep_prob) {
  VTK_TRAIN_CHECK(D % 8 == 0, "resid: D %% 8 required");
  VTK_TRAIN_CHECK(!keep || (rows_per_img > 0 && keep_prob > 0.f), "resid: drop_path needs rows_per_img > 0 and keep_prob > 0");
  if (M <= 0) return 0;
  resid_fwd_kernel<<<grid_for((long long)M * (D / 8), 256), 256, 0, st>>>(x, y, gamma, out, M, D, keep, rows_per_img, keep_prob);
  return check_cuda(cudaGetLastError(), "resid_fwd launch");
}
int launch_ln_fwd(const bf16* x, bf16* out, int M, int C, float eps, cudaStream_t st) {
  VTK_TRAIN_CHECK(C <= 256, "layernorm: C <= 256 required (C=%d)", C);
  if (M <= 0) return 0;
  ln_fwd_kernel<<<grid_for(M, 8), 256, 0, st>>>(x, out, M, C, eps);
  return check_cuda(cudaGetLastError(), "ln_fwd launch");
}
int launch_resid_bwd(const bf16* dx, const bf16* y, const bf16* gamma, bf16* dy, float* dgamma, int M, int D, cudaStream_t st,
                     const float* keep, int rows_per_img, float keep_prob) {
  VTK_TRAIN_CHECK(D % 8 == 0, "resid_bwd: D %% 8 required");
  VTK_TRAIN_CHECK(!keep || (rows_per_img > 0 && keep_prob > 0.f), "resid_bwd: drop_path needs rows_per_img > 0 and keep_prob > 0");
  if (M <= 0) return 0;
  dim3 grid((D + 255) / 256, (unsigned)std::min<long long>(((long long)M + 7) / 8, 4LL * num_sms()));
  resid_bwd_kernel<<<grid, 256, 0, st>>>(dx, y, gamma, dy, dgamma, M, D, keep, rows_per_img, keep_prob);
  return check_cuda(cudaGetLastError(), "resid_bwd launch");
}
int launch_colsum(const bf16* in, long long ld, float* out, int M, int C, cudaStream_t st) {
  VTK_TRAIN_CHECK(C % 8 == 0 && ld % 8 == 0, "colsum: C, ld %% 8 required");
  if (M <= 0) return 0;
  dim3 grid((C + 255) / 256, (unsigned)std::min<long long>(((long long)M + 7) / 8, 4LL * num_sms()));
  colsum_kernel<<<grid, 256, 0, st>>>(in, ld, out, M, C);
  return check_cuda(cudaGetLastError(), "colsum launch");
}
int launch_swiglu_bwd(const bf16* dact, long long ldd, const bf16* zraw, long long ldz, int qp, bf16* dz, long long lddz, int M,
                      int Hf, int layout, cudaStream_t st) {
  VTK_TRAIN_CHECK(Hf % 16 == 0 && ldd % 8 == 0 && ldz % 8 == 0 && lddz % 8 == 0, "swiglu_bwd: Hf %% 16 and strides %% 8 required");
  if (M <= 0) return 0;
  if ((long long)M * (Hf / 8) + (long long)num_sms() * 16 * 256 < (1ll << 32))
    swiglu_bwd_kernel<unsigned><<<grid_for((long long)M * (Hf / 8), 256), 256, 0, st>>>(dact, ldd, zraw, ldz, qp, dz, lddz, M, Hf, layout);
  else swiglu_bwd_kernel<long long><<<grid_for((long long)M * (Hf / 8), 256), 256, 0, st>>>(dact, ldd, zraw, ldz, qp, dz, lddz, M, Hf, layout);
  return check_cuda(cudaGetLastError(), "swiglu_bwd launch");
}
int launch_qk_norm_rope_bwd(bf16* dz, long long lddz, const bf16* zraw, long long ldz, const bf16* wq, const bf16* wk,
                            const bf16* rope, float* dw, int M, int heads, int d, float eps, cudaStream_t st) {
  VTK_TRAIN_CHECK(head_dim_supported(d), "qk_norm_rope_bwd: head_dim %d unsupported (supported: multiples of 8 from 8 to 128)", d);
  if (M <= 0) return 0;
  if (d != 64 && d != 128) {
    qk_norm_rope_bwd_any_kernel<<<grid_for((long long)M * 2 * heads, 8, 8), 256, 0, st>>>(dz, lddz, zraw, ldz, wq, wk, rope, dw, M, heads,
                                                                                            d, eps);
    return check_cuda(cudaGetLastError(), "qk_norm_rope_bwd (any d) launch");
  }
  const int hpw = 32 / (d / 8);
  if (heads % hpw == 0 && ldz % 8 == 0 && lddz % 8 == 0 && (long long)M * (2 * heads / hpw) < (1ll << 31) &&
      ((reinterpret_cast<uintptr_t>(zraw) | reinterpret_cast<uintptr_t>(dz) | reinterpret_cast<uintptr_t>(wq) | reinterpret_cast<uintptr_t>(wk) |
        reinterpret_cast<uintptr_t>(rope)) & 15) == 0) {
    const int g16 = grid_for(((long long)M * (2 * heads / hpw) + 3) / 4, 8, 4);
    if (d == 64) qk_norm_rope_bwd16_kernel<64, 4><<<g16, 256, 0, st>>>(dz, lddz, zraw, ldz, wq, wk, rope, dw, M, heads, eps);
    else qk_norm_rope_bwd16_kernel<128, 4><<<g16, 256, 0, st>>>(dz, lddz, zraw, ldz, wq, wk, rope, dw, M, heads, eps);
    return check_cuda(cudaGetLastError(), "qk_norm_rope_bwd16 launch");
  }
  const int grid = grid_for((long long)M * 2 * heads, 8, 8);
  if (d == 64) qk_norm_rope_bwd_kernel<64><<<grid, 256, 0, st>>>(dz, lddz, zraw, ldz, wq, wk, rope, dw, M, heads, eps);
  else qk_norm_rope_bwd_kernel<128><<<grid, 256, 0, st>>>(dz, lddz, zraw, ldz, wq, wk, rope, dw, M, heads, eps);
  return check_cuda(cudaGetLastError(), "qk_norm_rope_bwd launch");
}
int launch_rmsnorm_bwd(const bf16* x, const bf16* dh, const bf16* w, const bf16* dx_res, bf16* dx_out, float* dw, int M, int D,
                       float eps, cudaStream_t st) {
  VTK_TRAIN_CHECK(D % 8 == 0 && D <= 4096, "rmsnorm_bwd: D %% 8 == 0 and D <= 4096 required (D=%d)", D);
  if (M <= 0) return 0;
  if (((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dh) | reinterpret_cast<uintptr_t>(w) |
               reinterpret_cast<uintptr_t>(dx_res) | reinterpret_cast<uintptr_t>(dx_out)) & 15) == 0) {
    const int threads = ((D / 8) + 31) / 32 * 32;                       // <= 512 for D <= 4096
    const int per_sm = threads <= 192 ? 4 : threads <= 384 ? 2 : 1;
    const int RB = threads <= 384 ? 2 : 4;   // rows per pass: 2 x 3 x 16 bytes per thread and two CTAs per SM, or 4 x 3 x 16 and one
    long long g = ((long long)M + RB - 1) / RB;
    if (g > (long long)num_sms() * per_sm) g = (long long)num_sms() * per_sm;
    if (threads <= 384) rmsnorm_bwd_cols_kernel<2, 384, 2><<<(unsigned)g, threads, 0, st>>>(x, dh, w, dx_res, dx_out, dw, M, D, eps);
    else rmsnorm_bwd_cols_kernel<4, 512, 1><<<(unsigned)g, threads, 0, st>>>(x, dh, w, dx_res, dx_out, dw, M, D, eps);
    return check_cuda(cudaGetLastError(), "rmsnorm_bwd (columns) launch");
  }
  const int grid = grid_for(M, 8, 4);
  const size_t smem = (size_t)8 * D * sizeof(float);
  auto run = [&](auto kern) {
    if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<grid, 256, smem, st>>>(x, dh, w, dx_res, dx_out, dw, M, D, eps);
  };
  if (D <= 1024) run(rmsnorm_bwd_kernel<4>);
  else if (D <= 2048) run(rmsnorm_bwd_kernel<8>);
  else run(rmsnorm_bwd_kernel<16>);
  return check_cuda(cudaGetLastError(), "rmsnorm_bwd launch");
}
int launch_ln_bwd(const bf16* zlin, const bf16* dz, bf16* dx, int M, int C, float eps, cudaStream_t st) {
  VTK_TRAIN_CHECK(C <= 256, "layernorm_bwd: C <= 256 required (C=%d)", C);
  if (M <= 0) return 0;
  ln_bwd_kernel<<<grid_for(M, 8), 256, 0, st>>>(zlin, dz, dx, M, C, eps);
  return check_cuda(cudaGetLastError(), "ln_bwd launch");
}
int launch_charbonnier(const bf16* pred, const bf16* target, const uint8_t* mask, const int* n_valid, float* loss_sum, bf16* dpred,
                       int B, int N, int P, float eps, cudaStream_t st) {
  VTK_TRAIN_CHECK(P % 8 == 0, "charbonnier: P %% 8 required");
  if (B <= 0 || N <= 0) return 0;
  charbonnier_kernel<<<grid_for((long long)B * N, 8), 256, 0, st>>>(pred, target, mask, n_valid, loss_sum, dpred, B, N, P, eps);
  return check_cuda(cudaGetLastError(), "charbonnier launch");
}
// The next launch's share of the tensor table from tensors[i] on: at most ADAMW_MAX_T non-empty tensors and fewer than 2^30
// chunks.  Fills g / n / g_f32 / chunk0 of `bt` (all the norm pass reads) and src[k] = the table index of slot k; returns the
// batch's chunk count.
static long long next_adamw_batch(const AdamwTensor* tensors, int n_tensors, int& i, AdamwBatch& bt, int (&src)[ADAMW_MAX_T]) {
  bt.nt = 0;
  long long chunks = 0;
  for (; i < n_tensors && bt.nt < ADAMW_MAX_T; ++i) {
    const AdamwTensor& t = tensors[i];
    if (t.n <= 0) continue;
    const long long c = (t.n + ADAMW_CHUNK - 1) / ADAMW_CHUNK;
    if (chunks + c >= (1ll << 30)) break;
    const int k = bt.nt++;
    src[k] = i;
    bt.g[k] = t.g; bt.n[k] = t.n; bt.g_f32[k] = t.g_is_f32 ? 1 : 0;
    bt.chunk0[k] = (int)chunks;
    chunks += c;
  }
  bt.chunk0[bt.nt] = (int)chunks;
  return chunks;
}

template <bool kClip, bool kEma>
static int launch_adamw_t(const AdamwTensor* tensors, float* const* ema, int n_tensors, float lr, float b1, float b2, float eps,
                          float bc1, float bc2s, float grad_scale, const float* coef, float ema_w, cudaStream_t st) {
  int i = 0;
  while (i < n_tensors) {
    AdamwBatchT<kEma> bt;
    int src[ADAMW_MAX_T];
    const long long chunks = next_adamw_batch(tensors, n_tensors, i, bt, src);
    if (bt.nt == 0) continue;
    for (int k = 0; k < bt.nt; ++k) {
      const AdamwTensor& t = tensors[src[k]];
      VTK_TRAIN_CHECK(t.master && t.g && t.m && t.v, "adamw: null pointer in tensor %d", src[k]);
      bt.master[k] = t.master; bt.p16[k] = (bf16*)t.p16; bt.m[k] = t.m; bt.v[k] = t.v; bt.wd[k] = t.weight_decay;
      if constexpr (kEma) {
        VTK_TRAIN_CHECK(ema[src[k]], "adamw: null ema pointer for tensor %d", src[k]);
        bt.ema[k] = ema[src[k]];
      }
    }
    const int grid = (int)std::min<long long>(chunks, (long long)num_sms() * 8);
    adamw_multi_kernel<kClip, kEma><<<grid, 256, 0, st>>>(bt, lr, b1, b2, eps, bc1, bc2s, grad_scale, coef, ema_w);
    if (check_cuda(cudaGetLastError(), "adamw_multi launch")) return -1;
  }
  return 0;
}

int launch_adamw_multi(const AdamwTensor* tensors, float* const* ema, int n_tensors, float lr, float b1, float b2, float eps, int step,
                       float grad_scale, const float* coef, double ema_decay, cudaStream_t st) {
  VTK_TRAIN_CHECK(step >= 1, "adamw: step must be >= 1");
  VTK_TRAIN_CHECK(!ema || (ema_decay >= 0.0 && ema_decay < 1.0), "adamw: ema_decay must lie in [0, 1) (got %g)", ema_decay);
  const float bc1 = 1.f - powf(b1, (float)step), bc2s = sqrtf(1.f - powf(b2, (float)step));
  const float ema_w = (float)(1.0 - ema_decay);   // the weight torch._foreach_lerp_(ema, master, 1 - decay) rounds to fp32
  if (coef) {
    return ema ? launch_adamw_t<true, true>(tensors, ema, n_tensors, lr, b1, b2, eps, bc1, bc2s, grad_scale, coef, ema_w, st)
               : launch_adamw_t<true, false>(tensors, ema, n_tensors, lr, b1, b2, eps, bc1, bc2s, grad_scale, coef, ema_w, st);
  }
  return ema ? launch_adamw_t<false, true>(tensors, ema, n_tensors, lr, b1, b2, eps, bc1, bc2s, grad_scale, coef, ema_w, st)
             : launch_adamw_t<false, false>(tensors, ema, n_tensors, lr, b1, b2, eps, bc1, bc2s, grad_scale, coef, ema_w, st);
}

long long grad_norm_slots(const AdamwTensor* tensors, int n_tensors) {
  long long s = 0;
  for (int i = 0; i < n_tensors; ++i)
    if (tensors[i].n > 0) s += (tensors[i].n + ADAMW_CHUNK - 1) / ADAMW_CHUNK;
  return s;
}

int launch_grad_sumsq(const AdamwTensor* tensors, int n_tensors, float* partials, cudaStream_t st) {
  int i = 0;
  while (i < n_tensors) {
    AdamwBatch bt;
    int src[ADAMW_MAX_T];
    const long long chunks = next_adamw_batch(tensors, n_tensors, i, bt, src);
    if (bt.nt == 0) continue;
    for (int k = 0; k < bt.nt; ++k) VTK_TRAIN_CHECK(bt.g[k], "grad_norm: null gradient pointer in tensor %d", src[k]);
    const int grid = (int)std::min<long long>(chunks, (long long)num_sms() * 8);
    grad_sumsq_kernel<<<grid, 256, 0, st>>>(bt, partials);
    if (check_cuda(cudaGetLastError(), "grad_sumsq launch")) return -1;
    partials += chunks;
  }
  return 0;
}

int launch_grad_norm_finish(const float* partials, long long n_slots, float max_norm, float* norm_coef, cudaStream_t st) {
  grad_norm_finish_kernel<<<1, 256, 0, st>>>(partials, n_slots, max_norm, norm_coef);
  return check_cuda(cudaGetLastError(), "grad_norm_finish launch");
}
int launch_scale_by_dev(bf16* x, const float* scale, long long n, cudaStream_t st) {
  if (n <= 0) return 0;
  scale_by_dev_kernel<<<grid_for((n + 7) / 8, 256, 8), 256, 0, st>>>(x, scale, n);
  return check_cuda(cudaGetLastError(), "scale_by_dev launch");
}
int launch_attn_delta(const bf16* o, long long ldo, const bf16* dob, long long lddo, float* delta, int M, int heads, int d,
                      cudaStream_t st) {
  VTK_TRAIN_CHECK(head_dim_supported(d), "attn_delta: head_dim %d unsupported (supported: multiples of 8 from 8 to 128)", d);
  if (M <= 0) return 0;
  attn_delta_kernel<<<grid_for((long long)M * heads, 8), 256, 0, st>>>(o, ldo, dob, lddo, delta, M, heads, d);
  return check_cuda(cudaGetLastError(), "attn_delta launch");
}

}  // namespace vtk
