// vtk_elementwise.cu -- HBM-bound helper kernels of the AE path (coalesced, 16-byte vectorised).
//
//   rmsnorm      Block.norm1            vitok/models/modules/norm.py:17-25   (bf16 in/out, fp32 math)
//   rope_table   compute_2d_freqs_cis   vitok/models/modules/rotary_embedding.py:46-75 (+ the bf16 cast at :118-119)
//   kv_len       _get_attn_mask         vitok/models/ae.py:173-187 reduced to a per-image key count
//   casts        callers' .to(bf16)     scripts/train_vae.py:305-306
#include "vtk_common.cuh"
#include "vtk_kernels.h"

namespace vtk {

// one warp per row; D % 8 == 0.  Two passes over the row (second pass hits L1).
__global__ void __launch_bounds__(256) rmsnorm_kernel(const bf16* __restrict__ x, long long ldx,
                                                      const bf16* __restrict__ w, bf16* __restrict__ y, long long ldy,
                                                      int M, int D, float eps, const int* __restrict__ m_dev) {
  pdl_wait();      // PDL (vtk_common.cuh): this kernel may have been launched before its predecessor finished
  pdl_trigger();
  const int warps_per_block = blockDim.x >> 5;
  const int lane = threadIdx.x & 31;
  const int nvec = D >> 3;
  if (m_dev) M = min(M, __ldg(m_dev));
  for (long long row = (long long)blockIdx.x * warps_per_block + (threadIdx.x >> 5); row < M;
       row += (long long)gridDim.x * warps_per_block) {
    const bf16* xr = x + row * ldx;
    float ss = 0.f;
    for (int v = lane; v < nvec; v += 32) {
      uint4 q = ld_global_v4(xr + 8 * v);
      const uint32_t u[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float a = bf16_lo(u[i]), b = bf16_hi(u[i]);
        ss += a * a + b * b;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    const float rstd = rsqrtf(ss / (float)D + eps);
    bf16* yr = y + row * ldy;
    for (int v = lane; v < nvec; v += 32) {
      uint4 q = ld_global_v4(xr + 8 * v);
      uint4 g = ld_global_nc_v4(w + 8 * v);
      const uint32_t u[4] = {q.x, q.y, q.z, q.w};
      const uint32_t gw[4] = {g.x, g.y, g.z, g.w};
      uint32_t o[4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
        o[i] = pack_bf16x2(bf16_lo(u[i]) * rstd * bf16_lo(gw[i]), bf16_hi(u[i]) * rstd * bf16_hi(gw[i]));
      st_global_v4(yr + 8 * v, o[0], o[1], o[2], o[3]);
    }
  }
}

// Single-pass variant: the row (D <= NV * 256 elements) stays in registers between the sum of squares and the
// scaling, so x is read from HBM/L2 exactly once.  One warp per row, 16-byte vectors, lane-strided (coalesced).
template <int NV>
__global__ void __launch_bounds__(256) rmsnorm_reg_kernel(const bf16* __restrict__ x, long long ldx,
                                                          const bf16* __restrict__ w, bf16* __restrict__ y,
                                                          long long ldy, int M, int D, float eps,
                                                          const int* __restrict__ m_dev) {
  pdl_wait();      // PDL (vtk_common.cuh): this kernel may have been launched before its predecessor finished
  pdl_trigger();
  const int warps_per_block = blockDim.x >> 5;
  const int lane = threadIdx.x & 31;
  const int nvec = D >> 3;
  const float inv_d = 1.f / (float)D;
  if (m_dev) M = min(M, __ldg(m_dev));
  for (long long row = (long long)blockIdx.x * warps_per_block + (threadIdx.x >> 5); row < M;
       row += (long long)gridDim.x * warps_per_block) {
    const bf16* xr = x + row * ldx;
    uint4 q[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int v = lane + 32 * i;
      q[i] = v < nvec ? ld_global_v4(xr + 8 * v) : make_uint4(0, 0, 0, 0);
    }
    uint64_t ss2 = 0ull;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const uint32_t u[4] = {q[i].x, q[i].y, q[i].z, q[i].w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint64_t t = bf2_to_f2(u[k]);
        ss2 = f2_fma(t, t, ss2);
      }
    }
    float s0, s1;
    f2_unpack(ss2, s0, s1);
    float ss = s0 + s1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    const float rstd = rsqrtf(ss * inv_d + eps);
    const uint64_t rstd2 = f2_pack(rstd, rstd);
    bf16* yr = y + row * ldy;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int v = lane + 32 * i;
      if (v < nvec) {
        const uint4 g = ld_global_nc_v4(w + 8 * v);
        const uint32_t u[4] = {q[i].x, q[i].y, q[i].z, q[i].w};
        const uint32_t gw[4] = {g.x, g.y, g.z, g.w};
        uint32_t o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float a, b;
          f2_unpack(f2_mul(f2_mul(bf2_to_f2(u[k]), rstd2), bf2_to_f2(gw[k])), a, b);
          o[k] = bf2_cvt(a, b);
        }
        st_global_v4(yr + 8 * v, o[0], o[1], o[2], o[3]);
      }
    }
  }
}

int launch_rmsnorm(const bf16* x, long long ldx, const bf16* w, bf16* y, long long ldy, int M, int D, float eps,
                   cudaStream_t stream, const int* m_dev) {
  if (D % 8 || ldx % 8 || ldy % 8) { set_error("rmsnorm: D and strides must be multiples of 8"); return -2; }
  if (M <= 0) return 0;
  const int wpb = 8;
  long long blocks = ((long long)M + wpb - 1) / wpb;
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  if (D <= 1024) (void)launch_k(rmsnorm_reg_kernel<4>, dim3((int)blocks), dim3(wpb * 32), 0, stream, x, ldx, w, y, ldy, M, D, eps, m_dev);
  else if (D <= 3072) (void)launch_k(rmsnorm_reg_kernel<12>, dim3((int)blocks), dim3(wpb * 32), 0, stream, x, ldx, w, y, ldy, M, D, eps, m_dev);
  else if (D <= 4096) (void)launch_k(rmsnorm_reg_kernel<16>, dim3((int)blocks), dim3(wpb * 32), 0, stream, x, ldx, w, y, ldy, M, D, eps, m_dev);
  else (void)launch_k(rmsnorm_kernel, dim3((int)blocks), dim3(wpb * 32), 0, stream, x, ldx, w, y, ldy, M, D, eps, m_dev);
  return check_cuda(cudaGetLastError(), "rmsnorm launch");
}

// Pair-expanded, chunk-major RoPE table consumed by the QKV GEMM epilogue (vtk_gemm.cu, rope_row_ptr):
//   per token row 2d bf16 = C2[d] = (c_0, c_0, c_1, c_1, ...) | S2[d] = (-s_0, +s_0, -s_1, +s_1, ...),
//   c_j = bf16(cos(angle_j)), s_j = bf16(sin(angle_j)), angle_j = row*f_j for j < d/4, col*f_{j-d/4} for j >= d/4
//   (fp32 angles like the reference, rotary_embedding.py:46-75; the bf16 cast is the one at :118-119);
//   bf16 element offset(row m, element e) = ((m >> 5) * (d / 4) + (e >> 3)) * 256 + (m & 31) * 8 + (e & 7).
// Rows are grouped by 32 so that one warp of the epilogue (32 consecutive rows) reads each 16-byte chunk
// as 512 contiguous bytes.  The table holds ceil(M / 32) * 32 rows.
__global__ void rope_table_kernel(const int64_t* __restrict__ row_idx, const int64_t* __restrict__ col_idx,
                                  const float* __restrict__ inv_freq, bf16* __restrict__ table, int M, int d,
                                  const int* __restrict__ src_map, const int* __restrict__ m_dev) {
  pdl_wait();      // PDL (vtk_common.cuh): this kernel may have been launched before its predecessor finished
  pdl_trigger();
  const int half = d >> 1, quarter = d >> 2;
  if (m_dev) M = min(M, __ldg(m_dev));
  const long long groups = ((long long)M + 31) >> 5;
  const long long total = groups * half * 32;   // thread <-> (group, pair j, row-in-group): coalesced-ish writes
  uint32_t* tw = reinterpret_cast<uint32_t*>(table);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int ml = (int)(i & 31);
    const long long t = i >> 5;
    const int j = (int)(t % half);
    const long long grp = t / half;
    const long long m = grp * 32 + ml;
    if (m >= M) continue;
    // packed NaFlex batches: table row m belongs to source token src_map[m] (pad rows: position 0)
    const long long src = src_map ? (long long)src_map[m] : m;
    const float pos = src < 0 ? 0.f : (j < quarter ? (float)row_idx[src] : (float)col_idx[src]);
    const float f = inv_freq[j < quarter ? j : j - quarter];
    const float ang = pos * f;
    const uint32_t c = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(cosf(ang)));
    const uint32_t sn = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(sinf(ang)));
    // 32-bit word w of the row (w < d/2: C2 pair w; w >= d/2: S2 pair w - d/2) lives in chunk w/4, slot w%4
    const long long base = grp * (long long)(d >> 2);
    const int wc = j, ws = half + j;
    tw[((base + (wc >> 2)) * 32 + ml) * 4 + (wc & 3)] = c | (c << 16);
    tw[((base + (ws >> 2)) * 32 + ml) * 4 + (ws & 3)] = (sn ^ 0x8000u) | (sn << 16);
  }
}

int launch_rope_table(const int64_t* row_idx, const int64_t* col_idx, const float* inv_freq, bf16* table, int M, int d,
                      cudaStream_t stream, const int* src_map, const int* m_dev) {
  if (d % 8) { set_error("rope: head dimension must be a multiple of 8 (2D RoPE needs d %% 4 == 0; table chunks need 8)"); return -2; }
  if (M <= 0) return 0;
  const long long total = (((long long)M + 31) >> 5) * (d / 2) * 32;
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  (void)launch_k(rope_table_kernel, dim3((int)blocks), dim3(256), 0, stream, row_idx, col_idx, inv_freq, table, M, d, src_map, m_dev);
  return check_cuda(cudaGetLastError(), "rope_table launch");
}

__global__ void cast_f32_bf16_kernel(const float* __restrict__ in, bf16* __restrict__ out, long long n) {
  pdl_wait();      // PDL (vtk_common.cuh): this kernel may have been launched before its predecessor finished
  pdl_trigger();
  const long long nvec = n >> 3;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += stride) {
    const float4 a = reinterpret_cast<const float4*>(in)[2 * v];
    const float4 b = reinterpret_cast<const float4*>(in)[2 * v + 1];
    st_global_v4(out + 8 * v, pack_bf16x2(a.x, a.y), pack_bf16x2(a.z, a.w), pack_bf16x2(b.x, b.y), pack_bf16x2(b.z, b.w));
  }
  for (long long i = (nvec << 3) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    out[i] = __float2bfloat16_rn(in[i]);
}
static int cast_grid(long long n) {
  long long blocks = (n / 8 + 255) / 256 + 1;
  const long long cap = (long long)num_sms() * 16;
  return (int)(blocks > cap ? cap : blocks);
}
int launch_cast_f32_bf16(const float* in, bf16* out, long long n, cudaStream_t stream) {
  if (n <= 0) return 0;
  if ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 15) { set_error("cast: pointers must be 16-byte aligned"); return -2; }
  (void)launch_k(cast_f32_bf16_kernel, dim3(cast_grid(n)), dim3(256), 0, stream, in, out, n);
  return check_cuda(cudaGetLastError(), "cast launch");
}

// ------------------------------------------------------------------------------------------------
// FP8 inference (reference AE.quantize, ae.py:253-270: torchao Float8DynamicActivationFloat8Weight on every Linear of the
// blocks): dynamic activation quantisation.  One warp per row: amax over the row, scale = amax / 448, q = e4m3(x / scale)
// (round to nearest even, saturating); the GEMM epilogue multiplies its accumulator row by scale[row] * weight_scale.
// Per-row scales (torchao's PerRow granularity) need no grid-wide reduction before the first byte can be written.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t e4m3x4(float a, float b, float c, float d) {   // bytes (a, b, c, d), a in the low byte
  uint16_t lo, hi;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(lo) : "f"(b), "f"(a));
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(hi) : "f"(d), "f"(c));
  return (uint32_t)lo | ((uint32_t)hi << 16);
}

// amax_all != nullptr: PER-TENSOR dynamic scale (torchao's default granularity for Float8DynamicActivationFloat8WeightConfig): every row
// uses the amax of the whole tensor, computed by amax_kernel below; scale[row] is still written (all equal) so the GEMM epilogue is the same.
__global__ void __launch_bounds__(256) quant_rows_e4m3_kernel(const bf16* __restrict__ x, long long ldx, uint8_t* __restrict__ q,
                                                              long long ldq, float* __restrict__ scale, int M, int K,
                                                              const int* __restrict__ m_dev, const float* __restrict__ amax_all) {
  pdl_wait();      // PDL (vtk_common.cuh): this kernel may have been launched before its predecessor finished
  pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int nvec = K >> 3;   // 8 bf16 = 16 bytes in, 8 bytes out
  if (m_dev) M = min(M, __ldg(m_dev));
  for (long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); row < M; row += (long long)gridDim.x * 8) {
    const bf16* xr = x + row * ldx;
    float amax = 0.f;
    if (amax_all) {
      amax = __ldg(amax_all);
    } else {
      for (int v = lane; v < nvec; v += 32) {
        const uint4 u = ld_global_v4(xr + 8 * v);
        const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) amax = fmaxf(amax, fmaxf(fabsf(bf16_lo(w[i])), fabsf(bf16_hi(w[i]))));
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    }
    const float sc = amax > 0.f ? amax / 448.f : 1.f;
    const float inv = amax > 0.f ? 448.f / amax : 1.f;
    if (lane == 0) scale[row] = sc;
    uint8_t* qr = q + row * ldq;
    for (int v = lane; v < nvec; v += 32) {   // second pass: the row comes from L1 / L2
      const uint4 u = ld_global_v4(xr + 8 * v);
      uint2 o;
      o.x = e4m3x4(bf16_lo(u.x) * inv, bf16_hi(u.x) * inv, bf16_lo(u.y) * inv, bf16_hi(u.y) * inv);
      o.y = e4m3x4(bf16_lo(u.z) * inv, bf16_hi(u.z) * inv, bf16_lo(u.w) * inv, bf16_hi(u.w) * inv);
      *reinterpret_cast<uint2*>(qr + 8 * v) = o;
    }
  }
}

// amax_out[0] = max |x| over the [M, K] tensor (non-negative floats order like their bit patterns: one atomicMax per warp); zero it first
__global__ void __launch_bounds__(256) amax_kernel(const bf16* __restrict__ x, long long ldx, float* __restrict__ amax_out, int M, int K,
                                                   const int* __restrict__ m_dev) {
  pdl_wait();
  pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int nvec = K >> 3;
  if (m_dev) M = min(M, __ldg(m_dev));
  float amax = 0.f;
  for (long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); row < M; row += (long long)gridDim.x * 8) {
    const bf16* xr = x + row * ldx;
    for (int v = lane; v < nvec; v += 32) {
      const uint4 u = ld_global_v4(xr + 8 * v);
      const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) amax = fmaxf(amax, fmaxf(fabsf(bf16_lo(w[i])), fabsf(bf16_hi(w[i]))));
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
  if (lane == 0 && amax > 0.f) atomicMax(reinterpret_cast<int*>(amax_out), __float_as_int(amax));
}

int launch_quant_rows_e4m3(const bf16* x, long long ldx, uint8_t* q, long long ldq, float* scale, int M, int K, const int* m_dev,
                           cudaStream_t stream, float* amax_ws) {
  if (K % 8 || ldx % 8 || ldq % 8) { set_error("quant_rows: K and the row strides must be multiples of 8"); return -2; }
  if (M <= 0) return 0;
  long long blocks = ((long long)M + 7) / 8;
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  if (amax_ws) {   // per-tensor scale: one more read of x for the global amax
    if (check_cuda(cudaMemsetAsync(amax_ws, 0, sizeof(float), stream), "amax memset")) return -1;
    (void)launch_k(amax_kernel, dim3((int)blocks), dim3(256), 0, stream, x, ldx, amax_ws, M, K, m_dev);
  }
  (void)launch_k(quant_rows_e4m3_kernel, dim3((int)blocks), dim3(256), 0, stream, x, ldx, q, ldq, scale, M, K, m_dev, (const float*)amax_ws);
  return check_cuda(cudaGetLastError(), "quant_rows launch");
}

// one warp per image: kv_len = 1 + index of the last valid token (0 if none)
__global__ void kv_len_kernel(const uint8_t* __restrict__ mask, int* __restrict__ kv_len, int B, int N) {
  pdl_wait();      // PDL (vtk_common.cuh): this kernel may have been launched before its predecessor finished
  pdl_trigger();
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= B) return;
  const int lane = threadIdx.x & 31;
  int last = -1;
  for (int i = lane; i < N; i += 32) {
    if (mask[(long long)b * N + i]) last = i;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
  if (lane == 0) kv_len[b] = last + 1;
}
int launch_kv_len(const uint8_t* mask, int* kv_len, int B, int N, cudaStream_t stream) {
  if (B <= 0) return 0;
  (void)launch_k(kv_len_kernel, dim3((B + 3) / 4), dim3(128), 0, stream, mask, kv_len, B, N);
  return check_cuda(cudaGetLastError(), "kv_len launch");
}

// ------------------------------------------------------------------------------------------------
// NaFlex token packing.  The reference runs every block over all B*N token rows and masks the padded keys inside
// SDPA (ae.py:173-187, attention.py:69-73).  Here the valid tokens of a masked batch are packed image after image
// (each image padded to a multiple of 128 rows so no attention tile straddles two images), every kernel of the block
// stack runs on the packed rows only, and the result is scattered back.  Any bool mask is handled: the valid tokens
// of an image keep their order, so inside the packed layout an image is always a dense prefix of n_i tokens.
// The packed row count sum(ceil128(n_i)) never visits the host: kernels read it from device memory (m_dev).
// ------------------------------------------------------------------------------------------------
// one CTA per image: rel[b, t] = rank of token t among the valid tokens of image b (-1 if masked), n_valid[b]
__global__ void __launch_bounds__(256) pack_count_kernel(const uint8_t* __restrict__ mask, int* __restrict__ rel,
                                                         int* __restrict__ n_valid, int N) {
  pdl_wait();      // PDL (vtk_common.cuh): this kernel may have been launched before its predecessor finished
  pdl_trigger();
  __shared__ int warp_tot[8];
  __shared__ int running;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) running = 0;
  __syncthreads();
  for (int t0 = 0; t0 < N; t0 += 256) {
    const int t = t0 + tid;
    const bool v = t < N && mask[(long long)b * N + t] != 0;
    const unsigned bal = __ballot_sync(0xffffffffu, v);
    if (lane == 0) warp_tot[warp] = __popc(bal);
    __syncthreads();
    int before = running;
    for (int w = 0; w < warp; ++w) before += warp_tot[w];
    if (t < N) rel[(long long)b * N + t] = v ? before + __popc(bal & ((1u << lane) - 1u)) : -1;
    __syncthreads();
    if (tid == 0) {
      int tot = 0;
      for (int w = 0; w < 8; ++w) tot += warp_tot[w];
      running += tot;
    }
    __syncthreads();
  }
  if (tid == 0) n_valid[b] = running;
}

// one CTA: cu[b] = packed row offset of image b (exclusive scan of n_valid rounded up to `pad` rows), cu[B] = packed row
// count; attention work groups (`qrows` = 128 or 256 query rows of ONE image each): cuq[b] = first group of image b,
// cuq[B] = number of groups, grp_img[g] = image of group g, grp_order = the groups sorted by the number of key tiles of
// their image, longest first (counting sort; ties in arbitrary order) -- the attention kernel deals its work items from
// this list so that every persistent CTA gets the same mix of long and short items.
__global__ void __launch_bounds__(1024) pack_plan_kernel(const int* __restrict__ n_valid, int* __restrict__ cu, int* __restrict__ cuq,
                                                         int* __restrict__ grp_img, int* __restrict__ grp_order, int B, int N, int pad,
                                                         int qrows) {
  pdl_wait();      // PDL (vtk_common.cuh): this kernel may have been launched before its predecessor finished
  pdl_trigger();
  constexpr int MAX_BINS = 2048;
  __shared__ int warp_tot[2][32];
  __shared__ int running[2];
  __shared__ int bins[MAX_BINS + 1];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < 2) running[tid] = 0;
  __syncthreads();
  for (int b0 = 0; b0 < B; b0 += 1024) {
    const int b = b0 + tid;
    const int n = b < B ? n_valid[b] : 0;
    const int padded = (n + pad - 1) / pad * pad;
    const int groups = (n + qrows - 1) / qrows;
    int incl_r = padded, incl_g = groups;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int vr = __shfl_up_sync(0xffffffffu, incl_r, o), vg = __shfl_up_sync(0xffffffffu, incl_g, o);
      if (lane >= o) { incl_r += vr; incl_g += vg; }
    }
    if (lane == 31) { warp_tot[0][warp] = incl_r; warp_tot[1][warp] = incl_g; }
    __syncthreads();
    int before_r = running[0], before_g = running[1];
    for (int w = 0; w < warp; ++w) { before_r += warp_tot[0][w]; before_g += warp_tot[1][w]; }
    if (b < B) {
      cu[b] = before_r + incl_r - padded;
      const int g0 = before_g + incl_g - groups;
      cuq[b] = g0;
      for (int q = 0; q < groups; ++q) grp_img[g0 + q] = b;
    }
    __syncthreads();
    if (tid == 1023) { running[0] = before_r + incl_r; running[1] = before_g + incl_g; }
    __syncthreads();
  }
  if (tid == 0) { cu[B] = running[0]; cuq[B] = running[1]; }
  // ---- group order: counting sort by key tiles per image, descending ----
  const int nbins = (N + 127) / 128;           // an image has 1 .. nbins key tiles
  const int ngroups = running[1];
  if (nbins > MAX_BINS) {                      // very long sequences: keep the natural order
    for (int t = tid; t < ngroups; t += 1024) grp_order[t] = t;
    return;
  }
  for (int i = tid; i <= nbins; i += 1024) bins[i] = 0;
  __syncthreads();
  for (int b = tid; b < B; b += 1024) {
    const int n = n_valid[b];
    if (n > 0) atomicAdd(&bins[(n + 127) >> 7], (n + qrows - 1) / qrows);
  }
  __syncthreads();
  if (tid == 0) {                              // start offset of each bin, longest images first
    int acc = 0;
    for (int k = nbins; k >= 1; --k) { const int c = bins[k]; bins[k] = acc; acc += c; }
  }
  __syncthreads();
  for (int b = tid; b < B; b += 1024) {
    const int n = n_valid[b];
    if (n > 0) {
      const int groups = (n + qrows - 1) / qrows;
      const int at = atomicAdd(&bins[(n + 127) >> 7], groups);
      const int first = cuq[b];
      for (int q = 0; q < groups; ++q) grp_order[at + q] = first + q;
    }
  }
}

// one CTA per image: src[packed row] = source token row b*N + t, or -1 for the pad rows of the image's last tile
__global__ void __launch_bounds__(256) pack_src_kernel(const int* __restrict__ rel, const int* __restrict__ n_valid,
                                                       const int* __restrict__ cu, int* __restrict__ src, int N, int pad) {
  pdl_wait();      // PDL (vtk_common.cuh): this kernel may have been launched before its predecessor finished
  pdl_trigger();
  const int b = blockIdx.x;
  const int base = cu[b], n = n_valid[b];
  for (int t = threadIdx.x; t < N; t += 256) {
    const int r = rel[(long long)b * N + t];
    if (r >= 0) src[base + r] = b * N + t;
  }
  for (int p = n + threadIdx.x; p < (n + pad - 1) / pad * pad; p += 256) src[base + p] = -1;
}

// packed[r, :] = in[src[r], :] (zeros for pad rows); rows of `width` bf16 (width % 8 == 0), 16-byte vectors
__global__ void __launch_bounds__(256) pack_rows_kernel(const bf16* __restrict__ in, long long ld_in, const int* __restrict__ src,
                                                        const int* __restrict__ m_dev, bf16* __restrict__ out, long long ld_out,
                                                        int width) {
  pdl_wait();      // PDL (vtk_common.cuh): this kernel may have been launched before its predecessor finished
  pdl_trigger();
  const int nvec = width >> 3;
  const long long total = (long long)__ldg(m_dev) * nvec;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / nvec;
    const int v = (int)(i - r * nvec);
    const int s = src[r];
    uint4 q = make_uint4(0, 0, 0, 0);
    if (s >= 0) q = ld_global_nc_v4(in + (long long)s * ld_in + 8 * v);
    st_global_v4(out + r * ld_out + 8 * v, q.x, q.y, q.z, q.w);
  }
}

// out[b, t, :] = packed[cu[b] + rel[b, t], :] for valid tokens, 0 for masked ones
__global__ void __launch_bounds__(256) unpack_rows_kernel(const bf16* __restrict__ packed, long long ld_p, const int* __restrict__ rel,
                                                          const int* __restrict__ cu, bf16* __restrict__ out, long long ld_out,
                                                          long long rows, int N, int width) {
  pdl_wait();      // PDL (vtk_common.cuh): this kernel may have been launched before its predecessor finished
  pdl_trigger();
  const int nvec = width >> 3;
  const long long total = rows * nvec;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long m = i / nvec;
    const int v = (int)(i - m * nvec);
    const int r = rel[m];
    uint4 q = make_uint4(0, 0, 0, 0);
    if (r >= 0) q = ld_global_nc_v4(packed + (long long)(cu[m / N] + r) * ld_p + 8 * v);
    st_global_v4(out + m * ld_out + 8 * v, q.x, q.y, q.z, q.w);
  }
}

int launch_pack_plan(const uint8_t* mask, int B, int N, const PackPlan& pl, cudaStream_t stream) {
  if (B <= 0 || N <= 0) return 0;
  (void)launch_k(pack_count_kernel, dim3(B), dim3(256), 0, stream, mask, pl.rel, pl.n_valid, N);
  if (pl.pad < 8 || pl.pad % 8 || (pl.qrows != 128 && pl.qrows != 256)) {
    set_error("pack_plan: row padding must be a positive multiple of 8 and the attention group 128 or 256 rows (got %d, %d)", pl.pad, pl.qrows);
    return -2;
  }
  (void)launch_k(pack_plan_kernel, dim3(1), dim3(1024), 0, stream, pl.n_valid, pl.cu, pl.cuq, pl.grp_img, pl.grp_order, B, N, pl.pad, pl.qrows);
  (void)launch_k(pack_src_kernel, dim3(B), dim3(256), 0, stream, pl.rel, pl.n_valid, pl.cu, pl.src, N, pl.pad);
  return check_cuda(cudaGetLastError(), "pack_plan launch");
}

static int row_copy_grid(long long rows, int width) {
  long long blocks = (rows * (width / 8) + 255) / 256;
  const long long cap = (long long)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  return (int)(blocks < 1 ? 1 : blocks);
}

int launch_pack_rows(const bf16* in, long long ld_in, const PackPlan& pl, long long row_cap, bf16* out, long long ld_out, int width,
                     cudaStream_t stream) {
  if (width % 8 || ld_in % 8 || ld_out % 8) { set_error("pack_rows: width and strides must be multiples of 8"); return -2; }
  (void)launch_k(pack_rows_kernel, dim3(row_copy_grid(row_cap, width)), dim3(256), 0, stream, in, ld_in, pl.src, pl.cu + pl.B, out, ld_out, width);
  return check_cuda(cudaGetLastError(), "pack_rows launch");
}

int launch_unpack_rows(const bf16* packed, long long ld_p, const PackPlan& pl, bf16* out, long long ld_out, int width,
                       cudaStream_t stream) {
  if (width % 8 || ld_p % 8 || ld_out % 8) { set_error("unpack_rows: width and strides must be multiples of 8"); return -2; }
  const long long rows = (long long)pl.B * pl.N;
  (void)launch_k(unpack_rows_kernel, dim3(row_copy_grid(rows, width)), dim3(256), 0, stream, packed, ld_p, pl.rel, pl.cu, out, ld_out, rows, pl.N, width);
  return check_cuda(cudaGetLastError(), "unpack_rows launch");
}

}  // namespace vtk
