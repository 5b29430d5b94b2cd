// vtk_ssim.cu -- per-tile SSIM of NaFlex patch batches (the SSIM tile loss of scripts/train_vae.py:328-368), forward and
// backward, read straight from the [B, N, 3p^2] token layout: no canvas is written to HBM.
//
// Definition (oracle/ae_oracle.py: ssim = torchmetrics' StructuralSimilarityIndexMeasure defaults): 11 x 11 gaussian window,
// sigma 1.5, K1 = 0.01, K2 = 0.03, data_range 1, per channel, averaged over the 3 channels and every window position that lies
// entirely inside the tile.  Pixel values are those of unpatchify's canvas (same cell map: masked tokens and cells without a
// token read 0, token 0 is re-scattered into cell 0) mapped to [0, 1]: (v + 1) / 2 for minus_one_to_one, v for zero_to_one.
//
// Forward: one CTA per (tile, 32 x 32 block of window positions).  It stages the block's 42 x 42 pixels of both images (one
// channel at a time) in shared memory, runs the separable gaussian (horizontal, then vertical) for the five moments
// mu_a, mu_b, E[aa], E[bb], E[ab], forms the SSIM map and writes the block's sum.  ssim_reduce_kernel adds a tile's block sums
// in a fixed order (the tile's own block rows and columns), so a tile's value does not depend on the other tiles of the call.
//
// Backward: one CTA per (image, 32 x 32 pixel block).  Nothing is saved by the forward: the CTA recomputes the moments of the
// 42 x 42 window positions whose windows touch its pixels (a 20-px halo of pixels), forms the per-position coefficients
//   c1 = w dS/dmu_a,  c2 = w dS/dE[aa],  c3 = w dS/dE[ab],   w(p) = sum over the tiles t that contain window p of gout[t] / count_t
// (tiles summed in tile order), applies the transposed separable gaussian (the gaussian is symmetric, so it is the same
// correlation) and writes dpred = s (G*c1 + 2 a G*c2 + b G*c3), s = the format's chain-rule factor, into the token layout.
// Overlapping tiles share one pass; pixels outside every tile get 0.  No float atomics anywhere.
#include "vtk_common.cuh"
#include "vtk_kernels.h"

namespace vtk {

namespace {

constexpr int SS_WIN = 11;              // gaussian window
constexpr int SS_BLK = 32;              // window positions (forward) / pixels (backward) per CTA side
constexpr int SS_IN = SS_BLK + SS_WIN - 1;        // 42: pixels per side of a forward block; window positions per side of a backward block
constexpr int SS_IN2 = SS_BLK + 2 * (SS_WIN - 1); // 52: pixels per side of a backward block
constexpr int SS_LIST = 128;            // tiles a backward CTA gathers per round
constexpr float SS_C1 = 0.01f * 0.01f, SS_C2 = 0.03f * 0.03f;

// exp(-(k - 5)^2 / (2 * 1.5^2)) normalised to sum 1, computed in float64 and rounded to fp32 (symmetric: g[k] == g[10 - k])
__constant__ float kGauss[SS_WIN] = {1.028380124e-03f, 7.598758209e-03f, 3.600077331e-02f, 1.093606874e-01f, 2.130055428e-01f,
                                     2.660117149e-01f, 2.130055428e-01f, 1.093606874e-01f, 3.600077331e-02f, 7.598758209e-03f,
                                     1.028380124e-03f};

constexpr size_t SS_BWD_SMEM = sizeof(float) * (2 * SS_IN2 * SS_IN2 + 5 * SS_IN2 * SS_IN + 3 * SS_IN * SS_IN + SS_IN * SS_IN) +
                               sizeof(int) * SS_LIST;

__device__ __forceinline__ float ss_load(const void* p, int dtype, long long i) {
  if (dtype == 0) return __ldg(reinterpret_cast<const float*>(p) + i);
  return __uint_as_float((uint32_t)__ldg(reinterpret_cast<const unsigned short*>(p) + i) << 16);
}

// element offset of channel ch of canvas pixel (y, x) of image b in the token layout, or -1 where unpatchify's canvas reads 0
__device__ __forceinline__ long long ss_offset(const SsimArgs& a, int b, int ch, int y, int x) {
  if (y < 0 || x < 0 || b < 0 || b >= a.B) return -1;
  const int p = a.patch, r = y / p, c = x / p;
  if (r >= a.gy || c >= a.gx) return -1;
  const int cell = r * a.gx + c;
  // unpatchify_kernel's lookup: token 0 is re-scattered into cell 0 after the main scatter (ops.py:332-333)
  const int tok = (cell == 0) ? (a.patch_mask[(long long)b * a.N] ? 0 : -1) : a.cell_map[(long long)b * a.gy * a.gx + cell];
  if (tok < 0) return -1;
  return ((long long)b * a.N + tok) * 3 * p * p + (long long)ch * p * p + (y - r * p) * p + (x - c * p);
}

__device__ __forceinline__ float ss_map(float v, int fmt) { return fmt == 0 ? (v + 1.f) * 0.5f : v; }

// pixels [y0, y0 + rows) x [x0, x0 + cols) of channel ch of both images -> sa / sb (row pitch cols), mapped to [0, 1]
__device__ __forceinline__ void ss_stage(const SsimArgs& a, int b, int ch, int y0, int x0, int rows, int cols, float* sa, float* sb) {
  for (int i = threadIdx.x; i < rows * cols; i += blockDim.x) {
    const int r = i / cols, c = i - r * cols;
    const long long o = ss_offset(a, b, ch, y0 + r, x0 + c);
    const float va = o >= 0 ? ss_load(a.pred, a.pred_dtype, o) : 0.f;
    const float vb = o >= 0 ? ss_load(a.target, a.target_dtype, o) : 0.f;
    sa[i] = ss_map(va, a.format);
    sb[i] = ss_map(vb, a.format);
  }
}

// horizontal gaussian pass of the five moments: sh[m][r][j] for rows [0, rows), window columns [0, outc) (pixel columns j..j+10)
__device__ __forceinline__ void ss_hpass(const float* sa, const float* sb, int rows, int inc, int outc, float* sh) {
  const int plane = rows * outc;
  for (int i = threadIdx.x; i < plane; i += blockDim.x) {
    const int r = i / outc, j = i - r * outc;
    const float* pa = sa + r * inc + j;
    const float* pb = sb + r * inc + j;
    float m0 = 0.f, m1 = 0.f, m2 = 0.f, m3 = 0.f, m4 = 0.f;
#pragma unroll
    for (int k = 0; k < SS_WIN; ++k) {
      const float g = kGauss[k], x = pa[k], y = pb[k];
      m0 = fmaf(g, x, m0);
      m1 = fmaf(g, y, m1);
      m2 = fmaf(g * x, x, m2);
      m3 = fmaf(g * y, y, m3);
      m4 = fmaf(g * x, y, m4);
    }
    sh[i] = m0; sh[plane + i] = m1; sh[2 * plane + i] = m2; sh[3 * plane + i] = m3; sh[4 * plane + i] = m4;
  }
}

// vertical gaussian pass at window position (r, j) of the horizontal moments sh ([5][rows][cols])
__device__ __forceinline__ void ss_vpass(const float* sh, int rows, int cols, int r, int j, float (&m)[5]) {
  const int plane = rows * cols;
#pragma unroll
  for (int q = 0; q < 5; ++q) m[q] = 0.f;
#pragma unroll
  for (int k = 0; k < SS_WIN; ++k) {
    const float g = kGauss[k];
    const float* s = sh + (r + k) * cols + j;
#pragma unroll
    for (int q = 0; q < 5; ++q) m[q] = fmaf(g, s[q * plane], m[q]);
  }
}

struct SsTerms {
  float a1, a2, b1, b2;
};
__device__ __forceinline__ SsTerms ss_terms(const float (&m)[5]) {
  const float mab = m[0] * m[1], maa = m[0] * m[0], mbb = m[1] * m[1];
  SsTerms t;
  t.a1 = 2.f * mab + SS_C1;
  t.a2 = 2.f * (m[4] - mab) + SS_C2;
  t.b1 = maa + mbb + SS_C1;
  t.b2 = (m[2] - maa) + (m[3] - mbb) + SS_C2;
  return t;
}

// Fixed-order CTA sum (warp butterfly, then the warps in order); the result is valid in thread 0.
__device__ __forceinline__ float ss_block_sum(float v, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[warp] = v;
  __syncthreads();
  float s = 0.f;
  if (threadIdx.x == 0)
    for (int w = 0; w < nw; ++w) s += red[w];
  return s;
}

__device__ __forceinline__ void tile_of(const SsimArgs& a, int t, int& b, int& y0, int& x0, int& h, int& w) {
  const int* tl = a.tiles + 5 * (long long)t;
  b = tl[0]; y0 = tl[1]; x0 = tl[2]; h = tl[3]; w = tl[4];
}

__host__ __device__ __forceinline__ int ss_blocks(int n) { return (n - (SS_WIN - 1) + SS_BLK - 1) / SS_BLK; }

__global__ void __launch_bounds__(256) ssim_fwd_kernel(const SsimArgs a) {
  pdl_wait();      // PDL (vtk_common.cuh): the cell map is written by the previous kernel of the stream
  pdl_trigger();
  __shared__ float sa[SS_IN * SS_IN], sb[SS_IN * SS_IN];
  __shared__ float sh[5 * SS_IN * SS_BLK];
  __shared__ float red[32];
  const int t = blockIdx.y;
  int b, y0, x0, h, w;
  tile_of(a, t, b, y0, x0, h, w);
  const int nbx_cap = ss_blocks(a.max_tile_w);
  const int by = blockIdx.x / nbx_cap, bx = blockIdx.x - by * nbx_cap;
  const int oh = h - (SS_WIN - 1), ow = w - (SS_WIN - 1);     // window positions of the tile
  if (by * SS_BLK >= oh || bx * SS_BLK >= ow) return;         // outside this tile (the reduction never reads it)
  if (h > a.max_tile_h || w > a.max_tile_w) return;           // a tile the caller's bounds do not cover: the reduction writes NaN
  const int py = by * SS_BLK, px = bx * SS_BLK;
  float acc = 0.f;
  for (int ch = 0; ch < 3; ++ch) {
    __syncthreads();
    ss_stage(a, b, ch, y0 + py, x0 + px, SS_IN, SS_IN, sa, sb);
    __syncthreads();
    ss_hpass(sa, sb, SS_IN, SS_IN, SS_BLK, sh);
    __syncthreads();
    for (int i = threadIdx.x; i < SS_BLK * SS_BLK; i += blockDim.x) {
      const int r = i / SS_BLK, j = i - r * SS_BLK;
      if (py + r >= oh || px + j >= ow) continue;
      float m[5];
      ss_vpass(sh, SS_IN, SS_BLK, r, j, m);
      const SsTerms s = ss_terms(m);
      acc += (s.a1 * s.a2) / (s.b1 * s.b2);
    }
  }
  const float total = ss_block_sum(acc, red);
  if (threadIdx.x == 0) a.partial[(long long)t * gridDim.x + blockIdx.x] = total;
}

// one thread per tile: its block sums in row-major order of the tile's own blocks, in double
__global__ void ssim_reduce_kernel(const SsimArgs a, int blocks_cap) {
  pdl_wait();
  pdl_trigger();
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= a.T) return;
  int b, y0, x0, h, w;
  tile_of(a, t, b, y0, x0, h, w);
  const int nbx_cap = ss_blocks(a.max_tile_w), nby = ss_blocks(h), nbx = ss_blocks(w);
  if (h < SS_WIN || w < SS_WIN || h > a.max_tile_h || w > a.max_tile_w) {   // outside the caller's contract: never read past the sums
    a.out[t] = __int_as_float(0x7fc00000);
    return;
  }
  const float* part = a.partial + (long long)t * blocks_cap;
  double s = 0.0;
  for (int by = 0; by < nby; ++by)
    for (int bx = 0; bx < nbx; ++bx) s += (double)part[by * nbx_cap + bx];
  a.out[t] = (float)(s / (3.0 * (double)(h - (SS_WIN - 1)) * (double)(w - (SS_WIN - 1))));
}

__global__ void __launch_bounds__(256) ssim_bwd_kernel(const SsimArgs a) {
  pdl_wait();      // PDL: the cell map and the zeroed dpred come from the previous operations of the stream
  pdl_trigger();
  extern __shared__ float smem[];
  float* sa = smem;                                   // [52][52] pixels of pred, mapped
  float* sb = sa + SS_IN2 * SS_IN2;                   // [52][52] pixels of target, mapped
  float* sh = sb + SS_IN2 * SS_IN2;                   // [5][52][42] horizontal moments; later [3][42][32] transposed pass
  float* sc = sh + 5 * SS_IN2 * SS_IN;                // [3][42][42] coefficients c1, c2, c3 per window position
  float* sw = sc + 3 * SS_IN * SS_IN;                 // [42][42] w(p)
  int* list = reinterpret_cast<int*>(sw + SS_IN * SS_IN);   // [SS_LIST] tiles of this round
  __shared__ int s_n, s_next;
  const int nbx = (a.gx * a.patch + SS_BLK - 1) / SS_BLK, nby = (a.gy * a.patch + SS_BLK - 1) / SS_BLK;
  const int b = blockIdx.x / (nbx * nby);
  const int rem = blockIdx.x - b * (nbx * nby);
  const int qy = (rem / nbx) * SS_BLK, qx = (rem % nbx) * SS_BLK;   // first pixel of the block
  const int wy = qy - (SS_WIN - 1), wx = qx - (SS_WIN - 1);        // first window position whose window touches it

  for (int i = threadIdx.x; i < SS_IN * SS_IN; i += blockDim.x) sw[i] = 0.f;
  // w(p) for the 42 x 42 window positions [wy, wy + 42) x [wx, wx + 42): warp 0 gathers, in tile order, the tiles of image b
  // whose window positions meet that square (up to SS_LIST per round); every position then adds their weights in list order
  bool any = false;
  int t0 = 0;
  while (t0 < a.T) {
    if (threadIdx.x < 32) {
      const int lane = threadIdx.x;
      int n = 0, t = t0;
      for (; t < a.T && n + 32 <= SS_LIST; t += 32) {
        bool hit = false;
        if (t + lane < a.T) {
          int tb, y0, x0, h, w;
          tile_of(a, t + lane, tb, y0, x0, h, w);
          hit = tb == b && y0 < wy + SS_IN && y0 + h - SS_WIN >= wy && x0 < wx + SS_IN && x0 + w - SS_WIN >= wx;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, hit);
        if (hit) list[n + __popc(bal & ((1u << lane) - 1u))] = t + lane;
        n += __popc(bal);
      }
      if (lane == 0) { s_n = n; s_next = t; }
    }
    __syncthreads();
    const int n = s_n;
    t0 = s_next;
    any = any || n > 0;
    for (int i = threadIdx.x; i < SS_IN * SS_IN && n > 0; i += blockDim.x) {
      const int y = wy + i / SS_IN, x = wx + i % SS_IN;
      float s = sw[i];
      for (int k = 0; k < n; ++k) {
        int tb, y0, x0, h, w;
        tile_of(a, list[k], tb, y0, x0, h, w);
        if (y >= y0 && y <= y0 + h - SS_WIN && x >= x0 && x <= x0 + w - SS_WIN)
          s += a.gout[list[k]] / (3.f * (float)(h - (SS_WIN - 1)) * (float)(w - (SS_WIN - 1)));
      }
      sw[i] = s;
    }
    __syncthreads();
  }
  if (!any) return;                 // no tile reaches these pixels: their gradient is the zero the caller's memset wrote

  const float fscale = a.format == 0 ? 0.5f : 1.f;   // d value / d token element: (v + 1) / 2 or v
  const int Hc = a.gy * a.patch, Wc = a.gx * a.patch;
  constexpr int PC = SS_IN * SS_IN, PT = SS_IN * SS_BLK;
  for (int ch = 0; ch < 3; ++ch) {
    __syncthreads();
    ss_stage(a, b, ch, wy, wx, SS_IN2, SS_IN2, sa, sb);
    __syncthreads();
    ss_hpass(sa, sb, SS_IN2, SS_IN2, SS_IN, sh);
    __syncthreads();
    for (int i = threadIdx.x; i < PC; i += blockDim.x) {
      const float wgt = sw[i];
      float c1 = 0.f, c2 = 0.f, c3 = 0.f;
      if (wgt != 0.f) {
        const int r = i / SS_IN, j = i - r * SS_IN;
        float m[5];
        ss_vpass(sh, SS_IN2, SS_IN, r, j, m);
        const SsTerms s = ss_terms(m);
        // S = N / D with N = a1 a2, D = b1 b2 (b1 >= C1, b2 ~ var_a + var_b + C2 > 0): only D is divided by
        const float inv_d = 1.f / (s.b1 * s.b2), S = s.a1 * s.a2 * inv_d;
        c1 = wgt * 2.f * (m[1] * (s.a2 - s.a1) - S * m[0] * (s.b2 - s.b1)) * inv_d;   // dS / d mu_a
        c2 = -wgt * S * s.b1 * inv_d;                                                // dS / d E[aa]
        c3 = wgt * 2.f * s.a1 * inv_d;                                               // dS / d E[ab]
      }
      sc[i] = c1; sc[PC + i] = c2; sc[2 * PC + i] = c3;
    }
    __syncthreads();
    // transposed gaussian, horizontal: pixel column u gets the window columns u..u+10 (g is symmetric)
    for (int i = threadIdx.x; i < PT; i += blockDim.x) {
      const int r = i / SS_BLK, u = i - r * SS_BLK;
      float g0 = 0.f, g1 = 0.f, g2 = 0.f;
#pragma unroll
      for (int k = 0; k < SS_WIN; ++k) {
        const float g = kGauss[k];
        const float* c = sc + r * SS_IN + u + k;
        g0 = fmaf(g, c[0], g0); g1 = fmaf(g, c[PC], g1); g2 = fmaf(g, c[2 * PC], g2);
      }
      sh[i] = g0; sh[PT + i] = g1; sh[2 * PT + i] = g2;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < SS_BLK * SS_BLK; i += blockDim.x) {
      const int v = i / SS_BLK, u = i - v * SS_BLK;
      const int y = qy + v, x = qx + u;
      if (y >= Hc || x >= Wc) continue;
      const long long o = ss_offset(a, b, ch, y, x);
      if (o < 0) continue;
      float g0 = 0.f, g1 = 0.f, g2 = 0.f;
#pragma unroll
      for (int k = 0; k < SS_WIN; ++k) {
        const float g = kGauss[k];
        const float* c = sh + (v + k) * SS_BLK + u;
        g0 = fmaf(g, c[0], g0); g1 = fmaf(g, c[PT], g1); g2 = fmaf(g, c[2 * PT], g2);
      }
      const int px = (v + SS_WIN - 1) * SS_IN2 + u + SS_WIN - 1;
      const float d = fscale * (g0 + 2.f * sa[px] * g1 + sb[px] * g2);
      if (a.pred_dtype == 0) reinterpret_cast<float*>(a.dpred)[o] = d;
      else reinterpret_cast<bf16*>(a.dpred)[o] = __float2bfloat16_rn(d);
    }
  }
}

}  // namespace

size_t ssim_workspace_bytes(int B, int gy, int gx, int T, int max_tile_h, int max_tile_w) {
  if (B <= 0 || gy <= 0 || gx <= 0 || T <= 0 || max_tile_w < SS_WIN || max_tile_h < SS_WIN) return 0;
  const size_t cells = ((size_t)B * gy * gx * sizeof(int) + 255) / 256 * 256;
  return cells + (size_t)T * ss_blocks(max_tile_h) * ss_blocks(max_tile_w) * sizeof(float);
}

int launch_ssim(const SsimArgs& in, bool backward, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  if (in.B <= 0 || in.N <= 0 || in.T <= 0) { set_error("ssim: empty batch or no tiles (B=%d, N=%d, T=%d)", in.B, in.N, in.T); return -2; }
  if (in.patch <= 0 || in.gy <= 0 || in.gx <= 0) { set_error("ssim: bad patch %d or canvas grid %dx%d", in.patch, in.gy, in.gx); return -2; }
  if (in.max_tile_h < SS_WIN || in.max_tile_w < SS_WIN) {
    set_error("ssim: tiles must be at least %d px on each side (max_tile_h=%d, max_tile_w=%d)", SS_WIN, in.max_tile_h, in.max_tile_w);
    return -2;
  }
  if (in.T > 65535) { set_error("ssim: at most 65535 tiles per call (got %d)", in.T); return -2; }
  const size_t need = ssim_workspace_bytes(in.B, in.gy, in.gx, in.T, in.max_tile_h, in.max_tile_w);
  if (workspace_bytes < need) { set_error("ssim: workspace of %zu bytes, %zu needed", workspace_bytes, need); return -2; }
  const long long blocks_bwd = (long long)in.B * ((in.gy * in.patch + SS_BLK - 1) / SS_BLK) * ((in.gx * in.patch + SS_BLK - 1) / SS_BLK);
  if (backward && blocks_bwd >= (1ll << 31)) { set_error("ssim: canvas too large"); return -2; }
  SsimArgs a = in;
  a.cell_map = reinterpret_cast<int*>(workspace);
  a.partial = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + ((size_t)in.B * in.gy * in.gx * sizeof(int) + 255) / 256 * 256);
  UnpatchifyArgs u{};
  u.patches = in.pred; u.dtype = in.pred_dtype; u.patch_mask = in.patch_mask; u.row_idx = in.row_idx; u.col_idx = in.col_idx;
  u.B = in.B; u.N = in.N; u.patch = in.patch; u.gy = in.gy; u.gx = in.gx; u.cell_map = a.cell_map; u.status = nullptr;
  if (int rc = launch_cellmap(u, st)) return rc;
  if (!backward) {
    const int blocks_cap = ss_blocks(in.max_tile_h) * ss_blocks(in.max_tile_w);
    (void)launch_k(ssim_fwd_kernel, dim3((unsigned)blocks_cap, (unsigned)in.T), dim3(256), 0, st, a);
    (void)launch_k(ssim_reduce_kernel, dim3((unsigned)((in.T + 127) / 128)), dim3(128), 0, st, a, blocks_cap);
    return check_cuda(cudaGetLastError(), "ssim forward launch");
  }
  const size_t nelem = (size_t)in.B * in.N * 3 * in.patch * in.patch;
  if (check_cuda(cudaMemsetAsync(a.dpred, 0, nelem * (in.pred_dtype == 0 ? 4 : 2), st), "ssim dpred memset")) return -1;
  if (int rc = ensure_max_smem((const void*)ssim_bwd_kernel, (int)SS_BWD_SMEM, "ssim backward smem")) return rc;
  (void)launch_k(ssim_bwd_kernel, dim3((unsigned)blocks_bwd), dim3(256), SS_BWD_SMEM, st, a);
  return check_cuda(cudaGetLastError(), "ssim backward launch");
}

}  // namespace vtk
