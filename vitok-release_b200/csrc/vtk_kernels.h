// vtk_kernels.h -- internal (C++) launch interface between the C-ABI layer (vtk_api.cu) and the
// kernels.  Nothing here is exported; the exported surface is include/vitok_b200.h.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace vtk {

typedef __nv_bfloat16 bf16;

// error plumbing (vtk_api.cu)
void set_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);
int num_sms();
int usable_sms();   // num_sms() minus the "reserve_sms" flag: grid size of the persistent kernels

// Kernel launch with programmatic dependent launch (PDL, vtk_common.cuh: pdl_wait / pdl_trigger): the kernel's prologue
// overlaps the tail of the previous kernel of the stream.  Works inside CUDA-graph capture (programmatic edges).  Only for
// kernels that call pdl_wait() before their first access to global memory.  VTK_PDL=0 launches them fully serialised.
bool pdl_enabled();
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel, device): the attribute is per device, and one process may drive
// several GPUs (a model on cuda:1 while cuda:0 is current, torch DataParallel-style callers)
int ensure_max_smem(const void* kern, int bytes, const char* what);
int current_device();
// runtime switches (include/vitok_b200.h: vtk_set_flag)
int flag_gemm_splitk();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// Encode a 2-D bf16 row-major tensor map with 128-byte swizzle: inner box = 64 elements.
int encode_tmap_bf16_sw128(CUtensorMap* out, const void* base, uint64_t inner_elems, uint64_t rows,
                           uint64_t row_stride_elems, uint32_t box_rows);
// fp8 (1-byte elements): inner box = 128 elements, 128-byte swizzle
int encode_tmap_u8_sw128(CUtensorMap* out, const void* base, uint64_t inner_elems, uint64_t rows, uint64_t row_stride_bytes,
                         uint32_t box_rows);
// General form: box = box_inner x box_rows elements, swizzle_bytes in {0, 32, 64, 128} (box_inner * 2 <= swizzle span).
int encode_tmap_bf16(CUtensorMap* out, const void* base, uint64_t inner_elems, uint64_t rows, uint64_t row_stride_elems,
                     uint32_t box_inner, uint32_t box_rows, int swizzle_bytes);
// Attention head tiles: a 3-D bf16 map {d, heads, rows} with byte strides {2d, 2 * row_stride_elems}, box {64, 1, box_rows},
// 128-byte swizzle.  Box columns at or past d (a head narrower than its 64-column tile block) load as zeros and are never stored.
int encode_tmap_heads(CUtensorMap* out, const void* base, int d, int heads, uint64_t rows, uint64_t row_stride_elems, uint32_t box_rows);

// Head dims of the attention kernels and the block path: d % 8 == 0 (a TMA stride is a multiple of 16 bytes) and d <= 128 (the
// d = 128 kernel already uses all 512 TMEM columns).  A head runs on the kernel of the next tile width, 64 or 128.
__host__ __device__ inline bool head_dim_supported(int d) { return d >= 8 && d <= 128 && d % 8 == 0; }
__host__ __device__ inline int head_tile(int d) { return d <= 64 ? 64 : 128; }
// QKV GEMM epilogue: QK-norm + RoPE run inside it for these d only (its walk over a tile's heads needs whole heads per 64- or
// d-column unit); at other head dims it copies q and k raw and launch_qk_norm_rope_fwd normalises them in place.
__host__ __device__ inline bool qk_norm_fused(int d) { return d == 32 || d == 64 || d == 128; }

// ---------------------------------------------------------------------------------------------
// GEMM  out = epilogue(A[M,K] * B[N,K]^T), bf16 in, fp32 accumulate in TMEM (vtk_gemm.cu)
// ---------------------------------------------------------------------------------------------
enum EpiKind {
  EPI_BIAS = 0,        // out = bf16(acc + bias)            (bias may be null)
  EPI_BIAS_LN = 1,     // out = LN_noaffine(bf16(acc+bias)) over the N (= C <= 256) columns
  EPI_QKV_SWIGLU = 2,  // packed [q|k|v|pad|(v16,g16)*] columns: QK-RMSNorm + 2D RoPE, V copy, SwiGLU gate
  EPI_RESID = 3,       // x = bf16(x + bf16(bf16(acc) * gamma))   (in place on out)
};

struct EpiParams {
  bf16* out;            // EPI_BIAS / EPI_BIAS_LN: [M, N]; EPI_RESID: x (read + written)
  long long ldo;        // row stride of out (elements)
  const bf16* bias;     // [N] or null
  float eps;
  // EPI_QKV_SWIGLU
  bf16* qkv;            // [M, 3D]
  long long ld_qkv;
  bf16* act;            // [M, Hf] view (row stride ld_act)
  long long ld_act;
  const bf16* normq;    // [d]
  const bf16* normk;    // [d]
  const bf16* rope;     // pair-expanded chunk-major table [ceil(M/32)*32, 2d] (see rope_table_kernel)
  int D, d, Hf, qp;     // qp = 3D rounded up to the tile width (start of the SwiGLU columns)
  // EPI_RESID
  const bf16* gamma;    // [N]
  // Fused Block.norm1 (norm.py:17-25): instead of a separate RMSNorm pass the producer of x (EPI_BIAS / EPI_RESID) also
  // writes, per row, the sum of squares of its bf16 outputs for every 64-column unit (ss_out[row * ss_ld + col / 64];
  // fixed summation order, no atomics), and the consumer (EPI_QKV_SWIGLU, whose weight has norm1.weight folded into its
  // columns) multiplies each accumulator row by rsqrt(sum(ss_in[row, 0..ss_units)) * ss_inv_d + eps) before anything else.
  float* ss_out; int ss_ld;
  const float* ss_in; int ss_units; float ss_inv_d;
  // FP8 operands (GemmArgs::fp8): every accumulator row is multiplied by a_scale[row] * w_scale (per-row activation scale
  // of the dynamic quantisation x per-tensor weight scale) before anything else, on top of the fused-norm1 scale
  const float* a_scale; float w_scale;
  int accumulate;       // EPI_BIAS: out = bf16(acc + bias + float(out)) -- the GEMM adds to what `out` already holds
  int k_split;          // > 0 (pair kernel, EPI_BIAS, K-major operands): k-blocks at or beyond k_split read their B tile from the
                        // SECOND weight matrix (GemmArgs::B2, k coordinate - k_split): out = A[:, :k_split] B^T + A[:, k_split:] B2^T
                        // in one accumulator -- [out_proj | fc2] without a packed copy (training forward); a multiple of 64
  const int* m_dev;     // optional: number of rows to process, read on the device (<= GemmArgs::M, which is then the row
                        // capacity of the buffers); used by the packed NaFlex path where sum(n_i) is only known on the GPU
  unsigned long long* prof;  // perf experiments only (env VTK_GEMM_PROF): per-role clock64 accumulators, or null
};

struct GemmArgs {
  const bf16* A; long long lda;   // [M, K], row stride lda
  const bf16* B; long long ldb;   // [N_rows, K], row stride ldb (N_rows may be < N: OOB rows read as 0)
  long long b_rows;
  const bf16* B2; long long ldb2;   // second weight matrix [N_rows, K - k_split] (EpiParams::k_split > 0), else null
  int M, N, K;                    // N = number of output (packed) columns to cover
  int trans;                      // 3: A is [K, M] and B is [K, N] row-major (out = A^T B); 2: only B is [K, N] (out = A B); CTA-pair kernel, EPI_BIAS
  int fp8;                        // 1: A and B hold e4m3 bytes (lda / ldb / K in elements = bytes); CTA-pair kernel only
  EpiParams epi;
};

int launch_gemm(EpiKind kind, const GemmArgs& a, cudaStream_t stream);

// descriptor probe (tests only): D[128, N] fp32 = A[128,K] * op(B); b_mn_major selects B = [K, N] row-major.
int launch_umma_probe(const bf16* A, const bf16* B, float* D, int N, int K, int b_mn_major, uint32_t lbo_bytes,
                      uint32_t sbo_bytes, uint32_t kstep_bytes, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------
// attention (vtk_attention.cu): softmax(q k^T / sqrt(d)) v per (image, head); q/k/v rows are
// [B*N, ld] with heads along columns.  kv_len[b] = number of leading key rows to visit (null = N).
// ---------------------------------------------------------------------------------------------
struct AttnArgs {
  const bf16* q; const bf16* k; const bf16* v; long long ld_qkv;  // row stride (elements)
  bf16* out; long long ld_out;
  const int* kv_len;            // [B] or null
  int B, N, heads, d;
  int zero_invalid_rows;        // 1: rows >= kv_len[b] are written as 0 (packed: the image's pad rows)
  int window;                   // sliding window: keys j with |i - j| <= window (flash_attn window_size=(w,w)); < 0 = none
  float* lse;                   // optional [B*N, heads] fp32: log2-domain logsumexp of the scaled scores (for the backward pass)
  // packed NaFlex layout (PackPlan): rows of image b start at cu[b] and hold kv_len[b] valid tokens; work group g
  // (128 query rows at d = 64, 256 at d = 128) belongs to image grp_img[g] and is the (g - cuq[grp_img[g]])-th of that image
  const int* cu = nullptr; const int* cuq = nullptr; const int* grp_img = nullptr; const int* grp_order = nullptr;
  long long row_cap = 0;   // rows of the q / k / v / out buffers
  int grp_cap = 0;         // capacity of the group arrays (grid size of the one-shot kernel)
};
int launch_attention(const AttnArgs& a, cudaStream_t stream);

// attention backward (vtk_attention_bwd.cu): dq, dk, dv [B*N, ld_d] from q, k, v, dO, lse (log2 domain) and
// delta = rowsum(dO * O).  Same masking arguments as the forward.
struct AttnBwdArgs {
  const bf16* q; const bf16* k; const bf16* v; long long ld_qkv;
  const bf16* dout; long long ld_do;
  const float* lse; const float* delta;   // [B*N, heads] (packed: [row_cap, heads])
  bf16* dq; bf16* dk; bf16* dv; long long ld_d;
  const int* kv_len;
  int B, N, heads, d, zero_invalid_rows, window;
  // packed NaFlex layout (PackPlan with qrows = 128): image b = rows [cu[b], cu[b+1]) with kv_len[b] valid tokens in front; one CTA
  // per (128-row group, head) of each pass, groups taken in grp_order
  const int* cu = nullptr; const int* cuq = nullptr; const int* grp_img = nullptr; const int* grp_order = nullptr;
  long long row_cap = 0;   // rows of the q / k / v / dO / dq / dk / dv buffers
  int grp_cap = 0;         // groups the grid covers (>= cuq[B]; CTAs beyond cuq[B] exit at once)
};
int launch_attention_bwd(const AttnBwdArgs& a, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------
// elementwise / HBM-bound kernels (vtk_elementwise.cu)
// ---------------------------------------------------------------------------------------------
// m_dev (optional): row count read on the device (M is then the capacity); src_map (optional): table row -> source token
int launch_rmsnorm(const bf16* x, long long ldx, const bf16* w, bf16* y, long long ldy, int M, int D, float eps,
                   cudaStream_t stream, const int* m_dev = nullptr);
int launch_rope_table(const int64_t* row_idx, const int64_t* col_idx, const float* inv_freq, bf16* table, int M, int d,
                      cudaStream_t stream, const int* src_map = nullptr, const int* m_dev = nullptr);

// NaFlex token packing (vtk_elementwise.cu): valid tokens of a masked [B, N] batch packed image after image, each image
// padded to `pad` rows (16: row tiles of the GEMMs may straddle images; only 16-byte alignment of the rows matters).
// Attention works on groups of `qrows` query rows of one image (128, or 256 for the two-tile CTAs of d = 128); a group's
// last tile may be partial -- its rows beyond n_valid belong to the next image and are neither attended to (keys are
// masked by n_valid) nor stored.  All arrays live in device memory (carved from the caller's workspace).
struct PackPlan {
  int B, N;
  int pad = 16;     // rows every image is padded to in the packed layout
  int qrows = 128;  // query rows per attention work group
  int* n_valid;    // [B]      valid tokens per image (= key count of the image in the packed layout)
  int* rel;        // [B * N]  rank of a token among the valid tokens of its image, -1 if masked
  int* cu;         // [B + 1]  packed row offset per image; cu[B] = packed row count (the m_dev of every kernel)
  int* cuq;        // [B + 1]  first attention group of each image; cuq[B] = number of groups
  int* grp_img;    // [B * ceil(N / qrows)]  image of each group
  int* grp_order;  // [B * ceil(N / qrows)]  groups sorted by key tiles of their image, longest first (attention work list)
  int* src;        // [row capacity]         packed row -> source row b * N + t, -1 for pad rows
  const int* m_dev() const { return cu + B; }
  const int* n_groups() const { return cuq + B; }
  static long long row_capacity(int B, int N, int pad = 16) { return (long long)B * ((N + pad - 1) / pad * pad); }
  static long long group_capacity(int B, int N, int qrows) { return (long long)B * ((N + qrows - 1) / qrows); }
};
int launch_pack_plan(const uint8_t* mask, int B, int N, const PackPlan& pl, cudaStream_t stream);
int launch_pack_rows(const bf16* in, long long ld_in, const PackPlan& pl, long long row_cap, bf16* out, long long ld_out, int width,
                     cudaStream_t stream);
int launch_unpack_rows(const bf16* packed, long long ld_p, const PackPlan& pl, bf16* out, long long ld_out, int width,
                       cudaStream_t stream);
int launch_cast_f32_bf16(const float* in, bf16* out, long long n, cudaStream_t stream);
// dynamic per-row FP8 (e4m3) quantisation: q[row, :K] = e4m3(x[row, :K] / scale[row]), scale[row] = amax(row) / 448
// amax_ws (optional, one device float): per-TENSOR scale instead (amax of the whole tensor, torchao's default granularity)
int launch_quant_rows_e4m3(const bf16* x, long long ldx, uint8_t* q, long long ldq, float* scale, int M, int K, const int* m_dev,
                           cudaStream_t stream, float* amax_ws = nullptr);
int launch_kv_len(const uint8_t* mask, int* kv_len, int B, int N, cudaStream_t stream);

// ---------------------------------------------------------------------------------------------
// NaFlex pre/post-processing (vtk_pp.cu)
// ---------------------------------------------------------------------------------------------
struct PatchifyArgs {
  const void* images;          // base pointer of the packed image buffer
  const int64_t* img_table;    // device [B, 3] = {element offset, H, W}
  int in_dtype;                // 0 = fp32 CHW (already normalised), 1 = uint8 HWC (to_tensor|normalize fused)
  int B, patch, max_tokens;
  int out_dtype;               // 0 = fp32, 1 = bf16
  void* patches;               // [B, T, 3 p^2]
  uint8_t* patch_mask;         // [B, T]
  int64_t* row_idx; int64_t* col_idx; int64_t* time_idx;  // [B, T]
  int64_t* meta;               // [4, B] = orig_height, orig_width, grid_rows, grid_cols
  int* status;                 // device int: set to 1 if any grid exceeds max_tokens
  int max_h = 0, max_w = 0;    // optional: largest image height / width of the batch (host knowledge); > 0 selects the row-coalesced
                               // uint8 kernel, which walks the batch's bounding box
};
int launch_patchify(const PatchifyArgs& a, cudaStream_t stream);
int launch_patchify_selftest(int* mismatches, cudaStream_t stream);   // norm_u8_fast == norm_u8 for all 256 inputs

// resize to the token budget + patchify (vtk_pp.cu).  img_table [B, 5] = {element offset, H, W, h', w'}.  The workspace holds a
// header (per-image offsets, computed on the device) and, per image, its resample tables and width-pass scratch image.
// Table of one axis n_in -> n_out: [resize_kt + 2][n_out] floats, tap-major: row 0 = xmin, row 1 = taps (int bits), then the
// weights (zero beyond the tap count); resize_kt bounds
// ATen's ceil(support) * 2 + 1 taps (support = 2 * n_in / n_out when shrinking, 2 otherwise).
__host__ __device__ inline int resize_kt(int n_in, int n_out) { return 4 * ((n_in + n_out - 1) / n_out) + 1; }
struct ResizeImage {
  long long off;
  int H, W, h, w;   // source size, target size
  __host__ __device__ bool sized() const { return H >= 1 && W >= 1 && h >= 1 && w >= 1; }
  __host__ __device__ long long table_floats() const {
    if (!sized()) return 0;
    return (w != W ? (long long)w * (resize_kt(W, w) + 2) : 0) + (h != H ? (long long)h * (resize_kt(H, h) + 2) : 0);
  }
  __host__ __device__ long long width_rows() const { return sized() && w != W ? H : 0; }
  __host__ __device__ long long region_floats() const { return table_floats() + 3 * width_rows() * (sized() ? w : 0); }
};
__host__ __device__ inline ResizeImage resize_image(const int64_t* tab, int b) {
  const int64_t* r = tab + 5 * (long long)b;
  return ResizeImage{(long long)r[0], (int)r[1], (int)r[2], (int)r[3], (int)r[4]};
}
__host__ __device__ inline size_t resize_header_bytes(int B) { return ((size_t)(2 * B + 3) * 8 + 255) / 256 * 256; }
struct ResizePatchifyArgs {
  const void* images; const int64_t* img_table;
  int in_dtype, B, patch, max_tokens, out_dtype;
  void* patches; uint8_t* patch_mask; int64_t* row_idx; int64_t* col_idx; int64_t* time_idx; int64_t* meta;
  void* workspace; size_t workspace_bytes;
  int* status;   // 1: a target grid exceeds max_tokens; 2: a size < 1 or the workspace is too small
};
int launch_resize_patchify(const ResizePatchifyArgs& a, cudaStream_t stream);
size_t resize_workspace_bytes(const int64_t* img_table_host, int B);

struct UnpatchifyArgs {
  const void* patches;         // [B, N, 3 p^2]
  int dtype;                   // 0 fp32, 1 bf16
  const uint8_t* patch_mask; const int64_t* row_idx; const int64_t* col_idx;  // [B, N]
  int B, N, patch, gy, gx;
  int* cell_map;               // workspace [B, gy*gx] int32
  void* out;                   // [B, 3, gy*p, gx*p], same dtype unless out_u8
  int out_format;              // 0 = same dtype, no conversion; 1 = uint8 "0_255" from minus_one_to_one;
                               // 2 = zero_to_one from minus_one_to_one (same dtype)
  int* status;                 // set to 1 when a valid token falls outside the canvas
};
int launch_unpatchify(const UnpatchifyArgs& a, cudaStream_t stream);
// unpatchify's cell -> token map alone (memset to -1, then the scatter of the valid tokens); uses patch_mask, row_idx, col_idx,
// B, N, gy, gx, cell_map and status of `a`
int launch_cellmap(const UnpatchifyArgs& a, cudaStream_t stream);
int launch_grid_extent(const uint8_t* mask, const int64_t* row, const int64_t* col, int B, int N, int* out2,
                       cudaStream_t stream);

// ---------------------------------------------------------------------------------------------
// training step (vtk_train.cu, vtk_attention_bwd.cu)
// ---------------------------------------------------------------------------------------------
int launch_qk_norm_rope_fwd(const bf16* zraw, long long ldz, const bf16* wq, const bf16* wk, const bf16* rope, bf16* qkv,
                            long long ldq, int M, int heads, int d, float eps, cudaStream_t st);
int launch_swiglu_fwd(const bf16* zraw, long long ldz, int qp, bf16* act, long long lda, int M, int Hf, int layout, cudaStream_t st);
int launch_resid_fwd(const bf16* x, const bf16* y, const bf16* gamma, bf16* out, int M, int D, cudaStream_t st,
                     const float* keep = nullptr, int rows_per_img = 0, float keep_prob = 1.f);
int launch_ln_fwd(const bf16* x, bf16* out, int M, int C, float eps, cudaStream_t st);
int launch_resid_bwd(const bf16* dx, const bf16* y, const bf16* gamma, bf16* dy, float* dgamma, int M, int D, cudaStream_t st,
                     const float* keep = nullptr, int rows_per_img = 0, float keep_prob = 1.f);
int launch_colsum(const bf16* in, long long ld, float* out, int M, int C, cudaStream_t st);
int launch_swiglu_bwd(const bf16* dact, long long ldd, const bf16* zraw, long long ldz, int qp, bf16* dz, long long lddz, int M,
                      int Hf, int layout, cudaStream_t st);
int launch_qk_norm_rope_bwd(bf16* dz, long long lddz, const bf16* zraw, long long ldz, const bf16* wq, const bf16* wk,
                            const bf16* rope, float* dw, int M, int heads, int d, float eps, cudaStream_t st);
int launch_rmsnorm_bwd(const bf16* x, const bf16* dh, const bf16* w, const bf16* dx_res, bf16* dx_out, float* dw, int M, int D,
                       float eps, cudaStream_t st);
int launch_ln_bwd(const bf16* zlin, const bf16* dz, bf16* dx, int M, int C, float eps, cudaStream_t st);
int launch_charbonnier(const bf16* pred, const bf16* target, const uint8_t* mask, const int* n_valid, float* loss_sum, bf16* dpred,
                       int B, int N, int P, float eps, cudaStream_t st);
// per-tile SSIM on the token layout (vtk_ssim.cu; include/vitok_b200.h: vtk_ssim_fwd / vtk_ssim_bwd)
struct SsimArgs {
  const void* pred; int pred_dtype;       // [B, N, 3 p^2], 0 = fp32, 1 = bf16
  const void* target; int target_dtype;
  const uint8_t* patch_mask; const int64_t* row_idx; const int64_t* col_idx;   // [B, N]
  int B, N, patch, gy, gx;                // canvas grid (unpatchify's)
  const int* tiles; int T;                // [T, 5] int32 (image, y0, x0, h, w)
  int max_tile_h, max_tile_w;             // bounds of the tiles' h / w (size the forward grid and workspace)
  int format;                             // 0 = minus_one_to_one, 1 = zero_to_one
  float* out;                             // forward: [T] fp32
  const float* gout; void* dpred;         // backward: [T] fp32, [B, N, 3 p^2] in pred's dtype
  int* cell_map = nullptr; float* partial = nullptr;   // carved from the workspace by launch_ssim
};
size_t ssim_workspace_bytes(int B, int gy, int gx, int T, int max_tile_h, int max_tile_w);
int launch_ssim(const SsimArgs& a, bool backward, void* workspace, size_t workspace_bytes, cudaStream_t st);
int launch_attn_delta(const bf16* o, long long ldo, const bf16* dob, long long lddo, float* delta, int M, int heads, int d,
                      cudaStream_t st);
// one tensor of a multi-tensor AdamW step (mirrors vtk_adamw_tensor of include/vitok_b200.h)
struct AdamwTensor {
  float* master; void* p16; const void* g; float* m; float* v; long long n; float weight_decay; int g_is_f32;
};
// ema (optional, one fp32 pointer per tensor) follows the new master with decay ema_decay; coef (optional, device) scales every gradient
int launch_adamw_multi(const AdamwTensor* tensors, float* const* ema, int n_tensors, float lr, float b1, float b2, float eps, int step,
                       float grad_scale, const float* coef, double ema_decay, cudaStream_t st);
long long grad_norm_slots(const AdamwTensor* tensors, int n_tensors);
int launch_grad_sumsq(const AdamwTensor* tensors, int n_tensors, float* partials, cudaStream_t st);
int launch_grad_norm_finish(const float* partials, long long n_slots, float max_norm, float* norm_coef, cudaStream_t st);
int launch_scale_by_dev(bf16* x, const float* scale, long long n, cudaStream_t st);

}  // namespace vtk
