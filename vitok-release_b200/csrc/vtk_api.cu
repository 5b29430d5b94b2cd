// vtk_api.cu -- the exported C ABI (include/vitok_b200.h): argument checking, error plumbing,
// tensor-map encoding, and the AE encode/decode layer loops.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <set>
#include <utility>
#include <vector>

#include "../../include/vitok_b200.h"
#include "vtk_kernels.h"

namespace vtk {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return 0;
  set_error("%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
  return VTK_ERR_CUDA;
}

int num_sms() {   // of the CURRENT device (cached per device: one process may drive several GPUs)
  static int sms[64] = {0};
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return -1;
  if (dev >= 0 && dev < 64 && sms[dev] > 0) return sms[dev];
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
  if (dev >= 0 && dev < 64) sms[dev] = n;
  return n;
}

int current_device() {
  int dev = 0;
  return cudaGetDevice(&dev) == cudaSuccess ? dev : 0;
}

int ensure_max_smem(const void* kern, int bytes, const char* what) {
  static std::mutex mu;
  static std::set<std::pair<const void*, int>> done;
  const int dev = current_device();
  std::lock_guard<std::mutex> lock(mu);
  if (done.count({kern, dev})) return 0;
  const int r = check_cuda(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes), what);
  if (r == 0) done.insert({kern, dev});
  return r;
}

static int g_flag_pdl = -1, g_flag_splitk = -1, g_flag_reserve = -1;
// SMs the persistent kernels (GEMMs, d = 64 attention) may occupy: all of them, minus the ones a concurrent communication kernel needs
// ("reserve_sms": NCCL's all-reduce CTAs run next to the backward GEMMs of the data-parallel training step; a persistent grid sized for
// every SM would leave some of its CTAs waiting for the whole collective to finish before they can start)
int usable_sms() {
  if (g_flag_reserve < 0) g_flag_reserve = getenv("VTK_RESERVE_SMS") ? atoi(getenv("VTK_RESERVE_SMS")) : 0;
  const int n = num_sms() - g_flag_reserve;
  return n < 2 ? 2 : n;
}
bool pdl_enabled() {
  if (g_flag_pdl < 0) g_flag_pdl = getenv("VTK_PDL") ? atoi(getenv("VTK_PDL")) : 1;
  return g_flag_pdl != 0;
}
int flag_gemm_splitk() {
  if (g_flag_splitk < 0) g_flag_splitk = getenv("VTK_GEMM_SPLITK") ? atoi(getenv("VTK_GEMM_SPLITK")) : 1;
  return g_flag_splitk;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !p) {
    set_error("cuTensorMapEncodeTiled entry point unavailable (%s)", cudaGetErrorString(e));
    return nullptr;
  }
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

int encode_tmap_bf16(CUtensorMap* out, const void* base, uint64_t inner_elems, uint64_t rows, uint64_t row_stride_elems,
                     uint32_t box_inner, uint32_t box_rows, int swizzle_bytes) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return VTK_ERR_CUDA;
  cuuint64_t gdim[2] = {inner_elems, rows};
  cuuint64_t gstride[1] = {row_stride_elems * 2};
  cuuint32_t box[2] = {box_inner, box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                                      : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (CUresult %d) base=%p inner=%llu rows=%llu stride=%llu box=%ux%u swizzle=%d",
              (int)r, base, (unsigned long long)inner_elems, (unsigned long long)rows, (unsigned long long)row_stride_elems,
              box_inner, box_rows, swizzle_bytes);
    return VTK_ERR_CUDA;
  }
  return 0;
}

// 2-D row-major tensor of bytes (fp8 e4m3), 128-byte swizzle: inner box = 128 elements = 128 bytes
int encode_tmap_u8_sw128(CUtensorMap* out, const void* base, uint64_t inner_elems, uint64_t rows, uint64_t row_stride_bytes,
                         uint32_t box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return VTK_ERR_CUDA;
  cuuint64_t gdim[2] = {inner_elems, rows};
  cuuint64_t gstride[1] = {row_stride_bytes};
  cuuint32_t box[2] = {128, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(u8) failed (CUresult %d) base=%p inner=%llu rows=%llu stride=%llu box_rows=%u", (int)r, base,
              (unsigned long long)inner_elems, (unsigned long long)rows, (unsigned long long)row_stride_bytes, box_rows);
    return VTK_ERR_CUDA;
  }
  return 0;
}

int encode_tmap_bf16_sw128(CUtensorMap* out, const void* base, uint64_t inner_elems, uint64_t rows,
                           uint64_t row_stride_elems, uint32_t box_rows) {
  return encode_tmap_bf16(out, base, inner_elems, rows, row_stride_elems, 64, box_rows, 128);
}

int encode_tmap_heads(CUtensorMap* out, const void* base, int d, int heads, uint64_t rows, uint64_t row_stride_elems, uint32_t box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return VTK_ERR_CUDA;
  cuuint64_t gdim[3] = {(cuuint64_t)d, (cuuint64_t)heads, rows};
  cuuint64_t gstride[2] = {(cuuint64_t)d * 2, row_stride_elems * 2};
  cuuint32_t box[3] = {64, 1, box_rows};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(heads) failed (CUresult %d) base=%p d=%d heads=%d rows=%llu stride=%llu box_rows=%u", (int)r,
              base, d, heads, (unsigned long long)rows, (unsigned long long)row_stride_elems, box_rows);
    return VTK_ERR_CUDA;
  }
  return 0;
}

// -------------------------------------------------------------------------------------------------
// AE handle
// -------------------------------------------------------------------------------------------------
struct Side {
  int width = 0, depth = 0, heads = 0, hidden = 0;
  const bf16 *w_a = nullptr, *b_a = nullptr, *w_b = nullptr, *b_b = nullptr;
  std::vector<vtk_block_weights> blocks;
  std::vector<vtk_block_fp8> fp8;   // non-empty: the block GEMMs run with e4m3 operands (AE.quantize)
  float* inv_freq = nullptr;  // device, d/4 floats
  bool norm_folded = false;   // w_in has norm1.weight folded into its columns: norm1 runs inside the GEMM epilogues
  int head_dim() const { return heads ? width / heads : 0; }
  int qp() const { return ((3 * width + 255) / 256) * 256; }
  // row pitch of [attn | act] and of the packed [out_proj | fc2]: D + Hf rounded up to 64 elements so every
  // row starts on a 128-byte line (a misaligned pitch makes each 128-byte TMA box row straddle two lines)
  int kp() const { return ((width + hidden + 63) / 64) * 64; }
};

struct Workspace {
  bf16 *x, *h, *qkv, *a2, *rope;
  uint8_t *x8, *a28;    // FP8 inference: e4m3 copies of x and of [attn | act], and their per-row scales
  float *sx, *sa;
  float* amax;          // FP8 per-tensor activation scale: two device floats (x, [attn | act])
  float* ss;            // [rows, D / 64] per-unit sums of squares of x (fused norm1)
  PackPlan plan;        // NaFlex token packing (masked batches): plan arrays + packed input / output staging rows
  bf16 *pin, *pout;
  size_t bytes;
};

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// M = row capacity of the activation buffers = B * ceil128(N) (the packed layout pads every image to 128 rows)
static Workspace carve(const Side& s, void* base, int B, int N, int io_cols) {
  Workspace w;
  size_t off = 0;
  auto take = [&](size_t nbytes) {
    void* p = base ? static_cast<uint8_t*>(base) + off : nullptr;
    off += align_up(nbytes, 1024);
    return p;
  };
  const int qrows = head_tile(s.head_dim()) == 128 ? 256 : 128;   // query rows per attention work group
  const long long M = PackPlan::row_capacity(B, N, 16);   // >= B * N, so it also holds the padded (un-packed) layout
  const long long G = PackPlan::group_capacity(B, N, qrows);
  const long long D = s.width, d = s.head_dim();
  w.x = static_cast<bf16*>(take((size_t)M * D * 2));
  w.h = static_cast<bf16*>(take((size_t)M * D * 2));
  w.qkv = static_cast<bf16*>(take((size_t)M * 3 * D * 2));
  w.a2 = static_cast<bf16*>(take((size_t)M * s.kp() * 2));
  w.rope = static_cast<bf16*>(take((size_t)((M + 31) / 32 * 32) * 2 * d * 2));   // pair-expanded table, 32-row groups
  w.ss = static_cast<float*>(take((size_t)M * ((D + 63) / 64) * 4));
  w.x8 = w.a28 = nullptr; w.sx = w.sa = nullptr; w.amax = nullptr;
  if (!s.fp8.empty()) {
    w.x8 = static_cast<uint8_t*>(take((size_t)M * D));
    w.a28 = static_cast<uint8_t*>(take((size_t)M * s.kp()));
    w.sx = static_cast<float*>(take((size_t)M * 4));
    w.sa = static_cast<float*>(take((size_t)M * 4));
    w.amax = static_cast<float*>(take(1024));
  }
  w.plan.B = B; w.plan.N = N; w.plan.pad = 16; w.plan.qrows = qrows;
  w.plan.n_valid = static_cast<int*>(take((size_t)B * 4));
  w.plan.rel = static_cast<int*>(take((size_t)B * N * 4));
  w.plan.cu = static_cast<int*>(take((size_t)(B + 1) * 4));
  w.plan.cuq = static_cast<int*>(take((size_t)(B + 1) * 4));
  w.plan.grp_img = static_cast<int*>(take((size_t)G * 4));
  w.plan.grp_order = static_cast<int*>(take((size_t)G * 4));
  w.plan.src = static_cast<int*>(take((size_t)M * 4));
  w.pin = static_cast<bf16*>(take((size_t)M * io_cols * 2));
  w.pout = static_cast<bf16*>(take((size_t)M * io_cols * 2));
  w.bytes = off;
  return w;
}

static int io_cols(const vtk_ae_config& c) { return c.pixels_per_token > c.channels_per_token ? c.pixels_per_token : c.channels_per_token; }

}  // namespace vtk

// kernel classes for the optional per-launch CUDA-event timing (bench.py roofline)
enum { CLS_LINEAR = 0, CLS_RMSNORM = 1, CLS_QKV_SWIGLU = 2, CLS_ATTENTION = 3, CLS_PROJ_RESID = 4, CLS_MISC = 5, CLS_COUNT = 6 };

struct vtk_ae_s {
  vtk_ae_config cfg;
  vtk::Side side[2];
  int last_launches = 0;
  bool fp8_per_tensor = false;   // FP8 activations quantised with one dynamic scale per tensor instead of per row (vtk_ae_set_fp8_granularity)
  // timing: one (start, stop) event pair per launch of the last encode/decode call
  bool timing = false;
  std::vector<cudaEvent_t> ev;      // 2 per launch
  std::vector<int> ev_cls;
  int ev_used = 0;
};

// RAII helper: records an event pair around one launch when timing is on
struct LaunchTimer {
  vtk_ae_s* h; cudaStream_t st; int idx = -1;
  LaunchTimer(vtk_ae_s* h_, cudaStream_t st_, int cls) : h(h_), st(st_) {
    if (!h->timing) return;
    if ((size_t)(2 * h->ev_used + 2) > h->ev.size()) {
      for (int i = 0; i < 2; ++i) { cudaEvent_t e; cudaEventCreate(&e); h->ev.push_back(e); }
      h->ev_cls.push_back(cls);
    }
    idx = h->ev_used++;
    h->ev_cls[idx] = cls;
    cudaEventRecord(h->ev[2 * idx], st);
  }
  ~LaunchTimer() { if (idx >= 0) cudaEventRecord(h->ev[2 * idx + 1], st); }
};

using namespace vtk;

#define VTK_REQUIRE(cond, ...)        \
  do {                                \
    if (!(cond)) {                    \
      set_error(__VA_ARGS__);         \
      return VTK_ERR_BAD_ARG;         \
    }                                 \
  } while (0)

extern "C" {

const char* vtk_last_error(void) { return g_err; }
int vtk_abi_version(void) { return VTK_ABI_VERSION; }
int vtk_sm_count(void) { return num_sms(); }

int vtk_set_flag(const char* name, int value) {
  VTK_REQUIRE(name, "vtk_set_flag: null name");
  if (!strcmp(name, "pdl")) { g_flag_pdl = value ? 1 : 0; return VTK_OK; }
  if (!strcmp(name, "gemm_splitk")) { g_flag_splitk = value ? 1 : 0; return VTK_OK; }
  if (!strcmp(name, "reserve_sms")) { g_flag_reserve = value < 0 ? 0 : value; return VTK_OK; }
  set_error("vtk_set_flag: unknown flag '%s' (pdl, gemm_splitk, reserve_sms)", name);
  return VTK_ERR_BAD_ARG;
}

int vtk_patchify_ex(const void* images, const int64_t* img_table, int in_dtype, int B, int patch, int max_tokens, int out_dtype,
                    void* patches, uint8_t* patch_mask, int64_t* row_idx, int64_t* col_idx, int64_t* time_idx, int64_t* meta, int* status,
                    int max_h, int max_w, void* stream) {
  VTK_REQUIRE(images && img_table && patches && patch_mask && row_idx && col_idx && time_idx && meta, "vtk_patchify_ex: null pointer");
  VTK_REQUIRE(in_dtype == 0 || in_dtype == 1, "vtk_patchify_ex: in_dtype must be 0 (f32 CHW) or 1 (u8 HWC)");
  VTK_REQUIRE(out_dtype == 0 || out_dtype == 1, "vtk_patchify_ex: out_dtype must be 0 (f32) or 1 (bf16)");
  VTK_REQUIRE(B >= 0 && max_tokens >= 0 && max_h >= 0 && max_w >= 0, "vtk_patchify_ex: negative size");
  PatchifyArgs a;
  a.images = images; a.img_table = img_table; a.in_dtype = in_dtype; a.B = B; a.patch = patch; a.max_tokens = max_tokens;
  a.out_dtype = out_dtype; a.patches = patches; a.patch_mask = patch_mask; a.row_idx = row_idx; a.col_idx = col_idx;
  a.time_idx = time_idx; a.meta = meta; a.status = status; a.max_h = max_h; a.max_w = max_w;
  return launch_patchify(a, (cudaStream_t)stream);
}

int vtk_resize_patchify(const void* images, const int64_t* img_table, int in_dtype, int B, int patch, int max_tokens, int out_dtype,
                        void* patches, uint8_t* patch_mask, int64_t* row_idx, int64_t* col_idx, int64_t* time_idx, int64_t* meta,
                        void* workspace, size_t workspace_bytes, int* status, void* stream) {
  VTK_REQUIRE(images && img_table && patches && patch_mask && row_idx && col_idx && time_idx && meta && workspace,
              "vtk_resize_patchify: null pointer");
  VTK_REQUIRE(in_dtype == 0 || in_dtype == 1, "vtk_resize_patchify: in_dtype must be 0 (f32 CHW) or 1 (u8 HWC)");
  VTK_REQUIRE(out_dtype == 0 || out_dtype == 1, "vtk_resize_patchify: out_dtype must be 0 (f32) or 1 (bf16)");
  VTK_REQUIRE(B >= 0 && max_tokens >= 0, "vtk_resize_patchify: negative size");
  ResizePatchifyArgs a;
  a.images = images; a.img_table = img_table; a.in_dtype = in_dtype; a.B = B; a.patch = patch; a.max_tokens = max_tokens;
  a.out_dtype = out_dtype; a.patches = patches; a.patch_mask = patch_mask; a.row_idx = row_idx; a.col_idx = col_idx;
  a.time_idx = time_idx; a.meta = meta; a.workspace = workspace; a.workspace_bytes = workspace_bytes; a.status = status;
  return launch_resize_patchify(a, (cudaStream_t)stream);
}

size_t vtk_resize_patchify_workspace_bytes(const int64_t* img_table_host, int B) {
  if (!img_table_host || B <= 0) return 0;
  return resize_workspace_bytes(img_table_host, B);
}

int vtk_patchify_selftest(int* mismatches, void* stream) {
  VTK_REQUIRE(mismatches, "vtk_patchify_selftest: null pointer");
  return launch_patchify_selftest(mismatches, (cudaStream_t)stream);
}

int vtk_grid_extent(const uint8_t* patch_mask, const int64_t* row_idx, const int64_t* col_idx, int B, int N, int* out2,
                    void* stream) {
  VTK_REQUIRE(patch_mask && row_idx && col_idx && out2, "vtk_grid_extent: null pointer");
  return launch_grid_extent(patch_mask, row_idx, col_idx, B, N, out2, (cudaStream_t)stream);
}

int vtk_unpatchify(const void* patches, int dtype, const uint8_t* patch_mask, const int64_t* row_idx,
                   const int64_t* col_idx, int B, int N, int patch, int gy, int gx, int* cell_map, void* out,
                   int out_format, int* status, void* stream) {
  VTK_REQUIRE(patches && patch_mask && row_idx && col_idx && cell_map && out, "vtk_unpatchify: null pointer");
  VTK_REQUIRE(dtype == 0 || dtype == 1, "vtk_unpatchify: dtype must be 0 (f32) or 1 (bf16)");
  VTK_REQUIRE(out_format >= 0 && out_format <= 2, "vtk_unpatchify: out_format must be 0, 1 or 2");
  UnpatchifyArgs a;
  a.patches = patches; a.dtype = dtype; a.patch_mask = patch_mask; a.row_idx = row_idx; a.col_idx = col_idx;
  a.B = B; a.N = N; a.patch = patch; a.gy = gy; a.gx = gx; a.cell_map = cell_map; a.out = out; a.out_format = out_format;
  a.status = status;
  return launch_unpatchify(a, (cudaStream_t)stream);
}

static int ssim_call(const void* pred, int pred_dtype, const void* target, int target_dtype, const uint8_t* patch_mask,
                     const int64_t* row_idx, const int64_t* col_idx, int B, int N, int patch, int gy, int gx, const int* tiles, int T,
                     int max_tile_h, int max_tile_w, int format, float* out, const float* gout, void* dpred, void* workspace,
                     size_t workspace_bytes, void* stream) {
  VTK_REQUIRE(pred && target && patch_mask && row_idx && col_idx && tiles && workspace, "vtk_ssim: null pointer");
  VTK_REQUIRE((pred_dtype == 0 || pred_dtype == 1) && (target_dtype == 0 || target_dtype == 1),
              "vtk_ssim: dtypes must be 0 (f32) or 1 (bf16)");
  VTK_REQUIRE(format == 0 || format == 1, "vtk_ssim: format must be 0 (minus_one_to_one) or 1 (zero_to_one)");
  SsimArgs a;
  a.pred = pred; a.pred_dtype = pred_dtype; a.target = target; a.target_dtype = target_dtype;
  a.patch_mask = patch_mask; a.row_idx = row_idx; a.col_idx = col_idx;
  a.B = B; a.N = N; a.patch = patch; a.gy = gy; a.gx = gx; a.tiles = tiles; a.T = T; a.max_tile_h = max_tile_h;
  a.max_tile_w = max_tile_w; a.format = format; a.out = out; a.gout = gout; a.dpred = dpred;
  return launch_ssim(a, out == nullptr, workspace, workspace_bytes, (cudaStream_t)stream);
}

size_t vtk_ssim_workspace_bytes(int B, int gy, int gx, int T, int max_tile_h, int max_tile_w) {
  return ssim_workspace_bytes(B, gy, gx, T, max_tile_h, max_tile_w);
}

int vtk_ssim_fwd(const void* pred, int pred_dtype, const void* target, int target_dtype, const uint8_t* patch_mask,
                 const int64_t* row_idx, const int64_t* col_idx, int B, int N, int patch, int gy, int gx, const int* tiles, int T,
                 int max_tile_h, int max_tile_w, int format, float* out, void* workspace, size_t workspace_bytes, void* stream) {
  VTK_REQUIRE(out, "vtk_ssim_fwd: null pointer");
  return ssim_call(pred, pred_dtype, target, target_dtype, patch_mask, row_idx, col_idx, B, N, patch, gy, gx, tiles, T, max_tile_h,
                   max_tile_w, format, out, nullptr, nullptr, workspace, workspace_bytes, stream);
}

int vtk_ssim_bwd(const void* pred, int pred_dtype, const void* target, int target_dtype, const uint8_t* patch_mask,
                 const int64_t* row_idx, const int64_t* col_idx, int B, int N, int patch, int gy, int gx, const int* tiles, int T,
                 int max_tile_h, int max_tile_w, int format, const float* gout, void* dpred, void* workspace, size_t workspace_bytes,
                 void* stream) {
  VTK_REQUIRE(gout && dpred, "vtk_ssim_bwd: null pointer");
  return ssim_call(pred, pred_dtype, target, target_dtype, patch_mask, row_idx, col_idx, B, N, patch, gy, gx, tiles, T, max_tile_h,
                   max_tile_w, format, nullptr, gout, dpred, workspace, workspace_bytes, stream);
}

int vtk_rmsnorm_bf16(const void* x, int64_t ldx, const void* w, void* y, int64_t ldy, int M, int D, float eps,
                     void* stream) {
  VTK_REQUIRE(x && w && y, "vtk_rmsnorm_bf16: null pointer");
  return launch_rmsnorm((const bf16*)x, ldx, (const bf16*)w, (bf16*)y, ldy, M, D, eps, (cudaStream_t)stream);
}

int vtk_rope_table(const int64_t* row_idx, const int64_t* col_idx, const float* inv_freq, void* table, int M, int d,
                   void* stream) {
  VTK_REQUIRE(row_idx && col_idx && inv_freq && table, "vtk_rope_table: null pointer");
  return launch_rope_table(row_idx, col_idx, inv_freq, (bf16*)table, M, d, (cudaStream_t)stream);
}

int vtk_cast_f32_to_bf16(const float* in, void* out, int64_t n, void* stream) {
  VTK_REQUIRE(in && out, "vtk_cast_f32_to_bf16: null pointer");
  return launch_cast_f32_bf16(in, (bf16*)out, n, (cudaStream_t)stream);
}

int vtk_kv_len(const uint8_t* patch_mask, int* kv_len, int B, int N, void* stream) {
  VTK_REQUIRE(patch_mask && kv_len, "vtk_kv_len: null pointer");
  return launch_kv_len(patch_mask, kv_len, B, N, (cudaStream_t)stream);
}

int vtk_pack_plan(const uint8_t* patch_mask, int B, int N, int pad, int qrows, int* n_valid, int* rel, int* cu, int* cuq,
                  int* grp_img, int* grp_order, int* src, void* stream) {
  VTK_REQUIRE(patch_mask && n_valid && rel && cu && cuq && grp_img && grp_order && src, "vtk_pack_plan: null pointer");
  VTK_REQUIRE(B > 0 && N > 0 && pad > 0 && PackPlan::row_capacity(B, N, pad) < (1ll << 31), "vtk_pack_plan: bad batch shape B=%d N=%d", B, N);
  PackPlan pl;
  pl.B = B; pl.N = N; pl.pad = pad; pl.qrows = qrows;
  pl.n_valid = n_valid; pl.rel = rel; pl.cu = cu; pl.cuq = cuq; pl.grp_img = grp_img; pl.grp_order = grp_order; pl.src = src;
  return launch_pack_plan(patch_mask, B, N, pl, (cudaStream_t)stream);
}
int vtk_pack_rows(const void* in, int64_t ld_in, const int* src, const int* cu, int B, int64_t row_cap, void* packed, int64_t ld_packed,
                  int width, void* stream) {
  VTK_REQUIRE(in && src && cu && packed, "vtk_pack_rows: null pointer");
  VTK_REQUIRE(B > 0 && row_cap > 0 && width > 0, "vtk_pack_rows: empty problem");
  PackPlan pl;
  pl.B = B; pl.N = 0; pl.n_valid = nullptr; pl.rel = nullptr; pl.cu = const_cast<int*>(cu); pl.cuq = nullptr; pl.grp_img = nullptr;
  pl.grp_order = nullptr; pl.src = const_cast<int*>(src);
  return launch_pack_rows((const bf16*)in, ld_in, pl, row_cap, (bf16*)packed, ld_packed, width, (cudaStream_t)stream);
}
int vtk_unpack_rows(const void* packed, int64_t ld_packed, const int* rel, const int* cu, int B, int N, void* out,
                    int64_t ld_out, int width, void* stream) {
  VTK_REQUIRE(packed && rel && cu && out, "vtk_unpack_rows: null pointer");
  VTK_REQUIRE(B > 0 && N > 0 && width > 0, "vtk_unpack_rows: empty problem");
  PackPlan pl;
  pl.B = B; pl.N = N; pl.n_valid = nullptr; pl.rel = const_cast<int*>(rel); pl.cu = const_cast<int*>(cu); pl.cuq = nullptr;
  pl.grp_img = nullptr; pl.grp_order = nullptr; pl.src = nullptr;
  return launch_unpack_rows((const bf16*)packed, ld_packed, pl, (bf16*)out, ld_out, width, (cudaStream_t)stream);
}

static GemmArgs base_args(const void* A, int64_t lda, const void* W, int64_t ldw, int64_t w_rows, int M, int N, int K) {
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.A = (const bf16*)A; g.lda = lda; g.B = (const bf16*)W; g.ldb = ldw; g.b_rows = w_rows; g.M = M; g.N = N; g.K = K;
  g.epi.eps = 1e-6f;
  return g;
}

int vtk_linear_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, const void* bias, void* out, int64_t ldo,
                    int M, int N, int K, void* stream) {
  VTK_REQUIRE(A && W && out, "vtk_linear_bf16: null pointer");
  VTK_REQUIRE(ldo % 8 == 0, "vtk_linear_bf16: ldo must be a multiple of 8");
  GemmArgs g = base_args(A, lda, W, ldw, N, M, N, K);
  g.epi.out = (bf16*)out; g.epi.ldo = ldo; g.epi.bias = (const bf16*)bias;
  return launch_gemm(EPI_BIAS, g, (cudaStream_t)stream);
}

int vtk_linear_tn_bf16(const void* At, int64_t lda, const void* Bt, int64_t ldb, void* out, int64_t ldo, int M, int N, int K,
                       void* stream) {
  VTK_REQUIRE(At && Bt && out, "vtk_linear_tn_bf16: null pointer");
  VTK_REQUIRE(ldo % 8 == 0, "vtk_linear_tn_bf16: ldo must be a multiple of 8");
  GemmArgs g = base_args(At, lda, Bt, ldb, N, M, N, K);
  g.trans = 3;
  g.epi.out = (bf16*)out; g.epi.ldo = ldo;
  return launch_gemm(EPI_BIAS, g, (cudaStream_t)stream);
}

int vtk_linear_nn_acc_bf16(const void* A, int64_t lda, const void* Bt, int64_t ldb, void* out, int64_t ldo, int M, int N, int K,
                           int accumulate, void* stream) {
  VTK_REQUIRE(A && Bt && out, "vtk_linear_nn_acc_bf16: null pointer");
  VTK_REQUIRE(ldo % 8 == 0, "vtk_linear_nn_acc_bf16: ldo must be a multiple of 8");
  GemmArgs g = base_args(A, lda, Bt, ldb, N, M, N, K);
  g.trans = 2;
  g.epi.out = (bf16*)out; g.epi.ldo = ldo; g.epi.accumulate = accumulate ? 1 : 0;
  return launch_gemm(EPI_BIAS, g, (cudaStream_t)stream);
}

int vtk_linear2_bf16(const void* A, int64_t lda, const void* W0, int64_t ldw0, const void* W1, int64_t ldw1, void* out, int64_t ldo,
                     int M, int N, int K0, int K1, void* stream) {
  VTK_REQUIRE(A && W0 && W1 && out, "vtk_linear2_bf16: null pointer");
  VTK_REQUIRE(ldo % 8 == 0 && K0 > 0 && K1 > 0, "vtk_linear2_bf16: ldo must be a multiple of 8 and both K parts non-empty");
  const bool aligned = ((reinterpret_cast<uintptr_t>(W1) | reinterpret_cast<uintptr_t>(A)) & 15) == 0;
  if (M > 128 && N > 128 && K0 % 64 == 0 && ldw1 % 8 == 0 && aligned) {
    GemmArgs g = base_args(A, lda, W0, ldw0, N, M, N, K0 + K1);       // one accumulator over both K ranges
    g.B2 = (const bf16*)W1; g.ldb2 = ldw1; g.epi.k_split = K0;
    g.epi.out = (bf16*)out; g.epi.ldo = ldo;
    return launch_gemm(EPI_BIAS, g, (cudaStream_t)stream);
  }
  // small / oddly shaped problems: two GEMMs, the second one adding to the first one's output
  GemmArgs g0 = base_args(A, lda, W0, ldw0, N, M, N, K0);
  g0.epi.out = (bf16*)out; g0.epi.ldo = ldo;
  int r = launch_gemm(EPI_BIAS, g0, (cudaStream_t)stream);
  if (r) return r;
  GemmArgs g1 = base_args((const bf16*)A + K0, lda, W1, ldw1, N, M, N, K1);
  g1.epi.out = (bf16*)out; g1.epi.ldo = ldo; g1.epi.accumulate = 1;
  return launch_gemm(EPI_BIAS, g1, (cudaStream_t)stream);
}

int vtk_linear_ln_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, const void* bias, void* out, int64_t ldo,
                       int M, int N, int K, float eps, void* stream) {
  VTK_REQUIRE(A && W && out && bias, "vtk_linear_ln_bf16: null pointer");
  VTK_REQUIRE(ldo % 8 == 0, "vtk_linear_ln_bf16: ldo must be a multiple of 8");
  GemmArgs g = base_args(A, lda, W, ldw, N, M, N, K);
  g.epi.out = (bf16*)out; g.epi.ldo = ldo; g.epi.bias = (const bf16*)bias; g.epi.eps = eps;
  return launch_gemm(EPI_BIAS_LN, g, (cudaStream_t)stream);
}

int vtk_qkv_swiglu_bf16(const void* h, int64_t ldh, const void* Wp, int64_t ldw, int64_t w_rows, int M, int D, int d,
                        int Hf, int qp, const void* norm_q, const void* norm_k, const void* rope_table, float eps,
                        void* qkv, int64_t ld_qkv, void* act, int64_t ld_act, void* stream) {
  VTK_REQUIRE(h && Wp && norm_q && norm_k && rope_table && qkv && act, "vtk_qkv_swiglu_bf16: null pointer");
  VTK_REQUIRE(qp >= 3 * D && w_rows == (int64_t)qp + 2 * Hf, "vtk_qkv_swiglu_bf16: packed weight must have qp + 2*Hf rows");
  VTK_REQUIRE(ld_qkv % 8 == 0 && ld_act % 8 == 0, "vtk_qkv_swiglu_bf16: output strides must be multiples of 8");
  GemmArgs g = base_args(h, ldh, Wp, ldw, w_rows, M, qp + 2 * Hf, D);
  g.epi.qkv = (bf16*)qkv; g.epi.ld_qkv = ld_qkv; g.epi.act = (bf16*)act; g.epi.ld_act = ld_act;
  g.epi.normq = (const bf16*)norm_q; g.epi.normk = (const bf16*)norm_k; g.epi.rope = (const bf16*)rope_table;
  g.epi.D = D; g.epi.d = d; g.epi.Hf = Hf; g.epi.qp = qp; g.epi.eps = eps;
  int r = launch_gemm(EPI_QKV_SWIGLU, g, (cudaStream_t)stream);
  if (r || qk_norm_fused(d)) return r;
  return launch_qk_norm_rope_fwd((const bf16*)qkv, ld_qkv, (const bf16*)norm_q, (const bf16*)norm_k, (const bf16*)rope_table, (bf16*)qkv,
                                 ld_qkv, M, D / d, d, eps, (cudaStream_t)stream);
}

int vtk_proj_residual_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, const void* gamma, void* x,
                           int64_t ldx, int M, int N, int K, void* stream) {
  VTK_REQUIRE(A && W && gamma && x, "vtk_proj_residual_bf16: null pointer");
  VTK_REQUIRE(ldx % 8 == 0, "vtk_proj_residual_bf16: ldx must be a multiple of 8");
  GemmArgs g = base_args(A, lda, W, ldw, N, M, N, K);
  g.epi.out = (bf16*)x; g.epi.ldo = ldx; g.epi.gamma = (const bf16*)gamma;
  return launch_gemm(EPI_RESID, g, (cudaStream_t)stream);
}

int vtk_quant_rows_e4m3(const void* x, int64_t ldx, void* q, int64_t ldq, float* scale, int M, int K, void* stream) {
  VTK_REQUIRE(x && q && scale, "vtk_quant_rows_e4m3: null pointer");
  return launch_quant_rows_e4m3((const bf16*)x, ldx, (uint8_t*)q, ldq, scale, M, K, nullptr, (cudaStream_t)stream);
}
int vtk_quant_tensor_e4m3(const void* x, int64_t ldx, void* q, int64_t ldq, float* scale, float* amax_ws, int M, int K, void* stream) {
  VTK_REQUIRE(x && q && scale && amax_ws, "vtk_quant_tensor_e4m3: null pointer");
  return launch_quant_rows_e4m3((const bf16*)x, ldx, (uint8_t*)q, ldq, scale, M, K, nullptr, (cudaStream_t)stream, amax_ws);
}

int vtk_proj_residual_fp8(const void* A8, int64_t lda, const float* a_scale, const void* W8, int64_t ldw, float w_scale,
                          const void* gamma, void* x, int64_t ldx, int M, int N, int K, void* stream) {
  VTK_REQUIRE(A8 && a_scale && W8 && gamma && x, "vtk_proj_residual_fp8: null pointer");
  VTK_REQUIRE(ldx % 8 == 0, "vtk_proj_residual_fp8: ldx must be a multiple of 8");
  GemmArgs g = base_args(A8, lda, W8, ldw, N, M, N, K);
  g.fp8 = 1;
  g.epi.out = (bf16*)x; g.epi.ldo = ldx; g.epi.gamma = (const bf16*)gamma; g.epi.a_scale = a_scale; g.epi.w_scale = w_scale;
  return launch_gemm(EPI_RESID, g, (cudaStream_t)stream);
}

int vtk_attention_bf16(const void* q, const void* k, const void* v, int64_t ld_qkv, void* out, int64_t ld_out,
                       const int* kv_len, int B, int N, int heads, int d, int zero_invalid_rows, int window, float* lse, void* stream) {
  VTK_REQUIRE(q && k && v && out, "vtk_attention_bf16: null pointer");
  AttnArgs a;
  a.q = (const bf16*)q; a.k = (const bf16*)k; a.v = (const bf16*)v; a.ld_qkv = ld_qkv; a.out = (bf16*)out; a.ld_out = ld_out;
  a.kv_len = kv_len; a.B = B; a.N = N; a.heads = heads; a.d = d;
  a.zero_invalid_rows = zero_invalid_rows;
  a.window = window;
  a.lse = lse;
  return launch_attention(a, (cudaStream_t)stream);
}

int vtk_attention_packed_lse_bf16(const void* q, const void* k, const void* v, int64_t ld_qkv, void* out, int64_t ld_out,
                                  const int* n_valid, const int* cu, const int* cuq, const int* grp_img, const int* grp_order, int B, int N,
                                  int heads, int d, int64_t row_cap, int grp_cap, float* lse, void* stream) {
  VTK_REQUIRE(q && k && v && out && n_valid && cu && cuq && grp_img && grp_order, "vtk_attention_packed_lse_bf16: null pointer");
  AttnArgs a;
  a.q = (const bf16*)q; a.k = (const bf16*)k; a.v = (const bf16*)v; a.ld_qkv = ld_qkv; a.out = (bf16*)out; a.ld_out = ld_out;
  a.kv_len = n_valid; a.B = B; a.N = N; a.heads = heads; a.d = d;
  a.zero_invalid_rows = lse ? 1 : 0;   // with lse: the image's pad rows get out 0, lse +inf; without: they are not written
  a.window = -1; a.lse = lse;
  a.cu = cu; a.cuq = cuq; a.grp_img = grp_img; a.grp_order = grp_order; a.row_cap = row_cap; a.grp_cap = grp_cap;
  return launch_attention(a, (cudaStream_t)stream);
}

int vtk_umma_probe(const void* A, const void* B, float* D, int N, int K, int b_mn_major, uint32_t lbo_bytes,
                   uint32_t sbo_bytes, uint32_t kstep_bytes, void* stream) {
  VTK_REQUIRE(A && B && D, "vtk_umma_probe: null pointer");
  return launch_umma_probe((const bf16*)A, (const bf16*)B, D, N, K, b_mn_major, lbo_bytes, sbo_bytes, kstep_bytes,
                           (cudaStream_t)stream);
}

// -------------------------------------------------------------------------------------------------
// training step (BASELINE config 5): kernel-level entry points driven by vitok_b200/train.py
// -------------------------------------------------------------------------------------------------
int vtk_qk_norm_rope_fwd(const void* zraw, int64_t ldz, const void* norm_q, const void* norm_k, const void* rope_table,
                         void* qkv, int64_t ld_qkv, int M, int heads, int d, float eps, void* stream) {
  VTK_REQUIRE(zraw && norm_q && norm_k && rope_table && qkv, "vtk_qk_norm_rope_fwd: null pointer");
  return launch_qk_norm_rope_fwd((const bf16*)zraw, ldz, (const bf16*)norm_q, (const bf16*)norm_k, (const bf16*)rope_table,
                                 (bf16*)qkv, ld_qkv, M, heads, d, eps, (cudaStream_t)stream);
}
int vtk_swiglu_fwd(const void* zraw, int64_t ldz, int qp, void* act, int64_t ld_act, int M, int Hf, int layout, void* stream) {
  VTK_REQUIRE(zraw && act, "vtk_swiglu_fwd: null pointer");
  VTK_REQUIRE(layout == 0 || layout == 1, "vtk_swiglu_fwd: layout must be 0 (16-column value|gate groups) or 1 ([value | gate])");
  return launch_swiglu_fwd((const bf16*)zraw, ldz, qp, (bf16*)act, ld_act, M, Hf, layout, (cudaStream_t)stream);
}
int vtk_resid_fwd_dp(const void* x, const void* y, const void* gamma, void* out, int M, int D, const float* keep, int rows_per_image,
                     float keep_prob, void* stream) {
  VTK_REQUIRE(x && y && gamma && out, "vtk_resid_fwd_dp: null pointer");
  return launch_resid_fwd((const bf16*)x, (const bf16*)y, (const bf16*)gamma, (bf16*)out, M, D, (cudaStream_t)stream, keep, rows_per_image,
                          keep_prob);
}
int vtk_resid_bwd_dp(const void* dx, const void* y, const void* gamma, void* dy, float* dgamma, int M, int D, const float* keep,
                     int rows_per_image, float keep_prob, void* stream) {
  VTK_REQUIRE(dx && y && gamma && dy && dgamma, "vtk_resid_bwd_dp: null pointer");
  return launch_resid_bwd((const bf16*)dx, (const bf16*)y, (const bf16*)gamma, (bf16*)dy, dgamma, M, D, (cudaStream_t)stream, keep,
                          rows_per_image, keep_prob);
}
int vtk_layernorm_fwd(const void* x, void* out, int M, int C, float eps, void* stream) {
  VTK_REQUIRE(x && out, "vtk_layernorm_fwd: null pointer");
  return launch_ln_fwd((const bf16*)x, (bf16*)out, M, C, eps, (cudaStream_t)stream);
}
int vtk_colsum(const void* in, int64_t ld, float* out, int M, int C, void* stream) {
  VTK_REQUIRE(in && out, "vtk_colsum: null pointer");
  return launch_colsum((const bf16*)in, ld, out, M, C, (cudaStream_t)stream);
}
int vtk_swiglu_bwd(const void* dact, int64_t ldd, const void* zraw, int64_t ldz, int qp, void* dz, int64_t lddz, int M, int Hf, int layout,
                   void* stream) {
  VTK_REQUIRE(dact && zraw && dz, "vtk_swiglu_bwd: null pointer");
  VTK_REQUIRE(layout == 0 || layout == 1, "vtk_swiglu_bwd: layout must be 0 or 1");
  return launch_swiglu_bwd((const bf16*)dact, ldd, (const bf16*)zraw, ldz, qp, (bf16*)dz, lddz, M, Hf, layout, (cudaStream_t)stream);
}
int vtk_qk_norm_rope_bwd(void* dz, int64_t lddz, const void* zraw, int64_t ldz, const void* norm_q, const void* norm_k,
                         const void* rope_table, float* dw, int M, int heads, int d, float eps, void* stream) {
  VTK_REQUIRE(dz && zraw && norm_q && norm_k && rope_table && dw, "vtk_qk_norm_rope_bwd: null pointer");
  return launch_qk_norm_rope_bwd((bf16*)dz, lddz, (const bf16*)zraw, ldz, (const bf16*)norm_q, (const bf16*)norm_k,
                                 (const bf16*)rope_table, dw, M, heads, d, eps, (cudaStream_t)stream);
}
int vtk_rmsnorm_bwd(const void* x, const void* dh, const void* w, const void* dx_res, void* dx_out, float* dw, int M, int D,
                    float eps, void* stream) {
  VTK_REQUIRE(x && dh && w && dx_res && dx_out && dw, "vtk_rmsnorm_bwd: null pointer");
  return launch_rmsnorm_bwd((const bf16*)x, (const bf16*)dh, (const bf16*)w, (const bf16*)dx_res, (bf16*)dx_out, dw, M, D, eps,
                            (cudaStream_t)stream);
}
int vtk_layernorm_bwd(const void* zlin, const void* dz, void* dx, int M, int C, float eps, void* stream) {
  VTK_REQUIRE(zlin && dz && dx, "vtk_layernorm_bwd: null pointer");
  return launch_ln_bwd((const bf16*)zlin, (const bf16*)dz, (bf16*)dx, M, C, eps, (cudaStream_t)stream);
}
int vtk_charbonnier(const void* pred, const void* target, const uint8_t* patch_mask, const int* n_valid, float* loss_sum,
                    void* dpred, int B, int N, int P, float eps, void* stream) {
  VTK_REQUIRE(pred && target && loss_sum, "vtk_charbonnier: null pointer");
  VTK_REQUIRE(!patch_mask || n_valid, "vtk_charbonnier: n_valid is required with a patch_mask");
  return launch_charbonnier((const bf16*)pred, (const bf16*)target, patch_mask, n_valid, loss_sum, (bf16*)dpred, B, N, P, eps,
                            (cudaStream_t)stream);
}
int vtk_adamw_multi_ex(const vtk_adamw_tensor* tensors, float* const* ema, int n_tensors, float lr, float beta1, float beta2, float eps,
                       int step, float grad_scale, const float* coef, double ema_decay, void* stream) {
  VTK_REQUIRE(tensors || n_tensors == 0, "vtk_adamw_multi: null tensor table");
  static_assert(sizeof(vtk_adamw_tensor) == sizeof(AdamwTensor), "vtk_adamw_tensor layout");
  return launch_adamw_multi(reinterpret_cast<const AdamwTensor*>(tensors), ema, n_tensors, lr, beta1, beta2, eps, step, grad_scale, coef,
                            ema_decay, (cudaStream_t)stream);
}
int vtk_adamw_multi(const vtk_adamw_tensor* tensors, int n_tensors, float lr, float beta1, float beta2, float eps, int step,
                    float grad_scale, void* stream) {
  return vtk_adamw_multi_ex(tensors, nullptr, n_tensors, lr, beta1, beta2, eps, step, grad_scale, nullptr, 0.0, stream);
}
int64_t vtk_grad_norm_slots(const vtk_adamw_tensor* tensors, int n_tensors) {
  if (!tensors || n_tensors <= 0) return 0;
  return grad_norm_slots(reinterpret_cast<const AdamwTensor*>(tensors), n_tensors);
}
int vtk_grad_sumsq_multi(const vtk_adamw_tensor* tensors, int n_tensors, float* partials, int64_t slot0, void* stream) {
  VTK_REQUIRE(tensors || n_tensors == 0, "vtk_grad_sumsq_multi: null tensor table");
  VTK_REQUIRE(partials || n_tensors == 0, "vtk_grad_sumsq_multi: null partials");
  VTK_REQUIRE(slot0 >= 0, "vtk_grad_sumsq_multi: slot0 must be >= 0");
  return launch_grad_sumsq(reinterpret_cast<const AdamwTensor*>(tensors), n_tensors, partials + slot0, (cudaStream_t)stream);
}
int vtk_grad_norm_finish(const float* partials, int64_t n_slots, float max_norm, float* norm_coef, void* stream) {
  VTK_REQUIRE(norm_coef && (partials || n_slots == 0), "vtk_grad_norm_finish: null pointer");
  VTK_REQUIRE(n_slots >= 0, "vtk_grad_norm_finish: n_slots must be >= 0");
  return launch_grad_norm_finish(partials, n_slots, max_norm, norm_coef, (cudaStream_t)stream);
}
int vtk_scale_by_dev(void* x, const float* scale, int64_t n, void* stream) {
  VTK_REQUIRE(x && scale, "vtk_scale_by_dev: null pointer");
  return launch_scale_by_dev((bf16*)x, scale, n, (cudaStream_t)stream);
}
int vtk_attn_delta(const void* o, int64_t ldo, const void* dout, int64_t lddo, float* delta, int M, int heads, int d, void* stream) {
  VTK_REQUIRE(o && dout && delta, "vtk_attn_delta: null pointer");
  return launch_attn_delta((const bf16*)o, ldo, (const bf16*)dout, lddo, delta, M, heads, d, (cudaStream_t)stream);
}
int vtk_attention_bwd_bf16(const void* q, const void* k, const void* v, int64_t ld_qkv, const void* dout, int64_t ld_do,
                           const float* lse, const float* delta, void* dq, void* dk, void* dv, int64_t ld_d, const int* kv_len,
                           int B, int N, int heads, int d, int zero_invalid_rows, int window, void* stream) {
  VTK_REQUIRE(q && k && v && dout && lse && delta && dq && dk && dv, "vtk_attention_bwd_bf16: null pointer");
  AttnBwdArgs a;
  a.q = (const bf16*)q; a.k = (const bf16*)k; a.v = (const bf16*)v; a.ld_qkv = ld_qkv; a.dout = (const bf16*)dout; a.ld_do = ld_do;
  a.lse = lse; a.delta = delta; a.dq = (bf16*)dq; a.dk = (bf16*)dk; a.dv = (bf16*)dv; a.ld_d = ld_d; a.kv_len = kv_len;
  a.B = B; a.N = N; a.heads = heads; a.d = d; a.zero_invalid_rows = zero_invalid_rows; a.window = window;
  return launch_attention_bwd(a, (cudaStream_t)stream);
}

int vtk_attention_bwd_packed_bf16(const void* q, const void* k, const void* v, int64_t ld_qkv, const void* dout, int64_t ld_do,
                                  const float* lse, const float* delta, void* dq, void* dk, void* dv, int64_t ld_d, const int* n_valid,
                                  const int* cu, const int* cuq, const int* grp_img, const int* grp_order, int B, int heads, int d,
                                  int64_t row_cap, int grp_cap, void* stream) {
  VTK_REQUIRE(q && k && v && dout && lse && delta && dq && dk && dv && n_valid && cu && cuq && grp_img && grp_order,
              "vtk_attention_bwd_packed_bf16: null pointer");
  AttnBwdArgs a;
  a.q = (const bf16*)q; a.k = (const bf16*)k; a.v = (const bf16*)v; a.ld_qkv = ld_qkv; a.dout = (const bf16*)dout; a.ld_do = ld_do;
  a.lse = lse; a.delta = delta; a.dq = (bf16*)dq; a.dk = (bf16*)dk; a.dv = (bf16*)dv; a.ld_d = ld_d; a.kv_len = n_valid;
  a.B = B; a.N = 0; a.heads = heads; a.d = d; a.zero_invalid_rows = 1; a.window = -1;
  a.cu = cu; a.cuq = cuq; a.grp_img = grp_img; a.grp_order = grp_order; a.row_cap = row_cap; a.grp_cap = grp_cap;
  return launch_attention_bwd(a, (cudaStream_t)stream);
}

// -------------------------------------------------------------------------------------------------
// AE
// -------------------------------------------------------------------------------------------------
int vtk_ae_create(const vtk_ae_config* cfg, vtk_ae_t* out) {
  VTK_REQUIRE(cfg && out, "vtk_ae_create: null pointer");
  VTK_REQUIRE(cfg->enc_depth > 0 || cfg->dec_depth > 0 || cfg->enc_width > 0 || cfg->dec_width > 0,
              "At least one of encoder or decoder must be True");
  vtk_ae_s* h = new vtk_ae_s();
  h->cfg = *cfg;
  Side& e = h->side[0];
  e.width = cfg->enc_width; e.depth = cfg->enc_depth; e.heads = cfg->enc_heads; e.hidden = cfg->enc_hidden;
  Side& d = h->side[1];
  d.width = cfg->dec_width; d.depth = cfg->dec_depth; d.heads = cfg->dec_heads; d.hidden = cfg->dec_hidden;
  for (int s = 0; s < 2; ++s) {
    Side& sd = h->side[s];
    if (sd.width <= 0) continue;
    if (sd.heads <= 0 || sd.width % sd.heads) {
      set_error("vtk_ae_create: width %d not divisible by heads %d", sd.width, sd.heads);
      delete h;
      return VTK_ERR_BAD_ARG;
    }
    const int hd = sd.head_dim();
    if (sd.depth > 0 && !head_dim_supported(hd)) {
      set_error("vtk_ae_create: head_dim %d unsupported by the sm_100a attention kernels (supported: multiples of 8 from 8 to 128)", hd);
      delete h;
      return VTK_ERR_UNSUPPORTED;
    }
    if (sd.width % 8 || sd.hidden % 16) {
      set_error("vtk_ae_create: width must be a multiple of 8 and hidden of 16 (width=%d hidden=%d)", sd.width, sd.hidden);
      delete h;
      return VTK_ERR_BAD_ARG;
    }
  }
  *out = h;
  return VTK_OK;
}

int vtk_ae_destroy(vtk_ae_t h) {
  if (!h) return VTK_OK;
  for (int s = 0; s < 2; ++s)
    if (h->side[s].inv_freq) cudaFree(h->side[s].inv_freq);
  for (cudaEvent_t e : h->ev) cudaEventDestroy(e);
  delete h;
  return VTK_OK;
}

int vtk_ae_set_weights(vtk_ae_t h, int side, const void* w_a, const void* b_a, const void* w_b, const void* b_b,
                       const vtk_block_weights* blocks, int nblocks, const float* inv_freq_host, int n_inv_freq) {
  VTK_REQUIRE(h && (side == 0 || side == 1), "vtk_ae_set_weights: bad handle/side");
  Side& s = h->side[side];
  VTK_REQUIRE(s.width > 0, "vtk_ae_set_weights: side %d is absent from this model", side);
  VTK_REQUIRE(w_a && b_a && w_b && b_b, "vtk_ae_set_weights: null projection weights");
  VTK_REQUIRE(nblocks == s.depth, "vtk_ae_set_weights: expected %d blocks, got %d", s.depth, nblocks);
  VTK_REQUIRE(nblocks == 0 || blocks, "vtk_ae_set_weights: null blocks");
  VTK_REQUIRE(n_inv_freq == s.head_dim() / 4 && inv_freq_host, "vtk_ae_set_weights: inv_freq must have head_dim/4 entries");
  s.w_a = (const bf16*)w_a; s.b_a = (const bf16*)b_a; s.w_b = (const bf16*)w_b; s.b_b = (const bf16*)b_b;
  s.norm_folded = false;
  s.fp8.clear();
  s.blocks.assign(blocks, blocks + nblocks);
  for (int i = 0; i < nblocks; ++i) {
    const vtk_block_weights& b = s.blocks[i];
    VTK_REQUIRE(b.w_in && b.w_out && b.norm1 && b.norm_q && b.norm_k && b.gamma, "vtk_ae_set_weights: null pointer in block %d", i);
  }
  if (!s.inv_freq) {
    int r = check_cuda(cudaMalloc(&s.inv_freq, sizeof(float) * n_inv_freq), "cudaMalloc(inv_freq)");
    if (r) return r;
  }
  return check_cuda(cudaMemcpy(s.inv_freq, inv_freq_host, sizeof(float) * n_inv_freq, cudaMemcpyHostToDevice), "cudaMemcpy(inv_freq)");
}

size_t vtk_ae_workspace_bytes(vtk_ae_t h, int side, int B, int N) {
  if (!h || side < 0 || side > 1 || B <= 0 || N <= 0) return 0;
  return carve(h->side[side], nullptr, B, N, io_cols(h->cfg)).bytes;
}

// A masked batch runs on its packed valid tokens.  A side without blocks keeps the padded rows: it has no attention to mask.
static bool use_packing(const Side& s, const uint8_t* patch_mask) { return patch_mask != nullptr && s.depth > 0; }

// rows = row capacity of the activation buffers; with `pl` the kernels read the live row count from pl->m_dev()
static int run_blocks(vtk_ae_s* h, const Side& s, const Workspace& w, const int64_t* row_idx, const int64_t* col_idx, int B, int N,
                      int rows, const PackPlan* pl, cudaStream_t st, int& launches) {
  const int M = rows, D = s.width, d = s.head_dim(), Hf = s.hidden, qp = s.qp(), kp = s.kp();
  const float eps = h->cfg.norm_eps;
  const int* m_dev = pl ? pl->m_dev() : nullptr;
  int r;
  if (s.depth > 0) {
    { LaunchTimer t(h, st, CLS_MISC); r = launch_rope_table(row_idx, col_idx, s.inv_freq, w.rope, M, d, st, pl ? pl->src : nullptr, m_dev); }
    if (r) return r;
    ++launches;
  }
  for (int i = 0; i < s.depth; ++i) {
    const vtk_block_weights& b = s.blocks[i];
    const bool fused = s.norm_folded;   // norm1 inside the epilogues: x is the A operand, rows scaled by rsqrt(mean(x^2)+eps)
    if (!fused) {
      { LaunchTimer t(h, st, CLS_RMSNORM); r = launch_rmsnorm(w.x, D, (const bf16*)b.norm1, w.h, D, M, D, eps, st, m_dev); }
      if (r) return r;
      ++launches;
    }
    const bool f8 = !s.fp8.empty();     // AE.quantize: e4m3 operands for both block GEMMs (needs the fused norm)
    if (f8) {
      { LaunchTimer t(h, st, CLS_MISC); r = launch_quant_rows_e4m3(w.x, D, w.x8, D, w.sx, M, D, m_dev, st, h->fp8_per_tensor ? w.amax : nullptr); }
      if (r) return r;
      launches += h->fp8_per_tensor ? 2 : 1;
    }
    GemmArgs g1 = f8 ? base_args(w.x8, D, s.fp8[i].w_in8, D, (int64_t)qp + 2 * Hf, M, qp + 2 * Hf, D)
                     : base_args(fused ? w.x : w.h, D, b.w_in, D, (int64_t)qp + 2 * Hf, M, qp + 2 * Hf, D);
    if (f8) { g1.fp8 = 1; g1.epi.a_scale = w.sx; g1.epi.w_scale = s.fp8[i].w_in_scale; }
    if (fused) { g1.epi.ss_in = w.ss; g1.epi.ss_units = D / 64; g1.epi.ss_inv_d = 1.f / (float)D; }
    g1.epi.qkv = w.qkv; g1.epi.ld_qkv = 3 * D; g1.epi.act = w.a2 + D; g1.epi.ld_act = kp;
    g1.epi.normq = (const bf16*)b.norm_q; g1.epi.normk = (const bf16*)b.norm_k; g1.epi.rope = w.rope;
    g1.epi.D = D; g1.epi.d = d; g1.epi.Hf = Hf; g1.epi.qp = qp; g1.epi.eps = eps;
    g1.epi.m_dev = m_dev;
    { LaunchTimer t(h, st, CLS_QKV_SWIGLU); r = launch_gemm(EPI_QKV_SWIGLU, g1, st); }
    if (r) return r;
    if (!qk_norm_fused(d)) {   // the epilogue copied q and k raw: QK-norm + RoPE in place on the qkv rows
      LaunchTimer t(h, st, CLS_MISC);
      r = launch_qk_norm_rope_fwd(w.qkv, 3 * D, (const bf16*)b.norm_q, (const bf16*)b.norm_k, w.rope, w.qkv, 3 * D, M, s.heads, d, eps, st);
      if (r) return r;
      ++launches;
    }
    AttnArgs a;
    a.q = w.qkv; a.k = w.qkv + D; a.v = w.qkv + 2 * D; a.ld_qkv = 3 * D; a.out = w.a2; a.ld_out = kp;
    a.B = B; a.N = N; a.heads = s.heads; a.d = d;
    a.zero_invalid_rows = 0;
    a.lse = nullptr;
    if (pl) {
      // packed: image b = packed rows [cu[b], cu[b+1]) with its n_valid[b] tokens in front -- no key mask left
      a.kv_len = pl->n_valid;
      a.cu = pl->cu; a.cuq = pl->cuq; a.grp_img = pl->grp_img; a.grp_order = pl->grp_order; a.row_cap = M;
      a.grp_cap = (int)PackPlan::group_capacity(B, N, pl->qrows);
      a.window = -1;
    } else {
      // no mask: every key of the image, or those of the sliding window (flash backend, attention.py:113-116)
      a.kv_len = nullptr;
      a.window = h->cfg.sliding_window > 0 ? h->cfg.sliding_window : -1;
    }
    { LaunchTimer t(h, st, CLS_ATTENTION); r = launch_attention(a, st); }
    if (r) return r;
    if (f8) {
      { LaunchTimer t(h, st, CLS_MISC); r = launch_quant_rows_e4m3(w.a2, kp, w.a28, kp, w.sa, M, D + Hf, m_dev, st, h->fp8_per_tensor ? w.amax + 1 : nullptr); }
      if (r) return r;
      launches += h->fp8_per_tensor ? 2 : 1;
    }
    GemmArgs g2 = f8 ? base_args(w.a28, kp, s.fp8[i].w_out8, kp, D, M, D, D + Hf) : base_args(w.a2, kp, b.w_out, kp, D, M, D, D + Hf);
    if (f8) { g2.fp8 = 1; g2.epi.a_scale = w.sa; g2.epi.w_scale = s.fp8[i].w_out_scale; }
    g2.epi.out = w.x; g2.epi.ldo = D; g2.epi.gamma = (const bf16*)b.gamma;
    g2.epi.m_dev = m_dev;
    if (fused && i + 1 < s.depth) { g2.epi.ss_out = w.ss; g2.epi.ss_ld = D / 64; }
    { LaunchTimer t(h, st, CLS_PROJ_RESID); r = launch_gemm(EPI_RESID, g2, st); }
    if (r) return r;
    launches += 3;
  }
  return 0;
}

// [embed -> blocks -> head] over either the padded [B*N] rows or the packed rows of a masked batch
static int run_side(vtk_ae_s* h, int side, const void* in, const int64_t* row_idx, const int64_t* col_idx,
                    const uint8_t* patch_mask, int B, int N, void* out, void* workspace, cudaStream_t st) {
  const Side& s = h->side[side];
  const int P = h->cfg.pixels_per_token, C = h->cfg.channels_per_token, D = s.width;
  const int cin = side == 0 ? P : C, cout = side == 0 ? C : P;
  Workspace w = carve(s, workspace, B, N, io_cols(h->cfg));
  const bool packed = use_packing(s, patch_mask);
  const PackPlan* pl = packed ? &w.plan : nullptr;
  const int rows = packed ? (int)PackPlan::row_capacity(B, N, w.plan.pad) : B * N;   // capacity; the live count is pl->m_dev()
  const int* m_dev = packed ? pl->m_dev() : nullptr;
  int launches = 0, r;
  h->ev_used = 0;
  const bf16* a_in = (const bf16*)in;
  if (packed) {
    { LaunchTimer t(h, st, CLS_MISC); r = launch_pack_plan(patch_mask, B, N, *pl, st); }
    if (r) return r;
    { LaunchTimer t(h, st, CLS_MISC); r = launch_pack_rows((const bf16*)in, cin, *pl, rows, w.pin, cin, cin, st); }
    if (r) return r;
    launches += 4;
    a_in = w.pin;
  }
  GemmArgs g = base_args(a_in, cin, s.w_a, cin, D, rows, D, cin);       // patch_embed ae.py:191 / decoder_embed ae.py:220
  g.epi.out = w.x; g.epi.ldo = D; g.epi.bias = s.b_a; g.epi.m_dev = m_dev;
  if (s.norm_folded && s.depth > 0) { g.epi.ss_out = w.ss; g.epi.ss_ld = D / 64; }
  { LaunchTimer t(h, st, CLS_LINEAR); r = launch_gemm(EPI_BIAS, g, st); }
  if (r) return r;
  ++launches;
  if ((r = run_blocks(h, s, w, row_idx, col_idx, B, N, rows, pl, st, launches))) return r;
  bf16* o = packed ? w.pout : (bf16*)out;
  GemmArgs gz = base_args(w.x, D, s.w_b, D, cout, rows, cout, D);
  gz.epi.out = o; gz.epi.ldo = cout; gz.epi.bias = s.b_b; gz.epi.eps = h->cfg.norm_eps; gz.epi.m_dev = m_dev;
  if (side == 0) { LaunchTimer t(h, st, CLS_MISC); r = launch_gemm(EPI_BIAS_LN, gz, st); }     // to_code + output_fn, ae.py:207
  else { LaunchTimer t(h, st, CLS_LINEAR); r = launch_gemm(EPI_BIAS, gz, st); }                 // to_pixels, ae.py:242
  if (r) return r;
  ++launches;
  if (packed) {   // scatter back to [B, N, cout]; masked tokens read as 0
    { LaunchTimer t(h, st, CLS_MISC); r = launch_unpack_rows(w.pout, cout, *pl, (bf16*)out, cout, cout, st); }
    if (r) return r;
    ++launches;
  }
  h->last_launches = launches;
  return VTK_OK;
}

static int check_io(vtk_ae_t h, int side, const void* in, const int64_t* row_idx, const int64_t* col_idx, int B, int N,
                    void* out, void* workspace, size_t workspace_bytes, const char* fn) {
  VTK_REQUIRE(h, "%s: null handle", fn);
  const Side& s = h->side[side];
  VTK_REQUIRE(s.width > 0 && s.w_a, "%s: this model has no %s weights set", fn, side ? "decoder" : "encoder");
  VTK_REQUIRE(in && row_idx && col_idx && out && workspace, "%s: null pointer", fn);
  VTK_REQUIRE(B > 0 && N > 0, "%s: empty batch (B=%d N=%d)", fn, B, N);
  VTK_REQUIRE(PackPlan::row_capacity(B, N, 16) < (1ll << 31), "%s: B*N too large", fn);
  VTK_REQUIRE(workspace_bytes >= vtk_ae_workspace_bytes(h, side, B, N), "%s: workspace too small (%zu < %zu)", fn,
              workspace_bytes, vtk_ae_workspace_bytes(h, side, B, N));
  VTK_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0, "%s: workspace must be 1024-byte aligned", fn);
  return 0;
}

int vtk_ae_encode(vtk_ae_t h, const void* patches, const int64_t* row_idx, const int64_t* col_idx,
                  const uint8_t* patch_mask, int B, int N, void* z_out, void* workspace, size_t workspace_bytes,
                  void* stream) {
  int r = check_io(h, 0, patches, row_idx, col_idx, B, N, z_out, workspace, workspace_bytes, "vtk_ae_encode");
  if (r) return r;
  return run_side(h, 0, patches, row_idx, col_idx, patch_mask, B, N, z_out, workspace, (cudaStream_t)stream);
}

int vtk_ae_decode(vtk_ae_t h, const void* z, const int64_t* row_idx, const int64_t* col_idx, const uint8_t* patch_mask,
                  int B, int N, void* patches_out, void* workspace, size_t workspace_bytes, void* stream) {
  int r = check_io(h, 1, z, row_idx, col_idx, B, N, patches_out, workspace, workspace_bytes, "vtk_ae_decode");
  if (r) return r;
  return run_side(h, 1, z, row_idx, col_idx, patch_mask, B, N, patches_out, workspace, (cudaStream_t)stream);
}

int vtk_ae_set_norm_folded(vtk_ae_t h, int side, int folded) {
  VTK_REQUIRE(h && (side == 0 || side == 1), "vtk_ae_set_norm_folded: bad handle/side");
  Side& s = h->side[side];
  VTK_REQUIRE(!folded || (s.width > 0 && s.width % 256 == 0), "vtk_ae_set_norm_folded: the fused norm needs width %% 256 == 0 (width=%d)", s.width);
  s.norm_folded = folded != 0;
  return VTK_OK;
}

int vtk_ae_set_fp8_weights(vtk_ae_t h, int side, const vtk_block_fp8* blocks, int nblocks) {
  VTK_REQUIRE(h && (side == 0 || side == 1), "vtk_ae_set_fp8_weights: bad handle/side");
  Side& s = h->side[side];
  if (nblocks == 0) { s.fp8.clear(); return VTK_OK; }
  VTK_REQUIRE(blocks && nblocks == s.depth, "vtk_ae_set_fp8_weights: expected %d blocks, got %d", s.depth, nblocks);
  VTK_REQUIRE(s.norm_folded, "vtk_ae_set_fp8_weights: the FP8 path needs the fused norm1 (vtk_ae_set_norm_folded, width %% 256 == 0)");
  VTK_REQUIRE((s.width + s.hidden) % 16 == 0, "vtk_ae_set_fp8_weights: width + hidden must be a multiple of 16");
  for (int i = 0; i < nblocks; ++i)
    VTK_REQUIRE(blocks[i].w_in8 && blocks[i].w_out8 && blocks[i].w_in_scale > 0.f && blocks[i].w_out_scale > 0.f,
                "vtk_ae_set_fp8_weights: null pointer / non-positive scale in block %d", i);
  s.fp8.assign(blocks, blocks + nblocks);
  return VTK_OK;
}

int vtk_ae_set_fp8_granularity(vtk_ae_t h, int per_tensor) {
  VTK_REQUIRE(h, "vtk_ae_set_fp8_granularity: null handle");
  h->fp8_per_tensor = per_tensor != 0;
  return VTK_OK;
}

int vtk_ae_last_launch_count(vtk_ae_t h) { return h ? h->last_launches : 0; }

int vtk_ae_set_timing(vtk_ae_t h, int enable) {
  VTK_REQUIRE(h, "vtk_ae_set_timing: null handle");
  h->timing = enable != 0;
  h->ev_used = 0;
  return VTK_OK;
}

int vtk_ae_collect_timing(vtk_ae_t h, float* ms_by_class, int* launches_by_class) {
  VTK_REQUIRE(h && ms_by_class && launches_by_class, "vtk_ae_collect_timing: null pointer");
  for (int c = 0; c < CLS_COUNT; ++c) { ms_by_class[c] = 0.f; launches_by_class[c] = 0; }
  if (h->ev_used == 0) return VTK_OK;
  int r = check_cuda(cudaEventSynchronize(h->ev[2 * (h->ev_used - 1) + 1]), "cudaEventSynchronize(timing)");
  if (r) return r;
  for (int i = 0; i < h->ev_used; ++i) {
    float ms = 0.f;
    if ((r = check_cuda(cudaEventElapsedTime(&ms, h->ev[2 * i], h->ev[2 * i + 1]), "cudaEventElapsedTime"))) return r;
    ms_by_class[h->ev_cls[i]] += ms;
    launches_by_class[h->ev_cls[i]] += 1;
  }
  h->ev_used = 0;
  return VTK_OK;
}

}  // extern "C"
