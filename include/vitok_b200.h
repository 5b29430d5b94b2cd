/* vitok_b200.h -- C ABI of libvitok_b200.so: the drop-in boundary for the ViTok-v2 AE hot path.
 *
 * The reference (Na-VAE/vitok-release) has no FFI; its boundary for this path is the Python surface of
 * vitok/models/ae.py and vitok/pp.  Each entry point below names the reference call site it replaces
 * (paths relative to the reference repo root).  Conventions:
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream); no hidden syncs or
 *     allocations on the data path, so every call is CUDA-graph capturable;
 *   - every function returns 0 on success or a negative vtk_status; the message for the calling thread
 *     is available from vtk_last_error();
 *   - bf16 tensors are row-major; row strides are in elements and must be multiples of 8; base pointers
 *     16-byte aligned;
 *   - there is no CPU fallback: without a CUDA device every compute call fails with VTK_ERR_CUDA.
 */
#ifndef VITOK_B200_H_
#define VITOK_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define VTK_ABI_VERSION 6

typedef enum {
  VTK_OK = 0,
  VTK_ERR_CUDA = -1,        /* CUDA runtime / driver error, text in vtk_last_error()          -> RuntimeError */
  VTK_ERR_BAD_ARG = -2,     /* shape / alignment / null-pointer violation                      -> ValueError   */
  VTK_ERR_UNSUPPORTED = -3  /* valid in the reference but not implemented here (e.g. a head_dim outside d % 8 == 0, 8 <= d <= 128)
                               -> NotImplementedError */
} vtk_status;

const char* vtk_last_error(void);
int vtk_abi_version(void);
int vtk_sm_count(void); /* of the current device; <0 when no CUDA device is usable */
/* Runtime switches of the kernels (process-wide; no reference counterpart -- they select between implementations of the same
 * arithmetic).  "pdl": launch every kernel of the path with programmatic dependent launch (prologue overlaps the previous kernel's
 * tail; default 1, env VTK_PDL).  "gemm_splitk": split-K over the two CTA pairs of a 4-CTA cluster for the out_proj+fc2 residual
 * GEMM of small batches (<= 37 output tiles; default 1, env VTK_GEMM_SPLITK) -- the two K-halves are summed in fp32, so results
 * differ from the un-split kernel in the last bit of the accumulator; set 0 where bit-identical results across batch sizes
 * matter.  "reserve_sms" = n: the persistent kernels (GEMMs, d = 64 attention) size their grids for n SMs fewer (default 0, env
 * VTK_RESERVE_SMS) -- room for NCCL's all-reduce CTAs when the gradient exchange overlaps the backward pass.
 * Returns VTK_ERR_BAD_ARG for an unknown name. */
int vtk_set_flag(const char* name, int value);

/* ------------------------------------------------------------------------------------------------
 * NaFlex pre/post-processing                                   vitok/pp/ops.py, vitok/pp/io.py
 * ---------------------------------------------------------------------------------------------- */

/* patchify + patch_collate_fn for a whole batch.           vitok/pp/ops.py:217-285, vitok/data.py:77-94
 * images     : packed image buffer; img_table [B,3] int64 = {element offset, H, W} per image.
 * in_dtype   : 0 = float32 CHW already normalised; 1 = uint8 HWC (fuses to_tensor|normalize(minus_one_to_one),
 *              vitok/pp/ops.py:140-155).
 * out_dtype  : 0 = float32 (what the reference returns), 1 = bfloat16.
 * outputs    : patches [B,T,3p^2], patch_mask [B,T] (bool bytes), row/col/time_idx [B,T] int64,
 *              meta [4,B] int64 = orig_height, orig_width, grid_rows, grid_cols.
 * status     : optional device int, set to 1 if an image's grid exceeds max_tokens (the reference raises at :260).
 * max_h/max_w: a host-side hint, the largest image height / width of the batch (0 = unknown).  With the hint the uint8 front end
 *              runs a row-coalesced kernel over the batch's bounding box (thread = 4 pixels of an image row, 384 contiguous bytes
 *              per warp) with the normalisation done arithmetically; results are bit-identical to the call without it. */
int vtk_patchify_ex(const void* images, const int64_t* img_table, int in_dtype, int B, int patch, int max_tokens, int out_dtype,
                    void* patches, uint8_t* patch_mask, int64_t* row_idx, int64_t* col_idx, int64_t* time_idx, int64_t* meta, int* status,
                    int max_h, int max_w, void* stream);
/* resize_to_token_budget | patchify + patch_collate_fn for a ragged batch. vitok/pp/ops.py:169-214, :217-285, vitok/data.py:77-94
 * img_table  : [B,5] int64 = {element offset, H, W, h', w'} per image; (h', w') is the target size, normally
 *              _fit_to_token_budget(H, W, patch, max_tokens) (ops.py:169-196).  An axis whose size is unchanged is not resampled,
 *              so an image with (h', w') == (H, W) comes out bit-identical to vtk_patchify_ex.
 * resampling : TF.resize(BICUBIC, antialias=True) on the normalised fp32 image = ATen's _upsample_bicubic2d_aa (align_corners=False):
 *              cubic a = -0.5, support 2 * scale when shrinking, weights divided by their sum; width pass first, then height, each
 *              output summed in fp32 in tap order.  Weights equal torch's; outputs agree with TF.resize to a few fp32 ulps.
 * in_dtype / out_dtype / outputs: as vtk_patchify_ex; meta holds the RESIZED height and width (patchify sees the resized tensor).
 * workspace  : device memory of at least vtk_resize_patchify_workspace_bytes.  Layout: a header of 2B+3 int64 (rounded up to 256
 *              bytes): [0..B] = offset of each image's region in floats after the header, [B+1..2B+1] = row prefix of the width pass,
 *              [2B+2] = 1 if the batch was usable.  An image's region holds its resample tables (width then height; only for axes
 *              that change; [4*ceil(n_in/n_out)+3][n_out] floats, tap-major: row 0 = xmin and row 1 = tap count as int32 bits, then
 *              one row per tap of weights)
 *              and, if its width changes, the fp32 [3, H, w'] image of the width pass.
 * status     : optional device int: 1 if a target grid exceeds max_tokens (only for a target not produced by _fit_to_token_budget);
 *              2 if a size is < 1 or the workspace is too small (the resized images' patches are then left zero). */
int vtk_resize_patchify(const void* images, const int64_t* img_table, int in_dtype, int B, int patch, int max_tokens, int out_dtype,
                        void* patches, uint8_t* patch_mask, int64_t* row_idx, int64_t* col_idx, int64_t* time_idx, int64_t* meta,
                        void* workspace, size_t workspace_bytes, int* status, void* stream);
/* Workspace of vtk_resize_patchify for a batch: img_table_host = the same [B,5] table in HOST memory.  Header + per image the tables
 * and 3 * H * w' * 4 bytes of width-pass scratch (none for an image whose width is unchanged). */
size_t vtk_resize_patchify_workspace_bytes(const int64_t* img_table_host, int B);
/* test hook: *mismatches (device int) = number of uint8 values for which the arithmetic to_tensor|normalize of the row kernel differs
 * from the IEEE-division form (u / 255 - 0.5) / 0.5 of vitok/pp/ops.py:140-161; must be 0 */
int vtk_patchify_selftest(int* mismatches, void* stream);

/* max(row)+1, max(col)+1 over valid tokens -> out2[2] (device).        vitok/pp/ops.py:319-321 */
int vtk_grid_extent(const uint8_t* patch_mask, const int64_t* row_idx, const int64_t* col_idx, int B, int N, int* out2,
                    void* stream);

/* unpatchify (+ optional fused _convert_format).          vitok/pp/ops.py:295-335, vitok/pp/io.py:91-121
 * dtype      : 0 = float32, 1 = bfloat16 (patches and, unless out_format==1, the canvas).
 * cell_map   : workspace, B*gy*gx int32.
 * out        : [B,3,gy*p,gx*p].  out_format 0 = as is; 1 = uint8 "0_255"; 2 = "zero_to_one" (input is minus_one_to_one).
 * status     : optional device int, set to 1 if a valid token lies outside the canvas (reference: index error). */
int vtk_unpatchify(const void* patches, int dtype, const uint8_t* patch_mask, const int64_t* row_idx,
                   const int64_t* col_idx, int B, int N, int patch, int gy, int gx, int* cell_map, void* out,
                   int out_format, int* status, void* stream);

/* Per-tile SSIM of a NaFlex patch batch against its target, forward and backward: the SSIM tile loss of
 * scripts/train_vae.py:328-368 (the reference unpatchifies with torch fold / scatter, crops tiles and runs torchmetrics'
 * StructuralSimilarityIndexMeasure on them).  The canvas is read straight from the token layout, never written: pixel (y, x) of
 * image b is unpatchify's (vtk_unpatchify's cell map on the grid gy x gx; masked tokens and empty cells read 0), mapped to
 * [0, 1] by format 0 = minus_one_to_one ((v + 1) / 2) or 1 = zero_to_one (v), no clamping.  SSIM: 11 x 11 gaussian window,
 * sigma 1.5, K1 = 0.01, K2 = 0.03, data_range 1, per channel, averaged over the 3 channels and every window position lying
 * entirely inside the tile.
 * pred / target: [B, N, 3 p^2], dtype 0 = float32, 1 = bfloat16 each; patch_mask [B, N] bool bytes; row / col [B, N] int64.
 * tiles      : [T, 5] int32 (image, y0, x0, h, w) in canvas pixels; the caller keeps each inside its image (h, w >= 11).
 *              max_tile_h / max_tile_w bound every tile's h / w (they size the forward grid and the workspace).
 * out        : [T] fp32 tile values (vtk_ssim_fwd).  Per-tile sums run in a fixed order with no float atomics: bit-identical run to
 *              run, and a tile's value does not depend on the other tiles of the call.
 * gout, dpred: vtk_ssim_bwd writes dpred [B, N, 3 p^2] in pred's dtype = sum_t gout[t] d out[t] / d pred (recomputing the
 *              moments, nothing is kept from the forward); 0 for masked tokens, tokens that own no canvas pixel and pixels outside
 *              every tile.
 * workspace  : vtk_ssim_workspace_bytes(B, gy, gx, T, max_tile_h, max_tile_w) bytes of device memory (cell map + block sums). */
size_t vtk_ssim_workspace_bytes(int B, int gy, int gx, int T, int max_tile_h, int max_tile_w);
int vtk_ssim_fwd(const void* pred, int pred_dtype, const void* target, int target_dtype, const uint8_t* patch_mask,
                 const int64_t* row_idx, const int64_t* col_idx, int B, int N, int patch, int gy, int gx, const int* tiles, int T,
                 int max_tile_h, int max_tile_w, int format, float* out, void* workspace, size_t workspace_bytes, void* stream);
int vtk_ssim_bwd(const void* pred, int pred_dtype, const void* target, int target_dtype, const uint8_t* patch_mask,
                 const int64_t* row_idx, const int64_t* col_idx, int B, int N, int patch, int gy, int gx, const int* tiles, int T,
                 int max_tile_h, int max_tile_w, int format, const float* gout, void* dpred, void* workspace, size_t workspace_bytes,
                 void* stream);

/* ------------------------------------------------------------------------------------------------
 * Kernel-level entry points (used by the parity tests and by vtk_ae_* internally)
 * ---------------------------------------------------------------------------------------------- */

/* y = bf16(rms(x) * w), fp32 math, eps inside the rsqrt.                 vitok/models/modules/norm.py:17-25 */
int vtk_rmsnorm_bf16(const void* x, int64_t ldx, const void* w, void* y, int64_t ldy, int M, int D, float eps,
                     void* stream);

/* table [M,d] bf16 = cos | sin of the 2-D RoPE angles.     vitok/models/modules/rotary_embedding.py:46-75,118-119
 * inv_freq [d/4] float32 (device). */
int vtk_rope_table(const int64_t* row_idx, const int64_t* col_idx, const float* inv_freq, void* table, int M, int d,
                   void* stream);

int vtk_cast_f32_to_bf16(const float* in, void* out, int64_t n, void* stream);

/* kv_len[b] = 1 + last valid index: the key length of a prefix mask.   vitok/models/ae.py:173-187 */
int vtk_kv_len(const uint8_t* patch_mask, int* kv_len, int B, int N, void* stream);

/* NaFlex token packing plan for a masked [B, N] batch (replaces the reference's [B,1,N,N] mask, vitok/models/ae.py:173-187,
 * and its work on padded tokens).  Valid tokens are packed image after image, each image padded to `pad` rows (a multiple
 * of 8; the AE uses 16), and attention works on groups of `qrows` (128 or 256) query rows of one image:
 *   n_valid [B]                  valid tokens per image
 *   rel     [B*N]                rank of token t among the valid tokens of its image, -1 if masked
 *   cu      [B+1]                packed row offset of each image; cu[B] = packed row count (stays on the device)
 *   cuq     [B+1]                first attention group of each image; cuq[B] = number of groups
 *   grp_img [B*ceil(N/qrows)]    image of each group (entries >= cuq[B] are not written)
 *   grp_order[B*ceil(N/qrows)]   a permutation of the groups [0, cuq[B]), groups of images with more 128-key tiles first
 *                                (ties in any order): the work list the attention kernel deals to its CTAs
 *   src     [B*ceil(N/pad)*pad]  packed row -> source row b*N+t, -1 for pad rows (entries >= cu[B] are not written)
 * vtk_pack_rows gathers rows of `width` bf16 (packed[r] = in[src[r]], 0 for pad rows) for r < cu[B] (row_cap = capacity of
 * `packed` / `src`, sizes the grid); vtk_unpack_rows scatters them back (out[b,t] = packed[cu[b] + rel[b,t]], 0 for masked tokens). */
int vtk_pack_plan(const uint8_t* patch_mask, int B, int N, int pad, int qrows, int* n_valid, int* rel, int* cu, int* cuq,
                  int* grp_img, int* grp_order, int* src, void* stream);
int vtk_pack_rows(const void* in, int64_t ld_in, const int* src, const int* cu, int B, int64_t row_cap, void* packed, int64_t ld_packed,
                  int width, void* stream);
int vtk_unpack_rows(const void* packed, int64_t ld_packed, const int* rel, const int* cu, int B, int N, void* out,
                    int64_t ld_out, int width, void* stream);

/* out [M, N] = At^T Bt for At [K, M] and Bt [K, N] row-major (row strides lda / ldb): the weight gradient dW = dY^T X of the
 * training step without transposing either operand (the tensor core reads both tiles MN-major).  M, N multiples of 8. */
int vtk_linear_tn_bf16(const void* At, int64_t lda, const void* Bt, int64_t ldb, void* out, int64_t ldo, int M, int N, int K,
                       void* stream);

/* FP8 inference building blocks (reference AE.quantize, vitok/models/ae.py:253-270 = torchao
 * Float8DynamicActivationFloat8WeightConfig on the Linears of every block).
 * vtk_quant_rows_e4m3: dynamic per-row activation quantisation, q[row,:K] = e4m3(x[row,:K] / scale[row]), scale = amax / 448.
 * vtk_proj_residual_fp8: x += gamma * (scale_a[row] * w_scale * (A8 W8^T)) with e4m3 operands on the tcgen05 kind::f8f6f4 path
 * (lda / ldw / K in bytes = elements, multiples of 16). */
int vtk_quant_rows_e4m3(const void* x, int64_t ldx, void* q, int64_t ldq, float* scale, int M, int K, void* stream);
/* The same with ONE dynamic scale for the whole tensor (torchao's default PerTensor granularity of
 * Float8DynamicActivationFloat8WeightConfig, the reference's ae.py:253-270): amax_ws = one device float of workspace; scale[row] is
 * written for every row (all equal) so the GEMM epilogues are unchanged.  Costs one more read of x. */
int vtk_quant_tensor_e4m3(const void* x, int64_t ldx, void* q, int64_t ldq, float* scale, float* amax_ws, int M, int K, void* stream);
int vtk_proj_residual_fp8(const void* A8, int64_t lda, const float* a_scale, const void* W8, int64_t ldw, float w_scale,
                          const void* gamma, void* x, int64_t ldx, int M, int N, int K, void* stream);

/* out = bf16(A W^T + bias); bias may be null.                      nn.Linear: vitok/models/ae.py:191,220,242 */
int vtk_linear_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, const void* bias, void* out, int64_t ldo,
                    int M, int N, int K, void* stream);

/* out = LayerNorm_noaffine(bf16(A W^T + bias)), N = channels_per_token <= 256.   vitok/models/ae.py:207 */
int vtk_linear_ln_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, const void* bias, void* out, int64_t ldo,
                       int M, int N, int K, float eps, void* stream);

/* Fused first half of Block.forward after norm1 (vitok/models/ae.py:61-63):
 *   qkv_proj -> norm_q/norm_k -> 2-D RoPE (modules/attention.py:95-107) and fc1 -> silu(g)*v (modules/mlp.py:21-22).
 * Wp [w_rows, K=D] is the packed weight [Wq; Wk; Wv; 0-pad to qp; interleave16(W1_v, W1_g)]; qp = 3D rounded up to 256.
 * qkv [M,3D] receives roped q, roped k, v; act [M,Hf] receives silu(g)*v.  head_dim d: d % 8 == 0, 8 <= d <= 128.  At d = 32, 64 and
 * 128 the GEMM epilogue normalises and ropes q / k; at the other d it writes them raw and vtk_qk_norm_rope_fwd runs in place on
 * qkv after the GEMM, on the same stream (same rounding points). */
int vtk_qkv_swiglu_bf16(const void* h, int64_t ldh, const void* Wp, int64_t ldw, int64_t w_rows, int M, int D, int d,
                        int Hf, int qp, const void* norm_q, const void* norm_k, const void* rope_table, float eps,
                        void* qkv, int64_t ld_qkv, void* act, int64_t ld_act, void* stream);

/* Fused second half: x = bf16(x + bf16(bf16(A W^T) * gamma)) with A = [attn | act], W = [Wout | Wfc2]
 * (modules/attention.py:129, modules/mlp.py:22, modules/layerscale.py:23, vitok/models/ae.py:64-65). */
int vtk_proj_residual_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, const void* gamma, void* x,
                           int64_t ldx, int M, int N, int K, void* stream);

/* softmax(q k^T / sqrt(d)) v per (image, head); q,k,v,out rows = tokens, heads along columns.
 * kv_len null = no masking (reference flash backend, modules/attention.py:109-117); otherwise image b attends to its first
 * kv_len[b] keys: the sdpa backend's key masking (modules/attention.py:118-127) for a prefix mask (vtk_kv_len).
 * zero_invalid_rows = 1: query rows >= kv_len[b] are written as 0 (lse +inf).
 * window >= 0: sliding-window attention, query i sees keys j with |i - j| <= window on the token index, i.e.
 * flash_attn_func(window_size=(window, window)) as called at modules/attention.py:113-116; window < 0 = full.
 * lse (optional, may be null): [B*N, heads] fp32, log2-domain logsumexp of the scaled scores (+inf for zeroed rows);
 * the training backward (vtk_attention_bwd_bf16) consumes it.
 * head_dim d: d % 8 == 0 and 8 <= d <= 128 (else VTK_ERR_UNSUPPORTED).  d <= 64 runs on the d = 64 kernel, 64 < d <= 128 on the
 * d = 128 one; only the d columns of each head are read and written.  Row strides and q / k / v / out: multiples of 8 elements. */
int vtk_attention_bf16(const void* q, const void* k, const void* v, int64_t ld_qkv, void* out, int64_t ld_out,
                       const int* kv_len, int B, int N, int heads, int d, int zero_invalid_rows, int window, float* lse, void* stream);
/* The same on the packed NaFlex layout of vtk_pack_plan (the form the layer stack runs masked batches in): image b owns packed rows
 * [cu[b], cu[b+1]) with its n_valid[b] tokens in front; q / k / v / out have row_cap rows.  qrows of the plan must be 128 (d <= 64)
 * or 256 (64 < d <= 128).  For image b it writes packed rows [cu[b], cu[b+1]) only, and rows below n_valid[b] get out as
 * vtk_attention_bf16 with kv_len = n_valid.  Rows of other images -- the rest of a partial last tile -- are not touched.
 * lse (optional, may be null; the training step on packed rows, vitok/models/modules/attention.py:118-127 under autograd):
 * [row_cap, heads] fp32.  With lse, the image's pad rows [cu[b] + n_valid[b], cu[b+1]) get out = 0 and lse = +inf; without it,
 * they are not written. */
int vtk_attention_packed_lse_bf16(const void* q, const void* k, const void* v, int64_t ld_qkv, void* out, int64_t ld_out,
                                  const int* n_valid, const int* cu, const int* cuq, const int* grp_img, const int* grp_order, int B, int N,
                                  int heads, int d, int64_t row_cap, int grp_cap, float* lse, void* stream);

/* out [M,N] (+)= A [M,K] @ Bt [K,N] with B read as stored: the data gradient dX = dY W with the weight W [out, in] used as stored.
 * accumulate != 0 adds to what `out` already holds, in fp32 before the bf16 rounding (dh = dz_qkv Wqkv + dz_fc1 W1 without a
 * separate add pass). */
int vtk_linear_nn_acc_bf16(const void* A, int64_t lda, const void* Bt, int64_t ldb, void* out, int64_t ldo, int M, int N, int K,
                           int accumulate, void* stream);
/* out [M,N] = A[:, :K0] W0^T + A[:, K0:K0+K1] W1^T with W0 [N,K0], W1 [N,K1] as stored: out_proj(attn) + fc2(act)
 * (modules/attention.py:129 + modules/mlp.py:22) over the concatenated activations WITHOUT a packed [out_proj | fc2] copy -- the
 * training step's weights change every step.  One accumulator when K0 is a multiple of 64 (pair kernel), else two GEMMs. */
int vtk_linear2_bf16(const void* A, int64_t lda, const void* W0, int64_t ldw0, const void* W1, int64_t ldw1, void* out, int64_t ldo,
                     int M, int N, int K0, int K1, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Training step (BASELINE config 5; scripts/train_vae.py:304-320,371-372 = forward, Charbonnier loss, backward,
 * AdamW).  The GEMMs of forward and backward are vtk_linear_bf16 (forward), vtk_linear2_bf16 (out_proj + fc2),
 * vtk_linear_nn_acc_bf16 (dgrad against the weights as stored) and vtk_linear_tn_bf16 (wgrad) calls; everything else is
 * below.  All tensors bf16 unless noted; gradient accumulators of norm weights / gamma / biases are fp32 and ADDED to (zero
 * them first).
 * ---------------------------------------------------------------------------------------------- */
/* zraw [M, >=3D] raw q|k|v -> qkv [M,3D]: QK-RMSNorm over d + 2D RoPE, v copied (modules/attention.py:95-107).
 * d % 8 == 0, 8 <= d <= 128.  qkv == zraw (with ld_qkv == ldz) runs in place and leaves v as it is. */
int vtk_qk_norm_rope_fwd(const void* zraw, int64_t ldz, const void* norm_q, const void* norm_k, const void* rope_table,
                         void* qkv, int64_t ld_qkv, int M, int heads, int d, float eps, void* stream);
/* zraw[:, qp:] (16-col groups value|gate, the packed fc1 order) -> act [M,Hf] = silu(g) * v (modules/mlp.py:21-22) */
/* layout: 0 = 16-column (value16 | gate16) groups (the packed w_in of the inference path), 1 = [value Hf | gate Hf] (fc1 rows as stored) */
int vtk_swiglu_fwd(const void* zraw, int64_t ldz, int qp, void* act, int64_t ld_act, int M, int Hf, int layout, void* stream);
/* out = x + gamma * y (vitok/models/ae.py:64-65); contiguous [M,D].  With stochastic depth (drop_path, vitok/models/ae.py:15-30,65;
 * decoder blocks in train mode): keep [B] fp32 holds the per-image draw floor(keep_prob + U[0,1)) in {0, 1}, image b = rows
 * [b * rows_per_image, (b+1) * rows_per_image): out = x + bf16(bf16(gamma * y) / keep_prob) * keep[b].  keep == NULL: no
 * stochastic depth. */
int vtk_resid_fwd_dp(const void* x, const void* y, const void* gamma, void* out, int M, int D, const float* keep, int rows_per_image,
                     float keep_prob, void* stream);
/* backward of vtk_resid_fwd_dp: the LayerScale output's gradient is bf16(dx * keep[b] / keep_prob); dy = that * gamma,
 * dgamma[D] += colsum(that * y).  keep == NULL: dy = dx * gamma, dgamma[D] += colsum(dx * y) */
int vtk_resid_bwd_dp(const void* dx, const void* y, const void* gamma, void* dy, float* dgamma, int M, int D, const float* keep,
                     int rows_per_image, float keep_prob, void* stream);
/* out = LayerNorm_noaffine(x) over C <= 256 (modules/norm.py:28-39) */
int vtk_layernorm_fwd(const void* x, void* out, int M, int C, float eps, void* stream);
/* out[C] += colsum(in [M,C]) (bias gradients) */
int vtk_colsum(const void* in, int64_t ld, float* out, int M, int C, void* stream);
/* d_act [M,Hf] + zraw -> dz[:, qp:] in the packed (value|gate) order */
int vtk_swiglu_bwd(const void* dact, int64_t ldd, const void* zraw, int64_t ldz, int qp, void* dz, int64_t lddz, int M, int Hf, int layout,
                   void* stream);
/* in place on dz[:, 0:2D] (dq|dk w.r.t. roped q/k) -> gradient w.r.t. raw q/k; dw [2][d] fp32 += norm_q / norm_k grads;
 * d % 8 == 0, 8 <= d <= 128 */
int vtk_qk_norm_rope_bwd(void* dz, int64_t lddz, const void* zraw, int64_t ldz, const void* norm_q, const void* norm_k,
                         const void* rope_table, float* dw, int M, int heads, int d, float eps, void* stream);
/* dx_out = dx_res + RMSNorm'(x; w)^T dh; dw[D] += colsum(dh * xhat) */
int vtk_rmsnorm_bwd(const void* x, const void* dh, const void* w, const void* dx_res, void* dx_out, float* dw, int M, int D,
                    float eps, void* stream);
int vtk_layernorm_bwd(const void* zlin, const void* dz, void* dx, int M, int C, float eps, void* stream);
/* Charbonnier loss (scripts/train_vae.py:314-320): loss_sum[B] fp32 += per-image masked mean (caller zeroes it and takes the
 * batch mean); dpred (optional) = d(batch-mean loss)/d pred; n_valid[B] int32 = clamp_min(patch_mask.sum(1), 1) */
int vtk_charbonnier(const void* pred, const void* target, const uint8_t* patch_mask, const int* n_valid, float* loss_sum,
                    void* dpred, int B, int N, int P, float eps, void* stream);
/* Multi-tensor AdamW with the reference's optimizer precision (scripts/train_vae.py:200-208: fp32 parameters and fp32 Adam moments under
 * autocast).  Per tensor: `master` = fp32 parameter values (for an fp32 model parameter: the parameter itself), `p16` = the bf16 model
 * parameter re-emitted from the master in the same pass (NULL for fp32 parameters), `g` = gradient (bf16, or fp32 when g_is_f32),
 * `m` / `v` = fp32 exp_avg / exp_avg_sq; torch.optim.AdamW semantics (decoupled weight decay, bias correction with `step` >= 1).
 * The table is read on the host; all tensor pointers are device pointers. */
typedef struct {
  float* master; void* p16; const void* g; float* m; float* v; long long n; float weight_decay; int g_is_f32;
} vtk_adamw_tensor;
int vtk_adamw_multi(const vtk_adamw_tensor* tensors, int n_tensors, float lr, float beta1, float beta2, float eps, int step,
                    float grad_scale, void* stream);
/* vtk_adamw_multi with gradient clipping and an EMA of the master weights in the same pass (vtk_adamw_multi = this with NULL, NULL).
 *   coef (optional): fp32 device scalar, e.g. norm_coef + 1 of vtk_grad_norm_finish; every gradient is multiplied by it after
 *     grad_scale (coef == 1 gives the unclipped step bit for bit).
 *   ema (optional): one fp32 device pointer of n elements per table entry (host array); after the update
 *     ema = lerp(ema, master, w) with w = (float)(1 - ema_decay), 0 <= ema_decay < 1, in torch.lerp's fp32 arithmetic -- the
 *     weight is formed in double, as torch._foreach_lerp_(ema, master, 1 - ema_decay) forms it from a Python float.
 * HBM traffic per bf16 parameter: 28 bytes; with ema 36. */
int vtk_adamw_multi_ex(const vtk_adamw_tensor* tensors, float* const* ema, int n_tensors, float lr, float beta1, float beta2, float eps,
                       int step, float grad_scale, const float* coef, double ema_decay, void* stream);
/* Global L2 norm of the gradients of a vtk_adamw_tensor table (only g, n and g_is_f32 are read), deterministic and without a host
 * sync.  vtk_grad_sumsq_multi writes partials[slot0 + j] = fp32 sum of g^2 over the j-th 8192-element chunk of the table
 * (chunks numbered tensor by tensor; vtk_grad_norm_slots(table) of them), so several calls can fill one workspace;
 * vtk_grad_norm_finish then sums partials[0, n_slots) in a fixed order in double and writes norm_coef[0] = the norm (fp32) and
 * norm_coef[1] = clamp(max_norm / (norm + 1e-6), max = 1), the clip coefficient of torch.nn.utils.clip_grad_norm_ (NaN for a NaN
 * norm, 0 for an inf norm; max_norm = inf never clips a finite norm).  HBM traffic: one read of the gradients, 2 bytes per bf16
 * value and 4 per fp32 value. */
int64_t vtk_grad_norm_slots(const vtk_adamw_tensor* tensors, int n_tensors);
int vtk_grad_sumsq_multi(const vtk_adamw_tensor* tensors, int n_tensors, float* partials, int64_t slot0, void* stream);
int vtk_grad_norm_finish(const float* partials, int64_t n_slots, float max_norm, float* norm_coef, void* stream);
/* x [n] bf16 *= *scale (fp32 scalar in device memory): the loss gradient arriving at vtk_charbonnier's dpred */
int vtk_scale_by_dev(void* x, const float* scale, int64_t n, void* stream);
/* delta [M, heads] fp32 = rowsum over d of dO * O; d % 8 == 0, 8 <= d <= 128 */
int vtk_attn_delta(const void* o, int64_t ldo, const void* dout, int64_t lddo, float* delta, int M, int heads, int d, void* stream);
/* attention backward: dq, dk, dv (row stride ld_d) from q,k,v,dO, lse (from vtk_attention_bf16) and delta; the head dims of
 * vtk_attention_bf16, only the d columns of each head written */
int vtk_attention_bwd_bf16(const void* q, const void* k, const void* v, int64_t ld_qkv, const void* dout, int64_t ld_do,
                           const float* lse, const float* delta, void* dq, void* dk, void* dv, int64_t ld_d, const int* kv_len,
                           int B, int N, int heads, int d, int zero_invalid_rows, int window, void* stream);
/* The same on the packed NaFlex layout (autograd of modules/attention.py:118-127 for the packed training step), same head dims:
 * lse from vtk_attention_packed_lse_bf16, delta [row_cap, heads] from vtk_attn_delta over the packed rows.  The plan must have
 * qrows = 128 at every head dim (the forward's plan at 64 < d <= 128 has qrows = 256: a second plan of the same mask, whose n_valid / cu
 * are the same).  Two passes, each one CTA per (128-row group, head) taken in grp_order: dK/dV per key tile, then dQ per query
 * tile; grp_cap (>= cuq[B], CTAs beyond cuq[B] exit) sizes the grid.  For image b it writes dq / dk / dv rows [cu[b], cu[b+1])
 * only: gradients for rows below n_valid[b], zeros for the image's pad rows; rows of other images are not touched.  Query rows
 * past n_valid[b] in a partial last tile (the next image's rows) contribute nothing to dK / dV whatever their dO. */
int vtk_attention_bwd_packed_bf16(const void* q, const void* k, const void* v, int64_t ld_qkv, const void* dout, int64_t ld_do,
                                  const float* lse, const float* delta, void* dq, void* dk, void* dv, int64_t ld_d, const int* n_valid,
                                  const int* cu, const int* cuq, const int* grp_img, const int* grp_order, int B, int heads, int d,
                                  int64_t row_cap, int grp_cap, void* stream);

/* test-only: D[128,N] fp32 = A[128,K] * op(B) through one tcgen05 tile with explicit descriptor fields */
int vtk_umma_probe(const void* A, const void* B, float* D, int N, int K, int b_mn_major, uint32_t lbo_bytes,
                   uint32_t sbo_bytes, uint32_t kstep_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Whole-model entry points                                       vitok/models/ae.py:68-251 (class AE)
 * ---------------------------------------------------------------------------------------------- */
typedef struct vtk_ae_s* vtk_ae_t;

typedef struct {
  int32_t pixels_per_token, channels_per_token;
  int32_t enc_width, enc_depth, enc_heads, enc_hidden; /* hidden = SwiGLU Hf; depth 0 = side absent */
  int32_t dec_width, dec_depth, dec_heads, dec_hidden;
  float norm_eps;                                       /* 1e-6 */
  int32_t sliding_window;                               /* AE(sw=...), vitok/models/ae.py:90,99; <= 0 = full attention */
} vtk_ae_config;

typedef struct {
  const void* w_in;   /* packed [qp + 2*Hf, D]: see vtk_qkv_swiglu_bf16 */
  const void* w_out;  /* packed [D, Kp] = [out_proj | fc2 | 0-pad], Kp = D + Hf rounded up to a multiple of 64 */
  const void* norm1;  /* [D] */
  const void* norm_q; /* [d] */
  const void* norm_k; /* [d] */
  const void* gamma;  /* [D] (ones when use_layer_scale=False) */
} vtk_block_weights;

/* The handle stores pointers only (weights stay owned by the caller) plus a small device table of RoPE
 * inverse frequencies it allocates itself. */
int vtk_ae_create(const vtk_ae_config* cfg, vtk_ae_t* out);
int vtk_ae_destroy(vtk_ae_t h);
/* side 0 = encoder (w_a = patch_embed, w_b = to_code), 1 = decoder (w_a = decoder_embed, w_b = to_pixels) */
int vtk_ae_set_weights(vtk_ae_t h, int side, const void* w_a, const void* b_a, const void* w_b, const void* b_b,
                       const vtk_block_weights* blocks, int nblocks, const float* inv_freq_host, int n_inv_freq);
size_t vtk_ae_workspace_bytes(vtk_ae_t h, int side, int B, int N);
/* AE.encode (vitok/models/ae.py:189-216): patches [B,N,P] bf16 -> z [B,N,C] bf16.  patch_mask null = flash semantics.
 * NaFlex token packing: when a patch_mask is given, vtk_ae_encode/decode gather the valid tokens of every image into a packed
 * row range (each image padded to 16 rows), run every kernel of the layer stack over the packed rows only -- the packed row count
 * stays in device memory, nothing syncs -- and scatter the result back; masked tokens of the output are 0.  This replaces the
 * reference's [B,1,N,N] mask (vitok/models/ae.py:173-187) and its work on padded tokens.  A side without blocks keeps the padded
 * rows (it has no attention to mask). */
int vtk_ae_encode(vtk_ae_t h, const void* patches, const int64_t* row_idx, const int64_t* col_idx,
                  const uint8_t* patch_mask, int B, int N, void* z_out, void* workspace, size_t workspace_bytes,
                  void* stream);
/* AE.decode (vitok/models/ae.py:218-243): z [B,N,C] bf16 -> patches [B,N,P] bf16. */
int vtk_ae_decode(vtk_ae_t h, const void* z, const int64_t* row_idx, const int64_t* col_idx, const uint8_t* patch_mask,
                  int B, int N, void* patches_out, void* workspace, size_t workspace_bytes, void* stream);
/* Fused Block.norm1 (vitok/models/ae.py:55, modules/norm.py:17-25).  Call after vtk_ae_set_weights with folded = 1 when
 * every block's w_in of that side was packed with norm1.weight multiplied into its columns (W'[j,k] = W[j,k] * w[k]).
 * Then no RMSNorm kernel runs: the GEMM that produces x (patch/decoder embed, out_proj+fc2 residual) also writes the
 * per-row sums of squares, and the QKV+fc1 GEMM reads x directly and scales every accumulator row by
 * rsqrt(mean(x^2) + eps): h W^T = rstd * (x (W*w)^T).  Needs width % 256 == 0.  folded = 0 (default): separate RMSNorm. */
int vtk_ae_set_norm_folded(vtk_ae_t h, int side, int folded);
/* FP8 inference (AE.quantize, vitok/models/ae.py:253-270).  After vtk_ae_set_weights + vtk_ae_set_norm_folded(.., 1): hand over, per
 * block, e4m3 copies of the packed weights (w_in8 [qp + 2*Hf, D], w_out8 [D, Kp], one byte per element, same packing and row
 * pitches in ELEMENTS as the bf16 ones) and their per-tensor scales (w ~= w8 * scale).  From then on the two GEMMs of every
 * block of that side run on the tcgen05 kind::f8f6f4 path: their A operands (x, [attn | act]) are quantised per row on the fly
 * (vtk_quant_rows_e4m3) and the epilogues rescale the accumulators; attention, embeds and the latent bottleneck stay bf16.
 * nblocks = 0 switches the side back to bf16.  The pointers must stay valid (caller-owned), like the bf16 weights. */
typedef struct vtk_block_fp8 {
  const void* w_in8;
  const void* w_out8;
  float w_in_scale;
  float w_out_scale;
} vtk_block_fp8;
int vtk_ae_set_fp8_weights(vtk_ae_t h, int side, const vtk_block_fp8* blocks, int nblocks);
/* FP8 activation scale granularity of the quantised block GEMMs: 0 = per row (default: finer, no extra pass), 1 = per tensor
 * (torchao-equivalent numerics). */
int vtk_ae_set_fp8_granularity(vtk_ae_t h, int per_tensor);
/* number of kernels launched by the last vtk_ae_encode/decode on this handle (for gpu_launches accounting) */
int vtk_ae_last_launch_count(vtk_ae_t h);
/* Optional per-launch CUDA-event timing (bench.py's live roofline).  With timing enabled every kernel launched by
 * vtk_ae_encode/decode is bracketed by an event pair on `stream`; vtk_ae_collect_timing synchronises on the last
 * event and returns the summed milliseconds and launch counts per kernel class:
 * 0 linear, 1 rmsnorm, 2 qkv+swiglu GEMM, 3 attention, 4 out_proj+fc2 residual GEMM, 5 misc (6 entries each). */
int vtk_ae_set_timing(vtk_ae_t h, int enable);
int vtk_ae_collect_timing(vtk_ae_t h, float* ms_by_class_host, int* launches_by_class_host);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* VITOK_B200_H_ */
