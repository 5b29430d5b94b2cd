"""ctypes binding of libvitok_b200.so (the C ABI declared in include/vitok_b200.h).

There is NO fallback: if the shared library is missing or a tensor is not on a
CUDA device the call raises.  torch is used only for device memory and the
current stream.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvitok_b200.so")

VTK_OK, VTK_ERR_CUDA, VTK_ERR_BAD_ARG, VTK_ERR_UNSUPPORTED = 0, -1, -2, -3

c_int, c_i64, c_f32, c_vp, c_u32, c_sz = (ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p,
                                          ctypes.c_uint32, ctypes.c_size_t)


class AEConfig(ctypes.Structure):
    _fields_ = [("pixels_per_token", ctypes.c_int32), ("channels_per_token", ctypes.c_int32),
                ("enc_width", ctypes.c_int32), ("enc_depth", ctypes.c_int32), ("enc_heads", ctypes.c_int32),
                ("enc_hidden", ctypes.c_int32),
                ("dec_width", ctypes.c_int32), ("dec_depth", ctypes.c_int32), ("dec_heads", ctypes.c_int32),
                ("dec_hidden", ctypes.c_int32),
                ("norm_eps", ctypes.c_float), ("sliding_window", ctypes.c_int32)]


class BlockWeights(ctypes.Structure):
    _fields_ = [("w_in", c_vp), ("w_out", c_vp), ("norm1", c_vp), ("norm_q", c_vp), ("norm_k", c_vp), ("gamma", c_vp)]


class BlockFp8(ctypes.Structure):
    _fields_ = [("w_in8", c_vp), ("w_out8", c_vp), ("w_in_scale", ctypes.c_float), ("w_out_scale", ctypes.c_float)]


class AdamwTensor(ctypes.Structure):
    _fields_ = [("master", c_vp), ("p16", c_vp), ("g", c_vp), ("m", c_vp), ("v", c_vp), ("n", ctypes.c_longlong),
                ("weight_decay", ctypes.c_float), ("g_is_f32", ctypes.c_int)]


# name -> (restype, argtypes); must list every symbol include/vitok_b200.h declares
SIGNATURES = {
    "vtk_last_error": (ctypes.c_char_p, []),
    "vtk_abi_version": (c_int, []),
    "vtk_sm_count": (c_int, []),
    "vtk_set_flag": (c_int, [ctypes.c_char_p, c_int]),
    "vtk_patchify_ex": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_vp]),
    "vtk_resize_patchify": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_sz,
                                    c_vp, c_vp]),
    "vtk_resize_patchify_workspace_bytes": (c_sz, [c_vp, c_int]),
    "vtk_patchify_selftest": (c_int, [c_vp, c_vp]),
    "vtk_grid_extent": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp]),
    "vtk_unpatchify": (c_int, [c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_int, c_vp, c_vp]),
    "vtk_ssim_workspace_bytes": (c_sz, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "vtk_ssim_fwd": (c_int, [c_vp, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_vp, c_int, c_int, c_int,
                             c_int, c_vp, c_vp, c_sz, c_vp]),
    "vtk_ssim_bwd": (c_int, [c_vp, c_int, c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_vp, c_int, c_int, c_int,
                             c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "vtk_rmsnorm_bf16": (c_int, [c_vp, c_i64, c_vp, c_vp, c_i64, c_int, c_int, c_f32, c_vp]),
    "vtk_rope_table": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_vp]),
    "vtk_cast_f32_to_bf16": (c_int, [c_vp, c_vp, c_i64, c_vp]),
    "vtk_kv_len": (c_int, [c_vp, c_vp, c_int, c_int, c_vp]),
    "vtk_pack_plan": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "vtk_pack_rows": (c_int, [c_vp, c_i64, c_vp, c_vp, c_int, c_i64, c_vp, c_i64, c_int, c_vp]),
    "vtk_unpack_rows": (c_int, [c_vp, c_i64, c_vp, c_vp, c_int, c_int, c_vp, c_i64, c_int, c_vp]),
    "vtk_quant_rows_e4m3": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_int, c_int, c_vp]),
    "vtk_quant_tensor_e4m3": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_int, c_int, c_vp]),
    "vtk_proj_residual_fp8": (c_int, [c_vp, c_i64, c_vp, c_vp, c_i64, c_f32, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_vp]),
    "vtk_linear_bf16": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_vp]),
    "vtk_linear_tn_bf16": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_int, c_int, c_int, c_vp]),
    "vtk_linear_nn_acc_bf16": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_int, c_int, c_int, c_int, c_vp]),
    "vtk_linear2_bf16": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_int, c_int, c_int, c_int, c_vp]),
    "vtk_resid_fwd_dp": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_int, c_f32, c_vp]),
    "vtk_resid_bwd_dp": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_int, c_f32, c_vp]),
    "vtk_adamw_multi": (c_int, [ctypes.POINTER(AdamwTensor), c_int, c_f32, c_f32, c_f32, c_f32, c_int, c_f32, c_vp]),
    "vtk_adamw_multi_ex": (c_int, [ctypes.POINTER(AdamwTensor), ctypes.POINTER(c_vp), c_int, c_f32, c_f32, c_f32, c_f32, c_int, c_f32,
                                   c_vp, ctypes.c_double, c_vp]),
    "vtk_grad_norm_slots": (c_i64, [ctypes.POINTER(AdamwTensor), c_int]),
    "vtk_grad_sumsq_multi": (c_int, [ctypes.POINTER(AdamwTensor), c_int, c_vp, c_i64, c_vp]),
    "vtk_grad_norm_finish": (c_int, [c_vp, c_i64, c_f32, c_vp, c_vp]),
    "vtk_scale_by_dev": (c_int, [c_vp, c_vp, c_i64, c_vp]),
    "vtk_linear_ln_bf16": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_f32, c_vp]),
    "vtk_qkv_swiglu_bf16": (c_int, [c_vp, c_i64, c_vp, c_i64, c_i64, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp,
                                    c_f32, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "vtk_proj_residual_bf16": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_vp]),
    "vtk_attention_bf16": (c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp]),
    "vtk_attention_packed_lse_bf16": (c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int,
                                              c_int, c_i64, c_int, c_vp, c_vp]),
    "vtk_qk_norm_rope_fwd": (c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_int, c_f32, c_vp]),
    "vtk_swiglu_fwd": (c_int, [c_vp, c_i64, c_int, c_vp, c_i64, c_int, c_int, c_int, c_vp]),
    "vtk_layernorm_fwd": (c_int, [c_vp, c_vp, c_int, c_int, c_f32, c_vp]),
    "vtk_colsum": (c_int, [c_vp, c_i64, c_vp, c_int, c_int, c_vp]),
    "vtk_swiglu_bwd": (c_int, [c_vp, c_i64, c_vp, c_i64, c_int, c_vp, c_i64, c_int, c_int, c_int, c_vp]),
    "vtk_qk_norm_rope_bwd": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_f32, c_vp]),
    "vtk_rmsnorm_bwd": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_f32, c_vp]),
    "vtk_layernorm_bwd": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_f32, c_vp]),
    "vtk_charbonnier": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_f32, c_vp]),
    "vtk_attn_delta": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_int, c_int, c_int, c_vp]),
    "vtk_attention_bwd_bf16": (c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp,
                                       c_int, c_int, c_int, c_int, c_int, c_int, c_vp]),
    "vtk_attention_bwd_packed_bf16": (c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp,
                                              c_vp, c_vp, c_vp, c_int, c_int, c_int, c_i64, c_int, c_vp]),
    "vtk_umma_probe": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_int, c_u32, c_u32, c_u32, c_vp]),
    "vtk_ae_create": (c_int, [ctypes.POINTER(AEConfig), ctypes.POINTER(c_vp)]),
    "vtk_ae_destroy": (c_int, [c_vp]),
    "vtk_ae_set_weights": (c_int, [c_vp, c_int, c_vp, c_vp, c_vp, c_vp, ctypes.POINTER(BlockWeights), c_int,
                                   ctypes.POINTER(c_f32), c_int]),
    "vtk_ae_workspace_bytes": (c_sz, [c_vp, c_int, c_int, c_int]),
    "vtk_ae_encode": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_sz, c_vp]),
    "vtk_ae_decode": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_sz, c_vp]),
    "vtk_ae_last_launch_count": (c_int, [c_vp]),
    "vtk_ae_set_timing": (c_int, [c_vp, c_int]),
    "vtk_ae_set_fp8_granularity": (c_int, [c_vp, c_int]),
    "vtk_ae_set_fp8_weights": (c_int, [c_vp, c_int, ctypes.POINTER(BlockFp8), c_int]),
    "vtk_ae_set_norm_folded": (c_int, [c_vp, c_int, c_int]),
    "vtk_ae_collect_timing": (c_int, [c_vp, ctypes.POINTER(c_f32), ctypes.POINTER(c_int)]),
}

_lib: Optional[ctypes.CDLL] = None


def load() -> ctypes.CDLL:
    """dlopen the in-tree library and type every export.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: the sm_100a CUDA library has not been built "
            "(run `python vitok-release_b200/build.py`).  vitok_b200 has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def set_flag(name: str, value: int) -> None:
    """Process-wide kernel switch (include/vitok_b200.h: vtk_set_flag): "pdl", "gemm_splitk", "reserve_sms" (the persistent
    kernels -- GEMMs and attention at d <= 64 -- size their grids for that many SMs fewer)."""
    check(load().vtk_set_flag(name.encode(), int(value)))


def last_error() -> str:
    return (load().vtk_last_error() or b"").decode("utf-8", "replace")


def check(rc: int) -> None:
    if rc == VTK_OK:
        return
    msg = last_error()
    if rc == VTK_ERR_BAD_ARG:
        raise ValueError(msg)
    if rc == VTK_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(msg)


def stream_ptr() -> int:
    """Current stream of the CURRENT device: call under ``device_of(tensor)`` so that it is the tensors' device."""
    return torch.cuda.current_stream().cuda_stream


def device_of(*tensors) -> "torch.cuda.device":
    """Context manager that makes the CUDA device of ``tensors`` current for the C calls inside it (kernel launches,
    tensor-map encoding, ``stream_ptr()`` and the per-device SM count all use the current device).  Raises on tensors
    that live on different devices or on the host."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("vitok_b200: tensors must live on a CUDA device (there is no CPU path)")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"vitok_b200: tensors on different devices ({dev} and {t.device})")
    if dev is None:
        raise RuntimeError("vitok_b200: no CUDA tensor given")
    return torch.cuda.device(dev)


def _on_device(fn):
    """Run ``fn`` with the device of its first tensor argument current (see device_of)."""
    import functools

    @functools.wraps(fn)
    def wrapped(*args, **kwargs):
        first = next((a for a in args if isinstance(a, torch.Tensor)), None)
        if first is None or not first.is_cuda:
            return fn(*args, **kwargs)      # the wrapper's own checks raise the "no CPU path" error
        with torch.cuda.device(first.device):
            return fn(*args, **kwargs)
    return wrapped


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("vitok_b200: tensors must live on a CUDA device (there is no CPU path)")
    return t.data_ptr()


def _req(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"vitok_b200: {name} must be a CUDA tensor (there is no CPU path)")
    if t.dtype != dtype:
        raise RuntimeError(f"vitok_b200: {name} must have dtype {dtype}, got {t.dtype}")
    if t.stride(-1) != 1:
        raise ValueError(f"vitok_b200: {name} must be contiguous in its last dimension")
    return t


# ---------------------------------------------------------------------------
# thin kernel-level wrappers (used by the parity tests; the model path goes
# through vtk_ae_encode / vtk_ae_decode)
# ---------------------------------------------------------------------------
@_on_device
def linear(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None) -> torch.Tensor:
    _req(a, torch.bfloat16, "a"); _req(w, torch.bfloat16, "w")
    M, K = a.shape
    N = w.shape[0]
    out = torch.empty(M, N, dtype=torch.bfloat16, device=a.device)
    check(load().vtk_linear_bf16(ptr(a), a.stride(0), ptr(w), w.stride(0), ptr(bias), ptr(out), out.stride(0), M, N, K,
                                 stream_ptr()))
    return out


@_on_device
def linear_tn(at: torch.Tensor, bt: torch.Tensor) -> torch.Tensor:
    """out [M, N] = at^T @ bt for at [K, M], bt [K, N] (row-major, any row pitch): transposed-operand GEMM."""
    _req(at, torch.bfloat16, "at"); _req(bt, torch.bfloat16, "bt")
    K, M = at.shape
    N = bt.shape[1]
    out = torch.empty(M, N, dtype=torch.bfloat16, device=at.device)
    check(load().vtk_linear_tn_bf16(ptr(at), at.stride(0), ptr(bt), bt.stride(0), ptr(out), out.stride(0), M, N, K, stream_ptr()))
    return out


@_on_device
def linear_nn(a: torch.Tensor, bt: torch.Tensor) -> torch.Tensor:
    """out [M, N] = a @ bt for a [M, K], bt [K, N] (row-major, any row pitch): B is read MN-major, no transposed copy."""
    _req(a, torch.bfloat16, "a"); _req(bt, torch.bfloat16, "bt")
    M, K = a.shape
    N = bt.shape[1]
    out = torch.empty(M, N, dtype=torch.bfloat16, device=a.device)
    check(load().vtk_linear_nn_acc_bf16(ptr(a), a.stride(0), ptr(bt), bt.stride(0), ptr(out), out.stride(0), M, N, K, 0, stream_ptr()))
    return out


@_on_device
def linear_ln(a: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, eps: float = 1e-6) -> torch.Tensor:
    _req(a, torch.bfloat16, "a"); _req(w, torch.bfloat16, "w"); _req(bias, torch.bfloat16, "bias")
    M, K = a.shape
    N = w.shape[0]
    out = torch.empty(M, N, dtype=torch.bfloat16, device=a.device)
    check(load().vtk_linear_ln_bf16(ptr(a), a.stride(0), ptr(w), w.stride(0), ptr(bias), ptr(out), out.stride(0), M, N, K,
                                    eps, stream_ptr()))
    return out


@_on_device
def rmsnorm(x: torch.Tensor, w: torch.Tensor, eps: float = 1e-6) -> torch.Tensor:
    _req(x, torch.bfloat16, "x"); _req(w, torch.bfloat16, "w")
    M, D = x.shape
    y = torch.empty_like(x)
    check(load().vtk_rmsnorm_bf16(ptr(x), x.stride(0), ptr(w), ptr(y), y.stride(0), M, D, eps, stream_ptr()))
    return y


@_on_device
def rope_table(row_idx: torch.Tensor, col_idx: torch.Tensor, inv_freq: torch.Tensor, head_dim: int) -> torch.Tensor:
    _req(row_idx, torch.int64, "row_idx"); _req(col_idx, torch.int64, "col_idx"); _req(inv_freq, torch.float32, "inv_freq")
    M = row_idx.numel()
    # pair-expanded, chunk-major layout (csrc/vtk_elementwise.cu: rope_table_kernel); decode with rope_table_decode
    table = torch.zeros((M + 31) // 32 * 32, 2 * head_dim, dtype=torch.bfloat16, device=row_idx.device)
    check(load().vtk_rope_table(ptr(row_idx.contiguous()), ptr(col_idx.contiguous()), ptr(inv_freq), ptr(table), M,
                                head_dim, stream_ptr()))
    return table


def rope_table_decode(table: torch.Tensor, M: int, head_dim: int):
    """Undo the kernel layout: returns (C2 [M, d], S2 [M, d]) with C2 = (c0,c0,c1,c1,..), S2 = (-s0,+s0,-s1,+s1,..)."""
    d = head_dim
    g = table.shape[0] // 32
    t = table.reshape(g, 2 * d // 8, 32, 8).permute(0, 2, 1, 3).reshape(g * 32, 2 * d)[:M]
    return t[:, :d], t[:, d:]


@_on_device
def cast_to_bf16(x: torch.Tensor) -> torch.Tensor:
    _req(x, torch.float32, "x")
    x = x.contiguous()
    out = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    check(load().vtk_cast_f32_to_bf16(ptr(x), ptr(out), x.numel(), stream_ptr()))
    return out


@_on_device
def kv_len(mask: torch.Tensor) -> torch.Tensor:
    """[B] int32: 1 + index of the last valid token of each image (the key length of a prefix mask)."""
    B, N = mask.shape
    m = mask.contiguous().view(torch.uint8) if mask.dtype == torch.bool else mask.contiguous()
    kl = torch.empty(B, dtype=torch.int32, device=mask.device)
    check(load().vtk_kv_len(ptr(m), ptr(kl), B, N, stream_ptr()))
    return kl


@_on_device
def pack_plan(mask: torch.Tensor, pad: int = 16, qrows: int = 128):
    """NaFlex token-packing plan of a [B, N] bool mask (include/vitok_b200.h: vtk_pack_plan).  Arrays the kernel leaves
    unwritten (beyond the packed row / group counts) are pre-filled with -2."""
    B, N = mask.shape
    m = mask.contiguous().view(torch.uint8) if mask.dtype == torch.bool else mask.contiguous()
    cap = B * ((N + pad - 1) // pad * pad)
    gcap = B * ((N + qrows - 1) // qrows)
    i32 = dict(dtype=torch.int32, device=mask.device)
    n_valid, rel, cu, cuq = torch.empty(B, **i32), torch.empty(B * N, **i32), torch.empty(B + 1, **i32), torch.empty(B + 1, **i32)
    grp_img, grp_order, src = torch.full((gcap,), -2, **i32), torch.full((gcap,), -2, **i32), torch.full((cap,), -2, **i32)
    check(load().vtk_pack_plan(ptr(m), B, N, pad, qrows, ptr(n_valid), ptr(rel), ptr(cu), ptr(cuq), ptr(grp_img), ptr(grp_order),
                               ptr(src), stream_ptr()))
    return {"n_valid": n_valid, "rel": rel, "cu": cu, "cuq": cuq, "grp_img": grp_img, "grp_order": grp_order, "src": src}


@_on_device
def pack_rows(x: torch.Tensor, plan: dict) -> torch.Tensor:
    """x [B, N, W] bf16 -> packed [row capacity of the plan, W] (rows beyond cu[B] are left as allocated: zeros here)."""
    _req(x, torch.bfloat16, "x")
    B, N, W = x.shape
    x = x.contiguous()
    cap = plan["src"].numel()
    out = torch.zeros(cap, W, dtype=torch.bfloat16, device=x.device)
    check(load().vtk_pack_rows(ptr(x), W, ptr(plan["src"]), ptr(plan["cu"]), B, cap, ptr(out), W, W, stream_ptr()))
    return out


@_on_device
def unpack_rows(packed: torch.Tensor, plan: dict, B: int, N: int) -> torch.Tensor:
    _req(packed, torch.bfloat16, "packed")
    W = packed.shape[1]
    out = torch.empty(B, N, W, dtype=torch.bfloat16, device=packed.device)
    check(load().vtk_unpack_rows(ptr(packed), packed.stride(0), ptr(plan["rel"]), ptr(plan["cu"]), B, N, ptr(out), W, W, stream_ptr()))
    return out


@_on_device
def quant_rows_e4m3(x: torch.Tensor):
    """Dynamic per-row FP8 quantisation: returns (q [M, K] float8_e4m3fn, scale [M] fp32) with x ~= q * scale[:, None]."""
    _req(x, torch.bfloat16, "x")
    M, K = x.shape
    q = torch.empty(M, K, dtype=torch.uint8, device=x.device)
    scale = torch.empty(M, dtype=torch.float32, device=x.device)
    check(load().vtk_quant_rows_e4m3(ptr(x), x.stride(0), ptr(q), q.stride(0), ptr(scale), M, K, stream_ptr()))
    return q.view(torch.float8_e4m3fn), scale


@_on_device
@_on_device
def quant_tensor_e4m3(x: torch.Tensor):
    """Dynamic per-TENSOR FP8 quantisation (torchao's default granularity): returns (q [M, K] float8_e4m3fn, scale [M] fp32, all equal)."""
    _req(x, torch.bfloat16, "x")
    M, K = x.shape
    q = torch.empty(M, K, dtype=torch.uint8, device=x.device)
    scale = torch.empty(M, dtype=torch.float32, device=x.device)
    ws = torch.zeros(1, dtype=torch.float32, device=x.device)
    check(load().vtk_quant_tensor_e4m3(ptr(x), x.stride(0), ptr(q), q.stride(0), ptr(scale), ptr(ws), M, K, stream_ptr()))
    return q.view(torch.float8_e4m3fn), scale


def proj_residual_fp8(a8, a_scale, w8, w_scale: float, gamma, x):
    """x += gamma * (a_scale[:, None] * w_scale * (a8 @ w8^T)) with e4m3 operands (tcgen05 kind::f8f6f4)."""
    M, K = a8.shape
    N = w8.shape[0]
    check(load().vtk_proj_residual_fp8(ptr(a8), a8.stride(0), ptr(a_scale), ptr(w8), w8.stride(0), float(w_scale), ptr(gamma),
                                       ptr(x), x.stride(0), M, N, K, stream_ptr()))
    return x


@_on_device
def qkv_swiglu(h, w_packed, D, d, Hf, qp, norm_q, norm_k, table, eps=1e-6):
    """QKV + fc1 GEMM with QK-norm, RoPE and SwiGLU (vtk_qkv_swiglu_bf16); d % 8 == 0, 8 <= d <= 128.  At d other than 32, 64 and
    128 the QK-norm + RoPE run as a second kernel after the GEMM."""
    M = h.shape[0]
    qkv = torch.empty(M, 3 * D, dtype=torch.bfloat16, device=h.device)
    act = torch.empty(M, Hf, dtype=torch.bfloat16, device=h.device)
    check(load().vtk_qkv_swiglu_bf16(ptr(h), h.stride(0), ptr(w_packed), w_packed.stride(0), w_packed.shape[0], M, D, d,
                                     Hf, qp, ptr(norm_q), ptr(norm_k), ptr(table), eps, ptr(qkv), qkv.stride(0),
                                     ptr(act), act.stride(0), stream_ptr()))
    return qkv, act


@_on_device
def proj_residual(a, w, gamma, x):
    M, K = a.shape
    N = w.shape[0]
    check(load().vtk_proj_residual_bf16(ptr(a), a.stride(0), ptr(w), w.stride(0), ptr(gamma), ptr(x), x.stride(0), M, N, K,
                                        stream_ptr()))
    return x


@_on_device
def attention(qkv: torch.Tensor, B: int, N: int, heads: int, d: int, mask: Optional[torch.Tensor] = None,
              window: int = -1, lse: Optional[torch.Tensor] = None) -> torch.Tensor:
    """qkv [B*N, 3*heads*d] (q | k | v).  mask [B,N] bool -> sdpa semantics (masked query rows read 0); None -> flash semantics.
    The mask must be a prefix mask (every image's valid tokens first, what patchify emits): a mask with holes raises ValueError
    (a host check; masked batches with holes run on the packed layout, see ``attention_packed``).
    window >= 0: sliding window |i - j| <= window (flash_attn window_size=(window, window)).
    head_dim d: d % 8 == 0 and 8 <= d <= 128 (NotImplementedError otherwise)."""
    D = heads * d
    out = torch.empty(B * N, D, dtype=torch.bfloat16, device=qkv.device)
    kl = None
    if mask is not None:
        m = mask.bool()
        if not bool((m == (torch.arange(N, device=m.device) < m.sum(dim=1, keepdim=True))).all()):
            raise ValueError("vitok_b200.attention: the mask must be a prefix mask (valid tokens first in every image)")
        kl = kv_len(mask)
    base = qkv.data_ptr()
    check(load().vtk_attention_bf16(base, base + 2 * D, base + 4 * D, qkv.stride(0), ptr(out), out.stride(0), ptr(kl),
                                    B, N, heads, d, 1 if mask is not None else 0, int(window), ptr(lse), stream_ptr()))
    return out


@_on_device
def umma_probe(a: torch.Tensor, b: torch.Tensor, n: int, k: int, b_mn_major: bool, lbo: int, sbo: int, kstep: int):
    d = torch.zeros(128, n, dtype=torch.float32, device=a.device)
    check(load().vtk_umma_probe(ptr(a), ptr(b), ptr(d), n, k, 1 if b_mn_major else 0, lbo, sbo, kstep, stream_ptr()))
    return d


@_on_device
def attention_packed(qkv: torch.Tensor, plan: dict, B: int, N: int, heads: int, d: int, lse: Optional[torch.Tensor] = None,
                     out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Attention over the packed NaFlex layout of ``pack_plan`` (qkv [row capacity, 3*heads*d]; the plan's qrows must be 128 for
    d <= 64, 256 for 64 < d <= 128).  Without ``lse`` the pad rows of ``out`` are never written; with ``lse`` ([rows, heads] fp32) they
    are written as 0 and lse as +inf.  ``out`` (optional) = a preallocated [rows, heads*d]."""
    D = heads * d
    if out is None:
        out = torch.empty(qkv.shape[0], D, dtype=torch.bfloat16, device=qkv.device)
    base = qkv.data_ptr()
    check(load().vtk_attention_packed_lse_bf16(base, base + 2 * D, base + 4 * D, qkv.stride(0), ptr(out), out.stride(0),
                                               ptr(plan["n_valid"]), ptr(plan["cu"]), ptr(plan["cuq"]), ptr(plan["grp_img"]),
                                               ptr(plan["grp_order"]), B, N, heads, d, qkv.shape[0], plan["grp_img"].numel(), ptr(lse),
                                               stream_ptr()))
    return out
