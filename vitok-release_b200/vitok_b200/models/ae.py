"""B200-native drop-in for ``vitok.models.ae`` (reference: /root/reference/vitok/models/ae.py).

Same public surface -- ``AE(**decode_variant(v))``, ``.encode(d)['z']``, ``.decode(d)['patches']``,
``.forward``, ``.quantize``, identical parameter names/shapes so ``load_state_dict`` of reference or
Hub weights works -- but no tensor math happens in PyTorch: ``encode``/``decode`` each make ONE call
into libvitok_b200.so (``vtk_ae_encode`` / ``vtk_ae_decode``), which runs the whole layer stack as
hand-written sm_100a kernels on the current CUDA stream.  The nn.Module tree below only *holds*
parameters.  There is no CPU / eager fallback.

Semantics kept from the reference (file:line in the reference tree):
  * dict contract: pass-through of patch_mask/row_idx/col_idx/orig_height/orig_width as the same
    tensor objects, 'patches' dropped by encode, 'z' dropped by decode (ae.py:209-216, 236-243);
  * ``attn_backend="flash"``: attention over all N tokens, patch_mask ignored (attention.py:109-117);
    ``attn_backend="sdpa"``: keys masked by patch_mask (ae.py:173-187, attention.py:118-127).  Both
    run on the same tcgen05 attention kernel; padded keys are skipped, not masked after the fact;
  * unknown kwargs ignored (ae.py:92); ``sw <= 0`` -> None (ae.py:99).
``sw``: sliding-window attention |i-j| <= sw on the token index with the flash backend (attention.py:113-116);
    ignored by the sdpa backend, as in the reference.
Training: ``model(batch)`` in train mode builds one autograd node (vitok_b200/train.py) that computes only the gradients
    autograd asks for: frozen parameters (``requires_grad=False``) cost no weight-gradient GEMM and get no ``.grad``, and the
    backward pass stops below the lowest block that needs one.  ``AE(encoder=False)`` trains on ``batch["z"]``, ``AE(decoder=False)``
    returns the encode dict with z carrying the graph.  encode/decode alone are inference-only.  ``quantize()`` (FP8 block GEMMs) needs widths that are multiples of 256 and raises otherwise.
"""
from __future__ import annotations

import ctypes
import itertools
import re
import weakref
from typing import Any, Dict, List, Optional

import torch
import torch.nn as nn

from .. import _lib

__all__ = ["AE", "Model", "decode_variant", "pack_w_in", "pack_w_out"]

# --------------------------------------------------------------------------------------
# variant strings:  "{enc}-{dec}/{T}x{S}x{C}"                      (ae.py:280-346)
# --------------------------------------------------------------------------------------
_PRESETS = {  # letter: (width, depth, heads)
    "B": (768, 12, 12), "L": (1024, 24, 16), "G": (1728, 32, 24), "T": (3072, 40, 24), "E": (4096, 48, 32),
}
_DEFAULT_MLP = 2.67
_MOD = {"w": r"w(\d+)", "d": r"d(\d+)", "h": r"h(\d+)", "m": r"m(\d+(?:\.\d+)?)"}


def _side_config(name: str) -> Dict[str, Any]:
    """One side of a variant: preset letter with inline w/d/h/m overrides, or ``w{W}_d{D}_h{H}[_m{M}]``."""
    if name.startswith("w") and "_d" in name and "_h" in name:
        f = name.split("_")
        mlp = float(f[3][1:]) if len(f) > 3 and f[3].startswith("m") else _DEFAULT_MLP
        return {"width": int(f[0][1:]), "depth": int(f[1][1:]), "heads": int(f[2][1:]), "mlp_factor": mlp}
    found = {k: re.search(rx, name) for k, rx in _MOD.items()}
    base = re.sub("|".join(_MOD[k] for k in ("w", "d", "h", "m")), "", name)
    if base and base not in _PRESETS:
        raise ValueError(f"Unknown base variant: {base}. Available: {list(_PRESETS.keys())}")
    pw, pd, ph = _PRESETS.get(base, (768, 12, 12))
    return {
        "width": int(found["w"].group(1)) if found["w"] else pw,
        "depth": int(found["d"].group(1)) if found["d"] else pd,
        "heads": int(found["h"].group(1)) if found["h"] else ph,
        "mlp_factor": float(found["m"].group(1)) if found["m"] else _DEFAULT_MLP,
    }


def decode_variant(variant: str) -> Dict[str, Any]:
    """Variant string -> AE kwargs; same keys/values as the reference's ``decode_variant`` (ae.py:318-346)."""
    arch, geom = variant.split("/")
    enc_name, dec_name = arch.split("-") if "-" in arch else (arch, arch)
    dims = [int(t) for t in geom.split("x")]
    if len(dims) == 2:
        dims = [1] + dims
    if len(dims) != 3:
        raise ValueError(f"Invalid variant format: {variant}")
    t_stride, s_stride, channels = dims
    enc, dec = _side_config(enc_name), _side_config(dec_name)
    return {
        "encoder_width": enc["width"], "decoder_width": dec["width"],
        "encoder_depth": enc["depth"], "decoder_depth": dec["depth"],
        "encoder_heads": enc["heads"], "decoder_heads": dec["heads"],
        "mlp_factor": max(enc["mlp_factor"], dec["mlp_factor"]),
        "temporal_stride": t_stride, "spatial_stride": s_stride, "channels_per_token": channels,
        "pixels_per_token": 3 * s_stride * s_stride * t_stride,
    }


def _ffn_hidden(width: int, mlp_factor: float) -> int:
    """SwiGLU hidden size: int(width*mlp_factor) (ae.py:128) rounded to a multiple of 16 (mlp.py:14)."""
    return ((int(width * mlp_factor) + 8) // 16) * 16


def pack_w_in(qkv_w: torch.Tensor, fc1_w: torch.Tensor) -> torch.Tensor:
    """[Wq; Wk; Wv; zeros up to qp = roundup(3D, 256); fc1 value/gate halves interleaved in 16-row groups].

    The interleave puts value column j and gate column j in the same 32-column accumulator chunk so the
    GEMM epilogue can apply silu(g)*v without leaving registers.
    """
    three_d, width = qkv_w.shape
    hf = fc1_w.shape[0] // 2
    qp = ((three_d + 255) // 256) * 256
    w_in = torch.zeros(qp + 2 * hf, width, dtype=qkv_w.dtype, device=qkv_w.device)
    w_in[:three_d] = qkv_w
    w_in[qp:] = fc1_w.view(2, hf // 16, 16, width).permute(1, 0, 2, 3).reshape(2 * hf, width)
    return w_in


def _quantize_e4m3(w: torch.Tensor):
    """Per-tensor e4m3 quantisation of a packed weight matrix: returns (uint8 view of the e4m3 bytes, scale) with w ~= w8 * scale."""
    wf = w.float()
    amax = float(wf.abs().max())
    scale = amax / 448.0 if amax > 0 else 1.0
    return (wf / scale).to(torch.float8_e4m3fn).view(torch.uint8).contiguous(), scale


def pack_w_out(out_w: torch.Tensor, fc2_w: torch.Tensor) -> torch.Tensor:
    """[out_proj | fc2 | 0-pad] along K: attn_out + mlp_out becomes one GEMM over the concatenated activations.

    The row pitch is rounded up to 64 elements (128 bytes) so that every row of the TMA boxes starts on a
    128-byte line; the pad columns are zero and lie beyond K, so they are never multiplied.
    """
    k = out_w.shape[1] + fc2_w.shape[1]
    kp = (k + 63) // 64 * 64
    w = torch.zeros(out_w.shape[0], kp, dtype=out_w.dtype, device=out_w.device)
    w[:, :out_w.shape[1]] = out_w
    w[:, out_w.shape[1]:k] = fc2_w
    return w


# --------------------------------------------------------------------------------------
# parameter holders (names = the reference's state_dict keys; no forward math here)
# --------------------------------------------------------------------------------------
class _NoTorchPath(nn.Module):
    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("vitok_b200 modules hold parameters only; the math runs in libvitok_b200.so "
                           "via AE.encode / AE.decode (there is no PyTorch fallback)")


class _Scale(_NoTorchPath):
    def __init__(self, dim: int, init: float, name: str):
        super().__init__()
        self.register_parameter(name, nn.Parameter(torch.full((dim,), float(init))))


class _Attn(_NoTorchPath):
    def __init__(self, dim: int, heads: int):
        super().__init__()
        self.dim, self.num_heads, self.head_dim = dim, heads, dim // heads
        self.norm_q = _Scale(self.head_dim, 1.0, "weight")
        self.norm_k = _Scale(self.head_dim, 1.0, "weight")
        self.qkv_proj = nn.Linear(dim, 3 * dim, bias=False)
        self.out_proj = nn.Linear(dim, dim, bias=False)


class _Ffn(_NoTorchPath):
    def __init__(self, dim: int, hidden: int):
        super().__init__()
        self.fc1 = nn.Linear(dim, 2 * hidden, bias=False)
        self.fc2 = nn.Linear(hidden, dim, bias=False)


class Block(_NoTorchPath):
    """Parallel attention + SwiGLU block with LayerScale (reference Block, ae.py:33-65) -- parameters only."""

    def __init__(self, dim: int, ffn_dim: int, num_heads: int, use_layer_scale: bool = True,
                 layer_scale_init: float = 1e-6, drop_path: float = 0.0, sliding_window: Optional[int] = None,
                 attn_backend: str = "flash"):
        super().__init__()
        self.sliding_window = sliding_window
        self.drop_path_rate = drop_path
        self.norm1 = _Scale(dim, 1.0, "weight")
        self.attn = _Attn(dim, num_heads)
        self.ffn = _Ffn(dim, ((ffn_dim + 8) // 16) * 16)
        self.layer_scale = _Scale(dim, layer_scale_init, "gamma") if use_layer_scale else nn.Identity()


class _OutputNorm(_NoTorchPath):
    """LayerNorm without affine parameters (no state_dict entries), fused into the to_code GEMM epilogue."""


# ----------------------------------------------------------------------------------------------------------------
# vitok_b200::ae_run -- the one opaque torch op behind AE.encode / AE.decode.  It exists so that TorchDynamo can trace
# encode / decode (torch.compile(model.encode, fullgraph=True), reference README.md:57-58): the graph holds a single
# call to this op, whose eager body does the C-ABI call.  Models are looked up by id (weak references).
# ----------------------------------------------------------------------------------------------------------------
_MODELS: "weakref.WeakValueDictionary[int, AE]" = weakref.WeakValueDictionary()
_MODEL_IDS = itertools.count(1)


@torch.library.custom_op("vitok_b200::ae_run", mutates_args=())
def _ae_run(model_id: int, side: int, x: torch.Tensor, row: torch.Tensor, col: torch.Tensor,
            mask: Optional[torch.Tensor]) -> torch.Tensor:
    return _MODELS[model_id]._run_native(side, x, row, col, mask)


@_ae_run.register_fake
def _ae_run_fake(model_id, side, x, row, col, mask):
    m = _MODELS[model_id]
    return x.new_empty((x.shape[0], x.shape[1], m.channels_per_token if side == 0 else m.pixels_per_token), dtype=m._out_dtype())


class AE(nn.Module):
    """ViTok-v2 autoencoder; see module docstring."""

    def __init__(self, pixels_per_token=768, channels_per_token=32, encoder_width=1024, decoder_width=1024,
                 encoder_depth=4, decoder_depth=24, encoder_heads=12, decoder_heads=12, mlp_factor=2.67,
                 checkpoint: int = 0, spatial_stride: int = 16, temporal_stride: int = 1, use_layer_scale: bool = True,
                 layer_scale_init: float = 1e-4, drop_path_rate: float = 0.0, encoder: bool = True, decoder: bool = True,
                 sw: Optional[int] = None, attn_backend: str = "flash", **kwargs):
        super().__init__()
        if not encoder and not decoder:
            raise ValueError("At least one of encoder or decoder must be True")
        if attn_backend not in ("flash", "sdpa"):
            raise ValueError(f"attn_backend must be 'flash' or 'sdpa', got {attn_backend!r}")
        sw = sw if (sw is None or sw > 0) else None
        self.pixels_per_token, self.channels_per_token = pixels_per_token, channels_per_token
        self.rope_theta = 10000.0
        self.encoder_depth, self.decoder_depth = encoder_depth, decoder_depth
        self.encoder_width, self.decoder_width = encoder_width, decoder_width
        self.encoder_heads, self.decoder_heads = encoder_heads, decoder_heads
        self.mlp_factor = mlp_factor
        self.checkpoint = checkpoint
        self.spatial_stride = spatial_stride
        self.temporal_stride = temporal_stride
        self.is_encoder, self.is_decoder = encoder, decoder
        self.sw = sw
        self.attn_backend = attn_backend
        self._quantization_applied = False

        def stack(width, depth, heads, rates):
            return nn.ModuleList([
                Block(width, int(width * mlp_factor), heads, use_layer_scale, layer_scale_init, rates[i], sw, attn_backend)
                for i in range(depth)])

        if encoder:
            self.patch_embed = nn.Linear(pixels_per_token, encoder_width)
            self.to_code = nn.Linear(encoder_width, channels_per_token)
            self.output_fn = _OutputNorm()
            self.encoder_blocks = stack(encoder_width, encoder_depth, encoder_heads, [0.0] * encoder_depth)
        if decoder:
            self.decoder_embed = nn.Linear(channels_per_token, decoder_width)
            self.to_pixels = nn.Linear(decoder_width, pixels_per_token)
            rates = [drop_path_rate * i / max(decoder_depth - 1, 1) for i in range(decoder_depth)]
            self.decoder_blocks = stack(decoder_width, decoder_depth, decoder_heads, rates)

        # native state (not part of the state_dict)
        self._handle: Optional[int] = None
        self._packed: Dict[int, List[torch.Tensor]] = {}
        self._packed_sig = None
        self._ws: Dict[Any, torch.Tensor] = {}
        self._plist: Optional[List[torch.Tensor]] = None
        self.last_launch_count = 0
        self._model_id = next(_MODEL_IDS)       # key of this instance for the vitok_b200::ae_run op
        _MODELS[self._model_id] = self
        # Masked (sdpa-backend) inference batches always run on their packed valid tokens (include/vitok_b200.h: vtk_ae_encode).
        # The same for the training step (train mode, sdpa backend with a patch_mask; vitok_b200/train.py: _Packing): GEMMs, kernels
        # and saved activations cover the valid tokens only.  Off by default: the result differs from the padded step in the order of
        # the weight-gradient sums, and masked tokens of the output are 0.  No effect without a mask or under the flash backend.
        self.train_token_packing = False
        # Block.norm1 fused into the GEMM epilogues (widths that are multiples of 256): no RMSNorm kernel, no h buffer
        # round trip.  False keeps the separate RMSNorm kernel (rounds h to bf16 exactly where the reference does).
        self.fuse_norm = True
        # quantize(): dynamic FP8 activation scale per "row" (default: finer, no extra pass over the activations) or per "tensor"
        # (torchao's default granularity for Float8DynamicActivationFloat8WeightConfig, the reference's numerics)
        self.fp8_activation_scale = "row"
        # True: re-pack the weights on every call (for code that writes parameters through ``.data``; see invalidate_packed)
        self.always_repack = False

    # ------------------------------------------------------------------ native plumbing
    def _sides(self):
        out = []
        if self.is_encoder:
            out.append((0, self.patch_embed, self.to_code, self.encoder_blocks, self.encoder_width, self.encoder_heads))
        if self.is_decoder:
            out.append((1, self.decoder_embed, self.to_pixels, self.decoder_blocks, self.decoder_width, self.decoder_heads))
        return out

    def _signature(self):
        # (device, storage pointers, versions) of every parameter: changes on .to(), load_state_dict, optimizer steps.
        # The module-tree walk is cached (it costs more than the check itself); anything that can replace a Parameter
        # object goes through _apply / load_state_dict / train(), which drop the cache.
        ps = self._plist
        if ps is None:
            ps = self._plist = list(self.parameters())
        return (ps[0].device, tuple(p.data_ptr() for p in ps), tuple(p._version for p in ps))

    def _apply(self, fn, *args, **kwargs):
        self._plist = None
        return super()._apply(fn, *args, **kwargs)

    def load_state_dict(self, *args, **kwargs):
        self._plist = None
        return super().load_state_dict(*args, **kwargs)

    def train(self, mode: bool = True):
        self._plist = None
        return super().train(mode)

    def __del__(self):
        try:
            if self._handle:
                _lib.load().vtk_ae_destroy(self._handle)
        except Exception:  # noqa: BLE001  (interpreter shutdown)
            pass

    def invalidate_packed(self) -> "AE":
        """Drop the packed / folded / FP8 weight copies so that the next encode / decode rebuilds them from the parameters.
        The copies are re-built automatically when a parameter's storage or ``_version`` changes (``load_state_dict``,
        ``.to()``, in-place ops, optimizer steps); writes that bypass the version counter -- ``p.data.copy_(ema)``,
        ``torch._foreach_*`` on ``.data``, custom optimizers -- must call this (or set ``model.always_repack = True``)."""
        self._packed_sig = None
        self._plist = None
        return self

    refresh_weights = invalidate_packed

    @torch.no_grad()
    def _ensure_packed(self, device: torch.device, fold_norm: bool = True) -> int:
        """(Re)build the packed bf16 weights the kernels read and hand their pointers to the C handle.

        w_in  [qp + 2*Hf, D] = [Wq; Wk; Wv; zeros up to qp; 16-row interleave of fc1's value/gate halves]
        w_out [D, Kp]        = [out_proj | fc2 | 0-pad to a multiple of 64]   (one GEMM over the concatenated K)
        Rebuilt whenever a parameter's storage or version changes (load_state_dict, .to(), optimizer step).
        """
        sig = (self._signature(), bool(fold_norm and self.fuse_norm), bool(self._quantization_applied and fold_norm))
        if self._handle is not None and sig == self._packed_sig and not self.always_repack:
            return self._handle
        fold = sig[1]
        fp8 = sig[2]
        sig0 = sig
        sig = sig[0]
        lib = _lib.load()
        if sig[0].type != "cuda":
            raise RuntimeError("vitok_b200.AE: parameters must be on a CUDA device (model.to('cuda')); there is no CPU path")
        if self._handle is None:
            cfg = _lib.AEConfig()
            cfg.pixels_per_token, cfg.channels_per_token = self.pixels_per_token, self.channels_per_token
            if self.is_encoder:
                cfg.enc_width, cfg.enc_depth, cfg.enc_heads = self.encoder_width, self.encoder_depth, self.encoder_heads
                cfg.enc_hidden = _ffn_hidden(self.encoder_width, self.mlp_factor)
            if self.is_decoder:
                cfg.dec_width, cfg.dec_depth, cfg.dec_heads = self.decoder_width, self.decoder_depth, self.decoder_heads
                cfg.dec_hidden = _ffn_hidden(self.decoder_width, self.mlp_factor)
            cfg.norm_eps = 1e-6
            cfg.sliding_window = int(self.sw) if self.sw else 0
            h = ctypes.c_void_p()
            _lib.check(lib.vtk_ae_create(ctypes.byref(cfg), ctypes.byref(h)))
            self._handle = h.value
        bf = torch.bfloat16

        def dev(t):
            return t.detach().to(device=device, dtype=bf).contiguous()

        for side, lin_a, lin_b, blocks, width, heads in self._sides():
            keep: List[torch.Tensor] = []
            Hf = _ffn_hidden(width, self.mlp_factor)
            qp = ((3 * width + 255) // 256) * 256
            arr = (_lib.BlockWeights * max(len(blocks), 1))()
            arr8 = (_lib.BlockFp8 * max(len(blocks), 1))()
            for i, blk in enumerate(blocks):
                if fold and width % 256 == 0:
                    # norm1 folded into the GEMM: h W^T = rstd * (x (W * w)^T)  (include/vitok_b200.h: vtk_ae_set_norm_folded)
                    n1 = blk.norm1.weight.detach().to(device=device, dtype=torch.float32)[None, :]
                    w_in = pack_w_in((blk.attn.qkv_proj.weight.detach().to(device=device, dtype=torch.float32) * n1).to(bf),
                                     (blk.ffn.fc1.weight.detach().to(device=device, dtype=torch.float32) * n1).to(bf))
                else:
                    w_in = pack_w_in(dev(blk.attn.qkv_proj.weight), dev(blk.ffn.fc1.weight))
                w_out = pack_w_out(dev(blk.attn.out_proj.weight), dev(blk.ffn.fc2.weight))
                gamma = dev(blk.layer_scale.gamma) if isinstance(blk.layer_scale, _Scale) else torch.ones(width, dtype=bf, device=device)
                tens = [w_in, w_out, dev(blk.norm1.weight), dev(blk.attn.norm_q.weight), dev(blk.attn.norm_k.weight), gamma]
                keep.extend(tens)
                (arr[i].w_in, arr[i].w_out, arr[i].norm1, arr[i].norm_q, arr[i].norm_k, arr[i].gamma) = [t.data_ptr() for t in tens]
                if fp8:      # e4m3 copies of the packed matrices, one scale each (w ~= w8 * scale)
                    q_in, s_in = _quantize_e4m3(w_in)
                    q_out, s_out = _quantize_e4m3(w_out)
                    keep.extend([q_in, q_out])
                    arr8[i].w_in8, arr8[i].w_out8, arr8[i].w_in_scale, arr8[i].w_out_scale = q_in.data_ptr(), q_out.data_ptr(), s_in, s_out
            proj = [dev(lin_a.weight), dev(lin_a.bias), dev(lin_b.weight), dev(lin_b.bias)]
            keep.extend(proj)
            axis = (width // heads) // 2
            inv = (1.0 / (self.rope_theta ** (torch.arange(0, axis, 2).float() / axis))).contiguous()
            inv_c = (ctypes.c_float * inv.numel())(*inv.tolist())
            _lib.check(lib.vtk_ae_set_weights(self._handle, side, *[t.data_ptr() for t in proj], arr, len(blocks), inv_c,
                                              inv.numel()))
            _lib.check(lib.vtk_ae_set_norm_folded(self._handle, side, 1 if (fold and width % 256 == 0 and len(blocks) > 0) else 0))
            _lib.check(lib.vtk_ae_set_fp8_weights(self._handle, side, arr8, len(blocks) if (fp8 and len(blocks) > 0) else 0))
            self._packed[side] = keep
        self._packed_sig = sig0
        return self._handle

    def _workspace(self, side: int, B: int, N: int, device) -> torch.Tensor:
        key = (side, B, N, device, self._quantization_applied)
        ws = self._ws.get(key)
        if ws is None:
            nbytes = _lib.load().vtk_ae_workspace_bytes(self._handle, side, B, N)
            ws = torch.zeros(nbytes + 1024, dtype=torch.uint8, device=device)
            self._ws = {k: v for k, v in self._ws.items() if k[0] != side}  # one live workspace per side
            self._ws[key] = ws
        return ws

    def _run(self, side: int, x: torch.Tensor, d: Dict[str, torch.Tensor], out_cols: int) -> torch.Tensor:
        """Argument checks (traceable by TorchDynamo) + ONE opaque op, ``vitok_b200::ae_run``, that makes the C call.
        The op is what lets ``torch.compile(model.encode, fullgraph=True)`` (reference README.md:57-58) capture encode /
        decode as a single graph node instead of failing on the ctypes call."""
        if self._wants_grad():
            raise NotImplementedError("vitok_b200.AE: gradients flow through model(batch) (AE.forward) only; call encode/decode "
                                      "under model.eval() or torch.no_grad()")
        if not x.is_cuda:
            raise RuntimeError("vitok_b200.AE: inputs must be CUDA tensors (there is no CPU path)")
        if x.dim() != 3:
            raise ValueError(f"expected a [B, N, C] tensor, got shape {tuple(x.shape)}")
        B, N, cin = x.shape
        want = (self.pixels_per_token if side == 0 else self.channels_per_token)
        if cin != want:
            raise RuntimeError(f"shape mismatch: last dim {cin} != {want}")
        if x.dtype not in (torch.float32, torch.bfloat16):
            raise RuntimeError(f"vitok_b200.AE: unsupported input dtype {x.dtype} (float32 or bfloat16)")
        row, col = d["row_idx"], d["col_idx"]
        if row.shape != (B, N) or col.shape != (B, N):
            raise ValueError("x_positions and y_positions must have matching shapes [B, N]")
        mask = d.get("patch_mask") if self.attn_backend == "sdpa" else None
        return torch.ops.vitok_b200.ae_run(self._model_id, side, x, row, col, mask)

    def _out_dtype(self) -> torch.dtype:
        pdtype = next(self.parameters()).dtype
        return torch.float32 if (pdtype == torch.float32 and not torch.is_autocast_enabled()) else torch.bfloat16

    def _run_native(self, side: int, x: torch.Tensor, row: torch.Tensor, col: torch.Tensor,
                    mask: Optional[torch.Tensor]) -> torch.Tensor:
        """The body of ``vitok_b200::ae_run``: weight packing check, workspace, and the vtk_ae_encode / vtk_ae_decode call."""
        pdev = next(self.parameters()).device
        if pdev != x.device:
            raise RuntimeError(f"vitok_b200.AE: the model is on {pdev} but the input is on {x.device}")
        with torch.cuda.device(x.device):     # kernels, tensor maps and stream_ptr() follow the CURRENT device
            return self._run_on_device(side, x, row, col, mask)

    def _run_on_device(self, side: int, x: torch.Tensor, row: torch.Tensor, col: torch.Tensor,
                       mask: Optional[torch.Tensor]) -> torch.Tensor:
        B, N, _ = x.shape
        out_cols = self.channels_per_token if side == 0 else self.pixels_per_token
        h = self._ensure_packed(x.device)
        lib = _lib.load()
        xin = _lib.cast_to_bf16(x) if x.dtype == torch.float32 else x.contiguous()
        row = row.to(device=x.device, dtype=torch.int64).contiguous()
        col = col.to(device=x.device, dtype=torch.int64).contiguous()
        m8 = None
        if mask is not None:
            m8 = mask.to(device=x.device).bool().contiguous().view(torch.uint8)
        ws = self._workspace(side, B, N, x.device)
        ws_ptr = (ws.data_ptr() + 1023) // 1024 * 1024
        out = torch.empty(B, N, out_cols, dtype=torch.bfloat16, device=x.device)
        fn = lib.vtk_ae_encode if side == 0 else lib.vtk_ae_decode
        _lib.check(lib.vtk_ae_set_fp8_granularity(h, 1 if self.fp8_activation_scale == "tensor" else 0))
        _lib.check(fn(h, xin.data_ptr(), row.data_ptr(), col.data_ptr(), m8.data_ptr() if m8 is not None else None,
                      B, N, out.data_ptr(), ws_ptr, ws.numel() - (ws_ptr - ws.data_ptr()), _lib.stream_ptr()))
        self.last_launch_count = lib.vtk_ae_last_launch_count(h)
        if self._out_dtype() == torch.float32:
            out = out.float()
        return out

    # ------------------------------------------------------------------ public surface
    def encode(self, patch_dict: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        """patches [B,N,P] -> z [B,N,C]  (reference AE.encode, ae.py:189-216)."""
        if not self.is_encoder:
            raise AttributeError("this AE was built with encoder=False")
        z = self._run(0, patch_dict["patches"], patch_dict, self.channels_per_token)
        return {
            "patch_mask": patch_dict.get("patch_mask"), "row_idx": patch_dict["row_idx"], "col_idx": patch_dict["col_idx"],
            "orig_height": patch_dict.get("orig_height"), "orig_width": patch_dict.get("orig_width"), "z": z,
        }

    def decode(self, encode_dict: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        """z [B,N,C] -> patches [B,N,P]  (reference AE.decode, ae.py:218-243)."""
        if not self.is_decoder:
            raise AttributeError("this AE was built with decoder=False")
        patches = self._run(1, encode_dict["z"], encode_dict, self.pixels_per_token)
        return {
            "patch_mask": encode_dict.get("patch_mask"), "row_idx": encode_dict.get("row_idx"),
            "col_idx": encode_dict.get("col_idx"), "orig_height": encode_dict.get("orig_height"),
            "orig_width": encode_dict.get("orig_width"), "patches": patches,
        }

    def _wants_grad(self) -> bool:
        return self.training and torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())

    def forward(self, x: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        """encode then decode (ae.py:245-251); a model with one half runs that half.  In training mode with gradients enabled
        (some parameter requires grad) this is the training step's forward: one autograd node whose backward runs the sm_100a
        backward kernels for exactly the gradients autograd asks for (vitok_b200/train.py).  ``AE(encoder=False)`` decodes
        ``x["z"]`` (z gets a gradient when it requires grad); ``AE(decoder=False)`` returns the encode dict, whose ``z`` carries the
        graph back to the encoder parameters (and to ``x["patches"]`` when they require grad)."""
        if self._wants_grad():
            from ..train import train_forward
            return train_forward(self, x)
        if self.is_encoder:
            x = self.encode(x)
        if self.is_decoder:
            x = self.decode(x)
        return x

    def quantize(self) -> "AE":
        """FP8 inference (reference ae.py:253-270: torchao ``Float8DynamicActivationFloat8WeightConfig`` on every Linear of the
        blocks).  The packed block weights are quantised to e4m3 with one scale per packed matrix, the activations entering the
        two block GEMMs are quantised per row on the fly, and both GEMMs run on the tcgen05 ``kind::f8f6f4`` path; attention, the
        embeds and the latent bottleneck stay bf16, as in the reference.  Idempotent; inference only."""
        if self._quantization_applied:
            return self
        for _, _, _, blocks, width, _ in self._sides():
            if len(blocks) and width % 256:
                raise NotImplementedError(f"vitok_b200.AE.quantize: the FP8 path needs widths that are multiples of 256 (got {width})")
        if not self.fuse_norm:
            raise NotImplementedError("vitok_b200.AE.quantize: the FP8 path runs on the fused-norm GEMMs (fuse_norm must stay True)")
        self._quantization_applied = True
        self._packed_sig = None      # re-pack (and quantise) on the next call
        self._ws = {}                # the workspace grows by the e4m3 activation copies
        return self


def Model(**kw):
    return AE(**kw)
