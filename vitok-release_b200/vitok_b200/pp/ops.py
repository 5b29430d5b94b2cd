"""NaFlex patchify / unpatchify / unpack on the GPU + the host-side op registry.

Hot-path ops (``patchify_batch``, ``patchify``, ``unpatchify``, ``unpack``) call libvitok_b200.so;
results are bit-identical to vitok/pp/ops.py:217-360.  The PIL-level augmentation ops are NOT on
the encode/decode path (SURVEY.md section 8a row A15/A16); they are thin host wrappers over
PIL/torchvision kept only so that reference DSL strings keep working.
"""
from __future__ import annotations

import math
import random
from typing import Callable, Dict, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from .. import _lib

_FMT = {"as_is": 0, "0_255": 1, "zero_to_one": 2}


# --------------------------------------------------------------------------------------
# patchify
# --------------------------------------------------------------------------------------
def _grid(h: int, w: int, patch: int) -> Tuple[int, int]:
    return -(-h // patch), -(-w // patch)


def patchify_batch(images: Union[torch.Tensor, Sequence[torch.Tensor], Sequence[np.ndarray]], patch: int = 16,
                   max_tokens: int = 256, out_dtype: torch.dtype = torch.float32,
                   device: Union[str, torch.device] = "cuda", resize_to_budget: bool = False) -> Dict[str, torch.Tensor]:
    """patchify + collate for a whole (possibly ragged) batch in one kernel launch.

    images: a [B,3,H,W] float32 tensor, or a list of [3,H_i,W_i] float32 tensors (already normalised,
    i.e. the output of ``to_tensor|normalize``), or a list of uint8 HWC arrays/tensors (then
    ``to_tensor|normalize(minus_one_to_one)`` is fused into the kernel).  Returns the batched NaFlex
    dict of vitok/pp/ops.py:274-284 + vitok/data.py:77-94 on ``device``.
    Raises RuntimeError when an image's patch grid exceeds ``max_tokens`` (reference: ops.py:260), unless
    ``resize_to_budget``: then such images are first resized on the device to ``_fit_to_token_budget(h, w, patch,
    max_tokens)`` as ``resize_to_token_budget`` does (ops.py:169-214; antialiased bicubic, within a few fp32 ulps of
    torchvision's, not bit-identical), in the same launch sequence as the patchify.  ``orig_height`` / ``orig_width``
    are then the resized sizes.
    """
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("vitok_b200.patchify_batch: device must be a CUDA device (there is no CPU path)")
    if (isinstance(images, torch.Tensor) and images.dim() == 4 and images.dtype == torch.uint8 and images.shape[-1] == 3
            and images.is_contiguous() and (images.shape[1] * images.shape[2] * 3) % 4 == 0):
        # a batched [B,H,W,3] uint8 tensor (decoded images): one H2D copy (if on the host) and one launch, with
        # to_tensor|normalize(minus_one_to_one) fused into the kernel (ops.py:140-161)
        B, H, W, _ = images.shape
        packed = images.to(dev, non_blocking=True).reshape(-1)
        return _patchify_packed(packed, [i * H * W * 3 for i in range(B)], [(H, W)] * B, 1, patch, max_tokens, out_dtype, dev,
                                resize_to_budget)
    if isinstance(images, torch.Tensor) and images.dim() == 4:
        imgs: List = list(images.unbind(0)) if not images.is_contiguous() else None
        if imgs is None:
            B, C, H, W = images.shape
            if C != 3 or images.dtype != torch.float32:
                raise ValueError("patchify_batch: a batched tensor must be [B,3,H,W] float32")
            sizes = [(H, W)] * B
            packed = images.to(dev).reshape(-1)
            offsets = [i * 3 * H * W for i in range(B)]
            in_dtype = 0
            return _patchify_packed(packed, offsets, sizes, in_dtype, patch, max_tokens, out_dtype, dev, resize_to_budget)
        images = imgs
    imgs = [torch.from_numpy(i) if isinstance(i, np.ndarray) else i for i in images]
    if not imgs:
        return {}
    u8 = imgs[0].dtype == torch.uint8
    sizes, offsets, flat, off = [], [], [], 0
    for t in imgs:
        if u8:
            if t.dtype != torch.uint8 or t.dim() != 3 or t.shape[2] != 3:
                raise ValueError("patchify_batch: uint8 images must be [H,W,3]")
            h, w = int(t.shape[0]), int(t.shape[1])
        else:
            if t.dtype != torch.float32 or t.dim() != 3 or t.shape[0] != 3:
                raise ValueError("patchify_batch: float images must be [3,H,W] float32")
            h, w = int(t.shape[1]), int(t.shape[2])
        sizes.append((h, w))
        offsets.append(off)
        n = 3 * h * w
        flat.append(t.reshape(-1))
        off += (n + 3) // 4 * 4  # keep every image 16-byte aligned for the vector path
    if all(t.is_cuda for t in flat):
        packed = torch.zeros(off, dtype=flat[0].dtype, device=dev)
        for t, o in zip(flat, offsets):
            packed[o:o + t.numel()] = t
    else:
        host = torch.zeros(off, dtype=flat[0].dtype).pin_memory()
        for t, o in zip(flat, offsets):
            host[o:o + t.numel()] = t.cpu()
        packed = host.to(dev, non_blocking=True)
    return _patchify_packed(packed, offsets, sizes, 1 if u8 else 0, patch, max_tokens, out_dtype, dev, resize_to_budget)


def pack_images(images: Sequence[Union[torch.Tensor, np.ndarray]], pin: bool = True):
    """Flatten a ragged list of images (all uint8 [H,W,3] or all float32 [3,H,W]) into ONE host buffer so that a
    serving loop moves a NaFlex batch to the GPU with a single H2D copy.  Returns (flat, offsets, sizes); feed the
    device copy of ``flat`` to ``patchify_packed``.  Every image starts on a 16-byte boundary."""
    imgs = [torch.from_numpy(i) if isinstance(i, np.ndarray) else i for i in images]
    u8 = imgs[0].dtype == torch.uint8
    sizes, offsets, off = [], [], 0
    for t in imgs:
        if u8 and (t.dtype != torch.uint8 or t.dim() != 3 or t.shape[2] != 3):
            raise ValueError("pack_images: uint8 images must be [H,W,3]")
        if not u8 and (t.dtype != torch.float32 or t.dim() != 3 or t.shape[0] != 3):
            raise ValueError("pack_images: float images must be [3,H,W] float32")
        h, w = (int(t.shape[0]), int(t.shape[1])) if u8 else (int(t.shape[1]), int(t.shape[2]))
        sizes.append((h, w))
        offsets.append(off)
        step = 16 if u8 else 4
        off += (3 * h * w + step - 1) // step * step
    flat = torch.zeros(off, dtype=imgs[0].dtype)
    if pin:
        flat = flat.pin_memory()
    for t, o in zip(imgs, offsets):
        flat[o:o + t.numel()] = t.reshape(-1).cpu()
    return flat, offsets, sizes


def patchify_packed(flat: torch.Tensor, offsets: Sequence[int], sizes: Sequence[Tuple[int, int]], patch: int = 16,
                    max_tokens: int = 256, out_dtype: torch.dtype = torch.float32,
                    resize_to_budget: bool = False) -> Dict[str, torch.Tensor]:
    """patchify + collate of a batch laid out by ``pack_images`` (``flat`` already on the GPU): one kernel launch.
    ``resize_to_budget``: as in ``patchify_batch``."""
    if not flat.is_cuda:
        raise RuntimeError("vitok_b200.patchify_packed: the packed image buffer must be on a CUDA device")
    if flat.dtype not in (torch.uint8, torch.float32):
        raise ValueError("patchify_packed: the packed buffer must be uint8 (HWC images) or float32 (CHW images)")
    return _patchify_packed(flat, list(offsets), list(sizes), 1 if flat.dtype == torch.uint8 else 0, patch, max_tokens,
                            out_dtype, flat.device, resize_to_budget)


_TABLE_CACHE: Dict = {}


def _patchify_packed(packed, offsets, sizes, in_dtype, patch, max_tokens, out_dtype, dev, resize_to_budget=False):
    B = len(sizes)
    targets = [_fit_to_token_budget(h, w, patch, max_tokens) for (h, w) in sizes] if resize_to_budget else sizes
    if list(targets) != list(sizes):
        return _resize_patchify_packed(packed, offsets, sizes, targets, in_dtype, patch, max_tokens, out_dtype, dev)
    for (h, w) in sizes:
        gr, gc = _grid(h, w, patch)
        if gr * gc > max_tokens:
            raise RuntimeError(f"patchify: image {h}x{w} needs {gr}x{gc}={gr * gc} patches > max_tokens={max_tokens} "
                               "(use resize_to_token_budget first)")
    if out_dtype not in (torch.float32, torch.bfloat16):
        raise ValueError("patchify: out_dtype must be float32 or bfloat16")
    key = (dev, tuple(offsets), tuple(sizes))
    table = _TABLE_CACHE.get(key)
    if table is None:       # {offset, H, W} per image; cached so that a steady-state loop issues no pageable H2D copy
        if len(_TABLE_CACHE) > 64:
            _TABLE_CACHE.clear()
        table = torch.tensor([[o, h, w] for o, (h, w) in zip(offsets, sizes)], dtype=torch.int64).to(dev)
        _TABLE_CACHE[key] = table
    P = 3 * patch * patch
    T = max_tokens
    patches = torch.empty(B, T, P, dtype=out_dtype, device=dev)
    mask = torch.empty(B, T, dtype=torch.bool, device=dev)
    idx = torch.empty(3, B, T, dtype=torch.int64, device=dev)
    meta = torch.empty(4, B, dtype=torch.int64, device=dev)
    with _lib.device_of(packed, patches):       # the launch and stream_ptr() follow the tensors' device, not the current one
        _lib.check(_lib.load().vtk_patchify_ex(packed.data_ptr(), table.data_ptr(), in_dtype, B, patch, T,
                                               0 if out_dtype == torch.float32 else 1, patches.data_ptr(), mask.data_ptr(),
                                               idx[0].data_ptr(), idx[1].data_ptr(), idx[2].data_ptr(), meta.data_ptr(), None,
                                               max(h for h, _ in sizes), max(w for _, w in sizes), _lib.stream_ptr()))
    return {"patches": patches, "patch_mask": mask, "row_idx": idx[0], "col_idx": idx[1], "time_idx": idx[2],
            "orig_height": meta[0], "orig_width": meta[1], "grid_rows": meta[2], "grid_cols": meta[3]}


def _resize_patchify_packed(packed, offsets, sizes, targets, in_dtype, patch, max_tokens, out_dtype, dev):
    """Over-budget images of the batch resized to ``targets`` on the device, fused with patchify (vtk_resize_patchify)."""
    if out_dtype not in (torch.float32, torch.bfloat16):
        raise ValueError("patchify: out_dtype must be float32 or bfloat16")
    for (h, w), (th, tw) in zip(sizes, targets):
        gr, gc = _grid(th, tw, patch)
        if gr * gc > max_tokens:    # _fit_to_token_budget keeps a 1-patch side at 1 patch: 1 x 4500 -> 1 x 4288 at p = 16
            raise RuntimeError(f"patchify: image {h}x{w} resized to {th}x{tw} needs {gr}x{gc}={gr * gc} patches > "
                               f"max_tokens={max_tokens} (the reference's patchify raises here too)")
    B = len(sizes)
    key = ("resize", dev, tuple(offsets), tuple(sizes), tuple(targets))
    cached = _TABLE_CACHE.get(key)
    if cached is None:      # {offset, H, W, h', w'} per image + the workspace size it needs
        if len(_TABLE_CACHE) > 64:
            _TABLE_CACHE.clear()
        host = torch.tensor([[o, h, w, th, tw] for o, (h, w), (th, tw) in zip(offsets, sizes, targets)], dtype=torch.int64)
        cached = (host.to(dev), int(_lib.load().vtk_resize_patchify_workspace_bytes(host.data_ptr(), B)))
        _TABLE_CACHE[key] = cached
    table, ws_bytes = cached
    P = 3 * patch * patch
    T = max_tokens
    patches = torch.empty(B, T, P, dtype=out_dtype, device=dev)
    mask = torch.empty(B, T, dtype=torch.bool, device=dev)
    idx = torch.empty(3, B, T, dtype=torch.int64, device=dev)
    meta = torch.empty(4, B, dtype=torch.int64, device=dev)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    with _lib.device_of(packed, patches):
        _lib.check(_lib.load().vtk_resize_patchify(packed.data_ptr(), table.data_ptr(), in_dtype, B, patch, T,
                                                   0 if out_dtype == torch.float32 else 1, patches.data_ptr(), mask.data_ptr(),
                                                   idx[0].data_ptr(), idx[1].data_ptr(), idx[2].data_ptr(), meta.data_ptr(),
                                                   ws.data_ptr(), ws_bytes, None, _lib.stream_ptr()))
    return {"patches": patches, "patch_mask": mask, "row_idx": idx[0], "col_idx": idx[1], "time_idx": idx[2],
            "orig_height": meta[0], "orig_width": meta[1], "grid_rows": meta[2], "grid_cols": meta[3]}


def patchify(patch: int = 16, max_tokens: int = 256):
    """OPS factory (``patchify(16, 256)`` in the DSL): [C,H,W] tensor -> per-image dict (ops.py:217-285).

    The tensor is patchified on the current CUDA device; the returned dict lives there.
    """
    def _patchify(img: torch.Tensor) -> dict:
        dev = img.device if img.is_cuda else torch.device("cuda")
        d = patchify_batch([img], patch, max_tokens, torch.float32, dev)
        return {k: v[0] for k, v in d.items()}
    _patchify.patch, _patchify.max_tokens = patch, max_tokens
    return _patchify


# --------------------------------------------------------------------------------------
# unpatchify / unpack
# --------------------------------------------------------------------------------------
def unpatchify(patch_dict: dict, patch: int = 16, max_grid_size: Optional[int] = None,
               output_format: str = "as_is") -> torch.Tensor:
    """patches -> [B,3,Gy*p,Gx*p] canvas (ops.py:295-335).  ``output_format`` optionally fuses the
    ``minus_one_to_one -> 0_255 | zero_to_one`` conversion of io.py:91-121 into the same kernel."""
    patches, mask = patch_dict["patches"], patch_dict["patch_mask"]
    row, col = patch_dict["row_idx"], patch_dict["col_idx"]
    if not patches.is_cuda:
        raise RuntimeError("vitok_b200.unpatchify: tensors must be on a CUDA device (there is no CPU path)")
    if patches.dtype not in (torch.float32, torch.bfloat16):
        raise RuntimeError(f"unpatchify: unsupported dtype {patches.dtype}")
    dev = patches.device
    B, N, dim = patches.shape
    if dim != 3 * patch * patch:
        raise RuntimeError(f"unpatchify: patch dim {dim} != 3*{patch}*{patch}")
    patches = patches.contiguous()
    m8 = mask.to(dev).bool().contiguous().view(torch.uint8)
    row = row.to(device=dev, dtype=torch.int64).contiguous()
    col = col.to(device=dev, dtype=torch.int64).contiguous()
    lib = _lib.load()
    with _lib.device_of(patches, m8, row, col):
        if max_grid_size is None:
            ext = torch.empty(2, dtype=torch.int32, device=dev)
            _lib.check(lib.vtk_grid_extent(m8.data_ptr(), row.data_ptr(), col.data_ptr(), B, N, ext.data_ptr(), _lib.stream_ptr()))
            gy, gx = (int(v) for v in ext.tolist())  # the reference syncs here too (ops.py:320-321)
            if gy == 0 or gx == 0:
                raise RuntimeError("unpatchify: no valid patches (max() of an empty tensor in the reference)")
        else:
            gy = gx = int(max_grid_size)
        fmt = _FMT[output_format]
        out_dtype = torch.uint8 if fmt == 1 else patches.dtype
        out = torch.empty(B, 3, gy * patch, gx * patch, dtype=out_dtype, device=dev)
        cell = torch.empty(B * gy * gx, dtype=torch.int32, device=dev)
        _lib.check(lib.vtk_unpatchify(patches.data_ptr(), 0 if patches.dtype == torch.float32 else 1, m8.data_ptr(),
                                      row.data_ptr(), col.data_ptr(), B, N, patch, gy, gx, cell.data_ptr(), out.data_ptr(), fmt,
                                      None, _lib.stream_ptr()))
    return out


def unpack(images: torch.Tensor, orig_h, orig_w) -> List[torch.Tensor]:
    """Crop each canvas to its original size (ops.py:338-360); one D2H copy instead of 2B ``.item()`` syncs."""
    if images.ndim == 3:
        images = images.unsqueeze(0)
    hs = orig_h.tolist() if isinstance(orig_h, torch.Tensor) else list(orig_h)
    ws = orig_w.tolist() if isinstance(orig_w, torch.Tensor) else list(orig_w)
    return [img[:, :int(h), :int(w)] for img, h, w in zip(images, hs, ws)]


# --------------------------------------------------------------------------------------
# token budget (host integers, ops.py:169-214)
# --------------------------------------------------------------------------------------
def _fit_to_token_budget(h: int, w: int, patch: int, max_tokens: int, eps: float = 1e-5) -> Tuple[int, int]:
    gh, gw = _grid(h, w, patch)
    if gh * gw <= max_tokens:
        return h, w
    s = math.sqrt(max_tokens / (gh * gw))
    nh = max(1, math.floor(gh * s + eps)) * patch
    nw = max(1, math.floor(gw * s + eps)) * patch
    return min(nh, h), min(nw, w)


def resize_to_token_budget(patch: int, max_tokens: int):
    import torchvision.transforms.functional as TF

    def _resize(img: torch.Tensor) -> torch.Tensor:
        _, h, w = img.shape
        th, tw = _fit_to_token_budget(h, w, patch, max_tokens)
        if (th, tw) != (h, w):
            img = TF.resize(img, [th, tw], interpolation=TF.InterpolationMode.BICUBIC, antialias=True)
        return img
    return _resize


# --------------------------------------------------------------------------------------
# host-side PIL ops (off the hot path; thin wrappers so reference DSL strings still parse and run)
# --------------------------------------------------------------------------------------
def resize_longest_side(max_size: int):
    import torchvision.transforms.functional as TF

    def _op(img):
        w, h = img.size
        longest = max(h, w)
        if longest <= max_size:
            return img
        f = max_size / longest
        return TF.resize(img, [int(round(h * f)), int(round(w * f))], interpolation=TF.InterpolationMode.LANCZOS, antialias=True)
    return _op


def center_crop(size: int):
    from PIL import Image

    def _op(img):
        while min(img.size) >= 2 * size:  # ADM-style pre-shrink by box filter
            img = img.resize((img.size[0] // 2, img.size[1] // 2), resample=Image.BOX)
        f = size / min(img.size)
        img = img.resize((round(img.size[0] * f), round(img.size[1] * f)), resample=Image.BICUBIC)
        left, top = (img.size[0] - size) // 2, (img.size[1] - size) // 2
        return img.crop((left, top, left + size, top + size))
    return _op


def random_resized_crop(size: int, scale=(0.8, 1.0), ratio=(0.75, 1.333)):
    import torchvision.transforms as T
    import torchvision.transforms.functional as TF
    return T.RandomResizedCrop(size, scale=scale, ratio=ratio, interpolation=TF.InterpolationMode.LANCZOS, antialias=True)


def flip(p: float = 0.5):
    import torchvision.transforms as T
    return T.RandomHorizontalFlip(p)


def identity() -> Callable:
    return lambda x: x


def random_choice(ops: Sequence[str], probs: Sequence[float]) -> Callable:
    if not ops:
        raise ValueError("ops cannot be empty")
    if len(ops) != len(probs):
        raise ValueError(f"ops and probs must have same length: {len(ops)} != {len(probs)}")
    from .registry import parse_op
    fns = []
    for spec in ops:
        name, args, kwargs = parse_op(spec)
        fns.append(OPS[name](*args, **kwargs))
    return lambda x: random.choices(fns, weights=probs, k=1)[0](x)


def to_tensor():
    import torchvision.transforms as T
    return T.ToTensor()


def normalize(mode: str = "minus_one_to_one"):
    import torchvision.transforms as T
    if mode == "minus_one_to_one":
        return T.Normalize(mean=[0.5] * 3, std=[0.5] * 3)
    if mode == "imagenet":
        return T.Normalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])
    if mode == "zero_to_one":
        return lambda x: x
    raise ValueError(f"Unknown normalize mode: '{mode}'. Use 'minus_one_to_one', 'imagenet', or 'zero_to_one'")


OPS = {
    "center_crop": center_crop, "random_resized_crop": random_resized_crop, "resize_longest_side": resize_longest_side,
    "resize_to_token_budget": resize_to_token_budget, "flip": flip, "identity": identity, "random_choice": random_choice,
    "to_tensor": to_tensor, "normalize": normalize, "patchify": patchify,
}

__all__ = ["OPS", "patchify", "patchify_batch", "pack_images", "patchify_packed", "unpatchify", "unpack", "resize_to_token_budget", "_fit_to_token_budget"]
