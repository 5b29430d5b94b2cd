"""``preprocess`` / ``postprocess`` over the NaFlex patch dictionary (mirror of vitok/pp/io.py).

preprocess : PIL image(s) -> batched patch dict on the GPU.  The DSL string is parsed exactly like the
             reference; every op up to ``patchify`` that works on PIL images runs on the host (they are
             not on the hot path), and the trailing ``to_tensor|normalize(minus_one_to_one)|patchify(p,T)``
             is executed as ONE kernel on uint8 HWC pixels (4x fewer H2D bytes than the reference's fp32
             upload, bit-identical output) writing straight into the batched buffers.  With ``fuse_resize=True`` a
             trailing ``...|normalize(minus_one_to_one)|resize_to_token_budget(p,T)|patchify(p,T)`` runs the same way, the
             resize done on the GPU inside the patchify launch sequence (within a few fp32 ulps of torchvision's resize).
postprocess: patch dict -> images; unpatchify + format conversion fused in one kernel, then ``unpack``.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Union

import numpy as np
import torch

from .ops import OPS, patchify_batch, unpack, unpatchify
from .registry import parse_pipeline

_FORMATS = ("minus_one_to_one", "zero_to_one", "0_255")


def preprocess(images, pp: str = "to_tensor|normalize(minus_one_to_one)|patchify(16, 256)",
               device: str = "cuda", fuse_resize: bool = False) -> Dict[str, torch.Tensor]:
    """PIL image(s) -> batched patch dict with fp32 patches on ``device`` (io.py:18-49).

    fuse_resize: when the pipeline ends in ``to_tensor|normalize(minus_one_to_one)|resize_to_token_budget(p,T)|patchify(p,T)``
    (same p and T in both ops), decode to uint8 and resize + normalize + patchify on the GPU (``patchify_batch(...,
    resize_to_budget=True)``) instead of running torchvision's resize per image on the host.  Off by default: the GPU resize
    is not bit-identical to torchvision's.
    """
    if not isinstance(images, (list, tuple)):
        images = [images]
    steps = parse_pipeline(pp)
    if not steps or steps[-1][0] != "patchify":
        # not a patchifying pipeline: exactly what the reference does (io.py:43-49) -- transform every image, collate, move the
        # dict's tensors to the device (for tensor- or PIL-valued pipelines that last step raises AttributeError there too)
        from ..data import patch_collate_fn
        from .registry import build_transform
        transform = build_transform(pp)
        batched = patch_collate_fn([transform(img) for img in images])
        return {k: v.to(device) if isinstance(v, torch.Tensor) else v for k, v in batched.items()}
    _, pargs, pkw = steps[-1]
    probe = OPS["patchify"](*pargs, **pkw)
    patch, max_tokens = probe.patch, probe.max_tokens
    head = steps[:-1]
    resize = fuse_resize and len(head) >= 3 and head[-1][0] == "resize_to_token_budget" and \
        _budget_args(head[-1]) == (patch, max_tokens)
    if resize:
        head = head[:-1]
    fused = (len(head) >= 2 and head[-2][0] == "to_tensor" and head[-1][0] == "normalize"
             and (head[-1][1] + ("minus_one_to_one",))[0] == "minus_one_to_one" and not head[-1][2])
    if resize and not fused:            # the resize only fuses behind to_tensor|normalize(minus_one_to_one): keep it a host step
        head, resize = steps[:-1], False
    host_steps = head[:-2] if fused else head
    fns = [OPS[n](*a, **k) for n, a, k in host_steps]
    outs = []
    for img in images:
        for fn in fns:
            img = fn(img)
        outs.append(img)
    if fused:
        arrs = []
        for img in outs:
            a = np.asarray(img.convert("RGB") if hasattr(img, "convert") and getattr(img, "mode", "RGB") != "RGB" else img)
            if a.ndim != 3 or a.shape[2] != 3 or a.dtype != np.uint8:
                raise ValueError("preprocess: expected 8-bit RGB PIL images")
            arrs.append(np.ascontiguousarray(a))
        return patchify_batch(arrs, patch, max_tokens, torch.float32, device, resize_to_budget=resize)
    return patchify_batch(outs, patch, max_tokens, torch.float32, device)


def _budget_args(step):
    """(patch, max_tokens) of a parsed ``resize_to_token_budget(...)`` step."""
    import inspect
    _, args, kwargs = step
    bound = inspect.signature(OPS["resize_to_token_budget"]).bind(*args, **kwargs).arguments
    return int(bound["patch"]), int(bound["max_tokens"])


def postprocess(output: Union[torch.Tensor, Dict[str, torch.Tensor]], output_format: str = "minus_one_to_one",
                current_format: str = "minus_one_to_one", do_unpack: bool = True, patch: int = 16,
                max_grid_size: Optional[int] = None) -> Union[torch.Tensor, List[torch.Tensor]]:
    """Model output -> images (io.py:52-88)."""
    if isinstance(output, torch.Tensor):
        return _convert_format(output, current_format, output_format)
    if do_unpack and (output.get("orig_height") is None or output.get("orig_width") is None):
        raise ValueError("do_unpack=True requires 'orig_height' and 'orig_width' in output")
    fused = current_format == "minus_one_to_one" and output_format in ("0_255", "zero_to_one")
    images = unpatchify(output, patch=patch, max_grid_size=max_grid_size, output_format=output_format if fused else "as_is")
    if not fused:
        images = _convert_format(images, current_format, output_format)
    if do_unpack:
        return unpack(images, output["orig_height"], output["orig_width"])
    return images


def _convert_format(images: torch.Tensor, from_format: str, to_format: str) -> torch.Tensor:
    """Stand-alone format conversion of an image tensor (io.py:91-121).  Elementwise and off the
    encode/decode path (the dict path fuses it into unpatchify); same operation order as the reference."""
    if from_format == to_format:
        return images
    if to_format == "minus_one_to_one":
        if from_format == "0_255":
            return (images.float() / 127.5 - 1.0).clamp(-1.0, 1.0)
        if from_format == "zero_to_one":
            return (images * 2.0 - 1.0).clamp(-1.0, 1.0)
    elif to_format == "zero_to_one":
        if from_format == "0_255":
            return (images.float() / 255.0).clamp(0.0, 1.0)
        if from_format == "minus_one_to_one":
            return ((images + 1.0) / 2.0).clamp(0.0, 1.0)
    elif to_format == "0_255":
        if from_format == "minus_one_to_one":
            return ((images.clamp(-1.0, 1.0) + 1.0) / 2.0 * 255).round().to(torch.uint8)
        if from_format == "zero_to_one":
            return (images.clamp(0.0, 1.0) * 255).round().to(torch.uint8)
    return images


preprocess_images = preprocess
postprocess_images = postprocess

__all__ = ["preprocess", "postprocess", "preprocess_images", "postprocess_images"]
