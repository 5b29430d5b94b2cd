"""numpy restatement of the antialiased bicubic resize behind resize_to_token_budget (vitok/pp/ops.py:169-214), i.e.
TF.resize(BICUBIC, antialias=True) = torch's CPU `_upsample_bicubic2d_aa`: the reference the device resize (vtk_resize_patchify) is
checked against, together with torchvision itself."""
from __future__ import annotations

import math
from typing import Dict, Tuple

import numpy as np

from oracle.pp_oracle import fit_to_token_budget, patchify


def _aa_cubic(x: np.ndarray) -> np.ndarray:
    """ATen's antialiasing bicubic filter (a = -0.5) in fp32; the CPU build contracts both polynomials into FMAs, emulated
    here through float64 (one rounding to fp32 of the exact a * b + c)."""
    f32, f64 = np.float32, np.float64

    def fma(a, b, c):
        return (f64(a) * f64(b) + f64(c)).astype(f32)
    x = np.abs(x.astype(f32))
    near = fma(fma(f32(1.5), x, f32(-2.5)) * x, x, f32(1.0))
    far = fma(fma(fma(f32(-0.5), x, f32(2.5)), x, f32(-4.0)), x, f32(2.0))
    return np.where(x < 1, near, np.where(x < 2, far, f32(0))).astype(f32)


def resize_table(n_in: int, n_out: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Resample table of one axis of an antialiased bicubic resize, torch's `_upsample_bicubic2d_aa` with align_corners=False
    (what TF.resize(BICUBIC, antialias=True) runs, vitok/pp/ops.py:198-214).  Returns (xmin [n_out], taps [n_out],
    weights [n_out, K]): output o = sum over j < taps[o] of in[xmin[o] + j] * weights[o, j].  Same float / double mix as
    ATen's _compute_indices_min_size_weights_aa."""
    f32, f64 = np.float32, np.float64
    scale = f32(f32(n_in) / f32(n_out))
    support = f32(2.0 * f64(scale)) if scale >= 1 else f32(2.0)
    K = int(math.ceil(f64(support))) * 2 + 1
    invscale = f32(1.0 / f64(scale)) if scale >= 1 else f32(1.0)
    o = np.arange(n_out)
    center = (f64(scale) * (o + 0.5)).astype(f32)
    xmin = np.maximum(((center - support).astype(f32).astype(f64) + 0.5).astype(np.int64), 0)
    taps = np.minimum(((center + support).astype(f32).astype(f64) + 0.5).astype(np.int64), n_in) - xmin
    taps = np.clip(taps, 0, K)
    j = np.arange(K)
    d = ((xmin[:, None] + j[None]).astype(f32) - center[:, None]).astype(f32)
    w = _aa_cubic(((d.astype(f64) + 0.5) * f64(invscale)).astype(f32))
    w = np.where(j[None] < taps[:, None], w, f32(0)).astype(f32)
    total = np.zeros(n_out, f32)
    for k in range(K):                      # fp32 running sum in tap order
        total = (total + w[:, k]).astype(f32)
    w = np.where(total[:, None] != 0, w / np.where(total == 0, f32(1), total)[:, None], w).astype(f32)
    return xmin, taps, w


def _resample_last_axis(x: np.ndarray, n_out: int) -> np.ndarray:
    xmin, taps, w = resize_table(x.shape[-1], n_out)
    idx = np.minimum(xmin[:, None] + np.arange(w.shape[1])[None], x.shape[-1] - 1)
    out = (x[..., idx[:, 0]] * w[:, 0]).astype(np.float32)
    for k in range(1, w.shape[1]):          # out = x0 * w0; out += xk * wk -- products rounded, summed in tap order
        out = np.where(k < taps, (out + (x[..., idx[:, k]] * w[:, k]).astype(np.float32)).astype(np.float32), out)
    return out


def resize_aa(img: np.ndarray, h: int, w: int) -> np.ndarray:
    """[C, H, W] float32 -> [C, h, w]: TF.resize(img, [h, w], BICUBIC, antialias=True) (vitok/pp/ops.py:198-214).  Width pass
    first, then height, as torch's CPU kernel; an axis whose size is unchanged is not resampled."""
    x = np.asarray(img, dtype=np.float32)
    if w != x.shape[2]:
        x = _resample_last_axis(x, w)
    if h != x.shape[1]:
        x = np.swapaxes(_resample_last_axis(np.swapaxes(x, 1, 2), h), 1, 2)
    return np.ascontiguousarray(x)


def resize_patchify(img: np.ndarray, patch: int = 16, max_tokens: int = 256) -> Dict[str, np.ndarray]:
    """resize_to_token_budget(p, T) | patchify(p, T): vitok/pp/ops.py:198-214 then :217-285."""
    _, h, w = img.shape
    th, tw = fit_to_token_budget(h, w, patch, max_tokens)
    return patchify(resize_aa(img, th, tw) if (th, tw) != (h, w) else img, patch, max_tokens)
