"""CPU tests of the antialiased bicubic resize behind ``resize_to_token_budget`` (vitok/pp/ops.py:169-214): the numpy oracle's
resample tables against torch's own weights, its outputs against TF.resize, and the C ABI's host-side workspace size."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import _resize_oracle as resize_oracle
from oracle import pp_oracle

# (H, W, patch, max_tokens): photo sizes, 1.1x to 15x downscales, one axis unchanged, 1-pixel and 4000-pixel sides, sizes that
# are not multiples of p, p = 32
BUDGET_CASES = [
    (375, 500, 16, 256),      # ImageNet photo, 1.56x
    (480, 640, 16, 256),
    (3024, 4032, 16, 256),    # 12 MP phone photo, 14.5x / 14x
    (64, 4000, 16, 256),      # 2x / 1.98x
    (1, 4500, 16, 256),       # 1-pixel height: only the width is resampled (4500 -> 4288)
    (4000, 1, 16, 64),        # 1-pixel width: only the height is resampled
    (300, 20, 16, 16),        # 1.46x height, width unchanged (min(n, w) clamps it)
    (17, 290, 16, 16),        # width resampled, height unchanged
    (333, 517, 32, 64),       # p = 32, 1.33x
    (263, 263, 16, 256),      # 1.1x
    (2049, 1537, 32, 64),     # p = 32, 8x
]


def _torch_weights(n_in, n_out):
    """torch's exact weight matrix [n_in, n_out]: resize one-hot rows (the height n_in is unchanged, so it is not resampled)."""
    return F.interpolate(torch.eye(n_in)[None, None], size=(n_in, n_out), mode="bicubic", antialias=True)[0, 0].numpy()


def _dense(n_in, table):
    xmin, taps, w = table
    m = np.zeros((n_in, len(xmin)), np.float32)
    for o in range(len(xmin)):
        m[xmin[o]:xmin[o] + taps[o], o] = w[o, :taps[o]]
    return m


@pytest.mark.parametrize("n_in,n_out", [(500, 320), (375, 240), (4032, 288), (3024, 208), (4000, 2016), (131, 96), (17, 16),
                                        (64, 32), (1000, 66), (4500, 4096), (7, 13), (900, 60)])
def test_oracle_tables_match_torch_weights(n_in, n_out):
    got = _dense(n_in, resize_oracle.resize_table(n_in, n_out))
    ref = _torch_weights(n_in, n_out)
    assert np.abs(got - ref).max() <= 3e-7
    xmin, taps, w = resize_oracle.resize_table(n_in, n_out)
    assert (taps >= 1).all() and (xmin >= 0).all() and (xmin + taps <= n_in).all()


@pytest.mark.parametrize("H,W,p,T", BUDGET_CASES)
def test_oracle_resize_matches_torchvision(H, W, p, T):
    import torchvision.transforms.functional as TF
    th, tw = pp_oracle.fit_to_token_budget(H, W, p, T)
    assert (th, tw) != (H, W)
    img = (np.random.default_rng(H * 7919 + W).random((3, H, W), dtype=np.float32) * 2 - 1).astype(np.float32)
    if W == 1:
        # torch's CPU kernel returns every output row equal to the first for a 1-pixel-wide NCHW input (its channels-last
        # layout gives the right result); the same resize of the transposed image is the reference here
        t = TF.resize(torch.from_numpy(img).transpose(1, 2), [tw, th], interpolation=TF.InterpolationMode.BICUBIC, antialias=True)
        ref = t.transpose(1, 2).numpy()
    else:
        ref = TF.resize(torch.from_numpy(img), [th, tw], interpolation=TF.InterpolationMode.BICUBIC, antialias=True).numpy()
    got = resize_oracle.resize_aa(img, th, tw)
    assert got.shape == ref.shape == (3, th, tw)
    assert np.abs(got - ref).max() <= 2e-6
    if th == H or tw == W:       # the unchanged axis is not resampled: an unchanged row / column is copied exactly
        ax = 1 if th == H else 2
        assert got.shape[ax] == img.shape[ax]


def test_oracle_resize_patchify_fits_the_budget():
    for H, W, p, T in BUDGET_CASES:
        th, tw = pp_oracle.fit_to_token_budget(H, W, p, T)
        if -(-th // p) * -(-tw // p) > T:
            # max(1, .) keeps a 1-patch side at one patch while the other side shrinks by the full factor: 1 x 4500 -> 1 x 4288,
            # 268 patches at p = 16.  The reference's patchify raises on it (ops.py:260); so do the oracle and the product.
            assert min(H, W) == 1
            with pytest.raises(RuntimeError):
                resize_oracle.resize_patchify(np.zeros((3, H, W), np.float32), p, T)
            continue
        d = resize_oracle.resize_patchify(np.zeros((3, H, W), np.float32), p, T)
        assert (int(d["orig_height"]), int(d["orig_width"])) == (th, tw)
        assert int(d["grid_rows"]) * int(d["grid_cols"]) <= T


def _kt(n_in, n_out):
    return 4 * (-(-n_in // n_out)) + 1


def test_kt_bounds_aten_tap_count():
    """The device tables give every output coordinate 4 * ceil(n_in / n_out) + 1 weight slots; ATen uses ceil(support) * 2 + 1."""
    for n_in in range(1, 300, 7):
        for n_out in range(1, 300, 5):
            assert resize_oracle.resize_table(n_in, n_out)[2].shape[1] <= _kt(n_in, n_out)


def test_workspace_bytes_restates_the_layout():
    from vitok_b200 import _lib
    lib = _lib.load()
    sizes = [(375, 500), (128, 128), (3024, 4032), (64, 4000), (300, 20), (17, 290)]
    rows = []
    for i, (h, w) in enumerate(sizes):
        th, tw = pp_oracle.fit_to_token_budget(h, w, 16, 256 if i < 4 else 16)
        rows.append([i * 1000, h, w, th, tw])
    table = np.ascontiguousarray(np.array(rows, dtype=np.int64))
    floats = 0
    for _, h, w, th, tw in rows:
        if tw != w:
            floats += tw * (_kt(w, tw) + 2) + 3 * h * tw
        if th != h:
            floats += th * (_kt(h, th) + 2)
    header = ((2 * len(rows) + 3) * 8 + 255) // 256 * 256
    got = lib.vtk_resize_patchify_workspace_bytes(table.ctypes.data_as(ctypes.c_void_p), len(rows))
    assert got == header + 4 * floats
    assert lib.vtk_resize_patchify_workspace_bytes(None, 0) == 0
