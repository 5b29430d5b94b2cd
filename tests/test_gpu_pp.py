"""GPU parity (bit-exact): patchify / unpatchify / index packing / format conversion vs oracle + golden."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

from oracle import pp_oracle
from oracle.make_golden import PP_CASES
from oracle.weights import C3_SIZES, synth_images

pytestmark = pytest.mark.gpu


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def ppmeta(golden_dir):
    with open(os.path.join(golden_dir, "pp.json")) as f:
        return json.load(f)


@pytest.mark.parametrize("ci", range(len(PP_CASES)))
def test_patchify_matches_reference_golden(ci, ppmeta):
    import vitok_b200 as vb
    H, W, p, T = PP_CASES[ci]
    m = ppmeta[f"case{ci}"]
    img = synth_images([(H, W)], seed=100 + ci)[0]
    d = vb.patchify_batch([torch.from_numpy(img)], p, T)
    for k in ("patches", "patch_mask", "row_idx", "col_idx", "time_idx", "orig_height", "orig_width", "grid_rows", "grid_cols"):
        assert sha(d[k][0].cpu().numpy()) == m[k], (ci, k)
    canvas = vb.unpatchify(d, patch=p)
    assert list(canvas.shape) == m["unpatchify_shape"]
    assert sha(canvas.cpu().numpy()) == m["unpatchify_sha"]
    assert sha(vb.postprocess(d, output_format="0_255", do_unpack=False, patch=p).cpu().numpy()) == m["u8_sha"]
    assert sha(vb.postprocess(d, output_format="zero_to_one", do_unpack=False, patch=p).cpu().numpy()) == m["zero_to_one_sha"]
    assert np.array_equal(canvas[0, :, :H, :W].cpu().numpy(), img)          # round trip
    # per-image OPS entry point (DSL "patchify(p, T)")
    d1 = vb.OPS["patchify"](p, T)(torch.from_numpy(img))
    assert sha(d1["patches"].cpu().numpy()) == m["patches"] and d1["orig_height"].item() == H


def test_ragged_batch_matches_reference_golden(ppmeta):
    import vitok_b200 as vb
    m = ppmeta["ragged"]
    imgs = [torch.from_numpy(i) for i in synth_images(C3_SIZES[:6], seed=77)]
    batch = vb.patchify_batch(imgs, 16, 1024)
    for k, v in batch.items():
        assert sha(v.cpu().numpy()) == m[k + "_sha"], k
    canvas = vb.unpatchify(batch, 16)
    assert list(canvas.shape) == m["canvas_shape"] and sha(canvas.cpu().numpy()) == m["canvas_sha"]
    assert sha(vb.unpatchify(batch, 16, max_grid_size=32).cpu().numpy()) == m["canvas32_sha"]
    crops = vb.postprocess(batch, output_format="0_255", do_unpack=True, patch=16)
    assert [list(c.shape) for c in crops] == m["crops_shape"]
    assert [sha(c.contiguous().cpu().numpy()) for c in crops] == m["crops_sha"]


@pytest.mark.parametrize("patch,sizes", [
    (16, [(256, 256), (130, 131), (37, 300)]),
    # the strip kernel's other paths: p = 32 (32-row strips), widths beyond one 256-pixel strip with aligned (512, 272) and unaligned
    # rows (517, 259), a one-pixel image, heights that are not multiples of the patch size
    (32, [(512, 512), (100, 517), (33, 259), (1, 1), (64, 272)]),
    (16, [(16, 512), (515, 16), (48, 272), (1, 700)]),
])
def test_uint8_fused_frontend_bit_exact(patch, sizes):
    """N1: uint8 HWC -> to_tensor|normalize|patchify in one kernel == oracle on the same pixels (fp32 and bf16 outputs)."""
    import vitok_b200 as vb
    rng = np.random.default_rng(0)
    u8 = [rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8) for h, w in sizes]
    T = max(((h + patch - 1) // patch) * ((w + patch - 1) // patch) for h, w in sizes) + 3      # a few padding tokens per image too
    got = vb.patchify_batch(u8, patch, T)
    want = pp_oracle.collate([pp_oracle.patchify(pp_oracle.normalize_u8(a), patch, T) for a in u8])
    for k in want:
        assert np.array_equal(got[k].cpu().numpy(), want[k]), k
    got16 = vb.patchify_batch(u8, patch, T, out_dtype=torch.bfloat16)
    assert torch.equal(got16["patches"], got["patches"].to(torch.bfloat16))
    assert torch.equal(got16["patch_mask"], got["patch_mask"]) and torch.equal(got16["row_idx"], got["row_idx"])


def test_uint8_batched_tensor_frontend_and_u8_roundtrip():
    """A [B,H,W,3] uint8 batch (host or device) takes the one-copy path; with the fused 0_255 back-end the
    uint8 -> patches -> uint8 round trip is the identity (io.py:115-119: round(clamp((x+1)/2)*255))."""
    import vitok_b200 as vb
    rng = np.random.default_rng(3)
    u8 = rng.integers(0, 256, size=(5, 96, 128, 3), dtype=np.uint8)
    want = pp_oracle.collate([pp_oracle.patchify(pp_oracle.normalize_u8(a), 16, 64) for a in u8])
    for src in (torch.from_numpy(u8), torch.from_numpy(u8).cuda(), torch.from_numpy(u8).pin_memory()):
        got = vb.patchify_batch(src, 16, 64)
        for k in want:
            assert np.array_equal(got[k].cpu().numpy(), want[k]), k
    back = vb.unpatchify(got, 16, max_grid_size=8, output_format="0_255")      # canvas 128 x 128, image in the top-left
    assert back.dtype == torch.uint8
    assert np.array_equal(back[:, :, :96, :128].permute(0, 2, 3, 1).cpu().numpy(), u8)


def test_arithmetic_normalisation_equals_ieee_division_for_all_bytes():
    """The three-FMA normalisation (no table, no division sequence) is bit-identical to (u / 255 - 0.5) / 0.5 for all 256 inputs
    (device-side exhaustive check), and the uint8 front end's output equals numpy's on them."""
    import vitok_b200 as vb
    from vitok_b200 import _lib
    bad = torch.full((1,), -1, dtype=torch.int32, device="cuda")
    _lib.check(_lib.load().vtk_patchify_selftest(bad.data_ptr(), _lib.stream_ptr()))
    assert int(bad.item()) == 0
    ramp = np.arange(256, dtype=np.uint8).reshape(16, 16, 1).repeat(3, axis=2)       # one 16 x 16 patch holding every byte value
    got = vb.patchify_batch([ramp], 16, 1)["patches"].cpu().numpy().reshape(3, 256)
    want = ((np.arange(256, dtype=np.float32) / np.float32(255.0)) - np.float32(0.5)) / np.float32(0.5)
    assert np.array_equal(got[0], want) and np.array_equal(got[2], want)


@pytest.mark.parametrize("out_format", ["as_is", "0_255", "zero_to_one"])
def test_unpatchify_row_and_cell_kernels_match_reference(out_format):
    """unpatchify has two kernels (row-coalesced writes for p = 16 / 32, cell-per-warp for any other patch size).  On a ragged batch
    with padding tokens and a canvas larger than every image, both equal the reference: fp32 patches bit for bit the numpy oracle,
    bf16 patches the io.py:91-121 operations evaluated by torch on a bf16 CPU tensor (each eager op rounds to bf16)."""
    import vitok_b200 as vb

    def io_convert(x):   # vitok/pp/io.py:91-121 from "minus_one_to_one"
        if out_format == "0_255":
            return ((x.clamp(-1.0, 1.0) + 1.0) / 2.0 * 255).round().to(torch.uint8)
        if out_format == "zero_to_one":
            return ((x + 1.0) / 2.0).clamp(0.0, 1.0)
        return x

    rng = np.random.default_rng(5)
    imgs = [torch.from_numpy(rng.standard_normal((3, h, w)).astype(np.float32)) for h, w in [(128, 128), (96, 64), (50, 120), (16, 16)]]
    for p, T, grid in ((8, 256, 18), (16, 64, 9)):       # generic kernel, row kernel
        for dt in (torch.float32, torch.bfloat16):
            d = vb.patchify_batch(imgs, p, T, out_dtype=dt)
            got = vb.unpatchify(d, p, max_grid_size=grid, output_format=out_format).cpu()
            canvas = pp_oracle.unpatchify({k: v.float().cpu().numpy() if k == "patches" else v.cpu().numpy() for k, v in d.items()},
                                          p, max_grid_size=grid)
            if dt == torch.float32:
                want = pp_oracle.convert_format(canvas, "minus_one_to_one", out_format)
                assert np.array_equal(got.numpy(), want), (p, dt)
            else:
                want = io_convert(torch.from_numpy(canvas).to(torch.bfloat16))
                assert got.dtype == want.dtype and torch.equal(got, want), (p, dt)


def test_full_size_roundtrip_and_bf16():
    """BASELINE config sizes: 64 x 256^2 (c2) and 8 x 512^2 (c4): patchify -> unpatchify is the identity."""
    import vitok_b200 as vb
    for B, S, T in [(64, 256, 256), (8, 512, 1024)]:
        g = torch.Generator().manual_seed(7)
        imgs = (torch.rand(B, 3, S, S, generator=g) * 2 - 1).cuda()
        d = vb.patchify_batch(imgs, 16, T)
        assert bool(d["patch_mask"].all())
        assert torch.equal(vb.unpatchify(d, 16), imgs)
        db = vb.patchify_batch(imgs, 16, T, out_dtype=torch.bfloat16)
        assert torch.equal(db["patches"], d["patches"].to(torch.bfloat16))
        assert torch.equal(vb.unpatchify(db, 16), imgs.to(torch.bfloat16))


def test_errors():
    import vitok_b200 as vb
    with pytest.raises(RuntimeError):
        vb.patchify_batch([torch.zeros(3, 640, 480)], 16, 256)      # grid exceeds the budget (ops.py:260)
    d = vb.patchify_batch([torch.zeros(3, 64, 64)], 16, 16)
    d2 = {k: v for k, v in d.items() if k not in ("orig_height", "orig_width")}
    with pytest.raises(ValueError):
        vb.postprocess(d2, do_unpack=True)                           # io.py:84-85
    with pytest.raises(RuntimeError):
        vb.unpatchify({k: v.cpu() for k, v in d.items()})            # no CPU path
