"""vitok_b200.ssim: per-tile SSIM on NaFlex patch batches (csrc/vtk_ssim.cu), forward and backward.

The reference here is float64 torch: a differentiable canvas gathered from the patches through unpatchify's cell map (checked
against ``vitok_b200.unpatchify`` bit for bit), mapped to [0, 1], cropped to each tile and run through a grouped ``conv2d`` with
the 11 x 11 gaussian.  Whole-image tiles are also checked against ``oracle.ae_oracle.ssim``.  Gradients are float64 autograd
through that canvas with a random upstream [T] gradient."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ae_oracle, pp_oracle
from oracle.weights import make_state_dict, synth_images

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
SIZES = [(11, 11), (16, 16), (17, 300), (130, 131), (500, 333), (512, 512)]
VAL_TOL = 1e-4
GRAD_TOL = {torch.float32: 1e-3, BF: 1e-2}


def _gauss64():
    ax = torch.arange(11, dtype=torch.float64) - 5
    g = torch.exp(-(ax / 1.5) ** 2 / 2)
    g = g / g.sum()
    return (g[:, None] * g[None, :]).expand(3, 1, 11, 11).contiguous()


def _canvas(patches, mask, row, col, patch):
    """Differentiable [B, 3, gy*p, gx*p] canvas of unpatchify (ops.py:295-335): grid = max(row)+1 x max(col)+1 over valid tokens,
    the later valid token wins a shared cell, token 0 is re-scattered into cell 0, cells without a token read 0."""
    B, N, P = patches.shape
    m = mask.bool()
    gy, gx = int(row[m].max()) + 1, int(col[m].max()) + 1
    cell = torch.full((B, gy * gx), -1, dtype=torch.int64, device=patches.device)
    tok = torch.arange(N, device=patches.device).expand(B, N)
    idx = torch.where(m, row * gx + col, torch.zeros_like(row))
    cell.scatter_reduce_(1, idx, torch.where(m, tok, torch.full_like(tok, -1)), reduce="amax")
    cell[:, 0] = torch.where(m[:, 0], 0, -1)
    src = patches.gather(1, cell.clamp_min(0)[:, :, None].expand(-1, -1, P)) * (cell >= 0)[:, :, None].to(patches.dtype)
    return src.reshape(B, gy, gx, 3, patch, patch).permute(0, 3, 1, 4, 2, 5).reshape(B, 3, gy * patch, gx * patch)


def _ssim_ref(pred, target, batch, patch, tiles, fmt="minus_one_to_one"):
    """float64 per-tile SSIM of the definition; differentiable w.r.t. pred (float64)."""
    cp = _canvas(pred, batch["patch_mask"], batch["row_idx"], batch["col_idx"], patch)
    ct = _canvas(target.double(), batch["patch_mask"], batch["row_idx"], batch["col_idx"], patch)
    if fmt == "minus_one_to_one":
        cp, ct = (cp + 1) / 2, (ct + 1) / 2
    k = _gauss64().to(pred.device)
    c1, c2 = 0.01 ** 2, 0.03 ** 2
    out = []
    for b, y0, x0, h, w in tiles.tolist():
        a, t = cp[b:b + 1, :, y0:y0 + h, x0:x0 + w], ct[b:b + 1, :, y0:y0 + h, x0:x0 + w]
        mo = F.conv2d(torch.cat([a, t, a * a, t * t, a * t]), k, groups=3)
        ma, mb, eaa, ebb, eab = mo.split(1)
        s = ((2 * ma * mb + c1) * (2 * (eab - ma * mb) + c2)) / ((ma * ma + mb * mb + c1) * ((eaa - ma * ma) + (ebb - mb * mb) + c2))
        out.append(s.mean())
    return torch.stack(out)


def _batch(sizes, patch, dtype, seed, noise=0.3):
    """Ragged batch of synthetic images (target) and a prediction = target + noise (blurred a little so that SSIM is neither 0 nor
    1) on every token; the prediction of masked tokens is garbage (must not matter)."""
    import vitok_b200 as vb
    imgs = [torch.from_numpy(i) for i in synth_images(sizes, seed=seed)]
    max_tok = max(((h + patch - 1) // patch) * ((w + patch - 1) // patch) for h, w in sizes)
    b = vb.patchify_batch(imgs, patch, max_tok, out_dtype=dtype, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(seed)
    pred = (b["patches"].float() * 0.8 + noise * torch.randn(b["patches"].shape, generator=g, device="cuda")).to(dtype)
    return b, pred


def _check(batch, pred, patch, tiles, fmt="minus_one_to_one", tag=""):
    """Kernel values and gradient against the float64 reference; returns (value error / bound, grad rel-Fro / bound)."""
    import vitok_b200 as vb
    p = pred.detach().clone().requires_grad_(True)
    val = vb.ssim(p, batch, patch, tiles=tiles, current_format=fmt)
    gen = torch.Generator(device="cuda").manual_seed(7)
    gout = torch.randn(val.shape, generator=gen, device="cuda")
    (val * gout).sum().backward()
    if tiles is None:
        tiles = torch.stack([torch.arange(len(batch["orig_height"])), torch.zeros(len(batch["orig_height"]), dtype=torch.int64),
                             torch.zeros(len(batch["orig_height"]), dtype=torch.int64), batch["orig_height"].cpu(),
                             batch["orig_width"].cpu()], 1)
    p64 = pred.detach().double().requires_grad_(True)
    ref = _ssim_ref(p64, batch["patches"], batch, patch, torch.as_tensor(tiles), fmt)
    (ref * gout.double()).sum().backward()
    verr = (val.double() - ref.detach()).abs().max().item()
    assert verr <= VAL_TOL, (tag, verr, val, ref)
    g, gr = p.grad.double(), p64.grad
    assert p.grad.dtype == pred.dtype
    assert torch.isfinite(g).all()
    rel = (torch.linalg.norm(g - gr) / torch.linalg.norm(gr)).item()
    bound = GRAD_TOL[pred.dtype]
    assert rel <= bound, (tag, rel)
    zero = gr == 0      # masked / duplicate / padding tokens, pad pixels, pixels outside every tile
    assert bool((g[zero] == 0).all()), (tag, int((g[zero] != 0).sum()))
    assert bool((p.grad[~batch["patch_mask"].bool()] == 0).all())
    print(f"[ssim] {tag}: value err {verr:.2e} ({verr / VAL_TOL:.3f} of bound), grad rel-Fro {rel:.2e} ({rel / bound:.3f} of bound), "
          f"{int(zero.sum())} exact zeros")
    return val, p.grad


def test_canvas_reference_is_unpatchify():
    import vitok_b200 as vb
    for patch, dtype in ((16, torch.float32), (32, BF)):
        b, _ = _batch(SIZES, patch, dtype, seed=1)
        ref = _canvas(b["patches"], b["patch_mask"], b["row_idx"], b["col_idx"], patch)
        assert torch.equal(vb.unpatchify(b, patch), ref)


@pytest.mark.parametrize("patch", [16, 32])
@pytest.mark.parametrize("dtype", [torch.float32, BF], ids=["fp32", "bf16"])
def test_ssim_whole_images(patch, dtype):
    b, pred = _batch(SIZES, patch, dtype, seed=3 + patch)
    val, _ = _check(b, pred, patch, None, tag=f"whole images p={patch} {dtype}")
    # the oracle's definition on each image's own region (the crop ``unpack`` returns)
    import vitok_b200 as vb
    cp, ct = vb.unpatchify({**b, "patches": pred}, patch).double().cpu(), vb.unpatchify(b, patch).double().cpu()
    for i, (h, w) in enumerate(SIZES):
        o = ae_oracle.ssim((cp[i:i + 1, :, :h, :w] + 1) / 2, (ct[i:i + 1, :, :h, :w] + 1) / 2)
        assert abs(val[i].item() - o) <= VAL_TOL, (i, val[i].item(), o)


@pytest.mark.parametrize("fmt", ["minus_one_to_one", "zero_to_one"])
def test_ssim_explicit_tiles(fmt):
    """Overlapping tiles, tiles at the right and bottom edges, 11-px tiles, several tiles on one image in any order."""
    sizes = [(130, 131), (500, 333), (64, 48)]
    b, pred = _batch(sizes, 16, torch.float32, seed=9)
    if fmt == "zero_to_one":
        b = {**b, "patches": (b["patches"] + 1) / 2}
        pred = (pred + 1) / 2
    tiles = torch.tensor([
        [1, 0, 0, 128, 128], [1, 64, 64, 128, 128], [1, 100, 30, 200, 150],      # overlapping
        [0, 130 - 40, 131 - 50, 40, 50], [1, 500 - 11, 333 - 11, 11, 11],       # bottom-right corners
        [0, 0, 120, 130, 11], [0, 119, 0, 11, 131],                             # right / bottom edge strips, 11 px wide
        [2, 0, 0, 11, 11], [2, 5, 7, 11, 11], [2, 0, 0, 64, 48], [0, 3, 4, 11, 11],
        [1, 64, 64, 128, 128],                                                   # a duplicate tile: contributes twice
    ])
    val, _ = _check(b, pred, 16, tiles, fmt=fmt, tag=f"explicit tiles {fmt}")
    assert val[1].item() == val[-1].item()


def test_ssim_mask_with_holes_and_duplicates():
    """Masked tokens read 0 and get gradient 0; a cell claimed by two valid tokens reads the later one, and the earlier one gets 0."""
    b, pred = _batch([(130, 131), (512, 300)], 16, BF, seed=13)
    m = b["patch_mask"].clone()
    g = torch.Generator(device="cuda").manual_seed(5)
    m &= torch.rand(m.shape, generator=g, device="cuda") > 0.2
    m[:, 0] = True
    row, col = b["row_idx"].clone(), b["col_idx"].clone()
    row[1, 40], col[1, 40] = row[1, 3], col[1, 3]      # token 40 takes token 3's cell (40 > 3 wins)
    m[1, 3] = m[1, 40] = True
    hb = {**b, "patch_mask": m, "row_idx": row, "col_idx": col}
    _, grad = _check(hb, pred, 16, None, tag="holes + duplicate cell")
    assert bool((grad[~m] == 0).all())
    assert bool((grad[1, 3] == 0).all()) and bool((grad[1, 40] != 0).any())


def test_ssim_bit_identical_runs_and_alone_vs_batch():
    import vitok_b200 as vb
    b, pred = _batch(SIZES, 16, BF, seed=21)
    gout = torch.randn(len(SIZES), generator=torch.Generator(device="cuda").manual_seed(2), device="cuda")

    def run(bb, pp, go):
        p = pp.clone().requires_grad_(True)
        v = vb.ssim(p, bb, 16)
        (v * go).sum().backward()
        return v.detach(), p.grad
    v0, g0 = run(b, pred, gout)
    v1, g1 = run(b, pred, gout)
    assert torch.equal(v0, v1) and torch.equal(g0, g1)
    for k in (0, 3, 5):
        alone = {key: (val[k:k + 1] if torch.is_tensor(val) and val.ndim >= 1 else val) for key, val in b.items()}
        va, ga = run(alone, pred[k:k + 1], gout[k:k + 1])
        assert torch.equal(va[0], v0[k]), k
        assert torch.equal(ga[0], g0[k]), k


def test_ssim_no_grad_and_detached():
    import vitok_b200 as vb
    b, pred = _batch([(130, 131)], 16, BF, seed=4)
    p = pred.clone().requires_grad_(True)
    with torch.no_grad():
        v = vb.ssim(p, b)
    assert v.grad_fn is None and not v.requires_grad
    v2 = vb.ssim(pred, b)          # pred without grad: no graph either
    assert v2.grad_fn is None and torch.equal(v, v2)


def test_ssim_errors():
    import vitok_b200 as vb
    b, pred = _batch([(130, 131), (64, 64)], 16, BF, seed=6)
    with pytest.raises(ValueError, match="at least 11"):
        vb.ssim(pred, b, tiles=torch.tensor([[0, 0, 0, 10, 40]]))
    with pytest.raises(ValueError, match="inside"):
        vb.ssim(pred, b, tiles=torch.tensor([[1, 60, 0, 11, 11]]))
    with pytest.raises(ValueError, match="inside"):
        vb.ssim(pred, b, tiles=torch.tensor([[0, -1, 0, 11, 11]]))
    with pytest.raises(ValueError, match="image"):
        vb.ssim(pred, b, tiles=torch.tensor([[2, 0, 0, 11, 11]]))
    with pytest.raises(ValueError, match="patch"):
        vb.ssim(pred, b, patch=32)
    with pytest.raises(ValueError, match="current_format"):
        vb.ssim(pred, b, current_format="0_255")
    with pytest.raises(ValueError, match="requires grad"):
        vb.ssim(pred, {**b, "patches": b["patches"].float().requires_grad_(True)})
    with pytest.raises(RuntimeError, match="CUDA"):
        vb.ssim(pred.cpu(), {k: v.cpu() for k, v in b.items()})


# ---------------------------------------------------------------------------------------------------------------------------
# the SSIM term in a training step
# ---------------------------------------------------------------------------------------------------------------------------
SMALL = "w128_d2_h2-w256_d3_h2/1x16x16"


def _cos(a, b):
    return F.cosine_similarity(a.float().cpu().flatten(), b.float().cpu().flatten(), dim=0).item()


def _rel(got, ref):
    got, ref = got.detach().float().cpu(), ref.detach().float().cpu()
    return (torch.linalg.norm(got - ref) / torch.linalg.norm(ref).clamp_min(1e-30)).item()


@pytest.mark.parametrize("packed", [False, True], ids=["padded", "packed"])
def test_training_step_with_ssim_vs_oracle(packed):
    """loss = charbonnier + 0.5 (1 - ssim).mean() on a masked ragged batch: parameter gradients against the fp32 oracle's autograd
    (forward of oracle.ae_oracle plus the same SSIM on a differentiable canvas), within the gates of the Charbonnier-only oracle
    tests: cosine >= 0.995, worst rel-Fro <= 8e-2."""
    import vitok_b200 as vb
    cfg = vb.decode_variant(SMALL)
    sd = make_state_dict(cfg, seed=1, stress=True)
    imgs = synth_images([(128, 128), (96, 64), (128, 112), (64, 128)], seed=11)
    batch = {k: torch.from_numpy(np.asarray(v)) for k, v in pp_oracle.collate([pp_oracle.patchify(i, 16, 64) for i in imgs]).items()}
    cb = {k: (v.cuda().to(BF) if v.dtype == torch.float32 else v.cuda()) for k, v in batch.items()}
    model = vb.AE(**cfg, attn_backend="sdpa").train()
    model.load_state_dict(sd, strict=True)
    model = model.to("cuda", BF)
    model.train_token_packing = packed
    out = model(cb)
    s = vb.ssim(out["patches"], cb)
    loss = vb.charbonnier_loss(out["patches"], cb["patches"], cb["patch_mask"]) + 0.5 * (1 - s).mean()
    loss.backward()
    grads = {n: p.grad for n, p in model.named_parameters()}

    params = {k: v.to(BF).float().clone().requires_grad_(True) for k, v in sd.items()}
    tb = dict(batch)
    tb["patches"] = batch["patches"].to(BF).float()
    enc = ae_oracle.encode(params, tb, cfg["encoder_heads"], attn_backend="sdpa")
    dec = ae_oracle.decode(params, enc, cfg["decoder_heads"], attn_backend="sdpa")
    B = len(imgs)
    tiles = torch.stack([torch.arange(B), torch.zeros(B, dtype=torch.int64), torch.zeros(B, dtype=torch.int64),
                         batch["orig_height"], batch["orig_width"]], 1)
    s_ref = _ssim_ref(dec["patches"].double(), tb["patches"], tb, 16, tiles).float()
    ref_loss = ae_oracle.charbonnier_loss(dec["patches"], tb["patches"], tb["patch_mask"]) + 0.5 * (1 - s_ref).mean()
    ref_loss.backward()
    assert abs(loss.item() - ref_loss.item()) <= 5e-3 * abs(ref_loss.item()), (loss.item(), ref_loss.item())
    worst = ("", 0.0)
    for name, g in grads.items():
        assert torch.isfinite(g).all(), name
        r = _rel(g, params[name].grad)
        assert _cos(g, params[name].grad) >= 0.995, (name, r)
        worst = max(worst, (name, r), key=lambda t: t[1])
    print(f"[parity] train step + ssim ({'packed' if packed else 'padded'}) vs oracle: loss {loss.item():.6f} / {ref_loss.item():.6f}, "
          f"ssim {s.mean().item():.5f} / {s_ref.mean().item():.5f}, worst rel-Fro {worst[1]:.3e} at {worst[0]}")
    assert worst[1] <= 8e-2, worst
