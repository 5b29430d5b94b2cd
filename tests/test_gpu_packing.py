"""GPU parity: NaFlex token packing (masked batches run on their valid tokens only).

The reference masks padded keys inside SDPA and still pushes every padded token through every GEMM
(vitok/models/ae.py:173-187, attention.py:69-73).  Our packed path must give the same result on the valid tokens:
  * the index plan is bit-exact vs the numpy oracle (oracle/pp_oracle.py: pack_plan);
  * gather / scatter are bit-exact copies;
  * every image of a masked ragged batch equals, bit for bit on its valid tokens, the same image run alone without padding
    -- every per-row kernel sees the same row and attention sees the same key tiles;
  * arbitrary (non-prefix) masks agree with the fp32 oracle within the bf16 tolerance of SURVEY.md section 8c;
  * BASELINE.json configs[2] (350M-f16x16, 64 mixed-aspect images of 128-512 px, max_tokens 1024): every image encoded
    and decoded inside the ragged batch equals the same image run alone without padding.
"""
import numpy as np
import pytest
import torch

from _util import report
from oracle import ae_oracle, pp_oracle
from oracle.weights import make_state_dict, synth_images

pytestmark = pytest.mark.gpu

D64 = "w128_d2_h2-w256_d3_h4/1x16x16"   # head_dim 64 on both sides -> both halves use the packed attention kernel


def _masks():
    g = torch.Generator().manual_seed(3)
    out = []
    m = torch.zeros(5, 300, dtype=torch.bool)
    for b, n in enumerate([300, 1, 128, 129, 0]):
        m[b, :n] = True
    out.append(m)                                              # prefix masks incl. an empty image and tile edges
    out.append(torch.rand(7, 257, generator=g) > 0.4)          # arbitrary masks
    out.append(torch.ones(3, 64, dtype=torch.bool))            # nothing masked
    big = torch.rand(1500, 40, generator=g) > 0.5              # more images than one scan block (1024)
    out.append(big)
    return out


@pytest.mark.parametrize("ci", range(4))
@pytest.mark.parametrize("pad,qrows", [(16, 128), (16, 256), (128, 128)])
def test_pack_plan_bit_exact(ci, pad, qrows):
    from vitok_b200 import _lib
    mask = _masks()[ci]
    ref = pp_oracle.pack_plan(mask.numpy(), pad, qrows)
    got = {k: v.cpu().numpy() for k, v in _lib.pack_plan(mask.cuda(), pad, qrows).items()}
    total, ngrp = int(ref["cu"][-1]), int(ref["cuq"][-1])
    for k in ("n_valid", "rel", "cu", "cuq"):
        assert np.array_equal(got[k], ref[k]), k
    assert np.array_equal(got["src"][:total], ref["src"])
    assert np.array_equal(got["grp_img"][:ngrp], ref["grp_img"])
    assert (got["src"][total:] == -2).all() and (got["grp_img"][ngrp:] == -2).all()   # nothing written past the end
    # grp_order: a permutation of the groups with non-increasing key-tile counts (ties may come in any order)
    order = got["grp_order"][:ngrp]
    assert np.array_equal(np.sort(order), np.arange(ngrp)) and (got["grp_order"][ngrp:] == -2).all()
    kt = ((ref["n_valid"] + 127) // 128)[ref["grp_img"]]
    assert np.array_equal(kt[order], kt[ref["grp_order"]]) and (np.diff(kt[order]) <= 0).all()


@pytest.mark.parametrize("ci", range(3))
@pytest.mark.parametrize("width", [16, 776])
def test_pack_unpack_rows_bit_exact(ci, width):
    from vitok_b200 import _lib
    mask = _masks()[ci]
    B, N = mask.shape
    x = torch.randn(B, N, width, generator=torch.Generator().manual_seed(ci)).to(torch.bfloat16)
    plan = _lib.pack_plan(mask.cuda())
    packed = _lib.pack_rows(x.cuda(), plan)
    ref = pp_oracle.pack_plan(mask.numpy())
    total = int(ref["cu"][-1])
    want = torch.zeros(total, width, dtype=torch.bfloat16)
    sel = torch.from_numpy(ref["src"] >= 0)
    want[sel] = x.reshape(B * N, width)[torch.from_numpy(ref["src"][ref["src"] >= 0]).long()]
    assert torch.equal(packed[:total].cpu(), want)
    back = _lib.unpack_rows(packed, plan, B, N).cpu()
    assert torch.equal(back, torch.where(mask[..., None], x, torch.zeros_like(x)))


def _model(variant, seed=1, stress=True, backend="sdpa"):
    import vitok_b200 as vb
    cfg = vb.decode_variant(variant)
    sd = make_state_dict(ae_oracle.decode_variant(variant), seed=seed, stress=stress)
    m = vb.AE(**cfg, attn_backend=backend).eval()
    m.load_state_dict(sd, strict=True)
    return m.to(device="cuda", dtype=torch.bfloat16), cfg, sd


def _ragged_batch(sizes, patch, T, seed):
    b = pp_oracle.collate([pp_oracle.patchify(i, patch, T) for i in synth_images(sizes, seed=seed)])
    return {k: torch.from_numpy(np.asarray(v)) for k, v in b.items()}


def _cuda(batch):
    return {k: (v.cuda().to(torch.bfloat16) if v.dtype == torch.float32 else v.cuda()) for k, v in batch.items()}


def _alone(model, batch, i, n):
    """Image i of a batch run alone without padding: N = n (its valid tokens, a prefix), flash backend (no mask)."""
    one = {k: (v[i:i + 1, :n].contiguous() if v.dim() >= 2 else v[i:i + 1]) for k, v in batch.items()}
    backend = model.attn_backend
    model.attn_backend = "flash"
    try:
        enc = model.encode(one)
        return enc, model.decode(enc)
    finally:
        model.attn_backend = backend


@pytest.fixture
def no_splitk():
    """A lone image is a small batch: its residual GEMM would run split-K, whose fp32 sum of the two K-halves differs from the
    un-split kernel in the last bit (tests/test_gpu_gemm.py).  Bit-exact comparisons across batch sizes run without it."""
    from vitok_b200 import _lib
    _lib.set_flag("gemm_splitk", 0)
    yield
    _lib.set_flag("gemm_splitk", 1)


D128 = "w128_d2_h2-w256_d3_h2/1x16x16"  # decoder head_dim 128: attention groups of 256 query rows (two query tiles per CTA)


@pytest.mark.parametrize("variant", [D64, D128])
def test_packed_equals_single_images(variant, no_splitk):
    """Every image of the packed ragged batch == the same image alone (N = n_i, no mask), bit for bit on its valid tokens."""
    model, cfg, _ = _model(variant)
    batch = _ragged_batch([(256, 320), (96, 64), (50, 120), (16, 16), (320, 256), (130, 131)], 16, 320, seed=11)
    cb = _cuda(batch)
    valid = batch["patch_mask"]
    n = valid.sum(1).tolist()
    with torch.no_grad():
        e1 = model.encode(cb); d1 = model.decode(e1)
        n_packed = model.last_launch_count
        model.attn_backend = "flash"      # the same [B, N] batch without a mask
        model.decode(e1)
        n_dense = model.last_launch_count
        model.attn_backend = "sdpa"
        for i in range(len(n)):
            e0, d0 = _alone(model, cb, i, n[i])
            assert torch.equal(e1["z"][i, :n[i]], e0["z"][0]), f"image {i}: packed encode differs from the image alone"
            assert torch.equal(d1["patches"][i, :n[i]], d0["patches"][0]), f"image {i}: packed decode differs from the image alone"
    assert (e1["z"].cpu()[~valid] == 0).all() and (d1["patches"].cpu()[~valid] == 0).all(), "masked tokens must read as 0"
    assert n_packed == n_dense + 5   # plan (3) + gather + scatter


def test_general_mask_vs_oracle():
    model, cfg, sd = _model(D64)
    batch = _ragged_batch([(128, 128), (128, 128), (128, 128)], 16, 64, seed=2)
    g = torch.Generator().manual_seed(9)
    mask = torch.rand(3, 64, generator=g) > 0.35            # holes anywhere, not a prefix
    mask[:, 0] = True
    batch["patch_mask"] = mask
    with torch.no_grad():
        enc = model.encode(_cuda(batch))
        dec = model.decode(enc)
    e_o = ae_oracle.encode(sd, batch, cfg["encoder_heads"], attn_backend="sdpa")
    d_o = ae_oracle.decode(sd, e_o, cfg["decoder_heads"], attn_backend="sdpa")
    sdb = {k: v.to(torch.bfloat16) for k, v in sd.items()}
    bb = {k: (v.to(torch.bfloat16) if v.dtype == torch.float32 else v) for k, v in batch.items()}
    e_b = ae_oracle.encode(sdb, bb, cfg["encoder_heads"], attn_backend="sdpa")
    d_b = ae_oracle.decode(sdb, e_b, cfg["decoder_heads"], attn_backend="sdpa")
    own_z = (e_b["z"].float() - e_o["z"])[mask].abs().max().item()
    own_p = (d_b["patches"].float() - d_o["patches"])[mask].abs().max().item()
    ma_z, _ = report("general mask z", enc["z"].cpu().float()[mask], e_o["z"][mask])
    ma_p, _ = report("general mask patches", dec["patches"].cpu().float()[mask], d_o["patches"][mask])
    print(f"[parity] reference-bf16 own error: z {own_z:.3e} patches {own_p:.3e}")
    assert ma_z <= max(2 * own_z, 5e-2) and ma_p <= max(2 * own_p, 5e-2)


def c3_sizes(n=64, seed=1234):
    """BASELINE.json configs[2]: mixed-aspect sizes in [128, 512]^2 incl. non-multiples of 16; all fit 1024 tokens."""
    rng = np.random.RandomState(seed)
    return [(int(rng.randint(128, 513)), int(rng.randint(128, 513))) for _ in range(n)]


def test_c3_ragged_batch_equals_single_images():
    """350M-f16x16 on the c3 batch: image i inside the packed ragged batch == image i alone (N = n_i, no mask)."""
    import vitok_b200 as vb
    variant = "Ld4-Ld24/1x16x16"
    cfg = vb.decode_variant(variant)
    torch.manual_seed(0)
    model = vb.AE(**cfg, attn_backend="sdpa").eval().to(device="cuda", dtype=torch.bfloat16)
    sizes = c3_sizes()
    g = torch.Generator().manual_seed(7)
    imgs = [torch.rand(3, h, w, generator=g) * 2 - 1 for h, w in sizes]
    batch = vb.patchify_batch(imgs, 16, 1024, out_dtype=torch.bfloat16, device="cuda")
    with torch.no_grad():
        enc = model.encode(batch)
        dec = model.decode(enc)
    n = batch["patch_mask"].sum(1).tolist()
    assert sum(n) == sum(-(-h // 16) * -(-w // 16) for h, w in sizes)
    model.attn_backend = "flash"      # single, unpadded images: the reference's default no-mask path
    worst_z = worst_p = 0.0
    from vitok_b200 import _lib
    _lib.set_flag("gemm_splitk", 0)   # a lone image is a small batch: its residual GEMM would run split-K, whose fp32 sum of the two
    try:                              # K-halves differs from the un-split kernel in the last bit (tests/test_gpu_gemm.py)
        for i in (0, 5, 17, 40, 63, int(np.argmin(n)), int(np.argmax(n))):
            one = {k: (v[i:i + 1, :n[i]].contiguous() if v.dim() >= 2 else v[i:i + 1]) for k, v in batch.items()}
            with torch.no_grad():
                e1 = model.encode(one)
                d1 = model.decode(e1)
            worst_z = max(worst_z, (e1["z"][0].float() - enc["z"][i, :n[i]].float()).abs().max().item())
            worst_p = max(worst_p, (d1["patches"][0].float() - dec["patches"][i, :n[i]].float()).abs().max().item())
    finally:
        _lib.set_flag("gemm_splitk", 1)
    print(f"[parity] c3 ragged-vs-single: z max-abs {worst_z:.3e}, patches max-abs {worst_p:.3e} (tokens: {sum(n)} of {64 * 1024})")
    assert worst_z == 0.0 and worst_p == 0.0
    assert (enc["z"][~batch["patch_mask"]] == 0).all()


def test_fully_masked_batch_is_all_zero_and_does_not_hang(no_splitk):
    """Edge case: no valid token at all (packed row count 0 -> every kernel gets an empty problem from device memory)."""
    model, cfg, _ = _model(D64)
    batch = _ragged_batch([(64, 64), (32, 48)], 16, 64, seed=3)
    batch["patch_mask"] = torch.zeros_like(batch["patch_mask"])
    with torch.no_grad():
        enc = model.encode(_cuda(batch))
        dec = model.decode(enc)
    torch.cuda.synchronize()
    assert (enc["z"] == 0).all() and (dec["patches"] == 0).all()
    # and a batch where only ONE image has tokens
    batch = _ragged_batch([(64, 64), (32, 48), (128, 16)], 16, 64, seed=4)
    batch["patch_mask"][0] = False
    batch["patch_mask"][2] = False
    cb = _cuda(batch)
    valid = batch["patch_mask"]
    n1 = int(valid[1].sum())
    with torch.no_grad():
        d1 = model.decode(model.encode(cb))
        _, d0 = _alone(model, cb, 1, n1)
    assert torch.equal(d1["patches"][1, :n1], d0["patches"][0]) and (d1["patches"].cpu()[~valid] == 0).all()
