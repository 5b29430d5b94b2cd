"""GPU: the training step computes only the gradients autograd asks for.  Frozen parameters (requires_grad=False) get no gradient and
cost no weight-gradient GEMM; the backward pass stops where gradients stop; AE(encoder=False) trains on z and AE(decoder=False) returns
z with its graph.  Every gradient that is computed is the full step's (bit-identical for the GEMM-produced ones), or the oracle's under
torch autograd for the single-half models."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ae_oracle, pp_oracle
from oracle.make_golden import SMALL
from oracle.weights import make_state_dict, synth_images

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = [(128, 128), (96, 64), (128, 112), (64, 128)]
ENC_PREFIXES = ("patch_embed.", "to_code.", "encoder_blocks.")


def _rel(got, ref):
    got, ref = got.detach().float().cpu(), ref.detach().float().cpu()
    return (torch.linalg.norm(got - ref) / torch.linalg.norm(ref).clamp_min(1e-30)).item()


def _batch(sizes, patch, T, seed):
    b = pp_oracle.collate([pp_oracle.patchify(i, patch, T) for i in synth_images(sizes, seed=seed)])
    return {k: torch.from_numpy(np.asarray(v)) for k, v in b.items()}


def _cuda(batch):
    return {k: (v.cuda().to(BF) if v.dtype == torch.float32 else v.cuda()) for k, v in batch.items()}


def _holes(batch, seed=3):
    g = torch.Generator().manual_seed(seed)
    mask = batch["patch_mask"].clone()
    mask &= torch.rand(mask.shape, generator=g) > 0.3
    mask[:, 0] = True
    batch["patch_mask"] = mask
    return batch


def _is_enc(name):
    return name.startswith(ENC_PREFIXES)


def _model(cfg, sd, **kw):
    import vitok_b200 as vb
    m = vb.AE(**cfg, **kw).train()
    m.load_state_dict({k: v for k, v in sd.items() if k in dict(m.named_parameters())}, strict=True)
    return m.to("cuda", BF)


def _step(m, cb, seed=9):
    """One step: (loss, output, {name: grad or None}, bytes held after the forward)."""
    import vitok_b200 as vb
    for p in m.parameters():
        p.grad = None
    torch.manual_seed(seed)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    out = m(cb)
    held = torch.cuda.memory_allocated() - base
    loss = vb.charbonnier_loss(out["patches"], cb["patches"], cb["patch_mask"], eps=1e-3)
    loss.backward()
    return loss.detach(), out["patches"].detach(), {n: (None if p.grad is None else p.grad.clone()) for n, p in m.named_parameters()}, held


def _same_grad(name, a, b):
    """GEMM-produced gradients bit-identical; vector gradients (fp32 atomic sums, then one bf16 rounding) within one bf16 ulp, as in
    test_gpu_train.py::test_activation_checkpointing_is_bit_identical."""
    assert a is not None and b is not None, name
    if a.ndim >= 2:
        assert torch.equal(a, b), name
    else:
        fa, fb = a.float(), b.float()
        tol = 2.0 ** -7 * torch.maximum(fa.abs(), fb.abs()) + 2.0 ** -8 * fa.abs().max()
        assert bool(((fa - fb).abs() <= tol).all()), (name, float((fa - fb).abs().max()))
        assert _rel(a, b) <= 2e-3, (name, _rel(a, b))


def _block_saved_bytes(cfg, side, M):
    """x, h, zraw, qkv, a2, lse and y of one block (vitok_b200/train.py: _block_forward)."""
    from vitok_b200.models.ae import _ffn_hidden
    D, heads = (cfg["encoder_width"], cfg["encoder_heads"]) if side == 0 else (cfg["decoder_width"], cfg["decoder_heads"])
    Hf = _ffn_hidden(D, cfg["mlp_factor"])
    qp = (3 * D + 255) // 256 * 256
    kp = (D + Hf + 63) // 64 * 64
    return 2 * M * (D + D + (qp + 2 * Hf) + 3 * D + kp + D) + 4 * M * heads


def test_frozen_encoder_matches_full_step():
    import vitok_b200 as vb
    cfg = vb.decode_variant(SMALL)
    sd = make_state_dict(cfg, seed=1, stress=True)
    cb = _cuda(_batch(SIZES, 16, 64, seed=11))
    full = _model(cfg, sd, attn_backend="sdpa", drop_path_rate=0.3)
    _step(full, cb)                                    # warm-up (library load, tensor-map caches)
    loss0, out0, g0, held0 = _step(full, cb)
    frozen = _model(cfg, sd, attn_backend="sdpa", drop_path_rate=0.3)
    for mod in (frozen.patch_embed, frozen.encoder_blocks, frozen.to_code):
        mod.requires_grad_(False)
    loss1, out1, g1, held1 = _step(frozen, cb)
    assert torch.equal(out0, out1)
    assert abs(float(loss0) - float(loss1)) <= 1e-6 * abs(float(loss0))
    for n in g0:
        if _is_enc(n):
            assert g1[n] is None, n
        else:
            _same_grad(n, g0[n], g1[n])
    B, N = cb["patch_mask"].shape
    enc_bytes = cfg["encoder_depth"] * _block_saved_bytes(cfg, 0, B * N)
    print(f"[frozen] held after forward: full {held0 / 2**20:.2f} MiB, frozen encoder {held1 / 2**20:.2f} MiB, "
          f"encoder blocks' activations {enc_bytes / 2**20:.2f} MiB")
    assert held0 - held1 >= 0.8 * enc_bytes


@pytest.mark.parametrize("packing", [False, True])
@pytest.mark.parametrize("ck", [0, 1])
def test_mixed_frozen_subset_matches_full_step(packing, ck):
    import vitok_b200 as vb
    cfg = vb.decode_variant(SMALL)
    sd = make_state_dict(cfg, seed=1, stress=True)
    cb = _cuda(_holes(_batch(SIZES, 16, 64, seed=13)))

    def make():
        m = _model(cfg, sd, attn_backend="sdpa", drop_path_rate=0.3, checkpoint=ck)
        m.train_token_packing = packing
        return m

    loss0, out0, g0, _ = _step(make(), cb)
    m = make()
    m.decoder_blocks[0].requires_grad_(False)
    for n, p in m.named_parameters():
        if "norm" in n:
            p.requires_grad_(False)
    m.patch_embed.requires_grad_(False)
    m.to_code.bias.requires_grad_(False)
    frozen = {n for n, p in m.named_parameters() if not p.requires_grad}
    loss1, out1, g1, _ = _step(m, cb)
    assert torch.equal(out0, out1)
    assert abs(float(loss0) - float(loss1)) <= 1e-6 * abs(float(loss0))
    for n in g0:
        if n in frozen:
            assert g1[n] is None, n
        else:
            _same_grad(n, g0[n], g1[n])


def _halves(cfg, sd, **kw):
    enc = _model(cfg, sd, encoder=True, decoder=False, **kw)
    dec = _model(cfg, sd, encoder=False, decoder=True, **kw)
    return enc, dec


def _oracle_sd(sd):
    return {k: v.to(BF).float() for k, v in sd.items()}


@pytest.mark.parametrize("backend,packing", [("sdpa", False), ("sdpa", True), ("flash", False)])
def test_decoder_only_model(backend, packing):
    import vitok_b200 as vb
    cfg = vb.decode_variant(SMALL)
    sd = make_state_dict(cfg, seed=1, stress=True)
    batch = _batch(SIZES if backend == "sdpa" else [(128, 128)] * 4, 16, 64, seed=11)
    cb = _cuda(batch)
    full = _model(cfg, sd, attn_backend=backend)
    full.train_token_packing = packing
    _, _, g_full, _ = _step(full, cb)
    enc, dec = _halves(cfg, sd, attn_backend=backend)
    enc.train_token_packing = dec.train_token_packing = packing
    z = enc(cb)["z"].detach()                        # the training-forward kernels of the full step
    # decoder gradients equal the full step's
    _, _, g_dec, _ = _step(dec, dict(cb, z=z))
    for n, g in g_dec.items():
        _same_grad(n, g_full[n], g)
    # vs the oracle under autograd, z requiring grad
    for p in dec.parameters():
        p.grad = None
    zg = z.clone().requires_grad_(True)
    out = dec(dict(cb, z=zg))
    assert set(out) == {"patch_mask", "row_idx", "col_idx", "orig_height", "orig_width", "patches"}
    loss = vb.charbonnier_loss(out["patches"], cb["patches"], cb["patch_mask"], eps=1e-3)
    loss.backward()
    assert zg.grad is not None and zg.grad.shape == z.shape
    sd_b = _oracle_sd(sd)
    zc = z.float().cpu().requires_grad_(True)
    ref_sd = {k: v.clone().requires_grad_(True) for k, v in sd_b.items() if not _is_enc(k)}
    mask = batch["patch_mask"]
    d_o = ae_oracle.decode(ref_sd, {"z": zc, "row_idx": batch["row_idx"], "col_idx": batch["col_idx"], "patch_mask": mask},
                           cfg["decoder_heads"], attn_backend=backend)
    ref_loss = ae_oracle.charbonnier_loss(d_o["patches"], batch["patches"].to(BF).float(), mask, 1e-3)
    ref_loss.backward()
    _vs_oracle(loss, ref_loss, {**{n: p.grad for n, p in dec.named_parameters()}, "z": zg.grad},
               {**{n: t.grad for n, t in ref_sd.items()}, "z": zc.grad}, "decoder-only")


def _vs_oracle(loss, ref_loss, got, ref, tag, loss_scale=None):
    """Loss within 5e-3 of ``loss_scale`` (default: |ref_loss|); every gradient cosine >= 0.995 and rel-Fro <= 8e-2."""
    scale = abs(float(ref_loss)) if loss_scale is None else float(loss_scale)
    assert abs(float(loss) - float(ref_loss)) <= 5e-3 * scale, (float(loss), float(ref_loss), scale)
    worst = ("", 0.0)
    for n, g in got.items():
        assert g is not None and torch.isfinite(g).all(), n
        r = _rel(g, ref[n])
        cos = F.cosine_similarity(g.float().cpu().flatten(), ref[n].float().flatten(), dim=0).item()
        assert cos >= 0.995, (n, cos, r)
        worst = max(worst, (n, r), key=lambda t: t[1])
    print(f"[frozen] {tag}: loss {float(loss):.6f} / oracle {float(ref_loss):.6f}, worst gradient rel-Fro {worst[1]:.3e} at {worst[0]}")
    assert worst[1] <= 8e-2


@pytest.mark.parametrize("packing", [False, True])
def test_encoder_only_model(packing):
    import vitok_b200 as vb
    cfg = vb.decode_variant(SMALL)
    sd = make_state_dict(cfg, seed=1, stress=True)
    batch = _holes(_batch(SIZES, 16, 64, seed=13))
    cb = _cuda(batch)
    enc = _model(cfg, sd, attn_backend="sdpa", encoder=True, decoder=False)
    enc.train_token_packing = packing
    cb["patches"] = cb["patches"].clone().requires_grad_(True)
    out = enc(cb)
    assert set(out) == {"patch_mask", "row_idx", "col_idx", "orig_height", "orig_width", "z"} and out["z"].requires_grad
    mask = batch["patch_mask"]
    r = (torch.randn(*out["z"].shape, generator=torch.Generator().manual_seed(5)) * mask[:, :, None]).cuda()
    loss = (out["z"].float() * r).sum()
    loss.backward()
    if packing:                                      # masked tokens come back as 0
        assert float(out["z"][~mask.cuda()].abs().max()) == 0.0
    sd_b = _oracle_sd(sd)
    ref_sd = {k: v.clone().requires_grad_(True) for k, v in sd_b.items() if _is_enc(k)}
    pc = batch["patches"].to(BF).float().requires_grad_(True)
    e_o = ae_oracle.encode(ref_sd, dict(batch, patches=pc), cfg["encoder_heads"], attn_backend="sdpa")
    ref_loss = (e_o["z"] * r.cpu()).sum()
    ref_loss.backward()
    # sum(z * r) cancels (z is LayerNorm-ed, r has mean 0): the bf16 rounding of z shows against the size of its terms, not of the sum
    _vs_oracle(loss, ref_loss, {**{n: p.grad for n, p in enc.named_parameters()}, "patches": cb["patches"].grad},
               {**{n: t.grad for n, t in ref_sd.items()}, "patches": pc.grad}, f"encoder-only packing={packing}",
               loss_scale=(e_o["z"] * r.cpu()).abs().sum())


def test_adamw_steps_with_frozen_encoder():
    """Three FusedAdamW steps with the encoder frozen vs the full model whose encoder gradients are dropped before each step.  The
    frozen encoder stays bitwise unchanged and gets no optimizer state.  The decoder matches: its matrix gradients are bit-identical
    (see above), its vector gradients are fp32 atomic sums whose order varies from run to run, so the parameters are compared to
    within the bf16 rounding such a difference can flip."""
    import vitok_b200 as vb
    cfg = vb.decode_variant(SMALL)
    sd = make_state_dict(cfg, seed=1, stress=True)
    cb = _cuda(_batch(SIZES, 16, 64, seed=11))
    a = _model(cfg, sd, attn_backend="sdpa")
    b = _model(cfg, sd, attn_backend="sdpa")
    for mod in (a.patch_embed, a.encoder_blocks, a.to_code):
        mod.requires_grad_(False)
    enc0 = {n: p.detach().clone() for n, p in a.named_parameters() if _is_enc(n)}
    oa = vb.FusedAdamW(a.parameters(), lr=1e-3, betas=(0.9, 0.99), weight_decay=0.01)
    ob = vb.FusedAdamW(b.parameters(), lr=1e-3, betas=(0.9, 0.99), weight_decay=0.01)
    for _ in range(3):
        _step(a, cb)
        _step(b, cb)
        for n, p in b.named_parameters():
            if _is_enc(n):
                p.grad = None
        oa.step()
        ob.step()
    pb = dict(b.named_parameters())
    exact = 0
    for n, p in a.named_parameters():
        if _is_enc(n):
            assert torch.equal(p.detach(), enc0[n]) and not oa.state[p], n
            assert torch.equal(pb[n].detach(), enc0[n]), n
        else:
            exact += int(torch.equal(p.detach(), pb[n].detach()))
            d = (p.detach().float() - pb[n].detach().float()).abs().max()
            assert float(d) <= 2.0 ** -7 * float(p.detach().float().abs().max()), (n, float(d))
            assert _rel(p, pb[n]) <= 1e-3, n
    n_dec = sum(1 for n, _ in a.named_parameters() if not _is_enc(n))
    print(f"[frozen] after 3 AdamW steps: {exact} of {n_dec} decoder parameters bit-identical to the full model's")


def test_unchanged_paths():
    import vitok_b200 as vb
    cfg = vb.decode_variant(SMALL)
    sd = make_state_dict(cfg, seed=1, stress=True)
    cb = _cuda(_batch(SIZES, 16, 64, seed=11))
    m = _model(cfg, sd, attn_backend="sdpa")
    m.encoder_blocks.requires_grad_(False)
    with pytest.raises(NotImplementedError):
        m.encode(cb)
    with pytest.raises(NotImplementedError):
        m.decode({**cb, "z": torch.zeros(*cb["patches"].shape[:2], cfg["channels_per_token"], dtype=BF, device="cuda")})
    m.requires_grad_(False)                          # nothing trainable, no input requiring grad: the inference path
    out = m(cb)["patches"]
    assert out.grad_fn is None and not out.requires_grad
    with torch.no_grad():
        ref = m.eval()(cb)["patches"]
    assert torch.equal(out, ref)


def test_grad_sync_frozen_encoder_two_ranks():
    """tools/ddp_train_check.py --frozen-encoder under torchrun: with enable_grad_sync, ranks hold identical decoder gradients equal to
    the mean of the local ones, and the frozen encoder has no gradient and stays identical across ranks."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29547", os.path.join(ROOT, "tools", "ddp_train_check.py"), "--frozen-encoder"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stderr[-3000:]
    assert "grad_sync frozen encoder OK" in r.stdout
