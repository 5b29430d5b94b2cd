"""GPU parity of the training step (BASELINE config 5 path; scripts/train_vae.py:304-320,371-372): every backward
kernel against torch autograd of the CPU oracle's restatement of the same op, then the whole step (loss + every
parameter gradient) against the oracle, then a few optimizer steps."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from _util import bf16_randn, report
from oracle import ae_oracle, pp_oracle
from oracle.make_golden import SMALL
from oracle.weights import make_state_dict, synth_images

pytestmark = pytest.mark.gpu
BF = torch.bfloat16


@pytest.fixture(scope="module")
def L():
    from vitok_b200 import _lib
    _lib.load()
    return _lib


def _rel(got, ref):
    got, ref = got.detach().float().cpu(), ref.detach().float().cpu()
    return (torch.linalg.norm(got - ref) / torch.linalg.norm(ref).clamp_min(1e-30)).item()


def test_colsum_and_resid_bwd(L):
    M, D = 777, 384
    dx, y = bf16_randn(M, D, seed=51), bf16_randn(M, D, seed=52)
    gamma = bf16_randn(D, seed=53, scale=0.5)
    out = torch.zeros(D, dtype=torch.float32, device="cuda")
    L.check(L.load().vtk_colsum(dx.data_ptr(), D, out.data_ptr(), M, D, L.stream_ptr()))
    report("colsum", out, dx.float().sum(0), rel_fro=1e-5)
    dy = torch.empty_like(dx)
    dg = torch.zeros(D, dtype=torch.float32, device="cuda")
    L.check(L.load().vtk_resid_bwd_dp(dx.data_ptr(), y.data_ptr(), gamma.data_ptr(), dy.data_ptr(), dg.data_ptr(), M, D, None, 0, 1.0,
                                      L.stream_ptr()))   # keep = NULL: no stochastic depth
    report("resid_bwd dgamma", dg, (dx.float() * y.float()).sum(0), rel_fro=1e-5)
    assert torch.equal(dy, (dx.float() * gamma.float()).to(BF))
    # forward counterpart: same rounding as the fused GEMM epilogue
    x = bf16_randn(M, D, seed=54)
    o = torch.empty_like(x)
    L.check(L.load().vtk_resid_fwd_dp(x.data_ptr(), y.data_ptr(), gamma.data_ptr(), o.data_ptr(), M, D, None, 0, 1.0, L.stream_ptr()))
    assert torch.equal(o, x + (y * gamma))


@pytest.mark.parametrize("M,heads,d", [(200, 2, 64), (96, 3, 128), (203, 4, 64), (97, 4, 128), (1001, 16, 64), (333, 24, 128)])
def test_qk_norm_rope_fwd_bwd(L, M, heads, d):
    D = heads * d
    z = bf16_randn(M, 3 * D, seed=55)
    g = torch.Generator().manual_seed(56)
    wq = (torch.rand(d, generator=g) + 0.5).to(BF).cuda()
    wk = (torch.rand(d, generator=g) + 0.5).to(BF).cuda()
    row, col = (torch.arange(M) // 9).cuda(), (torch.arange(M) % 9).cuda()
    table = L.rope_table(row, col, ae_oracle.rope_inv_freq(d).cuda(), d)
    qkv = torch.empty(M, 3 * D, dtype=BF, device="cuda")
    L.check(L.load().vtk_qk_norm_rope_fwd(z.data_ptr(), 3 * D, wq.data_ptr(), wk.data_ptr(), table.data_ptr(), qkv.data_ptr(), 3 * D,
                                          M, heads, d, 1e-6, L.stream_ptr()))
    # oracle in fp32 with autograd
    zc = z.float().cpu().reshape(1, M, 3, heads, d).requires_grad_(True)
    wqc, wkc = wq.float().cpu().requires_grad_(True), wk.float().cpu().requires_grad_(True)
    cos, sin = ae_oracle.rope_cos_sin(row.cpu()[None], col.cpu()[None], d)
    q = ae_oracle.apply_rope(ae_oracle.rms_norm(zc[:, :, 0], wqc), cos, sin)
    k = ae_oracle.apply_rope(ae_oracle.rms_norm(zc[:, :, 1], wkc), cos, sin)
    got = qkv.cpu().reshape(1, M, 3, heads, d)
    report("qk fwd q", got[:, :, 0], q, max_abs=6e-2, rel_fro=6e-3)
    report("qk fwd k", got[:, :, 1], k, max_abs=6e-2, rel_fro=6e-3)
    assert torch.equal(got[:, :, 2], z.cpu().reshape(1, M, 3, heads, d)[:, :, 2])
    dq, dk = bf16_randn(1, M, heads, d, seed=57).cpu().float(), bf16_randn(1, M, heads, d, seed=58).cpu().float()
    (q * dq).sum().backward(retain_graph=True)
    (k * dk).sum().backward()
    dz = torch.zeros(M, 3 * D, dtype=BF, device="cuda")
    dz.view(M, 3, heads, d)[:, 0] = dq[0].to(BF).cuda()
    dz.view(M, 3, heads, d)[:, 1] = dk[0].to(BF).cuda()
    dw = torch.zeros(2, d, dtype=torch.float32, device="cuda")
    L.check(L.load().vtk_qk_norm_rope_bwd(dz.data_ptr(), 3 * D, z.data_ptr(), 3 * D, wq.data_ptr(), wk.data_ptr(), table.data_ptr(),
                                          dw.data_ptr(), M, heads, d, 1e-6, L.stream_ptr()))
    gz = zc.grad[0]
    report("qk bwd dq_raw", dz.view(M, 3, heads, d)[:, 0], gz[:, 0], rel_fro=1.5e-2)
    report("qk bwd dk_raw", dz.view(M, 3, heads, d)[:, 1], gz[:, 1], rel_fro=1.5e-2)
    report("qk bwd dwq", dw[0], wqc.grad, rel_fro=1.5e-2)
    report("qk bwd dwk", dw[1], wkc.grad, rel_fro=1.5e-2)


def test_swiglu_fwd_bwd(L):
    from vitok_b200.models.ae import pack_w_in
    M, Hf, qp = 300, 336, 256
    u = bf16_randn(M, 2 * Hf, seed=59)                      # reference order [value | gate]
    # packed order: 16-column groups (value16 | gate16) after qp pad columns
    zraw = torch.zeros(M, qp + 2 * Hf, dtype=BF, device="cuda")
    zraw[:, qp:] = u.view(M, 2, Hf // 16, 16).permute(0, 2, 1, 3).reshape(M, 2 * Hf)
    act = torch.empty(M, Hf, dtype=BF, device="cuda")
    L.check(L.load().vtk_swiglu_fwd(zraw.data_ptr(), qp + 2 * Hf, qp, act.data_ptr(), Hf, M, Hf, 0, L.stream_ptr()))
    uc = u.float().cpu().requires_grad_(True)
    val, gate = uc.chunk(2, dim=-1)
    ref = F.silu(gate) * val
    report("swiglu fwd", act, ref, max_abs=6e-2, rel_fro=5e-3)
    dact = bf16_randn(M, Hf, seed=60)
    (ref * dact.float().cpu()).sum().backward()
    dz = torch.zeros_like(zraw)
    L.check(L.load().vtk_swiglu_bwd(dact.data_ptr(), Hf, zraw.data_ptr(), qp + 2 * Hf, qp, dz.data_ptr(), qp + 2 * Hf, M, Hf, 0, L.stream_ptr()))
    du = dz[:, qp:].view(M, Hf // 16, 2, 16).permute(0, 2, 1, 3).reshape(M, 2 * Hf)
    report("swiglu bwd", du, uc.grad, rel_fro=6e-3)
    # layout 1: fc1's own column order [value Hf | gate Hf] (training path, no weight repack) -- same numbers
    zplain = torch.zeros(M, qp + 2 * Hf, dtype=BF, device="cuda")
    zplain[:, qp:] = u
    act1 = torch.empty(M, Hf, dtype=BF, device="cuda")
    L.check(L.load().vtk_swiglu_fwd(zplain.data_ptr(), qp + 2 * Hf, qp, act1.data_ptr(), Hf, M, Hf, 1, L.stream_ptr()))
    assert torch.equal(act1, act)
    dz1 = torch.zeros_like(zplain)
    L.check(L.load().vtk_swiglu_bwd(dact.data_ptr(), Hf, zplain.data_ptr(), qp + 2 * Hf, qp, dz1.data_ptr(), qp + 2 * Hf, M, Hf, 1, L.stream_ptr()))
    assert torch.equal(dz1[:, qp:], du)


@pytest.mark.parametrize("M,D", [(100, 256), (64, 1024), (40, 3072), (4099, 3072), (77, 4096), (50, 768), (1500, 1024)])
def test_rmsnorm_bwd(L, M, D):
    x, dh, dres = bf16_randn(M, D, seed=61, scale=2.0), bf16_randn(M, D, seed=62), bf16_randn(M, D, seed=63)
    w = (torch.rand(D, generator=torch.Generator().manual_seed(64)) + 0.5).to(BF).cuda()
    xc, wc = x.float().cpu().requires_grad_(True), w.float().cpu().requires_grad_(True)
    (ae_oracle.rms_norm(xc, wc) * dh.float().cpu()).sum().backward()
    dx = torch.empty_like(x)
    dw = torch.zeros(D, dtype=torch.float32, device="cuda")
    L.check(L.load().vtk_rmsnorm_bwd(x.data_ptr(), dh.data_ptr(), w.data_ptr(), dres.data_ptr(), dx.data_ptr(), dw.data_ptr(), M, D, 1e-6,
                                     L.stream_ptr()))
    report(f"rmsnorm bwd dx D={D}", dx, xc.grad + dres.float().cpu(), rel_fro=5e-3)
    report(f"rmsnorm bwd dw D={D}", dw, wc.grad, rel_fro=1e-4)


@pytest.mark.parametrize("C", [16, 64, 256])
def test_layernorm_fwd_bwd(L, C):
    M = 130
    zl, dz = bf16_randn(M, C, seed=65, scale=2.0), bf16_randn(M, C, seed=66)
    out = torch.empty_like(zl)
    L.check(L.load().vtk_layernorm_fwd(zl.data_ptr(), out.data_ptr(), M, C, 1e-6, L.stream_ptr()))
    zc = zl.float().cpu().requires_grad_(True)
    ref = ae_oracle.layer_norm_noaffine(zc)
    report(f"ln fwd C={C}", out, ref, max_abs=3e-2, rel_fro=4e-3)
    (ref * dz.float().cpu()).sum().backward()
    dx = torch.empty_like(zl)
    L.check(L.load().vtk_layernorm_bwd(zl.data_ptr(), dz.data_ptr(), dx.data_ptr(), M, C, 1e-6, L.stream_ptr()))
    report(f"ln bwd C={C}", dx, zc.grad, rel_fro=6e-3)


@pytest.mark.parametrize("masked", [False, True])
def test_charbonnier(L, masked):
    import vitok_b200 as vb
    B, N, P = 3, 64, 768
    pred = bf16_randn(B, N, P, seed=67).requires_grad_(True)
    target = bf16_randn(B, N, P, seed=68)
    mask = None
    if masked:
        mask = torch.zeros(B, N, dtype=torch.bool)
        mask[0, :64], mask[1, :10] = True, True            # image 2 has no valid token (clamp_min(1) path)
    loss = vb.charbonnier_loss(pred, target, mask.cuda() if masked else None, eps=1e-3)
    loss.backward()
    pc = pred.detach().cpu().float().requires_grad_(True)
    ref = ae_oracle.charbonnier_loss(pc, target.cpu().float(), mask, 1e-3)
    ref.backward()
    assert abs(loss.item() - ref.item()) <= 1e-5 * max(1.0, abs(ref.item()))
    report(f"charbonnier dpred masked={masked}", pred.grad, pc.grad, rel_fro=4e-3)


def test_resid_drop_path_kernels(L):
    """vtk_resid_fwd_dp / vtk_resid_bwd_dp vs autograd of the oracle's drop_path (ae.py:15-30,65) with an explicit draw."""
    B, N, D, keep_prob = 5, 24, 384, 0.7
    M = B * N
    x, y = bf16_randn(M, D, seed=151), bf16_randn(M, D, seed=152)
    gamma = bf16_randn(D, seed=153, scale=0.5)
    keep = torch.tensor([1.0, 0.0, 1.0, 1.0, 0.0])
    o = torch.empty_like(x)
    L.check(L.load().vtk_resid_fwd_dp(x.data_ptr(), y.data_ptr(), gamma.data_ptr(), o.data_ptr(), M, D, keep.cuda().data_ptr(), N, keep_prob,
                                      L.stream_ptr()))
    comb = (y.cpu() * gamma.cpu()).reshape(B, N, D)                       # bf16, like the reference's LayerScale output
    ref = x.cpu().reshape(B, N, D) + ae_oracle.drop_path(comb, keep, keep_prob)
    assert torch.equal(o.cpu().reshape(B, N, D), ref)                     # same bf16 rounding points as the eager reference
    # backward: fp32 autograd of the same expression
    yc, gc = y.float().cpu().requires_grad_(True), gamma.float().cpu().requires_grad_(True)
    dx = bf16_randn(M, D, seed=154)
    (ae_oracle.drop_path((yc * gc).reshape(B, N, D), keep, keep_prob) * dx.float().cpu().reshape(B, N, D)).sum().backward()
    dy = torch.empty_like(x)
    dg = torch.zeros(D, dtype=torch.float32, device="cuda")
    L.check(L.load().vtk_resid_bwd_dp(dx.data_ptr(), y.data_ptr(), gamma.data_ptr(), dy.data_ptr(), dg.data_ptr(), M, D,
                                      keep.cuda().data_ptr(), N, keep_prob, L.stream_ptr()))
    report("resid_bwd_dp dy", dy, yc.grad, rel_fro=6e-3)
    report("resid_bwd_dp dgamma", dg, gc.grad, rel_fro=6e-3)
    assert float(dy.view(B, N, D)[1].abs().max()) == 0.0 and float(dy.view(B, N, D)[4].abs().max()) == 0.0   # dropped images: no gradient


def test_adamw_matches_torch(L):
    import vitok_b200 as vb
    torch.manual_seed(0)
    p0 = torch.randn(5000)
    ours = torch.nn.Parameter(p0.to(BF).cuda())
    ref = torch.nn.Parameter(p0.to(BF).float())             # torch AdamW on fp32 copies of the same bf16 values
    o1 = vb.FusedAdamW([ours], lr=1e-2, betas=(0.9, 0.99), weight_decay=0.05)
    o2 = torch.optim.AdamW([ref], lr=1e-2, betas=(0.9, 0.99), weight_decay=0.05)
    for s in range(5):
        g = torch.randn(5000, generator=torch.Generator().manual_seed(s)).to(BF)
        ours.grad, ref.grad = g.cuda(), g.float()
        o1.step(); o2.step()
    report("adamw 5 steps (bf16 param)", ours.data, ref.data.to(BF), max_abs=1.6e-2, rel_fro=2e-3)   # = bf16 rounding of the fp32 result
    report("adamw 5 steps (fp32 master)", o1.state[ours]["master"], ref.data, rel_fro=1e-6)
    report("adamw exp_avg_sq", o1.state[ours]["exp_avg_sq"], o2.state[ref]["exp_avg_sq"], rel_fro=1e-6)


@pytest.mark.parametrize("pdtype", [BF, torch.float32])
def test_adamw_small_lr_many_steps_vs_torch_fp32(L, pdtype):
    """The reference recipe (train_vae.py:200-208: lr 1e-4 ... 3e-4, fp32 parameters and moments).  With bf16 parameters and no
    master copy, an update below half a bf16 ulp is rounded away: weights of magnitude ~1 (all norm weights) would never move
    at lr 1e-4.  FusedAdamW keeps an fp32 master and fp32 moments: after 300 steps of a constant-sign gradient the bf16
    parameters have moved exactly as torch's fp32 AdamW moves them (also with beta2 = 0.999)."""
    import vitok_b200 as vb
    n = 4096 + 3                                                     # odd length: the scalar tail of the vector kernel
    p0 = torch.ones(n) + 0.25 * torch.randn(n, generator=torch.Generator().manual_seed(1))
    ours = torch.nn.Parameter(p0.to(pdtype).cuda())
    ref = torch.nn.Parameter(p0.to(pdtype).float().clone())           # (for fp32 the casts are no-ops: do not alias p0)
    o1 = vb.FusedAdamW([ours], lr=1e-4, betas=(0.9, 0.999), weight_decay=0.01)
    o2 = torch.optim.AdamW([ref], lr=1e-4, betas=(0.9, 0.999), weight_decay=0.01)
    gsign = torch.where(torch.arange(n) % 2 == 0, 1.0, -1.0)
    for s in range(300):
        g = (gsign * (1.0 + 0.1 * torch.randn(n, generator=torch.Generator().manual_seed(100 + s)))).to(BF)
        ours.grad, ref.grad = g.to(pdtype).cuda(), g.float()
        o1.step(); o2.step()
    moved = (ref.data - p0.to(pdtype).float()).abs()
    assert float(moved.min()) > 2e-2                                   # ~300 * 1e-4: several bf16 ulps at |w| ~ 1 (ulp 7.8e-3)
    master = o1.state[ours].get("master", ours.data)
    report(f"adamw 300 steps lr 1e-4 master ({pdtype})", master, ref.data, max_abs=2e-5, rel_fro=1e-5)
    if pdtype == BF:
        assert torch.equal(ours.data.cpu(), master.cpu().to(BF))       # the bf16 parameter is the rounded master
        assert float((ours.data.float().cpu() - p0.to(BF).float()).abs().min()) > 1e-2      # every bf16 weight moved


def test_linear2_and_dgrad_accumulate(L):
    """vtk_linear2_bf16 (out_proj(attn) + fc2(act) over two weight matrices, one accumulator) and the accumulating data-gradient
    GEMM: vs fp32 matmuls, for the pair-kernel shape (K0 % 64 == 0, large M) and for the two-GEMM fallback shapes."""
    for M, N, K0, K1 in [(1024, 1024, 1024, 2736), (2048, 3072, 3072, 8208), (300, 256, 256, 688), (96, 128, 128, 336), (512, 384, 72, 200)]:
        a = bf16_randn(M, K0 + K1 + 8, seed=160)[:, :K0 + K1]
        w0 = bf16_randn(N, K0, seed=161, scale=1 / math.sqrt(K0 + K1))
        w1 = bf16_randn(N, K1, seed=162, scale=1 / math.sqrt(K0 + K1))
        out = torch.empty(M, N, dtype=BF, device="cuda")
        L.check(L.load().vtk_linear2_bf16(a.data_ptr(), a.stride(0), w0.data_ptr(), K0, w1.data_ptr(), K1, out.data_ptr(), N, M, N, K0, K1,
                                          L.stream_ptr()))
        ref = a[:, :K0].float() @ w0.float().t() + a[:, K0:].float() @ w1.float().t()
        report(f"linear2 M={M} N={N} K={K0}+{K1}", out, ref, rel_fro=5e-3)
    M, N, K = 1000, 512, 264
    a, bt = bf16_randn(M, K, seed=163), bf16_randn(K, N, seed=164, scale=1 / math.sqrt(K))
    base = bf16_randn(M, N, seed=165)
    out = base.clone()
    L.check(L.load().vtk_linear_nn_acc_bf16(a.data_ptr(), K, bt.data_ptr(), N, out.data_ptr(), N, M, N, K, 1, L.stream_ptr()))
    report("linear_nn accumulate", out, base.float() + a.float() @ bt.float(), rel_fro=4e-3)
    out2 = base.clone()
    L.check(L.load().vtk_linear_nn_acc_bf16(a.data_ptr(), K, bt.data_ptr(), N, out2.data_ptr(), N, M, N, K, 0, L.stream_ptr()))
    report("linear_nn overwrite", out2, a.float() @ bt.float(), rel_fro=4e-3)


def _attn_inputs(B, N, heads, d, seed):
    qkv = bf16_randn(B * N, 3 * heads * d, seed=seed)
    do = bf16_randn(B * N, heads * d, seed=seed + 1)
    return qkv, do


@pytest.mark.parametrize("B,N,heads,d,lens,w", [
    (2, 256, 2, 64, None, -1), (1, 512, 2, 128, None, -1), (2, 384, 2, 64, [384, 130], -1), (1, 200, 1, 64, None, -1),
    (1, 512, 2, 64, None, 70), (2, 256, 1, 128, [100, 256], -1), (1, 1024, 1, 128, None, 200)])
def test_attention_backward(L, B, N, heads, d, lens, w):
    qkv, do = _attn_inputs(B, N, heads, d, 70)
    D = heads * d
    mask = None
    if lens is not None:
        mask = torch.zeros(B, N, dtype=torch.bool)
        for b, n in enumerate(lens):
            mask[b, :n] = True
    lse = torch.empty(B * N, heads, dtype=torch.float32, device="cuda")
    out = L.attention(qkv, B, N, heads, d, mask.cuda() if mask is not None else None, window=w, lse=lse)
    # oracle autograd (fp32 on the bf16 values)
    t = qkv.float().cpu().reshape(B, N, 3, heads, d).requires_grad_(True)
    ref = ae_oracle.attention_core(t[:, :, 0], t[:, :, 1], t[:, :, 2], mask, w if w >= 0 else None)
    report("attn fwd (train)", out, ref.reshape(B * N, D), max_abs=3e-2, rel_fro=1e-2)
    dof = do.float().cpu().reshape(B, N, D)
    if mask is not None:
        dof = dof * mask[:, :, None]                        # the loss never feeds gradient into padded rows
    (ref * dof).sum().backward()
    delta = torch.empty(B * N, heads, dtype=torch.float32, device="cuda")
    dod = dof.reshape(B * N, D).to(BF).cuda()
    L.check(L.load().vtk_attn_delta(out.data_ptr(), D, dod.data_ptr(), D, delta.data_ptr(), B * N, heads, d, L.stream_ptr()))
    dqkv = torch.full((B * N, 3 * D), float("nan"), dtype=BF, device="cuda")
    kl = L.kv_len(mask.cuda()) if mask is not None else None
    b0, g0 = qkv.data_ptr(), dqkv.data_ptr()
    L.check(L.load().vtk_attention_bwd_bf16(b0, b0 + 2 * D, b0 + 4 * D, 3 * D, dod.data_ptr(), D, lse.data_ptr(), delta.data_ptr(),
                                            g0, g0 + 2 * D, g0 + 4 * D, 3 * D, L.ptr(kl), B, N, heads, d, 1 if mask is not None else 0,
                                            w, L.stream_ptr()))
    got = dqkv.cpu().float().reshape(B, N, 3, heads, d)
    assert torch.isfinite(got).all()
    for i, nm in enumerate("qkv"):
        report(f"attn bwd d{nm} N={N} d={d} w={w}", got[:, :, i], t.grad[:, :, i], rel_fro=2e-2)


def _batch(sizes, patch, T, seed):
    b = pp_oracle.collate([pp_oracle.patchify(i, patch, T) for i in synth_images(sizes, seed=seed)])
    return {k: torch.from_numpy(np.asarray(v)) for k, v in b.items()}


@pytest.mark.parametrize("backend", ["sdpa", "flash"])
def test_training_step_gradients_vs_oracle(backend):
    """Loss and every parameter gradient of one training step vs the CPU oracle's autograd (fp32)."""
    import vitok_b200 as vb
    cfg = vb.decode_variant(SMALL)
    sd = make_state_dict(cfg, seed=1, stress=True)           # gamma ~ U(0.5, 1.5): the blocks matter
    sizes = [(128, 128), (96, 64), (128, 112), (64, 128)] if backend == "sdpa" else [(128, 128)] * 4
    batch = _batch(sizes, 16, 64, seed=11)
    model = vb.AE(**cfg, attn_backend=backend).train()
    model.load_state_dict(sd, strict=True)
    model = model.to("cuda", BF)
    cb = {k: (v.cuda().to(BF) if v.dtype == torch.float32 else v.cuda()) for k, v in batch.items()}
    out = model(cb)
    loss = vb.charbonnier_loss(out["patches"], cb["patches"], cb["patch_mask"], eps=1e-3)
    loss.backward()
    sd_b = {k: v.to(BF).float() for k, v in sd.items()}      # the oracle sees the same bf16-rounded weights and inputs
    bb = dict(batch)
    bb["patches"] = batch["patches"].to(BF).float()
    ref_loss, ref_g = ae_oracle.train_step_grads(sd_b, bb, cfg["encoder_heads"], cfg["decoder_heads"], attn_backend=backend)
    print(f"[parity] train step {backend}: loss ours {loss.item():.6f} oracle {ref_loss.item():.6f}")
    assert abs(loss.item() - ref_loss.item()) <= 5e-3 * abs(ref_loss.item())
    worst = ("", 0.0)
    for name, p in model.named_parameters():
        assert p.grad is not None and p.grad.shape == p.shape and torch.isfinite(p.grad).all(), name
        r = _rel(p.grad, ref_g[name])
        if r > worst[1]:
            worst = (name, r)
        cos = F.cosine_similarity(p.grad.float().cpu().flatten(), ref_g[name].flatten(), dim=0).item()
        assert cos >= 0.995, (name, cos, r)
    print(f"[parity] train step {backend}: worst rel-Frobenius gradient error {worst[1]:.3e} at {worst[0]}")
    assert worst[1] <= 8e-2


def test_training_loop_reduces_loss():
    import vitok_b200 as vb
    cfg = vb.decode_variant(SMALL)
    torch.manual_seed(0)
    model = vb.AE(**cfg, attn_backend="flash").train().to("cuda", BF)
    decay = [p for n, p in model.named_parameters() if p.ndim > 1 and "norm" not in n and "bias" not in n]
    no_decay = [p for n, p in model.named_parameters() if not (p.ndim > 1 and "norm" not in n and "bias" not in n)]
    opt = vb.FusedAdamW([{"params": decay, "weight_decay": 0.01}, {"params": no_decay, "weight_decay": 0.0}], lr=3e-3, betas=(0.9, 0.99))
    batch = _batch([(128, 128)] * 4, 16, 64, seed=3)
    cb = {k: (v.cuda().to(BF) if v.dtype == torch.float32 else v.cuda()) for k, v in batch.items()}
    losses = []
    for _ in range(12):
        opt.zero_grad(set_to_none=True)
        out = model(cb)
        loss = vb.charbonnier_loss(out["patches"], cb["patches"], cb["patch_mask"])
        loss.backward()
        opt.step()
        losses.append(loss.item())
    print("[parity] losses", [round(x, 4) for x in losses])
    assert losses[-1] < 0.9 * losses[0] and all(math.isfinite(x) for x in losses)
    # inference path sees the updated weights (packed copies were invalidated by the optimizer)
    model.eval()
    with torch.no_grad():
        o = model(cb)["patches"]
    l2 = vb.charbonnier_loss(o, cb["patches"], cb["patch_mask"]).item()
    assert l2 < losses[0]


def _train_once(model, cb):
    import vitok_b200 as vb
    for p in model.parameters():
        p.grad = None
    out = model(cb)
    loss = vb.charbonnier_loss(out["patches"], cb["patches"], cb["patch_mask"], eps=1e-3)
    loss.backward()
    return loss.detach(), out["patches"].detach(), {n: p.grad.clone() for n, p in model.named_parameters()}


def test_training_drop_path_vs_oracle(monkeypatch):
    """AE(drop_path_rate > 0) in train mode (ae.py:15-30,65,143-152): decoder block i drops images with rate * i / (depth - 1).
    The draws come from torch.rand exactly as in the reference; here torch.rand is patched so that the same draws can be
    handed to the oracle, and loss + gradients are compared.  Then: seeded runs repeat, other seeds differ, eval ignores it."""
    import vitok_b200 as vb
    cfg = vb.decode_variant(SMALL)
    sd = make_state_dict(cfg, seed=1, stress=True)
    batch = _batch([(128, 128)] * 6, 16, 64, seed=12)
    rate = 0.5
    model = vb.AE(**cfg, attn_backend="flash", drop_path_rate=rate).train()
    model.load_state_dict(sd, strict=True)
    model = model.to("cuda", BF)
    cb = {k: (v.cuda().to(BF) if v.dtype == torch.float32 else v.cuda()) for k, v in batch.items()}
    depth = cfg["decoder_depth"]
    draws = [torch.rand(6, generator=torch.Generator().manual_seed(200 + i)) for i in range(depth)]
    calls = []
    real_rand = torch.rand

    def fake_rand(shape, dtype=None, device=None, **kw):
        u = draws[1 + len(calls)]                      # block 0 has rate 0 and draws nothing
        calls.append(tuple(shape))
        return u.reshape(shape).to(dtype=dtype, device=device)

    monkeypatch.setattr(torch, "rand", fake_rand)
    loss, _, grads = _train_once(model, cb)
    monkeypatch.setattr(torch, "rand", real_rand)
    assert calls == [(6, 1, 1)] * (depth - 1)
    keep = {i: (1.0 - rate * i / (depth - 1) + draws[i].to(BF)).floor().float() for i in range(1, depth)}
    assert any(float(k.min()) == 0.0 for k in keep.values()) and any(float(k.max()) == 1.0 for k in keep.values())
    sd_b = {k: v.to(BF).float() for k, v in sd.items()}
    bb = dict(batch)
    bb["patches"] = batch["patches"].to(BF).float()
    ref_loss, ref_g = ae_oracle.train_step_grads(sd_b, bb, cfg["encoder_heads"], cfg["decoder_heads"], attn_backend="flash",
                                                 drop_keep=keep, drop_path_rate=rate)
    assert abs(loss.item() - ref_loss.item()) <= 5e-3 * abs(ref_loss.item())
    worst = max((_rel(grads[n], ref_g[n]), n) for n in grads)
    print(f"[parity] drop_path train step: loss {loss.item():.6f} / {ref_loss.item():.6f}, worst gradient rel-Fro {worst[0]:.3e} at {worst[1]}")
    assert worst[0] <= 8e-2
    # the real generator: same seed -> same step, another seed -> another set of dropped images; eval mode: no drop_path
    torch.manual_seed(5)
    l1, o1, _ = _train_once(model, cb)
    torch.manual_seed(5)
    l2, o2, _ = _train_once(model, cb)
    torch.manual_seed(6)
    l3, o3, _ = _train_once(model, cb)
    assert torch.equal(o1, o2) and not torch.equal(o1, o3)
    model.eval()
    with torch.no_grad():
        e1 = model(cb)["patches"]
        e2 = model(cb)["patches"]
    assert torch.equal(e1, e2)


@pytest.mark.parametrize("ck", [1, 2])
def test_activation_checkpointing_is_bit_identical(ck):
    """AE(checkpoint=k) (ae.py:159-160,202-205,231-233): blocks with i % k == 0 keep only their input and are re-run inside the
    backward pass.  Output and every weight gradient are bit-identical to the un-checkpointed step (also with drop_path: the
    block's draw is kept, not re-drawn), the vector gradients equal up to the order of their fp32 atomic sums, and the forward pass
    holds less memory."""
    import vitok_b200 as vb
    cfg = vb.decode_variant(SMALL)
    sd = make_state_dict(cfg, seed=1, stress=True)
    batch = _batch([(128, 128), (96, 64), (128, 112), (64, 128)], 16, 64, seed=11)
    cb = {k: (v.cuda().to(BF) if v.dtype == torch.float32 else v.cuda()) for k, v in batch.items()}
    res = {}
    for c in (0, ck):
        m = vb.AE(**cfg, attn_backend="sdpa", checkpoint=c, drop_path_rate=0.3).train()
        m.load_state_dict(sd, strict=True)
        m = m.to("cuda", BF)
        torch.manual_seed(9)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        out = m(cb)
        held = torch.cuda.memory_allocated() - base
        loss = vb.charbonnier_loss(out["patches"], cb["patches"], cb["patch_mask"], eps=1e-3)
        loss.backward()
        res[c] = (loss.detach(), out["patches"].detach(), {n: p.grad.clone() for n, p in m.named_parameters()}, held)
    assert torch.equal(res[0][1], res[ck][1])                                   # same forward (and the same stochastic-depth draws)
    assert abs(float(res[0][0]) - float(res[ck][0])) <= 1e-6 * abs(float(res[0][0]))   # the loss sums per-token terms with fp32 atomics
    for n in res[0][2]:
        a, b = res[0][2][n], res[ck][2][n]
        if a.ndim >= 2:
            assert torch.equal(a, b), n                                          # GEMM-produced gradients: bit-identical
        else:
            # norm weights / gamma / biases: fp32 atomic column sums whose order differs from run to run, then ONE rounding to the bf16
            # gradient -- a sum that lands next to a rounding boundary may come out one bf16 ulp (2^-8 relative) away, so: every
            # element within one ulp (+ a floor of 2^-8 of the vector's largest element, for sums that cancel to ~0), few of them
            fa, fb = a.float(), b.float()
            tol = 2.0 ** -7 * torch.maximum(fa.abs(), fb.abs()) + 2.0 ** -8 * fa.abs().max()
            assert bool(((fa - fb).abs() <= tol).all()), (n, float((fa - fb).abs().max()))
            assert _rel(a, b) <= 2e-3, (n, _rel(a, b))
    print(f"[parity] activations held after forward: checkpoint=0 {res[0][3] / 2**20:.1f} MiB, checkpoint={ck} {res[ck][3] / 2**20:.1f} MiB")
    assert res[ck][3] < (0.45 if ck == 1 else 0.8) * res[0][3]


def test_training_with_non_prefix_mask_vs_oracle():
    """The reference's autograd handles any patch_mask (ae.py:173-187).  Here a mask with holes is turned into a prefix mask by
    permuting tokens (positions travel in row_idx / col_idx), the prefix path runs, and the output is permuted back."""
    import vitok_b200 as vb
    cfg = vb.decode_variant(SMALL)
    sd = make_state_dict(cfg, seed=1, stress=True)
    batch = _batch([(128, 128), (96, 64), (128, 112), (64, 128)], 16, 64, seed=13)
    g = torch.Generator().manual_seed(3)
    mask = batch["patch_mask"].clone()
    mask &= torch.rand(mask.shape, generator=g) > 0.3          # knock holes into every image
    mask[:, 0] = True
    batch["patch_mask"] = mask
    model = vb.AE(**cfg, attn_backend="sdpa").train()
    model.load_state_dict(sd, strict=True)
    model = model.to("cuda", BF)
    cb = {k: (v.cuda().to(BF) if v.dtype == torch.float32 else v.cuda()) for k, v in batch.items()}
    loss, out, grads = _train_once(model, cb)
    sd_b = {k: v.to(BF).float() for k, v in sd.items()}
    bb = dict(batch)
    bb["patches"] = batch["patches"].to(BF).float()
    ref_loss, ref_g = ae_oracle.train_step_grads(sd_b, bb, cfg["encoder_heads"], cfg["decoder_heads"], attn_backend="sdpa")
    assert abs(loss.item() - ref_loss.item()) <= 5e-3 * abs(ref_loss.item())
    worst = max((_rel(grads[n], ref_g[n]), n) for n in grads)
    print(f"[parity] non-prefix mask train step: worst gradient rel-Fro {worst[0]:.3e} at {worst[1]}")
    assert worst[0] <= 8e-2
    # forward values on valid tokens equal the inference path's (which packs valid tokens)
    model.eval()
    with torch.no_grad():
        inf = model(cb)["patches"]
    report("train-mode vs eval-mode output on valid tokens", out[mask.cuda()], inf[mask.cuda()].float(), max_abs=6e-2, rel_fro=1e-2)


def test_double_backward_raises_and_patches_get_a_gradient():
    import vitok_b200 as vb
    cfg = vb.decode_variant(SMALL)
    sd = make_state_dict(cfg, seed=1, stress=True)
    batch = _batch([(128, 128)] * 2, 16, 64, seed=14)
    model = vb.AE(**cfg, attn_backend="flash").train()
    model.load_state_dict(sd, strict=True)
    model = model.to("cuda", BF)
    cb = {k: (v.cuda().to(BF) if v.dtype == torch.float32 else v.cuda()) for k, v in batch.items()}
    cb["patches"] = cb["patches"].clone().requires_grad_(True)
    out = model(cb)["patches"]
    w = bf16_randn(*out.shape, seed=15)
    (out * w).sum().backward(retain_graph=True)
    assert cb["patches"].grad is not None and cb["patches"].grad.shape == cb["patches"].shape
    # oracle: d sum(out * w) / d patches
    sd_b = {k: v.to(BF).float() for k, v in sd.items()}
    pc = batch["patches"].to(BF).float().requires_grad_(True)
    bb = dict(batch)
    bb["patches"] = pc
    enc = ae_oracle.encode(sd_b, bb, cfg["encoder_heads"], attn_backend="flash")
    dec = ae_oracle.decode(sd_b, enc, cfg["decoder_heads"], attn_backend="flash")
    (dec["patches"] * w.float().cpu()).sum().backward()
    report("d out / d patches", cb["patches"].grad, pc.grad, rel_fro=8e-2)
    with pytest.raises(RuntimeError, match="already run"):
        (out * w).sum().backward()


def test_5b_shape_training_gradients_vs_oracle():
    """BASELINE configs[4] at its real block shape: 5B-f32x256 widths (D = 3072, 24 heads of 128, Hf = 8208), patch 32
    (P = 3072), C = 256, N = 1024 tokens -- one encoder + one decoder block, one 1024 x 1024 image.  Loss and every parameter
    gradient vs fp32 CPU autograd of the oracle (the d = 128 attention backward at 8 x 8 tile pairs, the transposed-operand GEMMs
    at K = 1024 tokens, the two-weight forward GEMM at K = 3072 + 8208)."""
    import os
    import vitok_b200 as vb
    variant = "w3072_d1_h24-w3072_d1_h24/1x32x256"
    cfg = vb.decode_variant(variant)
    sd = make_state_dict(cfg, seed=4, stress=True)
    batch = _batch([(1024, 1024)], 32, 1024, seed=21)
    model = vb.AE(**cfg, attn_backend="flash").train()
    model.load_state_dict(sd, strict=True)
    model = model.to("cuda", BF)
    cb = {k: (v.cuda().to(BF) if v.dtype == torch.float32 else v.cuda()) for k, v in batch.items()}
    loss, _, grads = _train_once(model, cb)
    torch.set_num_threads(os.cpu_count() or 1)
    sd_b = {k: v.to(BF).float() for k, v in sd.items()}
    bb = dict(batch)
    bb["patches"] = batch["patches"].to(BF).float()
    ref_loss, ref_g = ae_oracle.train_step_grads(sd_b, bb, cfg["encoder_heads"], cfg["decoder_heads"], attn_backend="flash")
    print(f"[parity] 5B-shape train step: loss ours {loss.item():.6f} oracle {ref_loss.item():.6f}")
    assert abs(loss.item() - ref_loss.item()) <= 5e-3 * abs(ref_loss.item())
    worst = ("", 0.0)
    for name, g in grads.items():
        assert torch.isfinite(g).all(), name
        r = _rel(g, ref_g[name])
        cos = F.cosine_similarity(g.float().cpu().flatten(), ref_g[name].flatten(), dim=0).item()
        assert cos >= 0.995, (name, cos, r)
        worst = max(worst, (name, r), key=lambda t: t[1])
    print(f"[parity] 5B-shape train step: worst rel-Frobenius gradient error {worst[1]:.3e} at {worst[0]}")
    assert worst[1] <= 8e-2
