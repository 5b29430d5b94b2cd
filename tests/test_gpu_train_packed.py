"""Training on packed NaFlex rows (AE.train_token_packing; vitok_b200/train.py: _Packing).

Kernel level: the packed attention forward that also writes lse (vtk_attention_packed_lse_bf16) and the packed attention backward
(vtk_attention_bwd_packed_bf16) against their padded counterparts on the same data, bit for bit, with sentinel-filled buffers so that
a store outside an image's packed rows fails.  Model level: the packed training step against the padded one (same loss and
reconstruction, gradients within a summation-order tolerance) and against the fp32 CPU oracle's autograd.

The ragged batch has images of 1, 127, 128, 129, 300 and 1024 valid tokens and one with none: single-row, partial, exact and
one-past tiles, and an image whose rows are followed directly by the next image's in a partial last tile."""
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
LENS = [1, 127, 128, 129, 300, 1024, 0]
N_TOK = 1024
SENT = -12288.0      # sentinel of lse / gradient buffers (exact in bf16 and fp32)


@pytest.fixture(scope="module")
def L():
    from vitok_b200 import _lib
    _lib.load()
    return _lib


def _prefix_mask(lens, N):
    m = torch.zeros(len(lens), N, dtype=torch.bool)
    for b, n in enumerate(lens):
        m[b, :n] = True
    return m


def _rows(plan, B):
    """(cu, n_valid) on the host."""
    return plan["cu"].cpu().tolist(), plan["n_valid"].cpu().tolist()


def _subset_plan(plan, B, keep_imgs):
    """The plan restricted to the work groups of ``keep_imgs``: the kernels then run for those images only, and every row of the
    other images must keep what the buffers held."""
    gi = plan["grp_img"].cpu()
    ng = int(plan["cuq"][B])
    order = [g for g in range(ng) if int(gi[g]) in keep_imgs]
    sub = dict(plan)
    sub["grp_order"] = torch.tensor(order + [-2] * (gi.numel() - len(order)), dtype=torch.int32, device="cuda")
    cuq = plan["cuq"].clone()
    cuq[B] = len(order)
    sub["cuq"] = cuq
    return sub


def _packed_fwd(L, qkv_pk, plan, B, heads, d, fill_out=7.0):
    D = heads * d
    rows = qkv_pk.shape[0]
    out = torch.full((rows, D), fill_out, dtype=BF, device="cuda")
    lse = torch.full((rows, heads), SENT, dtype=torch.float32, device="cuda")
    L.attention_packed(qkv_pk, plan, B, N_TOK, heads, d, lse=lse, out=out)
    return out, lse


@pytest.mark.parametrize("heads,d", [(3, 64), (2, 128)])
def test_packed_forward_lse_matches_padded(L, heads, d):
    B, N, D = len(LENS), N_TOK, heads * d
    mask = _prefix_mask(LENS, N).cuda()
    qkv = bf16_randn(B * N, 3 * D, seed=80 + d)
    lse_pad = torch.empty(B * N, heads, dtype=torch.float32, device="cuda")
    out_pad = L.attention(qkv, B, N, heads, d, mask, lse=lse_pad)
    plan = L.pack_plan(mask, 16, 128 if d == 64 else 256)
    qkv_pk = L.pack_rows(qkv.view(B, N, 3 * D), plan)
    cu, nv = _rows(plan, B)
    out, lse = _packed_fwd(L, qkv_pk, plan, B, heads, d)
    for b in range(B):
        r0, n, r1 = cu[b], nv[b], cu[b + 1]
        assert torch.equal(out[r0:r0 + n], out_pad[b * N:b * N + n]), b
        assert torch.equal(lse[r0:r0 + n], lse_pad[b * N:b * N + n]), b
        assert bool((out[r0 + n:r1] == 0).all()) and bool(torch.isinf(lse[r0 + n:r1]).all() and (lse[r0 + n:r1] > 0).all()), b
    assert bool((lse[cu[B]:] == SENT).all()) and bool((out[cu[B]:] == 7.0).all())       # rows past the last image: untouched
    # only images 1, 3, 5 (127, 129, 1024 tokens: partial last tiles running into the next image's rows): every other image's rows
    # keep the sentinel, the selected ones come out as above
    sub = _subset_plan(plan, B, {1, 3, 5})
    out_s, lse_s = _packed_fwd(L, qkv_pk, sub, B, heads, d)
    for b in range(B):
        r0, r1 = cu[b], cu[b + 1]
        if b in (1, 3, 5):
            assert torch.equal(out_s[r0:r1], out[r0:r1]) and torch.equal(lse_s[r0:r1], lse[r0:r1]), b
        else:
            assert bool((lse_s[r0:r1] == SENT).all()) and bool((out_s[r0:r1] == 7.0).all()), b


def _attn_delta(L, out, do, rows, heads, d):
    D = heads * d
    delta = torch.zeros(out.shape[0], heads, dtype=torch.float32, device="cuda")     # rows >= `rows` stay 0
    L.check(L.load().vtk_attn_delta(out.data_ptr(), out.stride(0), do.data_ptr(), do.stride(0), delta.data_ptr(), rows, heads, d,
                                    L.stream_ptr()))
    return delta


def _packed_bwd(L, qkv_pk, do_pk, lse, delta, plan, B, heads, d):
    D = heads * d
    rows = qkv_pk.shape[0]
    dqkv = torch.full((rows, 3 * D), SENT, dtype=BF, device="cuda")
    b0, g0 = qkv_pk.data_ptr(), dqkv.data_ptr()
    L.check(L.load().vtk_attention_bwd_packed_bf16(b0, b0 + 2 * D, b0 + 4 * D, 3 * D, do_pk.data_ptr(), D, lse.data_ptr(), delta.data_ptr(),
                                                   g0, g0 + 2 * D, g0 + 4 * D, 3 * D, plan["n_valid"].data_ptr(), plan["cu"].data_ptr(),
                                                   plan["cuq"].data_ptr(), plan["grp_img"].data_ptr(), plan["grp_order"].data_ptr(), B,
                                                   heads, d, rows, plan["grp_img"].numel(), L.stream_ptr()))
    return dqkv


@pytest.mark.parametrize("heads,d", [(3, 64), (2, 128)])
def test_packed_attention_backward_matches_padded(L, heads, d):
    B, N, D = len(LENS), N_TOK, heads * d
    mask_h = _prefix_mask(LENS, N)
    mask = mask_h.cuda()
    qkv = bf16_randn(B * N, 3 * D, seed=90 + d)
    do = (bf16_randn(B * N, D, seed=91 + d).view(B, N, D) * mask[:, :, None]).view(B * N, D)   # no gradient enters padded rows
    # padded reference
    lse_pad = torch.empty(B * N, heads, dtype=torch.float32, device="cuda")
    out_pad = L.attention(qkv, B, N, heads, d, mask, lse=lse_pad)
    delta_pad = _attn_delta(L, out_pad, do, B * N, heads, d)
    kl = L.kv_len(mask)
    dqkv_pad = torch.empty(B * N, 3 * D, dtype=BF, device="cuda")
    b0, g0 = qkv.data_ptr(), dqkv_pad.data_ptr()
    L.check(L.load().vtk_attention_bwd_bf16(b0, b0 + 2 * D, b0 + 4 * D, 3 * D, do.data_ptr(), D, lse_pad.data_ptr(), delta_pad.data_ptr(),
                                            g0, g0 + 2 * D, g0 + 4 * D, 3 * D, kl.data_ptr(), B, N, heads, d, 1, -1, L.stream_ptr()))
    # sanity of the reference against fp32 autograd of the oracle
    t = qkv.float().cpu().reshape(B, N, 3, heads, d).requires_grad_(True)
    ref = ae_oracle.attention_core(t[:, :, 0], t[:, :, 1], t[:, :, 2], mask_h)
    (ref * do.float().cpu().reshape(B, N, D)).sum().backward()
    got = dqkv_pad.float().cpu().reshape(B, N, 3, heads, d)
    for i, nm in enumerate("qkv"):
        report(f"padded attn bwd d{nm} d={d}", got[:, :, i], t.grad[:, :, i], rel_fro=2e-2)
    # packed: the forward's lse, delta over the packed rows
    plan_f = L.pack_plan(mask, 16, 128 if d == 64 else 256)
    plan = L.pack_plan(mask, 16, 128)
    cu, nv = _rows(plan, B)
    qkv_pk = L.pack_rows(qkv.view(B, N, 3 * D), plan)
    do_pk = L.pack_rows(do.view(B, N, D), plan)
    out_pk, lse_pk = _packed_fwd(L, qkv_pk, plan_f, B, heads, d)
    delta_pk = _attn_delta(L, out_pk, do_pk, cu[B], heads, d)
    dqkv = _packed_bwd(L, qkv_pk, do_pk, lse_pk, delta_pk, plan, B, heads, d)

    def check(dq, subset=None):
        for b in range(B):
            r0, n, r1 = cu[b], nv[b], cu[b + 1]
            if subset is not None and b not in subset:
                assert bool((dq[r0:r1] == SENT).all()), b                             # another image's rows: untouched
                continue
            assert torch.equal(dq[r0:r0 + n], dqkv_pad[b * N:b * N + n]), b
            assert bool((dq[r0 + n:r1] == 0).all()), b                                # the image's pad rows: 0
        assert bool((dq[cu[B]:] == SENT).all())

    check(dqkv)
    # MODE 0's query-row rule: rows past an image's end must contribute nothing to its dK / dV whatever they hold.  Poison every
    # row outside the valid tokens (the images' pad rows and the rows past the last image) with non-zero dO, a finite lse and a
    # non-zero delta -- without the explicit row mask they would get P = exp2(S * scale) != 0.  The next image's rows after a
    # partial tile already carry non-zero dO, finite lse and delta in every run.
    valid = torch.zeros(qkv_pk.shape[0], dtype=torch.bool, device="cuda")
    for b in range(B):
        valid[cu[b]:cu[b] + nv[b]] = True
    do_p = torch.where(valid[:, None], do_pk, bf16_randn(*do_pk.shape, seed=92, scale=4.0))
    lse_p = torch.where(valid[:, None], lse_pk, torch.zeros_like(lse_pk))
    delta_p = torch.where(valid[:, None], delta_pk, torch.full_like(delta_pk, 0.75))
    check(_packed_bwd(L, qkv_pk, do_p, lse_p, delta_p, plan, B, heads, d))
    # only images 1, 3, 5: the rows of the others keep the sentinel
    check(_packed_bwd(L, qkv_pk, do_p, lse_p, delta_p, _subset_plan(plan, B, {1, 3, 5}), B, heads, d), subset={1, 3, 5})


# ---------------------------------------------------------------------------------------------------------------------------
# whole training step
# ---------------------------------------------------------------------------------------------------------------------------
def _ragged_batch(lens, N, P, seed, holes=False):
    """Square synthetic images of N tokens (patchified by the oracle); image b keeps its first lens[b] tokens, and with ``holes``
    about 30 % of those are knocked out as well."""
    patch = int(math.isqrt(P // 3))
    side = int(math.isqrt(N))
    imgs = synth_images([(side * patch, side * patch)] * len(lens), seed=seed)
    b = {k: torch.from_numpy(np.asarray(v)) for k, v in pp_oracle.collate([pp_oracle.patchify(i, patch, N) for i in imgs]).items()}
    mask = _prefix_mask(lens, N)
    if holes:
        mask &= torch.rand(mask.shape, generator=torch.Generator().manual_seed(seed)) > 0.3
        mask[:, 0] = torch.tensor(lens) > 0
    assert bool(b["patch_mask"].all())
    return {"patches": b["patches"].float(), "patch_mask": mask, "row_idx": b["row_idx"], "col_idx": b["col_idx"]}


def _model(cfg, sd, **kw):
    import vitok_b200 as vb
    m = vb.AE(**cfg, attn_backend=kw.pop("attn_backend", "sdpa"), **kw).train()
    m.load_state_dict(sd, strict=True)
    return m.to("cuda", BF)


def _cuda_batch(batch):
    return {k: (v.cuda().to(BF) if v.dtype == torch.float32 else v.cuda()) for k, v in batch.items()}


def _step(model, cb, seed=0):
    import vitok_b200 as vb
    for p in model.parameters():
        p.grad = None
    if cb["patches"].requires_grad:
        cb["patches"].grad = None
    torch.manual_seed(seed)
    out = model(cb)
    loss = vb.charbonnier_loss(out["patches"], cb["patches"], cb.get("patch_mask"), eps=1e-3)
    loss.backward()
    dp = cb["patches"].grad.clone() if cb["patches"].requires_grad else None
    return loss.detach(), out["patches"].detach(), {n: p.grad.clone() for n, p in model.named_parameters()}, dp


def _cos(a, b):
    return F.cosine_similarity(a.float().cpu().flatten(), b.float().cpu().flatten(), dim=0).item()


def _rel(got, ref):
    got, ref = got.detach().float().cpu(), ref.detach().float().cpu()
    return (torch.linalg.norm(got - ref) / torch.linalg.norm(ref).clamp_min(1e-30)).item()


def _vs_oracle(tag, cfg, sd, batch, loss, grads):
    sd_b = {k: v.to(BF).float() for k, v in sd.items()}
    bb = dict(batch)
    bb["patches"] = batch["patches"].to(BF).float()
    ref_loss, ref_g = ae_oracle.train_step_grads(sd_b, bb, cfg["encoder_heads"], cfg["decoder_heads"], attn_backend="sdpa")
    assert abs(loss.item() - ref_loss.item()) <= 5e-3 * abs(ref_loss.item()), (tag, loss.item(), ref_loss.item())
    worst = ("", 0.0)
    for name, g in grads.items():
        assert torch.isfinite(g).all(), name
        r = _rel(g, ref_g[name])
        assert _cos(g, ref_g[name]) >= 0.995, (tag, name, r)
        worst = max(worst, (name, r), key=lambda t: t[1])
    print(f"[parity] packed train step {tag} vs oracle: loss {loss.item():.6f} / {ref_loss.item():.6f}, worst rel-Fro {worst[1]:.3e} at {worst[0]}")
    assert worst[1] <= 8e-2, (tag, worst)


D128 = "w256_d1_h2-w256_d1_h2/1x16x16"     # one encoder + one decoder block, head_dim 128 on both sides


def _oracle_batch(holes):
    """The batch of the oracle gradient tests in test_gpu_train.py (4 images of 64 tokens at most), with their hole pattern."""
    imgs = synth_images([(128, 128), (96, 64), (128, 112), (64, 128)], seed=11)
    b = {k: torch.from_numpy(np.asarray(v)) for k, v in pp_oracle.collate([pp_oracle.patchify(i, 16, 64) for i in imgs]).items()}
    if holes:
        b["patch_mask"] = b["patch_mask"] & (torch.rand(b["patch_mask"].shape, generator=torch.Generator().manual_seed(3)) > 0.3)
        b["patch_mask"][:, 0] = True
    return b


@pytest.mark.parametrize("case", ["ragged", "drop_path", "checkpoint", "holes", "dpatches", "d128"])
def test_packed_training_step_vs_padded_and_oracle(case):
    """train_token_packing True vs False on the same ragged sdpa batch: the loss equal up to the order of the loss kernel's fp32
    atomics, the reconstruction bit-identical on valid tokens (0 on masked ones), every parameter gradient within cosine 0.9999 /
    rel-Fro 1e-2 (the weight gradients sum the same terms in another order and blocking).  Then the packed step vs the fp32 oracle
    within the gates of test_gpu_train.py, on the batch those tests use: with the 1024-token images of the ragged batch and stress
    init the bf16 step is further from the fp32 oracle than those gates in either layout (worst rel-Fro ~0.1 for padded and packed
    alike), which says nothing about packing."""
    import vitok_b200 as vb
    variant = D128 if case == "d128" else SMALL
    cfg = vb.decode_variant(variant)
    sd = make_state_dict(cfg, seed=1, stress=True)
    kw = {"drop_path_rate": 0.3} if case == "drop_path" else {"checkpoint": 2} if case == "checkpoint" else {}
    model = _model(cfg, sd, **kw)
    batch = _ragged_batch(LENS, N_TOK, cfg["pixels_per_token"], seed=31, holes=case == "holes")
    cb = _cuda_batch(batch)
    if case == "dpatches":
        cb["patches"] = cb["patches"].clone().requires_grad_(True)
    mask = cb["patch_mask"]
    res = {}
    for packed in (False, True):
        model.train_token_packing = packed
        res[packed] = _step(model, cb, seed=17)
    (l0, o0, g0, d0), (l1, o1, g1, d1) = res[False], res[True]
    assert abs(l1.item() - l0.item()) <= 1e-6 * abs(l0.item()), (l0.item(), l1.item())
    assert torch.equal(o1[mask], o0[mask])
    assert bool((o1[~mask] == 0).all())
    worst = ("", 0.0, 1.0)
    for n in g0:
        assert torch.isfinite(g1[n]).all(), n
        r, c = _rel(g1[n], g0[n]), _cos(g1[n], g0[n])
        assert c >= 0.9999 and r <= 1e-2, (n, c, r)
        worst = max(worst, (n, r, c), key=lambda t: t[1])
    print(f"[parity] packed vs padded train step ({case}): loss {l1.item():.6f} / {l0.item():.6f}, worst gradient rel-Fro {worst[1]:.3e} "
          f"(cos {worst[2]:.6f}) at {worst[0]}")
    if case == "dpatches":
        report("dpatches packed vs padded (valid tokens)", d1[mask], d0[mask].float(), rel_fro=1e-2)
        assert bool((d1[~mask] == 0).all())
    if case == "checkpoint":
        # the re-run blocks work on the packed tensors: every GEMM-produced gradient equals the un-checkpointed packed step's
        ref = _model(cfg, sd)
        ref.train_token_packing = True
        _, o2, g2, _ = _step(ref, cb, seed=17)
        assert torch.equal(o2, o1)
        for n in g2:
            if g2[n].ndim >= 2:
                assert torch.equal(g2[n], g1[n]), n
    if case != "drop_path":   # (the oracle's drop-path draws would have to be injected; test_gpu_train.py covers that path)
        small = _oracle_batch(case == "holes")
        cs = _cuda_batch(small)
        if case == "dpatches":
            cs["patches"] = cs["patches"].clone().requires_grad_(True)
        model.train_token_packing = True
        ls, _, gs, _ = _step(model, cs, seed=17)
        _vs_oracle(case, cfg, sd, small, ls, gs)


def test_packed_training_unaligned_batch_and_empty_batch():
    """B * N % 8 != 0: the padded step raises as before, the packed step trains (its row count is a multiple of 16).  A batch
    without a valid token raises ValueError."""
    import vitok_b200 as vb
    cfg = vb.decode_variant(SMALL)
    sd = make_state_dict(cfg, seed=1, stress=True)
    batch = _ragged_batch([5, 49, 0], 49, cfg["pixels_per_token"], seed=32)      # 3 x 49 = 147 rows
    cb = _cuda_batch(batch)
    model = _model(cfg, sd)
    with pytest.raises(ValueError, match="multiple of 8"):
        model(cb)
    model.train_token_packing = True
    loss, out, grads, _ = _step(model, cb)
    _vs_oracle("B*N=147", cfg, sd, batch, loss, grads)
    empty = dict(cb)
    empty["patch_mask"] = torch.zeros_like(cb["patch_mask"])
    with pytest.raises(ValueError, match="no valid token"):
        model(empty)


@pytest.mark.parametrize("backend", ["flash", "sdpa-no-mask"])
def test_flag_changes_nothing_without_a_mask(backend):
    """Flash backend (the mask is ignored) or no patch_mask: train_token_packing changes nothing.  Output and every GEMM-produced
    gradient bit-identical; the vector gradients (fp32 atomic column sums, whose order varies from run to run) within one bf16 ulp."""
    import vitok_b200 as vb
    cfg = vb.decode_variant(SMALL)
    sd = make_state_dict(cfg, seed=1, stress=True)
    cb = _cuda_batch(_ragged_batch(LENS, N_TOK, cfg["pixels_per_token"], seed=33))
    if backend != "flash":
        cb.pop("patch_mask")
    model = _model(cfg, sd, attn_backend="flash" if backend == "flash" else "sdpa")
    res = {}
    for packed in (False, True):
        model.train_token_packing = packed
        res[packed] = _step(model, cb)
    assert torch.equal(res[False][1], res[True][1])
    assert abs(res[False][0].item() - res[True][0].item()) <= 1e-6 * abs(res[False][0].item())
    for n, a in res[False][2].items():
        b = res[True][2][n]
        if a.ndim >= 2:
            assert torch.equal(a, b), n
        else:
            fa, fb = a.float(), b.float()
            tol = 2.0 ** -7 * torch.maximum(fa.abs(), fb.abs()) + 2.0 ** -8 * fa.abs().max()
            assert bool(((fa - fb).abs() <= tol).all()), n


def test_packed_training_loop_reduces_loss():
    """12 FusedAdamW steps on the packed path reduce the loss; the inference path then sees the updated weights."""
    import vitok_b200 as vb
    cfg = vb.decode_variant(SMALL)
    torch.manual_seed(0)
    model = vb.AE(**cfg, attn_backend="sdpa").train().to("cuda", BF)
    model.train_token_packing = True
    decay = [p for n, p in model.named_parameters() if p.ndim > 1 and "norm" not in n and "bias" not in n]
    no_decay = [p for n, p in model.named_parameters() if not (p.ndim > 1 and "norm" not in n and "bias" not in n)]
    opt = vb.FusedAdamW([{"params": decay, "weight_decay": 0.01}, {"params": no_decay, "weight_decay": 0.0}], lr=3e-3, betas=(0.9, 0.99))
    imgs = [pp_oracle.patchify(i, 16, 64) for i in synth_images([(128, 128), (96, 64), (128, 112), (64, 128)], seed=3)]
    batch = {k: torch.from_numpy(np.asarray(v)) for k, v in pp_oracle.collate(imgs).items()}
    cb = _cuda_batch(batch)
    losses = []
    for _ in range(12):
        opt.zero_grad(set_to_none=True)
        out = model(cb)
        loss = vb.charbonnier_loss(out["patches"], cb["patches"], cb["patch_mask"])
        loss.backward()
        opt.step()
        losses.append(loss.item())
    print("[parity] packed losses", [round(x, 4) for x in losses])
    assert losses[-1] < 0.9 * losses[0] and all(math.isfinite(x) for x in losses)
    model.eval()
    with torch.no_grad():
        o = model(cb)["patches"]
    assert vb.charbonnier_loss(o, cb["patches"], cb["patch_mask"]).item() < losses[0]
