"""Head dims other than 64 and 128 (d % 8 == 0, 8 <= d <= 128), from the kernels up to AE and the training step.

A head of width d runs on the attention kernel of the next tile width (64 or 128) through 3-D tensor maps that zero-fill the
columns d..63 / d..127, so these tests put poison in the columns a kernel must not read: every attention case has 4 heads, of
which heads 1 and 3 (the right-hand neighbours of the two checked heads 0 and 2) carry large q / k / v, and every output buffer
is wider than heads * d and filled with a sentinel that must survive.  The attention checks reuse the float64 reference and the
per-element bounds of test_gpu_attention_numerics.py."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from _util import bf16_randn, report
from oracle import ae_oracle, pp_oracle
from oracle.weights import make_state_dict, synth_images
from test_gpu_attention_numerics import (C_BWD, E32, POISON_V, SENT, Worst, _bwd_ref, _check_fwd, _fwd_ref, _grad_do, _inputs,
                                         _lens, _mask, _seed)

pytestmark = pytest.mark.gpu

BF = torch.bfloat16
DS = [16, 32, 48, 72, 96, 120]
H4 = 4                      # heads in the buffers; heads 0 and 2 are checked, 1 and 3 are poison
PAD_COLS = 24               # extra sentinel columns of every output buffer
REGIMES = ["diffuse", "qknorm2", "late_max", "uniform", "poison"]
NS = [1, 127, 129, 257, 1000]


@pytest.fixture(scope="module")
def L():
    from vitok_b200 import _lib
    _lib.load()
    return _lib


def _four(t, poison, g):
    """[B, N, 2, d] (the two checked heads) -> [B * N, 4 * d] with poison heads 1 and 3 of magnitude ``poison``."""
    B, N, _, d = t.shape
    x = torch.empty(B, N, H4, d)
    x[:, :, 0::2] = t
    x[:, :, 1::2] = poison * torch.sign(torch.randn(B, N, 2, d, generator=g))
    return x.reshape(B * N, H4 * d)


def _qkv4(q, k, v, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.cat([_four(q, 16.0, g), _four(k, 16.0, g), _four(v, POISON_V, g)], 1).to(BF).cuda()


def _real(x, d):
    """The checked heads of [rows, >= 4 d] (or [rows, 4]) -> [rows, 2, d] ([rows, 2])."""
    if d is None:
        return x[:, 0::2]
    return x[:, :H4 * d].reshape(x.shape[0], H4, d)[:, 0::2]


def _window_inputs(regime, N, d, seed, w):
    """One image for a window w.  The poison regime's offset-peaked scores need enough of a gap between the window's inside and its
    edge, which a few draws of the d / 2 frequencies miss at small d: take the first seed after ``seed`` that has it."""
    for s in range(seed, seed + 64):
        try:
            return _inputs(regime, [N], N, d, s, window=w)
        except AssertionError:
            continue
    raise AssertionError(f"no window-poison draw for N={N} d={d} w={w}")


def _fwd_padded(L, qkv, B, N, d, mask, w):
    D4 = H4 * d
    out = torch.full((B * N, D4 + PAD_COLS), SENT, dtype=BF, device="cuda")
    lse = torch.full((B * N, H4), SENT, device="cuda")
    kl = L.kv_len(mask) if mask is not None else None
    b0 = qkv.data_ptr()
    L.check(L.load().vtk_attention_bf16(b0, b0 + 2 * D4, b0 + 4 * D4, 3 * D4, out.data_ptr(), out.stride(0), L.ptr(kl), B, N, H4, d,
                                        1 if mask is not None else 0, w, lse.data_ptr(), L.stream_ptr()))
    assert bool((out[:, D4:] == SENT).all()), "columns past heads * d must stay untouched"
    return out, lse


def _packed(L, regime, lens, N, d, seed, qrows):
    """Padded inputs, the pack plan and the packed 4-head qkv whose pad rows (which no kernel may read) are poisoned."""
    q, k, v = _inputs(regime, lens, N, d, seed)
    B = len(lens)
    plan = L.pack_plan(_mask(lens, N).cuda(), 16, qrows)
    pk = L.pack_rows(_qkv4(q, k, v, seed).view(B, N, -1), plan)
    cu, nv = plan["cu"].cpu().tolist(), plan["n_valid"].cpu().tolist()
    g = torch.Generator().manual_seed(seed + 1)
    D4 = H4 * d
    for b in range(B):
        r0, r1 = cu[b] + nv[b], cu[b + 1]
        if r1 > r0:
            pk[r0:r1, :2 * D4] = (8.0 * torch.randn(r1 - r0, 2 * D4, generator=g)).to(BF).cuda()
            pk[r0:r1, 2 * D4:] = POISON_V * torch.sign(torch.randn(r1 - r0, D4, generator=g)).to(BF).cuda()
    return q, k, v, plan, pk, cu, nv


def _fwd_packed(L, pk, plan, B, N, d):
    D4 = H4 * d
    rows = pk.shape[0]
    out = torch.full((rows, D4 + PAD_COLS), SENT, dtype=BF, device="cuda")
    lse = torch.full((rows, H4), SENT, device="cuda")
    b0 = pk.data_ptr()
    L.check(L.load().vtk_attention_packed_lse_bf16(b0, b0 + 2 * D4, b0 + 4 * D4, pk.stride(0), out.data_ptr(), out.stride(0),
                                                   plan["n_valid"].data_ptr(), plan["cu"].data_ptr(), plan["cuq"].data_ptr(),
                                                   plan["grp_img"].data_ptr(), plan["grp_order"].data_ptr(), B, N, H4, d, rows,
                                                   plan["grp_img"].numel(), lse.data_ptr(), L.stream_ptr()))
    assert bool((out[:, D4:] == SENT).all()), "columns past heads * d must stay untouched"
    return out, lse


# ------------------------------------------------------------------------------------------------------------------------------
# attention forward
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["dense", "prefix", "window", "packed"])
@pytest.mark.parametrize("d", DS)
def test_attention_forward(L, d, layout):
    wst = Worst(f"fwd {layout} d={d}")
    for regime in REGIMES:
        for N in NS:
            seed = _seed("hd fwd", layout, d, regime, N)
            if layout == "dense":
                B = 2
                q, k, v = _inputs(regime, [N] * B, N, d, seed)
                out, lse = _fwd_padded(L, _qkv4(q, k, v, seed), B, N, d, None, -1)
                for b in range(B):
                    r = slice(b * N, (b + 1) * N)
                    _check_fwd(wst, f"{regime} N={N} img {b}", _real(out[r], d).reshape(N, -1), _real(lse[r], None), q[b], k[b], v[b])
            elif layout == "prefix":
                lens = _lens(N)
                B = len(lens)
                q, k, v = _inputs(regime, lens, N, d, seed)
                out, lse = _fwd_padded(L, _qkv4(q, k, v, seed), B, N, d, _mask(lens, N).cuda(), -1)
                for b, n in enumerate(lens):
                    r0 = b * N
                    if n:
                        _check_fwd(wst, f"{regime} N={N} img {b} (kv_len {n})", _real(out[r0:r0 + n], d).reshape(n, -1),
                                   _real(lse[r0:r0 + n], None), q[b, :n], k[b, :n], v[b, :n])
                    assert bool((out[r0 + n:r0 + N, :H4 * d] == 0).all()) and bool((lse[r0 + n:r0 + N] == float("inf")).all()), (N, b)
            elif layout == "window":
                for w in (0, 129, N + 7):
                    q, k, v = _window_inputs(regime, N, d, seed + w, w)
                    out, lse = _fwd_padded(L, _qkv4(q, k, v, seed), 1, N, d, None, w)
                    _check_fwd(wst, f"{regime} N={N} w={w}", _real(out, d).reshape(N, -1), _real(lse, None), q[0], k[0], v[0], w)
            else:
                lens = _lens(N)
                B = len(lens)
                q, k, v, plan, pk, cu, nv = _packed(L, regime, lens, N, d, seed, 128 if d <= 64 else 256)
                out, lse = _fwd_packed(L, pk, plan, B, N, d)
                for b, n in enumerate(nv):
                    if n:
                        r = slice(cu[b], cu[b] + n)
                        _check_fwd(wst, f"{regime} N={N} img {b} ({n} tokens)", _real(out[r], d).reshape(n, -1), _real(lse[r], None),
                                   q[b, :n], k[b, :n], v[b, :n])
                    assert bool((out[cu[b] + n:cu[b + 1], :H4 * d] == 0).all()), (N, b)
                    assert bool((lse[cu[b] + n:cu[b + 1]] == float("inf")).all()), (N, b)
                assert bool((out[cu[B]:] == SENT).all()) and bool((lse[cu[B]:] == SENT).all()), "rows past the last image"
    wst.report()


# ------------------------------------------------------------------------------------------------------------------------------
# attention backward
# ------------------------------------------------------------------------------------------------------------------------------
def _delta(L, out, do, rows, d):
    delta = torch.zeros(out.shape[0], H4, dtype=torch.float32, device="cuda")
    L.check(L.load().vtk_attn_delta(out.data_ptr(), out.stride(0), do.data_ptr(), do.stride(0), delta.data_ptr(), rows, H4, d,
                                    L.stream_ptr()))
    return delta


def _check_grads4(wst, tag, g_rows, q, k, v, do, b_o, tau, w=None):
    n, _, d = q.shape
    g = g_rows[:, :3 * H4 * d].reshape(n, 3, H4, d)[:, :, 0::2]
    dq, bdq, dk, bdk, dv, bdv = _bwd_ref(q, k, v, do, b_o, tau, w)
    for i, (nm, ref, bd) in enumerate((("dq", dq, bdq), ("dk", dk, bdk), ("dv", dv, bdv))):
        wst.check(f"{tag} {nm}", g[:, i], ref, bd + E32 * ref.abs().max(), C_BWD)


def _do4(do, seed):
    return _four(do, 1.0, torch.Generator().manual_seed(seed)).to(BF).cuda()


BWD_CASES = [("dense", 129, None), ("dense", 1000, None), ("prefix", 127, None), ("prefix", 257, None),
             ("window", 1000, 0), ("window", 1000, 129), ("packed", 257, None), ("packed", 1000, None)]


@pytest.mark.parametrize("d", DS)
def test_attention_backward(L, d):
    """vtk_attention_bwd_bf16 (dense, prefix with poisoned dO / lse / delta past kv_len, window) and vtk_attention_bwd_packed_bf16,
    with lse and delta from the forward kernel; the gradient buffer's extra columns keep their sentinel."""
    wst = Worst(f"bwd d={d}")
    D4 = H4 * d
    for regime in ("diffuse", "late_max", "poison"):
        for layout, N, w in BWD_CASES:
            seed = _seed("hd bwd", layout, d, regime, N, w)
            lens = _lens(N) if layout in ("prefix", "packed") else [N] * (1 if layout == "window" else 2)
            B = len(lens)
            do = _grad_do(lens, N, d, seed + 2, regime != "diffuse" and layout == "prefix")
            if layout == "packed":
                q, k, v, plan, pk, cu, nv = _packed(L, regime, lens, N, d, seed, 128)
                plan_f = plan if d <= 64 else L.pack_plan(_mask(lens, N).cuda(), 16, 256)
                do_x = L.pack_rows(_do4(do, seed).view(B, N, -1), plan)
                out, lse = _fwd_packed(L, pk, plan_f, B, N, d)
                rows = pk.shape[0]
                delta = _delta(L, out, do_x, cu[B], d)
                qkv = pk
            else:
                q, k, v = _inputs(regime, lens, N, d, seed) if w is None else _window_inputs(regime, N, d, seed, w)
                qkv = _qkv4(q, k, v, seed)
                do_x = _do4(do, seed)
                mask = _mask(lens, N).cuda() if layout == "prefix" else None
                out, lse = _fwd_padded(L, qkv, B, N, d, mask, -1 if w is None else w)
                rows = B * N
                delta = _delta(L, out, do_x, rows, d)
                if mask is not None:
                    live = mask.reshape(rows, 1)
                    lse = torch.where(live, lse, torch.zeros_like(lse))
                    delta = torch.where(live, delta, torch.full_like(delta, 0.75 * POISON_V))
            g = torch.full((rows, 3 * D4 + PAD_COLS), SENT, dtype=BF, device="cuda")
            b0, g0 = qkv.data_ptr(), g.data_ptr()
            if layout == "packed":
                L.check(L.load().vtk_attention_bwd_packed_bf16(b0, b0 + 2 * D4, b0 + 4 * D4, qkv.stride(0), do_x.data_ptr(), D4,
                                                               lse.data_ptr(), delta.data_ptr(), g0, g0 + 2 * D4, g0 + 4 * D4, g.stride(0),
                                                               plan["n_valid"].data_ptr(), plan["cu"].data_ptr(), plan["cuq"].data_ptr(),
                                                               plan["grp_img"].data_ptr(), plan["grp_order"].data_ptr(), B, H4, d, rows,
                                                               plan["grp_img"].numel(), L.stream_ptr()))
                starts = cu[:B]
            else:
                kl = L.kv_len(mask) if mask is not None else None
                L.check(L.load().vtk_attention_bwd_bf16(b0, b0 + 2 * D4, b0 + 4 * D4, qkv.stride(0), do_x.data_ptr(), D4, lse.data_ptr(),
                                                        delta.data_ptr(), g0, g0 + 2 * D4, g0 + 4 * D4, g.stride(0), L.ptr(kl), B, N,
                                                        H4, d, 1 if mask is not None else 0, -1 if w is None else w, L.stream_ptr()))
                starts = [b * N for b in range(B)]
            assert bool((g[:, 3 * D4:] == SENT).all()), (layout, N, "columns past the gradients must stay untouched")
            for b, n in enumerate(lens):
                r0 = starts[b]
                if n:
                    b_o, tau = _fwd_ref(q[b, :n], k[b, :n], v[b, :n], w)[1::2]
                    _check_grads4(wst, f"{regime} {layout} N={N} w={w} img {b}", g[r0:r0 + n], q[b, :n], k[b, :n], v[b, :n], do[b, :n],
                                  b_o, tau, w)
                r1 = cu[b + 1] if layout == "packed" else r0 + N
                assert bool((g[r0 + n:r1, :3 * D4] == 0).all()), (layout, N, b, "rows past kv_len get 0 gradients")
            if layout == "packed":
                assert bool((g[cu[B]:] == SENT).all()), (N, "rows past the last image must stay untouched")
    wst.report()


# ------------------------------------------------------------------------------------------------------------------------------
# QK-norm + RoPE, attn_delta
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", [8] + DS)
def test_qk_norm_rope_and_delta(L, d):
    M, heads = 203, 5
    D = heads * d
    z = bf16_randn(M, 3 * D, seed=55 + d)
    g = torch.Generator().manual_seed(56)
    wq = (torch.rand(d, generator=g) + 0.5).to(BF).cuda()
    wk = (torch.rand(d, generator=g) + 0.5).to(BF).cuda()
    row, col = (torch.arange(M) // 9).cuda(), (torch.arange(M) % 9).cuda()
    table = L.rope_table(row, col, ae_oracle.rope_inv_freq(d).cuda(), d)
    lib, st = L.load(), L.stream_ptr()
    qkv = torch.empty(M, 3 * D, dtype=BF, device="cuda")
    L.check(lib.vtk_qk_norm_rope_fwd(z.data_ptr(), 3 * D, wq.data_ptr(), wk.data_ptr(), table.data_ptr(), qkv.data_ptr(), 3 * D, M, heads, d,
                                     1e-6, st))
    zc = z.float().cpu().reshape(1, M, 3, heads, d).requires_grad_(True)
    wqc, wkc = wq.float().cpu().requires_grad_(True), wk.float().cpu().requires_grad_(True)
    cos, sin = ae_oracle.rope_cos_sin(row.cpu()[None], col.cpu()[None], d)
    q = ae_oracle.apply_rope(ae_oracle.rms_norm(zc[:, :, 0], wqc), cos, sin)
    k = ae_oracle.apply_rope(ae_oracle.rms_norm(zc[:, :, 1], wkc), cos, sin)
    got = qkv.cpu().reshape(1, M, 3, heads, d)
    report(f"qk fwd q d={d}", got[:, :, 0], q, max_abs=6e-2, rel_fro=6e-3)
    report(f"qk fwd k d={d}", got[:, :, 1], k, max_abs=6e-2, rel_fro=6e-3)
    assert torch.equal(got[:, :, 2], z.cpu().reshape(1, M, 3, heads, d)[:, :, 2])
    # in place (the inference path of the head dims the QKV epilogue leaves raw): same bits for q / k, v untouched
    zi = z.clone()
    L.check(lib.vtk_qk_norm_rope_fwd(zi.data_ptr(), 3 * D, wq.data_ptr(), wk.data_ptr(), table.data_ptr(), zi.data_ptr(), 3 * D, M, heads, d,
                                     1e-6, st))
    assert torch.equal(zi, qkv)
    # backward
    dq, dk = bf16_randn(1, M, heads, d, seed=57).cpu().float(), bf16_randn(1, M, heads, d, seed=58).cpu().float()
    (q * dq).sum().backward(retain_graph=True)
    (k * dk).sum().backward()
    dz = torch.zeros(M, 3 * D, dtype=BF, device="cuda")
    dz.view(M, 3, heads, d)[:, 0] = dq[0].to(BF).cuda()
    dz.view(M, 3, heads, d)[:, 1] = dk[0].to(BF).cuda()
    dw = torch.zeros(2, d, dtype=torch.float32, device="cuda")
    L.check(lib.vtk_qk_norm_rope_bwd(dz.data_ptr(), 3 * D, z.data_ptr(), 3 * D, wq.data_ptr(), wk.data_ptr(), table.data_ptr(),
                                     dw.data_ptr(), M, heads, d, 1e-6, st))
    gz = zc.grad[0]
    report(f"qk bwd dq_raw d={d}", dz.view(M, 3, heads, d)[:, 0], gz[:, 0], rel_fro=1.5e-2)
    report(f"qk bwd dk_raw d={d}", dz.view(M, 3, heads, d)[:, 1], gz[:, 1], rel_fro=1.5e-2)
    report(f"qk bwd dwq d={d}", dw[0], wqc.grad, rel_fro=1.5e-2)
    report(f"qk bwd dwk d={d}", dw[1], wkc.grad, rel_fro=1.5e-2)
    # delta = sum_d dO * O per (row, head), against float64 on the same bf16 values (strided rows)
    o, dob = bf16_randn(M, D + 8, seed=59), bf16_randn(M, D + 16, seed=60)
    delta = torch.full((M, heads), SENT, dtype=torch.float32, device="cuda")
    L.check(lib.vtk_attn_delta(o.data_ptr(), o.stride(0), dob.data_ptr(), dob.stride(0), delta.data_ptr(), M, heads, d, st))
    ref = (o[:, :D].double() * dob[:, :D].double()).view(M, heads, d).sum(-1)
    bound = d * E32 * (o[:, :D].double().abs() * dob[:, :D].double().abs()).view(M, heads, d).sum(-1) * 2 + 1e-30
    assert bool(((delta.double() - ref).abs() <= bound).all()), (delta.double() - ref).abs().max().item()


@pytest.mark.parametrize("M,D,heads", [(500, 1728, 24), (333, 768, 8)])
def test_qkv_swiglu_raw_copy_head_dims(L, M, D, heads):
    """vtk_qkv_swiglu_bf16 at d = 72 and d = 96: the GEMM epilogue copies q / k raw and the QK-norm + RoPE kernel runs after it on
    the caller's stream; same gates as test_gpu_gemm.py::test_qkv_swiglu."""
    from vitok_b200.models.ae import pack_w_in
    d = D // heads
    Hf = ae_oracle.ffn_hidden(D, 2.67)
    h = bf16_randn(M, D, seed=0)
    wqkv = bf16_randn(3 * D, D, seed=1, scale=1 / math.sqrt(D))
    w1 = bf16_randn(2 * Hf, D, seed=2, scale=1 / math.sqrt(D))
    g = torch.Generator().manual_seed(3)
    nq = (torch.rand(d, generator=g) + 0.5).to(BF).cuda()
    nk = (torch.rand(d, generator=g) + 0.5).to(BF).cuda()
    side = int(math.ceil(math.sqrt(M)))
    row, col = (torch.arange(M) // side).cuda(), (torch.arange(M) % side).cuda()
    table = L.rope_table(row, col, ae_oracle.rope_inv_freq(d).cuda(), d)
    wp = pack_w_in(wqkv, w1)
    qp = wp.shape[0] - 2 * Hf
    qkv, act = L.qkv_swiglu(h, wp, D, d, Hf, qp, nq, nk, table)
    hc = h.cpu()
    r_qkv = F.linear(hc.float(), wqkv.cpu().float()).to(BF).reshape(1, M, 3, heads, d)
    q, k, v = r_qkv.unbind(2)
    cos, sin = ae_oracle.rope_cos_sin(row.cpu()[None], col.cpu()[None], d)
    q = ae_oracle.apply_rope(ae_oracle.rms_norm(q, nq.cpu()), cos, sin)
    k = ae_oracle.apply_rope(ae_oracle.rms_norm(k, nk.cpu()), cos, sin)
    got = qkv.cpu().reshape(1, M, 3, heads, d)
    report(f"qkv.q d={d}", got[:, :, 0], q.float(), max_abs=1.3e-1, rel_fro=8e-3)
    report(f"qkv.k d={d}", got[:, :, 1], k.float(), max_abs=1.3e-1, rel_fro=8e-3)
    report(f"qkv.v d={d}", got[:, :, 2], v.float(), max_abs=6e-2, rel_fro=4e-3)
    u = F.linear(hc.float(), w1.cpu().float()).to(BF)
    val, gate = u.chunk(2, dim=-1)
    report(f"swiglu act d={d}", act, (F.silu(gate) * val).float(), max_abs=1.3e-1, rel_fro=8e-3)


# ------------------------------------------------------------------------------------------------------------------------------
# AE and training
# ------------------------------------------------------------------------------------------------------------------------------
V_A = "Lw512h8-Gd3m4/2x8x8"            # the pinned golden string: encoder d = 64 (fused norm), decoder d = 72 (not fused)
V_B = "w768_d2_h8-w768_d2_h8/1x16x64"  # d = 96 at a fused-norm width
V_C = "w384_d2_h8-w384_d2_h8/1x16x64"  # d = 48
GRIDS = [(8, 8), (5, 7), (3, 10)]       # N = 64 tokens (N != heads: SURVEY A10)


def _synth_batch(P, grids, N, seed):
    g = torch.Generator().manual_seed(seed)
    B = len(grids)
    b = {"patches": torch.zeros(B, N, P), "patch_mask": torch.zeros(B, N, dtype=torch.bool),
         "row_idx": torch.zeros(B, N, dtype=torch.int64), "col_idx": torch.zeros(B, N, dtype=torch.int64),
         "orig_height": torch.tensor([gh * 16 for gh, _ in grids]), "orig_width": torch.tensor([gw * 16 for _, gw in grids])}
    for i, (gh, gw) in enumerate(grids):
        n, t = gh * gw, torch.arange(gh * gw)
        b["patches"][i, :n] = (0.5 * torch.randn(n, P, generator=g)).clamp(-1, 1)
        b["patch_mask"][i, :n] = True
        b["row_idx"][i, :n], b["col_idx"][i, :n] = t // gw, t % gw
    return b


def _cuda(batch):
    return {k: (v.cuda().to(BF) if v.dtype == torch.float32 else v.cuda()) for k, v in batch.items()}


def _ae(cfg, sd, **kw):
    import vitok_b200 as vb
    m = vb.AE(**cfg, **kw)
    m.load_state_dict(sd, strict=True)
    return m.to("cuda", BF)


@pytest.mark.parametrize("mode", ["flash", "sdpa", "sw"])
@pytest.mark.parametrize("variant", [V_A, V_B, V_C])
def test_ae_vs_oracle(variant, mode):
    """encode + decode against the fp32 CPU oracle under stress init: error <= max(2 x the reference-bf16's own error, 5e-2), the gate
    of test_gpu_ae.py::test_5b_width_shallow_vs_oracle.  flash: no mask; sdpa: masked batch (the packed path); sw: flash, window 5."""
    import vitok_b200 as vb
    cfg = vb.decode_variant(variant)
    sd = make_state_dict(ae_oracle.decode_variant(variant), seed=3, stress=True)
    backend, sw = ("flash", 5) if mode == "sw" else (mode, None)
    model = _ae(cfg, sd, attn_backend=backend, sw=sw).eval()
    batch = _synth_batch(cfg["pixels_per_token"], GRIDS, 64, seed=9)
    with torch.no_grad():
        enc = model.encode(_cuda(batch))
        dec = model.decode(enc)
    valid = batch["patch_mask"] if backend == "sdpa" else torch.ones_like(batch["patch_mask"])
    eh, dh = cfg["encoder_heads"], cfg["decoder_heads"]
    e_o = ae_oracle.encode(sd, batch, eh, attn_backend=backend, sw=sw)
    d_o = ae_oracle.decode(sd, e_o, dh, attn_backend=backend, sw=sw)
    sdb = {k: v.to(BF) for k, v in sd.items()}
    bb = {k: (v.to(BF) if v.dtype == torch.float32 else v) for k, v in batch.items()}
    e_b = ae_oracle.encode(sdb, bb, eh, attn_backend=backend, sw=sw)
    d_b = ae_oracle.decode(sdb, e_b, dh, attn_backend=backend, sw=sw)
    own_z = (e_b["z"].float() - e_o["z"])[valid].abs().max().item()
    own_p = (d_b["patches"].float() - d_o["patches"])[valid].abs().max().item()
    ma_z, _ = report(f"{variant} {mode} z", enc["z"].cpu().float()[valid], e_o["z"][valid])
    ma_p, _ = report(f"{variant} {mode} patches", dec["patches"].cpu().float()[valid], d_o["patches"][valid])
    print(f"[parity] reference-bf16 own error: z {own_z:.3e} patches {own_p:.3e}")
    assert ma_z <= max(2 * own_z, 5e-2) and ma_p <= max(2 * own_p, 5e-2)
    if backend == "sdpa":
        assert bool((dec["patches"][~batch["patch_mask"].cuda()] == 0).all())


def test_quantize_d96_ssim():
    """AE.quantize() at d = 96 (width 768, a multiple of 256): FP8 vs bf16 reconstruction SSIM >= 0.99 under the default init, the
    gate of test_gpu_fp8.py::test_reference_acceptance_gate_ssim."""
    import vitok_b200 as vb
    cfg = vb.decode_variant(V_B)
    sd = make_state_dict(ae_oracle.decode_variant(V_B), seed=0, stress=False)
    model = _ae(cfg, sd, attn_backend="flash").eval()
    b = pp_oracle.collate([pp_oracle.patchify(i, 16, 256) for i in synth_images([(256, 256)] * 4, seed=1234)])
    cb = _cuda({k: torch.from_numpy(np.asarray(v)) for k, v in b.items()})
    with torch.no_grad():
        img16 = vb.unpatchify(model.decode(model.encode(cb)), 16, max_grid_size=16).float().cpu()
        model.quantize()
        img8 = vb.unpatchify(model.decode(model.encode(cb)), 16, max_grid_size=16).float().cpu()
    assert torch.isfinite(img8).all()
    s = ae_oracle.ssim(img8, img16, data_range=2.0)
    print(f"[parity] d=96 FP8 vs bf16 SSIM {s:.5f}")
    assert s >= 0.99


@pytest.mark.parametrize("backend", ["sdpa", "flash"])
def test_graphed_ae_d72_replay_equals_eager(backend):
    """GraphedAE on the golden-string model replays bit-identically, also for another ragged batch of the same shape.  Default init:
    under the stress init some seeds drive the 24-block encoder's bf16 activations to inf, and an inf output is no test of replay."""
    import vitok_b200 as vb
    cfg = vb.decode_variant(V_A)
    sd = make_state_dict(ae_oracle.decode_variant(V_A), seed=1, stress=False)
    model = _ae(cfg, sd, attn_backend=backend).eval()
    P = cfg["pixels_per_token"]
    b1 = _cuda(_synth_batch(P, GRIDS, 64, seed=5))
    b2 = _cuda(_synth_batch(P, [(4, 4), (8, 8), (2, 9)], 64, seed=6))
    graphed = vb.GraphedAE(model, b1)
    for b in (b2, b1):
        with torch.no_grad():
            eager = model.decode(model.encode(b))
        assert torch.isfinite(eager["patches"]).all()
        assert torch.equal(graphed(b)["patches"], eager["patches"])


def _rel(got, ref):
    got, ref = got.detach().float().cpu(), ref.detach().float().cpu()
    return (torch.linalg.norm(got - ref) / torch.linalg.norm(ref).clamp_min(1e-30)).item()


@pytest.mark.parametrize("case", ["padded", "packed", "window"])
def test_training_step_d72_vs_oracle(case):
    """One training step of the golden-string model (decoder d = 72): loss and every parameter gradient against the CPU oracle's fp32
    autograd, with the gates of test_gpu_train.py (loss within 5e-3, cosine >= 0.995, rel-Fro <= 8e-2) -- sdpa on a ragged batch in
    the padded layout and with train_token_packing, and flash with a sliding window."""
    import vitok_b200 as vb
    cfg = vb.decode_variant(V_A)
    sd = make_state_dict(ae_oracle.decode_variant(V_A), seed=1, stress=True)
    backend, sw = ("flash", 5) if case == "window" else ("sdpa", None)
    model = _ae(cfg, sd, attn_backend=backend, sw=sw).train()
    model.train_token_packing = case == "packed"
    batch = _synth_batch(cfg["pixels_per_token"], GRIDS if backend == "sdpa" else [(8, 8)] * 3, 64, seed=11)
    cb = _cuda(batch)
    out = model(cb)
    loss = vb.charbonnier_loss(out["patches"], cb["patches"], cb["patch_mask"], eps=1e-3)
    loss.backward()
    sd_b = {k: v.to(BF).float() for k, v in sd.items()}
    bb = dict(batch)
    bb["patches"] = batch["patches"].to(BF).float()
    ref_loss, ref_g = ae_oracle.train_step_grads(sd_b, bb, cfg["encoder_heads"], cfg["decoder_heads"], attn_backend=backend, sw=sw)
    print(f"[parity] d=72 train step {case}: loss ours {loss.item():.6f} oracle {ref_loss.item():.6f}")
    assert abs(loss.item() - ref_loss.item()) <= 5e-3 * abs(ref_loss.item())
    worst = ("", 0.0)
    for name, p in model.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), name
        r = _rel(p.grad, ref_g[name])
        worst = max(worst, (name, r), key=lambda t: t[1])
        cos = F.cosine_similarity(p.grad.float().cpu().flatten(), ref_g[name].flatten(), dim=0).item()
        assert cos >= 0.995, (name, cos, r)
    print(f"[parity] d=72 train step {case}: worst rel-Frobenius gradient error {worst[1]:.3e} at {worst[0]}")
    assert worst[1] <= 8e-2
