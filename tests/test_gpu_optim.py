"""FusedAdamW's gradient clipping (max_grad_norm) and EMA of the fp32 master weights (ema_decay), both inside the multi-tensor pass
(csrc/vtk_train.cu: grad_sumsq_kernel, grad_norm_finish_kernel, adamw_multi_kernel<kClip, kEma>)."""
import math

import numpy as np
import pytest
import torch

from _util import report
from oracle import pp_oracle
from oracle.make_golden import SMALL
from oracle.weights import synth_images

pytestmark = pytest.mark.gpu
BF = torch.bfloat16

# Relative error bound of FusedAdamW.grad_norm against sqrt(sum g.double()^2).  A chunk's fp32 partial sums its <= 8192 squares as
# 32 sequential fmaf per thread (+ 1 for the n % 8 tail of a tensor's last chunk), then a 5-level warp tree and a 3-level tree over
# the 8 warps: every square passes through at most k = 41 roundings, so with non-negative terms the partial's relative error is at
# most gamma_k = k u / (1 - k u), u = 2^-24.  The fp64 sum of the partials adds < 2^20 * 2^-53 (negligible), the square root halves
# the relative error, and the final fp32 rounding adds u: |norm - ref| / ref <= gamma_41 / 2 + u (+ fp64 terms) < 22 u.
NORM_RTOL = 22 * 2.0 ** -24


def _params(sizes, dtype, seed=0):
    g = torch.Generator().manual_seed(seed)
    return [torch.nn.Parameter(torch.randn(n, generator=g).to(dtype).cuda()) for n in sizes]


def _set_grads(params, seed, scales=None, dtype=None):
    g = torch.Generator().manual_seed(seed)
    for i, p in enumerate(params):
        s = 1.0 if scales is None else scales[i % len(scales)]
        p.grad = (s * torch.randn(p.shape, generator=g)).to(dtype or p.dtype).cuda()


def _ref_norm(params):
    return math.sqrt(sum(float((p.grad.double() ** 2).sum()) for p in params))


def _snapshot(opt, params):
    return [(p.detach().clone(), {k: (v.clone() if torch.is_tensor(v) else v) for k, v in opt.state[p].items()}) for p in params]


def _assert_same(a, b):
    for (pa, sa), (pb, sb) in zip(a, b):
        assert torch.equal(pa, pb)
        assert sa.keys() == sb.keys()
        for k in sa:
            assert (sa[k] == sb[k]) if not torch.is_tensor(sa[k]) else torch.equal(sa[k], sb[k]), k


# ------------------------------------------------------------------------------------------------------------------------------
# 1. the norm
# ------------------------------------------------------------------------------------------------------------------------------
SIZES = [1, 3, 8191, 8193, 5, 4099, 20000, 8192, 7, 16387]


@pytest.mark.parametrize("dtype", [BF, torch.float32])
@pytest.mark.parametrize("n_tensors", [len(SIZES), 70])
def test_grad_norm_vs_fp64(dtype, n_tensors):
    """bf16 and fp32 gradients; sizes 1, 3, 8191, 8193 and others with n % 4 != 0; 70 tensors (two launches of the norm pass);
    magnitudes over 10 decades; one gradient a view at an odd offset (the scalar path of the kernel)."""
    import vitok_b200 as vb
    sizes = [SIZES[i % len(SIZES)] for i in range(n_tensors)]
    params = _params(sizes, dtype)
    opt = vb.FusedAdamW(params, lr=0.0, max_grad_norm=float("inf"))
    _set_grads(params, 1, scales=[1.0, 1e-5, 3e4, 0.1, 1e-3])
    big = torch.randn(sizes[2] + 1, dtype=dtype, device="cuda")
    params[2].grad = big[1:]
    assert params[2].grad.data_ptr() % 16 != 0
    ref = _ref_norm(params)
    opt.step()
    got = float(opt.grad_norm)
    print(f"[parity] grad_norm {dtype} x{n_tensors}: got {got:.9e} ref {ref:.9e} rel {abs(got - ref) / ref:.3e} (bound {NORM_RTOL:.3e})")
    assert opt.grad_norm.dtype == torch.float32 and opt.grad_norm.ndim == 0 and opt.grad_norm.is_cuda
    assert abs(got - ref) <= NORM_RTOL * ref


def test_grad_norm_is_bit_identical_across_runs_and_groupings():
    import vitok_b200 as vb
    sizes = [SIZES[i % len(SIZES)] for i in range(70)]
    params = _params(sizes, BF)
    _set_grads(params, 2, scales=[1.0, 1e-3, 10.0])
    norms = []
    for groups in ([{"params": params}], [{"params": params}],
                   [{"params": params[:33]}, {"params": params[33:], "weight_decay": 0.0}],
                   [{"params": params[:1]}, {"params": params[1:65]}, {"params": params[65:]}]):
        opt = vb.FusedAdamW(groups, lr=0.0, max_grad_norm=1.0)
        opt.step()
        norms.append(opt.grad_norm.clone())
    for n in norms[1:]:
        assert torch.equal(n, norms[0])


# ------------------------------------------------------------------------------------------------------------------------------
# 2. clipping
# ------------------------------------------------------------------------------------------------------------------------------
def test_clipping_matches_torch_adamw_on_clipped_gradients():
    """K steps with clipping active vs fp32 torch.optim.AdamW fed the same gradients times a coefficient computed in fp64 (the
    tolerances of test_adamw_matches_torch)."""
    import vitok_b200 as vb
    torch.manual_seed(0)
    sizes = [5000, 333, 4097]
    p0 = [torch.randn(n) for n in sizes]
    ours = [torch.nn.Parameter(p.to(BF).cuda()) for p in p0]
    ref = [torch.nn.Parameter(p.to(BF).float()) for p in p0]
    o1 = vb.FusedAdamW(ours, lr=1e-2, betas=(0.9, 0.99), weight_decay=0.05, max_grad_norm=1.0)
    o2 = torch.optim.AdamW(ref, lr=1e-2, betas=(0.9, 0.99), weight_decay=0.05)
    for s in range(5):
        g = torch.Generator().manual_seed(s)
        gs = [((1 + s) * torch.randn(n, generator=g)).to(BF) for n in sizes]
        norm64 = math.sqrt(sum(float((x.double() ** 2).sum()) for x in gs))
        coef = min(1.0 / (norm64 + 1e-6), 1.0)
        assert coef < 0.05
        for o, r, x in zip(ours, ref, gs):
            o.grad, r.grad = x.cuda(), (x.double() * coef).float()
        o1.step(); o2.step()
        assert abs(float(o1.grad_norm) - norm64) <= NORM_RTOL * norm64
        assert o1.param_groups[0]["params"][0].grad.dtype == BF and torch.equal(ours[0].grad.cpu(), gs[0])   # .grad is not rewritten
    for i in range(len(sizes)):
        report(f"clipped adamw 5 steps (bf16 param {i})", ours[i].data, ref[i].data.to(BF), max_abs=1.6e-2, rel_fro=2e-3)
        report(f"clipped adamw 5 steps (fp32 master {i})", o1.state[ours[i]]["master"], ref[i].data, rel_fro=1e-6)
        report(f"clipped adamw exp_avg_sq {i}", o1.state[ours[i]]["exp_avg_sq"], o2.state[ref[i]]["exp_avg_sq"], rel_fro=1e-6)


@pytest.mark.parametrize("pdtype", [BF, torch.float32])
def test_unclipped_steps_are_bit_identical(pdtype):
    """A norm below max_grad_norm (coefficient 1) and max_grad_norm = inf leave masters, moments and parameters bit-identical to
    FusedAdamW without clipping."""
    import vitok_b200 as vb
    sizes = [5000, 3, 8193, 70]
    runs = []
    for kw in ({}, {"max_grad_norm": 1e6}, {"max_grad_norm": float("inf")}):
        params = _params(sizes, pdtype, seed=4)
        opt = vb.FusedAdamW(params, lr=1e-3, weight_decay=0.01, **kw)
        for s in range(3):
            _set_grads(params, 10 + s)
            opt.step()
        runs.append(_snapshot(opt, params))
        if kw:
            assert float(opt.grad_norm) < 1e6
    _assert_same(runs[0], runs[1])
    _assert_same(runs[0], runs[2])


def test_inf_gradient_gives_torch_norm_and_parameters():
    import vitok_b200 as vb
    sizes = [1000, 37]
    ours = _params(sizes, torch.float32, seed=5)
    ref = [torch.nn.Parameter(p.detach().clone()) for p in ours]
    o1 = vb.FusedAdamW(ours, lr=1e-2, weight_decay=0.0, max_grad_norm=1.0)
    o2 = torch.optim.AdamW(ref, lr=1e-2, weight_decay=0.0)
    _set_grads(ours, 6)
    ours[1].grad[5] = float("inf")
    for o, r in zip(ours, ref):
        r.grad = o.grad.clone()
    tn = torch.nn.utils.clip_grad_norm_(ref, 1.0, foreach=True)
    o1.step(); o2.step()
    assert math.isinf(float(tn)) and torch.equal(o1.grad_norm, tn)
    for o, r in zip(ours, ref):
        torch.testing.assert_close(o.detach(), r.detach(), rtol=0, atol=0, equal_nan=True)
    assert math.isnan(float(ours[1].detach()[5])) and int(torch.isnan(ours[0].detach()).sum()) == 0


# ------------------------------------------------------------------------------------------------------------------------------
# 3. EMA
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pdtype", [BF, torch.float32])
@pytest.mark.parametrize("decay", [0.999, 0.3, 0.0])
@pytest.mark.parametrize("clip", [None, 0.5])
def test_ema_is_foreach_lerp_of_the_master(pdtype, decay, clip):
    """After every step state["ema"] equals torch._foreach_lerp_(previous ema, new master, 1 - decay) bit for bit (decay 0.999 and
    0.3 take the two branches of torch's lerp, 0 gives the master); a parameter without a gradient in a step keeps its EMA."""
    import vitok_b200 as vb
    sizes = [4099, 3, 8192, 1]
    params = _params(sizes, pdtype, seed=7)
    opt = vb.FusedAdamW(params, lr=1e-2, weight_decay=0.01, max_grad_norm=clip, ema_decay=decay)
    prev = {p: p.detach().float().clone() for p in params}            # the EMA starts at the parameter's value
    for s in range(4):
        _set_grads(params, 20 + s)
        if s == 2:
            params[1].grad = None
        if s:
            prev = {p: opt.state[p]["ema"].clone() for p in params}
        opt.step()
        for p in params:
            stt = opt.state[p]
            if p.grad is None:
                assert torch.equal(stt["ema"], prev[p])
                continue
            master = stt["master"] if pdtype == BF else p.detach()
            exp = [prev[p].clone()]
            torch._foreach_lerp_(exp, [master.clone()], 1 - decay)
            assert torch.equal(stt["ema"], exp[0]), (s, int((stt["ema"] != exp[0]).sum()))
            if decay == 0.0:
                assert torch.equal(stt["ema"], master)
    assert opt.state[params[1]]["step"] == 3


# ------------------------------------------------------------------------------------------------------------------------------
# 4.-6. with the model
# ------------------------------------------------------------------------------------------------------------------------------
def _small(packed=True, seed=0):
    import vitok_b200 as vb
    torch.manual_seed(seed)
    model = vb.AE(**vb.decode_variant(SMALL), attn_backend="sdpa").train().to("cuda", BF)
    model.train_token_packing = packed
    return model


def _opt(model, **kw):
    import vitok_b200 as vb
    decay = [p for n, p in model.named_parameters() if p.ndim > 1 and "norm" not in n and "bias" not in n]
    no_decay = [p for n, p in model.named_parameters() if not (p.ndim > 1 and "norm" not in n and "bias" not in n)]
    return vb.FusedAdamW([{"params": decay, "weight_decay": 0.01}, {"params": no_decay, "weight_decay": 0.0}], lr=3e-3,
                         betas=(0.9, 0.99), **kw)


def _batch():
    imgs = [pp_oracle.patchify(i, 16, 64) for i in synth_images([(128, 128), (96, 64), (128, 112), (64, 128)], seed=3)]
    b = {k: torch.from_numpy(np.asarray(v)) for k, v in pp_oracle.collate(imgs).items()}
    return {k: (v.cuda().to(BF) if v.dtype == torch.float32 else v.cuda()) for k, v in b.items()}


def _train_step(model, opt, cb):
    import vitok_b200 as vb
    opt.zero_grad(set_to_none=True)
    out = model(cb)
    loss = vb.charbonnier_loss(out["patches"], cb["patches"], cb["patch_mask"])
    loss.backward()
    opt.step()
    return loss.detach()


def _synthetic_step(model, opt, seed):
    g = torch.Generator().manual_seed(seed)
    for p in model.parameters():
        p.grad = (1e-2 * torch.randn(p.shape, generator=g)).to(p.dtype).cuda()
    opt.step()


def _eval(model, cb):
    model.eval()
    with torch.no_grad():
        enc = model.encode(cb)
        out = (enc["z"].clone(), model.decode(enc)["patches"].clone())
    model.train()
    return out


def test_swap_ema_and_export():
    """Inside swap_ema the eval encode / decode equal those of a second model loaded with ema_state_dict(model), bit for bit; after
    exit the parameters and optimizer state are bit-identical to before entry, inference sees the training weights again, and the
    next step equals the step taken without the swap."""
    model, cb = _small(), _batch()
    opt = _opt(model, max_grad_norm=1.0, ema_decay=0.9)
    for _ in range(3):
        _train_step(model, opt, cb)
    params = list(model.parameters())
    before = _snapshot(opt, params)
    out_train = _eval(model, cb)
    with opt.swap_ema(model):
        out_ema = _eval(model, cb)
    assert not torch.equal(out_ema[1], out_train[1])
    _assert_same(_snapshot(opt, params), before)
    out_after = _eval(model, cb)
    assert torch.equal(out_after[0], out_train[0]) and torch.equal(out_after[1], out_train[1])
    ema_model = _small(seed=1)
    ema_model.load_state_dict(opt.ema_state_dict(model))
    out_ref = _eval(ema_model, cb)
    assert torch.equal(out_ema[0], out_ref[0]) and torch.equal(out_ema[1], out_ref[1])
    _synthetic_step(model, opt, 99)                                     # the step after the swap ...
    after_swap = _snapshot(opt, params)
    for p, (v, st) in zip(params, before):                              # ... vs the same step from the state before it
        p.data.copy_(v)
        opt.state[p].update({k: (x.clone() if torch.is_tensor(x) else x) for k, x in st.items()})
    _synthetic_step(model, opt, 99)
    _assert_same(_snapshot(opt, params), after_swap)


def test_checkpoint_round_trip_is_bit_identical():
    """3 steps, a state_dict round trip of model and optimizer into new objects, 3 more steps == 6 uninterrupted steps (gradients
    seeded per step, so the comparison sees the optimizer alone)."""
    model = _small()
    opt = _opt(model, max_grad_norm=0.05, ema_decay=0.99)
    ref_model = _small(seed=1)
    ref_model.load_state_dict(model.state_dict())
    ref_opt = _opt(ref_model, max_grad_norm=0.05, ema_decay=0.99)
    for s in range(3):
        _synthetic_step(model, opt, s)
        _synthetic_step(ref_model, ref_opt, s)
    model2 = _small(seed=2)
    model2.load_state_dict(model.state_dict())
    opt2 = _opt(model2, max_grad_norm=0.05, ema_decay=0.99)
    opt2.load_state_dict(opt.state_dict())
    del model, opt
    for s in range(3, 6):
        _synthetic_step(model2, opt2, s)
        _synthetic_step(ref_model, ref_opt, s)
        assert torch.equal(opt2.grad_norm, ref_opt.grad_norm)
    assert float(ref_opt.grad_norm) > 0.05                             # clipping was active
    _assert_same(_snapshot(opt2, list(model2.parameters())), _snapshot(ref_opt, list(ref_model.parameters())))


@pytest.mark.parametrize("packed", [False, True])
def test_training_with_clipping_and_ema_reduces_loss(packed):
    model, cb = _small(packed), _batch()
    opt = _opt(model, max_grad_norm=1e-3, ema_decay=0.9)
    losses, norms = [], []
    for _ in range(12):
        losses.append(float(_train_step(model, opt, cb)))
        norms.append(float(opt.grad_norm))
    print(f"[parity] {'packed' if packed else 'padded'} losses", [round(x, 4) for x in losses], "norms", [f"{x:.3g}" for x in norms])
    assert losses[-1] < 0.9 * losses[0] and all(math.isfinite(x) for x in losses)
    assert min(norms) > 1e-3                                            # every step was clipped
    for p in model.parameters():
        e = opt.state[p]["ema"]
        assert bool(torch.isfinite(e).all())


def test_frozen_encoder_only_trainable_parameters_get_ema():
    model, cb = _small(), _batch()
    for name in ("patch_embed", "encoder_blocks", "to_code"):
        getattr(model, name).requires_grad_(False)
    opt = _opt(model, max_grad_norm=1.0, ema_decay=0.99)
    _train_step(model, opt, cb)
    for n, p in model.named_parameters():
        assert ("ema" in opt.state[p]) == p.requires_grad, n
    sd = opt.ema_state_dict(model)
    for n, p in model.named_parameters():
        if not p.requires_grad:
            assert torch.equal(sd[n], p.detach()), n


def _step_kernels(opt):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        opt.step()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def test_step_kernel_lists():
    """Both options off: opt.step() launches exactly the AdamW kernels it launched before clipping and EMA existed -- one
    plain-instantiation launch per 64 tensors of each group, nothing else.  Clipping adds one norm launch per 64 tensors and the
    one-CTA finish kernel, ahead of the AdamW launches; the EMA adds no launch."""
    model, cb = _small(), _batch()
    counts = [math.ceil(len(g["params"]) / 64) for g in _opt(model).param_groups]
    n_all = math.ceil(sum(len(g["params"]) for g in _opt(model).param_groups) / 64)
    expect = {
        (None, None): ["adamw_multi_kernel<false, false>"] * sum(counts),
        (1.0, None): ["grad_sumsq_kernel"] * n_all + ["grad_norm_finish_kernel"] + ["adamw_multi_kernel<true, false>"] * sum(counts),
        (None, 0.9): ["adamw_multi_kernel<false, true>"] * sum(counts),
        (1.0, 0.9): ["grad_sumsq_kernel"] * n_all + ["grad_norm_finish_kernel"] + ["adamw_multi_kernel<true, true>"] * sum(counts),
    }
    for (clip, ema), want in expect.items():
        opt = _opt(model, max_grad_norm=clip, ema_decay=ema)
        _train_step(model, opt, cb)                                     # (state is created in the first step)
        names = _step_kernels(opt)
        got = [next(k for k in ("grad_sumsq_kernel", "grad_norm_finish_kernel", "adamw_multi_kernel<false, false>",
                                "adamw_multi_kernel<true, false>", "adamw_multi_kernel<false, true>", "adamw_multi_kernel<true, true>",
                                "?") if k in n or k == "?") for n in names]
        print(f"[parity] step kernels clip={clip} ema={ema}: {len(names)} launches")
        assert got == want, (clip, ema, names)
