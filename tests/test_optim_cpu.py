"""FusedAdamW's host-side surface without a GPU: argument validation of max_grad_norm / ema_decay, the one-device rule of
clipping, fp32 state across load_state_dict, and the EMA export / swap (pure tensor plumbing on optimizer state set by hand)."""
import math

import pytest
import torch

import vitok_b200 as vb

BF = torch.bfloat16


def _p(n=6, dtype=BF, device="cpu"):
    return torch.nn.Parameter(torch.linspace(-1, 1, n).to(device=device, dtype=dtype))


@pytest.mark.parametrize("bad", [1.0, 1.5, -0.1, float("nan"), float("inf"), True, "0.99", [0.9]])
def test_ema_decay_out_of_range_raises(bad):
    with pytest.raises(ValueError):
        vb.FusedAdamW([_p()], ema_decay=bad)


@pytest.mark.parametrize("bad", [0.0, -1.0, float("nan"), float("-inf"), False, "1.0"])
def test_max_grad_norm_invalid_raises(bad):
    with pytest.raises(ValueError):
        vb.FusedAdamW([_p()], max_grad_norm=bad)


def test_valid_arguments_are_kept():
    opt = vb.FusedAdamW([_p()], max_grad_norm=float("inf"), ema_decay=0)
    assert opt.max_grad_norm == math.inf and opt.ema_decay == 0.0 and opt.grad_norm is None
    opt = vb.FusedAdamW([_p()], max_grad_norm=1, ema_decay=0.9999)
    assert opt.max_grad_norm == 1.0 and opt.ema_decay == 0.9999
    opt = vb.FusedAdamW([_p()])
    assert opt.max_grad_norm is None and opt.ema_decay is None


def test_clipping_rejects_parameters_on_two_devices():
    a, b = _p(), _p(device="meta")
    vb.FusedAdamW([a, b])                                          # without clipping: allowed
    with pytest.raises(ValueError, match="one device"):
        vb.FusedAdamW([a, b], max_grad_norm=1.0)
    opt = vb.FusedAdamW([a], max_grad_norm=1.0)
    with pytest.raises(ValueError, match="one device"):
        opt.add_param_group({"params": [b]})


def _model():
    m = torch.nn.Sequential(torch.nn.Linear(3, 4), torch.nn.LayerNorm(4))
    m[0].to(BF)                                                    # a bf16 layer and an fp32 layer
    return m


def _fake_state(opt, m, ema=True):
    """State as FusedAdamW.step leaves it: bf16 parameters equal bf16(master)."""
    g = torch.Generator().manual_seed(0)
    for p in m.parameters():
        st = opt.state[p]
        st["step"] = 3
        if p.dtype == BF:
            st["master"] = p.detach().float() + 1e-4 * torch.randn(p.shape, generator=g)
            p.data.copy_(st["master"])
        st["exp_avg"] = torch.randn(p.shape, generator=g)
        st["exp_avg_sq"] = torch.rand(p.shape, generator=g)
        if ema:
            st["ema"] = p.detach().float() + torch.randn(p.shape, generator=g)


def test_load_state_dict_keeps_fp32_state():
    m = _model()
    opt = vb.FusedAdamW(m.parameters(), ema_decay=0.99)
    _fake_state(opt, m)
    sd = opt.state_dict()
    m2 = _model()
    opt2 = vb.FusedAdamW(m2.parameters(), ema_decay=0.99)
    opt2.load_state_dict(sd)
    for p, p2 in zip(m.parameters(), m2.parameters()):
        for k, v in opt.state[p].items():
            v2 = opt2.state[p2][k]
            if k == "step":
                assert v2 == v
            else:
                assert v2.dtype == torch.float32 and torch.equal(v2, v), k
                assert v2.data_ptr() != v.data_ptr()


def test_ema_state_dict_and_swap_without_ema_raise():
    m = _model()
    opt = vb.FusedAdamW(m.parameters())
    with pytest.raises(ValueError, match="ema_decay"):
        opt.ema_state_dict(m)
    with pytest.raises(ValueError, match="ema_decay"):
        with opt.swap_ema(m):
            pass


def test_ema_state_dict_casts_and_keeps_parameters_without_state():
    m = _model()
    opt = vb.FusedAdamW(m.parameters(), ema_decay=0.9)
    _fake_state(opt, m)
    frozen = m[1].bias
    del opt.state[frozen]                                           # a parameter that never got optimizer state
    sd = opt.ema_state_dict(m)
    assert list(sd) == list(m.state_dict())
    for n, p in m.named_parameters():
        if p is frozen:
            assert torch.equal(sd[n], p.detach())
        else:
            assert sd[n].dtype == p.dtype and torch.equal(sd[n], opt.state[p]["ema"].to(p.dtype))
            assert sd[n].data_ptr() != opt.state[p]["ema"].data_ptr()


def test_swap_ema_round_trip():
    m = _model()
    opt = vb.FusedAdamW(m.parameters(), ema_decay=0.9)
    _fake_state(opt, m)
    before = {n: p.detach().clone() for n, p in m.named_parameters()}
    emas = {n: opt.state[p]["ema"].clone() for n, p in m.named_parameters()}
    versions = {n: p._version for n, p in m.named_parameters()}
    with opt.swap_ema(m):
        for n, p in m.named_parameters():
            assert torch.equal(p.detach(), emas[n].to(p.dtype)), n
            assert p._version > versions[n]
    for n, p in m.named_parameters():
        assert torch.equal(p.detach(), before[n]), n
        assert torch.equal(opt.state[p]["ema"], emas[n]), n
    with pytest.raises(RuntimeError, match="inside"):              # an exception inside the block still restores the weights
        with opt.swap_ema(m):
            raise RuntimeError("inside")
    for n, p in m.named_parameters():
        assert torch.equal(p.detach(), before[n]), n
