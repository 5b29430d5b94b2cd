"""GPU parity: rmsnorm / rope table / casts / kv_len vs the CPU oracle."""
import pytest
import torch

from _util import bf16_randn, report
from oracle import ae_oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def L():
    from vitok_b200 import _lib
    _lib.load()
    return _lib


@pytest.mark.parametrize("M,D", [(1, 128), (1000, 1024), (4096, 3072), (77, 768)])
def test_rmsnorm(L, M, D):
    x = bf16_randn(M, D, seed=1, scale=3.0)
    w = (torch.rand(D, generator=torch.Generator().manual_seed(2)) + 0.5).to(torch.bfloat16).cuda()
    y = L.rmsnorm(x, w)
    ref = ae_oracle.rms_norm(x.cpu(), w.cpu())
    # identical rounding points: at most 1 bf16 ulp from fp32 summation order
    ma, _ = report(f"rmsnorm M={M} D={D}", y, ref.float(), rel_fro=2e-3)
    mism = (y.cpu() != ref).float().mean().item()
    print(f"[parity] rmsnorm mismatching elements: {mism:.2e}")
    assert mism < 2e-2


@pytest.mark.parametrize("d", [64, 128])
def test_rope_table(L, d):
    row = torch.arange(0, 64).repeat_interleave(64).cuda()
    col = torch.arange(0, 64).repeat(64).cuda()
    inv = ae_oracle.rope_inv_freq(d).cuda()
    M = row.numel()
    c2, s2 = L.rope_table_decode(L.rope_table(row, col, inv, d).cpu(), M, d)
    cos, sin = ae_oracle.rope_cos_sin(row.cpu(), col.cpu(), d)
    cos, sin = cos.to(torch.bfloat16), sin.to(torch.bfloat16)
    # pair-expanded layout: C2 = (c0,c0,c1,c1,...), S2 = (-s0,+s0,-s1,+s1,...)
    assert torch.equal(c2[:, 0::2], c2[:, 1::2]) and torch.equal(s2[:, 0::2], -s2[:, 1::2])
    t = torch.cat([c2[:, 0::2], s2[:, 1::2]], dim=-1)
    ref = torch.cat([cos, sin], dim=-1)
    mism = (t != ref).float().mean().item()
    print(f"[parity] rope table d={d}: mismatching bf16 entries {mism:.2e}, max_abs {(t.float() - ref.float()).abs().max():.3e}")
    assert (t.float() - ref.float()).abs().max().item() <= 2 ** -7   # never more than 1 bf16 ulp at |x|<=1
    assert mism < 5e-3


@pytest.mark.parametrize("M", [1, 33, 100])
def test_rope_table_ragged_rows(L, M):
    """M not a multiple of the 32-row group."""
    d = 64
    row = (torch.arange(M) // 7).cuda()
    col = (torch.arange(M) % 7).cuda()
    inv = ae_oracle.rope_inv_freq(d).cuda()
    c2, s2 = L.rope_table_decode(L.rope_table(row, col, inv, d).cpu(), M, d)
    cos, sin = ae_oracle.rope_cos_sin(row.cpu(), col.cpu(), d)
    assert (c2[:, 0::2].float() - cos).abs().max().item() <= 2 ** -7
    assert (s2[:, 1::2].float() - sin).abs().max().item() <= 2 ** -7


def test_casts_bit_exact(L):
    x = torch.randn(1000003, generator=torch.Generator().manual_seed(3)).cuda()
    assert torch.equal(L.cast_to_bf16(x), x.to(torch.bfloat16))


def test_kv_len(L):
    m = torch.zeros(5, 300, dtype=torch.bool)
    m[0, :300] = True
    m[1, :17] = True
    m[3, 5:9] = True          # not a prefix
    m[4, :100] = True
    m[4, 50] = False          # hole
    assert L.kv_len(m.cuda()).tolist() == [300, 17, 0, 9, 100]
