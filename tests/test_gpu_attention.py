"""GPU parity: tcgen05 varlen attention vs the CPU oracle."""
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


def _ref(qkv, B, N, heads, d, mask, window=None):
    t = qkv.cpu().reshape(B, N, 3, heads, d)
    q, k, v = t.unbind(2)
    return ae_oracle.attention_core(q, k, v, mask.cpu() if mask is not None else None, window).reshape(B * N, heads * d)


@pytest.mark.parametrize("B,N,heads,d", [(2, 128, 2, 64), (2, 256, 4, 64), (1, 1024, 2, 64), (2, 256, 2, 128),
                                         (1, 1024, 3, 128), (3, 64, 2, 64), (2, 200, 2, 64), (1, 384, 1, 128)])
def test_attention_dense(L, B, N, heads, d):
    qkv = bf16_randn(B * N, 3 * heads * d, seed=40)
    out = L.attention(qkv, B, N, heads, d, None)
    report(f"attn dense B={B} N={N} h={heads} d={d}", out, _ref(qkv, B, N, heads, d, None).float(), max_abs=3e-2, rel_fro=1e-2)


@pytest.mark.parametrize("N,heads,d,lens", [(256, 2, 64, [256, 100, 1, 129]), (1024, 2, 64, [64, 1024, 600, 130]),
                                            (512, 2, 128, [512, 77, 256, 300]), (64, 2, 64, [24, 64, 32])])
def test_attention_prefix_mask(L, N, heads, d, lens):
    B = len(lens)
    qkv = bf16_randn(B * N, 3 * heads * d, seed=41)
    mask = torch.zeros(B, N, dtype=torch.bool)
    for b, n in enumerate(lens):
        mask[b, :n] = True
    out = L.attention(qkv, B, N, heads, d, mask.cuda())
    ref = _ref(qkv, B, N, heads, d, mask)
    report(f"attn masked N={N} d={d}", out, ref.float(), max_abs=3e-2, rel_fro=1e-2)
    # padded query rows are defined as 0 here
    assert out.cpu().reshape(B, N, -1)[~mask].abs().max().item() == 0.0


def test_attention_general_mask(L):
    """A mask with holes runs on the packed layout, as the model runs it: pack_plan -> pack_rows -> attention_packed ->
    unpack_rows (masked tokens read 0, like the oracle's masked query rows)."""
    B, N, heads, d = 2, 256, 2, 64
    qkv = bf16_randn(B * N, 3 * heads * d, seed=42)
    g = torch.Generator().manual_seed(5)
    mask = torch.rand(B, N, generator=g) > 0.4
    plan = L.pack_plan(mask.cuda())
    packed = L.attention_packed(L.pack_rows(qkv.view(B, N, -1), plan), plan, B, N, heads, d)
    out = L.unpack_rows(packed, plan, B, N).view(B * N, heads * d)
    report("attn general mask", out, _ref(qkv, B, N, heads, d, mask).float(), max_abs=3e-2, rel_fro=1e-2)


def test_attention_rejects_mask_with_holes(L):
    """The padded layout masks keys by length only: a mask with holes is refused (it runs on the packed layout instead)."""
    B, N, heads, d = 2, 256, 2, 64
    qkv = bf16_randn(B * N, 3 * heads * d, seed=42)
    mask = torch.zeros(B, N, dtype=torch.bool)
    mask[:, :100] = True
    mask[1, 50] = False
    with pytest.raises(ValueError, match="prefix mask"):
        L.attention(qkv, B, N, heads, d, mask.cuda())


def test_masked_equals_unpadded(L):
    """Property (SURVEY 7.5): a padded image's valid rows == the same image run alone without padding."""
    heads, d, n = 2, 64, 100
    small = bf16_randn(n, 3 * heads * d, seed=43)
    alone = L.attention(small.contiguous(), 1, n, heads, d, None)
    N = 256
    padded = torch.zeros(N, 3 * heads * d, dtype=torch.bfloat16, device="cuda")
    padded[:n] = small
    padded[n:] = bf16_randn(N - n, 3 * heads * d, seed=44)   # garbage in the padding must not matter
    mask = torch.zeros(1, N, dtype=torch.bool)
    mask[0, :n] = True
    out = L.attention(padded, 1, N, heads, d, mask.cuda())
    assert torch.equal(out[:n], alone)


@pytest.mark.parametrize("B,N,heads,d,w", [(2, 256, 2, 64, 16), (1, 1024, 2, 64, 100), (1, 1024, 2, 128, 128), (2, 512, 2, 128, 1),
                                           (1, 640, 2, 64, 0), (1, 300, 2, 64, 37), (1, 1024, 1, 64, 5000), (1, 2048, 1, 128, 200)])
def test_attention_sliding_window(L, B, N, heads, d, w):
    """AE(sw=w) with the flash backend: |i - j| <= w (attention.py:113-116)."""
    qkv = bf16_randn(B * N, 3 * heads * d, seed=45)
    out = L.attention(qkv, B, N, heads, d, None, window=w)
    report(f"attn window={w} N={N} d={d}", out, _ref(qkv, B, N, heads, d, None, w).float(), max_abs=3e-2, rel_fro=1e-2)


@pytest.mark.parametrize("N,heads,d,w", [(512, 2, 64, 64), (1024, 2, 128, 100), (1024, 2, 64, -1),
                                         # high-resolution decode (SURVEY 8f N2): 2048 px / 4096 px at p = 16 with a sliding window
                                         (16384, 2, 64, 1024), (65536, 1, 128, 2048)])
def test_attention_vs_flash_attn_library(L, N, heads, d, w):
    """The reference's flash backend IS flash_attn_func (third-party, pinned 2.8.3 in scripts/modal/modal_config.py);
    when it is importable on the GPU box, compare against it directly, with and without window_size."""
    fa = pytest.importorskip("flash_attn")
    B = 2 if N <= 4096 else 1
    qkv = bf16_randn(B * N, 3 * heads * d, seed=46)
    out = L.attention(qkv, B, N, heads, d, None, window=w)
    q, k, v = qkv.reshape(B, N, 3, heads, d).unbind(2)
    try:
        ref = fa.flash_attn_func(q.contiguous(), k.contiguous(), v.contiguous(), window_size=(w, w))
    except RuntimeError as e:   # no kernel image for this device in the installed wheel
        pytest.skip(f"flash_attn cannot run here: {e}")
    report(f"attn vs flash_attn window={w} N={N} d={d}", out, ref.reshape(B * N, heads * d).float(), max_abs=2e-2, rel_fro=6e-3)
