"""CPU-only: the backward work list of the training step (vitok_b200.train._grad_plan) -- which blocks keep activations, how deep each
block's backward goes and which weight-gradient GEMMs run -- for frozen parameters and single-half models, on SMALL and on the 350M
shape.  The model is built on the meta device: only parameter names and requires_grad are read."""
import pytest
import torch

SMALL = "w128_d2_h2-w256_d3_h2/1x16x16"
M350 = "Ld4-Ld24/1x16x16"
ALL_W = (True, True, True, True)
NO_W = (False, False, False, False)


def _model(variant, **kw):
    import vitok_b200 as vb
    with torch.device("meta"):
        return vb.AE(**vb.decode_variant(variant), **kw)


def _plan(model, input_grad=False):
    from vitok_b200.train import _grad_plan
    needs = {n: p.requires_grad for n, p in model.named_parameters()}
    return _grad_plan(needs, {s[0]: len(s[3]) for s in model._sides()}, input_grad)


def _depths(model):
    return model.encoder_depth, model.decoder_depth


@pytest.mark.parametrize("variant", [SMALL, M350])
def test_all_trainable_is_the_full_plan(variant):
    m = _model(variant)
    de, dd = _depths(m)
    p = _plan(m)
    assert p[0].stages == (3,) * de and p[0].wgrads == (ALL_W,) * de and p[0].save_from == 0
    assert p[1].stages == (3,) * dd and p[1].wgrads == (ALL_W,) * dd and p[1].save_from == 0
    assert p[0].top and p[1].top and p[1].dinput and not p[0].dinput
    assert p[0].embed == p[0].head == p[1].embed == p[1].head == (True, True)
    assert _plan(m, input_grad=True)[0].dinput


@pytest.mark.parametrize("variant", [SMALL, M350])
def test_frozen_encoder(variant):
    m = _model(variant)
    for mod in (m.patch_embed, m.encoder_blocks, m.to_code):
        mod.requires_grad_(False)
    de, dd = _depths(m)
    p = _plan(m)
    assert p[0].stages == (0,) * de and p[0].wgrads == (NO_W,) * de and p[0].save_from == de
    assert not p[0].top and p[0].embed == p[0].head == (False, False)
    assert not p[1].dinput                                        # the decoder_embed dgrad is skipped
    assert p[1].stages == (3,) * dd and p[1].wgrads == (ALL_W,) * dd and p[1].save_from == 0
    # patches requiring grad bring the whole encoder backward back, with no encoder wgrad
    q = _plan(m, input_grad=True)
    assert q[1].dinput and q[0].top and q[0].dinput and q[0].stages == (3,) * de and q[0].wgrads == (NO_W,) * de


@pytest.mark.parametrize("variant", [SMALL, M350])
@pytest.mark.parametrize("norm1", [False, True])
def test_only_last_decoder_block_trainable(variant, norm1):
    m = _model(variant)
    m.requires_grad_(False)
    last = m.decoder_blocks[-1]
    for mod in (last.attn.qkv_proj, last.attn.out_proj, last.ffn, last.attn.norm_q, last.attn.norm_k, last.layer_scale):
        mod.requires_grad_(True)
    last.norm1.requires_grad_(norm1)
    de, dd = _depths(m)
    p = _plan(m)
    assert p[0].stages == (0,) * de and p[0].save_from == de and not p[0].top
    assert not p[1].dinput and p[1].embed == (False, False) and p[1].head == (False, False) and p[1].top
    assert p[1].save_from == dd - 1
    assert p[1].stages == (0,) * (dd - 1) + ((3 if norm1 else 2),)     # the dgrad to h and rmsnorm_bwd only for norm1's gradient
    assert p[1].wgrads == (NO_W,) * (dd - 1) + (ALL_W,)


def test_last_block_stage_follows_its_deepest_trainable_parameter():
    m = _model(SMALL)
    m.requires_grad_(False)
    last = m.decoder_blocks[-1]
    last.attn.out_proj.requires_grad_(True)
    assert _plan(m)[1].stages[-1] == 1 and _plan(m)[1].wgrads[-1] == (False, False, True, False)
    last.layer_scale.requires_grad_(True)
    assert _plan(m)[1].stages[-1] == 1
    last.attn.norm_k.requires_grad_(True)
    assert _plan(m)[1].stages[-1] == 2 and _plan(m)[1].wgrads[-1] == (False, False, True, False)
    last.ffn.fc1.requires_grad_(True)
    assert _plan(m)[1].stages[-1] == 2 and _plan(m)[1].wgrads[-1] == (False, True, True, False)


@pytest.mark.parametrize("variant", [SMALL, M350])
def test_only_patch_embed_trainable(variant):
    m = _model(variant)
    m.requires_grad_(False)
    m.patch_embed.requires_grad_(True)
    de, dd = _depths(m)
    p = _plan(m)
    for s, depth in ((0, de), (1, dd)):
        assert p[s].stages == (3,) * depth and p[s].wgrads == (NO_W,) * depth and p[s].save_from == 0 and p[s].top
    assert p[1].dinput and p[1].embed == p[1].head == (False, False) and p[0].head == (False, False)
    assert p[0].embed == (True, True) and not p[0].dinput


@pytest.mark.parametrize("variant", [SMALL, M350])
def test_decoder_only_model(variant):
    m = _model(variant, encoder=False)
    dd = m.decoder_depth
    p = _plan(m)
    assert set(p) == {1} and not p[1].dinput and p[1].stages == (3,) * dd and p[1].save_from == 0
    assert _plan(m, input_grad=True)[1].dinput                    # z requires grad: the decoder_embed dgrad runs
    # frozen decoder_embed and first block, z without grad: block 0 needs no input gradient
    m.decoder_embed.requires_grad_(False)
    m.decoder_blocks[0].requires_grad_(False)
    p = _plan(m)
    assert p[1].stages[0] == 0 and p[1].save_from == 1 and p[1].stages[1:] == (3,) * (dd - 1)
    assert p[1].stages[1] == 3                                    # norm1 of block 1 is trainable


@pytest.mark.parametrize("variant", [SMALL, M350])
def test_encoder_only_model(variant):
    m = _model(variant, decoder=False)
    de = m.encoder_depth
    p = _plan(m)
    assert set(p) == {0} and p[0].stages == (3,) * de and not p[0].dinput and p[0].head == (True, True)
    assert _plan(m, input_grad=True)[0].dinput


def test_mixed_subset():
    """The subset of the GPU test: decoder block 0, every norm weight, patch_embed and to_code.bias frozen."""
    m = _model(SMALL)
    m.decoder_blocks[0].requires_grad_(False)
    for n, p in m.named_parameters():
        if "norm" in n:
            p.requires_grad_(False)
    m.patch_embed.requires_grad_(False)
    m.to_code.bias.requires_grad_(False)
    p = _plan(m)
    # encoder block 0 still has trainable matrices but nothing below it: stage 2 (qkv / fc1 wgrads), no input gradient
    assert p[0].stages == (2, 3) and p[0].save_from == 0 and p[0].wgrads == (ALL_W, ALL_W) and not p[0].dinput
    assert p[0].head == (True, False) and p[0].embed == (False, False)
    assert p[1].dinput and p[1].stages == (3, 3, 3) and p[1].wgrads == (NO_W, ALL_W, ALL_W)
