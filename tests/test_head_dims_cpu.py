"""CPU-only: which head dims vtk_ae_create accepts (it only fills a host struct, no device is touched).  Supported: d % 8 == 0 and
8 <= d <= 128; anything else is VTK_ERR_UNSUPPORTED (NotImplementedError) with the supported set in the message."""
import ctypes

import pytest


def _create(cfg_dict):
    from vitok_b200 import _lib
    from vitok_b200.models.ae import _ffn_hidden
    lib = _lib.load()
    cfg = _lib.AEConfig()
    cfg.pixels_per_token, cfg.channels_per_token = cfg_dict["pixels_per_token"], cfg_dict["channels_per_token"]
    cfg.enc_width, cfg.enc_depth, cfg.enc_heads = cfg_dict["encoder_width"], cfg_dict["encoder_depth"], cfg_dict["encoder_heads"]
    cfg.enc_hidden = _ffn_hidden(cfg_dict["encoder_width"], cfg_dict["mlp_factor"])
    cfg.dec_width, cfg.dec_depth, cfg.dec_heads = cfg_dict["decoder_width"], cfg_dict["decoder_depth"], cfg_dict["decoder_heads"]
    cfg.dec_hidden = _ffn_hidden(cfg_dict["decoder_width"], cfg_dict["mlp_factor"])
    cfg.norm_eps = 1e-6
    cfg.sliding_window = 0
    h = ctypes.c_void_p()
    try:
        _lib.check(lib.vtk_ae_create(ctypes.byref(cfg), ctypes.byref(h)))
    finally:
        if h.value:
            lib.vtk_ae_destroy(h)


@pytest.mark.parametrize("variant", ["Gd4-G/1x16x64", "Lw512h8-Gd3m4/2x8x8", "Lh32-Bh16/1x16x64", "w768_d2_h8-w768_d2_h96/1x16x64"])
def test_head_dims_accepted(variant):
    import vitok_b200 as vb
    cfg = vb.decode_variant(variant)
    dims = {cfg["encoder_width"] // cfg["encoder_heads"], cfg["decoder_width"] // cfg["decoder_heads"]}
    assert all(d % 8 == 0 and 8 <= d <= 128 for d in dims), dims
    _create(cfg)


def test_g_preset_head_dim_is_72():
    import vitok_b200 as vb
    cfg = vb.decode_variant("Gd4-G/1x16x64")
    assert cfg["encoder_width"] // cfg["encoder_heads"] == 72 and cfg["decoder_width"] // cfg["decoder_heads"] == 72


@pytest.mark.parametrize("width,heads", [(576, 16), (640, 4)])   # d = 36 (not a multiple of 8), d = 160 (over 128)
def test_head_dims_refused(width, heads):
    import vitok_b200 as vb
    cfg = vb.decode_variant("Bd2-Bd2/1x16x64")
    cfg.update(decoder_width=width, decoder_heads=heads)
    with pytest.raises(NotImplementedError, match="multiples of 8 from 8 to 128"):
        _create(cfg)
