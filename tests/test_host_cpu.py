"""CPU-only tests: the C-ABI library loads and exports every declared symbol, host-side mirrors of the
reference interface behave like the reference, and there is no CPU fallback on the product path."""
import json
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from vitok_b200 import _lib
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "vitok_b200.h")).read()
    declared = set(re.findall(r"\b(vtk_[a-z0-9_]+)\s*\(", header))
    declared -= {"vtk_status"}
    assert declared, "no declarations parsed"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.vtk_abi_version() == 6


def test_decode_variant_matches_reference(golden_dir):
    import vitok_b200 as vb
    g = json.load(open(os.path.join(golden_dir, "variants.json")))
    for v, want in g["ok"].items():
        assert vb.decode_variant(v) == want, v
    for v, err in g["errors"].items():
        with pytest.raises(Exception) as ei:
            vb.decode_variant(v)
        assert type(ei.value).__name__ == err


def test_state_dict_names_shapes_and_init():
    import vitok_b200 as vb
    from oracle.weights import make_state_dict, state_dict_shapes
    for variant in ["Bd2-Bd4/1x16x32", "w128_d2_h2-w256_d3_h2/1x16x16"]:
        cfg = vb.decode_variant(variant)
        m = vb.AE(**cfg, variational=True, float8_mode=None)           # unknown kwargs ignored (ae.py:92)
        assert [(k, tuple(v.shape)) for k, v in m.state_dict().items()] == [(k, tuple(s)) for k, s in state_dict_shapes(cfg)]
        m.load_state_dict(make_state_dict(cfg), strict=True)
        assert float(m.decoder_blocks[0].layer_scale.gamma[0]) == pytest.approx(1e-4)
        assert len(m.encoder_blocks) == cfg["encoder_depth"] and len(m.decoder_blocks) == cfg["decoder_depth"]
    big = vb.AE(**vb.decode_variant("Ld4-Ld24/1x16x64"))
    assert len(big.state_dict()) == 232
    with pytest.raises(ValueError):
        vb.AE(encoder=False, decoder=False)
    assert vb.AE(**vb.decode_variant("Bd2-Bd4/1x16x32"), sw=0).sw is None
    enc = vb.AE(**vb.decode_variant("Bd2-Bd4/1x16x32"), decoder=False)
    assert not any(k.startswith("decoder") or k.startswith("to_pixels") for k in enc.state_dict())


def test_weight_packing_layout():
    from vitok_b200.models.ae import pack_w_in, pack_w_out
    D, Hf = 128, 336
    g = torch.Generator().manual_seed(0)
    qkv, fc1 = torch.randn(3 * D, D, generator=g), torch.randn(2 * Hf, D, generator=g)
    w = pack_w_in(qkv, fc1)
    qp = 512
    assert w.shape == (qp + 2 * Hf, D) and torch.equal(w[:3 * D], qkv) and not w[3 * D:qp].any()
    x = torch.randn(5, D, generator=g)
    u = x @ w[qp:].T                                    # packed columns: [v16 | g16] blocks
    u = u.view(5, Hf // 16, 2, 16)
    ref = x @ fc1.T
    assert torch.allclose(u[:, :, 0].reshape(5, Hf), ref[:, :Hf], atol=1e-5)
    assert torch.allclose(u[:, :, 1].reshape(5, Hf), ref[:, Hf:], atol=1e-5)
    o, f2 = torch.randn(D, D, generator=g), torch.randn(D, Hf, generator=g)
    wo = pack_w_out(o, f2)
    a, act = torch.randn(5, D, generator=g), torch.randn(5, Hf, generator=g)
    assert wo.shape == (D, 512) and not wo[:, D + Hf:].any()          # pitch padded to a multiple of 64
    assert torch.allclose(torch.cat([a, act], 1) @ wo[:, :D + Hf].T, a @ o.T + act @ f2.T, atol=1e-4)


def test_dsl_parsing_like_reference():
    """Same cases as the reference's tests/cpu/test_pp.py:94-127."""
    from vitok_b200.pp import OPS, build_transform, parse_op
    assert parse_op("flip") == ("flip", (), {})
    assert parse_op("center_crop(256)") == ("center_crop", (256,), {})
    assert parse_op("patchify(16, 256)") == ("patchify", (16, 256), {})
    assert parse_op("normalize(minus_one_to_one)") == ("normalize", ("minus_one_to_one",), {})
    assert parse_op("random_resized_crop(256, scale=(0.8, 1.0))") == ("random_resized_crop", (256,), {"scale": (0.8, 1.0)})
    with pytest.raises(ValueError):
        parse_op("")
    with pytest.raises(ValueError):
        parse_op("bad syntax(")
    with pytest.raises(KeyError):
        build_transform("to_tensor|not_an_op(3)")
    assert set(OPS) == {"center_crop", "random_resized_crop", "resize_longest_side", "resize_to_token_budget", "flip",
                        "identity", "random_choice", "to_tensor", "normalize", "patchify"}
    assert build_transform("")(5) == 5


def test_fit_to_token_budget_matches_oracle():
    from oracle.pp_oracle import fit_to_token_budget
    from vitok_b200.pp.ops import _fit_to_token_budget
    for h, w, p, t in [(640, 480, 16, 256), (256, 256, 16, 256), (1000, 37, 16, 64), (4096, 4096, 32, 1024), (17, 5000, 16, 100)]:
        assert _fit_to_token_budget(h, w, p, t) == fit_to_token_budget(h, w, p, t)


def test_collate_like_reference():
    from vitok_b200 import patch_collate_fn
    assert patch_collate_fn([]) == {}
    d = patch_collate_fn([{"a": torch.zeros(3), "n": 1, "s": "x"}, {"a": torch.ones(3), "n": 2, "s": "y"}])
    assert d["a"].shape == (2, 3) and d["n"].tolist() == [1, 2] and d["s"] == ["x", "y"]
    assert patch_collate_fn([torch.zeros(2), torch.ones(2)]).shape == (2, 2)


def test_no_cpu_fallback():
    """The product path must fail loudly without CUDA tensors; nothing routes through the oracle."""
    import vitok_b200 as vb
    cfg = vb.decode_variant("w128_d2_h2-w128_d2_h2/1x16x16")
    m = vb.AE(**cfg).eval()
    d = {"patches": torch.zeros(1, 16, 768), "row_idx": torch.zeros(1, 16, dtype=torch.long),
         "col_idx": torch.zeros(1, 16, dtype=torch.long), "patch_mask": torch.ones(1, 16, dtype=torch.bool)}
    with pytest.raises(RuntimeError):
        m.encode(d)
    with pytest.raises(RuntimeError):
        vb.patchify_batch([torch.zeros(3, 32, 32)], 16, 16, device="cpu")
    with pytest.raises(RuntimeError):
        vb.unpatchify(d, 16)
    src = ""
    pkg = os.path.join(ROOT, "vitok-release_b200", "vitok_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith(".py"):
                src += open(os.path.join(dp, f)).read()
    assert "import oracle" not in src and "from oracle" not in src


def test_pretrained_registry_and_local_safetensors_roundtrip(tmp_path):
    """vitok/pretrained.py: same registry / return shape; weights ingest from local safetensors files."""
    import json
    import os
    import torch
    import vitok_b200 as vb
    from vitok_b200 import pretrained as pt
    golden = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "variants.json")))
    assert pt.list_pretrained() == ["350M-f16x16", "350M-f16x32", "350M-f16x64", "5B-f16x16", "5B-f16x32", "5B-f16x64",
                                    "5B-f32x64", "5B-f32x128", "5B-f32x256"]
    for name in pt.list_pretrained():
        repo, files, variant = pt.get_pretrained_info(name)
        assert repo == f"philippehansen/ViTok-v2-{name}" and files == ["encoder.safetensors", "decoder.safetensors"]
        vb.decode_variant(variant)
        if variant in golden:
            assert vb.decode_variant(variant) == golden[variant]
    with pytest.raises(KeyError):
        pt.load_pretrained("1T-f1x1")
    # a registry name with a small stand-in architecture on disk (no network here)
    cfg = vb.decode_variant("w128_d2_h2-w256_d3_h2/1x16x16")
    torch.manual_seed(3)
    model = vb.AE(**cfg)
    paths = pt.save_pretrained(model, str(tmp_path), "350M-f16x16")
    assert [os.path.basename(p) for p in paths] == ["encoder.safetensors", "decoder.safetensors"]
    data = pt.load_pretrained("350M-f16x16", local_dir=str(tmp_path))
    assert data["variant"] == "Ld4-Ld24/1x16x16" and set(data) == {"variant", "encoder", "decoder"}
    fresh = vb.AE(**cfg)
    fresh.load_state_dict({**data["encoder"], **data["decoder"]})          # README.md:50-53
    for (k, a), (_, b) in zip(model.state_dict().items(), fresh.state_dict().items()):
        assert torch.equal(a, b), k
    enc_only = vb.AE(**cfg, decoder=False)                                 # README.md:68-82
    enc_only.load_state_dict(pt.load_pretrained("350M-f16x16", component="encoder", local_dir=str(tmp_path))["encoder"], strict=False)
    dec_only = vb.AE(**cfg, encoder=False)
    dec_only.load_state_dict(pt.load_pretrained("350M-f16x16", component="decoder", local_dir=str(tmp_path))["decoder"], strict=True)
    assert not any(k.startswith("decoder") for k in enc_only.state_dict()) and not any(k.startswith("encoder") for k in dec_only.state_dict())


def test_preprocess_without_patchify_behaves_like_the_reference():
    """vitok/pp/io.py:43-49 runs ANY pipeline through build_transform + patch_collate_fn and then moves dict values to the device;
    a pipeline that does not end in patchify therefore yields a stacked tensor and fails on `.items()` -- same here (no extra
    "must end with patchify" rule of our own)."""
    from PIL import Image
    import numpy as np
    import vitok_b200 as vb
    img = Image.fromarray(np.zeros((32, 32, 3), dtype=np.uint8))
    with pytest.raises(AttributeError):
        vb.preprocess([img, img], pp="to_tensor|normalize(minus_one_to_one)", device="cpu")
