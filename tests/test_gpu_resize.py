"""GPU tests of the fused resize_to_token_budget | normalize | patchify front end (vtk_resize_patchify), against the host chain
the reference runs: to_tensor -> normalize(minus_one_to_one) -> TF.resize(BICUBIC, antialias=True) on the CPU -> patchify.

Gates: mask, index arrays and meta bit-exact; fp32 patches max-abs <= 2e-6; bf16 patches within one bf16 ulp on under 0.1 % of
the elements; images within budget bit-identical to patchify_batch without resizing."""
import ctypes

import numpy as np
import pytest
import torch

import _resize_oracle as resize_oracle
from oracle import pp_oracle

pytestmark = pytest.mark.gpu

P, T = 16, 256
# (H, W): photo sizes over budget, a 12 MP photo, a long strip, one axis unchanged, and images within budget
SIZES = [(375, 500), (480, 640), (768, 1024), (3024, 4032), (64, 4000), (500, 333), (256, 256), (200, 160), (1, 300),
         (333, 517), (263, 263), (130, 131), (1000, 700), (300, 20), (17, 4000), (96, 64), (720, 1280), (50, 120)]


def _images(sizes=SIZES, seed=0):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8) for h, w in sizes]


def _host_chain(arrs, patch=P, T_=T, out_dtype=torch.float32):
    """What preprocess runs without fusion: per image to_tensor | normalize | resize_to_token_budget on the host, then patchify."""
    import torchvision.transforms.functional as TF
    import vitok_b200 as vb
    from vitok_b200.pp.ops import resize_to_token_budget
    rs = resize_to_token_budget(patch, T_)
    imgs = [rs(TF.normalize(TF.to_tensor(a), [0.5] * 3, [0.5] * 3)) for a in arrs]
    return imgs, vb.patchify_batch(imgs, patch, T_, out_dtype, "cuda")


def _check(got, ref, out_dtype=torch.float32, max_abs=2e-6):
    for k in ("patch_mask", "row_idx", "col_idx", "time_idx", "orig_height", "orig_width", "grid_rows", "grid_cols"):
        assert torch.equal(got[k], ref[k]), k
    g, r = got["patches"].float(), ref["patches"].float()
    d = (g - r).abs()
    if out_dtype == torch.float32:
        assert d.max().item() <= max_abs, d.max().item()
    else:
        ulp = torch.where(r == 0, torch.full_like(r, 2.0 ** -133), r.abs() * 2.0 ** -7)   # bf16 spacing at |r| (upper bound)
        assert (d <= ulp).all(), d.max().item()
        assert (d > 0).float().mean().item() < 1e-3


@pytest.fixture(scope="module")
def batch():
    arrs = _images()
    imgs, ref = _host_chain(arrs)
    return arrs, imgs, ref


def test_uint8_batch_matches_host_chain(batch):
    import vitok_b200 as vb
    arrs, _, ref = batch
    got = vb.patchify_batch(arrs, P, T, torch.float32, "cuda", resize_to_budget=True)
    _check(got, ref)


def test_in_budget_images_bit_identical_to_patchify(batch):
    import vitok_b200 as vb
    arrs, _, _ = batch
    for dt in (torch.float32, torch.bfloat16):
        got = vb.patchify_batch(arrs, P, T, dt, "cuda", resize_to_budget=True)
        inb = [i for i, (h, w) in enumerate(SIZES) if pp_oracle.fit_to_token_budget(h, w, P, T) == (h, w)]
        assert len(inb) >= 4
        plain = vb.patchify_batch([arrs[i] for i in inb], P, T, dt, "cuda")
        for j, i in enumerate(inb):
            assert torch.equal(got["patches"][i], plain["patches"][j]), (SIZES[i], dt)


def test_bf16_output(batch):
    import vitok_b200 as vb
    arrs, imgs, _ = batch
    ref = vb.patchify_batch(imgs, P, T, torch.bfloat16, "cuda")
    got = vb.patchify_batch(arrs, P, T, torch.bfloat16, "cuda", resize_to_budget=True)
    _check(got, ref, torch.bfloat16)


def test_fp32_chw_input(batch):
    import torchvision.transforms.functional as TF
    import vitok_b200 as vb
    arrs, _, ref = batch
    f32 = [TF.normalize(TF.to_tensor(a), [0.5] * 3, [0.5] * 3) for a in arrs]
    _check(vb.patchify_batch(f32, P, T, torch.float32, "cuda", resize_to_budget=True), ref)
    flat, offs, sizes = vb.pack_images(f32)
    _check(vb.patchify_packed(flat.cuda(), offs, sizes, P, T, resize_to_budget=True), ref)


def test_against_torch_cuda_interpolate(batch):
    """torch's CUDA antialiased bicubic is a different implementation from its CPU kernel (which TF.resize runs on a CPU tensor)
    and differs from it by ~1.6e-4 on this batch (B200, torch 2.11); ours must be no further from it than the CPU reference is,
    plus the fp32 gate."""
    import torch.nn.functional as F
    import vitok_b200 as vb
    arrs, _, host = batch
    imgs = []
    for a in arrs:
        x = (torch.from_numpy(a).cuda().permute(2, 0, 1).float() / 255.0 - 0.5) / 0.5
        th, tw = pp_oracle.fit_to_token_budget(a.shape[0], a.shape[1], P, T)
        if (th, tw) != tuple(a.shape[:2]):
            x = F.interpolate(x[None], size=(th, tw), mode="bicubic", antialias=True, align_corners=False)[0]
        imgs.append(x.contiguous())
    ref = vb.patchify_batch(imgs, P, T, torch.float32, "cuda")
    got = vb.patchify_batch(arrs, P, T, torch.float32, "cuda", resize_to_budget=True)
    cpu_vs_cuda = (host["patches"] - ref["patches"]).abs().max().item()
    print(f"[parity] max-abs vs torch CUDA interpolate: ours {(got['patches'] - ref['patches']).abs().max().item():.3e}, "
          f"torch CPU (TF.resize) {cpu_vs_cuda:.3e}")
    _check(got, ref, max_abs=cpu_vs_cuda + 2e-6)


def test_p32_and_packed_uint8():
    import vitok_b200 as vb
    sizes = [(333, 517), (2049, 1537), (64, 64), (300, 700)]
    arrs = _images(sizes, seed=3)
    _, ref = _host_chain(arrs, 32, 64)
    flat, offs, szs = vb.pack_images(arrs)
    _check(vb.patchify_packed(flat.cuda(), offs, szs, 32, 64, resize_to_budget=True), ref)


def _raw_call(arrs, out_dtype=torch.float32, targets=None):
    """vtk_resize_patchify through the C ABI with caller-owned buffers; returns (outputs, workspace, status, launch)."""
    import vitok_b200 as vb
    from vitok_b200 import _lib
    lib = _lib.load()
    flat, offs, sizes = vb.pack_images(arrs)
    flat = flat.cuda()
    if targets is None:
        targets = [pp_oracle.fit_to_token_budget(h, w, P, T) for h, w in sizes]
    host = torch.tensor([[o, h, w, th, tw] for o, (h, w), (th, tw) in zip(offs, sizes, targets)], dtype=torch.int64)
    ws_bytes = lib.vtk_resize_patchify_workspace_bytes(ctypes.c_void_p(host.data_ptr()), len(sizes))
    B = len(sizes)
    out = {"patches": torch.empty(B, T, 3 * P * P, dtype=out_dtype, device="cuda"),
           "patch_mask": torch.empty(B, T, dtype=torch.bool, device="cuda"),
           "idx": torch.empty(3, B, T, dtype=torch.int64, device="cuda"), "meta": torch.empty(4, B, dtype=torch.int64, device="cuda")}
    tab, ws = host.cuda(), torch.zeros(ws_bytes, dtype=torch.uint8, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")

    def launch():
        _lib.check(lib.vtk_resize_patchify(flat.data_ptr(), tab.data_ptr(), 1, B, P, T, 0 if out_dtype == torch.float32 else 1,
                                           out["patches"].data_ptr(), out["patch_mask"].data_ptr(), out["idx"][0].data_ptr(),
                                           out["idx"][1].data_ptr(), out["idx"][2].data_ptr(), out["meta"].data_ptr(),
                                           ws.data_ptr(), ws_bytes, status.data_ptr(), _lib.stream_ptr()))
    launch()
    torch.cuda.synchronize()
    return out, ws, status, launch, (flat, tab)


def test_device_tables_equal_oracle_tables():
    sizes = [(375, 500), (3024, 4032), (64, 4000), (300, 20), (17, 290), (128, 128)]
    targets = [pp_oracle.fit_to_token_budget(h, w, P, T) for h, w in sizes]
    targets[3] = pp_oracle.fit_to_token_budget(300, 20, P, 16)
    targets[4] = pp_oracle.fit_to_token_budget(17, 290, P, 16)
    _, ws, status, _, _ = _raw_call(_images(sizes, seed=4), targets=targets)
    assert int(status.item()) == 0
    B = len(sizes)
    hdr = ws[:(2 * B + 3) * 8].view(torch.int64).cpu().numpy()
    assert hdr[2 * B + 2] == 1
    data = ws[((2 * B + 3) * 8 + 255) // 256 * 256:].view(torch.float32).cpu().numpy()
    checked, changed = 0, sum((h != th) + (w != tw) for (h, w), (th, tw) in zip(sizes, targets))
    for b, ((h, w), (th, tw)) in enumerate(zip(sizes, targets)):
        off = int(hdr[b])
        for n_in, n_out in ((w, tw), (h, th)):
            if n_in == n_out:
                continue
            kt = 4 * (-(-n_in // n_out)) + 1
            ent = data[off:off + n_out * (kt + 2)].reshape(kt + 2, n_out).T    # stored tap-major
            xmin, taps, wts = resize_oracle.resize_table(n_in, n_out)
            assert np.array_equal(ent[:, 0].view(np.int32), xmin) and np.array_equal(ent[:, 1].view(np.int32), taps)
            k = wts.shape[1]
            assert np.array_equal(ent[:, 2:2 + k], wts), (n_in, n_out, np.abs(ent[:, 2:2 + k] - wts).max())
            assert not ent[:, 2 + k:].any()
            off += n_out * (kt + 2)
            checked += 1
    assert checked == changed == 10


def test_cuda_graph_replay_is_bit_identical():
    arrs = _images(SIZES[:8], seed=5)
    out, _, _, launch, _ = _raw_call(arrs)
    eager = {k: v.clone() for k, v in out.items()}
    for v in out.values():
        v.zero_()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        launch()                                   # warm-up on the capture stream
        s.synchronize()
        with torch.cuda.graph(g, stream=s):
            launch()
    for v in out.values():
        v.zero_()
    g.replay()
    g.replay()
    torch.cuda.synchronize()
    for k in eager:
        assert torch.equal(out[k], eager[k]), k


def test_status_and_errors():
    import vitok_b200 as vb
    arrs = _images([(375, 500), (64, 64)], seed=6)
    with pytest.raises(RuntimeError):
        vb.patchify_batch(arrs, P, T, torch.float32, "cuda")          # the default still raises on an over-budget image
    with pytest.raises(RuntimeError):
        vb.patchify_batch(arrs, P, T, torch.float32, "cuda", resize_to_budget=False)
    with pytest.raises(RuntimeError):                                  # _fit_to_token_budget leaves 1 x 4500 at 268 patches
        vb.patchify_batch(_images([(1, 4500)]), P, T, torch.float32, "cuda", resize_to_budget=True)
    out, _, status, _, _ = _raw_call(arrs, targets=[(375, 500), (64, 64)])   # a target over budget: status 1, no tokens
    assert int(status.item()) == 1 and not out["patch_mask"][0].any() and out["patch_mask"][1].sum().item() == 16


def test_preprocess_fuse_resize_matches_host_path():
    from PIL import Image
    import vitok_b200 as vb
    pil = [Image.fromarray(a) for a in _images(SIZES[:10], seed=7)]
    pp = "to_tensor|normalize(minus_one_to_one)|resize_to_token_budget(16, 256)|patchify(16, 256)"
    ref = vb.preprocess(pil, pp, device="cuda")
    _check(vb.preprocess(pil, pp, device="cuda", fuse_resize=True), ref)
    # another (p, T) in the resize than in patchify: not fused, the host path runs
    pp2 = "to_tensor|normalize(minus_one_to_one)|resize_to_token_budget(16, 64)|patchify(16, 256)"
    a, b = vb.preprocess(pil, pp2, device="cuda"), vb.preprocess(pil, pp2, device="cuda", fuse_resize=True)
    assert all(torch.equal(a[k], b[k]) for k in a)


def test_resized_batch_through_small_ae():
    """End to end: the resized batch through a small AE encode -> decode matches the same model on the host-path batch."""
    import vitok_b200 as vb
    from oracle.weights import make_state_dict
    variant = "w128_d2_h2-w256_d3_h2/1x16x16"
    cfg = vb.decode_variant(variant)
    model = vb.AE(**cfg, attn_backend="sdpa").eval()
    model.load_state_dict(make_state_dict(cfg, seed=1, stress=True), strict=True)
    model = model.to("cuda", torch.bfloat16)
    arrs = _images(SIZES[:8], seed=8)
    _, ref = _host_chain(arrs)
    got = vb.patchify_batch(arrs, P, T, torch.float32, "cuda", resize_to_budget=True)
    with torch.no_grad():
        e0, e1 = model.encode(ref), model.encode(got)
        d0, d1 = model.decode(e0), model.decode(e1)
    valid = ref["patch_mask"]
    ez = (e1["z"].float() - e0["z"].float())[valid].abs().max().item()
    ep = (d1["patches"].float() - d0["patches"].float())[valid].abs().max().item()
    print(f"[parity] resized vs host-path batch through {variant}: z {ez:.3e} patches {ep:.3e}")
    assert ez <= 5e-2 and ep <= 5e-2
