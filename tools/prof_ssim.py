"""Per-tile SSIM kernels (csrc/vtk_ssim.cu) vs the eager torch restatement of the same definition, and the SSIM term's cost in a
training step.

    python tools/prof_ssim.py [--out FILE] [--rounds R]

Shapes: the c3 batch (64 seeded images of 128-512 px, p = 16) with whole-image tiles; 64 x 256^2 with 4 random 128-px tiles per
image; 8 x 1024^2 at p = 32 with whole-image tiles.  Kernel times are the C entry points called back to back (the Python wrapper's
one validation sync is outside the window): CUDA events over windows of at least 0.5 s after warm-up, median of 3 windows; the
forward includes the cell map and the per-tile reduction, the backward the cell map and the zeroing of dpred.  The torch reference
is what a user would write without the kernels: an fp32 canvas gathered from the tokens under autograd, tiles cropped, a grouped
conv2d with the 11 x 11 gaussian, forward alone and forward + backward.  Algorithmic FLOPs: per window position and channel
2 * (55 + 55) for the separable moments + 3 products + ~20 for the SSIM map (forward); the backward recomputes that, ~30 for the
coefficients and 2 * 2 * 33 for the transposed gaussian.  Bytes: pred and target read once over the tiles' pixels (forward); the
backward also writes dpred and zeroes it first.  The FP32 pipe peak is SMs x 128 lanes x 2 x the max SM clock.  Then the
350M-f16x16 packed training step on the c3 batch with and without the SSIM term (w = 0.5), alternated R rounds in one process.
The card's name, power limit and max SM clock are read in the same run.
"""
import argparse
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "vitok-release_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402
import vitok_b200 as vb  # noqa: E402
from bench import c3_sizes  # noqa: E402
from oracle import pp_oracle  # noqa: E402
from oracle.weights import synth_images  # noqa: E402
from prof_train_packed import card  # noqa: E402
from vitok_b200 import _lib, train  # noqa: E402

FWD_FLOP, BWD_FLOP = 2 * 110 + 3 + 20, 2 * 110 + 3 + 20 + 30 + 132


def timed(fn, min_s=0.5, windows=3):
    """Median ms per call over `windows` CUDA-event windows of at least `min_s` seconds each, after warm-up."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    n = max(1, int(min_s * 1e3 / max(e0.elapsed_time(e1), 1e-3)) + 1)
    res = []
    for _ in range(windows):
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        res.append(e0.elapsed_time(e1) / n)
    return statistics.median(res)


def batch_of(sizes, patch):
    T = max(((h + patch - 1) // patch) * ((w + patch - 1) // patch) for h, w in sizes)
    imgs = [torch.from_numpy(i) for i in synth_images(sizes, seed=1234)]
    b = vb.patchify_batch(imgs, patch, T, out_dtype=torch.bfloat16, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(0)
    pred = (b["patches"].float() * 0.8 + 0.3 * torch.randn(b["patches"].shape, generator=g, device="cuda")).to(torch.bfloat16)
    return b, pred


def kernel_calls(b, pred, patch, tiles):
    """Closures calling vtk_ssim_fwd / vtk_ssim_bwd with the arguments vb.ssim prepares (validated once)."""
    lib = _lib.load()
    B, N, _ = pred.shape
    m8 = b["patch_mask"].contiguous().view(torch.uint8)
    row, col = b["row_idx"].contiguous(), b["col_idx"].contiguous()
    ext = torch.empty(2, dtype=torch.int32, device="cuda")
    _lib.check(lib.vtk_grid_extent(m8.data_ptr(), row.data_ptr(), col.data_ptr(), B, N, ext.data_ptr(), _lib.stream_ptr()))
    gy, gx = ext.tolist()
    th = tiles.cpu()
    train._ssim_check_tiles(th, b["orig_height"].cpu(), b["orig_width"].cpu())
    tl = tiles.to(device="cuda", dtype=torch.int32).contiguous()
    T, mh, mw = tl.shape[0], int(th[:, 3].max()), int(th[:, 4].max())
    wsb = lib.vtk_ssim_workspace_bytes(B, gy, gx, T, mh, mw)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    out = torch.empty(T, dtype=torch.float32, device="cuda")
    gout = torch.ones(T, dtype=torch.float32, device="cuda")
    dpred = torch.empty_like(pred)
    tgt = b["patches"]
    common = (pred.data_ptr(), 1, tgt.data_ptr(), 1, m8.data_ptr(), row.data_ptr(), col.data_ptr(), B, N, patch, gy, gx, tl.data_ptr(), T,
              mh, mw, 0)
    keep = (pred, tgt, m8, row, col, tl)      # the tensors behind the raw pointers of `common` live as long as the closures

    def fwd():
        assert keep
        _lib.check(lib.vtk_ssim_fwd(*common, out.data_ptr(), ws.data_ptr(), wsb, _lib.stream_ptr()))

    def bwd():
        assert keep
        _lib.check(lib.vtk_ssim_bwd(*common, gout.data_ptr(), dpred.data_ptr(), ws.data_ptr(), wsb, _lib.stream_ptr()))
    return fwd, bwd, out


def torch_reference(b, pred, patch, tiles):
    """Eager fp32 restatement: canvas gathered from the tokens (unpatchify's cell map), tiles cropped, grouped conv2d."""
    B, N, P = pred.shape
    m = b["patch_mask"].bool()
    row, col = b["row_idx"], b["col_idx"]
    gy, gx = int(row[m].max()) + 1, int(col[m].max()) + 1
    cell = torch.full((B, gy * gx), -1, dtype=torch.int64, device="cuda")
    tok = torch.arange(N, device="cuda").expand(B, N)
    cell.scatter_reduce_(1, torch.where(m, row * gx + col, torch.zeros_like(row)), torch.where(m, tok, torch.full_like(tok, -1)),
                         reduce="amax")
    cell[:, 0] = torch.where(m[:, 0], 0, -1)
    idx = cell.clamp_min(0)[:, :, None].expand(-1, -1, P)
    keep = (cell >= 0)[:, :, None].float()
    ax = torch.arange(11, dtype=torch.float32, device="cuda") - 5
    g1 = torch.exp(-(ax / 1.5) ** 2 / 2)
    g1 = g1 / g1.sum()
    k = (g1[:, None] * g1[None, :]).expand(3, 1, 11, 11).contiguous()
    tl = tiles.tolist()
    same = len({(h, w) for _, _, _, h, w in tl}) == 1

    def canvas(x):
        c = x.float().gather(1, idx) * keep
        return (c.reshape(B, gy, gx, 3, patch, patch).permute(0, 3, 1, 4, 2, 5).reshape(B, 3, gy * patch, gx * patch) + 1) / 2

    def ssim_map(a, t):
        mo = F.conv2d(torch.cat([a, t, a * a, t * t, a * t]), k, groups=3)
        ma, mb, eaa, ebb, eab = mo.split(a.shape[0])
        return ((2 * ma * mb + 1e-4) * (2 * (eab - ma * mb) + 9e-4)) / ((ma * ma + mb * mb + 1e-4) * (eaa - ma * ma + ebb - mb * mb + 9e-4))

    def fwd(p):
        cp, ct = canvas(p), canvas(b["patches"])
        if same:        # equal tiles: one batched conv
            a = torch.stack([cp[i, :, y:y + h, x:x + w] for i, y, x, h, w in tl])
            t = torch.stack([ct[i, :, y:y + h, x:x + w] for i, y, x, h, w in tl])
            return ssim_map(a, t).mean(dim=(1, 2, 3))
        return torch.stack([ssim_map(cp[i:i + 1, :, y:y + h, x:x + w], ct[i:i + 1, :, y:y + h, x:x + w]).mean() for i, y, x, h, w in tl])

    pr = pred.detach().clone().requires_grad_(True)

    def f_only():
        with torch.no_grad():
            fwd(pr)

    def f_b():
        pr.grad = None
        fwd(pr).sum().backward()
    return f_only, f_b, fwd(pr).detach()


def kernel_section(log, sms, clock_mhz):
    fp32_peak = sms * 128 * 2 * clock_mhz * 1e6
    shapes = []
    s = c3_sizes(64, 1234)
    shapes.append(("c3 batch (64 x 128-512 px), whole-image tiles", s, 16, None))
    rng = np.random.RandomState(3)
    t4 = torch.tensor([[i, int(rng.randint(0, 129)), int(rng.randint(0, 129)), 128, 128] for i in range(64) for _ in range(4)])
    shapes.append(("64 x 256^2, 4 random 128-px tiles per image", [(256, 256)] * 64, 16, t4))
    shapes.append(("8 x 1024^2 at p = 32, whole-image tiles", [(1024, 1024)] * 8, 32, None))
    log(f"FP32 pipe peak {fp32_peak / 1e12:.1f} TFLOP/s ({sms} SMs x 128 x 2 x {clock_mhz} MHz); HBM 7.7 TB/s (data sheet)")
    for name, sizes, patch, tiles in shapes:
        b, pred = batch_of(sizes, patch)
        if tiles is None:
            tiles = train._ssim_default_tiles(b["orig_height"], b["orig_width"]).cpu()
        fwd, bwd, out = kernel_calls(b, pred, patch, tiles)
        rf, rfb, ref = torch_reference(b, pred, patch, tiles)
        fwd()
        err = (out - ref).abs().max().item()
        pos = sum((h - 10) * (w - 10) for _, _, _, h, w in tiles.tolist()) * 3
        px = sum(h * w for _, _, _, h, w in tiles.tolist()) * 3
        tf, tb = timed(fwd), timed(bwd)
        trf, trfb = timed(rf), timed(rfb)
        el = pred.element_size()
        for tag, ms, fl, by in (("forward", tf, FWD_FLOP * pos, 2 * px * el),
                                ("backward", tb, BWD_FLOP * pos, 2 * px * el + 2 * pred.numel() * el)):
            t_fl, t_by = fl / fp32_peak, by / 7.7e12
            bound = "FP32 pipe" if t_fl >= t_by else "HBM"
            log(f"  {name} | {tag}: {ms * 1e3:8.1f} us | {fl / 1e9:7.2f} GFLOP {fl / ms / 1e9:6.2f} TFLOP/s | {by / 1e6:7.1f} MB "
                f"{by / ms / 1e6:7.1f} GB/s | bound by {bound}: {max(t_fl, t_by) * 1e3 / ms:.2f} of the least time")
        log(f"  {name} | torch reference: forward {trf * 1e3:8.1f} us, forward + backward {trfb * 1e3:8.1f} us | kernels "
            f"{trf / tf:.1f}x / {trfb / (tf + tb):.1f}x faster | T = {tiles.shape[0]} tiles, max |kernel - fp32 torch| = {err:.2e}")


def step_section(log, rounds):
    dev = torch.device("cuda", 0)
    cfg = vb.decode_variant("Ld4-Ld24/1x16x16")
    torch.manual_seed(0)
    with torch.device(dev):
        model = vb.AE(**cfg, attn_backend="sdpa")
    model = model.to(torch.bfloat16).train()
    model.train_token_packing = True
    opt = vb.FusedAdamW(model.parameters(), lr=1e-4, betas=(0.9, 0.99))
    b = pp_oracle.collate([pp_oracle.patchify(i, 16, 1024) for i in synth_images(c3_sizes(64, 1234), seed=1234)])
    pd = {k: torch.from_numpy(np.asarray(v)).to(dev) for k, v in b.items()}
    pd["patches"] = pd["patches"].to(torch.bfloat16)

    def step(with_ssim):
        opt.zero_grad(set_to_none=True)
        out = model(pd)
        loss = vb.charbonnier_loss(out["patches"], pd["patches"], pd["patch_mask"], eps=1e-3)
        if with_ssim:
            loss = loss + 0.5 * (1 - vb.ssim(out["patches"], pd)).mean()
        loss.backward()
        opt.step()

    times = {False: [], True: []}
    for v in (False, True):
        for _ in range(2):
            step(v)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for v in (False, True):
            torch.cuda.synchronize()
            e0.record()
            for _ in range(3):
                step(v)
            e1.record()
            torch.cuda.synchronize()
            times[v].append(e0.elapsed_time(e1) / 3)
    m0, m1 = statistics.median(times[False]), statistics.median(times[True])
    log(f"## 350M-f16x16 packed training step on the c3 batch (forward, loss, backward, FusedAdamW), {rounds} alternated rounds of 3 steps")
    log(f"  charbonnier only      : {m0:8.2f} ms/step (rounds: {', '.join(f'{t:.2f}' for t in times[False])})")
    log(f"  charbonnier + 0.5 ssim: {m1:8.2f} ms/step (rounds: {', '.join(f'{t:.2f}' for t in times[True])}) | +{m1 - m0:.2f} ms "
        f"({(m1 / m0 - 1) * 100:.1f} %)")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_ssim: needs a CUDA device")
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    c = card()
    log(f"# per-tile SSIM kernels vs eager torch, and the SSIM term in a training step; {c}; torch {torch.__version__}")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    try:
        clock = int(c.rsplit(",", 1)[1].strip().split()[0])
    except (IndexError, ValueError):
        clock = 1965
        log(f"(max SM clock not readable: FP32 peak computed at {clock} MHz)")
    kernel_section(log, sms, clock)
    step_section(log, a.rounds)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
