"""Cost of the head dims that run on a wider kernel tile (d = 72, 96 on the d = 128 kernels) next to d = 64 and 128.

    python tools/prof_head_dims.py [--out FILE]

(i)   attention forward and backward (both passes) at d in {64, 72, 96, 128}, 16 heads, B x N = 64 x 256 and 16 x 1024, no mask:
      CUDA events over many launches, TFLOP/s on the true-d FLOPs (forward 2 matmuls of 2 N^2 d per head and image, backward 5);
(ii)  Gd4-G/1x16x64 (d = 72 on both sides) encode + decode on 64 device-resident 256 x 256 images, images/s and launches per call;
(iii) one training step (forward + backward, no optimizer) of a two-block model of the G width (1728, 24 heads of 72), 64 images of
      256 tokens.
Prints the card name and its power limit first: every number belongs to them."""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "vitok-release_b200")]
import numpy as np  # noqa: E402
import torch  # noqa: E402

BF = torch.bfloat16


def _time(fn, iters, warmup=5):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def attention(lines):
    from vitok_b200 import _lib
    lib, st = _lib.load(), _lib.stream_ptr()
    h = 16
    for B, N in ((64, 256), (16, 1024)):
        for d in (64, 72, 96, 128):
            D = h * d
            g = torch.Generator().manual_seed(d)
            qkv = torch.randn(B * N, 3 * D, generator=g).to(BF).cuda()
            do = torch.randn(B * N, D, generator=g).to(BF).cuda()
            out = torch.empty(B * N, D, dtype=BF, device="cuda")
            lse = torch.empty(B * N, h, device="cuda")
            delta = torch.empty(B * N, h, device="cuda")
            dqkv = torch.empty(B * N, 3 * D, dtype=BF, device="cuda")
            b0, g0 = qkv.data_ptr(), dqkv.data_ptr()

            def fwd():
                _lib.check(lib.vtk_attention_bf16(b0, b0 + 2 * D, b0 + 4 * D, 3 * D, out.data_ptr(), D, None, B, N, h, d, 0, -1,
                                                  lse.data_ptr(), st))

            def bwd():
                _lib.check(lib.vtk_attention_bwd_bf16(b0, b0 + 2 * D, b0 + 4 * D, 3 * D, do.data_ptr(), D, lse.data_ptr(), delta.data_ptr(),
                                                      g0, g0 + 2 * D, g0 + 4 * D, 3 * D, None, B, N, h, d, 0, -1, st))
            fwd()
            _lib.check(lib.vtk_attn_delta(out.data_ptr(), D, do.data_ptr(), D, delta.data_ptr(), B * N, h, d, st))
            t_f = _time(fwd, 200)
            t_b = _time(bwd, 100)
            fl = 4.0 * N * N * d * h * B
            lines.append(f"attention B={B:3d} N={N:5d} h={h} d={d:3d}: forward {t_f * 1e3:8.1f} us {fl / t_f / 1e9:7.1f} TFLOP/s | "
                         f"backward {t_b * 1e3:8.1f} us {2.5 * fl / t_b / 1e9:7.1f} TFLOP/s")
            print(lines[-1], flush=True)


def codec(lines):
    import vitok_b200 as vb
    from oracle import ae_oracle, pp_oracle
    from oracle.weights import make_state_dict, synth_images
    variant = "Gd4-G/1x16x64"
    cfg = vb.decode_variant(variant)
    model = vb.AE(**cfg, attn_backend="flash").eval()
    model.load_state_dict(make_state_dict(ae_oracle.decode_variant(variant), seed=0), strict=True)
    model = model.to("cuda", BF)
    b = pp_oracle.collate([pp_oracle.patchify(i, 16, 256) for i in synth_images([(256, 256)] * 64, seed=1)])
    cb = {k: torch.from_numpy(np.asarray(v)).cuda() for k, v in b.items()}
    cb["patches"] = cb["patches"].to(BF)

    def run():
        with torch.no_grad():
            model.decode(model.encode(cb))
    ms = _time(run, 20, warmup=3)
    with torch.no_grad():
        model.encode(cb)
        n_enc = model.last_launch_count
        model.decode(model.encode(cb))
        n_dec = model.last_launch_count
    lines.append(f"{variant} encode+decode, 64 x 256^2 images (N = 256), flash: {ms:.2f} ms per call, {64 / ms * 1e3:.1f} images/s; "
                 f"launches: encode {n_enc}, decode {n_dec}")
    print(lines[-1], flush=True)


def train_step(lines):
    import vitok_b200 as vb
    from oracle import ae_oracle
    from oracle.weights import make_state_dict
    variant = "w1728_d1_h24-w1728_d1_h24/1x16x64"
    cfg = vb.decode_variant(variant)
    model = vb.AE(**cfg, attn_backend="flash").train()
    model.load_state_dict(make_state_dict(ae_oracle.decode_variant(variant), seed=0), strict=True)
    model = model.to("cuda", BF)
    B, N = 64, 256
    g = torch.Generator().manual_seed(2)
    t = torch.arange(N)
    cb = {"patches": (0.5 * torch.randn(B, N, cfg["pixels_per_token"], generator=g)).to(BF).cuda(),
          "patch_mask": torch.ones(B, N, dtype=torch.bool, device="cuda"),
          "row_idx": (t // 16).repeat(B, 1).cuda(), "col_idx": (t % 16).repeat(B, 1).cuda()}

    def step():
        for p in model.parameters():
            p.grad = None
        out = model(cb)
        vb.charbonnier_loss(out["patches"], cb["patches"], cb["patch_mask"], eps=1e-3).backward()
    ms = _time(step, 20, warmup=3)
    lines.append(f"training step (forward + backward) {variant}, {B} x {N} tokens: {ms:.2f} ms, {B / ms * 1e3:.1f} images/s")
    print(lines[-1], flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("prof_head_dims: needs a CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    lines = [f"device: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {q.stdout.strip() or 'unavailable'}"]
    print(lines[0], flush=True)
    attention(lines)
    codec(lines)
    train_step(lines)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
