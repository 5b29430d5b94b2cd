"""Resize-to-token-budget front end on photo-sized inputs: 64 seeded uint8 images, 16 each at 500x375, 640x480, 1024x768 and
4032x3024 (W x H), p = 16, T = 256 -- every one is over budget.

  (a) fused: patchify_packed(..., resize_to_budget=True) on the device-resident packed batch (CUDA events)
  (b) the host path preprocess runs today: PIL -> to_tensor -> normalize -> CPU bicubic resize -> fp32 H2D -> patchify
      (host clock ending in a synchronise, H2D included)
  (c) torch CUDA F.interpolate(bicubic, antialias=True) per image, then patchify_batch (CUDA events)
  (d) fused front end + 350M (Ld4-Ld24/1x16x64, bf16) encode + decode, images/s (CUDA events)

(a) is also reported as GB/s on its algorithmic bytes (uint8 pixels read, fp32 width-pass scratch written and read once,
patches written) and as a fraction of 6545.9 GB/s, the device-to-device copy rate measured on a B200 (DESIGN.md section 3.3).
The inputs (~0.7 GB of pixels) exceed the 126 MB L2.

    python tools/prof_resize.py [--reps 20] [--out profiles/resize_front_end.txt]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "vitok-release_b200")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

COPY_PEAK_GBS = 6545.9
SIZES_WH = [(500, 375), (640, 480), (1024, 768), (4032, 3024)]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as ex:  # noqa: BLE001
        pl = f"unknown ({type(ex).__name__})"
    return name, pl


def events(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps * 1e3      # us per call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--host-reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    ap.add_argument("--kernels", action="store_true", help="only (a), per kernel, under torch.profiler (a run of its own)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_resize.py needs a CUDA device")
    import torch.nn.functional as F
    from PIL import Image
    import vitok_b200 as vb
    from oracle.weights import make_state_dict
    from vitok_b200.pp.ops import _fit_to_token_budget

    P, T = 16, 256
    rng = np.random.default_rng(0)
    arrs = [rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8) for (w, h) in SIZES_WH for _ in range(16)]
    B = len(arrs)
    lines = []

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        lines.append(s)

    name, pl = card()
    emit({"card": name, "power_limit": pl, "images": B, "sizes_wh": SIZES_WH, "patch": P, "max_tokens": T})

    flat, offs, sizes = vb.pack_images(arrs)
    flat = flat.cuda()
    targets = [_fit_to_token_budget(h, w, P, T) for h, w in sizes]

    # (a) fused
    fused = lambda: vb.patchify_packed(flat, offs, sizes, P, T, resize_to_budget=True)   # noqa: E731
    if args.kernels:
        from torch.profiler import ProfilerActivity, profile
        for _ in range(3):
            fused()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                fused()
            torch.cuda.synchronize()
        for e in prof.key_averages():
            if e.device_type.name == "CUDA" and e.count:
                emit({"kernel": e.key[:90], "calls": e.count, "us_per_call": round(e.device_time_total / e.count, 1)})
        return
    us_a = events(fused, args.reps)
    px = sum(3 * h * w for h, w in sizes)
    scratch = sum(3 * h * tw * 4 for (h, w), (th, tw) in zip(sizes, targets) if tw != w)
    out = B * T * 3 * P * P * 4
    nbytes = px + 2 * scratch + out
    emit({"path": "a_fused", "us": round(us_a, 1), "images_per_s": round(B / us_a * 1e6), "alg_bytes": nbytes,
          "bytes_split": {"pixels_u8": px, "scratch_write_plus_read": 2 * scratch, "patches_f32": out},
          "GBps": round(nbytes / us_a / 1e3, 1), "frac_copy_peak": round(nbytes / us_a / 1e3 / COPY_PEAK_GBS, 3)})

    # (b) host path as preprocess runs it
    pil = [Image.fromarray(a) for a in arrs]
    pp = f"to_tensor|normalize(minus_one_to_one)|resize_to_token_budget({P}, {T})|patchify({P}, {T})"
    vb.preprocess(pil[:4], pp, device="cuda")
    torch.cuda.synchronize()
    ts = []
    for _ in range(args.host_reps):
        t0 = time.perf_counter()
        vb.preprocess(pil, pp, device="cuda")
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    us_b = min(ts) * 1e6
    emit({"path": "b_host_preprocess", "us": round(us_b), "images_per_s": round(B / us_b * 1e6, 1), "threads": torch.get_num_threads(),
          "reps_us": [round(t * 1e6) for t in ts]})

    # (c) torch CUDA interpolate + patchify_batch
    dev_u8 = [torch.from_numpy(a).cuda() for a in arrs]

    def torch_path():
        imgs = []
        for x, (th, tw) in zip(dev_u8, targets):
            f = (x.permute(2, 0, 1).float() / 255.0 - 0.5) / 0.5
            imgs.append(F.interpolate(f[None], size=(th, tw), mode="bicubic", antialias=True, align_corners=False)[0].contiguous())
        return vb.patchify_batch(imgs, P, T, torch.float32, "cuda")
    us_c = events(torch_path, max(3, args.reps // 4))
    emit({"path": "c_torch_cuda_interpolate_then_patchify", "us": round(us_c, 1), "images_per_s": round(B / us_c * 1e6)})

    # (d) fused front end + 350M encode/decode
    variant = "Ld4-Ld24/1x16x64"
    cfg = vb.decode_variant(variant)
    model = vb.AE(**cfg, attn_backend="flash").eval()
    model.load_state_dict(make_state_dict(cfg, seed=1, stress=True), strict=True)
    model = model.to("cuda", torch.bfloat16)

    def step(with_front=True, batch=None):
        d = fused() if with_front else batch
        with torch.no_grad():
            return model.decode(model.encode(d))
    b0 = fused()
    us_codec = events(lambda: step(False, b0), max(5, args.reps // 2))
    us_d = events(step, max(5, args.reps // 2))
    emit({"path": "d_fused_front_plus_350M_encode_decode", "us": round(us_d, 1), "images_per_s": round(B / us_d * 1e6),
          "codec_only_us": round(us_codec, 1), "codec_only_images_per_s": round(B / us_codec * 1e6), "variant": variant})

    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
