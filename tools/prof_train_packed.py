"""Training step on packed NaFlex rows (AE.train_token_packing = True) vs the padded step, on masked sdpa batches.

    python tools/prof_train_packed.py [--out FILE] [--rounds R]

Two workloads:
  * 350M-f16x16 (Ld4-Ld24/1x16x16) on the c3 batch: bench.c3_sizes(64, 1234), max_tokens = 1024, p = 16;
  * 5B (Td4-T/1x32x256, p = 32) on 8 images of seeded sizes in [512, 1024]^2, max_tokens = 1024.
Whole steps (forward, Charbonnier loss, backward, FusedAdamW) are timed with CUDA events after warm-up, padded and packed
alternated R times in this one process.  Reported per layout: ms/step (median of the rounds), images/s, valid tokens/s, peak
allocated memory of one step, the GEMM row count (B * N padded, cu[B] packed), and the device time of the attention backward kernels
of one step from torch.profiler (a separate, profiled step).  The card's name and power limit are read in the same run.
"""
import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "vitok-release_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import vitok_b200 as vb  # noqa: E402
from bench import c3_sizes  # noqa: E402
from oracle import pp_oracle  # noqa: E402
from oracle.weights import synth_images  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

WORKLOADS = {
    "350M-f16x16 c3": ("Ld4-Ld24/1x16x16", lambda: c3_sizes(64, 1234), 16, 1024, 3),
    "5B p32 mixed 512-1024": ("Td4-T/1x32x256", lambda: [(int(h), int(w)) for h, w in np.random.RandomState(7).randint(512, 1025, size=(8, 2))],
                              32, 1024, 2),
}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as ex:  # noqa: BLE001
        pl = f"unavailable ({type(ex).__name__})"
    return f"{name}, power limit / max SM clock: {pl}"


def run(tag, variant, sizes, patch, T, steps_per_round, rounds, log):
    dev = torch.device("cuda", 0)
    cfg = vb.decode_variant(variant)
    torch.manual_seed(0)
    with torch.device(dev):
        model = vb.AE(**cfg, attn_backend="sdpa")
    model = model.to(torch.bfloat16).train()
    decay = [p for n, p in model.named_parameters() if not (p.ndim <= 1 or "bias" in n or "norm" in n)]
    no_decay = [p for n, p in model.named_parameters() if (p.ndim <= 1 or "bias" in n or "norm" in n)]
    opt = vb.FusedAdamW([{"params": decay, "weight_decay": 0.01}, {"params": no_decay, "weight_decay": 0.0}], lr=1e-4, betas=(0.9, 0.99))
    b = pp_oracle.collate([pp_oracle.patchify(i, patch, T) for i in synth_images(sizes, seed=1234)])
    pd = {k: torch.from_numpy(np.asarray(v)).to(dev) for k, v in b.items()}
    pd["patches"] = pd["patches"].to(torch.bfloat16)
    B, N = pd["patch_mask"].shape
    n_valid = int(pd["patch_mask"].sum())
    m_packed = int(((pd["patch_mask"].sum(1) + 15) // 16 * 16).sum())

    def step():
        opt.zero_grad(set_to_none=True)
        out = model(pd)
        loss = vb.charbonnier_loss(out["patches"], pd["patches"], pd["patch_mask"], eps=1e-3)
        loss.backward()
        opt.step()
        return loss

    times = {False: [], True: []}
    peak = {}
    for packed in (False, True):             # warm-up of both layouts, then the peak memory of one step
        model.train_token_packing = packed
        for _ in range(2):
            step()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        step()
        torch.cuda.synchronize()
        peak[packed] = (torch.cuda.max_memory_allocated() - base) / 2**30
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for packed in (False, True):
            model.train_token_packing = packed
            torch.cuda.synchronize()
            e0.record()
            for _ in range(steps_per_round):
                step()
            e1.record()
            torch.cuda.synchronize()
            times[packed].append(e0.elapsed_time(e1) / steps_per_round)
    attn_bwd = {}
    for packed in (False, True):
        model.train_token_packing = packed
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step()
            torch.cuda.synchronize()
        ev = [r for r in prof.key_averages() if "attn_bwd_kernel" in r.key]
        attn_bwd[packed] = (sum(r.device_time_total for r in ev) / 1e3, sum(r.count for r in ev))
    log(f"## {tag}: {variant}, B = {B}, N = {N}, {n_valid} valid tokens ({n_valid / (B * N):.3f} of B*N), sdpa + patch_mask")
    for packed in (False, True):
        ms = statistics.median(times[packed])
        name = "packed" if packed else "padded"
        rows = m_packed if packed else B * N
        log(f"  {name:6s}: {ms:8.2f} ms/step (rounds: {', '.join(f'{t:.2f}' for t in times[packed])}) | {B / ms * 1e3:8.1f} images/s | "
            f"{n_valid / ms * 1e3 / 1e6:7.3f} M valid tokens/s | peak allocated in a step {peak[packed]:6.2f} GiB | GEMM rows {rows} | "
            f"attention backward {attn_bwd[packed][0]:7.2f} ms in {attn_bwd[packed][1]} launches")
    r = statistics.median(times[True]) / statistics.median(times[False])
    log(f"  packed / padded: step time {r:.3f}, rows {m_packed / (B * N):.3f}, peak memory {peak[True] / peak[False]:.3f}, "
        f"attention backward {attn_bwd[True][0] / attn_bwd[False][0]:.3f}")
    del model, opt
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--only", default=None, help="run the workloads whose name contains this string")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_train_packed: needs a CUDA device")
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"# packed vs padded training step; {card()}; torch {torch.__version__}")
    for tag, (variant, sizes, patch, T, spr) in WORKLOADS.items():
        if a.only and a.only not in tag:
            continue
        run(tag, variant, sizes(), patch, T, spr, a.rounds, log)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
