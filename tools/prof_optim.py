"""Cost of FusedAdamW's gradient clipping (max_grad_norm) and EMA (ema_decay) in the training step, and against the torch equivalent.

    python tools/prof_optim.py [--out FILE] [--rounds R] [--only TAG]

Workloads (the models, batches and layout of tools/prof_train_frozen.py, train_token_packing = True, every parameter trainable):
  * 350M-f16x16 (Ld4-Ld24/1x16x16) on the c3 batch;
  * 5B (Td4-T/1x32x256, p = 32) on 8 images of seeded sizes in [512, 1024]^2.
Variants, alternated R times in this one process on one model and one optimizer (the options are switched on the optimizer):
  plain        FusedAdamW as before;
  +clip        max_grad_norm = 1.0 (norm pass + finish kernel, the coefficient applied inside the AdamW pass);
  +ema         ema_decay = 0.999 (the fp32 EMA updated inside the AdamW pass);
  +both        both;
  torch        plain FusedAdamW plus what a user would write without the options: torch.nn.utils.clip_grad_norm_(foreach=True)
               before the step and torch._foreach_lerp_ of fp32 EMA copies toward the bf16 parameters (cast to fp32 in slices of
               at most 2^28 elements) after it.
Whole steps (forward, Charbonnier loss, backward, optimizer) are timed with CUDA events after warm-up; then opt.step() alone (the
gradients of the last step left in place) over windows of >= 0.5 s per variant, with its HBM rate from the byte counts of the kernels
(28 bytes per bf16 parameter, +8 with the EMA, +2 for the norm pass over bf16 gradients) against a device-to-device copy of 4 GiB timed
in the same run.  The card's name and power limit are read in the same run.
"""
import argparse
import math
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "vitok-release_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import vitok_b200 as vb  # noqa: E402
from bench import c3_sizes  # noqa: E402
from oracle import pp_oracle  # noqa: E402
from oracle.weights import synth_images  # noqa: E402
from prof_train_packed import card  # noqa: E402

WORKLOADS = {
    "350M-f16x16 c3": ("Ld4-Ld24/1x16x16", lambda: c3_sizes(64, 1234), 16, 1024, 3),
    "5B p32 mixed 512-1024": ("Td4-T/1x32x256", lambda: [(int(h), int(w)) for h, w in np.random.RandomState(7).randint(512, 1025, size=(8, 2))],
                              32, 1024, 2),
}
VARIANTS = {"plain": (None, None), "+clip": (1.0, None), "+ema": (None, 0.999), "+both": (1.0, 0.999), "torch": (None, None)}
BYTES = {"plain": 28, "+clip": 30, "+ema": 36, "+both": 38}
DECAY = 0.999


def copy_peak(log):
    n = 1 << 30
    src = torch.empty(n, dtype=torch.float32, device="cuda")
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 20
    log(f"device-to-device copy of 4 GiB: {ms:.3f} ms = {2 * 4 * n / ms / 1e6:.0f} GB/s (read + write)")
    del src, dst
    torch.cuda.empty_cache()


def run(tag, variant, sizes, patch, T, steps_per_round, rounds, log):
    dev = torch.device("cuda", 0)
    cfg = vb.decode_variant(variant)
    torch.manual_seed(0)
    with torch.device(dev):
        model = vb.AE(**cfg, attn_backend="sdpa")
    model = model.to(torch.bfloat16).train()
    model.train_token_packing = True
    params = list(model.parameters())
    decay = [p for n, p in model.named_parameters() if not (p.ndim <= 1 or "bias" in n or "norm" in n)]
    no_decay = [p for n, p in model.named_parameters() if (p.ndim <= 1 or "bias" in n or "norm" in n)]
    opt = vb.FusedAdamW([{"params": decay, "weight_decay": 0.01}, {"params": no_decay, "weight_decay": 0.0}], lr=1e-4, betas=(0.9, 0.99))
    b = pp_oracle.collate([pp_oracle.patchify(i, patch, T) for i in synth_images(sizes, seed=1234)])
    pd = {k: torch.from_numpy(np.asarray(v)).to(dev) for k, v in b.items()}
    pd["patches"] = pd["patches"].to(torch.bfloat16)
    B, N = pd["patch_mask"].shape
    P = sum(p.numel() for p in params)

    def opt_step(v):
        opt.max_grad_norm, opt.ema_decay = VARIANTS[v]
        if v == "torch":
            torch.nn.utils.clip_grad_norm_(params, 1.0, foreach=True)
        opt.step()
        if v == "torch":            # the EMA storage: the optimizer's fp32 ema tensors (allocated by the +ema warm-up)
            sl, n = [], 0
            for p in params:
                sl.append(p)
                n += p.numel()
                if n >= 1 << 28 or p is params[-1]:
                    torch._foreach_lerp_([opt.state[q]["ema"] for q in sl], [q.float() for q in sl], 1.0 - DECAY)
                    sl, n = [], 0

    def step(v):
        opt.zero_grad(set_to_none=True)
        out = model(pd)
        loss = vb.charbonnier_loss(out["patches"], pd["patches"], pd["patch_mask"], eps=1e-3)
        loss.backward()
        opt_step(v)

    for v in VARIANTS:                    # warm-up of every variant ("+ema" creates the EMA state before "torch" uses it)
        for _ in range(2):
            step(v)
    torch.cuda.synchronize()
    times = {v: [] for v in VARIANTS}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for v in VARIANTS:
            torch.cuda.synchronize()
            e0.record()
            for _ in range(steps_per_round):
                step(v)
            e1.record()
            torch.cuda.synchronize()
            times[v].append(e0.elapsed_time(e1) / steps_per_round)
    log(f"## {tag}: {variant}, {P / 1e6:.1f} M parameters (bf16, bf16 gradients), B = {B}, N = {N}, sdpa + patch_mask, train_token_packing")
    plain = statistics.median(times["plain"])
    log(f"  whole step, median of {rounds} rounds of {steps_per_round} steps:")
    for v in VARIANTS:
        ms = statistics.median(times[v])
        log(f"    {v:6s}: {ms:8.2f} ms/step (+{ms - plain:6.2f} ms vs plain; rounds: {', '.join(f'{t:.2f}' for t in times[v])})")

    # opt.step() alone, the last step's gradients in place; windows of >= 0.5 s, alternated
    win = {v: [] for v in VARIANTS}
    reps = {}
    for v in VARIANTS:
        torch.cuda.synchronize()
        e0.record()
        opt_step(v)
        e1.record()
        torch.cuda.synchronize()
        reps[v] = max(3, math.ceil(500.0 / max(e0.elapsed_time(e1), 1e-3)))
    for _ in range(3):
        for v in VARIANTS:
            torch.cuda.synchronize()
            e0.record()
            for _ in range(reps[v]):
                opt_step(v)
            e1.record()
            torch.cuda.synchronize()
            win[v].append((e0.elapsed_time(e1), reps[v]))
    log(f"  opt.step() alone ({P / 1e9:.3f} B parameters), 3 windows of >= 0.5 s each:")
    plain = statistics.median(t / r for t, r in win["plain"])
    for v in VARIANTS:
        ms = statistics.median(t / r for t, r in win[v])
        rate = f" | {BYTES[v]} B/param -> {BYTES[v] * P / ms / 1e6:5.0f} GB/s" if v in BYTES else ""
        log(f"    {v:6s}: {ms:8.3f} ms (+{ms - plain:6.3f} ms vs plain; windows {', '.join(f'{t:.0f} ms / {r}' for t, r in win[v])}){rate}")
    del model, opt, pd
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--only", default=None, help="run the workloads whose name contains this string")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_optim: needs a CUDA device")
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"# FusedAdamW clipping + EMA vs plain and vs the torch equivalent; {card()}; torch {torch.__version__}")
    copy_peak(log)
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
