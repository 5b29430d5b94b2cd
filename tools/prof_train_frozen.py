"""Training steps with frozen parameters (vitok_b200.train._grad_plan) vs the full step, on packed NaFlex batches.

    python tools/prof_train_frozen.py [--out FILE] [--rounds R] [--only TAG]

Workloads (the batches, seeds and layout of tools/prof_train_packed.py, train_token_packing = True):
  * 350M-f16x16 (Ld4-Ld24/1x16x16) on the c3 batch: full; frozen encoder; a decoder-only model (AE(encoder=False), the same decoder
    parameters) fed a cached z; only the last 8 decoder blocks trainable;
  * 5B (Td4-T/1x32x256, p = 32) on 8 images of seeded sizes in [512, 1024]^2: full; frozen encoder.
Whole steps (forward, Charbonnier loss, backward, FusedAdamW over every parameter -- frozen ones have no gradient and are skipped) are
timed with CUDA events after warm-up, the variants alternated R times in this one process on one set of parameters.  Reported per
variant: ms/step (median of the rounds, and the rounds), the spread of the full step's rounds, peak allocated memory of one step
above what is allocated before it, and the algorithmic FLOPs the step runs, counted from shapes and the backward plan: block GEMMs,
attention (forward 4 n^2 D, backward 10 n^2 D per image: S recomputed, dP, dV, dQ, dK) and the input / output projections.  The
card's name and power limit are read in the same run.
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
import vitok_b200 as vb  # noqa: E402
from bench import c3_sizes  # noqa: E402
from oracle import pp_oracle  # noqa: E402
from oracle.weights import synth_images  # noqa: E402
from prof_train_packed import card  # noqa: E402
from vitok_b200.models.ae import _ffn_hidden  # noqa: E402
from vitok_b200.train import _grad_plan  # noqa: E402

WORKLOADS = {
    "350M-f16x16 c3": ("Ld4-Ld24/1x16x16", lambda: c3_sizes(64, 1234), 16, 1024, 3, ("full", "frozen encoder", "decoder-only, cached z",
                                                                                      "last 8 decoder blocks")),
    "5B p32 mixed 512-1024": ("Td4-T/1x32x256", lambda: [(int(h), int(w)) for h, w in np.random.RandomState(7).randint(512, 1025, size=(8, 2))],
                              32, 1024, 2, ("full", "frozen encoder")),
}
ENC = ("patch_embed", "encoder_blocks", "to_code")


def step_flops(model, M: int, s2: int, input_grad: bool = False) -> float:
    """Algorithmic FLOPs of one training step of ``model`` as its parameters' requires_grad stand: M rows, s2 = sum over images of
    n_valid^2."""
    needs = {n: p.requires_grad for n, p in model.named_parameters()}
    sides = {s[0]: s for s in model._sides()}
    plan = _grad_plan(needs, {k: len(s[3]) for k, s in sides.items()}, input_grad)
    ck = int(model.checkpoint or 0)
    total = 0.0
    for side, (_, lin_a, lin_b, blocks, D, _) in sides.items():
        sp = plan[side]
        Hf = _ffn_hidden(D, model.mlp_factor)
        cin, cout = lin_a.weight.shape[1], lin_b.weight.shape[0]
        fwd = 2 * M * D * (3 * D + 2 * Hf) + 2 * M * (D + Hf) * D + 4 * s2 * D
        total += 2 * M * cin * D + 2 * M * D * cout + len(blocks) * fwd
        total += (sp.head[0] + sp.top) * 2 * M * D * cout + (sp.embed[0] + sp.dinput) * 2 * M * cin * D
        for i, st in enumerate(sp.stages):
            wq, wf, wo, w2 = sp.wgrads[i]
            if st and ck and i % ck == 0:
                total += fwd
            total += wo * 2 * M * D * D + w2 * 2 * M * Hf * D
            if st >= 2:
                total += 2 * M * D * (D + Hf) + 10 * s2 * D
            total += wq * 2 * M * 3 * D * D + wf * 2 * M * 2 * Hf * D
            if st >= 3:
                total += 2 * M * D * (3 * D + 2 * Hf)
    return total


def run(tag, variant, sizes, patch, T, steps_per_round, variants, rounds, log):
    dev = torch.device("cuda", 0)
    cfg = vb.decode_variant(variant)
    torch.manual_seed(0)
    with torch.device(dev):
        model = vb.AE(**cfg, attn_backend="sdpa")
    model = model.to(torch.bfloat16).train()
    model.train_token_packing = True
    decay = [p for n, p in model.named_parameters() if not (p.ndim <= 1 or "bias" in n or "norm" in n)]
    no_decay = [p for n, p in model.named_parameters() if (p.ndim <= 1 or "bias" in n or "norm" in n)]
    opt = vb.FusedAdamW([{"params": decay, "weight_decay": 0.01}, {"params": no_decay, "weight_decay": 0.0}], lr=1e-4, betas=(0.9, 0.99))
    b = pp_oracle.collate([pp_oracle.patchify(i, patch, T) for i in synth_images(sizes, seed=1234)])
    pd = {k: torch.from_numpy(np.asarray(v)).to(dev) for k, v in b.items()}
    pd["patches"] = pd["patches"].to(torch.bfloat16)
    B, N = pd["patch_mask"].shape
    nv = pd["patch_mask"].sum(1)
    n_valid, s2 = int(nv.sum()), int((nv.long() ** 2).sum())
    M = int(((nv + 15) // 16 * 16).sum())

    dec_only = None
    if "decoder-only, cached z" in variants:
        # AE(encoder=False) holding the very decoder parameters of ``model`` (one optimizer state), fed z encoded once
        dec_only = vb.AE(**cfg, attn_backend="sdpa", encoder=False)
        dec_only.decoder_embed, dec_only.to_pixels, dec_only.decoder_blocks = model.decoder_embed, model.to_pixels, model.decoder_blocks
        dec_only.train()
        dec_only.train_token_packing = True
        model.eval()
        with torch.no_grad():
            z = model.encode(pd)["z"]
        model.train()
        pd_z = dict(pd, z=z)

    def setup(v):
        model.requires_grad_(True)
        if v == "frozen encoder":
            for name in ENC:
                getattr(model, name).requires_grad_(False)
        elif v == "last 8 decoder blocks":
            model.requires_grad_(False)
            model.decoder_blocks[-8:].requires_grad_(True)
        elif v == "decoder-only, cached z":
            for name in ENC:
                getattr(model, name).requires_grad_(False)
        return (dec_only, pd_z) if v == "decoder-only, cached z" else (model, pd)

    def step(m, batch):
        opt.zero_grad(set_to_none=True)
        out = m(batch)
        loss = vb.charbonnier_loss(out["patches"], pd["patches"], pd["patch_mask"], eps=1e-3)
        loss.backward()
        opt.step()
        return loss

    times = {v: [] for v in variants}
    peak, flops = {}, {}
    for v in variants:                    # warm-up of every variant, then the peak memory of one step
        m, batch = setup(v)
        flops[v] = step_flops(m, M, s2)
        for _ in range(2):
            step(m, batch)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        step(m, batch)
        torch.cuda.synchronize()
        peak[v] = (torch.cuda.max_memory_allocated() - base) / 2**30
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for v in variants:
            m, batch = setup(v)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(steps_per_round):
                step(m, batch)
            e1.record()
            torch.cuda.synchronize()
            times[v].append(e0.elapsed_time(e1) / steps_per_round)
    model.requires_grad_(True)
    full = times["full"]
    log(f"## {tag}: {variant}, B = {B}, N = {N}, {n_valid} valid tokens, packed rows {M}, sdpa + patch_mask, train_token_packing")
    log(f"  full-step spread over {rounds} rounds: {min(full):.2f} .. {max(full):.2f} ms ({(max(full) - min(full)) / statistics.median(full) * 100:.1f} %)")
    for v in variants:
        ms = statistics.median(times[v])
        log(f"  {v:24s}: {ms:8.2f} ms/step (rounds: {', '.join(f'{t:.2f}' for t in times[v])}) | vs full {ms / statistics.median(full):.3f} | "
            f"peak allocated in a step {peak[v]:6.2f} GiB ({peak[v] / peak['full']:.3f} of full) | "
            f"{flops[v] / 1e12:7.2f} TFLOP/step ({flops[v] / flops['full']:.3f} of full) | {flops[v] / ms / 1e9:6.0f} TFLOP/s")
    del model, opt, dec_only
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--only", default=None, help="run the workloads whose name contains this string")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_train_frozen: needs a CUDA device")
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"# training steps with frozen parameters vs the full step; {card()}; torch {torch.__version__}")
    for tag, (variant, sizes, patch, T, spr, variants) in WORKLOADS.items():
        if a.only and a.only not in tag:
            continue
        run(tag, variant, sizes(), patch, T, spr, variants, a.rounds, log)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
