"""Micro-benchmark of the two block GEMMs at the c2 / c4 shapes (CUDA events, each kernel alone)."""
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "vitok-release_b200"))
import torch  # noqa: E402
from vitok_b200 import _lib  # noqa: E402
from vitok_b200.models.ae import pack_w_in, pack_w_out  # noqa: E402

which = sys.argv[1] if len(sys.argv) > 1 else "c2"
M, D, heads = (16384, 1024, 16) if which == "c2" else (8192, 3072, 24)
d = D // heads
Hf = ((int(D * 2.67) + 8) // 16) * 16
g = torch.Generator().manual_seed(0)
rn = lambda *s, sc=1.0: (torch.randn(*s, generator=g) * sc).to(torch.bfloat16).cuda()
h = rn(M, D)
wp = pack_w_in(rn(3 * D, D, sc=1 / math.sqrt(D)), rn(2 * Hf, D, sc=1 / math.sqrt(D)))
qp = wp.shape[0] - 2 * Hf
nq, nk = rn(d), rn(d)
idx = torch.arange(M)
inv = (1.0 / (10000.0 ** (torch.arange(0, d // 2, 2).float() / (d // 2)))).cuda()
table = _lib.rope_table((idx // 64).cuda(), (idx % 64).cuda(), inv, d)
kp = (D + Hf + 63) // 64 * 64
a2 = rn(M, kp)[:, :D + Hf]          # 128-byte aligned row pitch, like the AE workspace
wo = pack_w_out(rn(D, D, sc=1 / math.sqrt(D)), rn(D, Hf, sc=1 / math.sqrt(Hf)))
gamma = rn(D)
x = rn(M, D)


def timeit(fn, n=20):
    if len(sys.argv) > 2 and sys.argv[2] == "once":
        n = 4
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


t1 = timeit(lambda: _lib.qkv_swiglu(h, wp, D, d, Hf, qp, nq, nk, table))
t2 = timeit(lambda: _lib.proj_residual(a2, wo, gamma, x))
f1 = 2.0 * M * D * (3 * D + 2 * Hf)
f2 = 2.0 * M * (D + Hf) * D
print(f"{which}: qkv_swiglu {t1*1e3:.1f} us {f1/t1/1e9:.0f} TF/s | proj_resid {t2*1e3:.1f} us {f2/t2/1e9:.0f} TF/s")

if len(sys.argv) > 2 and sys.argv[2] == "sustain":
    # 2 s of back-to-back launches per GEMM with nvidia-smi clock sampling: is the kernel power-capped?
    import subprocess, tempfile, time, statistics
    for name, fn, fl in (("qkv_swiglu", lambda: _lib.qkv_swiglu(h, wp, D, d, Hf, qp, nq, nk, table), f1),
                         ("proj_resid", lambda: _lib.proj_residual(a2, wo, gamma, x), f2)):
        f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        p = subprocess.Popen(["nvidia-smi", "--id=0", "--query-gpu=clocks.sm,power.draw,clocks_event_reasons.sw_power_cap",
                              "--format=csv,noheader,nounits", "-lms", "50"], stdout=f, stderr=subprocess.DEVNULL)
        torch.cuda.synchronize()
        n = 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        while time.time() - t0 < 2.0:
            for _ in range(50):
                fn()
            n += 50
            torch.cuda.synchronize()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        p.terminate(); p.wait()
        rows = [r.split(",") for r in open(f.name).read().strip().splitlines() if r.strip()]
        clk = [float(r[0]) for r in rows[5:]] or [0.0]
        pw = [float(r[1]) for r in rows[5:]] or [0.0]
        cap = sum("Active" in r[2] and "Not" not in r[2] for r in rows)
        print(f"{which} sustain {name}: {ms*1e3:.1f} us {fl/ms/1e9:.0f} TF/s | sm clk median {statistics.median(clk):.0f} min {min(clk):.0f} MHz, "
              f"power median {statistics.median(pw):.0f} W, power-cap samples {cap}/{len(rows)}")
