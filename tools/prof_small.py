"""Per-kernel times of one 350M transformer block at small per-GPU batches (the strong-scaling shards of c2: 8 / 16 / 32 images),
each kernel replayed back to back from a CUDA graph (20 launches per replay, PDL edges like in the model) so that launch latency is
hidden the same way it is in the graphed step.  Env knob (read once per process): VTK_PDL."""
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "vitok-release_b200"))
import torch  # noqa: E402
from vitok_b200 import _lib  # noqa: E402
from vitok_b200.models.ae import pack_w_in, pack_w_out  # noqa: E402

D, heads, N = 1024, 16, 256
d = D // heads
Hf = ((int(D * 2.67) + 8) // 16) * 16
g = torch.Generator().manual_seed(0)
rn = lambda *s, sc=1.0: (torch.randn(*s, generator=g) * sc).to(torch.bfloat16).cuda()  # noqa: E731
wp = pack_w_in(rn(3 * D, D, sc=1 / math.sqrt(D)), rn(2 * Hf, D, sc=1 / math.sqrt(D)))
qp = wp.shape[0] - 2 * Hf
nq, nk = rn(d), rn(d)
inv = (1.0 / (10000.0 ** (torch.arange(0, d // 2, 2).float() / (d // 2)))).cuda()
kp = (D + Hf + 63) // 64 * 64
wo = pack_w_out(rn(D, D, sc=1 / math.sqrt(D)), rn(D, Hf, sc=1 / math.sqrt(Hf)))
gamma = rn(D)
REP = 20


def graph_time(fn):
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        for _ in range(REP):
            fn()
    for _ in range(3):
        gr.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        gr.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 10 / REP * 1e3


tag = " ".join(f"{k}={os.environ[k]}" for k in ("VTK_PDL",) if k in os.environ) or "default"
for B in [int(a) for a in sys.argv[1:]] or [8, 16, 32, 64]:
    M = B * N
    h = rn(M, D)
    idx = torch.arange(M)
    table = _lib.rope_table(((idx % N) // 16).cuda(), (idx % 16).cuda(), inv, d)
    a2 = rn(M, kp)[:, :D + Hf]
    x = rn(M, D)
    qkv = rn(M, 3 * D)
    t1 = graph_time(lambda: _lib.qkv_swiglu(h, wp, D, d, Hf, qp, nq, nk, table))
    t2 = graph_time(lambda: _lib.proj_residual(a2, wo, gamma, x))
    t3 = graph_time(lambda: _lib.attention(qkv, B, N, heads, d))
    f1, f2, f3 = 2.0 * M * D * (3 * D + 2 * Hf), 2.0 * M * (D + Hf) * D, 4.0 * B * N * N * D
    print(f"[{tag}] B={B:3d} M={M:6d}: qkv_swiglu {t1:6.1f} us {f1 / t1 / 1e6:5.0f} TF/s | proj_resid {t2:6.1f} us {f2 / t2 / 1e6:5.0f} TF/s | "
          f"attention {t3:6.1f} us {f3 / t3 / 1e6:5.0f} TF/s | block {t1 + t2 + t3:6.1f} us", flush=True)
