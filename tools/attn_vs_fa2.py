"""Attention forward: vtk_attention_bf16 against the reference's own attention library call (flash_attn 2.8.3, modules/attention.py:
109-117 -- the FA2 mma.sync kernel recompiled for sm_100, SURVEY K14 "the kernel to beat") on the same B200, same shapes:

    c2         64 images x 16 heads x N = 256, d = 64           c4   8 images x 24 heads x N = 1024, d = 128
    c3-packed  64 mixed-aspect images (bench.py's seeded list, 64..1024 tokens each), 16 heads, d = 64: flash_attn_varlen_func on the
               concatenated valid tokens vs vtk_attention_packed_lse_bf16 (lse = NULL) on the packed NaFlex layout
    2048px     1 image x 16 heads x N = 16384, d = 64 (dense), and the same with a sliding window of 1024 tokens

Both are replayed from CUDA graphs (20 calls per replay) so that the host-side wrappers do not enter the number; outputs are
compared first.  Prints a table and the SM clock seen during the run."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "vitok-release_b200"))
import torch  # noqa: E402
from flash_attn import flash_attn_func, flash_attn_varlen_func  # noqa: E402
from vitok_b200 import _lib  # noqa: E402
from bench import c3_sizes  # noqa: E402

REP = 20


def graph_ms(fn):
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(REP):
            fn()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 5 / REP


def clocks():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip()
        return out
    except Exception as ex:  # noqa: BLE001
        return f"nvidia-smi failed: {ex}"


rows = []
gen = torch.Generator().manual_seed(0)
for name, B, N, h, d, window in [("c2", 64, 256, 16, 64, -1), ("c4", 8, 1024, 24, 128, -1), ("350M-512", 16, 1024, 16, 64, -1),
                                 ("2048px dense", 1, 16384, 16, 64, -1), ("2048px sw=1024", 1, 16384, 16, 64, 1024)]:
    qkv = torch.randn(B * N, 3 * h * d, generator=gen).to(torch.bfloat16).cuda()
    q5 = qkv.view(B, N, 3, h, d)
    q, k, v = q5[:, :, 0], q5[:, :, 1], q5[:, :, 2]
    ws = (window, window) if window >= 0 else (-1, -1)
    ref = flash_attn_func(q, k, v, window_size=ws)
    out = _lib.attention(qkv, B, N, h, d, None, window=window)
    err = float((out.view(B, N, h, d).float() - ref.float()).abs().max())
    t_fa = graph_ms(lambda: flash_attn_func(q, k, v, window_size=ws))
    t_us = graph_ms(lambda: _lib.attention(qkv, B, N, h, d, None, window=window))
    fl = 4.0 * B * N * N * h * d if window < 0 else 4.0 * B * N * min(N, 2 * window + 1) * h * d
    rows.append((name, f"B={B} N={N} h={h} d={d}", t_fa * 1e3, t_us * 1e3, t_fa / t_us, fl / t_us / 1e9, err))

# c3: ragged batch, packed
sizes = c3_sizes(64, 1234)
n_i = [-(-hh // 16) * -(-ww // 16) for hh, ww in sizes]
B, N, h, d = 64, 1024, 16, 64
mask = torch.zeros(B, N, dtype=torch.bool)
for b, n in enumerate(n_i):
    mask[b, :n] = True
mask = mask.cuda()
plan = _lib.pack_plan(mask, 16, 128)
cap = plan["src"].numel()
x = torch.randn(B, N, 3 * h * d, generator=gen).to(torch.bfloat16).cuda()
packed = _lib.pack_rows(x, plan)                                        # [cap, 3D], image b at rows cu[b] .. cu[b] + n_b
cu = plan["cu"].cpu().tolist()
tot = sum(n_i)
cat = torch.cat([packed[cu[b]:cu[b] + n_i[b]] for b in range(B)]).view(tot, 3, h, d)      # what flash_attn_varlen_func wants
cu_seq = torch.tensor([0] + list(torch.tensor(n_i).cumsum(0)), dtype=torch.int32).cuda()
qv, kv_, vv = cat[:, 0].contiguous(), cat[:, 1].contiguous(), cat[:, 2].contiguous()
ref = flash_attn_varlen_func(qv, kv_, vv, cu_seq, cu_seq, max(n_i), max(n_i))
out = _lib.attention_packed(packed, plan, B, N, h, d)
got = torch.cat([out[cu[b]:cu[b] + n_i[b]] for b in range(B)]).view(tot, h, d)
err = float((got.float() - ref.float()).abs().max())
t_fa = graph_ms(lambda: flash_attn_varlen_func(qv, kv_, vv, cu_seq, cu_seq, max(n_i), max(n_i)))
t_us = graph_ms(lambda: _lib.attention_packed(packed, plan, B, N, h, d))
fl = sum(4.0 * n * n * h * d for n in n_i)
rows.append(("c3 packed", f"64 images, {tot} valid tokens, h=16 d=64", t_fa * 1e3, t_us * 1e3, t_fa / t_us, fl / t_us / 1e9, err))

print(f"{'shape':16s} {'detail':44s} {'flash_attn 2.8.3 (us)':>22s} {'vtk (us)':>10s} {'speed-up':>9s} {'vtk TFLOP/s':>12s} {'max |diff|':>11s}")
for r in rows:
    print(f"{r[0]:16s} {r[1]:44s} {r[2]:22.1f} {r[3]:10.1f} {r[4]:9.2f} {r[5]:12.1f} {r[6]:11.2e}")
print("clocks after the run (sm MHz, max, power, reasons):", clocks())
