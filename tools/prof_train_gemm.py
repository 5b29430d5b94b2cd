"""The three GEMM kinds of the 5B training step (BASELINE config 5: M = 8192 tokens, D = 3072, Hf = 8192) timed alone:
forward (K-major operands), data gradient (B read MN-major, `vtk_linear_nn_acc_bf16`) and weight gradient (both operands MN-major,
`vtk_linear_tn_bf16`), each at the shapes the step launches.  CUDA events over 10 back-to-back launches (operands larger than L2 in
total; no profiler).  VTK_GEMM_PROF=1 makes the library print a per-role cycle report after every launch."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "vitok-release_b200"))
import torch  # noqa: E402
from vitok_b200 import train as T  # noqa: E402

dev = "cuda"
M, D, Hf = 8192, 3072, 8192
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 10
g = torch.Generator(device=dev).manual_seed(0)


def rnd(*s):
    return (torch.randn(*s, device=dev, generator=g) * 0.05).to(torch.bfloat16)


def timed(name, fn, flops):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    print(f"{name:58s} {ms * 1e3:8.1f} us  {flops / ms / 1e9:7.1f} TFLOP/s", flush=True)


h, dy = rnd(M, D), rnd(M, D)
wqkv, w1, w2 = rnd(3 * D, D), rnd(2 * Hf, D), rnd(D, Hf)
dz1 = rnd(M, 2 * Hf)
act = rnd(M, Hf)
out_f = torch.empty(M, 2 * Hf, dtype=torch.bfloat16, device=dev)
out_d = torch.empty(M, D, dtype=torch.bfloat16, device=dev)
out_w = torch.empty(2 * Hf, D, dtype=torch.bfloat16, device=dev)
out_w2 = torch.empty(D, Hf, dtype=torch.bfloat16, device=dev)
out_a = torch.empty(M, Hf, dtype=torch.bfloat16, device=dev)
f = 2.0 * M * D * 2 * Hf
print(f"--- c5 shapes: M = {M}, D = {D}, Hf = {Hf}")
timed("forward  h[M,D] x W1[2Hf,D]^T            (K-major)", lambda: T._linear(h, D, w1, None, M, 2 * Hf, D, out=out_f), f)
timed("dgrad    dz[M,2Hf] x W1[2Hf,D]           (B MN-major)", lambda: T._dgrad(dz1, 2 * Hf, w1, M, D, 2 * Hf, out=out_d), f)
timed("dgrad    dy[M,D] x W2[D,Hf]              (B MN-major)", lambda: T._dgrad(dy, D, w2, M, Hf, D, out=out_a), 2.0 * M * D * Hf)
timed("wgrad    dz[M,2Hf]^T x h[M,D]            (A, B MN-major)", lambda: T._wgrad(dz1, 2 * Hf, 2 * Hf, h, D, D, M, out=out_w), f)
timed("wgrad    dy[M,D]^T x act[M,Hf]           (A, B MN-major)", lambda: T._wgrad(dy, D, D, act, Hf, Hf, M, out=out_w2), 2.0 * M * D * Hf)
