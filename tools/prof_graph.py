"""Eager vs CUDA-graph replay of encode+decode at small per-GPU batches (strong-scaling shape: 64 images over 8 GPUs)."""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "vitok-release_b200"))
import torch  # noqa: E402
import vitok_b200 as vb  # noqa: E402

print(f"VTK_PDL={os.environ.get('VTK_PDL', '1')}")

cfg = vb.decode_variant("Ld4-Ld24/1x16x64")
torch.manual_seed(0)
model = vb.AE(**cfg, attn_backend="flash").eval().to("cuda", torch.bfloat16)
for B in (1, 4, 8, 16, 32, 64):
    imgs = (torch.rand(B, 3, 256, 256) * 2 - 1).cuda()
    pd = vb.patchify_batch(imgs, 16, 256, out_dtype=torch.bfloat16)
    graphed = vb.GraphedAE(model, pd)

    def eager():
        with torch.no_grad():
            return model.decode(model.encode(pd))

    res = {}
    for name, fn in (("eager", eager), ("graph", lambda: graphed(pd))):
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        n = 50
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        res[name] = (e0.elapsed_time(e1) / n, (time.perf_counter() - t0) * 1e3 / n)
    print(f"B={B:3d}: eager {res['eager'][0]:7.3f} ms/step ({B / res['eager'][0] * 1e3:8.1f} images/s)   "
          f"graph {res['graph'][0]:7.3f} ms/step ({B / res['graph'][0] * 1e3:8.1f} images/s)")
