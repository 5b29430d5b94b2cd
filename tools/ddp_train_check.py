"""2+ GPU check of the data-parallel training step (reference: DDP at scripts/train_vae.py:172).

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29533 tools/ddp_train_check.py

Every rank runs model(batch) -> Charbonnier -> backward on ITS OWN batch under DistributedDataParallel (NCCL).  Checked:
  * after backward every rank holds the same gradients (bit-identical), and they equal the mean of the per-rank local
    gradients computed without DDP (all-reduce(mean) semantics);
  * after FusedAdamW steps the parameters stay identical across ranks and the loss goes down.
With ``--frozen-encoder`` it checks instead the overlapped all-reduce (vb.enable_grad_sync) of a model whose encoder is frozen: every
rank holds identical decoder gradients equal to the mean of the local ones, and the encoder has no gradient and stays identical.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "vitok-release_b200"))
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
from torch.nn.parallel import DistributedDataParallel as DDP  # noqa: E402

import vitok_b200 as vb  # noqa: E402


def _same_on_ranks(t, world):
    chk = t.float().sum().double().reshape(1)
    lst = [torch.zeros_like(chk) for _ in range(world)]
    dist.all_gather(lst, chk)
    return all(float(x) == float(lst[0]) for x in lst)


def frozen_encoder(cfg, dev, rank, world):
    enc = ("patch_embed.", "to_code.", "encoder_blocks.")

    def make():
        torch.manual_seed(0)
        m = vb.AE(**cfg, attn_backend="flash").train().to(dev, torch.bfloat16)
        for mod in (m.patch_embed, m.encoder_blocks, m.to_code):
            mod.requires_grad_(False)
        return m

    g = torch.Generator().manual_seed(100 + rank)
    imgs = torch.rand(4, 3, 256, 256, generator=g) * 2 - 1
    pd = vb.patchify_batch(imgs.to(dev), 16, 256, out_dtype=torch.bfloat16, device=dev)
    twin = make()
    vb.charbonnier_loss(twin(pd)["patches"], pd["patches"], pd["patch_mask"]).backward()
    local_g = {n: p.grad.float().clone() for n, p in twin.named_parameters() if p.grad is not None}
    assert not any(n.startswith(enc) for n in local_g) and len(local_g) == sum(1 for n, _ in twin.named_parameters() if not n.startswith(enc))
    for t in local_g.values():
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        t /= world
    m = make()
    vb.enable_grad_sync(m)
    vb.charbonnier_loss(m(pd)["patches"], pd["patches"], pd["patch_mask"]).backward()
    worst = 0.0
    for n, p in m.named_parameters():
        if n.startswith(enc):
            assert p.grad is None, f"{n}: a frozen parameter got a gradient"
            assert _same_on_ranks(p.detach(), world), f"{n}: frozen parameters differ across ranks"
            continue
        worst = max(worst, float((p.grad.float() - local_g[n]).norm() / local_g[n].norm().clamp_min(1e-30)))
        assert _same_on_ranks(p.grad, world), f"{n}: overlapped-sync gradients differ across ranks"
    assert worst < 2e-2, worst
    if rank == 0:
        print(f"grad_sync frozen encoder OK: world={world} worst decoder grad rel err vs hand-made mean {worst:.3e}")


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    args = [a for a in sys.argv[1:] if a != "--frozen-encoder"]
    variant = args[0] if args else "w256_d2_h4-w512_d3_h4/1x16x16"
    if "--frozen-encoder" in sys.argv[1:]:
        frozen_encoder(vb.decode_variant(variant), dev, rank, world)
        dist.destroy_process_group()
        return
    cfg = vb.decode_variant(variant)
    torch.manual_seed(0)
    model = vb.AE(**cfg, attn_backend="flash").train().to(dev, torch.bfloat16)
    # an un-wrapped twin for the hand-made reference: running the bare module's backward while DDP's hooks are
    # installed would be counted by the static-graph bookkeeping of the first iteration
    twin = vb.AE(**cfg, attn_backend="flash").train().to(dev, torch.bfloat16)
    twin.load_state_dict(model.state_dict())
    ddp = DDP(model, device_ids=[local], static_graph=True)
    g = torch.Generator().manual_seed(100 + rank)
    imgs = torch.rand(4, 3, 256, 256, generator=g) * 2 - 1
    pd = vb.patchify_batch(imgs.to(dev), 16, 256, out_dtype=torch.bfloat16, device=dev)

    # local gradients without DDP, then their mean over ranks by hand
    loss = vb.charbonnier_loss(twin(pd)["patches"], pd["patches"], pd["patch_mask"])
    loss.backward()
    local_g = {n: p.grad.float().clone() for n, p in twin.named_parameters()}
    for t in local_g.values():
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        t /= world
    # the same step under DDP
    model.zero_grad(set_to_none=True)
    loss = vb.charbonnier_loss(ddp(pd)["patches"], pd["patches"], pd["patch_mask"])
    loss.backward()
    worst = 0.0
    for n, p in model.named_parameters():
        ref = local_g[n]
        err = (p.grad.float() - ref).norm() / ref.norm().clamp_min(1e-30)
        worst = max(worst, float(err))
        chk = p.grad.float().sum().double().reshape(1)
        lst = [torch.zeros_like(chk) for _ in range(world)]
        dist.all_gather(lst, chk)
        assert all(float(x) == float(lst[0]) for x in lst), f"{n}: gradients differ across ranks"
    assert worst < 2e-2, worst     # bf16 all-reduce vs fp32 mean of bf16 gradients

    opt = vb.FusedAdamW(model.parameters(), lr=2e-3, betas=(0.9, 0.99), weight_decay=0.0)
    losses = []
    for _ in range(6):
        opt.zero_grad(set_to_none=True)
        loss = vb.charbonnier_loss(ddp(pd)["patches"], pd["patches"], pd["patch_mask"])
        loss.backward()
        if os.environ.get("DDP_CHECK_DEBUG"):
            for n, p in list(model.named_parameters())[:3]:
                for what, t in (("grad", p.grad), ("param", p.detach())):
                    lst = [torch.zeros_like(t) for _ in range(world)]
                    dist.all_gather(lst, t.contiguous())
                    if rank == 0:
                        print(f"step {len(losses)} {n} {what}: max |r0 - r1| = {(lst[0].float() - lst[1].float()).abs().max().item():.3e}", flush=True)
        opt.step()
        losses.append(float(loss))
    for n, p in model.named_parameters():
        chk = p.detach().float().sum().double().reshape(1)
        lst = [torch.zeros_like(chk) for _ in range(world)]
        dist.all_gather(lst, chk)
        assert all(float(x) == float(lst[0]) for x in lst), f"{n}: parameters diverged across ranks"
    assert losses[-1] < losses[0]
    if rank == 0:
        print(f"ddp_train_check OK: world={world} worst grad rel err vs hand-made mean {worst:.3e}; loss {losses[0]:.4f} -> {losses[-1]:.4f}")

    # ---- the same step with vb.enable_grad_sync (all-reduce issued from inside the backward loop, no DDP wrapper) ----
    torch.manual_seed(1 + rank)                      # different initial parameters per rank: the broadcast must fix that
    m2 = vb.AE(**cfg, attn_backend="flash").train().to(dev, torch.bfloat16)
    vb.enable_grad_sync(m2)
    for (n, p), (_, q) in zip(m2.named_parameters(), twin.named_parameters()):
        lst = [torch.zeros_like(p.data) for _ in range(world)]
        dist.all_gather(lst, p.data.contiguous())
        assert all(torch.equal(x, lst[0]) for x in lst), f"{n}: broadcast_parameters left ranks different"
    m2.load_state_dict(twin.state_dict())            # same weights as the hand-made reference above
    loss = vb.charbonnier_loss(m2(pd)["patches"], pd["patches"], pd["patch_mask"])
    loss.backward()
    worst2 = 0.0
    for n, p in m2.named_parameters():
        ref = local_g[n]
        worst2 = max(worst2, float((p.grad.float() - ref).norm() / ref.norm().clamp_min(1e-30)))
        chk = p.grad.float().sum().double().reshape(1)
        lst = [torch.zeros_like(chk) for _ in range(world)]
        dist.all_gather(lst, chk)
        assert all(float(x) == float(lst[0]) for x in lst), f"{n}: overlapped-sync gradients differ across ranks"
    assert worst2 < 2e-2, worst2
    if rank == 0:
        print(f"grad_sync (overlapped all-reduce) OK: worst grad rel err vs hand-made mean {worst2:.3e}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
