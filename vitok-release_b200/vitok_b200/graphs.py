"""CUDA-graph capture of the encode / decode hot path.

A full-size batch keeps the GPU busy for ~12 ms per step and the ~90 launches of an encode+decode are hidden behind it, but
at the small per-GPU batches of a strong-scaling or latency-bound deployment (SURVEY.md section 8e: 8 images per GPU are
~1.6 ms of GPU work) the host-side launch loop becomes the bottleneck.  Every C-ABI call of this path is capturable
(explicit stream, no allocation, no host sync -- with token packing even the packed row count stays on the device), so the
whole encode -> decode sequence for one (B, N) shape is captured once and replayed with ONE launch.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

_STATIC_KEYS = ("patches", "z", "patch_mask", "row_idx", "col_idx")


class GraphedAE:
    """``GraphedAE(model, example_batch)(batch)`` == ``model.decode(model.encode(batch))`` (or only the half the model has),
    replayed from a CUDA graph.  ``batch`` must have the shapes / dtypes of ``example_batch``; its tensors are copied into
    static buffers, the outputs are static tensors that the next call overwrites (clone them to keep them).  The model must
    be in eval mode; re-create the object after changing weights (``load_state_dict``, ``.to()``, ``quantize()``).
    """

    def __init__(self, model, example_batch: Dict[str, torch.Tensor], warmup: int = 2, private_workspace: bool = False):
        if model.training:
            raise RuntimeError("GraphedAE: put the model in eval mode first (model.eval())")
        self.model = model
        dev = next(model.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("GraphedAE: the model must be on a CUDA device")
        self.static_in = {k: (v.to(dev).clone() if isinstance(v, torch.Tensor) else v) for k, v in example_batch.items()}
        # private_workspace: capture with workspaces of its own instead of the model's (one per side, shared by every graph and eager call
        # of that shape), so that several graphs of one model may be replayed CONCURRENTLY on different streams -- two batches in flight
        # fill the SMs that the one-wave kernels of a small batch leave idle.  The model's own workspaces are put back afterwards.
        saved_ws = None
        if private_workspace:
            saved_ws, model._ws = model._ws, {}
        try:
            self._capture(model, dev, warmup)
        finally:
            if saved_ws is not None:
                model._ws = saved_ws

    def _capture(self, model, dev, warmup):
        with torch.cuda.device(dev):
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side), torch.no_grad():      # warm-up on a side stream: weight packing, workspaces, allocator
                for _ in range(max(warmup, 1)):
                    self._forward(self.static_in)
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            self._sig = self._state()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph), torch.no_grad():
                self.static_out = self._forward(self.static_in)
        # The graph has the raw addresses of the model's workspaces and packed weight copies baked in.  The model keeps only
        # one live workspace per side and replaces the packed copies when parameters change, so hold strong references here:
        # whatever the model does afterwards (another shape, another GraphedAE, eager calls), this memory stays allocated for
        # as long as this graph can be replayed.
        self._keep = (list(model._ws.values()), [t for lst in model._packed.values() for t in lst])

    def _state(self):
        m = self.model
        return (m._signature(), bool(m.fuse_norm), bool(m._quantization_applied), m.fp8_activation_scale, m.attn_backend, m.sw)

    def _forward(self, d):
        m = self.model
        if m.is_encoder:
            d = m.encode(d)
        if m.is_decoder:
            d = m.decode(d)
        return d

    def __call__(self, batch: Dict[str, torch.Tensor]) -> Dict[str, Optional[torch.Tensor]]:
        if self._state() != self._sig:
            raise RuntimeError("GraphedAE: the model's parameters or its fuse_norm / quantize state changed since "
                               "capture; build a new GraphedAE")
        for k in _STATIC_KEYS:
            src = batch.get(k)
            dst = self.static_in.get(k)
            if isinstance(dst, torch.Tensor):
                if src is None or src.shape != dst.shape:
                    raise ValueError(f"GraphedAE: '{k}' must have shape {tuple(dst.shape)} like the captured batch")
                if src.data_ptr() != dst.data_ptr():
                    dst.copy_(src, non_blocking=True)
        with torch.cuda.device(self.static_in["row_idx"].device):
            self.graph.replay()
        out = dict(self.static_out)
        for k in ("orig_height", "orig_width"):                # pass-through metadata of THIS batch (ae.py:209-216)
            out[k] = batch.get(k)
        return out


class GraphedCodec:
    """The whole serving step -- uint8 images -> ``patchify_batch`` (fused to_tensor|normalize|patchify) -> ``encode`` ->
    ``decode`` -> ``unpatchify(output_format=...)`` -- captured as ONE CUDA graph for one batch geometry.

    ``images``: a ``[B, H, W, 3]`` uint8 CUDA tensor, or ``(flat, offsets, sizes)`` as produced by ``pack_images`` (ragged
    NaFlex batch, ``flat`` on the GPU).  ``codec.static_in`` is the graph's input buffer: a serving loop copies the next
    batch straight into it (H2D) and calls ``codec()``; ``codec(images)`` copies device tensors for you.  The result is the
    static canvas tensor ``[B, 3, G*p, G*p]`` (``max_grid_size`` = G is required: a data-dependent canvas needs a host sync),
    overwritten by the next call.  At 8 images per GPU (a 64-image batch sharded over 8 GPUs) the ~100 launches of a step
    cost more host time than the GPU needs to run them; the replay is one launch.
    """

    def __init__(self, model, images, patch: int = 16, max_tokens: int = 256, max_grid_size: Optional[int] = None,
                 output_format: str = "0_255", warmup: int = 2, private_workspace: bool = False):
        from .pp import patchify_batch, patchify_packed, unpatchify
        if model.training:
            raise RuntimeError("GraphedCodec: put the model in eval mode first (model.eval())")
        if max_grid_size is None:
            raise ValueError("GraphedCodec: max_grid_size is required (the canvas size must not depend on the data)")
        self.model = model
        if isinstance(images, (tuple, list)):
            flat, offsets, sizes = images
            self.static_in = flat.clone()
            dev = flat.device

            def pre():
                return patchify_packed(self.static_in, offsets, sizes, patch, max_tokens, out_dtype=torch.bfloat16)
        else:
            if images.dtype != torch.uint8 or images.dim() != 4 or images.shape[-1] != 3:
                raise ValueError("GraphedCodec: images must be a [B, H, W, 3] uint8 tensor or (flat, offsets, sizes)")
            self.static_in = images.contiguous().clone()
            dev = images.device

            def pre():
                return patchify_batch(self.static_in, patch, max_tokens, out_dtype=torch.bfloat16, device=dev)
        if dev.type != "cuda":
            raise RuntimeError("GraphedCodec: the images must be on a CUDA device")
        self.launches = 0

        def run():
            d = pre()
            n = 1
            if model.is_encoder:
                d = model.encode(d)
                n += model.last_launch_count
            if model.is_decoder:
                d = model.decode(d)
                n += model.last_launch_count
            self.launches = n + 2                  # cell map + unpatchify
            return unpatchify(d, patch, max_grid_size=max_grid_size, output_format=output_format)

        saved_ws = None
        if private_workspace:                      # see GraphedAE: workspaces of its own, for concurrent replays on several streams
            saved_ws, model._ws = model._ws, {}
        try:
            with torch.cuda.device(dev):
                side = torch.cuda.Stream(device=dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(side), torch.no_grad():
                    for _ in range(max(warmup, 1)):
                        run()
                torch.cuda.current_stream(dev).wait_stream(side)
                torch.cuda.synchronize(dev)
                self._sig = GraphedAE._state(self)
                self.graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph), torch.no_grad():
                    self.static_out = run()
            self._keep = (list(model._ws.values()), [t for lst in model._packed.values() for t in lst])
        finally:
            if saved_ws is not None:
                model._ws = saved_ws
        self._dev = dev

    def __call__(self, images: Optional[torch.Tensor] = None) -> torch.Tensor:
        if GraphedAE._state(self) != self._sig:
            raise RuntimeError("GraphedCodec: the model changed since capture; build a new GraphedCodec")
        if images is not None and images.data_ptr() != self.static_in.data_ptr():
            if images.shape != self.static_in.shape or images.dtype != self.static_in.dtype:
                raise ValueError("GraphedCodec: images must match the captured batch")
            self.static_in.copy_(images, non_blocking=True)
        with torch.cuda.device(self._dev):
            self.graph.replay()
        return self.static_out


__all__ = ["GraphedAE", "GraphedCodec"]
