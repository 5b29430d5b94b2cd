"""Training step of the B200-native AE (BASELINE config 5; reference: scripts/train_vae.py:304-320,371-372).

``AE.forward`` in training mode routes here: one ``torch.autograd.Function`` runs the encoder + decoder forward
with hand-written sm_100a kernels while keeping what the backward pass needs, and its ``backward`` produces the
gradient of every parameter with the kernels of csrc/vtk_train.cu, csrc/vtk_attention_bwd.cu and the tcgen05
GEMM (data gradients against the weights as stored, weight gradients on transposed operands).  PyTorch only owns memory,
streams, the autograd graph edge, the random draw of stochastic depth and -- under DDP (train_vae.py:172) -- the NCCL
gradient all-reduce.

Also here: ``charbonnier_loss`` (train_vae.py:314-320), ``ssim`` (the SSIM tile loss term, train_vae.py:328-368; csrc/vtk_ssim.cu) and ``FusedAdamW`` (train_vae.py:200-208: AdamW with fp32 master
weights and fp32 moments, multi-tensor).

Saved per block (bf16 unless noted): x (block input), h = RMSNorm(x), zraw = [h Wqkv^T | pad | h W1^T], qkv (normed + roped),
a2 = [attention out | silu(g) v | pad], lse (fp32 [M, heads]), y = a2 [out_proj | fc2]^T.
``checkpoint = k`` (ae.py:159-160,202-205,231-233): blocks with ``i % k == 0`` keep only x (and their stochastic-depth draw)
and are re-run from it inside the backward pass -- config 5 at 8 x 1024 tokens per GPU saves ~0.9 GB per block, 40 GB for
44 blocks; with checkpoint = 1 the saved set shrinks to 50 MB per block.
``drop_path_rate > 0`` (ae.py:15-30,65,143-152): decoder block i drops its whole update for an image with probability
``rate * i / (depth - 1)`` and rescales the others by 1 / keep_prob; the draw uses torch's CUDA generator exactly as the
reference does (``keep_prob + torch.rand((B, 1, 1), dtype)`` floored), one draw per decoder block in block order.
Any ``patch_mask`` is accepted under the sdpa backend: tokens are permuted so that each image's valid tokens come first
(the model is equivariant to token order: positions travel in row_idx / col_idx), which turns every mask into the prefix
mask the attention backward understands; the output is permuted back.
``AE.train_token_packing`` (sdpa backend with a ``patch_mask``): the step runs on the packed NaFlex layout instead (``_Packing``,
include/vitok_b200.h: vtk_pack_plan) -- every image's valid tokens, in token order, padded to 16 rows, so every GEMM, elementwise
kernel and saved activation covers the valid tokens only; attention forward / backward are the packed kernels
(vtk_attention_packed_lse_bf16, vtk_attention_bwd_packed_bf16).  No permutation is needed for masks with holes.
Only the gradients autograd asks for are computed (``_grad_plan``): a parameter with ``requires_grad=False`` gets no
weight-gradient GEMM, no all-reduce and no ``.grad``, and the backward pass stops at the deepest block whose input gradient
something below still needs -- blocks below it keep no activations.  ``AE(encoder=False)`` trains on ``batch["z"]``,
``AE(decoder=False)`` returns z with its graph.
"""
from __future__ import annotations

import contextlib
import ctypes
from typing import Dict, NamedTuple, Optional, Tuple

import torch

from . import _lib

BF = torch.bfloat16


def _check(rc):
    _lib.check(rc)


def _linear(a: torch.Tensor, lda: int, w: torch.Tensor, bias: Optional[torch.Tensor], M: int, N: int, K: int,
            out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out [M, N] = a[:, :K] @ w[:N, :K]^T (+ bias) on the tcgen05 GEMM.  ``a`` / ``w`` may have a row pitch > K."""
    if out is None:
        out = torch.empty(M, N, dtype=BF, device=a.device)
    _check(_lib.load().vtk_linear_bf16(a.data_ptr(), lda, w.data_ptr(), w.stride(0), _lib.ptr(bias), out.data_ptr(), out.stride(0),
                                       M, N, K, _lib.stream_ptr()))
    return out


def _wgrad(dy: torch.Tensor, ld_dy: int, n1: int, x: torch.Tensor, ld_x: int, n2: int, M: int,
           out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """dW [n1, n2] = dy[:, :n1]^T @ x[:, :n2] on the transposed-operand GEMM (both tiles read MN-major; no transpose pass)."""
    if out is None:
        out = torch.empty(n1, n2, dtype=BF, device=dy.device)
    _check(_lib.load().vtk_linear_tn_bf16(dy.data_ptr(), ld_dy, x.data_ptr(), ld_x, out.data_ptr(), n2, n1, n2, M, _lib.stream_ptr()))
    return out


def _dgrad(dy: torch.Tensor, ld_dy: int, w: torch.Tensor, M: int, n_in: int, n_out: int, out: Optional[torch.Tensor] = None,
           accumulate: bool = False) -> torch.Tensor:
    """dX [M, n_in] (+)= dy[:, :n_out] @ w for a weight w [n_out, n_in] used as stored (B operand read MN-major).
    ``accumulate``: the GEMM epilogue adds to what ``out`` holds (fp32 sum, one bf16 rounding) instead of a separate add pass."""
    if out is None:
        out = torch.empty(M, n_in, dtype=BF, device=dy.device)
    _check(_lib.load().vtk_linear_nn_acc_bf16(dy.data_ptr(), ld_dy, w.data_ptr(), w.stride(0), out.data_ptr(), out.stride(0), M, n_in,
                                              n_out, 1 if accumulate else 0, _lib.stream_ptr()))
    return out


def _linear2(a: torch.Tensor, lda: int, w0: torch.Tensor, w1: torch.Tensor, M: int, N: int) -> torch.Tensor:
    """out [M, N] = a[:, :K0] @ w0^T + a[:, K0:K0+K1] @ w1^T: out_proj(attn) + fc2(act) in ONE accumulator, reading both weights as
    stored (no packed [out_proj | fc2] copy: the optimizer changes them every step)."""
    out = torch.empty(M, N, dtype=BF, device=a.device)
    _check(_lib.load().vtk_linear2_bf16(a.data_ptr(), lda, w0.data_ptr(), w0.stride(0), w1.data_ptr(), w1.stride(0), out.data_ptr(), N,
                                        M, N, w0.shape[1], w1.shape[1], _lib.stream_ptr()))
    return out


def _colsum(x: torch.Tensor, ld: int, M: int, C: int) -> torch.Tensor:
    out = torch.zeros(C, dtype=torch.float32, device=x.device)
    _check(_lib.load().vtk_colsum(x.data_ptr(), ld, out.data_ptr(), M, C, _lib.stream_ptr()))
    return out


class _GradSync:
    """Data-parallel gradient averaging overlapped with the backward loop.

    torch DDP (scripts/train_vae.py:172) also works with this model, but because ``model(batch)`` is ONE autograd node
    all gradients reach DDP's reducer together, after the last backward kernel, and the 10 GB all-reduce of the 5B
    model runs un-overlapped.  With ``enable_grad_sync(model)`` the backward loop itself issues an NCCL all-reduce
    (AVG) for each block's weight gradients as soon as its wgrad GEMMs are queued -- NCCL runs them on its own stream
    while the next block's kernels execute -- and the remaining small tensors go out as one flat bucket at the end.
    The gradients autograd hands to the optimizer are already averaged.
    """

    def __init__(self, group=None, min_numel: int = 1 << 16):
        import torch.distributed as dist
        self.dist, self.group, self.min_numel = dist, group, min_numel
        self.world = dist.get_world_size(group)
        self.avg = dist.get_backend(group) == "nccl"     # ReduceOp.AVG is NCCL-only; elsewhere (gloo in the CPU tests): SUM, then scale
        self.pending, self.small = [], []

    def _all_reduce(self, t: torch.Tensor, async_op: bool):
        if self.avg:
            return self.dist.all_reduce(t, op=self.dist.ReduceOp.AVG, group=self.group, async_op=async_op)
        w = self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.group, async_op=async_op)
        return (w, t) if async_op else t.div_(self.world)

    def reduce(self, t: torch.Tensor) -> None:
        if self.world == 1:
            return
        if t.numel() >= self.min_numel and t.is_contiguous():
            self.pending.append(self._all_reduce(t, True))
        else:
            self.small.append(t)

    def finish(self, named: Dict[str, torch.Tensor]) -> None:
        """Average everything not yet reduced (small or strided tensors) as one flat fp32 bucket, then make the
        current stream wait for every outstanding all-reduce."""
        if self.world == 1:
            return
        seen = {id(t) for t in self.small}
        rest = list(self.small) + [t for t in named.values() if t is not None and not getattr(t, "_vtk_reduced", False)
                                   and id(t) not in seen]
        if rest:
            flat = torch.cat([t.reshape(-1).float() for t in rest])
            self._all_reduce(flat, False)
            off = 0
            for t in rest:
                t.copy_(flat[off:off + t.numel()].view_as(t))
                off += t.numel()
        for w in self.pending:
            if isinstance(w, tuple):      # SUM fallback: scale once the sum has arrived
                w[0].wait()
                w[1].div_(self.world)
            else:
                w.wait()
        self.pending, self.small = [], []


def enable_grad_sync(model, process_group=None, broadcast_parameters: bool = True, reserve_sms: Optional[int] = None):
    """Turn on overlapped data-parallel gradient averaging for ``model`` (see _GradSync).  Call once after
    ``torch.distributed.init_process_group``; do NOT also wrap the model in DistributedDataParallel.  With
    ``broadcast_parameters`` the parameters of rank 0 are copied to every rank first (what DDP's constructor does).
    ``reserve_sms``: SMs the persistent GEMM / attention kernels leave free for NCCL's all-reduce CTAs, which run next to the
    backward kernels (include/vitok_b200.h: vtk_set_flag "reserve_sms"); None keeps the process-wide setting."""
    import torch.distributed as dist
    if reserve_sms is not None:
        _lib.set_flag("reserve_sms", int(reserve_sms))
    if process_group is None and dist.get_world_size() > 1 and dist.get_backend() == "nccl":
        # The per-block all-reduces run NEXT TO the backward kernels: give them their own communicator on a high-priority stream so
        # that their CTAs are placed as soon as SMs free up instead of queueing behind the next GEMM's grid.
        try:
            opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
            process_group = dist.new_group(backend="nccl", pg_options=opts)
        except Exception:     # older torch builds without the option: stay on the default group
            process_group = None
    if broadcast_parameters and dist.get_world_size(process_group) > 1:
        with torch.no_grad():
            for p in model.parameters():
                dist.broadcast(p.data, src=dist.get_global_rank(process_group, 0) if process_group is not None else 0,
                               group=process_group)
                torch.autograd.graph.increment_version(p)
    model._grad_sync_group = (process_group,)
    return model


class _SideWeights:
    """bf16 weights of one side (encoder / decoder) as the training kernels read them, taken straight from the parameters
    every step (the optimizer has just changed them) -- nothing is repacked, transposed or concatenated:
      * qkv_proj.weight [3D, D] and fc1.weight [2Hf, D] feed two forward GEMMs that write the column ranges [0, 3D) and
        [qp, qp + 2Hf) of zraw; their data gradients come from the same tensors read MN-major (vtk_linear_nn_acc_bf16, the
        second one accumulating into the first one's output) and their weight gradients from the transposed-operand GEMM
        (vtk_linear_tn_bf16), in the parameters' own row order;
      * out_proj.weight [D, D] and fc2.weight [D, Hf] feed ONE forward GEMM over the concatenated activations
        (vtk_linear2_bf16: two B tensor maps, one accumulator).
    bf16 parameters are used in place (no copy); fp32 parameters (the reference recipe under autocast) are cast once per step.
    """

    def __init__(self, model, side: int):
        from .models.ae import _Scale
        sd = {s[0]: s for s in model._sides()}[side]
        _, lin_a, lin_b, blocks, width, heads = sd
        dev = lin_a.weight.device
        D = width

        def b16(t):
            return t.detach().to(BF).contiguous()

        self.blocks = []
        self.drop = []
        for blk in blocks:
            gamma = b16(blk.layer_scale.gamma) if isinstance(blk.layer_scale, _Scale) else torch.ones(D, dtype=BF, device=dev)
            self.blocks.append((b16(blk.attn.qkv_proj.weight), b16(blk.ffn.fc1.weight), b16(blk.attn.out_proj.weight),
                                b16(blk.ffn.fc2.weight), b16(blk.norm1.weight), b16(blk.attn.norm_q.weight),
                                b16(blk.attn.norm_k.weight), gamma))
            self.drop.append(float(getattr(blk, "drop_path_rate", 0.0) or 0.0))
        self.wa, self.ba, self.wb, self.bb = b16(lin_a.weight), b16(lin_a.bias), b16(lin_b.weight), b16(lin_b.bias)


class _Packing:
    """The packed NaFlex layout of one training step: image b owns rows [cu[b], cu[b+1]) -- its valid tokens in token order, then
    zero rows up to a multiple of 16 -- and the step runs on M = cu[B] rows.  ``plan`` (128-row attention groups) is the work list of
    the attention backward at both head dims and of the d = 64 forward; the d = 128 forward takes 256-row groups (a second plan of
    the same mask: same rows, other groups).  Reading n_valid is the step's one host sync; it sizes every buffer."""

    def __init__(self, mask: torch.Tensor, B: int, N: int):
        self.B, self.N = B, N
        self.mask = mask.bool().contiguous()
        self.plan = _lib.pack_plan(self.mask, 16, 128)
        nv = self.plan["n_valid"].cpu().long()
        self.M = int(((nv + 15) // 16 * 16).sum())
        if self.M == 0:
            raise ValueError("vitok_b200 training: the batch has no valid token (patch_mask is all False)")
        self.groups = {q: int(((nv + q - 1) // q).sum()) for q in (128, 256)}
        self._plans = {128: self.plan}
        self._row_img = None

    def attn_plan(self, qrows: int) -> dict:
        if qrows not in self._plans:
            self._plans[qrows] = _lib.pack_plan(self.mask, 16, qrows)
        return self._plans[qrows]

    def pack(self, x: torch.Tensor) -> torch.Tensor:
        """[B*N, W] bf16 rows -> [M, W] (pad rows 0) with vtk_pack_rows."""
        W = x.shape[1]
        out = torch.empty(self.M, W, dtype=BF, device=x.device)
        _check(_lib.load().vtk_pack_rows(x.data_ptr(), x.stride(0), self.plan["src"].data_ptr(), self.plan["cu"].data_ptr(), self.B,
                                         self.M, out.data_ptr(), W, W, _lib.stream_ptr()))
        return out

    def unpack(self, x: torch.Tensor) -> torch.Tensor:
        """[M, W] -> [B, N, W] (masked tokens 0) with vtk_unpack_rows."""
        W = x.shape[1]
        out = torch.empty(self.B, self.N, W, dtype=BF, device=x.device)
        _check(_lib.load().vtk_unpack_rows(x.data_ptr(), x.stride(0), self.plan["rel"].data_ptr(), self.plan["cu"].data_ptr(), self.B,
                                           self.N, out.data_ptr(), W, W, _lib.stream_ptr()))
        return out

    def pack_index(self, idx: torch.Tensor) -> torch.Tensor:
        """[B, N] int64 token indices (row_idx / col_idx) -> [M], 0 on pad rows."""
        src = self.plan["src"][:self.M].long()
        return torch.where(src >= 0, idx.reshape(-1)[src.clamp_min(0)], 0).contiguous()

    def per_row(self, keep: torch.Tensor) -> torch.Tensor:
        """[B] per-image values -> [M] per packed row (a pad row takes its image's value)."""
        if self._row_img is None:
            cu = self.plan["cu"]
            self._row_img = torch.repeat_interleave(torch.arange(self.B, device=cu.device), (cu[1:] - cu[:-1]).long(),
                                                    output_size=self.M)
        return keep[self._row_img].contiguous()


# the four matrices of a block, in the order of its flat weight-gradient buffer
_BLOCK_MATS = ("attn.qkv_proj.weight", "ffn.fc1.weight", "attn.out_proj.weight", "ffn.fc2.weight")
_SIDE_NAMES = {0: ("patch_embed", "to_code", "encoder_blocks"), 1: ("decoder_embed", "to_pixels", "decoder_blocks")}


class SidePlan(NamedTuple):
    """What the backward pass of one side computes.

    ``stages[i]`` -- how deep block i's backward goes: 0 nothing; 1 ``resid_bwd``; 2 also the dgrad to [attn | act], the SwiGLU and
    attention backward and ``qk_norm_rope_bwd``; 3 also the dgrad to h and ``rmsnorm_bwd`` (the block's input gradient).
    ``wgrads[i]`` -- which of block i's weight-gradient GEMMs run: (qkv_proj, fc1, out_proj, fc2).
    ``save_from`` -- the first block that keeps its activations; blocks below it run their forward and keep nothing.
    ``top`` -- the gradient w.r.t. the last block's output is needed (the dgrad through the side's output projection runs).
    ``dinput`` -- the gradient w.r.t. the side's input (patches, or z) is needed (the dgrad through the input projection runs).
    ``embed`` / ``head`` -- (weight, bias) gradients of the input projection (patch_embed / decoder_embed) and of the output
    projection (to_code / to_pixels)."""
    stages: Tuple[int, ...]
    wgrads: Tuple[Tuple[bool, bool, bool, bool], ...]
    save_from: int
    top: bool
    dinput: bool
    embed: Tuple[bool, bool]
    head: Tuple[bool, bool]


def _grad_plan(needs: Dict[str, bool], depths: Dict[int, int], input_grad: bool) -> Dict[int, SidePlan]:
    """The backward pass's work list from what autograd asks for: ``needs`` maps every parameter name to its requires_grad
    (``ctx.needs_input_grad``), ``depths`` the present sides (0 encoder, 1 decoder) to their block counts, ``input_grad``
    says whether the step's input (patches, or z for a decoder-only model) requires grad.

    A block's input gradient is needed when anything below it needs a gradient: a trainable parameter of an earlier block or of the
    input projection, or the side's input -- for the decoder that is z, needed when anything of the encoder is trainable (or the
    patches require grad), for a decoder-only model when z requires grad.  A block then runs all three stages; otherwise it stops at
    the deepest stage that produces a gradient of one of its own trainable parameters."""

    def side(s: int, below: bool) -> SidePlan:
        emb, head, blk = _SIDE_NAMES[s]
        embed = (needs[emb + ".weight"], needs[emb + ".bias"])
        need = below or any(embed)                     # the gradient w.r.t. the current block's input is consumed below it
        trainable = {int(k.split(".")[1]) for k, v in needs.items() if v and k.startswith(blk + ".")}
        stages, wgrads = [], []
        for i in range(depths[s]):
            p = f"{blk}.{i}."
            w = tuple(needs[p + m] for m in _BLOCK_MATS)
            if need or needs[p + "norm1.weight"]:
                st = 3
            elif w[0] or w[1] or needs[p + "attn.norm_q.weight"] or needs[p + "attn.norm_k.weight"]:
                st = 2
            elif w[2] or w[3] or needs.get(p + "layer_scale.gamma", False):
                st = 1
            else:
                st = 0
            stages.append(st)
            wgrads.append(w)
            need = need or i in trainable
        save_from = next((i for i, st in enumerate(stages) if st), len(stages))
        return SidePlan(tuple(stages), tuple(wgrads), save_from, need, below, embed, (needs[head + ".weight"], needs[head + ".bias"]))

    plans = {}
    z_grad = input_grad
    if 0 in depths:
        plans[0] = side(0, input_grad)
        z_grad = plans[0].top or any(plans[0].head)    # the bottleneck backward (layernorm_bwd, to_code) runs
    if 1 in depths:
        plans[1] = side(1, z_grad)
    return plans


def _block_forward(lib, blk, x: torch.Tensor, rope, kv, B: int, N: int, dims, window: int, keep, keep_prob: float,
                   pk: Optional[_Packing] = None):
    """One transformer block (ae.py:55-65) with everything the backward needs: returns (x_new, (h, zraw, qkv, a2, lse, y)).
    ``pk``: the packed layout (M = pk.M rows; ``keep`` then holds one entry per row)."""
    M, D, heads, d, Hf, qp, ZP, kp = dims
    wqkv, w1, w_o, w_2, n1, nq, nk, gamma = blk
    st = _lib.stream_ptr()
    dev = x.device
    h = torch.empty(M, D, dtype=BF, device=dev)
    _check(lib.vtk_rmsnorm_bf16(x.data_ptr(), D, n1.data_ptr(), h.data_ptr(), D, M, D, 1e-6, st))
    zraw = torch.empty(M, ZP, dtype=BF, device=dev)       # [q | k | v | pad | fc1 value | fc1 gate]
    if qp > 3 * D:                                        # (3D is a multiple of 256 for every preset: no pad, no fill)
        zraw[:, 3 * D:qp].zero_()
    _linear(h, D, wqkv, None, M, 3 * D, D, out=zraw[:, :3 * D])
    _linear(h, D, w1, None, M, 2 * Hf, D, out=zraw[:, qp:])
    qkv = torch.empty(M, 3 * D, dtype=BF, device=dev)
    _check(lib.vtk_qk_norm_rope_fwd(zraw.data_ptr(), ZP, nq.data_ptr(), nk.data_ptr(), rope.data_ptr(), qkv.data_ptr(), 3 * D,
                                    M, heads, d, 1e-6, st))
    a2 = torch.empty(M, kp, dtype=BF, device=dev)
    if kp > D + Hf:
        a2[:, D + Hf:].zero_()
    lse = torch.empty(M, heads, dtype=torch.float32, device=dev)
    base = qkv.data_ptr()
    if pk is None:
        _check(lib.vtk_attention_bf16(base, base + 2 * D, base + 4 * D, 3 * D, a2.data_ptr(), kp, _lib.ptr(kv), B, N, heads, d,
                                      1 if kv is not None else 0, window, lse.data_ptr(), st))
    else:
        qrows = 128 if d <= 64 else 256                  # d <= 64 runs on the 128-row kernel, 64 < d <= 128 on the 256-row one
        pl = pk.attn_plan(qrows)
        _check(lib.vtk_attention_packed_lse_bf16(base, base + 2 * D, base + 4 * D, 3 * D, a2.data_ptr(), kp, pl["n_valid"].data_ptr(),
                                                 pl["cu"].data_ptr(), pl["cuq"].data_ptr(), pl["grp_img"].data_ptr(),
                                                 pl["grp_order"].data_ptr(), B, N, heads, d, M, pk.groups[qrows], lse.data_ptr(), st))
    _check(lib.vtk_swiglu_fwd(zraw.data_ptr(), ZP, qp, a2.data_ptr() + 2 * D, kp, M, Hf, 1, st))
    y = _linear2(a2, kp, w_o, w_2, M, D)
    x_new = torch.empty(M, D, dtype=BF, device=dev)
    _check(lib.vtk_resid_fwd_dp(x.data_ptr(), y.data_ptr(), gamma.data_ptr(), x_new.data_ptr(), M, D, _lib.ptr(keep),
                                N if pk is None else 1, float(keep_prob), st))
    return x_new, (h, zraw, qkv, a2, lse, y)


def _side_forward(lib, model, sw: _SideWeights, side: int, xin: torch.Tensor, row, col, kv, window: int, B: int, N: int, saved: Dict,
                  save_from: int, pk: Optional[_Packing] = None):
    """Blocks ``save_from`` and up keep what their backward needs (``saved["layers"]``); the blocks below keep nothing."""
    width = model.encoder_width if side == 0 else model.decoder_width
    heads = model.encoder_heads if side == 0 else model.decoder_heads
    d = width // heads
    M, D = (B * N if pk is None else pk.M), width
    from .models.ae import _ffn_hidden
    Hf = _ffn_hidden(width, model.mlp_factor)
    qp = ((3 * D + 255) // 256) * 256
    ZP = qp + 2 * Hf
    kp = (D + Hf + 63) // 64 * 64
    dims = (M, D, heads, d, Hf, qp, ZP, kp)
    st = _lib.stream_ptr()
    dev = xin.device
    cin = xin.shape[-1]
    x = _linear(xin, cin, sw.wa, sw.ba, M, D, cin)
    rope = None
    if sw.blocks:
        inv = (1.0 / (model.rope_theta ** (torch.arange(0, d // 2, 2).float() / (d // 2)))).to(dev)
        rope = torch.zeros((M + 31) // 32 * 32, 2 * d, dtype=BF, device=dev)
        _check(lib.vtk_rope_table(row.data_ptr(), col.data_ptr(), inv.data_ptr(), rope.data_ptr(), M, d, st))
    ck = int(getattr(model, "checkpoint", 0) or 0)
    layers = []
    for li, blk in enumerate(sw.blocks):
        keep, keep_prob = None, 1.0
        rate = sw.drop[li]
        if rate > 0.0:
            # stochastic depth (ae.py:15-30): the reference's own draw -- keep_prob + rand((B, 1, 1), dtype) floored -- from
            # torch's CUDA generator, one per block in block order, so a seeded run drops the same images as the reference
            keep_prob = 1.0 - rate
            keep = (keep_prob + torch.rand((B, 1, 1), dtype=BF, device=dev)).floor_().float().reshape(B).contiguous()
            if pk is not None:
                keep = pk.per_row(keep)
        x_new, inner = _block_forward(lib, blk, x, rope, kv, B, N, dims, window, keep, keep_prob, pk)
        if li < save_from:             # no backward reaches this block
            layers.append(None)
        else:                          # activation checkpointing (ae.py:159-160): block i with i % checkpoint == 0 keeps its input only
            layers.append((x, None if (ck > 0 and li % ck == 0) else inner, keep, keep_prob))
        x = x_new
    saved.update(dict(layers=layers, x_final=x, rope=rope if save_from < len(sw.blocks) else None, kv=kv, window=window, xin=xin,
                      dims=dims, pk=pk))
    return x


def _side_backward(lib, model, sw: _SideWeights, side: int, dx: Optional[torch.Tensor], saved: Dict, B: int, N: int, plan: SidePlan,
                   sync: Optional[_GradSync] = None):
    """dx = gradient w.r.t. the output of the last block (None when ``plan.top`` is False).  Runs the stages and weight gradients of
    ``plan``.  Returns ({block index: grads}, dW_a, db_a, d_input); the block grads include the vector gradients of every stage that
    ran, trainable or not (the caller keeps the trainable ones), and entries not computed are None."""
    dims = saved["dims"]
    M, D, heads, d, Hf, qp, ZP, kp = dims
    st = _lib.stream_ptr()
    rope, kv, window, pk = saved["rope"], saved["kv"], saved["window"], saved["pk"]
    grads: Dict[int, Dict[str, torch.Tensor]] = {}
    if dx is None:
        return grads, None, None, None
    dev = dx.device
    for li in range(len(sw.blocks) - 1, plan.save_from - 1, -1):
        stage = plan.stages[li]
        want = dict(zip(("qkv", "fc1", "out", "fc2"), plan.wgrads[li]))
        wqkv, w1, w_o, w_2, n1, nq, nk, gamma = sw.blocks[li]
        x, inner, keep, keep_prob = saved["layers"][li]
        if inner is None:      # checkpointed block: re-run its forward from x (same stochastic-depth draw)
            _, inner = _block_forward(lib, sw.blocks[li], x, rope, kv, B, N, dims, window, keep, keep_prob, pk)
        h, zraw, qkv, a2, lse, y = inner
        saved["layers"][li] = None                                                 # free this block's activations as we go
        dy = torch.empty(M, D, dtype=BF, device=dev)
        dgamma = torch.zeros(D, dtype=torch.float32, device=dev)
        _check(lib.vtk_resid_bwd_dp(dx.data_ptr(), y.data_ptr(), gamma.data_ptr(), dy.data_ptr(), dgamma.data_ptr(), M, D,
                                    _lib.ptr(keep), N if pk is None else 1, float(keep_prob), st))
        bg = dict(gamma=dgamma)
        # the trainable weight gradients of the block live in ONE flat buffer so that they leave as one all-reduce
        sizes = dict(qkv=(3 * D, D), fc1=(2 * Hf, D), out=(D, D), fc2=(D, Hf))
        flat = torch.empty(sum(r * c for k, (r, c) in sizes.items() if want[k]), dtype=BF, device=dev)
        off = 0
        for k, (r, c) in sizes.items():
            if want[k]:
                bg[k] = flat[off:off + r * c].view(r, c)
                off += r * c
        if stage >= 2:
            da2 = torch.empty(M, kp, dtype=BF, device=dev)                        # d[attn | act] = dy @ [out_proj | fc2]
            _dgrad(dy, D, w_o, M, D, D, out=da2[:, :D])
            _dgrad(dy, D, w_2, M, Hf, D, out=da2[:, D:D + Hf])
        if want["out"]:
            _wgrad(dy, D, D, a2, kp, D, M, out=bg["out"])                         # out_proj.weight grad [D, D] = dy^T attn
        if want["fc2"]:
            _wgrad(dy, D, D, a2[:, D:], kp, Hf, M, out=bg["fc2"])                 # fc2.weight grad [D, Hf] = dy^T act
        if stage >= 2:
            dz = torch.empty(M, ZP, dtype=BF, device=dev)
            if qp > 3 * D:
                dz[:, 3 * D:qp].zero_()
            _check(lib.vtk_swiglu_bwd(da2.data_ptr() + 2 * D, kp, zraw.data_ptr(), ZP, qp, dz.data_ptr(), ZP, M, Hf, 1, st))
            delta = torch.empty(M, heads, dtype=torch.float32, device=dev)
            _check(lib.vtk_attn_delta(a2.data_ptr(), kp, da2.data_ptr(), kp, delta.data_ptr(), M, heads, d, st))
            qb, zb = qkv.data_ptr(), dz.data_ptr()
            if pk is None:
                _check(lib.vtk_attention_bwd_bf16(qb, qb + 2 * D, qb + 4 * D, 3 * D, da2.data_ptr(), kp, lse.data_ptr(),
                                                  delta.data_ptr(), zb, zb + 2 * D, zb + 4 * D, ZP, _lib.ptr(kv), B, N, heads, d,
                                                  1 if kv is not None else 0, window, st))
            else:
                pl = pk.plan
                _check(lib.vtk_attention_bwd_packed_bf16(qb, qb + 2 * D, qb + 4 * D, 3 * D, da2.data_ptr(), kp, lse.data_ptr(),
                                                         delta.data_ptr(), zb, zb + 2 * D, zb + 4 * D, ZP, pl["n_valid"].data_ptr(),
                                                         pl["cu"].data_ptr(), pl["cuq"].data_ptr(), pl["grp_img"].data_ptr(),
                                                         pl["grp_order"].data_ptr(), B, heads, d, M, pk.groups[128], st))
            dwqk = torch.zeros(2, d, dtype=torch.float32, device=dev)
            _check(lib.vtk_qk_norm_rope_bwd(dz.data_ptr(), ZP, zraw.data_ptr(), ZP, nq.data_ptr(), nk.data_ptr(), rope.data_ptr(),
                                            dwqk.data_ptr(), M, heads, d, 1e-6, st))
            bg["norm_q"], bg["norm_k"] = dwqk[0], dwqk[1]
        if stage >= 3:
            dh = _dgrad(dz, ZP, wqkv, M, D, 3 * D)                                # dz[:, :3D] @ Wqkv ...
            _dgrad(dz[:, qp:], ZP, w1, M, D, 2 * Hf, out=dh, accumulate=True)     # ... + dz[:, qp:] @ W1, added in the GEMM epilogue
        if want["qkv"]:
            _wgrad(dz, ZP, 3 * D, h, D, D, M, out=bg["qkv"])                      # qkv_proj.weight grad [3D, D]
        if want["fc1"]:
            _wgrad(dz[:, qp:], ZP, 2 * Hf, h, D, D, M, out=bg["fc1"])             # fc1.weight grad [2Hf, D], fc1's own row order
        dx_in = None
        if stage >= 3:
            dx_in = torch.empty(M, D, dtype=BF, device=dev)
            dw1 = torch.zeros(D, dtype=torch.float32, device=dev)
            _check(lib.vtk_rmsnorm_bwd(x.data_ptr(), dh.data_ptr(), n1.data_ptr(), dx.data_ptr(), dx_in.data_ptr(), dw1.data_ptr(),
                                       M, D, 1e-6, st))
            bg["norm1"] = dw1
        if sync is not None and flat.numel():   # this block's weight gradients leave for the all-reduce while the next block computes
            sync.reduce(flat)
            for k in ("qkv", "fc1", "out", "fc2"):
                if want[k]:
                    bg[k]._vtk_reduced = True
        grads[li] = bg
        dx = dx_in
    xin = saved["xin"]
    cin = xin.shape[-1] if xin is not None else 0
    dwa = _wgrad(dx, D, D, xin.reshape(M, cin), cin, cin, M) if plan.embed[0] else None       # [D, cin]
    dba = _colsum(dx, D, M, D) if plan.embed[1] else None
    dxin = _dgrad(dx, D, sw.wa, M, sw.wa.shape[1], D) if plan.dinput else None                 # [M, cin]
    return grads, dwa, dba, dxin


class AETrainFunction(torch.autograd.Function):
    """The training forward of the sides the model has (reference AE.forward, ae.py:245-251): patches -> reconstructed patches,
    patches -> z (``AE(decoder=False)``) or z -> patches (``AE(encoder=False)``), with the gradients ``ctx.needs_input_grad`` asks
    for -- of the parameters and of the input -- and no others (``_grad_plan``)."""

    @staticmethod
    def forward(ctx, model, x, row, col, mask, *params):
        with _lib.device_of(x, *params):
            return AETrainFunction._forward(ctx, model, x, row, col, mask, *params)

    @staticmethod
    def _forward(ctx, model, x_in, row, col, mask, *params):
        lib = _lib.load()
        B, N, cin = x_in.shape
        want = model.pixels_per_token if model.is_encoder else model.channels_per_token
        if cin != want:
            raise RuntimeError(f"shape mismatch: last dim {cin} != {want}")
        dev = x_in.device
        names = [n for n, _ in model.named_parameters()]
        needs = dict(zip(names, ctx.needs_input_grad[5:]))
        sides = {s[0]: len(s[3]) for s in model._sides()}
        plan = _grad_plan(needs, sides, bool(ctx.needs_input_grad[1]))
        pk = _Packing(mask.to(dev), B, N) if _packs(model, mask) else None    # (packed row counts are multiples of 16)
        if pk is None and (B * N) % 8:
            raise ValueError("vitok_b200 training: B * N must be a multiple of 8 (token count is the K dimension of the wgrad GEMMs)")
        sw_ = {side: _SideWeights(model, side) for side in sorted(sides)}
        row = row.to(device=dev, dtype=torch.int64).contiguous()
        col = col.to(device=dev, dtype=torch.int64).contiguous()
        # padded step: each image's key length (train_forward has made every mask a prefix mask); the packed step's attention
        # reads the lengths from its plan.  The sdpa backend (a mask given) ignores the sliding window.
        kv = _lib.kv_len(mask.to(dev).bool()) if mask is not None and pk is None else None
        window = int(model.sw) if (model.sw and mask is None) else -1
        x = (_lib.cast_to_bf16(x_in) if x_in.dtype == torch.float32 else x_in).contiguous().view(B * N, cin)
        M, C = B * N, model.channels_per_token
        if pk is not None:
            x, row, col, M = pk.pack(x), pk.pack_index(row), pk.pack_index(col), pk.M
        saved = {}
        ctx.zlin = None
        for side, w in sw_.items():
            s = saved[side] = {}
            sp = plan[side]
            h = _side_forward(lib, model, w, side, x, row, col, kv, window, B, N, s, sp.save_from, pk)
            if not sp.embed[0]:
                s["xin"] = None
            if not sp.head[0]:
                s["x_final"] = None
            if side == 0:          # latent bottleneck: to_code, then LayerNorm without affine
                zlin = _linear(h, h.shape[1], w.wb, w.bb, M, C, h.shape[1])
                x = torch.empty(M, C, dtype=BF, device=dev)
                _check(lib.vtk_layernorm_fwd(zlin.data_ptr(), x.data_ptr(), M, C, 1e-6, _lib.stream_ptr()))
                if sp.top or any(sp.head):
                    ctx.zlin = zlin
            else:
                x = _linear(h, h.shape[1], w.wb, w.bb, M, model.pixels_per_token, h.shape[1])
        # activations live on ctx (not save_for_backward: they are workspace of the backward kernels, freed block by block while it
        # runs); a second backward through the same graph is therefore refused with a clear error in backward()
        ctx.model, ctx.sw, ctx.saved, ctx.plan = model, sw_, saved, plan
        ctx.shape, ctx.names, ctx.needs = (B, N, cin, C), names, needs
        ctx.param_dtypes = [p.dtype for p in params]
        ctx.in_dtype = x_in.dtype
        ctx.pk = pk
        return x.view(B, N, x.shape[1]) if pk is None else pk.unpack(x)

    @staticmethod
    def backward(ctx, dout):
        if ctx.saved is None:
            raise RuntimeError("vitok_b200 training: backward was already run through this forward pass -- its activations are "
                               "released while the backward kernels consume them (retain_graph / double backward is not "
                               "supported; run model(batch) again)")
        with _lib.device_of(dout):
            return AETrainFunction._backward(ctx, dout)

    @staticmethod
    def _backward(ctx, dout):
        lib = _lib.load()
        model, plan, sw_, saved = ctx.model, ctx.plan, ctx.sw, ctx.saved
        B, N, cin, C = ctx.shape
        pk = ctx.pk
        M = B * N if pk is None else pk.M
        cout = dout.shape[-1]
        dout = dout.to(BF).contiguous().view(B * N, cout)
        if pk is not None:
            dout = pk.pack(dout)           # pad rows 0: no gradient enters them, every weight gradient sums over valid tokens only
        g: Dict[str, Optional[torch.Tensor]] = {}
        grp = getattr(model, "_grad_sync_group", None)
        sync = _GradSync(grp[0]) if grp is not None else None
        dz = dout                          # gradient w.r.t. z (None: nothing below z needs one)
        dinput = None
        if 1 in plan:                      # decoder: to_pixels, blocks, decoder_embed
            sp, w, s = plan[1], sw_[1], saved[1]
            Dd = w.wb.shape[1]
            if sp.head[0]:
                g["to_pixels.weight"] = _wgrad(dout, cout, cout, s["x_final"], Dd, Dd, M)
            if sp.head[1]:
                g["to_pixels.bias"] = _colsum(dout, cout, M, cout)
            dx = _dgrad(dout, cout, w.wb, M, Dd, cout) if sp.top else None
            blocks, g["decoder_embed.weight"], g["decoder_embed.bias"], dz = _side_backward(lib, model, w, 1, dx, s, B, N, sp, sync)
            for i in sorted(blocks):
                _name_block(g, f"decoder_blocks.{i}.", blocks[i])
            dinput = dz
        if ctx.zlin is not None:           # latent bottleneck: LayerNorm (no affine) + to_code, then the encoder
            sp, w, s = plan[0], sw_[0], saved[0]
            dzlin = torch.empty(M, C, dtype=BF, device=dout.device)
            _check(lib.vtk_layernorm_bwd(ctx.zlin.data_ptr(), dz.data_ptr(), dzlin.data_ptr(), M, C, 1e-6, _lib.stream_ptr()))
            De = w.wb.shape[1]
            if sp.head[0]:
                g["to_code.weight"] = _wgrad(dzlin, C, C, s["x_final"], De, De, M)
            if sp.head[1]:
                g["to_code.bias"] = _colsum(dzlin, C, M, C)
            dx = _dgrad(dzlin, C, w.wb, M, De, C) if sp.top else None
            blocks, g["patch_embed.weight"], g["patch_embed.bias"], dinput = _side_backward(lib, model, w, 0, dx, s, B, N, sp, sync)
            for i in sorted(blocks):
                _name_block(g, f"encoder_blocks.{i}.", blocks[i])
        # frozen parameters get no gradient: drop what fell out of a stage that ran for another reason
        g = {n: t for n, t in g.items() if t is not None and ctx.needs.get(n, False)}
        if sync is not None:
            sync.finish(g)
        grads = []
        for name, dt in zip(ctx.names, ctx.param_dtypes):
            t = g.get(name)
            grads.append(None if t is None else t.to(dt).contiguous())
        ctx.saved = ctx.sw = ctx.zlin = ctx.pk = None
        if dinput is not None and ctx.needs_input_grad[1]:
            dinput = (dinput.view(B, N, cin) if pk is None else pk.unpack(dinput)).to(ctx.in_dtype)
        else:
            dinput = None
        return (None, dinput, None, None, None, *grads)


_BLOCK_GRAD_NAMES = dict(qkv="attn.qkv_proj.weight", out="attn.out_proj.weight", fc1="ffn.fc1.weight", fc2="ffn.fc2.weight",
                         norm1="norm1.weight", norm_q="attn.norm_q.weight", norm_k="attn.norm_k.weight", gamma="layer_scale.gamma")


def _name_block(g: Dict[str, torch.Tensor], prefix: str, bg: Dict[str, torch.Tensor]) -> None:
    for k, n in _BLOCK_GRAD_NAMES.items():
        if k in bg:
            g[prefix + n] = bg[k]


def _packs(model, mask: Optional[torch.Tensor]) -> bool:
    """The training step runs on packed rows: opt-in (AE.train_token_packing) and only for a masked (sdpa) batch."""
    return mask is not None and bool(getattr(model, "train_token_packing", False))


def _prefix_permutation(mask: torch.Tensor):
    """(perm, inv) [B, N] int64 such that mask.gather(1, perm) is a prefix mask (valid tokens first, order kept) and
    x.gather(1, perm).gather(1, inv) == x; None when the mask already is a prefix mask (what patchify emits, ops.py:262-263)."""
    m = mask.bool()
    n_valid = m.sum(dim=1, keepdim=True)
    ar = torch.arange(m.shape[1], device=m.device)[None, :]
    if bool((m == (ar < n_valid)).all()):
        return None
    perm = torch.sort((~m).to(torch.int8), dim=1, stable=True).indices
    inv = torch.empty_like(perm)
    inv.scatter_(1, perm, ar.expand_as(perm).contiguous())
    return perm, inv


def train_forward(model, patch_dict: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """AE.forward in training mode (ae.py:245-251): same dict contract as encode -> decode.  ``AE(encoder=False)`` decodes
    ``patch_dict["z"]``; ``AE(decoder=False)`` returns the encode dict, whose z carries the graph."""
    x = patch_dict["patches" if model.is_encoder else "z"]
    if not x.is_cuda:
        raise RuntimeError("vitok_b200.AE: inputs must be CUDA tensors (there is no CPU path)")
    mask = patch_dict.get("patch_mask") if model.attn_backend == "sdpa" else None
    params = [p for _, p in model.named_parameters()]
    row, col = patch_dict["row_idx"], patch_dict["col_idx"]
    # (the packed layout keeps every image's valid tokens in order for any mask: no permutation)
    pp = _prefix_permutation(mask.to(x.device)) if mask is not None and not _packs(model, mask) else None
    if pp is None:
        out = AETrainFunction.apply(model, x, row, col, mask, *params)
    else:
        # a mask with holes: move every image's valid tokens to the front (pure index plumbing; the model only sees positions
        # through row_idx / col_idx, which travel with the tokens), run the prefix-mask path, and move the outputs back
        perm, inv = pp
        pe = perm[:, :, None].expand(-1, -1, x.shape[-1])
        out_p = AETrainFunction.apply(model, x.gather(1, pe), row.to(perm.device).gather(1, perm), col.to(perm.device).gather(1, perm),
                                      mask.to(perm.device).gather(1, perm), *params)
        out = out_p.gather(1, inv[:, :, None].expand(-1, -1, out_p.shape[-1]))
    pdtype = params[0].dtype
    if pdtype == torch.float32 and not torch.is_autocast_enabled():
        out = out.float()
    if not model.is_decoder:
        return {
            "patch_mask": patch_dict.get("patch_mask"), "row_idx": patch_dict["row_idx"], "col_idx": patch_dict["col_idx"],
            "orig_height": patch_dict.get("orig_height"), "orig_width": patch_dict.get("orig_width"), "z": out,
        }
    return {
        "patch_mask": patch_dict.get("patch_mask"), "row_idx": patch_dict.get("row_idx"), "col_idx": patch_dict.get("col_idx"),
        "orig_height": patch_dict.get("orig_height"), "orig_width": patch_dict.get("orig_width"), "patches": out,
    }


class _Charbonnier(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, target, mask, eps):
        B, N, P = pred.shape
        dev = pred.device
        with _lib.device_of(pred):
            pb = pred.to(BF).contiguous()
            tb = target.to(device=dev, dtype=BF).contiguous()
            m8 = nv = None
            if mask is not None:
                mb = mask.to(dev).bool().contiguous()
                m8 = mb.view(torch.uint8)
                nv = mb.sum(dim=1).clamp_min(1).to(torch.int32).contiguous()
            loss_sum = torch.zeros(B, dtype=torch.float32, device=dev)
            dpred = torch.empty_like(pb)
            _check(_lib.load().vtk_charbonnier(pb.data_ptr(), tb.data_ptr(), _lib.ptr(m8), _lib.ptr(nv), loss_sum.data_ptr(),
                                               dpred.data_ptr(), B, N, P, float(eps), _lib.stream_ptr()))
        ctx.dpred = dpred
        ctx.in_dtype = pred.dtype
        return loss_sum.mean()

    @staticmethod
    def backward(ctx, gout):
        dpred = ctx.dpred
        if dpred is None:
            raise RuntimeError("vitok_b200.charbonnier_loss: backward was already run through this loss (its gradient buffer is scaled in place)")
        ctx.dpred = None
        with _lib.device_of(dpred):      # d loss / d pred was written by the forward kernel; times the incoming gradient, in place
            gs = gout.detach().to(device=dpred.device, dtype=torch.float32).reshape(1).contiguous()
            _check(_lib.load().vtk_scale_by_dev(dpred.data_ptr(), gs.data_ptr(), dpred.numel(), _lib.stream_ptr()))
        return dpred.to(ctx.in_dtype), None, None, None


def charbonnier_loss(pred: torch.Tensor, target: torch.Tensor, patch_mask: Optional[torch.Tensor] = None,
                     eps: float = 1e-3) -> torch.Tensor:
    """sqrt(diff^2 + eps^2) averaged over pixels, then over each image's valid tokens, then over the batch
    (scripts/train_vae.py:314-320), forward and gradient in one kernel."""
    return _Charbonnier.apply(pred, target, patch_mask, eps)


_SSIM_FORMATS = {"minus_one_to_one": (0, 0.5), "zero_to_one": (1, 1.0)}
_SSIM_WIN = 11


def _ssim_format(current_format: str) -> int:
    """Format code of the SSIM kernels: values are mapped to [0, 1] before SSIM, (v + 1) / 2 for "minus_one_to_one" and v for
    "zero_to_one"; anything else is a ValueError (SSIM's luminance term is not shift-invariant, so the mapping is part of the
    definition)."""
    if current_format not in _SSIM_FORMATS:
        raise ValueError(f"vitok_b200.ssim: current_format must be one of {sorted(_SSIM_FORMATS)}, got {current_format!r}")
    return _SSIM_FORMATS[current_format][0]


def _ssim_default_tiles(orig_height: torch.Tensor, orig_width: torch.Tensor) -> torch.Tensor:
    """One tile per image, (b, 0, 0, orig_height[b], orig_width[b]): the region ``unpack`` returns.  [B, 5] int32 on the device of
    the sizes."""
    oh = torch.as_tensor(orig_height).reshape(-1)
    ow = torch.as_tensor(orig_width).reshape(-1).to(oh.device)
    if oh.numel() != ow.numel():
        raise ValueError("vitok_b200.ssim: orig_height and orig_width differ in length")
    b = torch.arange(oh.numel(), device=oh.device)
    z = torch.zeros_like(b)
    return torch.stack([b, z, z, oh.to(b.dtype), ow.to(b.dtype)], dim=1).to(torch.int32)


def _ssim_check_tiles(tiles: torch.Tensor, orig_height, orig_width) -> None:
    """Host-side validation of a [T, 5] tile table (image, y0, x0, h, w) against the images' orig_height x orig_width: every tile
    lies inside its image and is at least 11 x 11 (one whole window).  Raises ValueError."""
    if tiles.ndim != 2 or tiles.shape[1] != 5:
        raise ValueError(f"vitok_b200.ssim: tiles must be [T, 5] (image, y0, x0, h, w), got {tuple(tiles.shape)}")
    if tiles.dtype.is_floating_point or tiles.dtype == torch.bool:
        raise ValueError(f"vitok_b200.ssim: tiles must be an integer tensor, got {tiles.dtype}")
    if tiles.shape[0] == 0:
        raise ValueError("vitok_b200.ssim: no tiles")
    if tiles.shape[0] > 65535:
        raise ValueError(f"vitok_b200.ssim: at most 65535 tiles per call, got {tiles.shape[0]}")
    t = tiles.to(torch.int64)
    oh = torch.as_tensor(orig_height).reshape(-1).to(torch.int64)
    ow = torch.as_tensor(orig_width).reshape(-1).to(torch.int64)
    b, y0, x0, h, w = t.unbind(1)
    bad_b = (b < 0) | (b >= oh.numel())
    if bool(bad_b.any()):
        i = int(bad_b.nonzero()[0])
        raise ValueError(f"vitok_b200.ssim: tile {i} names image {int(b[i])} of a batch of {oh.numel()}")
    small = (h < _SSIM_WIN) | (w < _SSIM_WIN)
    if bool(small.any()):
        i = int(small.nonzero()[0])
        raise ValueError(f"vitok_b200.ssim: tile {i} is {int(h[i])} x {int(w[i])}; tiles must be at least {_SSIM_WIN} x {_SSIM_WIN}")
    outside = (y0 < 0) | (x0 < 0) | (y0 + h > oh[b]) | (x0 + w > ow[b])
    if bool(outside.any()):
        i = int(outside.nonzero()[0])
        raise ValueError(f"vitok_b200.ssim: tile {i} = {t[i].tolist()} does not lie inside its image's "
                         f"{int(oh[b[i]])} x {int(ow[b[i]])} pixels")


class _SSIM(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, target, m8, row, col, tiles, geo, fmt):
        B, N, patch, gy, gx, max_h, max_w = geo
        dev = pred.device
        T = tiles.shape[0]
        lib = _lib.load()
        out = torch.empty(T, dtype=torch.float32, device=dev)
        with _lib.device_of(pred, target, tiles):
            ws_bytes = lib.vtk_ssim_workspace_bytes(B, gy, gx, T, max_h, max_w)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            _check(lib.vtk_ssim_fwd(pred.data_ptr(), 0 if pred.dtype == torch.float32 else 1, target.data_ptr(),
                                    0 if target.dtype == torch.float32 else 1, m8.data_ptr(), row.data_ptr(), col.data_ptr(), B, N, patch,
                                    gy, gx, tiles.data_ptr(), T, max_h, max_w, fmt, out.data_ptr(), ws.data_ptr(), ws_bytes,
                                    _lib.stream_ptr()))
        ctx.save_for_backward(pred, target, m8, row, col, tiles)
        ctx.geo, ctx.fmt = geo, fmt
        return out

    @staticmethod
    def backward(ctx, gout):
        pred, target, m8, row, col, tiles = ctx.saved_tensors
        B, N, patch, gy, gx, max_h, max_w = ctx.geo
        T = tiles.shape[0]
        lib = _lib.load()
        with _lib.device_of(pred):
            g = gout.detach().to(device=pred.device, dtype=torch.float32).contiguous()
            dpred = torch.empty_like(pred)
            ws_bytes = lib.vtk_ssim_workspace_bytes(B, gy, gx, T, max_h, max_w)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=pred.device)
            _check(lib.vtk_ssim_bwd(pred.data_ptr(), 0 if pred.dtype == torch.float32 else 1, target.data_ptr(),
                                    0 if target.dtype == torch.float32 else 1, m8.data_ptr(), row.data_ptr(), col.data_ptr(), B, N, patch,
                                    gy, gx, tiles.data_ptr(), T, max_h, max_w, ctx.fmt, g.data_ptr(), dpred.data_ptr(), ws.data_ptr(),
                                    ws_bytes, _lib.stream_ptr()))
        return dpred, None, None, None, None, None, None, None


def ssim(pred: torch.Tensor, batch: dict, patch: int = 16, tiles: Optional[torch.Tensor] = None,
         current_format: str = "minus_one_to_one") -> torch.Tensor:
    """Per-tile SSIM of ``pred`` against ``batch["patches"]`` on the images' canvases: the SSIM tile loss term of the reference's
    training loop (scripts/train_vae.py:328-368), ``loss = charbonnier + w * (1 - ssim(out["patches"], batch)).mean()``.

    pred   : [B, N, 3 p^2] bf16 / fp32 (e.g. ``model(batch)["patches"]``); the gradient flows to it, in its dtype and token layout.
    batch  : the NaFlex dict; "patches" (the target, must not require grad), "patch_mask", "row_idx", "col_idx", "orig_height",
             "orig_width" are used.
    tiles  : int [T, 5] of (image, y0, x0, h, w) in canvas pixels, each inside its image's orig_height x orig_width and at least
             11 x 11; None = one tile per image covering (0, 0, orig_height, orig_width), the region ``unpack`` returns.
    Returns fp32 [T].

    The canvas is the one ``unpatchify(batch, patch)`` builds (masked tokens read 0; where two valid tokens share a cell the
    later one wins), its values mapped to [0, 1] ((v + 1) / 2 for "minus_one_to_one", v for "zero_to_one", no clamping).  SSIM is
    torchmetrics' default (11 x 11 gaussian window, sigma 1.5, K1 = 0.01, K2 = 0.03, data_range 1) per channel, averaged over the 3
    channels and the window positions lying entirely inside the tile.  The kernels read pixels from the token layout and never
    write a canvas; forward and backward are deterministic (fixed reduction order, no float atomics), and a tile's value does not
    depend on the other images of the batch.  One device-to-host copy per call (the tile table, the image sizes and the canvas
    grid, for validation)."""
    fmt = _ssim_format(current_format)
    target = batch["patches"]
    if target.requires_grad:
        raise ValueError("vitok_b200.ssim: batch['patches'] requires grad; the SSIM gradient goes to pred only")
    if not isinstance(patch, int) or patch <= 0:
        raise ValueError(f"vitok_b200.ssim: patch must be a positive int, got {patch!r}")
    if pred.ndim != 3 or pred.shape[-1] != 3 * patch * patch:
        raise ValueError(f"vitok_b200.ssim: pred must be [B, N, 3 * patch^2] = [B, N, {3 * patch * patch}] for patch {patch}, "
                         f"got {tuple(pred.shape)}")
    if tuple(target.shape) != tuple(pred.shape):
        raise ValueError(f"vitok_b200.ssim: pred {tuple(pred.shape)} and batch['patches'] {tuple(target.shape)} differ in shape")
    for name, t in (("pred", pred), ("batch['patches']", target)):
        if t.dtype not in (torch.float32, BF):
            raise ValueError(f"vitok_b200.ssim: {name} must be float32 or bfloat16, got {t.dtype}")
    if not pred.is_cuda or not target.is_cuda:
        raise RuntimeError("vitok_b200.ssim: pred and batch['patches'] must be CUDA tensors (there is no CPU path)")
    dev = pred.device
    B, N, _ = pred.shape
    m8 = batch["patch_mask"].to(dev).bool().contiguous().view(torch.uint8)
    row = batch["row_idx"].to(device=dev, dtype=torch.int64).contiguous()
    col = batch["col_idx"].to(device=dev, dtype=torch.int64).contiguous()
    oh = torch.as_tensor(batch["orig_height"]).reshape(-1).to(device=dev, dtype=torch.int64)
    ow = torch.as_tensor(batch["orig_width"]).reshape(-1).to(device=dev, dtype=torch.int64)
    if oh.numel() != B or ow.numel() != B:
        raise ValueError(f"vitok_b200.ssim: orig_height / orig_width must hold one size per image ({B})")
    tl = _ssim_default_tiles(oh, ow) if tiles is None else torch.as_tensor(tiles)
    if tl.ndim != 2 or tl.shape[1] != 5 or tl.dtype.is_floating_point or tl.dtype == torch.bool:
        _ssim_check_tiles(tl, [1], [1])      # raises the shape / dtype error
    tl = tl.to(device=dev, dtype=torch.int32).contiguous()
    with _lib.device_of(pred, target, m8, row, col):
        ext = torch.empty(2, dtype=torch.int32, device=dev)
        _check(_lib.load().vtk_grid_extent(m8.data_ptr(), row.data_ptr(), col.data_ptr(), B, N, ext.data_ptr(), _lib.stream_ptr()))
        host = torch.cat([ext.long(), oh, ow, tl.reshape(-1).long()]).cpu()     # the one sync of the call
    gy, gx = int(host[0]), int(host[1])
    oh_h, ow_h, tl_h = host[2:2 + B], host[2 + B:2 + 2 * B], host[2 + 2 * B:].reshape(-1, 5)
    _ssim_check_tiles(tl_h, oh_h, ow_h)
    if gy == 0 or gx == 0:
        raise ValueError("vitok_b200.ssim: the batch has no valid token")
    geo = (B, N, patch, gy, gx, int(tl_h[:, 3].max()), int(tl_h[:, 4].max()))
    return _SSIM.apply(pred.contiguous(), target.contiguous(), m8, row, col, tl, geo, fmt)


class FusedAdamW(torch.optim.Optimizer):
    """Multi-tensor AdamW with the reference's optimizer precision (scripts/train_vae.py:200-208 keeps fp32 parameters and fp32
    Adam moments under autocast): every parameter has an fp32 MASTER copy and fp32 ``exp_avg`` / ``exp_avg_sq``; the update runs
    in fp32 on the master and the bf16 model parameter is re-emitted from it in the same pass, so an update smaller than half a
    bf16 ulp of the weight is not lost (at lr 1e-4 that is every weight above ~0.05 and all norm weights).  fp32 model
    parameters are their own master.  torch.optim.AdamW semantics (decoupled weight decay, bias correction); one kernel launch
    per 64 tensors of a param group; 28 bytes of HBM traffic per bf16 parameter.  ``state_dict()`` holds step, master (bf16
    parameters only), exp_avg, exp_avg_sq (and ema) per parameter; ``load_state_dict`` keeps them fp32.

    ``max_grad_norm``: clip by the global L2 norm of every gradient of the step (all groups), as
    ``torch.nn.utils.clip_grad_norm_(params, max_grad_norm)`` before the step would -- coefficient
    ``min(max_grad_norm / (norm + 1e-6), 1)`` in fp32 -- but the gradients are scaled inside the AdamW pass, so ``.grad`` is NOT
    rewritten.  The norm comes from a deterministic pass over the gradients (fp32 sums per 8192-value chunk, added in fp64;
    bit-identical from run to run, however the tensors are grouped) and stays on the device with the coefficient: no host sync.
    ``grad_norm`` is the pre-clip norm of the last step as a 0-dim fp32 CUDA tensor (reading it syncs).  ``float("inf")`` computes
    the norm and never clips.  The parameters must all live on one device.

    ``ema_decay`` (0 <= decay < 1): ``state[p]["ema"]``, an fp32 exponential moving average of the fp32 master weights (not of the
    bf16-rounded parameters, which stand still at small lr while the master moves), updated in the same pass after every step in
    which p has a gradient: ``ema = lerp(ema, master, 1 - decay)`` with torch.lerp's fp32 arithmetic.  It starts at the parameter's
    value when the parameter first gets optimizer state.  ``ema_state_dict(model)`` exports it, ``swap_ema(model)`` evaluates with it.
    HBM traffic: +8 bytes per parameter for the EMA, +2 (bf16 gradients) or +4 (fp32) for the norm pass."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, max_grad_norm=None, ema_decay=None):
        if max_grad_norm is not None:
            max_grad_norm = _real_arg("max_grad_norm", max_grad_norm)
            if not max_grad_norm > 0.0:
                raise ValueError(f"FusedAdamW: max_grad_norm must be > 0 (float('inf') computes the norm and never clips), got {max_grad_norm}")
        if ema_decay is not None:
            ema_decay = _real_arg("ema_decay", ema_decay)
            if not 0.0 <= ema_decay < 1.0:
                raise ValueError(f"FusedAdamW: ema_decay must satisfy 0 <= ema_decay < 1, got {ema_decay}")
        self.max_grad_norm, self.ema_decay = max_grad_norm, ema_decay
        self.grad_norm: Optional[torch.Tensor] = None
        self._norm_ws: Optional[torch.Tensor] = None
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))

    def add_param_group(self, param_group):
        super().add_param_group(param_group)
        if self.max_grad_norm is not None:
            devs = {p.device for g in self.param_groups for p in g["params"]}
            if len(devs) > 1:
                raise ValueError(f"FusedAdamW: max_grad_norm needs every parameter on one device (the global norm is not reduced across "
                                 f"devices); got {sorted(str(d) for d in devs)}")

    @staticmethod
    def _table(items) -> ctypes.Array:
        table = (_lib.AdamwTensor * len(items))()
        for e, (group, p, gr, stt) in zip(table, items):
            master = stt.get("master")
            e.master = (master if master is not None else p).data_ptr()
            e.p16 = p.data_ptr() if master is not None else None
            e.g = gr.data_ptr()
            e.m, e.v = stt["exp_avg"].data_ptr(), stt["exp_avg_sq"].data_ptr()
            e.n = p.numel()
            e.weight_decay = float(group["weight_decay"])
            e.g_is_f32 = 1 if gr.dtype == torch.float32 else 0
        return table

    def _clip_coef(self, lib, items) -> torch.Tensor:
        """Queue the norm pass over every gradient of ``items``; returns the device coefficient [1] and sets ``grad_norm``."""
        devs = {it[1].device for it in items}
        if len(devs) > 1:
            raise ValueError(f"FusedAdamW: max_grad_norm needs every parameter on one device; got {sorted(str(d) for d in devs)}")
        dev = devs.pop()
        table = self._table(items)
        slots = int(lib.vtk_grad_norm_slots(table, len(items)))
        if self._norm_ws is None or self._norm_ws.numel() != max(slots, 1) or self._norm_ws.device != dev:
            self._norm_ws = torch.empty(max(slots, 1), dtype=torch.float32, device=dev)
        norm_coef = torch.empty(2, dtype=torch.float32, device=dev)     # fresh per step: a grad_norm the caller holds stays valid
        with torch.cuda.device(dev):
            st = _lib.stream_ptr()
            _check(lib.vtk_grad_sumsq_multi(table, len(items), self._norm_ws.data_ptr(), 0, st))
            _check(lib.vtk_grad_norm_finish(self._norm_ws.data_ptr(), slots, float(self.max_grad_norm), norm_coef.data_ptr(), st))
        self.grad_norm = norm_coef[0]
        return norm_coef[1:]

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        lib = _lib.load()
        per_group = []            # (group, p, grad, state) of every parameter with a gradient, group by group
        for group in self.param_groups:
            items = []
            for p in group["params"]:
                if p.grad is None:
                    continue
                if p.dtype not in (BF, torch.float32) or not p.is_cuda:
                    raise RuntimeError("FusedAdamW: parameters must be bf16 or fp32 CUDA tensors")
                if not p.is_contiguous():
                    raise RuntimeError("FusedAdamW: parameters must be contiguous")
                stt = self.state[p]
                if not stt:
                    stt["step"] = 0
                    if p.dtype == BF:
                        stt["master"] = p.detach().float()
                    stt["exp_avg"] = torch.zeros(p.shape, dtype=torch.float32, device=p.device)
                    stt["exp_avg_sq"] = torch.zeros(p.shape, dtype=torch.float32, device=p.device)
                if self.ema_decay is not None and "ema" not in stt:
                    stt["ema"] = p.detach().to(torch.float32, copy=True)
                stt["step"] += 1
                gr = p.grad
                if gr.dtype not in (BF, torch.float32):
                    gr = gr.float()
                gr = gr.contiguous()
                items.append((group, p, gr, stt))
            per_group.append(items)
        coef = None
        if self.max_grad_norm is not None and any(per_group):
            coef = self._clip_coef(lib, [it for items in per_group for it in items])
        for group, items in zip(self.param_groups, per_group):
            b1, b2 = group["betas"]
            by_dev: Dict[torch.device, list] = {}
            for it in items:
                by_dev.setdefault(it[1].device, []).append(it)
            for dev, dev_items in by_dev.items():
                # parameters of a group share lr / betas / eps / weight decay; their step counts agree unless a parameter
                # got its first gradient later -- launch per distinct step
                for step in sorted({it[3]["step"] for it in dev_items}):
                    sel = [it for it in dev_items if it[3]["step"] == step]
                    table = self._table(sel)
                    ema = None
                    if self.ema_decay is not None:
                        ema = (ctypes.c_void_p * len(sel))(*[it[3]["ema"].data_ptr() for it in sel])
                    with torch.cuda.device(dev):
                        _check(lib.vtk_adamw_multi_ex(table, ema, len(sel), float(group["lr"]), float(b1), float(b2), float(group["eps"]),
                                                      int(step), 1.0, _lib.ptr(coef), float(self.ema_decay or 0.0), _lib.stream_ptr()))
                    for _, p, _, _ in sel:
                        torch.autograd.graph.increment_version(p)   # the kernel wrote p in place: invalidate packed copies
        return loss

    def load_state_dict(self, state_dict):
        """torch.optim.Optimizer.load_state_dict, except that the fp32 state (master, exp_avg, exp_avg_sq, ema) stays fp32: the base
        class casts floating-point state to each parameter's dtype, which would round it to bf16 for bf16 parameters."""
        super().load_state_dict(state_dict)
        saved_ids = [i for g in state_dict["param_groups"] for i in g["params"]]
        params = [p for g in self.param_groups for p in g["params"]]
        for i, p in zip(saved_ids, params):
            saved = state_dict["state"].get(i)
            if not saved:
                continue
            for k in _FP32_STATE:
                if k in saved:
                    self.state[p][k] = saved[k].to(device=p.device, dtype=torch.float32, copy=True)

    def _ema_params(self, model, remove_duplicate: bool = True):
        if self.ema_decay is None:
            raise ValueError("FusedAdamW: this optimizer keeps no EMA (construct it with ema_decay)")
        return [(n, p, self.state[p]) for n, p in model.named_parameters(remove_duplicate=remove_duplicate)
                if p in self.state and "ema" in self.state[p]]

    @torch.no_grad()
    def ema_state_dict(self, model) -> Dict[str, torch.Tensor]:
        """``model.state_dict()`` with every parameter that has an EMA replaced by the EMA cast to the parameter's dtype (the release
        weights of the run); parameters without optimizer state (frozen, or never given a gradient) and buffers keep their current
        values.  The EMA tensors are copied, never aliased."""
        sd = model.state_dict()
        for n, p, stt in self._ema_params(model, remove_duplicate=False):
            sd[n] = stt["ema"].to(dtype=p.dtype, copy=True)
        return sd

    @contextlib.contextmanager
    def swap_ema(self, model):
        """Evaluate ``model`` with its EMA weights, in place and without extra memory::

            with opt.swap_ema(model):
                model.eval(); ...

        On entry a bf16 parameter with an EMA is overwritten by bf16(ema) and an fp32 one swaps storage with its EMA; on exit a bf16
        parameter is re-emitted from its fp32 master and an fp32 one swaps back.  The bf16 exit is exact because after every step a
        bf16 parameter equals bf16(master) -- the invariant this relies on: do not write a bf16 parameter other than through this
        optimizer while it has state (a change made inside the block is lost on exit).  Version counters are bumped both ways, so
        AE's packed inference weights rebuild.  Parameters without an EMA are left alone."""
        swapped = []
        try:
            for _, p, stt in self._ema_params(model):
                if p.dtype == BF:
                    p.data.copy_(stt["ema"])
                else:
                    p.data, stt["ema"] = stt["ema"], p.data
                torch.autograd.graph.increment_version(p)
                swapped.append((p, stt))
            yield model
        finally:
            for p, stt in swapped:
                if p.dtype == BF:
                    p.data.copy_(stt["master"])
                else:
                    p.data, stt["ema"] = stt["ema"], p.data
                torch.autograd.graph.increment_version(p)


_FP32_STATE = ("master", "exp_avg", "exp_avg_sq", "ema")


def _real_arg(name: str, value) -> float:
    if isinstance(value, bool) or not isinstance(value, (int, float)):
        raise ValueError(f"FusedAdamW: {name} must be a real number or None, got {value!r}")
    return float(value)
