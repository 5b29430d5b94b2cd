"""vitok_b200 -- B200-native drop-in for the ViTok-v2 AE encode/decode hot path.

Mirrors the hot-path surface of the reference package ``vitok`` (vitok/__init__.py:3-28):
``AE``, ``decode_variant``, ``preprocess``, ``postprocess``, ``unpatchify``, ``unpack``,
``patchify``, ``patch_collate_fn``, ``build_transform``, ``OPS``.  All tensor work runs in
libvitok_b200.so (hand-written sm_100a kernels); there is no CPU fallback.
"""
from .models.ae import AE, Model, decode_variant
from .pp import (OPS, build_transform, pack_images, parse_op, patchify_batch, patchify_packed, postprocess, preprocess,
                 unpack, unpatchify)
from .data import patch_collate_fn
from .graphs import GraphedAE, GraphedCodec
from .parallel import shard_by_tokens, shard_range
from .pretrained import list_pretrained, load_pretrained, save_pretrained
from .train import FusedAdamW, charbonnier_loss, enable_grad_sync, ssim

__version__ = "0.1.0"
__all__ = ["AE", "Model", "decode_variant", "build_transform", "parse_op", "OPS", "patch_collate_fn", "preprocess",
           "postprocess", "unpatchify", "unpack", "patchify_batch", "pack_images", "patchify_packed", "charbonnier_loss", "ssim", "FusedAdamW", "enable_grad_sync", "load_pretrained", "list_pretrained",
           "save_pretrained", "shard_range", "shard_by_tokens", "GraphedAE", "GraphedCodec"]
