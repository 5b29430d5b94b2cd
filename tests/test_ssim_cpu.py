"""vitok_b200.ssim: everything that runs before the kernels -- default tiles, the format mapping and argument validation."""
import pytest
import torch

import vitok_b200 as vb
from vitok_b200 import train


def test_default_tiles_cover_each_image():
    oh, ow = torch.tensor([11, 130, 512]), torch.tensor([300, 131, 16])
    t = train._ssim_default_tiles(oh, ow)
    assert t.dtype == torch.int32
    assert t.tolist() == [[0, 0, 0, 11, 300], [1, 0, 0, 130, 131], [2, 0, 0, 512, 16]]
    train._ssim_check_tiles(t, oh, ow)        # the default tiles are always valid


def test_format_mapping():
    assert train._ssim_format("minus_one_to_one") == 0
    assert train._ssim_format("zero_to_one") == 1
    for bad in ("0_255", "as_is", "", None):
        with pytest.raises(ValueError, match="current_format"):
            train._ssim_format(bad)


@pytest.mark.parametrize("tile,msg", [
    ([0, 0, 0, 10, 20], "at least 11"),
    ([0, 0, 0, 20, 10], "at least 11"),
    ([0, -1, 0, 11, 11], "inside"),
    ([0, 0, -3, 11, 11], "inside"),
    ([0, 20, 0, 11, 11], "inside"),           # 20 + 11 > 30
    ([1, 0, 30, 11, 11], "inside"),           # 30 + 11 > 40
    ([2, 0, 0, 11, 11], "image"),
    ([-1, 0, 0, 11, 11], "image"),
])
def test_bad_tiles(tile, msg):
    oh, ow = torch.tensor([30, 64]), torch.tensor([64, 40])
    with pytest.raises(ValueError, match=msg):
        train._ssim_check_tiles(torch.tensor([[0, 0, 0, 11, 11], tile]), oh, ow)


def test_tile_table_shape_and_dtype():
    oh, ow = torch.tensor([30]), torch.tensor([30])
    train._ssim_check_tiles(torch.tensor([[0, 19, 19, 11, 11], [0, 0, 0, 30, 30]]), oh, ow)   # edge tiles are inside
    with pytest.raises(ValueError, match=r"\[T, 5\]"):
        train._ssim_check_tiles(torch.tensor([[0, 0, 0, 11]]), oh, ow)
    with pytest.raises(ValueError, match="integer"):
        train._ssim_check_tiles(torch.tensor([[0.0, 0, 0, 11, 11]]), oh, ow)
    with pytest.raises(ValueError, match="no tiles"):
        train._ssim_check_tiles(torch.zeros(0, 5, dtype=torch.int64), oh, ow)


def _batch(B=2, N=4, patch=4):
    return {"patches": torch.zeros(B, N, 3 * patch * patch), "patch_mask": torch.ones(B, N, dtype=torch.bool),
            "row_idx": torch.zeros(B, N, dtype=torch.int64), "col_idx": torch.zeros(B, N, dtype=torch.int64),
            "orig_height": torch.full((B,), 8), "orig_width": torch.full((B,), 8)}


def test_argument_errors_before_any_device_work():
    b = _batch()
    pred = torch.zeros_like(b["patches"])
    with pytest.raises(ValueError, match="current_format"):
        vb.ssim(pred, b, 4, current_format="0_255")
    with pytest.raises(ValueError, match="requires grad"):
        vb.ssim(pred, {**b, "patches": b["patches"].clone().requires_grad_(True)}, 4)
    with pytest.raises(ValueError, match="patch"):
        vb.ssim(pred, b, 16)
    with pytest.raises(ValueError, match="patch"):
        vb.ssim(pred, b, 0)
    with pytest.raises(ValueError, match="differ in shape"):
        vb.ssim(pred[:1], b, 4)
    with pytest.raises(ValueError, match="float32 or bfloat16"):
        vb.ssim(pred.half(), b, 4)
    with pytest.raises(RuntimeError, match="CUDA"):
        vb.ssim(pred, b, 4)
