"""Host side of the training augmentation (nerf_rpn_b200/augment.py): the random draws and the box transforms against the reference's own
BaseDataset.augment_rpn_inputs (datasets.py:109-163), stored under tests/golden/reference/ (tests/reference_golden.py); the grid kernel is
covered by tests/test_gpu_augment.py."""
import os
import random
import sys

import numpy as np
import pytest
import torch

from tests.reference_golden import recorded

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ref():
    stub = os.path.join(ROOT, "tools", "ref_stub")                 # import-time stand-in for the reference's native op on a CPU-only host
    sys.path.insert(0, stub)
    try:
        from oracle import ref_gpu
        return ref_gpu.load(need_k1=False)
    finally:
        sys.path.remove(stub)


def _cases(obb):
    dims = (20, 26, 12)
    g = torch.Generator().manual_seed(5)
    for seed in range(40):
        grid = torch.rand(4, *dims, generator=g)
        ctr = torch.rand(9, 3, generator=g) * torch.tensor(dims, dtype=torch.float32)
        size = 2 + torch.rand(9, 3, generator=g) * 6
        boxes = torch.cat([ctr, size, (torch.rand(9, 1, generator=g) - 0.5) * 3], 1) if obb else torch.cat([ctr - size / 2, ctr + size / 2], 1)
        yield seed, dims, grid, boxes


@pytest.mark.parametrize("obb", [True, False])
def test_draws_and_boxes_match_reference(obb):
    """Boxes and the number of `random` draws against the reference's augment_rpn_inputs (stored: its boxes, and the next draw of the
    `random` stream after it, which matches only when both consumed the same draws)."""
    from nerf_rpn_b200 import augment

    def reference():
        ref = _ref()
        boxes, after = [], []
        for seed, dims, grid, b in _cases(obb):
            random.seed(seed)
            boxes.append(ref.datasets.BaseDataset.augment_rpn_inputs(grid, b, 0.5, 0.5, 0.6)[1].numpy())
            after.append(random.random())
        return dict(boxes=np.stack(boxes), next_draw=np.array(after))
    want = recorded(f"augment_boxes_{'obb' if obb else 'aabb'}", reference)
    for seed, dims, grid, boxes in _cases(obb):
        random.seed(seed)
        aug = augment.draw_augmentation(0.5, 0.5, 0.6, obb)
        assert random.random() == want["next_draw"][seed]
        assert (aug.angle is not None) <= obb
        got = augment.augment_boxes(boxes, aug, dims)
        assert torch.allclose(got, torch.from_numpy(want["boxes"][seed]), rtol=0, atol=1e-5), (seed, aug)


def test_probability_validation_and_identity():
    from nerf_rpn_b200 import augment
    with pytest.raises(ValueError):
        augment.draw_augmentation(1.5, 0.0, 0.0, True)
    with pytest.raises(ValueError):
        augment.draw_augmentation(0.0, -0.1, 0.0, True)
    a = augment.draw_augmentation(0.0, 0.0, 0.0, True)
    assert a.identity
    b = torch.rand(3, 7)
    assert torch.equal(augment.augment_boxes(b, a, (8, 8, 8)), b)
    assert augment.augment_boxes(None, a, (8, 8, 8)) is None
