"""Device-side training augmentation (nerf_rpn_b200/augment.py, nrpn_augment_scene) against the reference's own
BaseDataset.augment_rpn_inputs / rotate_and_scale_scene (datasets.py:109-163, 290-329) run on the CPU with the same seeded `random`
stream (stored under tests/golden/reference/, tests/reference_golden.py): same decisions, same boxes, same grid."""
import hashlib
import random

import numpy as np
import pytest
import torch

from tests.reference_golden import recorded, sample_index

pytestmark = pytest.mark.gpu


def _scene(dims, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand((*dims, 4), generator=g).permute(3, 0, 1, 2)           # the dataset's (4, W, L, H) view of a (W, L, H, 4) array


def _boxes(dims, n, obb, seed):
    g = torch.Generator().manual_seed(seed + 100)
    ctr = torch.rand(n, 3, generator=g) * torch.tensor(dims, dtype=torch.float32)
    size = 2 + torch.rand(n, 3, generator=g) * 6
    if obb:
        return torch.cat([ctr, size, (torch.rand(n, 1, generator=g) - 0.5) * 3.0], 1)
    return torch.cat([ctr - size / 2, ctr + size / 2], 1)


GRID_SAMPLE = 512                                                            # stored values of each rotated grid


def _reference_results(obb, dims):
    """The reference's augment_rpn_inputs on each seed: the next `random` draw after it, its boxes, the grid's shape, a digest of the grid
    (exact cases) and a fixed sample of its values (compared where the grid was rotated: our trilinear weights round differently)."""
    from oracle import ref_gpu
    ref = ref_gpu.load(need_k1=False)
    out = {"next_draw": [], "boxes": [], "digest": [], "grid": [], "shape": []}
    for seed in range(24):
        grid = _scene(dims, seed)
        boxes = None if obb is None else _boxes(dims, 9, obb, seed)
        random.seed(seed)
        want_g, want_b = ref.datasets.BaseDataset.augment_rpn_inputs(grid, boxes, 0.5, 0.5, 0.6)
        out["next_draw"].append(random.random())
        out["boxes"].append(np.zeros((9, 7 if obb else 6), np.float32) if want_b is None else want_b.numpy())
        out["digest"].append(_digest(want_g))
        out["grid"].append(want_g.reshape(-1)[torch.from_numpy(sample_index(want_g.numel(), GRID_SAMPLE, seed))].numpy() if obb
                           else np.zeros(GRID_SAMPLE, np.float32))              # no rotation without oriented boxes: the digest decides
        out["shape"].append(want_g.shape)
    return {k: np.array(v) for k, v in out.items()}


def _digest(t):
    return hashlib.sha256(t.contiguous().numpy().tobytes()).hexdigest() + str(tuple(t.shape))


@pytest.mark.parametrize("obb", [True, False, None])
def test_augment_rpn_inputs_matches_reference(obb):
    """Same decisions, boxes and grid as the reference's augment_rpn_inputs (stored: tests/golden/reference/)."""
    from nerf_rpn_b200 import augment
    dims = (20, 26, 12)
    want = recorded(f"augment_grids_{ {True: 'obb', False: 'aabb', None: 'none'}[obb]}", lambda: _reference_results(obb, dims))
    seen = set()
    for seed in range(24):
        grid = _scene(dims, seed)
        boxes = None if obb is None else _boxes(dims, 9, obb, seed)
        random.seed(seed)
        aug = augment.draw_augmentation(0.5, 0.5, 0.6, bool(obb))
        assert random.random() == want["next_draw"][seed]                     # the same number of draws in the same order
        seen.add((aug.rot90, aug.flip_x, aug.flip_y, aug.angle is not None))
        random.seed(seed)
        got_g, got_b = augment.augment_rpn_inputs(grid.cuda(), boxes, 0.5, 0.5, 0.6)
        got_g = got_g.cpu()
        assert tuple(got_g.shape) == tuple(want["shape"][seed])
        if aug.angle is None:
            assert _digest(got_g) == want["digest"][seed], (seed, aug)
        else:                                                                 # trilinear weights differ in the last fp32 bits
            v = got_g.reshape(-1)[torch.from_numpy(sample_index(got_g.numel(), GRID_SAMPLE, seed))]
            assert (v - torch.from_numpy(want["grid"][seed])).abs().max().item() < 2e-5, (seed, aug)
        if boxes is None:
            assert got_b is None
        else:
            assert torch.allclose(got_b, torch.from_numpy(want["boxes"][seed]), rtol=0, atol=1e-5), (seed, aug)
    assert len(seen) >= (10 if obb else 6)                                    # the seeds exercised the combinations


def test_augment_full_size_round_trip_and_layouts():
    """160x256x256: four rot90 are the identity, a flip twice is the identity; NCDHW-contiguous input gives the same result as the dataset view."""
    from nerf_rpn_b200 import augment
    g = torch.rand((160, 256, 256, 4), device="cuda").permute(3, 0, 1, 2)
    a = augment.Augmentation(rot90=True)
    x = g
    for _ in range(4):
        x = augment.augment_scene(x, a)
    assert torch.equal(x, g)
    f = augment.Augmentation(flip_x=True, flip_y=True)
    assert torch.equal(augment.augment_scene(augment.augment_scene(g, f), f), g)
    r = augment.Augmentation(rot90=True, flip_y=True, angle=0.1, scale=1.05)
    assert torch.equal(augment.augment_scene(g.contiguous(), r), augment.augment_scene(g, r))
    ident = augment.Augmentation(angle=0.0, scale=1.0)
    assert (augment.augment_scene(g, ident) - g).abs().max().item() < 1e-4   # resampling at the voxel centres themselves


def test_augment_rejects_cpu_and_z_down():
    from nerf_rpn_b200 import augment
    with pytest.raises(RuntimeError):
        augment.augment_scene(torch.zeros(4, 4, 4, 4), augment.Augmentation(rot90=True))
    with pytest.raises(NotImplementedError):
        augment.augment_rpn_inputs(torch.zeros(4, 4, 4, 4, device="cuda"), None, 0.5, 0.5, 0.5, z_up=False)
