"""GPU: the FCOS training loss kernels (csrc/fcos_loss.cu through nerf_rpn_b200/model/fcos/loss.py) against
  * tests/golden/fcos_loss.npz = outputs of the unmodified reference (fcos/loss.py) from tools/make_golden.py: targets, losses, gradients;
  * the reference itself run on a B200 (stored under tests/golden/reference/: digests of the exact results, fixed samples), at the locations of BASELINE config 3 (200 x 200 x 130, strides 4..32),
    every loss type of both heads -- including the rotated-IoU losses that only exist on a GPU (K1 vertex sort);
  * the numpy oracle for the streamed-ground-truth path (G > one shared-memory chunk).
Tolerances: labels identical; targets bit-identical (AABB) / 1e-5 (OBB corner arithmetic); losses 1e-5 .. 1e-4 relative; gradients 2e-4
element-wise for the kernels' own terms, 3e-3 of the gradient's norm for the rotated-IoU term (IoU backward = fp64 clip + central differences; 2e-2
without centre sampling, where barely-overlapping positives sit at the IoU's kinks)."""
import argparse
import hashlib
import math
import os

import numpy as np
import pytest
import torch

from oracle import fcos_loss_oracle as O
from oracle import ref_gpu
from tests.reference_golden import recorded, sample_index

from .test_fcos_loss_cpu import CASES, STRIDES, WEIGHTS, load_case, per_scene

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, "fcos_loss.npz"))


def fcos_args(rotated, loss_type, radius, add_l1, proj2d=0.0):
    return argparse.Namespace(num_convs=1, norm_reg_targets=True, centerness_on_reg=True, rotated_bbox=rotated, pre_nms_thresh=0.0, pre_nms_top_n=100,
                              nms_thresh=0.3, fpn_post_nms_top_n=100, min_size=0.0, center_sampling_radius=radius, iou_loss_type=loss_type,
                              use_additional_l1_loss=add_l1, proj2d_loss_weight=proj2d)


def our_module(rotated, loss_type, radius, add_l1, proj2d=0.0):
    from nerf_rpn_b200.model.fcos.fcos import FCOSModule
    return FCOSModule(fcos_args(rotated, loss_type, radius, add_l1, proj2d), 256, STRIDES)


@pytest.mark.parametrize("name", list(CASES))
def test_kernels_match_reference_golden(golden, name):
    c = load_case(golden, name)
    mod = our_module(c["rotated"], c["loss_type"], c["radius"], c["add_l1"], c["proj2d"])
    cls, reg, ctr = ([torch.tensor(a, device="cuda", requires_grad=True) for a in c[k]] for k in ("cls", "reg", "ctr"))
    locs = mod.compute_locations(cls)
    sizes = golden[f"{name}/sizes"]
    masks = mod.compute_padding_masks(locs, [tuple(int(v) for v in s) for s in sizes]) if c["batch"] > 1 else None
    gts = [torch.tensor(g, device="cuda") for g in c["gt"]]
    lab, rt = mod.loss_evaluator.prepare_targets(locs, gts)
    for l in range(4):
        np.testing.assert_array_equal(lab[l].cpu().numpy(), c["labels"][l])
        if c["rotated"]:
            np.testing.assert_allclose(rt[l].cpu().numpy(), c["reg_targets"][l], rtol=1e-5, atol=1e-5)
        else:
            np.testing.assert_array_equal(rt[l].cpu().numpy(), c["reg_targets"][l])
    _, _, losses = mod._forward_train(locs, cls, reg, ctr, gts, masks)
    got = [losses[k].item() for k in ("loss_cls", "loss_reg", "loss_centerness")]
    rotated_iou = c["rotated"] and c["loss_type"] != "smooth_l1"
    gathered = rotated_iou or c["proj2d"] > 0                    # terms evaluated on the gathered positives (torch ops around the IoU kernels)
    np.testing.assert_allclose(got[0], c["losses"][0], rtol=1e-5)
    np.testing.assert_allclose(got[2], c["losses"][2], rtol=1e-5)
    np.testing.assert_allclose(got[1], c["losses"][1], rtol=2e-4 if rotated_iou else 2e-5)      # golden rotated IoU: CPU run with a stand-in vertex sort
    (WEIGHTS[0] * losses["loss_cls"] + WEIGHTS[1] * losses["loss_reg"] + WEIGHTS[2] * losses["loss_centerness"]).backward()
    for l in range(4):
        np.testing.assert_allclose(cls[l].grad.cpu().numpy(), c["dcls"][l], rtol=2e-4, atol=1e-7)
        np.testing.assert_allclose(ctr[l].grad.cpu().numpy(), c["dctr"][l], rtol=2e-4, atol=1e-7)
        if not gathered:
            np.testing.assert_allclose(reg[l].grad.cpu().numpy(), c["dreg"][l], rtol=2e-4, atol=1e-7)
    if gathered:
        a = torch.cat([t.grad.flatten() for t in reg]).cpu().double(); b = torch.cat([torch.tensor(t).flatten() for t in c["dreg"]]).double()
        assert ((a - b).norm() / b.norm()).item() < (3e-3 if rotated_iou else 1e-4)


def test_deterministic_and_forward_only(golden):
    c = load_case(golden, "aabb_giou")
    mod = our_module(False, "giou", 1.5, False)
    cls, reg, ctr = ([torch.tensor(a, device="cuda") for a in c[k]] for k in ("cls", "reg", "ctr"))
    locs = mod.compute_locations(cls)
    masks = mod.compute_padding_masks(locs, [tuple(int(v) for v in s) for s in golden["aabb_giou/sizes"]])
    gts = [torch.tensor(g, device="cuda") for g in c["gt"]]
    runs = [mod.loss_evaluator(locs, cls, reg, ctr, gts, masks) for _ in range(3)]          # no requires_grad: the forward-only launch
    for r in runs[1:]:
        assert all(torch.equal(a, b) for a, b in zip(r, runs[0]))
    assert not runs[0][0].requires_grad
    np.testing.assert_allclose([t.item() for t in runs[0]], c["losses"], rtol=1e-5)


def scene_inputs(rotated, batch, seed, mesh=(200, 200, 130), n_gt=30):
    g = torch.Generator().manual_seed(seed)
    grids = [tuple(int(math.ceil(m / s)) for m in mesh) for s in STRIDES]
    cls = [(torch.randn(batch, 1, *gr, generator=g) * 2 - 2).cuda().requires_grad_(True) for gr in grids]
    reg = [torch.cat([torch.rand(batch, 6, *gr, generator=g) * 3 + 0.1] + ([torch.randn(batch, 2, *gr, generator=g) * 0.3] if rotated else []), 1)
           .cuda().requires_grad_(True) for gr in grids]
    ctr = [torch.randn(batch, 1, *gr, generator=g).cuda().requires_grad_(True) for gr in grids]
    sizes = [mesh, (180, 200, 120)][:batch]
    gts = []
    for b in range(batch):
        sz = torch.tensor(sizes[b], dtype=torch.float32)
        ext = torch.rand(n_gt, 3, generator=g) * torch.tensor([90.0, 90.0, 60.0]) + 6.0
        ctrs = torch.rand(n_gt, 3, generator=g) * sz
        gts.append((torch.cat([ctrs, ext, (torch.rand(n_gt, 1, generator=g) - 0.5) * math.pi], 1) if rotated
                    else torch.cat([ctrs - ext / 2, ctrs + ext / 2], 1)).cuda())
    return grids, sizes, cls, reg, ctr, gts


FULL_CASES = [(False, "iou", 1.5, False, 2, 0.0), (False, "giou", 0.0, False, 1, 0.0), (False, "linear_iou", 1.5, False, 1, 0.0),
              (False, "smooth_l1", 1.5, False, 2, 0.0), (True, "smooth_l1", 1.5, False, 2, 0.0), (True, "iou", 1.5, True, 2, 0.0),
              (True, "linear_iou", 1.5, False, 1, 0.0), (True, "giou", 1.5, True, 1, 0.0), (True, "diou", 0.0, False, 1, 0.0),
              (True, "smooth_l1", 1.5, False, 1, 0.5), (True, "iou", 1.5, True, 1, 0.3)]


FULL_SAMPLE = 4096                                           # stored reference values per tensor


def _digest(ts):
    h = hashlib.sha256()
    for t in ts:
        h.update(str(tuple(t.shape)).encode()); h.update(t.detach().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()


def _sample(t, seed):
    return t.detach().reshape(-1)[torch.from_numpy(sample_index(t.numel(), FULL_SAMPLE, seed)).to(t.device)].cpu()


def _full_size_reference(args, cls, reg, ctr, sizes, gts, batch, rotated):
    """FCOSLossComputation of the reference on a B200: digests of its locations, padding masks, labels (and AABB targets), fixed samples of the
    OBB targets and of every input gradient, its three losses; for the gathered regression gradient, a sample of its non-zero entries."""
    ref = ref_gpu.load()
    rmod = ref.fcos.FCOSModule(args, 256, STRIDES).cuda()
    locs = rmod.compute_locations(cls)
    masks = rmod.compute_padding_masks(locs, sizes) if batch > 1 else None
    lab, rt = rmod.loss_evaluator.prepare_targets(locs, [t.clone() for t in gts])
    out = dict(locs=_digest(locs), masks=_digest(masks or []), labels=_digest(lab), n_pos=sum(int((x > 0).sum()) for x in lab))
    if rotated:
        out.update({f"rt{l}": _sample(rt[l], 10 + l).numpy() for l in range(4)})
    else:
        out["rt"] = _digest(rt)
    w = rmod.loss_evaluator(locs, cls, reg, ctr, gts, masks)
    out["losses"] = np.array([t.item() for t in w])
    (WEIGHTS[0] * w[0] + WEIGHTS[1] * w[1] + WEIGHTS[2] * w[2]).backward()
    for name, lst in (("cls", cls), ("reg", reg), ("ctr", ctr)):
        out.update({f"d{name}{l}": _sample(t.grad, 20 + l).numpy() for l, t in enumerate(lst)})
    b = torch.cat([t.grad.flatten() for t in reg])
    nz = torch.nonzero(b).reshape(-1)
    pick = nz[torch.from_numpy(sample_index(nz.numel(), FULL_SAMPLE, 30)).to(nz.device)]
    out.update(dreg_nonzero=np.array(nz.numel()), dreg_index=pick.cpu().numpy(), dreg_values=b[pick].cpu().numpy())
    for t in cls + reg + ctr:
        t.grad = None
    return out


@pytest.mark.parametrize("rotated,loss_type,radius,add_l1,batch,proj2d", FULL_CASES)
def test_full_size_against_reference_on_the_gpu(rotated, loss_type, radius, add_l1, batch, proj2d):
    """FCOSLossComputation of the reference, run on a B200, at BASELINE config 3's locations (94 k per scene); stored under tests/golden/reference/
    (exact results as digests, fixed samples of the targets and gradients)."""
    grids, sizes, cls, reg, ctr, gts = scene_inputs(rotated, batch, 40 + len(loss_type) + int(rotated))
    name = f"fcos_loss_full_{'obb' if rotated else 'aabb'}_{loss_type}_r{radius:g}_l1{int(add_l1)}_b{batch}_p{proj2d:g}"
    want = recorded(name, lambda: _full_size_reference(fcos_args(rotated, loss_type, radius, add_l1, proj2d), cls, reg, ctr, sizes, gts, batch, rotated))
    mod = our_module(rotated, loss_type, radius, add_l1, proj2d)
    locs = mod.compute_locations(cls)
    assert _digest(locs) == want["locs"]
    masks = mod.compute_padding_masks(locs, sizes) if batch > 1 else None
    assert _digest(masks or []) == want["masks"]
    got_lab, got_rt = mod.loss_evaluator.prepare_targets(locs, gts)
    assert _digest(got_lab) == want["labels"]
    assert int(want["n_pos"]) > 200
    if rotated:
        for l in range(4):
            torch.testing.assert_close(_sample(got_rt[l], 10 + l), torch.from_numpy(want[f"rt{l}"]), rtol=1e-5, atol=2e-5)
    else:
        assert _digest(got_rt) == want["rt"]
    g_cls, g_reg, g_ctr = mod.loss_evaluator(locs, cls, reg, ctr, gts, masks)
    (WEIGHTS[0] * g_cls + WEIGHTS[1] * g_reg + WEIGHTS[2] * g_ctr).backward()
    w_cls, w_reg, w_ctr = (torch.tensor(float(v), device="cuda") for v in want["losses"])
    rotated_iou = rotated and loss_type != "smooth_l1"
    gathered = rotated_iou or proj2d > 0
    torch.testing.assert_close(g_cls, w_cls, rtol=2e-5, atol=0)
    torch.testing.assert_close(g_ctr, w_ctr, rtol=2e-5, atol=0)
    torch.testing.assert_close(g_reg, w_reg, rtol=1e-4 if rotated_iou else 2e-5, atol=0)
    for l in range(4):
        torch.testing.assert_close(_sample(cls[l].grad, 20 + l), torch.from_numpy(want[f"dcls{l}"]), rtol=2e-4, atol=1e-8)
        torch.testing.assert_close(_sample(ctr[l].grad, 20 + l), torch.from_numpy(want[f"dctr{l}"]), rtol=2e-4, atol=1e-8)
        if not gathered:
            torch.testing.assert_close(_sample(reg[l].grad, 20 + l), torch.from_numpy(want[f"dreg{l}"]), rtol=2e-4, atol=1e-8)
    if gathered:
        a_full = torch.cat([t.grad.flatten() for t in reg])
        a = a_full[torch.from_numpy(want["dreg_index"]).to(a_full.device)].cpu().double(); b = torch.from_numpy(want["dreg_values"]).double()
        # without centre sampling every location inside a box is a positive, also those whose predicted box barely touches the target: there the
        # intersection polygon changes its vertex set within the finite-difference step of the IoU backward (measured 7.6e-3 on the B200)
        assert ((a - b).norm() / b.norm()).item() < ((3e-3 if radius > 0 else 2e-2) if rotated_iou else 1e-4)
        nz_a, nz_b = int((a_full != 0).sum()), int(want["dreg_nonzero"])
        assert nz_a == nz_b or abs(nz_a - nz_b) < 0.01 * nz_b


@pytest.mark.parametrize("dim", [6, 7])
def test_streamed_ground_truth_beyond_one_chunk(dim):
    """G = 700 boxes: three shared-memory chunks; labels / targets == the numpy oracle (first minimum across chunk borders)."""
    from nerf_rpn_b200 import ops
    rng = np.random.default_rng(dim)
    grids = [(20, 24, 16), (10, 12, 8), (5, 6, 4), (3, 3, 2)]
    locs = O.compute_locations(grids, STRIDES)
    G = 700
    ext = rng.random((G, 3)) * 50 + 4
    ctrs = rng.random((G, 3)) * np.array([80, 96, 64])
    ext[100:400] = (12.0, 20.0, 8.0)                          # integer boxes of equal volume: exact ties, the FIRST must win, also across chunks
    ctrs[100:400] = np.floor(ctrs[100:400])
    gt = (np.concatenate([ctrs - ext / 2, ctrs + ext / 2], 1) if dim == 6 else np.concatenate([ctrs, ext, (rng.random((G, 1)) - 0.5) * math.pi], 1)).astype(np.float32)
    if dim == 7:
        gt[100:400, 6] = 0.0
    want_l, want_r = O.targets(locs, STRIDES, gt, 1.5, True)
    got_l, got_r = ops.fcos_targets(torch.tensor(np.concatenate(locs)).cuda(), [len(p) for p in locs], STRIDES, torch.tensor(gt).cuda(), 1.5, True)
    assert want_l.sum() > 200
    np.testing.assert_array_equal(got_l.cpu().numpy(), want_l)
    pos = want_l > 0                                          # the reference leaves box 0's distances at the negatives: compared too
    np.testing.assert_allclose(got_r.cpu().numpy(), want_r, rtol=1e-5, atol=1e-5)
    assert pos.any()


def test_rejects_cpu_tensors_and_bad_shapes():
    from nerf_rpn_b200 import ops
    mod = our_module(False, "iou", 1.5, False)
    cls = [torch.zeros(1, 1, 2, 2, 2)]
    with pytest.raises(RuntimeError, match="CUDA"):
        mod.loss_evaluator([torch.zeros(8, 3)], cls, [torch.zeros(1, 6, 2, 2, 2)], cls, [torch.zeros(0, 6)], None)
    with pytest.raises(ValueError):
        ops.fcos_targets(torch.zeros(8, 3, device="cuda"), [7], [4], torch.zeros(1, 6, device="cuda"), 1.5)
