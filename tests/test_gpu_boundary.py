"""GPU: the stand-alone forward() surfaces of the drop-in boundary (SURVEY.md 8(b)) against the UNMODIFIED reference modules in fp32 on a
B200, same seeded weights (stored results, tests/reference_golden.py: fixed samples of the large outputs): Bottleneck.forward, FPN.forward, RPNHead.forward, RegionProposalNetwork.forward (eval),
FCOSHead.forward, --output_voxel_scores, and the training-mode forward of NeRFRegionProposalNetwork driven by torch.autograd +
torch.optim exactly as run_rpn.py:384-395 drives it.  Tolerance: 2e-3 norm-wise (fp16 activations; weights fp16 or hi+lo pairs)."""
import math
import os

import numpy as np
import pytest
import torch

from oracle import ref_gpu
from tests.reference_golden import recorded, sample_index

pytestmark = [pytest.mark.gpu]
SAMPLE = 1024                                                    # stored reference values per output tensor


def _rel(a, b):
    return ((a.float() - b.float()).norm() / (b.float().norm() + 1e-30)).item()


def _sampled(ts, seed):
    """Shape and a fixed sample of the values of each tensor (flat index order)."""
    out = {}
    for i, t in enumerate(ts):
        idx = torch.from_numpy(sample_index(t.numel(), SAMPLE, seed + i)).to(t.device)
        out[f"shape{i}"], out[f"val{i}"] = np.array(t.shape), t.reshape(-1)[idx].float().cpu().numpy()
    return out


def _check_sampled(ts, want, seed, tol):
    for i, t in enumerate(ts):
        assert tuple(t.shape) == tuple(want[f"shape{i}"]), (t.shape, want[f"shape{i}"])
        v = t.reshape(-1)[torch.from_numpy(sample_index(t.numel(), SAMPLE, seed + i)).to(t.device)].float().cpu()
        rel = _rel(v, torch.from_numpy(want[f"val{i}"]))
        assert rel <= tol, (i, rel)


@pytest.fixture(autouse=True)
def _no_tf32():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False; torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _randomise_bn(m, g):
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm3d):
            mod.running_mean.copy_(torch.randn(mod.running_mean.shape, generator=g) * 0.1)
            mod.running_var.copy_(torch.rand(mod.running_var.shape, generator=g) * 0.5 + 0.75)
            mod.weight.data.copy_(torch.rand(mod.weight.shape, generator=g) * 0.5 + 0.75)
            mod.bias.data.copy_(torch.randn(mod.bias.shape, generator=g) * 0.1)


@pytest.mark.parametrize("inplanes,planes,stride", [(64, 64, 1), (256, 128, 2), (512, 128, 1)])
def test_bottleneck_forward(inplanes, planes, stride):
    from nerf_rpn_b200.model.feature_extractor import Bottleneck
    def block(cls):                                              # seeded init, then BatchNorm statistics and affine parameters off their defaults
        torch.manual_seed(inplanes + planes)
        ds = None
        if stride != 1 or inplanes != planes * 4:
            ds = torch.nn.Sequential(torch.nn.Conv3d(inplanes, planes * 4, 1, stride=stride, bias=False), torch.nn.BatchNorm3d(planes * 4))
        m = cls(inplanes, planes, stride, ds)
        g = torch.Generator().manual_seed(inplanes + planes)
        with torch.no_grad():
            _randomise_bn(m, g)
        return m.cuda().eval(), torch.randn(2, inplanes, 9, 12, 10, generator=g).cuda()

    def reference():
        rb, x = block(ref_gpu.load().feature_extractor.Bottleneck)
        with torch.no_grad():
            return _sampled([rb(x)], 1)
    want = recorded(f"bottleneck_{inplanes}_{planes}_{stride}", reference)
    ours, x = block(Bottleneck)
    with torch.no_grad():
        got = ours(x)
    _check_sampled([got], want, 1, 2e-3)


def test_fpn_forward():
    from nerf_rpn_b200.model.fpn import FPN
    g = torch.Generator().manual_seed(4)
    xs = [torch.randn(1, c, *d, generator=g).cuda() for c, d in zip([128, 256, 512, 512], [(25, 20, 13), (13, 10, 7), (7, 5, 4), (4, 3, 2)])]

    def reference():
        torch.manual_seed(3)
        rf = ref_gpu.load().fpn.FPN([128, 256, 512, 512], 256, 4).cuda().eval()
        with torch.no_grad():
            return _sampled(rf(xs), 10)
    want = recorded("fpn", reference)
    torch.manual_seed(3)
    ours = FPN([128, 256, 512, 512], 256, 4).cuda().eval()
    with torch.no_grad():
        got = ours(xs)
    assert isinstance(got, tuple) and len(got) == 4
    _check_sampled(got, want, 10, 2e-3)


@pytest.mark.parametrize("rotated", [False, True])
def test_rpn_head_and_region_proposal_network_forward(rotated):
    """RPNHead.forward -> (logits, bbox_reg) and RegionProposalNetwork.forward(meshes, features, sizes) -> (boxes, levels, {}, scores): head
    outputs within 2e-3 of the reference's; proposals: same count within 2 % and >= 95 % of the reference's top-100 matched at IoU >= 0.7."""
    from nerf_rpn_b200 import ops
    from nerf_rpn_b200.model.anchor import AnchorGenerator3D, RPNHead
    from nerf_rpn_b200.model.feature_extractor import Bottleneck, ResNet_FPN_256
    from nerf_rpn_b200.model.rpn import RegionProposalNetwork
    g = torch.Generator().manual_seed(8)
    dims = (64, 96, 80)
    fd = [(16, 24, 20), (8, 12, 10), (4, 6, 5), (2, 3, 3)]
    feats = [torch.randn(1, 256, *d, generator=g).cuda() * 0.5 for d in fd]
    meshes = torch.zeros(1, 4, *dims, device="cuda")

    def reference():
        rm = ref_gpu.build_reference_model(rotated=rotated, seed=0, spread=30.0).cuda().eval()
        with torch.no_grad():
            wl, wb = rm.rpn.head(feats)
            wboxes, wlv, _, wscores = rm.rpn(meshes, feats, [dims])
        return dict(_sampled(wl + wb, 20), count=np.array(wboxes[0].shape[0]), top_boxes=wboxes[0][:100].cpu().numpy())
    want = recorded(f"rpn_head_and_rpn_{'obb' if rotated else 'aabb'}", reference)
    torch.manual_seed(0)                                         # the reference's init order (run_rpn.py): backbone, anchor generator, head
    ResNet_FPN_256(Bottleneck, [3, 4, 6, 3], input_dim=4, is_max_pool=True)
    ag = AnchorGenerator3D(ref_gpu.ANCHOR_SIZES, ref_gpu.ASPECT)
    head = RPNHead(256, 13, 4, rotate=rotated)
    with torch.no_grad():
        head.cls_logits.weight.mul_(30.0)
    rpn = RegionProposalNetwork(ag, head, 0.35, 0.2, 256, 0.5, dict(training=2500, testing=2500), dict(training=2500, testing=2500), 0.3,
                                score_thresh=0.0, rotated_bbox=rotated).cuda().eval()
    with torch.no_grad():
        gl, gb = head(feats)
        _check_sampled(gl + gb, want, 20, 2e-3)
        gboxes, glv, losses, gscores = rpn(meshes, feats, [dims])
    assert losses == {} and len(gboxes) == 1
    nw, ng = int(want["count"]), gboxes[0].shape[0]
    print(f"RegionProposalNetwork.forward ({'OBB' if rotated else 'AABB'}): {ng} proposals, reference {nw}")
    assert abs(nw - ng) <= max(3, 0.02 * nw)
    k = min(100, nw, ng)
    iou = ops.iou3d_matrix(torch.from_numpy(want["top_boxes"][:k]).contiguous().cuda(), gboxes[0].contiguous().cuda())
    matched = (iou.max(dim=1)[0] >= 0.7).float().mean().item()
    assert matched >= 0.95, matched


def test_fcos_head_forward():
    from nerf_rpn_b200.model.fcos.fcos import FCOSHead
    def head(cls):
        torch.manual_seed(5)
        h = cls(256, 4, [4, 8, 16, 32], True, True, True)
        with torch.no_grad():
            for i, sc in enumerate(h.scales):
                sc.scale.fill_(1.0 + 0.1 * i)
            h.cls_logits.weight.mul_(20.0); h.bbox_pred.weight.mul_(20.0); h.bbox_pred.bias.fill_(0.5)
        return h.cuda().eval()
    g = torch.Generator().manual_seed(6)
    feats = [torch.randn(1, 256, *d, generator=g).cuda() for d in [(12, 10, 8), (6, 5, 4), (3, 3, 2)]]

    def reference():
        with torch.no_grad():
            return _sampled([t for out in head(ref_gpu.load().fcos.FCOSHead)(feats) for t in out], 30)
    want = recorded("fcos_head", reference)
    with torch.no_grad():
        got = head(FCOSHead)(feats)
    _check_sampled([t for out in got for t in out], want, 30, 4e-3)        # 4 GroupNorm'ed layers deep, fp16 activations


def test_output_voxel_scores(tmp_path):
    """--output_voxel_scores (rpn.py:538-549): npz with the per-level maximum objectness logit, same keys / shapes as the reference's file."""
    from nerf_rpn_b200.model.anchor import AnchorGenerator3D, RPNHead
    from nerf_rpn_b200.model.feature_extractor import Bottleneck, ResNet_FPN_256
    from nerf_rpn_b200.model.nerf_rpn import NeRFRegionProposalNetwork
    g = torch.Generator().manual_seed(1000)
    x = torch.rand(48, 64, 40, 4, generator=g).permute(3, 0, 1, 2).contiguous().cuda()
    pw, pg = str(tmp_path / "ref.npz"), str(tmp_path / "ours.npz")

    def reference():
        rm = ref_gpu.build_reference_model(rotated=False, seed=0, spread=30.0).cuda().eval()
        with torch.no_grad():
            rm([x.clone()], objectness_output_paths=[pw])
        with np.load(pw) as z:
            return {k: z[k] for k in z.files}
    w = recorded("output_voxel_scores", reference)
    torch.manual_seed(0)                                         # the reference's init order: backbone, anchor generator, head
    backbone = ResNet_FPN_256(Bottleneck, [3, 4, 6, 3], input_dim=4, is_max_pool=True)
    ag = AnchorGenerator3D(ref_gpu.ANCHOR_SIZES, ref_gpu.ASPECT)
    head = RPNHead(256, 13, 4, rotate=False)
    with torch.no_grad():
        head.cls_logits.weight.mul_(30.0)
    model = NeRFRegionProposalNetwork(backbone, ag, head, rpn_pre_nms_top_n_test=2500, rpn_post_nms_top_n_test=2500, rpn_nms_thresh=0.3).cuda().eval()
    with torch.no_grad():
        model([x.clone()], objectness_output_paths=[pg])
    o = np.load(pg)
    assert sorted(w) == sorted(o.files) == ["0", "1", "2", "3"]
    for k in sorted(w):
        assert w[k].shape == o[k].shape
        assert np.linalg.norm(w[k] - o[k]) <= 3e-3 * np.linalg.norm(w[k]) + 1e-6


def test_training_forward_is_autograd_and_optimizer_compatible():
    """The reference's own loop (run_rpn.py:384-395) on our module mirror: losses = model(grids, boxes); weighted sum; loss.backward();
    clip_grad_norm_; torch.optim.AdamW.step() -- three iterations, the loss on a fixed scene must go down and every parameter must
    receive a finite gradient."""
    from nerf_rpn_b200.model.anchor import AnchorGenerator3D, RPNHead
    from nerf_rpn_b200.model.feature_extractor import Bottleneck, ResNet_FPN_256
    from nerf_rpn_b200.model.nerf_rpn import NeRFRegionProposalNetwork
    torch.manual_seed(0)
    backbone = ResNet_FPN_256(Bottleneck, [3, 4, 6, 3], input_dim=4, is_max_pool=True)
    head = RPNHead(256, 13, 4, rotate=True)
    model = NeRFRegionProposalNetwork(backbone, AnchorGenerator3D(ref_gpu.ANCHOR_SIZES, ref_gpu.ASPECT), head, rpn_fg_iou_thresh=0.35, rpn_bg_iou_thresh=0.2,
                                      rotated_bbox=True).cuda().train()
    g = torch.Generator().manual_seed(11)
    dims = (64, 96, 80)
    grid = torch.rand(*dims, 4, generator=g).permute(3, 0, 1, 2).contiguous().cuda()
    d = torch.tensor(dims, dtype=torch.float32)
    gt = torch.cat([torch.rand(12, 3, generator=g) * (d - 8) + 4, torch.rand(12, 3, generator=g) * 20 + 6, (torch.rand(12, 1, generator=g) - 0.5) * math.pi], 1).cuda()
    opt = torch.optim.AdamW(model.parameters(), lr=3e-4, weight_decay=0.01)
    hist = []
    for it in range(4):
        torch.manual_seed(7)                                            # same sampled anchors every iteration
        _, losses, _ = model([grid], [gt])
        losses["loss_rpn_box_reg"] *= 5.0
        losses["loss_rpn_box_reg_2d"] *= 0.0
        loss = losses["loss_objectness"] + losses["loss_rpn_box_reg"] + losses["loss_rpn_box_reg_2d"]
        loss.backward()
        assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in model.parameters())
        torch.nn.utils.clip_grad_norm_(model.parameters(), 0.1)
        opt.step(); opt.zero_grad()
        hist.append(loss.item())
    print("loss over 4 autograd-driven steps:", [round(v, 4) for v in hist])
    assert hist[-1] < hist[0]


PAIRS = 256                                                      # stored reference results: a fixed sample of the box pairs


def _pairs(n, seed):
    g = torch.Generator().manual_seed(seed)
    a = torch.cat([torch.rand(n, 3, generator=g) * 6, torch.rand(n, 3, generator=g) * 8 + 2, (torch.rand(n, 1, generator=g) - 0.5) * math.pi], 1).cuda()
    b = a + torch.cat([torch.randn(n, 3, generator=g), torch.randn(n, 3, generator=g) * 0.5, torch.randn(n, 1, generator=g) * 0.3], 1).cuda()
    b[:, 3:6] = b[:, 3:6].abs() + 0.5
    return a, b, torch.from_numpy(sample_index(n, PAIRS, seed)).cuda()


def test_cal_iou_3d_verbose_and_autograd_vs_reference():
    """cal_iou_3d(verbose=True) and its gradient (the IoU-type regression losses: RotatedIOULoss rpn.py:133-165) against the reference's torch
    chain + autograd on a B200, on a fixed sample of 256 of 4 000 pairs: values bit-identical (iou, corners, z_range, u3d), gradients of the loss
    -log((I + 1) / (U + 1)) within 1e-3 of the gradient's scale on the pairs away from a change of polygon topology (>= 99 % of them)."""
    from nerf_rpn_b200.model.rotated_iou.oriented_iou_loss import cal_iou_3d
    from nerf_rpn_b200._lib import lib
    lib().nrpn_set_iou_mode(3)                     # the reference's CUDA build's rounding order (the library default; conftest pins 0 for this module)
    n = 4000
    a, b, idx = _pairs(n, 31)

    def run(fn):
        a1, b1 = a.clone().requires_grad_(True), b.clone().requires_grad_(True)
        iou, c1, c2, zr, u = fn(a1[None], b1[None], verbose=True)
        loss = -torch.log((iou * u + 1.0) / (u + 1.0)).sum()
        loss.backward()
        return [t[idx] for t in (iou.detach()[0], c1.detach()[0], c2.detach()[0], zr.detach()[0], u.detach()[0], a1.grad, b1.grad)], \
            [a1.grad.abs().max().item(), b1.grad.abs().max().item()]

    def reference():
        vals, scales = run(ref_gpu.load().oriented_iou_loss.cal_iou_3d)
        return dict({f"out{k}": v.cpu().numpy() for k, v in enumerate(vals)}, scale=np.array(scales))
    want = recorded("cal_iou_3d_verbose", reference)
    r = [torch.from_numpy(want[f"out{k}"]).cuda() for k in range(7)]
    o, _ = run(cal_iou_3d)
    assert (r[0] > 0).sum() > 0.8 * PAIRS
    for k in range(5):
        assert torch.equal(r[k].view(torch.int32), o[k].view(torch.int32)), f"verbose output {k} differs"
    for k in (5, 6):
        err = (r[k] - o[k]).abs().max(dim=1)[0]
        scale = float(want["scale"][k - 5])
        frac = (err <= 1e-3 * scale).float().mean().item()
        print(f"cal_iou_3d backward, grad {'a' if k == 5 else 'b'}: {frac:.4f} of the pairs within 1e-3 of the gradient scale {scale:.3f}, median err {err.median().item():.2e}")
        assert frac >= 0.99
    # without requires_grad and verbose the fast path returns the same values
    assert torch.equal(cal_iou_3d(a[None], b[None])[0][idx], o[0])


@pytest.mark.parametrize("enclosing", ["smallest", "aligned", "pca"])
def test_cal_giou_diou_3d_vs_reference(enclosing):
    """cal_giou_3d / cal_diou_3d (oriented_iou_loss.py:109-150) against the reference's own functions on a B200, on a fixed sample of 256 of 3 000
    pairs: values within 1e-5 (1e-4 for the pca variant), gradients of the summed loss within 1e-3 of the gradient's scale on >= 99 % of the
    pairs (the IoU part is differentiated numerically on our side)."""
    from nerf_rpn_b200.model.rotated_iou.oriented_iou_loss import cal_diou_3d, cal_giou_3d
    from nerf_rpn_b200._lib import lib
    lib().nrpn_set_iou_mode(3)
    a, b, idx = _pairs(3000, 37)

    def run(fn):
        a1, b1 = a.clone().requires_grad_(True), b.clone().requires_grad_(True)
        out = fn(a1[None], b1[None], enclosing)
        out[0].sum().backward()
        return [out[0].detach()[0][idx], a1.grad[idx], b1.grad[idx]], [a1.grad.abs().max().item(), b1.grad.abs().max().item()]

    def reference():
        oil = ref_gpu.load().oriented_iou_loss
        out = {}
        for name, fn in (("giou", oil.cal_giou_3d), ("diou", oil.cal_diou_3d)):
            vals, scales = run(fn)
            out.update({f"{name}{k}": v.cpu().numpy() for k, v in enumerate(vals)}, **{f"{name}_scale": np.array(scales)})
        return out
    want = recorded(f"cal_giou_diou_3d_{enclosing}", reference)
    for name, ours in (("giou", cal_giou_3d), ("diou", cal_diou_3d)):
        r = [torch.from_numpy(want[f"{name}{k}"]).cuda() for k in range(3)]
        o, _ = run(ours)
        err = (r[0] - o[0]).abs().max().item()
        print(f"{name} [{enclosing}] loss max abs err {err:.2e}")
        assert err <= (1e-4 if enclosing == "pca" else 1e-5)          # pca: closed-form eigenvectors of a nearly isotropic 2x2 matrix amplify the last bits
        for k in (1, 2):
            e = (r[k] - o[k]).abs().max(dim=1)[0]
            scale = float(want[f"{name}_scale"][k - 1])
            frac = (e <= 1e-3 * scale).float().mean().item()
            print(f"{name} [{enclosing}] grad {'a' if k == 1 else 'b'}: {frac:.4f} within 1e-3 of scale {scale:.3f}")
            assert frac >= 0.99
