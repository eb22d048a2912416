"""GPU: the CUDA path against the UNMODIFIED reference run on a B200: its real native op K1 (`sort_vertices`, built by its own setup.py
for sm_100), its torch-CUDA IoU chain and Python NMS loop, its fp32 cuDNN network, and its unmodified driver run_rpn.py launched on top of
the drop-in shims.

The reference's results are stored under tests/golden/reference/ (tests/reference_golden.py: samples of the large outputs) and refreshed by
running this module with NRPN_RECORD_REFERENCE=<dir> where oracle/_ref is staged.  The two driver tests run the reference's own script and
are skipped where oracle/_ref is not staged."""
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import pytest
import torch

from oracle import ref_gpu
from tests.reference_golden import recorded, recording, sample_index

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = [pytest.mark.gpu]
needs_staged_reference = pytest.mark.skipif(not ref_gpu.available(), reason="runs the reference's own run_rpn.py: oracle/_ref not staged")


def rand_obb(n, g, extent=30.0, smin=1.0, smax=11.0):
    return torch.cat([torch.rand(n, 3, generator=g) * extent, torch.rand(n, 3, generator=g) * (smax - smin) + smin,
                      (torch.rand(n, 1, generator=g) - 0.5) * math.pi], 1)


# ------------------------------------------------------------------------------------------------ K1 (row a16)
def _reference_polygons():
    """The tensors box_intersection_2d.py:121-141 hands to the reference's kernel for 200 000 random box pairs, and its answer, on 3 072 of
    the defined polygons (num_valid <= 8; num_valid > 8 writes out of bounds in the reference, :103), most of them with >= 3 vertices."""
    ref = ref_gpu.load()
    b2d, oil = ref.box_intersection_2d, ref.oriented_iou_loss
    g = torch.Generator().manual_seed(21)
    n = 200_000
    a, b = rand_obb(n, g, extent=12.0).cuda()[None], rand_obb(n, g, extent=12.0).cuda()[None]
    c1 = oil.box2corners_th(a[..., [0, 1, 3, 4, 6]]); c2 = oil.box2corners_th(b[..., [0, 1, 3, 4, 6]])
    inters, mask_inter = b2d.box_intersection_th(c1, c2)
    c12, c21 = b2d.box_in_box_th(c1, c2)
    vertices, mask = b2d.build_vertices(c1, c2, c12, c21, inters, mask_inter)
    num_valid = torch.sum(mask.int(), dim=2).int()
    mean = torch.sum(vertices * mask.float().unsqueeze(-1), dim=2, keepdim=True) / num_valid.unsqueeze(-1).unsqueeze(-1)
    vn = (vertices - mean).float().contiguous()
    want = ref.sort_vertices.sort_vertices_forward(vn, mask.contiguous(), num_valid.contiguous())
    nv = num_valid[0].cpu().numpy()
    assert int((nv <= 8).sum()) > 0.99 * n and int((nv >= 3).sum()) > 1000
    poly = np.flatnonzero((nv >= 3) & (nv <= 8)), np.flatnonzero(nv < 3)
    rows = np.sort(np.concatenate([poly[0][sample_index(len(poly[0]), 2688, 23)], poly[1][sample_index(len(poly[1]), 384, 24)]]))
    return dict(vertices=vn[0].cpu().numpy()[rows], mask=mask[0].cpu().numpy()[rows], num_valid=nv[rows],
                idx=want[0].cpu().numpy()[rows].astype(np.uint8))


def _smoke_input():
    """The reference's own smoke input (cuda_ext.py:19-31): random vertices, random masks, every polygon kept at <= 8 valid vertices -- with
    more the reference writes PAST its 9 output slots into the next polygon's first slot (:103-106), so only those rows are defined."""
    g2 = torch.Generator().manual_seed(22)
    v = torch.rand(8, 1024, 24, 2, generator=g2).cuda()
    v = (v - v.mean(dim=2, keepdim=True)).contiguous()
    m = torch.rand(8, 1024, 24, generator=g2) > 0.8
    m[m.int().sum(-1) > 8] = False
    m = m.cuda()
    return v, m, m.int().sum(-1).int()


def test_sort_vertices_bit_identical_to_reference_kernel():
    """nrpn_sort_vertices == the reference's own compiled sort_vertices_kernel (cuda_op/sort_vert_kernel.cu:15-140), on polygons of real box
    pairs (the tensors box_intersection_2d.py:121-141 hands to it) and on the random-mask input of the reference's own smoke block."""
    from nerf_rpn_b200 import ops
    polys = recorded("sort_vertices_box_pairs", _reference_polygons)
    got = ops.sort_vertices_forward(torch.from_numpy(polys["vertices"]).cuda()[None], torch.from_numpy(polys["mask"]).cuda()[None],
                                    torch.from_numpy(polys["num_valid"]).cuda()[None])
    assert np.array_equal(got[0].cpu().numpy(), polys["idx"].astype(np.int64))
    v, m, nv = _smoke_input()

    def reference_smoke():
        return dict(idx=ref_gpu.load().sort_vertices.sort_vertices_forward(v, m, nv).cpu().numpy().astype(np.uint8))
    want = torch.from_numpy(recorded("sort_vertices_smoke", reference_smoke)["idx"].astype(np.int64)).cuda()
    got = ops.sort_vertices_forward(v, m, nv)
    rows = (got == want).all(dim=-1)
    bad = (~rows).nonzero()
    print(f"reference smoke input (random masks): {int(rows.sum())} of {rows.numel()} polygons identical")
    for gi in bad[:3].tolist():
        print("  differing polygon", gi, "nv", int(nv[gi[0], gi[1]]), "got", got[gi[0], gi[1]].tolist(), "want", want[gi[0], gi[1]].tolist(),
              "mask", m[gi[0], gi[1]].int().tolist(), "v", v[gi[0], gi[1]].flatten().tolist())
    assert bool(rows.all())


# ------------------------------------------------------------------------------------------------ IoU + NMS (rows a12-a15)
def test_iou_pairs_vs_reference_on_this_gpu():
    """cal_iou_3d of the reference (torch-CUDA chain + K1) vs nrpn_iou3d_pairs (library default NRPN_IOU_MODE 3: CUDA sinf / cosf,
    bmm as fma, ATen's CUDA summation orders -- measured by tools/ref_gpu_probe.py) on 400 000 random OBB pairs, compared on a fixed
    sample of 65 536 of them: bit-identical."""
    from nerf_rpn_b200 import ops
    g = torch.Generator().manual_seed(5)
    n = 400_000
    a, b = rand_obb(n, g, extent=14.0).cuda(), rand_obb(n, g, extent=14.0).cuda()
    idx = torch.from_numpy(sample_index(n, 65536, 5)).cuda()
    want = torch.from_numpy(recorded("iou_pairs", lambda: dict(iou=ref_gpu.load().oriented_iou_loss.cal_iou_3d(a[None], b[None])[0][idx].cpu().numpy()))["iou"]).cuda()
    got = ops.iou3d_pairs(a, b)[idx]
    a, b = a[idx], b[idx]
    nz = want > 0
    eq = (want.view(torch.int32) == got.view(torch.int32))
    print(f"IoU vs reference on {torch.cuda.get_device_name(0)}: {int(nz.sum())} overlapping pairs, bit-equal {eq[nz].float().mean().item():.5f} "
          f"(all pairs {eq.float().mean().item():.5f}), max |diff| {(want - got).abs().max().item():.3e}")
    bad = (~eq).nonzero().reshape(-1)
    for i in bad[:5].tolist():
        print(f"  differs: a={a[i].tolist()} b={b[i].tolist()} reference={want[i].item():.9g} ours={got[i].item():.9g}")
    assert int(nz.sum()) > 4000
    assert (want - got).abs().max().item() <= 2e-6
    assert eq.float().mean().item() >= 0.99999, "NRPN_IOU_MODE 3 should reproduce the torch-CUDA chain bit for bit"


@pytest.mark.parametrize("tag,nb,groups,extent", [("2500x4_levels", 10000, 4, 60.0), ("10000_one_level", 10000, 1, 60.0),
                                                  ("3000_dense", 3000, 1, 25.0)])
def test_nms_keep_sets_identical_to_reference_loop(tag, nb, groups, extent):
    """nrpn_nms keep lists == the reference's Python greedy loop (utils.py:215-265) run on a B200 with its real IoU chain,
    at the sizes the verdict asked for (2 500 boxes x 4 levels; 10 000 boxes in one group)."""
    from nerf_rpn_b200 import ops
    g = torch.Generator().manual_seed(77 + nb + groups)
    boxes = rand_obb(nb, g, extent=extent, smin=2.0, smax=14.0)
    scores = torch.rand(nb, generator=g)
    lv = torch.randint(0, groups, (nb,), generator=g)

    def reference_keep():
        ref = ref_gpu.load()
        keep = ref.utils.nms(boxes, scores, 0.3) if groups == 1 else ref.utils.batched_nms(boxes, scores, lv, 0.3)
        return dict(keep=keep.cpu().numpy().astype(np.int32))
    want = torch.from_numpy(recorded(f"nms_{tag}", reference_keep)["keep"].astype(np.int64))
    torch.cuda.synchronize(); t0 = time.perf_counter()
    keep, nk = ops.nms_device(boxes.cuda(), scores.cuda(), lv.to(torch.int32).cuda() if groups > 1 else None, 0.3)
    got = keep[: int(nk.item())].cpu()
    t_our = time.perf_counter() - t0
    diff = set(want.tolist()) ^ set(got.tolist())
    print(f"NMS {tag}: reference keeps {want.numel()}, ours keeps {got.numel()} in {t_our * 1e3:.2f} ms, symmetric difference {len(diff)}")
    assert got.numel() == want.numel() and not diff, f"keep sets differ in {len(diff)} boxes: {sorted(diff)[:10]}"
    # order: score descending in both; boxes with EQUAL scores (torch.rand draws collide among 10 000 fp32 values) come in whatever
    # order torch.sort leaves them in the reference and lowest-index-first here: compare the sequences modulo ties
    sw, sg = scores[want], scores[got]
    assert torch.equal(sw, sg)
    neq = (want != got).nonzero().reshape(-1)
    for i in neq.tolist():
        assert ((sw == sw[i]).sum() > 1), "order differs outside a tie group"


# ------------------------------------------------------------------------------------------------ network at full size (rows a3, a6)
FEATURE_SAMPLE = 16384                                       # stored reference values per pyramid level


def _scene(dims):
    g = torch.Generator().manual_seed(1000)
    return torch.rand(*dims, 4, generator=g).permute(3, 0, 1, 2).contiguous()


def _sampled(feats, seed):
    """Each pyramid level's shape and a fixed sample of its values (flat index order of the NCDHW tensor)."""
    out = {}
    for i, f in enumerate(feats):
        idx = torch.from_numpy(sample_index(f.numel(), FEATURE_SAMPLE, seed + i)).to(f.device)
        out[f"shape{i}"], out[f"val{i}"] = np.array(f.shape), f.reshape(-1)[idx].float().cpu().numpy()
    return out


def _rel_on_sample(f, want, i, seed):
    assert tuple(f.shape) == tuple(want[f"shape{i}"]), (f.shape, want[f"shape{i}"])
    r = torch.from_numpy(want[f"val{i}"])
    v = f.reshape(-1)[torch.from_numpy(sample_index(f.numel(), FEATURE_SAMPLE, seed + i)).to(f.device)].float().cpu()
    return ((v - r).norm() / r.norm()).item()


def _reference_features(dims):
    """fp32 cuDNN forward of the reference's own ResNet_FPN_256 (TF32 off), seed-0 weights, one U[0,1) scene: a fixed sample of every
    pyramid level, and how far the reference's own TF32-default run lands from it (norm-wise, whole levels)."""
    model = ref_gpu.build_reference_model(rotated=False, seed=0).cuda().eval()
    x = _scene(dims).cuda()
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    feats = {}
    try:
        with torch.no_grad():
            for tf32 in (False, True):
                torch.backends.cudnn.allow_tf32 = tf32; torch.backends.cuda.matmul.allow_tf32 = tf32
                feats[tf32] = [f.float() for f in model.backbone(x[None])]
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    out = _sampled(feats[False], 7)
    out["rel_tf32"] = np.array([((t - r).norm() / r.norm()).item() for t, r in zip(feats[True], feats[False])])
    return out


FEATURE_TOL = {"fp16_w2": 1.0e-3, "fp16": 1.25e-3, "bf16": 1.2e-2}      # north_star: <= 1e-3 -> the fp16_w2 mode (bench default)


@pytest.mark.parametrize("dims", [(160, 256, 256), (200, 200, 130)])
@pytest.mark.parametrize("precision", ["fp16_w2", "fp16", "bf16"])
def test_full_size_feature_maps_vs_reference_fp32_on_this_gpu(dims, precision):
    """BASELINE config 2 (160x256x256) and config 3's grid (200x200x130): every pyramid level of OUR backbone+FPN against the
    reference's own modules in fp32 on a B200 (same seed-0 weights), norm-wise relative error over a fixed sample of 16 384 values per level;
    tolerance = north_star's 1e-3 for the benched mode."""
    from nerf_rpn_b200.model.anchor import AnchorGenerator3D, RPNHead
    from nerf_rpn_b200.model.feature_extractor import Bottleneck, ResNet_FPN_256
    from nerf_rpn_b200.model.nerf_rpn import NeRFRegionProposalNetwork
    want = recorded(f"features_{dims[0]}x{dims[1]}x{dims[2]}", lambda: _reference_features(dims))
    torch.manual_seed(0)                                     # the reference's init order: backbone, anchor generator, head
    backbone = ResNet_FPN_256(Bottleneck, [3, 4, 6, 3], input_dim=4, is_max_pool=True)
    ag = AnchorGenerator3D(ref_gpu.ANCHOR_SIZES, ref_gpu.ASPECT)
    head = RPNHead(256, 13, 4, rotate=False)
    if recording():
        rm = ref_gpu.build_reference_model(rotated=False, seed=0)
        assert all(torch.equal(v, rm.backbone.state_dict()[k]) for k, v in backbone.state_dict().items())
    model = NeRFRegionProposalNetwork(backbone, ag, head, rpn_pre_nms_top_n_test=2500, rpn_post_nms_top_n_test=2500, rpn_nms_thresh=0.3,
                                      precision=precision).cuda().eval()
    with torch.no_grad():
        (feats, props, lv), _, scores = model([_scene(dims).cuda()])
    torch.cuda.synchronize()
    rels = []
    for i, f in enumerate(feats):
        rel = _rel_on_sample(f, want, i, 7)
        rels.append(rel)
        print(f"{dims} [{precision}] P{i + 2} {tuple(f.shape[2:])}: ours vs reference-fp32 {rel:.3e}   (reference TF32-default vs its fp32: "
              f"{want['rel_tf32'][i]:.3e})")
    assert max(rels) <= FEATURE_TOL[precision], rels


SWIN_TOL = {"fp16_w2": 2.5e-3, "fp16": 2.5e-3, "bf16": 2.0e-2}
SWIN_KW = dict(patch_size=[4, 4, 4], embed_dim=96, depths=[2, 2, 18, 2], num_heads=[3, 6, 12, 24], window_size=[4, 4, 4], stochastic_depth_prob=0.0,
               expand_dim=True)


def _reference_swin_features():
    """Pyramid of the reference's own SwinTransformer_FPN in fp32 (TF32 off) on one 200x200x130 scene, seed-0 weights (the FCOS head is
    created right after the backbone, as in run_fcos.py, so that both take the same initial values as in the test): a fixed sample per level."""
    ref = ref_gpu.load()
    torch.manual_seed(0)
    rbb = ref.feature_extractor.SwinTransformer_FPN(**SWIN_KW).cuda().eval()
    ref.fcos.FCOSHead(256, 4, [4, 8, 16, 32], norm_reg_targets=True, centerness_on_reg=True, use_obb=True)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False; torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            rf = rbb(_scene((200, 200, 130)).cuda()[None])
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    return _sampled(rf, 17)


@pytest.mark.parametrize("precision", ["fp16_w2", "bf16"])
def test_config3_swin_s_fcos_full_size_vs_reference_on_this_gpu(precision):
    """BASELINE config 3 at ITS size (Swin-S 3D window attention + FPN + FCOS head, --rotated_bbox, one 200x200x130 grid): pyramid features of
    OUR modules against the reference's own modules in fp32 on a B200 (same seed-0 weights), norm-wise over a fixed sample of each level."""
    import argparse
    from nerf_rpn_b200.model.fcos.fcos import FCOSHead, FCOSOverNeRF
    from nerf_rpn_b200.model.feature_extractor import SwinTransformer_FPN
    want = recorded("swin_s_features_200x200x130", _reference_swin_features)
    fa = argparse.Namespace(num_convs=4, norm_reg_targets=True, centerness_on_reg=True, rotated_bbox=True, pre_nms_thresh=0.0, pre_nms_top_n=2500,
                            nms_thresh=0.3, fpn_post_nms_top_n=2500, min_size=0.0)
    torch.manual_seed(0)
    bb = SwinTransformer_FPN(**SWIN_KW)
    head = FCOSHead(256, 4, [4, 8, 16, 32], norm_reg_targets=True, centerness_on_reg=True, use_obb=True)
    model = FCOSOverNeRF(fa, bb, [4, 8, 16, 32], precision=precision)
    model.fcos_module.head.load_state_dict(head.state_dict())
    model = model.cuda().eval()
    with torch.no_grad():
        boxes, _, scores = model([_scene((200, 200, 130)).cuda()])
        plan = model.engine()._plans[next(iter(model.engine()._plans))]
        feats = [f[..., :256].permute(0, 4, 1, 2, 3).float() for f in plan.features]      # channels-last pyramid buffers of the plan
    torch.cuda.synchronize()
    assert boxes[0].shape[0] > 0 and torch.isfinite(boxes[0]).all()
    rels = []
    for i, f in enumerate(feats):
        rel = _rel_on_sample(f, want, i, 17)
        rels.append(rel)
        print(f"config 3 [{precision}] P{i + 2} {tuple(f.shape[2:])}: ours vs reference-fp32 {rel:.3e}")
    assert max(rels) <= SWIN_TOL[precision], rels


# ------------------------------------------------------------------------------------------------ the unmodified driver (row b)
def _write_scenes(tmp, n_scenes, dims, n_gt=12):
    import pandas as pd
    rows = []
    for i in range(n_scenes):
        g = torch.Generator().manual_seed(3000 + i)
        grid = torch.rand(*dims, 4, generator=g).numpy().astype(np.float32)
        d = torch.tensor(dims, dtype=torch.float32)
        size = torch.rand(n_gt, 3, generator=g) * 20.0 + 6.0
        ctr = torch.rand(n_gt, 3, generator=g) * (d - 8.0) + 4.0
        theta = (torch.rand(n_gt, 1, generator=g) - 0.5) * math.pi
        np.savez(os.path.join(tmp, f"s{i}.npz"), rgbsigma=grid)
        np.save(os.path.join(tmp, f"s{i}.npy"), torch.cat([ctr, size, theta], 1).numpy().astype(np.float32))
        rows.append(dict(scene=f"s{i}", rgbsigma_path=os.path.join(tmp, f"s{i}.npz"), boxes_path=os.path.join(tmp, f"s{i}.npy")))
    pd.DataFrame(rows).to_csv(os.path.join(tmp, "test.csv"))
    return os.path.join(tmp, "test.csv")


def _checkpoint(tmp):
    """Seed-0 reference init with spread objectness, saved in the reference's checkpoint format (run_rpn.py:294-300)."""
    model = ref_gpu.build_reference_model(rotated=True, seed=0, spread=30.0)
    path = os.path.join(tmp, "ckpt.pt")
    torch.save({"epoch": 0, "backbone_state_dict": model.backbone.state_dict(), "rpn_head_state_dict": model.rpn.head.state_dict(),
                "train_args": {}}, path)
    return path


def _run_driver(via, args, tmp, timeout=1500):
    ref_root = ref_gpu.load().root
    script = os.path.join(ref_root, "run_rpn.py")
    env = dict(os.environ, WANDB_MODE="disabled", PYTHONUNBUFFERED="1")
    if via == "b200":
        cmd = [sys.executable, os.path.join(ROOT, "dropin", "run.py"), script] + args
    else:                                                    # the reference itself, untouched, with its own K1 extension
        from oracle.build_ref import CUDA_OP
        env["PYTHONPATH"] = CUDA_OP + os.pathsep + env.get("PYTHONPATH", "")
        cmd = [sys.executable, script] + args
    t0 = time.perf_counter()
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env, cwd=tmp)
    return r, time.perf_counter() - t0


@needs_staged_reference
def test_unmodified_run_rpn_eval_through_dropin_matches_reference_run(tmp_path):
    """`run_rpn.py --mode eval` (the reference's file, byte for byte) over 4 scenes with planted OBBs: once on the reference's own
    modules (cuDNN + Python NMS + K1) and once through dropin/run.py on the B200 engine, same checkpoint.  Both must finish and write
    eval.json; recall@0.25 from the two runs within 0.5 pt... on 48 boxes that is a zero-box difference at top-2500, one box elsewhere."""
    tmp = str(tmp_path)
    csv = _write_scenes(tmp, 4, (64, 96, 80))
    ckpt = _checkpoint(tmp)
    base = ["--mode", "eval", "--dataset_name", "general", "--test_csv", csv, "--backbone_type", "resnet", "--rotated_bbox",
            "--rpn_nms_thresh", "0.3", "--checkpoint", ckpt, "--batch_size", "1", "--output_proposals"]
    out = {}
    for via in ("reference", "b200"):
        save = os.path.join(tmp, via)
        r, dt = _run_driver(via, base + ["--save_path", save], tmp)
        assert r.returncode == 0, f"{via}: {r.stderr[-3000:]}"
        with open(os.path.join(save, "eval.json")) as f:
            out[via] = json.load(f)
        print(f"run_rpn.py --mode eval via {via}: {dt:.1f} s wall; recall@0.25 top-300/1000/2500 = "
              f"{[round(out[via][f'recall_25_top_{k}']['ar'], 4) for k in (300, 1000, 2500)]}  AP@25 {out[via]['ap_25']['ap']:.4f}")
    for k in (300, 1000, 2500):
        a, b = out["reference"][f"recall_25_top_{k}"]["ar"], out["b200"][f"recall_25_top_{k}"]["ar"]
        assert abs(a - b) <= 1.0 / 48 + 1e-6, (k, a, b)
    assert abs(out["reference"]["recall_25_top_2500"]["ar"] - out["b200"]["recall_25_top_2500"]["ar"]) <= 0.005 + 1e-6


@needs_staged_reference
def test_unmodified_run_rpn_benchmark_through_dropin(tmp_path):
    """`run_rpn.py --mode benchmark` (run_rpn.py:594-617: randn(4,200,200,130), 10 warm-up + 300 timed forwards, CUDA events) runs
    unchanged on the B200 engine and prints its own timing line."""
    r, dt = _run_driver("b200", ["--mode", "benchmark", "--dataset_name", "general", "--backbone_type", "resnet"], str(tmp_path))
    assert r.returncode == 0, r.stderr[-3000:]
    line = [l for l in r.stdout.splitlines() if "Average inference time" in l]
    assert line, r.stdout[-2000:]
    print(f"unmodified run_rpn.py --mode benchmark through dropin/: {line[-1]}  ({dt:.1f} s wall)")
