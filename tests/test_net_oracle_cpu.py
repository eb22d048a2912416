"""CPU: oracle/net.py (functional fp32 restatement of ResNet50-FPN + RPN head) against the reference's golden
feature maps / logits / proposals, using weights rebuilt from seeds through OUR module mirror (which also checks
that nerf_rpn_b200.model reproduces the reference's parameter order, init and state_dict keys)."""
import os

import numpy as np
import pytest
import torch

from nerf_rpn_b200.model import anchor, feature_extractor
from oracle import net as onet
from tests import recipes


class NS:
    ResNet_FPN_256 = feature_extractor.ResNet_FPN_256
    Bottleneck = feature_extractor.Bottleneck
    AnchorGenerator3D = anchor.AnchorGenerator3D
    RPNHead = anchor.RPNHead
    VGG_FPN = feature_extractor.VGG_FPN


@pytest.mark.parametrize("name,rot", [("rpn_small_aabb", False), ("rpn_small_obb", True)])
def test_net_oracle_matches_reference(golden_dir, name, rot):
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    backbone, ag, head = recipes.build_small_model(NS, rot, g)
    assert len(backbone.state_dict()) == 332 and len(head.state_dict()) == 12          # SURVEY.md section 5
    x = recipes.golden_input(g)[None]
    feats, (b, s, lv) = onet.full_forward(backbone.state_dict(), head.state_dict(), x, ag.cell_anchors_np(), rot)
    for i, f in enumerate(feats):
        ref = torch.from_numpy(g[f"feat{i}"].astype(np.float32))
        rel = (f[0] - ref).norm() / ref.norm()
        assert rel < 1e-3, f"feature level {i}: rel {rel}"                               # golden stored in fp16
    logits, deltas = onet.head_forward(head.state_dict(), feats)
    for i in range(4):
        np.testing.assert_allclose(logits[i][0].numpy(), g[f"logits{i}"], rtol=1e-3, atol=2e-3)
    assert b.shape == g["proposals"].shape
    if rot:                        # a yaw on the +-pi/2 boundary can come out at either end after last-bit differences: the same box
        b = np.array(b, dtype=np.float64)
        b[:, 6] -= np.pi * np.round((b[:, 6] - g["proposals"][:, 6]) / np.pi)
    np.testing.assert_allclose(b, g["proposals"], rtol=1e-3, atol=1e-2)
    np.testing.assert_array_equal(lv, g["level_index"])


def test_vgg_fpn_oracle_matches_reference(golden_dir):
    """BASELINE config 1 (VGG19-FPN + anchor head on a 32^3 grid): module mirror reproduces the reference's seeded weights
    and state_dict keys (135 backbone tensors); the functional oracle reproduces its features / logits / proposals."""
    from oracle import rpn_post as rp
    g = np.load(os.path.join(golden_dir, "vgg_small_aabb.npz"))
    backbone, ag, head = recipes.build_vgg_small(NS, g)
    sd = backbone.state_dict()
    assert len(sd) == 135 and "fpn_neck.lateral_convs.0.weight" in sd and "layers.3.0.weight" in sd
    x = recipes.golden_input(g)[None]
    feats = onet.vgg_fpn_forward(sd, x)
    for i, f in enumerate(feats):
        st = int(g["fstride"][i])
        ref = torch.from_numpy(g[f"feat{i}"].astype(np.float32))
        got = f[0][:, ::st, ::st, ::st]
        assert ((got - ref).norm() / ref.norm()).item() < 1e-3
    logits, deltas = onet.head_forward(head.state_dict(), feats)
    for i in range(4):
        st = int(g["lstride"][i])
        np.testing.assert_allclose(logits[i][0][:, ::st, ::st, ::st].numpy(), g[f"logits{i}"], rtol=1e-3, atol=2e-3)
    lg, dl = onet.flatten_predictions(logits, deltas, 13, 6)
    grids = [tuple(f.shape[-3:]) for f in feats]
    strides = [tuple(32 // gr[k] for k in range(3)) for gr in grids]
    b, s_, lv = rp.rpn_proposals(lg, dl, grids, strides, ag.cell_anchors_np(), (32, 32, 32), False)
    assert b.shape == g["proposals"].shape
    np.testing.assert_allclose(b, g["proposals"], rtol=1e-3, atol=1e-2)
    np.testing.assert_array_equal(lv, g["level_index"])


def test_swin_fpn_oracle_matches_reference(golden_dir):
    """BASELINE config 3 backbone (Swin-S 3-D shifted-window attention + FPN) on a 40x52x34 grid: the module mirror reproduces
    the reference's 365 seeded tensors, the functional oracle its feature maps."""
    from nerf_rpn_b200.model.fcos import fcos as fcos_mod

    class NSW(NS):
        SwinTransformer_FPN = feature_extractor.SwinTransformer_FPN
        FCOSOverNeRF = fcos_mod.FCOSOverNeRF
    g = np.load(os.path.join(golden_dir, "swin_small_fcos_obb.npz"))
    model = recipes.build_swin_fcos_small(NSW, g)
    sd = model.backbone.state_dict()
    assert len(sd) == 365
    x = recipes.seed1000_input((40, 52, 34))[None]
    feats = onet.swin_fpn_forward(sd, x, recipes.SWIN_S["depths"], recipes.SWIN_S["num_heads"])
    for i, f in enumerate(feats):
        ref = torch.from_numpy(g[f"feat{i}"].astype(np.float32))
        assert ((f[0] - ref).norm() / ref.norm()).item() < 1e-3
