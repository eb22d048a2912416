"""CPU: the drop-in shims make the reference's UNMODIFIED driver resolve `model.*` to this package and construct its model
through our module mirror with the reference's own constructor calls (run_rpn.py:171-216, 274-292). They run the reference's own driver
scripts, so they are skipped where the reference is not staged under oracle/_ref (oracle/build_ref.py)."""
import os
import subprocess
import sys
import textwrap

import pytest

from oracle.build_ref import ref_root

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = ref_root() or ""


@pytest.mark.skipif(not os.path.isdir(REF), reason="oracle/_ref not staged")
@pytest.mark.parametrize("backbone", ["resnet", "vgg_EF", "swin_s"])
def test_reference_driver_builds_our_modules(backbone, tmp_path):
    code = textwrap.dedent(f"""
        import sys, types
        sys.path[:0] = [{os.path.join(ROOT, 'dropin')!r}, {ROOT!r}, {REF!r}]
        sys.modules['wandb'] = types.ModuleType('wandb')                 # optional logger, not needed to build the model
        import model                                                     # dropin/model.py -> nerf_rpn_b200.model
        import numpy as np, pandas as pd, torch
        np.savez('{tmp_path}/s.npz', rgbsigma=np.random.rand(32, 32, 32, 4).astype('float32'))
        np.save('{tmp_path}/s.npy', np.array([[2, 2, 2, 9, 9, 9]], dtype='float32'))
        pd.DataFrame(dict(scene=['s'], rgbsigma_path=['{tmp_path}/s.npz'], boxes_path=['{tmp_path}/s.npy'])).to_csv('{tmp_path}/t.csv')
        sys.argv = ['run_rpn.py', '--mode', 'eval', '--dataset_name', 'general', '--test_csv', '{tmp_path}/t.csv',
                    '--backbone_type', '{backbone}', '--resolution', '32', '--rpn_nms_thresh', '0.3']
        import run_rpn                                                   # the reference's unmodified driver
        args = run_rpn.parse_args()
        tr = run_rpn.Trainer(args)
        m = tr.model
        assert type(m).__module__.startswith('nerf_rpn_b200.'), type(m).__module__
        assert type(tr.backbone).__module__.startswith('nerf_rpn_b200.') and type(tr.rpn_head).__module__.startswith('nerf_rpn_b200.')
        assert m.rpn.nms_thresh == 0.3 and m.rpn._pre_nms_top_n['testing'] == 2500 and m.rpn.head is tr.rpn_head
        sd = tr.backbone.state_dict()
        print('OK', type(tr.backbone).__name__, len(sd))
    """)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600,
                       env={**os.environ, "CUDA_VISIBLE_DEVICES": "", "WANDB_MODE": "disabled"})
    assert r.returncode == 0, r.stderr[-3000:]
    assert "OK" in r.stdout


@pytest.mark.skipif(not os.path.isdir(REF), reason="oracle/_ref not staged")
def test_reference_fcos_driver_builds_our_modules(tmp_path):
    code = textwrap.dedent(f"""
        import sys, types
        sys.path[:0] = [{os.path.join(ROOT, 'dropin')!r}, {ROOT!r}, {REF!r}]
        sys.modules['wandb'] = types.ModuleType('wandb')
        import model
        import numpy as np, pandas as pd, torch
        np.savez('{tmp_path}/s.npz', rgbsigma=np.random.rand(32, 32, 32, 4).astype('float32'))
        np.save('{tmp_path}/s.npy', np.array([[2, 2, 2, 9, 9, 9, 0.1]], dtype='float32'))
        pd.DataFrame(dict(scene=['s'], rgbsigma_path=['{tmp_path}/s.npz'], boxes_path=['{tmp_path}/s.npy'])).to_csv('{tmp_path}/t.csv')
        sys.argv = ['run_fcos.py', '--mode', 'eval', '--dataset_name', 'general', '--test_csv', '{tmp_path}/t.csv', '--backbone_type', 'swin_s',
                    '--resolution', '32', '--norm_reg_targets', '--centerness_on_reg', '--rotated_bbox', '--nms_thresh', '0.3']
        import run_fcos                                                  # the reference's unmodified FCOS driver
        args = run_fcos.parse_args()
        tr = run_fcos.Trainer(args)
        m = tr.model
        assert type(m).__module__ == 'nerf_rpn_b200.model.fcos.fcos' and type(m.backbone).__name__ == 'SwinTransformer_FPN'
        assert m.fcos_module.box_selector_test.use_obb and m.fcos_module.head.use_obb
        print('OK', len(m.fcos_module.state_dict()))
    """)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600,
                       env={**os.environ, "CUDA_VISIBLE_DEVICES": "", "WANDB_MODE": "disabled"})
    assert r.returncode == 0, r.stderr[-3000:]
    assert "OK" in r.stdout
