"""CPU suite: the FCOS-R50 oracle is pinned to the reference through committed fixtures (tools/make_golden_fcos.py)."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, 'tests', 'golden')
sys.path.insert(0, os.path.join(ROOT, 'tools'))


@pytest.fixture(scope='module')
def sd():
    from cvpytorch_b200 import synth
    return synth.fcos_state_dict(True)


def test_fcos_state_dict_keys_equal_reference():
    from cvpytorch_b200 import synth
    g = np.load(os.path.join(GOLD, 'fcos_keys.npz'))
    t = synth.fcos_template_state_dict()
    assert list(t.keys()) == list(g['keys']) and [str(tuple(v.shape)) for v in t.values()] == list(g['shapes'])


def test_fcos_oracle_forward_matches_reference(sd):
    from oracle import fcos_oracle as FO
    g = np.load(os.path.join(GOLD, 'fcos_fwd128.npz'))
    torch.manual_seed(1029)
    x = torch.randn(2, 3, 128, 128)
    feats, levels, cls, cnt, reg = FO.forward(x, sd)
    rel = lambda a, b: float((a.double() - torch.from_numpy(b).double()).abs().max() / (np.abs(b).max() + 1e-12))
    assert rel(feats[2][:, ::3], g['C5']) < 1e-5  # the fixture keeps every 3rd C5 channel
    for i in range(5):
        assert rel(levels[i], g[f'P{i + 3}']) < 1e-5 and rel(cls[i], g[f'cls{i}']) < 1e-5
        assert rel(cnt[i], g[f'cnt{i}']) < 1e-5 and rel(reg[i], g[f'reg{i}']) < 1e-5


def test_fcos_oracle_detect_matches_reference():
    """FCOSDetect (top-k, sqrt(cls*ctr), 1-based classes, class-offset '+1'-area NMS) on the reference's own head outputs."""
    from oracle import fcos_oracle as FO
    g = np.load(os.path.join(GOLD, 'fcos_det256.npz'))
    cls = [torch.from_numpy(g[f'cls{i}']) for i in range(5)]
    cnt = [torch.from_numpy(g[f'cnt{i}']) for i in range(5)]
    reg = [torch.from_numpy(g[f'reg{i}']) for i in range(5)]
    dets, _ = FO.fcos_detect(cls, cnt, reg)
    s, c, b, loc = dets[0]
    assert np.array_equal(s, g['scores']) and np.array_equal(c, g['classes']) and np.array_equal(b, g['boxes'])
    assert s.shape[0] > 100 and int(c.min()) >= 1


@pytest.mark.parametrize('name', ['dense', 'sparse'])
def test_fcos_oracle_nms_matches_reference(name):
    from make_golden_fcos import make_fcos_candidates
    from oracle import fcos_oracle as FO
    g = np.load(os.path.join(GOLD, 'fcos_nms_stress.npz'))
    s, c, b = make_fcos_candidates(2, dense=(name == 'dense'))
    for bi in range(2):
        top = np.argsort(-s[bi], kind='stable')[:1000]
        m = s[bi][top] >= np.float32(0.05)
        sm, cm, bm = s[bi][top][m], c[bi][top][m], b[bi][top][m]
        off = cm.astype(np.float32) * (bm.max() + np.float32(1))
        keep = FO.box_nms(bm + off[:, None], sm, 0.6)
        assert np.array_equal(sm[keep], g[f'{name}_{bi}_scores']) and np.array_equal(bm[keep], g[f'{name}_{bi}_boxes'])
        assert np.array_equal(cm[keep], g[f'{name}_{bi}_classes'])


def test_resnet_stem_space_to_depth_equivalence():
    """7x7/s2/p3 conv == 4x4 conv (2 rows/cols of padding before, 1 after) over the 2x2 space-to-depth input."""
    import torch.nn.functional as F
    from cvpytorch_b200.fcos_models import resnet_stem_weights_to_s2d
    g = torch.Generator().manual_seed(4)
    x = torch.randn(1, 3, 16, 24, generator=g, dtype=torch.float64)
    w = torch.randn(5, 3, 7, 7, generator=g, dtype=torch.float64)
    ref = F.conv2d(x, w, None, 2, 3)
    s2d = torch.zeros(1, 16, 8, 12, dtype=torch.float64)
    for dy in range(2):
        for dx in range(2):
            for c in range(3):
                s2d[:, (dy * 2 + dx) * 3 + c] = x[:, c, dy::2, dx::2]
    got = F.conv2d(F.pad(s2d, (2, 1, 2, 1)), resnet_stem_weights_to_s2d(w))
    assert got.shape == ref.shape and float((got - ref).abs().max()) < 1e-12
