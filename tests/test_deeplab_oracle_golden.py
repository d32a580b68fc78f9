"""CPU suite: the DeepLabv3+ oracle is pinned to the reference through committed fixtures (tools/make_golden_deeplab.py)."""
import os

import numpy as np
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def test_deeplab_keys_equal_reference():
    from cvpytorch_b200 import synth
    g = np.load(os.path.join(GOLD, 'deeplab_keys.npz'))
    t = synth.deeplab_template_state_dict()
    assert list(t.keys()) == list(g['keys']) and [str(tuple(v.shape)) for v in t.values()] == list(g['shapes'])


def test_deeplab_oracle_matches_reference():
    from cvpytorch_b200 import synth
    from oracle import deeplab_oracle as DO
    g = np.load(os.path.join(GOLD, 'deeplab_fwd.npz'))
    torch.manual_seed(1029)
    x = torch.randn(2, 3, 128, 256)
    feats, logits, labels = DO.forward(x, synth.deeplab_state_dict(True))
    rel = lambda a, b: float((a.double() - torch.from_numpy(b).double()).abs().max() / (np.abs(b).max() + 1e-12))
    assert rel(feats[0][:, ::8], g['low_sub']) < 1e-5 and rel(feats[1][:, ::3], g['high']) < 1e-5 and rel(logits, g['logits']) < 1e-5
    assert float((labels.numpy() == g['labels']).mean()) > 0.9999  # exact unless a 1e-6 logit tie flips across CPUs


def test_deep_stem_space_to_depth_equivalence():
    import torch.nn.functional as F
    from cvpytorch_b200.fcos_models import deep_stem_weights_to_s2d
    g = torch.Generator().manual_seed(4)
    x = torch.randn(1, 3, 16, 24, generator=g, dtype=torch.float64)
    w = torch.randn(5, 3, 3, 3, generator=g, dtype=torch.float64)
    ref = F.conv2d(x, w, None, 2, 1)
    s2d = torch.zeros(1, 16, 8, 12, dtype=torch.float64)
    for dy in range(2):
        for dx in range(2):
            for c in range(3):
                s2d[:, (dy * 2 + dx) * 3 + c] = x[:, c, dy::2, dx::2]
    got = F.conv2d(F.pad(s2d, (1, 0, 1, 0)), deep_stem_weights_to_s2d(w))
    assert got.shape == ref.shape and float((got - ref).abs().max()) < 1e-12
