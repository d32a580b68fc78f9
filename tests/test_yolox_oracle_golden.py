"""CPU suite: the YOLOX oracle (oracle/yolox_oracle.py) against fixtures produced by the REFERENCE itself
(tools/make_golden_yolox.py), and the drop-in's state_dict surface."""
import os

import numpy as np
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def test_yolox_state_dict_keys_equal_reference():
    from cvpytorch_b200 import synth
    g = np.load(os.path.join(GOLD, 'yolox_keys.npz'))
    t = synth.yolox_template_state_dict()
    assert list(t.keys()) == list(g['keys'])
    assert [str(tuple(v.shape)) for v in t.values()] == list(g['shapes'])
    n = sum(v.numel() for k, v in t.items() if not k.endswith(('num_batches_tracked', 'running_mean', 'running_var')))
    assert n == 4212672 + 2834688 + 1920895  # 8.97 M parameters (SURVEY.md 3.5 row 3)


def test_yolox_forward_matches_reference_fixture():
    from cvpytorch_b200 import synth
    from oracle import yolox_oracle as XO
    g = np.load(os.path.join(GOLD, 'yolox_fwd128.npz'))
    sd = synth.yolox_state_dict(True)
    torch.manual_seed(1029)
    x = torch.randn(2, 3, 128, 128)
    with torch.no_grad():
        b = XO.backbone(x, sd)
        n = XO.neck(b, sd)
        o = XO.head(n, sd)
    for name, ts in (('backbone', b), ('neck', n), ('head', o)):
        for i, t in enumerate(ts):
            ref = g[f'{name}{i}']
            t = t if name == 'backbone' else t[:, ::3]  # the fixture keeps every 3rd neck / head channel
            assert t.shape == ref.shape
            err = float(np.abs(t.numpy() - ref).max() / (np.abs(ref).max() + 1e-12))
            assert err <= 2e-5, (name, i, err)  # bit-identical in the build container; other CPUs/BLAS differ in the last bits
    assert o[0].shape[-2:] == (18, 18)  # 1x1 stems with padding=1: 16 + 2


def test_yolox_post_process_matches_reference_fixture():
    from oracle import yolox_oracle as XO
    g = np.load(os.path.join(GOLD, 'yolox_post320.npz'))
    outs = [torch.from_numpy(g[f'head{i}']) for i in range(3)]
    rec = XO.records(XO.decode(outs))
    assert np.array_equal(rec[0], g['records'])
    rows, loc = XO.nms_records(rec[0])
    assert np.array_equal(XO.canonical_rows(rows), XO.canonical_rows(g['det'])) and np.array_equal(loc, g['loc'])


def test_yolox_nms_stress_matches_reference_fixture():
    """score filter + torchvision.ops.batched_nms, both regimes (<= 1000 boxes: coordinate trick, more: per-class NMS)."""
    from oracle import yolox_oracle as XO
    g = np.load(os.path.join(GOLD, 'yolox_nms.npz'))
    seen = set()
    for regime in ('few', 'typical', 'all'):
        for seed in (2, 3):
            rec = XO.make_stress_records(regime=regime, seed=seed)
            seen.add(int((rec[:, 7] >= 0.01).sum()) > 1000)
            rows, loc = XO.nms_records(rec)
            assert np.array_equal(XO.canonical_rows(rows), XO.canonical_rows(g[f'{regime}_{seed}_det'])), (regime, seed)
            assert np.array_equal(loc, g[f'{regime}_{seed}_loc'])
    assert seen == {True, False}
