"""YOLOX-s inference path (SURVEY.md 8 row a16) on the B200 through the C ABI: components and fused graph against the reference's
golden outputs / the oracle (fp32 tolerance 1e-3 of max|ref|), post-processing bit-exact on identical candidate records."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
TOL = 1e-3


def _rel(a, b):
    b = torch.as_tensor(b)
    return float((a.double().cpu() - b.double()).abs().max() / (b.double().abs().max() + 1e-12))


@pytest.fixture(scope='module')
def model(cuda):
    from cvpytorch_b200 import synth
    return synth.build_yolox(True)


def test_components_vs_reference_golden_128(model):
    g = np.load(os.path.join(GOLD, 'yolox_fwd128.npz'))
    torch.manual_seed(1029)
    x = torch.randn(2, 3, 128, 128).cuda()
    b = model.backbone(x)
    for i, t in enumerate(b):
        assert _rel(t, g[f'backbone{i}']) < TOL, ('backbone', i)
    b_ref = [torch.from_numpy(g[f'backbone{i}']) for i in range(3)]
    n = model.neck([t.cuda() for t in b_ref])
    for i, t in enumerate(n):  # the fixture keeps every 3rd neck / head channel
        assert _rel(t[:, ::3], g[f'neck{i}']) < TOL, ('neck', i)
    from cvpytorch_b200 import synth
    from oracle import yolox_oracle as XO
    with torch.no_grad():
        n_ref = XO.neck(b_ref, synth.yolox_state_dict(True))  # the head's input: the oracle's neck on the reference's backbone tensors
    o = model.head([t.cuda() for t in n_ref])
    for i, t in enumerate(o):
        assert tuple(t[:, ::3].shape) == g[f'head{i}'].shape
        assert _rel(t[:, ::3], g[f'head{i}']) < TOL, ('head', i)


def test_nms_bit_exact_on_stress_records(cuda):
    """cvb_yolox_nms on foreign candidate records == the oracle (pinned to the reference + torchvision.ops.batched_nms), both regimes."""
    from cvpytorch_b200 import ops
    from oracle import yolox_oracle as XO
    recs = [XO.make_stress_records(regime=r, seed=s) for r in ('few', 'typical', 'all') for s in (2, 3)]
    A = recs[0].shape[0]
    ws = ops.YoloxWorkspace(len(recs), A)
    det, cnt = ops.yolox_nms(ws, 0.01, 0.65, cand=torch.from_numpy(np.stack(recs)).cuda())
    torch.cuda.synchronize()
    det, cnt = det.cpu().numpy(), cnt.cpu().numpy()
    for b, rec in enumerate(recs):
        rows, _ = XO.nms_records(rec, 0.01, 0.65)
        assert cnt[b] == rows.shape[0], (b, cnt[b], rows.shape[0])
        assert np.array_equal(det[b, :cnt[b]], rows), b
    # empty image and a single candidate
    ws1 = ops.YoloxWorkspace(2, 64)
    c = torch.zeros((2, 64, 8))
    c[1, 5] = torch.tensor([10., 10., 50., 60., 0.9, 0.8, 3., 0.9 * 0.8])
    det, cnt = ops.yolox_nms(ws1, 0.01, 0.65, cand=c.cuda())
    torch.cuda.synchronize()
    assert cnt.tolist() == [0, 1] and torch.equal(det[1, 0].cpu(), c[1, 5, :7])


def test_fused_320_vs_oracle_with_post_process(model):
    from cvpytorch_b200 import synth
    from oracle import yolox_oracle as XO
    sd = synth.yolox_state_dict(True)
    torch.manual_seed(1029)
    x = torch.randn(1, 3, 320, 320)
    det, cnt = model.predict(x.cuda())
    torch.cuda.synchronize()
    G = model._graph_for(x.cuda())
    rec_gpu = G['ws'].cand.cpu().numpy()
    rec_or = XO.records(XO.decode(XO.forward(x, sd)))
    g = np.load(os.path.join(GOLD, 'yolox_post320.npz'))
    # decoded records vs oracle / reference fixture (class_pred compared where the top-2 class gap is not a rounding tie)
    for col in (0, 1, 2, 3, 4, 5, 7):
        e = np.abs(rec_gpu[0, :, col] - rec_or[0, :, col]).max() / (np.abs(rec_or[0, :, col]).max() + 1e-12)
        assert e < TOL, (col, e)
    assert float((rec_gpu[0, :, 6] == rec_or[0, :, 6]).mean()) > 0.99
    e_gold = np.abs(rec_gpu[0, :, :5] - g['records'][:, :5]).max() / np.abs(g['records'][:, :5]).max()
    assert e_gold < TOL
    # post-process bit-exact on the GPU's own records
    rows, _ = XO.nms_records(rec_gpu[0], model.conf_thr, model.nms_thr)
    k = int(cnt[0])
    assert k == rows.shape[0] and np.array_equal(det[0, :k].cpu().numpy(), rows)
    # and agreement of the two end-to-end pipelines for the bulk of the detections
    ref_rows = g['det']
    common = len(set(map(tuple, np.round(rows[:, :4], 1).tolist())) & set(map(tuple, np.round(ref_rows[:, :4], 1).tolist())))
    print('kept', k, 'reference kept', ref_rows.shape[0], 'boxes in common (0.1 px):', common)
    assert common >= 0.9 * ref_rows.shape[0]


def test_forward_val_contract_and_batch_independence(model):
    torch.manual_seed(1)
    x = torch.randn(3, 3, 160, 160).cuda()
    targets = [{'labels': torch.zeros(1), 'boxes': torch.zeros(1, 4), 'scales': torch.tensor([1.0, 1.0]), 'pads': torch.tensor([0.0, 0.0]),
                'height': torch.tensor(160), 'width': torch.tensor(160)} for _ in range(3)]
    out = model(x, targets, 'val')
    assert isinstance(out, tuple) and isinstance(out[0], dict) and len(out[1]) == 3
    for o in out[1]:
        assert set(o.keys()) == {'boxes', 'labels', 'scores'} and o['boxes'].shape[1] == 4
        assert float(o['boxes'].min()) >= 0.0 and float(o['boxes'].max()) <= 160.0
    assert model(x, None, 'infer') is None
    det, cnt = [t.clone() for t in model.predict(x)]
    d1, c1 = model.predict(x[1:2].contiguous())
    torch.cuda.synchronize()
    assert int(c1[0]) == int(cnt[1]) and torch.equal(d1[0, :int(c1[0])], det[1, :int(cnt[1])])
