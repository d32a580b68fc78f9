"""Parity of the drop-in YOLOv5-s path (fused B200 graph through the C ABI) against
  (1) the committed golden fixtures produced by the REFERENCE on CPU and (2) the oracle run on this host.
Tolerance (north_star): fp32 logits / decoded outputs within 1e-3 relative (max|a-b|/max|b|); NMS kept indices
bit-exact on identical candidate tensors."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, 'tests', 'golden')
sys.path.insert(0, os.path.join(ROOT, 'tools'))
TOL = 1e-3


@pytest.fixture(scope='module')
def model(cuda):
    from cvpytorch_b200 import synth
    return synth.build_yolov5s(calibrated=True)


@pytest.fixture(scope='module')
def sd():
    from cvpytorch_b200 import synth
    return synth.yolov5s_state_dict(True)


def _rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).abs().max() / (b.abs().max() + 1e-12))


def test_components_vs_reference_golden_128(model):
    """backbone / neck / detect called one by one with the reference's NCHW fp32 tensors (component-level drop-in)."""
    g = np.load(os.path.join(GOLD, 'yolov5s_fwd128.npz'))
    torch.manual_seed(1029)
    x = torch.randn(2, 3, 128, 128).cuda()
    feats = model.backbone(x)
    errs = {}
    for i in range(3):  # the fixture keeps every 3rd channel / anchor row
        assert tuple(feats[i][:, ::3].shape) == g[f'backbone{i}'].shape
        errs[f'backbone{i}'] = _rel(feats[i][:, ::3], g[f'backbone{i}'])
    nfe = model.neck(feats)
    for i in range(3):
        errs[f'neck{i}'] = _rel(nfe[i][:, ::3], g[f'neck{i}'])
    lst = list(nfe)
    z, raws = model.detect(lst)
    errs['z'] = _rel(z[:, ::3], g['z'])
    assert lst[0] is raws[0] and tuple(raws[0].shape) == (2, 3, 16, 16, 85)  # list mutated in place like the reference
    print(errs)
    assert max(errs.values()) < TOL, errs


def test_fused_graph_vs_reference_golden_128(model):
    g = np.load(os.path.join(GOLD, 'yolov5s_fwd128.npz'))
    torch.manual_seed(1029)
    x = torch.randn(2, 3, 128, 128).cuda()
    model.predict(x)
    z = model._graph_for(x)['z']
    err = _rel(z[:, ::3], g['z'])
    print('fused z rel err vs reference golden', err)
    assert err < TOL


def test_fused_640_vs_golden_and_oracle_with_nms(model, sd):
    from oracle import nms_oracle as NO
    from oracle import yolov5_oracle as YO
    g = np.load(os.path.join(GOLD, 'yolov5s_fwd640.npz'))
    torch.manual_seed(1029)
    x = torch.randn(1, 3, 640, 640)
    det, idx, cnt = model.predict(x.cuda())
    torch.cuda.synchronize()
    z = model._graph_for(x.cuda())['z'].cpu()
    e_gold = _rel(z[0, ::16], g['z_sub'])
    zo, raws_o = YO.forward(x, sd)
    e_or = _rel(z, zo)
    print('z rel err vs golden', e_gold, 'vs oracle', e_or)
    assert e_gold < TOL and e_or < TOL
    # bit-exact NMS on identical candidates: the GPU's own z through the oracle NMS
    rd, ri = NO.non_max_suppression(z.numpy(), 0.001, 0.6, multi_label=True)[0]
    k = int(cnt[0])
    assert k == rd.shape[0] == 300
    assert np.array_equal(idx[0, :k].cpu().numpy().astype(np.int64), ri)
    assert np.array_equal(det[0, :k].cpu().numpy(), rd)
    # ... and the CUDA NMS over the ORACLE's z reproduces the oracle's result for it
    from cvpytorch_b200 import models as M
    dets, idxs = M.non_max_suppression(zo.cuda(), 0.001, 0.6, multi_label=True, return_indices=True)
    od, oi = NO.non_max_suppression(zo.numpy(), 0.001, 0.6, multi_label=True)[0]
    assert np.array_equal(dets[0].cpu().numpy(), od) and np.array_equal(idxs[0].cpu().numpy().astype(np.int64), oi)
    if np.array_equal(zo[0, ::16].numpy(), g['z_sub']):  # same CPU arithmetic as the build container -> compare to the reference's own NMS rows
        assert np.array_equal(od, g['nms_det'])
    # box-level agreement of the two end-to-end pipelines (fp32 CPU vs B200): same kept candidates for the bulk
    common = len(set(ri.tolist()) & set(oi.tolist()))
    print('kept candidates in common with the oracle pipeline:', common, '/ 300')
    assert common >= 270


def test_ragged_input_shape_and_batch(model, sd):
    from oracle import yolov5_oracle as YO
    torch.manual_seed(5)
    x = torch.randn(3, 3, 96, 160)
    model.predict(x.cuda())
    z = model._graph_for(x.cuda())['z'].cpu()
    zo, _ = YO.forward(x, sd)
    assert z.shape == zo.shape
    assert _rel(z, zo) < TOL


def test_forward_val_contract(model):
    torch.manual_seed(1)
    x = torch.randn(2, 3, 128, 128).cuda()
    targets = [{'labels': torch.zeros(1), 'boxes': torch.zeros(1, 4), 'scales': torch.tensor([1.0, 1.0]),
                'pads': torch.tensor([0.0, 0.0]), 'height': torch.tensor(128), 'width': torch.tensor(128)} for _ in range(2)]
    out = model(x, targets, 'val')
    assert isinstance(out, tuple) and isinstance(out[0], dict)  # trainer.py:210-213 disambiguates with isinstance(out, tuple)
    losses, outputs = out
    assert len(outputs) == 2
    for o in outputs:
        assert set(o.keys()) == {'boxes', 'labels', 'scores'}
        assert o['boxes'].shape[1] == 4 and o['boxes'].device.type == 'cpu'
        assert float(o['boxes'].min()) >= 0.0 and float(o['boxes'].max()) <= 128.0
        assert o['boxes'].shape[0] == o['labels'].shape[0] == o['scores'].shape[0] <= 300
    # non-identity letterbox geometry: the device-side rescale/clip must equal the reference's numpy lines (yolov5.py:274-281)
    targets2 = [{'labels': torch.zeros(1), 'boxes': torch.zeros(1, 4), 'scales': torch.tensor([0.4, 0.5]), 'pads': torch.tensor([3.0, 7.0]),
                 'height': torch.tensor(300), 'width': torch.tensor(240)} for _ in range(2)]
    _, outs2 = model(x, targets2, 'val')
    det, _, cnt = model.predict(x)
    for b, o in enumerate(outs2):
        bb = det[b, :int(cnt[b]), :4].cpu().numpy().copy()
        bb[:, [0, 2]] -= np.float32(7.0)
        bb[:, [1, 3]] -= np.float32(3.0)
        bb[:, [0, 2]] /= np.float32(0.5)
        bb[:, [1, 3]] /= np.float32(0.4)
        bb[:, [0, 2]] = bb[:, [0, 2]].clip(0, 240)
        bb[:, [1, 3]] = bb[:, [1, 3]].clip(0, 300)
        assert np.array_equal(o['boxes'].numpy(), bb)


def test_cuda_graph_replay_matches_eager(model):
    torch.manual_seed(2)
    x = torch.randn(2, 3, 128, 128).cuda()
    G = model.build_graph(2, 128, 128, x.device)
    G['holder']['x'] = x
    G['g'].run()
    torch.cuda.synchronize()
    z_eager = G['z'].clone()
    d_eager = G['ws'].det.clone()
    G['g'].capture()
    G['z'].zero_()
    G['g'].replay()
    torch.cuda.synchronize()
    assert torch.equal(G['z'], z_eager) and torch.equal(G['ws'].det, d_eager)


def test_inference_pipeline_matches_predict(model):
    from cvpytorch_b200.runtime import InferencePipeline
    torch.manual_seed(3)
    xs = [torch.randn(2, 3, 128, 128).pin_memory() for _ in range(5)]
    pipe = InferencePipeline(model, 2, 128, 128, torch.device('cuda:0'))
    outs = []
    for i, xh in enumerate(xs):
        s = pipe.submit(xh)
        d, ix, c = pipe.result(s)
        outs.append((d.clone(), ix.clone(), c.clone()))
    for xh, (d, ix, c) in zip(xs, outs):
        dd, ii, cc = model.predict(xh.cuda())
        torch.cuda.synchronize()
        assert torch.equal(cc.cpu(), c) and torch.equal(dd.cpu(), d) and torch.equal(ii.cpu(), ix)


def test_uint8_frames_stem_bit_identical_and_model_equal(cuda):
    """SURVEY.md 8(f) rank 1: uint8 HWC frames with ToTensor + Normalize fused into the stem loader.  The space-to-depth tensor must
    be bit-identical to the fp32 path fed with the reference's transformed tensor (golden fixture from the reference's own
    classes), and model-level detections must be identical."""
    import os
    import numpy as np
    from cvpytorch_b200 import ops, synth
    from oracle import yolov5_oracle as YO
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'input_transform.npz'))
    frames = torch.from_numpy(g['frames']).cuda()
    ref = torch.from_numpy(g['tensor']).cuda()
    norm = dict(mean=g['mean'].tolist(), std=g['std'].tolist(), reverse_channels=True)
    B, H, W = frames.shape[0], frames.shape[1], frames.shape[2]
    for padded in (False, True):
        Wd = W // 2 + (3 if padded else 0)
        a, b = ops.SplitTensor(B, H // 2, Wd, 16), ops.SplitTensor(B, H // 2, Wd, 16)
        ops.stem_s2d(ref, a.view())
        ops.stem_s2d(frames, b.view(), norm=norm)
        torch.cuda.synchronize()
        assert torch.equal(a.data, b.data)
    # W % 4 != 0 takes the one-pixel-per-thread kernel; reference tensor from the (fixture-pinned) oracle restatement
    fr46 = g['frames'][:, :, :46].copy()
    x46 = YO.input_transform(fr46, norm['mean'], norm['std'], True).cuda()
    a, b = ops.SplitTensor(B, H // 2, 23, 16), ops.SplitTensor(B, H // 2, 23, 16)
    ops.stem_s2d(x46, a.view())
    ops.stem_s2d(torch.from_numpy(fr46).cuda(), b.view(), norm=norm)
    torch.cuda.synchronize()
    assert torch.equal(a.data, b.data)
    # model level: random frames at 128x128
    m = synth.build_yolov5s(True)
    rng = np.random.default_rng(5)
    fr = torch.from_numpy(rng.integers(0, 256, size=(2, 128, 128, 3), dtype=np.uint8))
    x = YO.input_transform(fr, m.input_norm['mean'], m.input_norm['std'], True)
    d0, i0, c0 = [t.clone() for t in m.predict(x.cuda())]
    d1, i1, c1 = m.predict_frames(fr.cuda())
    torch.cuda.synchronize()
    assert torch.equal(c0, c1) and torch.equal(i0, i1) and torch.equal(d0, d1)


def test_full_size_bs64_properties(model):
    """BASELINE.json configs[1] at full size (64 x 3 x 640 x 640), through properties that need no oracle run:
    (1) determinism: two passes are bit-identical; (2) images are independent: image i of the batch equals the same image run
    alone (different tile boxes, same arithmetic); (3) NMS invariants on every image: scores non-increasing, counts <= 300,
    kept boxes of one class have IoU <= thr (torchvision's float IoU compared in double), kept ids unique and consistent
    with the decoded tensor; (4) batch permutation permutes the outputs."""
    torch.manual_seed(1029)
    x = torch.randn(64, 3, 640, 640).cuda()
    det, idx, cnt = [t.clone() for t in model.predict(x)]
    z = model._graph_for(x)['z']
    det2, idx2, cnt2 = model.predict(x)
    torch.cuda.synchronize()
    assert torch.equal(det, det2) and torch.equal(idx, idx2) and torch.equal(cnt, cnt2)
    # (3) invariants, checked on the host for all 64 images
    d, ix, c = det.cpu().double(), idx.cpu().long(), cnt.cpu().long()
    zc = z.cpu()
    nc = zc.shape[2] - 5
    for b in range(64):
        k = int(c[b])
        assert 0 < k <= 300
        s = d[b, :k, 4]
        assert bool((s[:-1] >= s[1:]).all())
        ids = ix[b, :k]
        assert ids.unique().numel() == k
        anchor, cls = ids // nc, ids % nc
        assert torch.equal(cls.double(), d[b, :k, 5])
        # score and box recomputed from the decoded tensor exactly as yolov5.py:106,52-59 does
        row = zc[b, anchor]
        assert torch.equal((row[:, 5:].gather(1, cls[:, None])[:, 0] * row[:, 4]).double(), s)
        box = torch.stack([row[:, 0] - row[:, 2] / 2, row[:, 1] - row[:, 3] / 2, row[:, 0] + row[:, 2] / 2, row[:, 1] + row[:, 3] / 2], 1)
        assert torch.equal(box.double(), d[b, :k, :4])
        if b % 16 == 0:  # pairwise IoU of same-class kept boxes (float32 arithmetic like torchvision, compared in double)
            bo = box + (cls.float() * 4096.0)[:, None]
            area = (bo[:, 2] - bo[:, 0]) * (bo[:, 3] - bo[:, 1])
            lt = torch.max(bo[:, None, :2], bo[None, :, :2])
            rb = torch.min(bo[:, None, 2:], bo[None, :, 2:])
            wh = (rb - lt).clamp(min=0)
            inter = wh[..., 0] * wh[..., 1]
            iou = inter / (area[:, None] + area[None, :] - inter)
            iou = torch.nan_to_num(iou, nan=0.0)  # 0/0 for degenerate boxes: NaN > thr is false in torchvision, nothing is suppressed
            iou.fill_diagonal_(0)
            assert float(iou.double().max()) <= 0.6
    # (2) independence + (4) permutation
    for b in (0, 37, 63):
        d1, i1, c1 = model.predict(x[b:b + 1].contiguous())
        torch.cuda.synchronize()
        assert int(c1[0]) == int(cnt[b]) and torch.equal(i1[0], idx[b]) and torch.equal(d1[0], det[b])
    perm = torch.randperm(64, generator=torch.Generator().manual_seed(1))
    dp, ip, cp = model.predict(x[perm.cuda()].contiguous())
    torch.cuda.synchronize()
    assert torch.equal(cp.cpu(), cnt.cpu()[perm]) and torch.equal(ip.cpu(), idx.cpu()[perm]) and torch.equal(dp.cpu(), det.cpu()[perm])


def test_headline_batch_vs_reference_rows_and_end_to_end_agreement(model, sd):
    """The 8 reference-golden images of the headline batch (tests/golden/yolov5s_batch640.npz, incl. the exact-score-tie images 3 and 5):
    (a) the CUDA NMS over the reference's candidates (the oracle's z when this host reproduces the build container's arithmetic, which
        the fixture's z_sub decides) keeps the reference's SET, in the reference's ORDER up to exact-score ties, with bit-identical rows;
    (b) end to end (B200 conv stack + decode + NMS vs the reference pipeline) the kept candidate ids are compared and the agreement is
        RECORDED (printed, and asserted against the level measured in round 2) instead of a loose bound;
    (c) the same 8 images inside the full bs64 batch give the same rows as the 8-image batch (two in-batch images vs the oracle)."""
    from cvpytorch_b200 import models as M
    from oracle import nms_oracle as NO
    from oracle import yolov5_oracle as YO
    g = np.load(os.path.join(GOLD, 'yolov5s_batch640.npz'))
    torch.manual_seed(1029)
    x64 = torch.randn(64, 3, 640, 640)
    x = x64[:8].contiguous()
    zo, _ = YO.forward(x, sd)
    assert YO.rel_err(zo[:, ::128], torch.from_numpy(g['z_sub'])) < 1e-5
    ref_arith = np.array_equal(zo[:, ::128].numpy(), g['z_sub'])
    dets, idxs = M.non_max_suppression(zo.cuda(), 0.001, 0.6, multi_label=True, return_indices=True)
    ores = NO.non_max_suppression(zo.numpy(), 0.001, 0.6, multi_label=True)
    for i in range(8):
        ci = idxs[i].cpu().numpy().astype(np.int64)
        assert np.array_equal(ci, ores[i][1]) and np.array_equal(dets[i].cpu().numpy(), ores[i][0]), i   # bit-exact vs the oracle
        if ref_arith:
            rd, ri = g[f'det_{i}'], g[f'idx_{i}']
            assert set(ci.tolist()) == set(ri.tolist()), i
            assert NO.same_up_to_score_ties(rd[:, 4], ri, ci), i
            assert np.array_equal(rd[np.argsort(ri, kind='stable')], dets[i].cpu().numpy()[np.argsort(ci, kind='stable')]), i
    # (b) end to end
    det, idx, cnt = [t.clone() for t in model.predict(x.cuda())]
    torch.cuda.synchronize()
    z = model._graph_for(x.cuda())['z'].cpu()
    print('end-to-end decoded z rel err vs oracle:', _rel(z, zo))
    assert _rel(z, zo) < TOL
    common = []
    for i in range(8):
        k = int(cnt[i])
        mine = set(idx[i, :k].cpu().numpy().astype(np.int64).tolist())
        common.append(len(mine & set(g[f'idx_{i}'].tolist())))
    print('end-to-end kept candidate ids in common with the REFERENCE pipeline, per image (of 300):', common)
    assert min(common) >= 240 and sum(common) >= 8 * 270, common
    # (c) two of these images inside the BASELINE-shaped bs64 batch equal the same image in the 8-image batch, and the oracle NMS over
    #     the batch's own z reproduces the rows (bit-exact on identical candidates)
    d64, i64, c64 = model.predict(x64.cuda())
    torch.cuda.synchronize()
    z64 = model._graph_for(x64.cuda())['z']
    for b in (3, 5):
        assert int(c64[b]) == int(cnt[b]) and torch.equal(i64[b], idx[b]) and torch.equal(d64[b], det[b])
        od, oi = NO.non_max_suppression(z64[b:b + 1].cpu().numpy(), 0.001, 0.6, multi_label=True)[0]
        k = int(c64[b])
        assert np.array_equal(i64[b, :k].cpu().numpy().astype(np.int64), oi) and np.array_equal(d64[b, :k].cpu().numpy(), od)


def test_brick_level_convmodule_standalone(cuda):
    """ConvModule / Conv called on their own (brick-level drop-in, SURVEY.md 8b): NCHW fp32 in / out == conv -> BN(eval) -> act of torch."""
    from cvpytorch_b200.bricks import B200ConvModule
    from cvpytorch_b200.modules import Conv
    torch.manual_seed(3)
    for (cin, cout, k, s, p, act) in [(32, 64, 3, 1, 1, 'SiLU'), (3, 16, 3, 2, 1, 'ReLU'), (64, 40, 1, 1, 0, None)]:
        m = B200ConvModule(cin, cout, k, stride=s, padding=p, conv_cfg=dict(type='B200Conv2d'), norm_cfg=dict(type='BN', eps=1e-3),
                           act_cfg=dict(type=act) if act else None).cuda().eval()
        with torch.no_grad():
            m.bn.running_mean.normal_(0, 0.3)
            m.bn.running_var.uniform_(0.5, 1.5)
            m.bn.weight.uniform_(0.5, 1.5)
            m.bn.bias.normal_(0, 0.2)
        x = torch.randn(2, cin, 24, 40, device='cuda')
        y = m(x)
        ref = torch.nn.functional.batch_norm(torch.nn.functional.conv2d(x, m.conv.weight, None, s, p), m.bn.running_mean, m.bn.running_var,
                                             m.bn.weight, m.bn.bias, False, 0.0, m.bn.eps)
        ref = torch.nn.functional.silu(ref) if act == 'SiLU' else (torch.relu(ref) if act == 'ReLU' else ref)
        assert _rel(y, ref) < 2e-5, (cin, cout, k)
        assert _rel(m(x), ref) < 2e-5  # cached plan
    c = Conv(32, 32, 3, 1).cuda().eval()
    x = torch.randn(1, 32, 16, 16, device='cuda')
    ref = torch.nn.functional.silu(torch.nn.functional.batch_norm(torch.nn.functional.conv2d(x, c.conv.weight, None, 1, 1), c.bn.running_mean,
                                                                  c.bn.running_var, c.bn.weight, c.bn.bias, False, 0.0, c.bn.eps))
    assert _rel(c(x), ref) < 2e-5


def test_drop_in_through_the_reference_trainer_val_step(model):
    """The val branch of the reference's Trainer.run_step (trainer.py:209-231) restated around the drop-in model, including the
    `cfg.distributed` path: reduce_dict(losses) stacks the loss values (src/utils/distributed.py:108-125) and must not see an empty dict."""
    class Logger:
        def __init__(self):
            self.seen = {}

        def update(self, *a, **k):
            self.seen.update(k)
            self.args = a

    def reduce_dict_distributed(d):  # the world_size >= 2 branch of src/utils/distributed.py:112-125 (mean over the stacked values)
        names = sorted(d.keys())
        values = torch.stack([d[k] for k in names], dim=0)
        return {k: torch.mean(v) for k, v in zip(names, values)}

    torch.manual_seed(4)
    imgs = torch.randn(2, 3, 128, 128).cuda()
    targets = [{'labels': torch.zeros(1), 'boxes': torch.zeros(1, 4), 'scales': torch.tensor([1.0, 1.0]), 'pads': torch.tensor([0.0, 0.0]),
                'height': torch.tensor(128), 'width': torch.tensor(128)} for _ in range(2)]
    for distributed in (False, True):
        loss_logger, perf_logger = Logger(), Logger()
        out = model(imgs, targets, 'val')                      # trainer.py:209
        if not isinstance(out, tuple):                         # :210-213
            losses, predicts = None, out
        else:
            losses, predicts = out
        if losses is not None:                                 # :215-222
            loss_logger.update(**(reduce_dict_distributed(losses) if distributed else losses))
        if predicts is not None:                               # :224-231 (the reference's reduce_dict of a LIST of dicts is its own bug)
            perf_logger.update(targets, predicts)
        assert 'loss' in loss_logger.seen and float(loss_logger.seen['loss']) == 0.0
        assert len(perf_logger.args[1]) == 2 and set(perf_logger.args[1][0].keys()) == {'boxes', 'labels', 'scores'}


def test_yolov6_yolov7_blocks_vs_reference_golden(cuda):
    """RepVGGBlock (training form and re-parameterised), BepC3 (BottleRep chain with learnable shortcut weights) and E-ELAN mirrors load the
    REFERENCE's state_dict (identical key lists) and reproduce the reference outputs (tools/make_golden_blocks.py) within 1e-3 -- measured
    ~1e-5: every RepVGG block is one folded 3x3 tcgen05 conv, every torch.cat is buffer aliasing."""
    from cvpytorch_b200 import yolo_blocks as YB
    from make_golden_blocks import case_inputs
    g = np.load(os.path.join(GOLD, 'yolo_blocks.npz'))
    ctors = {'rep_id': lambda: YB.RepVGGBlock(32, 32), 'rep_s2': lambda: YB.RepVGGBlock(32, 64, stride=2), 'rep_deploy': lambda: YB.RepVGGBlock(32, 32),
             'bepc3': lambda: YB.BepC3(64, 64, n=4), 'eelan': lambda: YB.EELAN(64, 32, 128)}
    for name, ctor in ctors.items():
        m = ctor()
        keys = [str(k) for k in g[f'{name}_keys']]
        assert list(m.state_dict().keys()) == keys, name
        sd, x = case_inputs(name, m.state_dict())
        m.load_state_dict(sd, strict=True)
        m = m.cuda().eval()
        if name == 'rep_deploy':
            m.switch_to_deploy()
            assert list(m.state_dict().keys()) == ['rbr_reparam.weight', 'rbr_reparam.bias']
        y = m(x.cuda())
        err = _rel(y[:, ::3], g[f'{name}_y'])  # the fixture keeps every 3rd channel
        print(name, 'rel err vs reference', err)
        assert err < TOL and err < 1e-4, (name, err)
