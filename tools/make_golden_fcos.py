"""Generates the FCOS-R50 fixtures under tests/golden/ by running the REFERENCE (/root/reference) on CPU.

Run once in the build container:  python tools/make_golden_fcos.py
  fcos_keys.npz     state_dict keys/shapes of the reference ResNet / FCOSFPN / FCOSHead
  fcos_calib.npz    BN running statistics of the calibrated synthetic ResNet-50 + head scales (see cvpytorch_b200/synth.py)
  fcos_fwd128.npz   reference forward, 2x3x128x128 (seed 1029): every 3rd channel of C5, P3..P7, per-level cls / cnt / reg
  fcos_det256.npz   reference FCOSDetect on the reference's own head outputs, 1x3x256x256: scores / classes / boxes
  fcos_nms_stress.npz  reference _post_process (batched_nms + box_nms) on seeded synthetic candidates
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

import ref_shim  # noqa: E402
from cvpytorch_b200 import synth  # noqa: E402
from oracle import fcos_oracle as FO  # noqa: E402

GOLD = os.path.join(ROOT, 'tests', 'golden')
torch.set_num_threads(8)


def make_fcos_candidates(B, N=13343, nc=80, seed=3, dense=True):
    """Seeded synthetic (scores, classes, boxes) for the FCOS post-processing stress test (unique scores)."""
    rng = np.random.default_rng(seed)
    G = 60
    gxy = rng.uniform(40, 760, size=(B, G, 2))
    gwh = rng.uniform(20, 200, size=(B, G, 2))
    gcl = rng.integers(1, nc + 1, size=(B, G))
    owner = rng.integers(0, G, size=(B, N))
    ctr = np.take_along_axis(gxy, owner[..., None].repeat(2, -1), 1) + rng.normal(0, 6, size=(B, N, 2))
    wh = np.take_along_axis(gwh, owner[..., None].repeat(2, -1), 1) * (1 + rng.normal(0, 0.08, size=(B, N, 2)))
    boxes = np.concatenate([ctr - wh / 2, ctr + wh / 2], -1).astype(np.float32)
    classes = np.take_along_axis(gcl, owner, 1).astype(np.int32)
    scores = (rng.beta(2, 5, size=(B, N)) if dense else rng.beta(1, 30, size=(B, N))).astype(np.float32)
    scores += (np.arange(B * N).reshape(B, N) % 1009).astype(np.float32) * np.float32(2.0 ** -22)  # de-duplicate
    return scores, classes, boxes


def main():
    ref_shim.install()
    import src.models.backbones.seg.resnet as R
    R.ResNet.load_pretrained_weights = R.ResNet.init_weights
    from src.models.backbones import build_backbone
    from src.models.detects import build_detect
    from src.models.heads import build_head
    from src.models.necks import build_neck
    cfg = synth.FCOS_CFG
    bb = build_backbone({**cfg['BACKBONE'], 'pretrained': False})
    nk = build_neck(cfg['NECK'])
    hd = build_head({**cfg['HEAD'], 'num_classes': 80})
    dt = build_detect(cfg['DETECT'])
    tmpl = synth.fcos_template_state_dict()
    ref_keys = {**{'backbone.' + k: v for k, v in bb.state_dict().items()}, **{'neck.' + k: v for k, v in nk.state_dict().items()},
                **{'head.' + k: v for k, v in hd.state_dict().items()}}
    assert list(tmpl.keys()) == list(ref_keys.keys()) and all(tmpl[k].shape == ref_keys[k].shape for k in tmpl)
    np.savez_compressed(os.path.join(GOLD, 'fcos_keys.npz'), keys=np.array(list(ref_keys.keys())),
                        shapes=np.array([str(tuple(v.shape)) for v in ref_keys.values()]))

    def load(sd):
        bb.load_state_dict(synth.split_prefix(sd, 'backbone.'), strict=True)
        nk.load_state_dict(synth.split_prefix(sd, 'neck.'), strict=True)
        hd.load_state_dict(synth.split_prefix(sd, 'head.'), strict=True)

    # ---------------------------------------------------------------- calibration
    sd = synth.base_state_dict(tmpl)
    load(sd)
    bns = [m for m in bb.modules() if isinstance(m, torch.nn.BatchNorm2d)]
    for m in bns:
        m.momentum = 1.0
    bb.train()
    torch.manual_seed(7)
    xc = torch.randn(4, 3, 256, 256)
    with torch.no_grad():
        bb(xc)
    for m in bns:
        m.momentum = 0.1
    bb.eval()
    nk.eval()
    hd.eval()
    calib = {'backbone.' + k: v.numpy().copy() for k, v in bb.state_dict().items() if k.endswith('running_mean') or k.endswith('running_var')}
    with torch.no_grad():
        cls, cnt, reg = hd(nk(bb(xc)))
        std = lambda xs: float(torch.cat([x.flatten() for x in xs]).std())
        cls_std = std([c - sd['head.cls_logits.bias'].view(1, -1, 1, 1) for c in cls])
        cnt_std = std(cnt)
        reg_std = std([torch.log(r) for r in reg])
    calib['head_scale'] = np.asarray([2.0 / cls_std, 2.0 / cnt_std, 1.0 / reg_std], dtype=np.float64)
    np.savez_compressed(os.path.join(GOLD, 'fcos_calib.npz'), **calib)
    print('calibration: head logits std (cls, cnt, log reg) =', cls_std, cnt_std, reg_std)

    sd = synth.fcos_state_dict(calibrated=True)
    load(sd)

    # ---------------------------------------------------------------- forward goldens
    torch.manual_seed(1029)
    x128 = torch.randn(2, 3, 128, 128)
    with torch.no_grad():
        feats = bb(x128)
        levels = nk(feats)
        cls, cnt, reg = hd(levels)
    ofe, olv, ocls, ocnt, oreg = FO.forward(x128, sd)
    errs = [float((a - b).abs().max() / b.abs().max()) for a, b in zip(list(ofe) + list(olv) + ocls + ocnt + oreg, list(feats) + list(levels) + cls + cnt + reg)]
    print('oracle vs reference @128 max rel err over all tensors:', max(errs))
    out = {'C5': feats[2][:, ::3].numpy()}
    for i in range(5):
        out[f'P{i + 3}'] = levels[i].numpy()
        out[f'cls{i}'] = cls[i].numpy()
        out[f'cnt{i}'] = cnt[i].numpy()
        out[f'reg{i}'] = reg[i].numpy()
    np.savez_compressed(os.path.join(GOLD, 'fcos_fwd128.npz'), **out)
    print('feature std: C5 %.3f, P3 %.3f, cls logits %.3f, reg median %.3f' % (float(feats[2].std()), float(levels[0].std()), float(cls[0].std()), float(reg[0].median())))

    # ---------------------------------------------------------------- detect golden (reference FCOSDetect on its own head outputs)
    torch.manual_seed(1029)
    x256 = torch.randn(1, 3, 256, 256)
    with torch.no_grad():
        cls, cnt, reg = hd(nk(bb(x256)))
        sc, cl, bx = dt([[c.clone() for c in cls], [c.clone() for c in cnt], [r.clone() for r in reg]])
    dets, _ = FO.fcos_detect(cls, cnt, reg)
    same = np.array_equal(dets[0][0], sc[0].numpy()) and np.array_equal(dets[0][1], cl[0].numpy()) and np.array_equal(dets[0][2], bx[0].numpy())
    print('reference FCOSDetect kept', sc.shape[1], ' oracle == reference:', same)
    np.savez_compressed(os.path.join(GOLD, 'fcos_det256.npz'), scores=sc[0].numpy(), classes=cl[0].numpy(), boxes=bx[0].numpy(),
                        **{f'cls{i}': cls[i].numpy() for i in range(5)}, **{f'cnt{i}': cnt[i].numpy() for i in range(5)},
                        **{f'reg{i}': reg[i].numpy() for i in range(5)})

    # ---------------------------------------------------------------- NMS stress goldens (reference _post_process itself)
    out = {}
    for name, dense in (('dense', True), ('sparse', False)):
        s, c, b = make_fcos_candidates(2, dense=dense)
        for bi in range(2):
            top = np.argsort(-s[bi], kind='stable')[:1000]
            rs, rc, rb = dt._post_process([torch.from_numpy(s[bi][top])[None], torch.from_numpy(c[bi][top].astype(np.int64))[None],
                                           torch.from_numpy(b[bi][top])[None]])
            m = s[bi][top] >= np.float32(0.05)
            sm, cm, bm = s[bi][top][m], c[bi][top][m], b[bi][top][m]
            off = cm.astype(np.float32) * (bm.max() + np.float32(1))
            keep = FO.box_nms(bm + off[:, None], sm, 0.6)
            ok = np.array_equal(sm[keep], rs[0].numpy()) and np.array_equal(bm[keep], rb[0].numpy()) and np.array_equal(cm[keep], rc[0].numpy())
            print(f'nms stress {name} img {bi}: candidates {int(m.sum())}, kept {len(keep)}, oracle == reference: {ok}')
            assert ok
            out[f'{name}_{bi}_scores'] = rs[0].numpy()
            out[f'{name}_{bi}_classes'] = rc[0].numpy()
            out[f'{name}_{bi}_boxes'] = rb[0].numpy()
    np.savez_compressed(os.path.join(GOLD, 'fcos_nms_stress.npz'), **out)
    for f in sorted(os.listdir(GOLD)):
        if f.startswith('fcos'):
            print('  ', f, os.path.getsize(os.path.join(GOLD, f)))


if __name__ == '__main__':
    main()
