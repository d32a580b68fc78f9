"""Generates the YOLOX fixtures under tests/golden/ by running the REFERENCE (/root/reference) on CPU (build container only).

  yolox_keys.npz     state_dict keys / shapes of the reference composite (CSPDarknet + YOLOXNeck + YOLOXHead, SURVEY.md 3.5 row 3)
  yolox_calib.npz    BN running statistics of the calibration pass + predictor scales (cvpytorch_b200/synth.py)
  yolox_fwd128.npz   reference forward at 2x3x128x128 (seed 1029): backbone outputs, every 3rd channel of the neck / head outputs
  yolox_post320.npz  reference forward + yolox_post_process at 1x3x320x320: decoded tensor sample, detections
  yolox_nms.npz      reference yolox_post_process tail (score filter + torchvision.ops.batched_nms) on seeded candidate records,
                     both batched_nms regimes
"""
import importlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

import ref_shim  # noqa: E402
from cvpytorch_b200 import synth  # noqa: E402
from oracle import yolox_oracle as XO  # noqa: E402

GOLD = os.path.join(ROOT, 'tests', 'golden')
torch.set_num_threads(8)


def build_reference():
    ref_shim.install()
    from src.models.backbones import build_backbone
    from src.models.yolox import yolox_post_process
    bb = build_backbone({'name': 'CSPDarknet', 'subtype': 'yolox_s', 'out_stages': [2, 3, 4]})
    nk = importlib.import_module('src.models.necks.yolox_neck').YOLOXNeck('yolox_s', [256, 512, 1024], depth_mul=.33, width_mul=.5)
    hd = importlib.import_module('src.models.heads.yolox_head').YOLOXHead(num_classes=80, subtype='yolox_s', in_channels=[256, 512, 1024],
                                                                          depth_mul=.33, width_mul=.5)
    return bb, nk, hd, yolox_post_process


def load_parts(bb, nk, hd, sd):
    bb.load_state_dict(synth.split_prefix(sd, 'backbone.'), strict=True)
    nk.load_state_dict(synth.split_prefix(sd, 'neck.'), strict=True)
    hd.load_state_dict(synth.split_prefix(sd, 'head.'), strict=True)


def ref_tail(post, rec, conf, thr):
    """The reference's own filter + batched_nms lines (yolox.py:54-67) on ONE image's already decoded prediction rows."""
    import torchvision
    image_pred = torch.from_numpy(rec)
    class_conf, class_pred = image_pred[:, 5:6], image_pred[:, 6:7]
    conf_mask = (image_pred[:, 4] * class_conf.squeeze() >= conf).squeeze()
    detections = torch.cat((image_pred[:, :5], class_conf, class_pred.float()), 1)[conf_mask]
    if not detections.size(0):
        return np.zeros((0, 7), np.float32)
    idx = torchvision.ops.batched_nms(detections[:, :4], detections[:, 4] * detections[:, 5], detections[:, 6], thr)
    return detections[idx].numpy()


def main():
    bb, nk, hd, post = build_reference()
    tmpl = synth.yolox_template_state_dict()
    ref_keys = {**{'backbone.' + k: v for k, v in bb.state_dict().items()}, **{'neck.' + k: v for k, v in nk.state_dict().items()},
                **{'head.' + k: v for k, v in hd.state_dict().items()}}
    assert list(tmpl.keys()) == list(ref_keys.keys()), 'drop-in keys differ from the reference'
    assert all(tmpl[k].shape == ref_keys[k].shape for k in tmpl)
    np.savez_compressed(os.path.join(GOLD, 'yolox_keys.npz'), keys=np.array(list(ref_keys.keys())),
                        shapes=np.array([str(tuple(v.shape)) for v in ref_keys.values()]))

    # ---------------------------------------------------------------- calibration
    sd = synth.base_state_dict(tmpl)
    load_parts(bb, nk, hd, sd)
    mods = (bb, nk, hd)
    bns = [m for mod in mods for m in mod.modules() if isinstance(m, torch.nn.BatchNorm2d)]
    for m in bns:
        m.momentum = 1.0
    for mod in mods:
        mod.train()
    torch.manual_seed(7)
    xc = torch.randn(4, 3, 640, 640)
    with torch.no_grad():
        hd(nk(bb(xc)))
    for m in bns:
        m.momentum = 0.03
    for mod in mods:
        mod.eval()
    calib = {}
    for p, mod in (('backbone.', bb), ('neck.', nk), ('head.', hd)):
        for k, v in mod.state_dict().items():
            if k.endswith('running_mean') or k.endswith('running_var'):
                calib[p + k] = v.numpy().copy()
    # predictor scales: logits (without bias) with std 2.0 (cls, obj) / 0.5 (reg) on the calibration batch
    sd_c = {k: v.clone() for k, v in sd.items()}
    for k in sd_c:
        if k in calib:
            sd_c[k] = torch.from_numpy(calib[k]).clone()
    with torch.no_grad():
        feats = XO.neck(XO.backbone(xc, sd_c), sd_c)
        scales = np.zeros((3, 3))
        for i, f in enumerate(feats):
            xx = XO.conv_bn_silu(f, sd_c, f'head.stems.{i}', 1, 1)
            cf = XO.conv_bn_silu(XO.conv_bn_silu(xx, sd_c, f'head.cls_convs.{i}.0', 1, 1), sd_c, f'head.cls_convs.{i}.1', 1, 1)
            rf = XO.conv_bn_silu(XO.conv_bn_silu(xx, sd_c, f'head.reg_convs.{i}.0', 1, 1), sd_c, f'head.reg_convs.{i}.1', 1, 1)
            F = torch.nn.functional
            scales[i, 0] = 2.0 / float(F.conv2d(cf, sd_c[f'head.cls_preds.{i}.weight']).std())
            scales[i, 1] = 0.5 / float(F.conv2d(rf, sd_c[f'head.reg_preds.{i}.weight']).std())
            scales[i, 2] = 2.0 / float(F.conv2d(rf, sd_c[f'head.obj_preds.{i}.weight']).std())
    calib['pred_scale'] = scales
    np.savez_compressed(os.path.join(GOLD, 'yolox_calib.npz'), **calib)
    print('calibration saved; predictor scales', scales.round(2).tolist())

    sd = synth.yolox_state_dict(calibrated=True)
    load_parts(bb, nk, hd, sd)

    def ref_forward(x):
        with torch.no_grad():
            b = bb(x)
            n = nk(b)
            o = hd(n)
        return b, n, o

    torch.manual_seed(1029)
    x128 = torch.randn(2, 3, 128, 128)
    b, n, o = ref_forward(x128)
    oo = XO.forward(x128, sd)
    print('oracle vs reference @128: head rel err', max(float((a - r).abs().max() / r.abs().max()) for a, r in zip(oo, o)))
    np.savez_compressed(os.path.join(GOLD, 'yolox_fwd128.npz'), **{f'backbone{i}': t.numpy() for i, t in enumerate(b)},
                        **{f'neck{i}': t[:, ::3].numpy() for i, t in enumerate(n)}, **{f'head{i}': t[:, ::3].numpy() for i, t in enumerate(o)})

    torch.manual_seed(1029)
    x320 = torch.randn(1, 3, 320, 320)
    _, _, o = ref_forward(x320)
    dets = post([t.clone() for t in o], [8, 16, 32], 80, 0.01, 0.65)
    od = XO.post_process([t.clone() for t in o])
    rd = dets[0].numpy() if dets[0] is not None else np.zeros((0, 7), np.float32)
    dec = XO.decode([t.clone() for t in o])
    rec = XO.records(dec)
    print('@320: candidates >= 0.01:', int((rec[0, :, 7] >= 0.01).sum()), 'of', rec.shape[1], ' reference kept', rd.shape[0],
          ' oracle == reference (canonical tie order):', np.array_equal(XO.canonical_rows(od[0][0]), XO.canonical_rows(rd)),
          ' identical order:', np.array_equal(od[0][0], rd))
    assert np.array_equal(XO.canonical_rows(od[0][0]), XO.canonical_rows(rd))
    np.savez_compressed(os.path.join(GOLD, 'yolox_post320.npz'), det=rd, loc=od[0][1], records=rec[0], **{f'head{i}': t.numpy() for i, t in enumerate(o)})

    # ---------------------------------------------------------------- post-process tail on seeded records (both batched_nms regimes)
    out = {}
    for regime in ('few', 'typical', 'all'):
        for seed in (2, 3):
            rec = XO.make_stress_records(regime=regime, seed=seed)
            r = ref_tail(post, rec, 0.01, 0.65)
            o_rows, o_loc = XO.nms_records(rec, 0.01, 0.65)
            n_pass = int((rec[:, 7] >= 0.01).sum())
            assert np.array_equal(XO.canonical_rows(o_rows), XO.canonical_rows(r)), (regime, seed)
            print(f'stress {regime}/{seed}: pass {n_pass} ({"vanilla" if n_pass > 1000 else "trick"}), kept {r.shape[0]}  oracle == reference')
            out[f'{regime}_{seed}_det'] = r
            out[f'{regime}_{seed}_loc'] = o_loc
    np.savez_compressed(os.path.join(GOLD, 'yolox_nms.npz'), **out)
    for f in sorted(os.listdir(GOLD)):
        if f.startswith('yolox'):
            print('  ', f, os.path.getsize(os.path.join(GOLD, f)))


if __name__ == '__main__':
    main()
