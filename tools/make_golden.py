"""Generates the committed fixtures under tests/golden/ by running the REFERENCE (/root/reference) on CPU.

Run once in the build container:  python tools/make_golden.py
(The GPU box has no /root/reference; tests only read the .npz files written here.)

Outputs
  yolov5s_calib.npz   BN running statistics + Detect scales of the calibrated synthetic model (see cvpytorch_b200/synth.py)
  yolov5s_fwd128.npz  reference forward, 2x3x128x128 (seed 1029): backbone outs, neck outs, decoded z (every 3rd channel / anchor row of each)
  yolov5s_fwd640.npz  reference forward, 1x3x640x640 (seed 1029): every 16th anchor row of z + reference NMS result on the full z
  nms_stress.npz      reference non_max_suppression (+torchvision.ops.nms) kept rows on the seeded stress set (4 regimes x 2 modes)
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
from oracle import nms_oracle as NO  # noqa: E402
from oracle import yolov5_oracle as YO  # noqa: E402

GOLD = os.path.join(ROOT, 'tests', 'golden')
os.makedirs(GOLD, exist_ok=True)
torch.set_num_threads(8)


def load_parts(bb, nk, dt, sd):
    bb.load_state_dict(synth.split_prefix(sd, 'backbone.'), strict=True)
    nk.load_state_dict(synth.split_prefix(sd, 'neck.'), strict=True)
    dt.load_state_dict(synth.split_prefix(sd, 'detect.'), strict=True)


def main():
    bb, nk, dt, ref_nms = ref_shim.build_yolov5s()
    # the drop-in template must equal the reference's keys/shapes
    tmpl = synth.template_state_dict()
    ref_keys = {**{'backbone.' + k: v for k, v in bb.state_dict().items()}, **{'neck.' + k: v for k, v in nk.state_dict().items()},
                **{'detect.' + k: v for k, v in dt.state_dict().items()}}
    assert list(tmpl.keys()) == list(ref_keys.keys())
    assert all(tmpl[k].shape == ref_keys[k].shape for k in tmpl)
    np.savez_compressed(os.path.join(GOLD, 'yolov5s_keys.npz'), keys=np.array(list(ref_keys.keys())),
                        shapes=np.array([str(tuple(v.shape)) for v in ref_keys.values()]))

    # ---------------------------------------------------------------- calibration (SURVEY.md §8d recipe)
    sd = synth.base_state_dict(tmpl)
    load_parts(bb, nk, dt, sd)
    bns = [m for mod in (bb, nk) for m in mod.modules() if isinstance(m, torch.nn.BatchNorm2d)]
    for m in bns:
        m.momentum = 1.0
    bb.train()
    nk.train()
    torch.manual_seed(7)
    xc = torch.randn(4, 3, 640, 640)
    with torch.no_grad():
        feats = nk(bb(xc))
    for m in bns:
        m.momentum = 0.03
    bb.eval()
    nk.eval()
    dt.eval()
    calib = {}
    for p, mod in (('backbone.', bb), ('neck.', nk)):
        for k, v in mod.state_dict().items():
            if k.endswith('running_mean') or k.endswith('running_var'):
                calib[p + k] = v.numpy().copy()
    with torch.no_grad():
        feats = nk(bb(xc))  # eval-mode features with the calibrated statistics
        scales = []
        for i, f in enumerate(feats):
            logit = torch.nn.functional.conv2d(f, sd[f'detect.m.{i}.weight'])
            scales.append(1.5 / float(logit.std()))
    calib['detect_scale'] = np.asarray(scales, dtype=np.float64)
    np.savez_compressed(os.path.join(GOLD, 'yolov5s_calib.npz'), **calib)
    print('calibration saved; detect scales', scales, 'feature std', [float(f.std()) for f in feats])

    sd = synth.yolov5s_state_dict(calibrated=True)
    load_parts(bb, nk, dt, sd)

    # ---------------------------------------------------------------- forward goldens
    def ref_forward(x):
        with torch.no_grad():
            b = bb(x)
            n = nk(b)
            z, raws = dt(list(n))
        return b, n, z, raws

    torch.manual_seed(1029)
    x128 = torch.randn(2, 3, 128, 128)
    b, n, z, raws = ref_forward(x128)
    oz, oraws = YO.forward(x128, sd)
    print('oracle vs reference @128: z rel err', YO.rel_err(oz, z))
    np.savez_compressed(os.path.join(GOLD, 'yolov5s_fwd128.npz'), z=z[:, ::3].numpy(), **{f'backbone{i}': t[:, ::3].numpy() for i, t in enumerate(b)},
                        **{f'neck{i}': t[:, ::3].numpy() for i, t in enumerate(n)})

    torch.manual_seed(1029)
    x640 = torch.randn(1, 3, 640, 640)
    b, n, z, raws = ref_forward(x640)
    oz, _ = YO.forward(x640, sd)
    print('oracle vs reference @640: z rel err', YO.rel_err(oz, z), ' raw logits std', float(raws[0].std()), 'max', float(raws[0].abs().max()))
    obj = z[0, :, 4]
    conf = z[0, :, 5:] * obj[:, None]
    print('anchors obj>0.001:', int((obj > 0.001).sum()), ' (anchor,class) pairs > 0.001:', int(((conf > 0.001) & (obj[:, None] > 0.001)).sum()))
    dets = ref_nms(z.clone(), 0.001, 0.6, multi_label=True)
    odet = NO.non_max_suppression(z.numpy(), 0.001, 0.6, multi_label=True)
    print('reference NMS kept', dets[0].shape[0], ' oracle == reference:', np.array_equal(odet[0][0], dets[0].numpy()))
    np.savez_compressed(os.path.join(GOLD, 'yolov5s_fwd640.npz'), z_sub=z[0, ::16].numpy(), nms_det=dets[0].numpy(),
                        nms_idx=odet[0][1], z_absmean=z[0].abs().mean(0).numpy())

    # ---------------------------------------------------------------- NMS stress goldens (reference NMS itself)
    out = {}
    for regime in ('few', 'sparse', 'typical', 'capped'):
        pred = NO.make_stress_prediction(2, regime=regime, seed=2)
        for ml in (True, False):
            r = ref_nms(torch.from_numpy(pred.copy()), 0.001, 0.6, multi_label=ml)
            o = NO.non_max_suppression(pred, 0.001, 0.6, multi_label=ml)
            for bi in range(2):
                assert np.array_equal(o[bi][0], r[bi].numpy()), (regime, ml, bi)
                out[f'{regime}_{int(ml)}_{bi}_det'] = r[bi].numpy()
                out[f'{regime}_{int(ml)}_{bi}_idx'] = o[bi][1]
    np.savez_compressed(os.path.join(GOLD, 'nms_stress.npz'), **out)
    print('golden fixtures written to', GOLD)
    for f in sorted(os.listdir(GOLD)):
        print('  ', f, os.path.getsize(os.path.join(GOLD, f)))


if __name__ == '__main__':
    main()
