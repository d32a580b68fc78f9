"""Generates the DeepLabv3+ (R50v1c) fixtures under tests/golden/ by running the REFERENCE (/root/reference) on CPU.
  deeplab_keys.npz   state_dict keys/shapes of the reference ResNet('resnet50v1c') / Deeplabv3PlusHead
  deeplab_calib.npz  BN running statistics of the calibrated synthetic model + cls_seg scale
  deeplab_fwd.npz    reference forward, 2x3x128x256 (seed 1029): every 8th / 3rd channel of the low / high features, logits, upsampled argmax labels
"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

import ref_shim  # noqa: E402
from cvpytorch_b200 import synth  # noqa: E402
from oracle import deeplab_oracle as DO  # noqa: E402

GOLD = os.path.join(ROOT, 'tests', 'golden')
torch.set_num_threads(8)


def main():
    ref_shim.install()
    import src.models.backbones.seg.resnet as R
    R.ResNet.load_pretrained_weights = R.ResNet.init_weights
    from src.models.backbones import build_backbone
    from src.models.heads import build_head
    cfg = synth.DEEPLAB_CFG
    bb = build_backbone({**cfg['BACKBONE'], 'pretrained': False})
    hd = build_head(cfg['HEAD'])
    tmpl = synth.deeplab_template_state_dict()
    ref_keys = {**{'backbone.' + k: v for k, v in bb.state_dict().items()}, **{'head.' + k: v for k, v in hd.state_dict().items()}}
    assert list(tmpl.keys()) == list(ref_keys.keys()), sorted(set(tmpl) ^ set(ref_keys))[:10]
    assert all(tmpl[k].shape == ref_keys[k].shape for k in tmpl)
    np.savez_compressed(os.path.join(GOLD, 'deeplab_keys.npz'), keys=np.array(list(ref_keys.keys())),
                        shapes=np.array([str(tuple(v.shape)) for v in ref_keys.values()]))

    def load(sd):
        bb.load_state_dict(synth.split_prefix(sd, 'backbone.'), strict=True)
        hd.load_state_dict(synth.split_prefix(sd, 'head.'), strict=True)

    sd = synth.base_state_dict(tmpl)
    load(sd)
    bns = [m for mod in (bb, hd) for m in mod.modules() if isinstance(m, torch.nn.BatchNorm2d)]
    for m in bns:
        m.momentum = 1.0
    bb.train()
    hd.train()
    torch.manual_seed(7)
    xc = torch.randn(4, 3, 256, 512)
    with torch.no_grad():
        logits = hd(bb(xc))
    for m in bns:
        m.momentum = 0.1
    bb.eval()
    hd.eval()
    calib = {}
    for p, mod in (('backbone.', bb), ('head.', hd)):
        for k, v in mod.state_dict().items():
            if k.endswith('running_mean') or k.endswith('running_var'):
                calib[p + k] = v.numpy().copy()
    with torch.no_grad():
        logits = hd(bb(xc))
    calib['cls_scale'] = np.asarray(2.0 / float(logits.std()))
    np.savez_compressed(os.path.join(GOLD, 'deeplab_calib.npz'), **calib)
    sd = synth.deeplab_state_dict(True)
    load(sd)

    torch.manual_seed(1029)
    x = torch.randn(2, 3, 128, 256)
    with torch.no_grad():
        feats = bb(x)
        logits = hd(feats)
        labels = torch.argmax(F.interpolate(logits, size=x.shape[2:], mode='bilinear', align_corners=False), dim=1)  # encoder_decoder.py:132-133
    ofe, olog, olab = DO.forward(x, sd)
    print('oracle vs reference: logits rel err', float((olog - logits).abs().max() / logits.abs().max()), 'labels equal', bool((olab == labels).all()))
    print('logits std %.3f, classes present %d, high feat std %.3f' % (float(logits.std()), int(labels.unique().numel()), float(feats[1].std())))
    np.savez_compressed(os.path.join(GOLD, 'deeplab_fwd.npz'), low_sub=feats[0].numpy()[:, ::8].copy(), high=feats[1].numpy()[:, ::3].copy(), logits=logits.numpy(),
                        labels=labels.numpy().astype(np.uint8))
    for f in sorted(os.listdir(GOLD)):
        if f.startswith('deeplab'):
            print('  ', f, os.path.getsize(os.path.join(GOLD, f)))


if __name__ == '__main__':
    main()
