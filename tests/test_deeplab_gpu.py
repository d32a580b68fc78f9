"""DeepLabv3+ (R50v1c) path on the B200 vs the reference goldens.  Tolerances: features / logits within 1e-3 relative;
labels: >= 99.99 % identical, every mismatch has a top-2 gap below 1e-3 * max|logit| (SURVEY.md 8d)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
TOL = 1e-3


def _rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).abs().max() / (b.abs().max() + 1e-12))


def test_deeplab_kernels(cuda):
    from cvpytorch_b200 import ops
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 64, 19, 23, generator=g).cuda()
    t = ops.SplitTensor(2, 19, 23, 64)
    ops.nchw_to_split(x, t.view())
    xr = ops.split_to_nchw(t.view())
    # depthwise dilated conv + ReLU
    for dil in (1, 2, 12):
        w = torch.randn(64, 1, 3, 3, generator=g, dtype=torch.float64)
        b = torch.randn(64, generator=g, dtype=torch.float64)
        w9c, bias = ops.pack_dw_weights(w, b)
        y = ops.SplitTensor(2, 19, 23, 64)
        ops.dwconv3x3(t.view(), w9c, bias, dil, y.view(), True)
        ref = F.relu(F.conv2d(xr, w.float().cuda(), b.float().cuda(), 1, dil, dil, groups=64))
        assert _rel(ops.split_to_nchw(y.view()), ref) < 2e-6, dil
    # global average pool
    p = ops.SplitTensor(2, 1, 1, 64)
    ops.global_avgpool(t.view(), p.view())
    assert _rel(ops.split_to_nchw(p.view()), xr.mean((2, 3), keepdim=True)) < 2e-6
    # bilinear resize (align_corners=False): x8 up, odd sizes, and the 1x1 broadcast
    for (ho, wo) in ((152, 184), (37, 51)):
        y = ops.SplitTensor(2, ho, wo, 64)
        ops.bilinear_resize(t.view(), y.view())
        assert _rel(ops.split_to_nchw(y.view()), F.interpolate(xr, size=(ho, wo), mode='bilinear', align_corners=False)) < 2e-6
    y = ops.SplitTensor(2, 5, 7, 64)
    ops.bilinear_resize(p.view(), y.view())
    assert _rel(ops.split_to_nchw(y.view()), ops.split_to_nchw(p.view()).expand(2, 64, 5, 7)) < 1e-7
    # fused upsample + argmax
    lg = ops.F32Tensor(2, 16, 24, 32)
    lg.data.normal_(0, 2)
    labels = torch.zeros((2, 64, 96), dtype=torch.int64, device='cuda')
    ops.upsample_argmax(lg.view(0, 19), 19, labels)
    up = F.interpolate(lg.data[..., :19].permute(0, 3, 1, 2), size=(64, 96), mode='bilinear', align_corners=False)
    ref = up.argmax(1)
    mism = labels != ref
    assert float(mism.float().mean()) < 1e-4
    if mism.any():
        top2 = up.topk(2, dim=1).values
        assert float((top2[:, 0] - top2[:, 1])[mism].max()) < 1e-4


def test_deeplab_forward_vs_reference_golden(cuda):
    from cvpytorch_b200 import ops, synth
    g = np.load(os.path.join(GOLD, 'deeplab_fwd.npz'))
    model = synth.build_deeplab(True)
    torch.manual_seed(1029)
    x = torch.randn(2, 3, 128, 256).cuda()
    labels = model(x, torch.zeros(2, 128, 256), 'val')
    torch.cuda.synchronize()
    assert labels.dtype == torch.int64 and tuple(labels.shape) == (2, 128, 256)
    G = model._graph_for(x, (128, 256))
    errs = {'low': _rel(ops.split_to_nchw(G['feats'][0].view())[:, ::8], g['low_sub']),
            'high': _rel(ops.split_to_nchw(G['feats'][1].view())[:, ::3], g['high']),
            'logits': _rel(G['logits'].data[..., :19].permute(0, 3, 1, 2), g['logits'])}
    print(errs)
    assert max(errs.values()) < TOL, errs
    ref = torch.from_numpy(g['labels'].astype(np.int64))
    mism = labels.cpu() != ref
    frac = float(mism.float().mean())
    print('label mismatch fraction', frac)
    up = F.interpolate(torch.from_numpy(g['logits']), size=(128, 256), mode='bilinear', align_corners=False)
    top2 = up.topk(2, dim=1).values
    gap = (top2[:, 0] - top2[:, 1])
    assert frac <= 1e-4 or float(gap[mism].max()) < 1e-3 * float(up.abs().max())
    if mism.any():
        assert float(gap[mism].max()) < 1e-3 * float(up.abs().max())
    # component-level API
    feats = model.backbone(x)
    logits = model.head(feats)
    assert _rel(logits, g['logits']) < TOL
