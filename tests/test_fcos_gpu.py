"""FCOS-R50 path on the B200 (through the C ABI) vs reference goldens / the oracle.
Tolerances: fp32 activations / logits within 1e-3 relative (max|a-b|/max|b|); NMS-kept rows bit-exact on identical candidates."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, 'tests', 'golden')
sys.path.insert(0, os.path.join(ROOT, 'tools'))
TOL = 1e-3


def _rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).abs().max() / (b.abs().max() + 1e-12))


@pytest.fixture(scope='module')
def model(cuda):
    from cvpytorch_b200 import synth
    return synth.build_fcos(True)


def test_maxpool_and_groupnorm_kernels(cuda):
    from cvpytorch_b200 import ops
    x = torch.randn(2, 64, 37, 50, device='cuda')
    t = ops.SplitTensor(2, 37, 50, 64)
    ops.nchw_to_split(x, t.view())
    xr = ops.split_to_nchw(t.view())
    y = ops.SplitTensor(2, 19, 25, 64)
    ops.maxpool3x3s2(t.view(), y.view())
    assert torch.equal(ops.split_to_nchw(y.view()), F.max_pool2d(xr, 3, 2, 1))
    # GroupNorm(32, 256) + ReLU
    x = torch.randn(3, 256, 13, 17, device='cuda') * 3 + 1
    t = ops.SplitTensor(3, 13, 17, 256)
    ops.nchw_to_split(x, t.view())
    gamma, beta = torch.rand(256, device='cuda') + 0.5, torch.randn(256, device='cuda')
    z = ops.SplitTensor(3, 13, 17, 256)
    ws = ops.GroupNormWorkspace(3, 32)
    ops.groupnorm_relu(t.view(), 32, gamma, beta, 1e-5, z.view(), ws)
    ref = F.relu(F.group_norm(ops.split_to_nchw(t.view()), 32, gamma, beta, 1e-5))
    assert _rel(ops.split_to_nchw(z.view()), ref) < 2e-5
    # split -> fp32 copy
    f = ops.F32Tensor(3, 13, 17, 256)
    ops.split_to_f32(t.view(), f.view())
    assert torch.equal(f.data.permute(0, 3, 1, 2), ops.split_to_nchw(t.view()))


def test_resnet_stem_window_conv(cuda):
    """7x7/s2/p3 stem as 4 filter rows over the space-to-depth input (row-window mode, pad_left = 2)."""
    from cvpytorch_b200 import ops
    from cvpytorch_b200.fcos_models import resnet_stem_weights_to_s2d
    g = torch.Generator().manual_seed(6)
    B, H, W = 2, 64, 96
    x = torch.randn(B, 3, H, W, generator=g)
    w = torch.randn(64, 3, 7, 7, generator=g) / 147 ** 0.5
    b = torch.randn(64, generator=g)
    ref = F.relu(F.conv2d(x.cuda(), w.cuda(), b.cuda(), 2, 3))
    t = ops.SplitTensor(B, H // 2, W // 2 + 3, 16)
    ops.stem_s2d(x.cuda().contiguous(), t.view(), pad_left=2)
    wp, bp = ops.pack_conv_weights(ops.window_weights(resnet_stem_weights_to_s2d(w.double()), 4), b.double())
    out = ops.SplitTensor(B, H // 2, W // 2, 64)
    ops.ConvPlan(t.view(), out.view(), wp, bp, 4, 1, 2, 1, 'relu', w_window=4).run()
    torch.cuda.synchronize()
    assert _rel(ops.split_to_nchw(out.view()), ref) < 2e-5


def test_conv_residual_before_activation(cuda):
    from cvpytorch_b200 import ops
    g = torch.Generator().manual_seed(9)
    x = torch.randn(2, 64, 20, 20, generator=g)
    w = torch.randn(256, 64, 1, 1, generator=g) / 8
    b = torch.randn(256, generator=g)
    r = torch.randn(2, 256, 20, 20, generator=g)
    ref = F.relu(F.conv2d(x.cuda(), w.cuda(), b.cuda()) + r.cuda())
    tin, tres, tout = ops.SplitTensor(2, 20, 20, 64), ops.SplitTensor(2, 20, 20, 256), ops.SplitTensor(2, 20, 20, 256)
    ops.nchw_to_split(x.cuda(), tin.view())
    ops.nchw_to_split(r.cuda(), tres.view())
    wp, bp = ops.pack_conv_weights(w.double(), b.double())
    ops.ConvPlan(tin.view(), tout.view(), wp, bp, 1, 1, 0, 1, 'relu', residual=tres.view(), residual_before_act=1).run()
    torch.cuda.synchronize()
    assert _rel(ops.split_to_nchw(tout.view()), ref) < 2e-5


def test_fcos_forward_vs_reference_golden_128(model):
    g = np.load(os.path.join(GOLD, 'fcos_fwd128.npz'))
    torch.manual_seed(1029)
    x = torch.randn(2, 3, 128, 128).cuda()
    model.predict(x)
    torch.cuda.synchronize()
    G = model._graph_for(x)
    from cvpytorch_b200 import ops
    errs = {'C5': _rel(ops.split_to_nchw(G['feats'][2].view())[:, ::3], g['C5'])}  # the fixture keeps every 3rd C5 channel
    for i in range(5):
        errs[f'P{i + 3}'] = _rel(ops.split_to_nchw(G['levels'][i].view()), g[f'P{i + 3}'])
        cls, rc = G['head'][i]
        errs[f'cls{i}'] = _rel(cls.data[..., :80].permute(0, 3, 1, 2), g[f'cls{i}'])
        errs[f'cnt{i}'] = _rel(rc.data[..., 4:5].permute(0, 3, 1, 2), g[f'cnt{i}'])
        errs[f'logreg{i}'] = _rel(rc.data[..., 0:4].permute(0, 3, 1, 2), np.log(g[f'reg{i}']))  # reg = exp(raw * scale), scale = 1
    print(errs)
    assert max(errs.values()) < TOL, errs


def test_fcos_components_nchw_api(model):
    """backbone / neck / head called one by one with the reference's NCHW tensors."""
    g = np.load(os.path.join(GOLD, 'fcos_fwd128.npz'))
    torch.manual_seed(1029)
    x = torch.randn(2, 3, 128, 128).cuda()
    feats = model.backbone(x)
    assert _rel(feats[2][:, ::3], g['C5']) < TOL
    levels = model.neck(feats)
    cls, cnt, reg = model.head(levels)
    for i in range(5):
        assert _rel(levels[i], g[f'P{i + 3}']) < TOL and _rel(cls[i], g[f'cls{i}']) < TOL
        assert _rel(cnt[i], g[f'cnt{i}']) < TOL and _rel(reg[i], g[f'reg{i}']) < 2 * TOL


@pytest.mark.parametrize('name', ['dense', 'sparse'])
def test_fcos_nms_bit_exact_vs_reference_golden(cuda, name):
    from cvpytorch_b200 import ops
    from make_golden_fcos import make_fcos_candidates
    g = np.load(os.path.join(GOLD, 'fcos_nms_stress.npz'))
    s, c, b = make_fcos_candidates(2, dense=(name == 'dense'))
    ws = ops.FcosWorkspace(2, s.shape[1], 1000)
    sc, cl, bx, loc, cnt = ops.fcos_nms(ws, 0.05, 0.6, torch.from_numpy(s).cuda(), torch.from_numpy(c).cuda(), torch.from_numpy(b).cuda().contiguous())
    torch.cuda.synchronize()
    assert int(ws.status[0]) == 0
    for bi in range(2):
        k = int(cnt[bi])
        assert k == g[f'{name}_{bi}_scores'].shape[0]
        assert np.array_equal(sc[bi, :k].cpu().numpy(), g[f'{name}_{bi}_scores'])
        assert np.array_equal(bx[bi, :k].cpu().numpy(), g[f'{name}_{bi}_boxes'])
        assert np.array_equal(cl[bi, :k].cpu().numpy().astype(np.int64), g[f'{name}_{bi}_classes'].astype(np.int64))


def test_fcos_end_to_end_detect_256(model):
    """Whole pipeline at 1x3x256x256: decoded candidates vs the oracle, and the CUDA NMS on the GPU's own candidates
    vs the oracle NMS on the same arrays (bit-exact)."""
    from cvpytorch_b200 import synth
    from oracle import fcos_oracle as FO
    torch.manual_seed(1029)
    x = torch.randn(1, 3, 256, 256)
    sc, cl, bx, loc, cnt = model.predict(x.cuda())
    torch.cuda.synchronize()
    ws = model._graph_for(x.cuda())['ws']
    sd = synth.fcos_state_dict(True)
    _, _, cls, cntl, reg = FO.forward(x, sd)
    dets, (osc, ocl, obx) = FO.fcos_detect(cls, cntl, reg)
    assert _rel(ws.scores, osc) < TOL and _rel(ws.boxes, obx) < TOL
    assert float((ws.classes.cpu() == ocl.int()).float().mean()) > 0.98
    # NMS exactness on the GPU's own candidate arrays
    s_np, c_np, b_np = ws.scores[0].cpu().numpy(), ws.classes[0].cpu().numpy(), ws.boxes[0].cpu().numpy()
    top = np.argsort(-s_np, kind='stable')[:1000]
    m = s_np[top] >= np.float32(0.05)
    sm, cm, bm, lm = s_np[top][m], c_np[top][m], b_np[top][m], top[m]
    off = cm.astype(np.float32) * (bm.max() + np.float32(1))
    keep = FO.box_nms(bm + off[:, None], sm, 0.6)
    k = int(cnt[0])
    assert k == len(keep)
    assert np.array_equal(loc[0, :k].cpu().numpy().astype(np.int64), lm[keep])
    assert np.array_equal(sc[0, :k].cpu().numpy(), sm[keep]) and np.array_equal(bx[0, :k].cpu().numpy(), bm[keep])
    # contract of forward(..., 'val')
    out = model(x.cuda(), None, 'val')
    assert isinstance(out, tuple) and set(out[1][0].keys()) == {'boxes', 'labels', 'scores'}
