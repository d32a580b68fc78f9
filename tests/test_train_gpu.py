"""SURVEY.md 8(f) rank 3 -- the YOLOX C3 block's TRAINING step (forward + backward) on the B200 kernels (cvpytorch_b200/train.py,
csrc/train_kernels.cu) against (1) torch on the same GPU, kernel by kernel, on bf16-representable inputs, and (2) the committed reference
fixture tests/golden/c3_train.npz = the reference CSPLayer + torch.autograd in fp32 on CPU (tools/make_golden_train.py).

Tolerances (bf16 step: 8-bit mantissa, |rounding| <= 2^-9 = 2e-3 per stored activation / gradient; fp32 accumulation everywhere):
  single kernels, bf16 outputs        max|a-b| / max|b| <= 6e-3        fp32 outputs (wgrad, BN statistics)  <= 2e-3
  whole block vs the fp32 reference   forward <= 3e-2, d/dx and every parameter gradient <= 6e-2  (5-9 bf16 layers deep each way)"""
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


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / (b.abs().max() + 1e-12))


def _bf(t):
    return t.to(torch.bfloat16).float()


@pytest.mark.parametrize('B,H,W,cin,cout,k', [(2, 16, 16, 64, 64, 1), (3, 20, 20, 128, 64, 3), (2, 13, 9, 64, 128, 3), (1, 40, 40, 128, 128, 1), (5, 8, 8, 256, 64, 1), (2, 10, 10, 256, 512, 1), (1, 12, 12, 512, 256, 3)])  # (incl. the 256 / 512-channel layers of dark4 / dark5)
def test_conv_forward_backward_data_backward_weight(cuda, B, H, W, cin, cout, k):
    from cvpytorch_b200 import train as T
    g = torch.Generator().manual_seed(B * 100 + H + cin + k)
    x = _bf(torch.randn(B, cin, H, W, generator=g)).cuda().requires_grad_(True)
    w = _bf(torch.randn(cout, cin, k, k, generator=g) / (cin * k * k) ** 0.5).cuda().requires_grad_(True)
    dy = _bf(torch.randn(B, cout, H, W, generator=g)).cuda()
    y_ref = F.conv2d(x, w, None, 1, k // 2)
    y_ref.backward(dy)
    xh = x.detach().permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)
    dyh = dy.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)
    wf, wb = T.pack_weights(w.detach())
    y = T.conv(xh, wf, cout, k).float().permute(0, 3, 1, 2)
    dx = T.conv(dyh, wb, cin, k).float().permute(0, 3, 1, 2)
    dw = T.conv_wgrad(xh, dyh, k)
    torch.cuda.synchronize()
    e = dict(y=_rel(y, y_ref), dx=_rel(dx, x.grad), dw=_rel(dw, w.grad))
    print(e)
    assert e['y'] < 6e-3 and e['dx'] < 6e-3 and e['dw'] < 2e-3, e


def test_bn_silu_forward_backward_and_fused_silu_grad_epilogue(cuda):
    from cvpytorch_b200 import _lib, train as T
    B, H, W, C = 3, 12, 20, 128
    g = torch.Generator().manual_seed(7)
    y = _bf(torch.randn(B, C, H, W, generator=g) * 1.5 + 0.3).cuda().requires_grad_(True)
    gamma = (torch.rand(C, generator=g) + 0.5).cuda().requires_grad_(True)
    beta = (torch.randn(C, generator=g) * 0.3).cuda().requires_grad_(True)
    da = _bf(torch.randn(B, C, H, W, generator=g)).cuda()
    rm, rv = torch.zeros(C).cuda(), torch.ones(C).cuda()
    a_ref = F.silu(F.batch_norm(y, rm.clone(), rv.clone(), gamma, beta, True, 0.03, 1e-3))
    a_ref.backward(da)
    rm_ref, rv_ref = torch.zeros(C).cuda(), torch.ones(C).cuda()
    F.batch_norm(y.detach(), rm_ref, rv_ref, gamma.detach(), beta.detach(), True, 0.03, 1e-3)
    L = _lib.lib()
    yh = y.detach().permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)
    dah = da.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)
    npix = B * H * W
    stat, scratch = torch.empty(4, C, device='cuda'), torch.empty(2, C, device='cuda')
    _lib.check(L.cvb_train_bn_stats(T._p(yh), npix, C, T._p(gamma.detach()), T._p(beta.detach()), 1e-3, 0.03, T._p(rm), T._p(rv), T._p(scratch), T._p(stat), T._stream()), 'stats')
    a = torch.empty_like(yh)
    _lib.check(L.cvb_train_bn_silu_fwd(T._p(yh), npix, C, T._p(stat), T._p(a), T._stream()), 'fwd')
    sums, dy = torch.empty(2, C, device='cuda'), torch.empty_like(yh)
    _lib.check(L.cvb_train_bn_silu_bwd(T._p(dah), 0, T._p(yh), npix, C, T._p(stat), T._p(gamma.detach()), T._p(sums), T._p(dy), T._stream()), 'bwd')
    torch.cuda.synchronize()
    e = dict(a=_rel(a.float().permute(0, 3, 1, 2), a_ref), dy=_rel(dy.float().permute(0, 3, 1, 2), y.grad), dgamma=_rel(sums[1], gamma.grad), dbeta=_rel(sums[0], beta.grad),
             rm=_rel(rm, rm_ref), rv=_rel(rv, rv_ref), mean=_rel(stat[0], y.detach().mean((0, 2, 3))))
    print(e)
    assert e['a'] < 6e-3 and e['dy'] < 6e-3 and max(e['dgamma'], e['dbeta'], e['rm'], e['rv'], e['mean']) < 2e-3, e
    # the backward-data convolution with the producer's SiLU' in its epilogue == backward-data, then * silu'(z) (the separate pass)
    cout2 = 64
    w2 = _bf(torch.randn(cout2, C, 3, 3, generator=g) / (C * 9) ** 0.5).cuda()
    dy2 = _bf(torch.randn(B, H, W, cout2, generator=g)).cuda().to(torch.bfloat16)
    _, wb2 = T.pack_weights(w2)
    fused = T.conv(dy2, wb2, C, 3, y_prev=yh, stat_prev=stat).float()
    plain = T.conv(dy2, wb2, C, 3).float()
    z = yh.float() * stat[2] + stat[3]
    sg = torch.sigmoid(z)
    ref = plain * (sg * (1 + z * (1 - sg)))
    torch.cuda.synchronize()
    assert _rel(fused, ref) < 8e-3, _rel(fused, ref)  # (`plain` was rounded to bf16 before the multiplication, `fused` after)


@pytest.mark.parametrize('case', ['c3_n1', 'c3_n2'])
def test_c3_training_step_vs_reference_fixture(cuda, case):
    from cvpytorch_b200 import train as T
    from make_golden_train import case_inputs, sub
    g = np.load(os.path.join(GOLD, 'c3_train.npz'))
    cin, cout, n, B, H, W = [int(v) for v in g[f'{case}_cfg']]
    m = T.CSPLayer(cin, cout, n=n)
    keys = [str(k) for k in g[f'{case}_keys']]
    assert list(m.state_dict().keys()) == keys  # same module tree / parameter names as the reference block
    sd, x, G = case_inputs(case, m.state_dict())
    m.load_state_dict(sd)
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.eps, mod.momentum = 1e-3, 0.03
    m.cuda().train()
    x = x.cuda().requires_grad_(True)
    y = m(x)
    (y * G.cuda()).sum().backward()
    torch.cuda.synchronize()
    errs = {'y': _rel(sub(y), torch.from_numpy(g[f'{case}_y'])), 'dx': _rel(sub(x.grad), torch.from_numpy(g[f'{case}_dx']))}
    for k, p in m.named_parameters():
        assert p.grad is not None, k
        errs['grad ' + k] = _rel(sub(p.grad), torch.from_numpy(g[f'{case}_grad_{k}']))
    for k, v in m.state_dict().items():
        if 'running_' in k:
            errs['after ' + k] = _rel(v, torch.from_numpy(g[f'{case}_after_{k}']))
    print({k: round(v, 4) for k, v in errs.items()})
    assert errs['y'] < 3e-2, errs
    assert errs['dx'] < 6e-2 and max(v for k, v in errs.items() if k.startswith('grad ')) < 6e-2, errs
    assert max(v for k, v in errs.items() if k.startswith('after ')) < 1e-2, errs
    # one SGD step through the unchanged torch optimiser keeps working on the drop-in's parameters
    opt = torch.optim.SGD(m.parameters(), lr=0.01, momentum=0.9)
    opt.step()
    opt.zero_grad(set_to_none=True)
    y2 = m(x.detach())
    assert torch.isfinite(y2).all()


def test_c3_dropin_through_the_reference_trainer_train_step(cuda):
    """The drop-in block inside a copy of the reference's training-step logic (trainer.py:177-207: amp.autocast(enabled=cfg.AMP) ->
    scaler.scale(losses['loss']).backward() -> clip_grad -> scaler.step(optimizer) -> scaler.update() -> optimizer.zero_grad(set_to_none=True)),
    with unchanged torch modules before and after it: the loss goes down and every parameter of the block receives finite gradients."""
    from cvpytorch_b200 import train as T
    torch.manual_seed(3)
    stem = torch.nn.Conv2d(3, 128, 3, 2, 1).cuda()          # reference-side layer in front of the block
    block = T.CSPLayer(128, 128, n=2).cuda().train()
    head = torch.nn.Conv2d(128, 8, 1).cuda()                # reference-side layer behind it
    params = list(stem.parameters()) + list(block.parameters()) + list(head.parameters())
    optimizer = torch.optim.SGD(params, lr=0.02, momentum=0.9)
    scaler = torch.amp.GradScaler('cuda', enabled=True)
    imgs = torch.randn(4, 3, 64, 64, device='cuda')
    target = torch.randn(4, 8, 32, 32, device='cuda') * 0.1
    hist = []
    for it in range(8):
        with torch.autocast('cuda', enabled=True):           # cfg.AMP
            out = head(block(stem(imgs)))
            losses = {'loss': (out.float() - target).pow(2).mean()}
        scaler.scale(losses['loss']).backward()
        scaler.unscale_(optimizer)
        torch.nn.utils.clip_grad_norm_(params, 10.0)          # cfg.GRAD_CLIP
        if it == 0:
            for k, p in block.named_parameters():
                assert p.grad is not None and torch.isfinite(p.grad).all() and float(p.grad.abs().max()) > 0, k
        scaler.step(optimizer)
        scaler.update()
        optimizer.zero_grad(set_to_none=True)
        hist.append(float(losses['loss']))
    assert all(np.isfinite(hist)) and hist[-1] < 0.7 * hist[0], hist


@pytest.mark.parametrize('B,H,W,cin,cout', [(2, 16, 16, 64, 64), (2, 13, 9, 64, 128), (3, 26, 18, 128, 64), (1, 7, 30, 64, 128)])
def test_stride2_conv_forward_backward_data_backward_weight(cuda, B, H, W, cin, cout):
    """3x3 / stride 2 / pad 1 (the downsampling BaseConv of every dark stage): forward through four parity tensor maps, backward-data as four
    parity sub-convolutions (with and without the SiLU' epilogue), backward-weight -- vs torch on bf16-representable inputs, odd sizes included."""
    from cvpytorch_b200 import train as T
    g = torch.Generator().manual_seed(B * 31 + H + W + cin)
    x = _bf(torch.randn(B, cin, H, W, generator=g)).cuda().requires_grad_(True)
    w = _bf(torch.randn(cout, cin, 3, 3, generator=g) / (cin * 9) ** 0.5).cuda().requires_grad_(True)
    y_ref = F.conv2d(x, w, None, 2, 1)
    dy = _bf(torch.randn(y_ref.shape, generator=g)).cuda()
    y_ref.backward(dy)
    xh = x.detach().permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)
    dyh = dy.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)
    wf, wb = T.pack_weights(w.detach())
    y = T.conv(xh, wf, cout, 3, stride=2)
    assert tuple(y.shape) == (B, y_ref.shape[2], y_ref.shape[3], cout)
    dx = T.conv_dgrad_s2(dyh, wb, cin, H, W)
    dw = T.conv_wgrad(xh, dyh, 3, stride=2)
    torch.cuda.synchronize()
    e = dict(y=_rel(y.float().permute(0, 3, 1, 2), y_ref), dx=_rel(dx.float().permute(0, 3, 1, 2), x.grad), dw=_rel(dw, w.grad))
    print(e)
    assert e['y'] < 6e-3 and e['dx'] < 6e-3 and e['dw'] < 2e-3, e
    # SiLU' epilogue on the strided stores
    yp = _bf(torch.randn(B, H, W, cin, generator=g)).cuda().to(torch.bfloat16)
    stat = torch.stack([torch.zeros(cin), torch.ones(cin), torch.rand(cin, generator=g) + 0.5, torch.randn(cin, generator=g) * 0.2]).cuda().contiguous()
    fused = T.conv_dgrad_s2(dyh, wb, cin, H, W, y_prev=yp, stat_prev=stat).float()
    z = yp.float() * stat[2] + stat[3]
    sg = torch.sigmoid(z)
    torch.cuda.synchronize()
    assert _rel(fused, dx.float() * (sg * (1 + z * (1 - sg)))) < 8e-3


def test_dark_stage_training_step_vs_reference_fixture(cuda):
    """stride-2 BaseConv + CSPLayer (one `dark` stage) forward + backward vs the reference modules + torch.autograd (fixture case 'dark')."""
    from cvpytorch_b200 import train as T
    from make_golden_train import case_inputs, sub
    g = np.load(os.path.join(GOLD, 'c3_train.npz'))
    down, csp = T.BaseConv(64, 128, 3, 2), T.CSPLayer(128, 128, n=1)
    m = torch.nn.Sequential(down, csp)
    keys = [str(k) for k in g['dark_keys']]
    assert list(m.state_dict().keys()) == keys
    sd, x, G = case_inputs('dark', m.state_dict())
    m.load_state_dict(sd)
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.eps, mod.momentum = 1e-3, 0.03
    m.cuda().train()
    x = x.cuda().requires_grad_(True)
    y = csp.forward_nhwc(down(x.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16))).permute(0, 3, 1, 2).float()
    (y * G.cuda()).sum().backward()
    torch.cuda.synchronize()
    errs = {'y': _rel(sub(y), torch.from_numpy(g['dark_y'])), 'dx': _rel(sub(x.grad), torch.from_numpy(g['dark_dx']))}
    for k, p in m.named_parameters():
        errs['grad ' + k] = _rel(sub(p.grad), torch.from_numpy(g[f'dark_grad_{k}']))
    for k, v in m.state_dict().items():
        if 'running_' in k:
            errs['after ' + k] = _rel(v, torch.from_numpy(g[f'dark_after_{k}']))
    print({k: round(v, 4) for k, v in errs.items()})
    assert errs['y'] < 3e-2 and errs['dx'] < 6e-2 and max(v for k, v in errs.items() if k.startswith('grad ')) < 6e-2, errs
    assert max(v for k, v in errs.items() if k.startswith('after ')) < 1e-2, errs


@pytest.mark.parametrize('c,n,shortcut', [(256, 1, True), (512, 1, False)])
def test_wider_c3_blocks_vs_oracle(cuda, c, n, shortcut):
    """dark4 / dark5 widths (256 / 512 channels; dark5 has shortcut=False): the drop-in vs the oracle's training step (reference block restated,
    torch.autograd, fp32 on the host) on seeded parameters -- same tolerances as the fixture test."""
    from cvpytorch_b200 import train as T
    from oracle import c3_train_oracle as CO
    sd = CO.synthetic_state(c, c, n, seed=c)
    g = torch.Generator().manual_seed(c + 1)
    x = torch.randn(2, c, 10, 12, generator=g)
    G = torch.randn(2, c, 10, 12, generator=g)
    sdt = {k: torch.as_tensor(v).clone().requires_grad_(True) if (torch.as_tensor(v).dtype.is_floating_point and 'running_' not in k) else torch.as_tensor(v).clone()
           for k, v in sd.items()}
    xr = x.clone().requires_grad_(True)
    yr = CO.csp_layer(xr, sdt, n, shortcut=shortcut)
    (yr * G).sum().backward()
    m = T.CSPLayer(c, c, n=n, shortcut=shortcut)
    m.load_state_dict({k: torch.as_tensor(v) for k, v in sd.items()})
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.eps, mod.momentum = CO.BN_EPS, CO.BN_MOMENTUM
    m.cuda().train()
    xg = x.cuda().requires_grad_(True)
    y = m(xg)
    (y * G.cuda()).sum().backward()
    torch.cuda.synchronize()
    errs = {'y': _rel(y, yr), 'dx': _rel(xg.grad, xr.grad)}
    for k, p in m.named_parameters():
        errs['grad ' + k] = _rel(p.grad, sdt[k].grad)
    print({k: round(v, 4) for k, v in errs.items()})
    assert errs['y'] < 3e-2 and errs['dx'] < 6e-2 and max(v for k, v in errs.items() if k.startswith('grad ')) < 6e-2, errs
