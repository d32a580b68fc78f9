"""tests/golden/c3_train.npz: the REFERENCE's CSPLayer (src/models/modules/yolox_modules.py:99-129: BaseConv = Conv2d -> BatchNorm2d -> SiLU,
Bottleneck, C3) in TRAINING mode on CPU in fp32, forward AND backward through torch.autograd (what trainer.py:177-207 runs): seeded weights,
loss = sum(out * G) with a fixed random G.  Stored: the state_dict (key list + tensors), input, output, d(loss)/d(input), every parameter
gradient and the BatchNorm running statistics after the step.  The B200 training drop-in (cvpytorch_b200/train.py) loads the SAME state_dict
and must reproduce them at the bf16 tolerance the GPU test states.

To keep the file small, the parameters, the input and G are not stored: tests regenerate them bit for bit from the seeds in CASES
(case_inputs), and every 4-D output (y, d/dx, conv weight gradients) is stored as every 7th channel (sub)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
import ref_shim  # noqa: E402


# case -> (cin, cout, n, B, H, W), stride of the first conv, seeds of (parameters, input, G)
CASES = {'c3_n1': ((128, 128, 1, 2, 16, 16), 1, (20, 30, 40)),
         'c3_n2': ((128, 128, 2, 3, 20, 20), 1, (21, 31, 41)),
         'dark': ((64, 128, 1, 2, 26, 18), 2, (78, 79, 80))}


def seeded_state(template, seed):
    """Seeded parameters in state_dict (= module) order: conv weight ~ N(0, 1.4^2 / fan_in), BatchNorm weight ~ U(0.5, 1.5), bias ~
    N(0, 0.3^2); buffers keep the template's values (fresh BatchNorm statistics)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, v in template.items():
        if k.endswith('conv.weight'):
            sd[k] = torch.randn(v.shape, generator=g) * (1.4 / v[0].numel() ** 0.5)
        elif k.endswith('bn.weight'):
            sd[k] = torch.rand(v.shape, generator=g) + 0.5
        elif k.endswith('bn.bias'):
            sd[k] = torch.randn(v.shape, generator=g) * 0.3
        else:
            sd[k] = v.clone()
    return sd


def case_inputs(case, template):
    """(state_dict, x, G) of a fixture case; template: a state_dict with the reference block's keys and shapes."""
    (cin, cout, n, B, H, W), s, (s_sd, s_x, s_G) = CASES[case]
    x = torch.randn(B, cin, H, W, generator=torch.Generator().manual_seed(s_x))
    G = torch.randn(B, cout, (H - 1) // s + 1, (W - 1) // s + 1, generator=torch.Generator().manual_seed(s_G))
    return seeded_state(template, s_sd), x, G


def sub(a):
    """The stored part of an output: every 7th channel of a 4-D tensor, all of a vector."""
    return a[:, ::7] if a.ndim == 4 else a


def run_case(name, m, out):
    sd, x, G = case_inputs(name, m.state_dict())
    m.load_state_dict(sd)
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.eps = 1e-3       # src/models/yolox.py init_params sets eps / momentum of every BN
            mod.momentum = 0.03
    m.train()
    x.requires_grad_(True)
    y = m(x)
    (y * G).sum().backward()
    out[f'{name}_cfg'] = np.array(CASES[name][0])
    out[f'{name}_keys'] = np.array(list(sd.keys()))
    out[f'{name}_y'] = sub(y.detach().numpy())
    out[f'{name}_dx'] = sub(x.grad.numpy())
    for k, p in m.named_parameters():
        out[f'{name}_grad_{k}'] = sub(p.grad.numpy())
    for k, v in m.state_dict().items():
        if 'running_' in k:
            out[f'{name}_after_{k}'] = v.numpy()
    print(name, 'x', tuple(x.shape), 'y', tuple(y.shape), 'y std', float(y.std()), 'dx std', float(x.grad.std()))


def main():
    ref_shim.install()
    from src.models.modules.yolox_modules import BaseConv, CSPLayer
    out = {}
    for name in ('c3_n1', 'c3_n2'):
        cin, cout, n = CASES[name][0][:3]
        run_case(name, CSPLayer(cin, cout, n=n), out)
    # one `dark` stage: stride-2 BaseConv in front of a CSPLayer (the structure of every stage of src/models/backbones/det/csp_darknet.py:57-91),
    # odd map sizes (26x18 -> 13x9) so that the stride-2 parity classes are ragged
    run_case('dark', torch.nn.Sequential(BaseConv(64, 128, 3, 2), CSPLayer(128, 128, n=1)), out)
    np.savez_compressed(os.path.join(ROOT, 'tests/golden/c3_train.npz'), **out)


if __name__ == '__main__':
    main()
