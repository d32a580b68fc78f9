"""tests/golden/yolo_blocks.npz: the REFERENCE's YOLOv6 / YOLOv7 blocks (src/models/modules/yolo_modules.py: RepVGGBlock :268, BepC3 :427,
EELAN :565) run on CPU in the build container (tools/ref_shim.py), with seeded weights and BN statistics, in eval mode; the drop-in
mirrors (cvpytorch_b200/yolo_blocks.py) load the SAME state_dict (the key lists must be equal) and must reproduce the outputs.

To keep the file small, the parameters and inputs are not stored: tests regenerate them bit for bit from the seeds in CASES (case_inputs),
and the outputs are stored as every 3rd channel."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
import ref_shim  # noqa: E402


# case -> (input channels, seed offset)
CASES = {'rep_id': (32, 0), 'rep_s2': (32, 1), 'rep_deploy': (32, 2), 'bepc3': (64, 3), 'eelan': (64, 4)}


def seeded_state(template, seed):
    """Seeded weights and BN statistics in state_dict (= module) order: conv weight ~ N(0, 1.6^2 / fan_in), conv bias ~ N(0, 0.1^2), BN weight
    ~ U(0.5, 1.5), bias ~ N(0, 0.2^2), running mean ~ N(0, 0.3^2), running var ~ U(0.5, 1.5); then every shortcut weight `alpha` ~
    U(0.5, 1.5).  Other buffers keep the template's values."""
    g = torch.Generator().manual_seed(seed)
    is_conv = {k.rpartition('.')[0]: v.dim() == 4 for k, v in template.items() if k.endswith('.weight')}
    sd = {}
    for k, v in template.items():
        mod, _, name = k.rpartition('.')
        conv = is_conv.get(mod)
        if conv and name == 'weight':
            sd[k] = torch.randn(v.shape, generator=g) * (1.6 / v[0].numel() ** 0.5)
        elif conv and name == 'bias':
            sd[k] = torch.randn(v.shape, generator=g) * 0.1
        elif conv is False and name in ('weight', 'running_var'):
            sd[k] = torch.rand(v.shape, generator=g) + 0.5
        elif conv is False and name == 'bias':
            sd[k] = torch.randn(v.shape, generator=g) * 0.2
        elif conv is False and name == 'running_mean':
            sd[k] = torch.randn(v.shape, generator=g) * 0.3
        else:
            sd[k] = v.clone()
    for k in sd:
        if k.endswith('alpha'):
            sd[k] = torch.rand(1, generator=g) + 0.5
    return sd


def case_inputs(name, template):
    """(state_dict, x) of a fixture case; template: a state_dict with the reference block's keys and shapes."""
    cin, i = CASES[name]
    return seeded_state(template, 200 + i), torch.randn(2, cin, 24, 40, generator=torch.Generator().manual_seed(300 + i))


def main():
    ref_shim.install()
    from src.models.modules import yolo_modules as YM
    out = {}
    ctors = {'rep_id': lambda: YM.RepVGGBlock(32, 32), 'rep_s2': lambda: YM.RepVGGBlock(32, 64, stride=2), 'rep_deploy': lambda: YM.RepVGGBlock(32, 32),
             'bepc3': lambda: YM.BepC3(64, 64, n=4), 'eelan': lambda: YM.EELAN(64, 32, 128)}
    for name, ctor in ctors.items():
        m = ctor()
        sd, x = case_inputs(name, m.state_dict())
        m.load_state_dict(sd)
        m.eval()
        with torch.no_grad():
            y = m(x)
            # 'rep_deploy': the reference's own switch_to_deploy() raises (its _fuse_bn_tensor :338-352 tests isinstance(branch, nn.Sequential)
            # but the branches are ConvModules), so the deployed form has no runnable reference; the fixture keeps the training-form
            # output and the test checks that the mirror's re-parameterised single conv reproduces it
        out[f'{name}_keys'] = np.array(list(sd.keys()))
        out[f'{name}_y'] = y.numpy()[:, ::3]
        print(name, 'in', tuple(x.shape), 'out', tuple(y.shape), 'keys', len(sd), 'out std', float(y.std()))
    np.savez_compressed(os.path.join(ROOT, 'tests/golden/yolo_blocks.npz'), **out)
    print('wrote tests/golden/yolo_blocks.npz', os.path.getsize(os.path.join(ROOT, 'tests/golden/yolo_blocks.npz')))


if __name__ == '__main__':
    main()
