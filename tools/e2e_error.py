"""Prints the end-to-end decoded-output error of the YOLOv5-s graph vs the reference goldens (128x128 and 640x640)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
from cvpytorch_b200 import synth
m = synth.build_yolov5s(True)
rel = lambda a, b: float((a.double().cpu() - torch.as_tensor(b).double()).abs().max() / (np.abs(b).max() + 1e-12))
g = np.load(os.path.join(ROOT, 'tests/golden/yolov5s_fwd128.npz'))
torch.manual_seed(1029); x = torch.randn(2, 3, 128, 128).cuda()
m.predict(x); e128 = rel(m._graph_for(x)['z'][:, ::3], g['z'])
g = np.load(os.path.join(ROOT, 'tests/golden/yolov5s_fwd640.npz'))
torch.manual_seed(1029); x = torch.randn(1, 3, 640, 640).cuda()
m.predict(x); e640 = rel(m._graph_for(x)['z'][0, ::16], g['z_sub'])
print(f'CVB_MAX_CHAIN={os.environ.get("CVB_MAX_CHAIN", "160(default)")}: decoded z rel err vs reference golden: 128x128 {e128:.2e}, 640x640 {e640:.2e}')
