"""Reference goldens on the HEADLINE data (build container only; imports /root/reference through tools/ref_shim.py):
the first 8 images of the seed-1029 640x640 batch that bench.py times, through the UNMODIFIED reference forward and the reference's own
`non_max_suppression` (+ torchvision.ops.nms) at the call-site thresholds (conf 0.001, IoU 0.6, multi_label).

Saturated sigmoids make exact score ties routine on real head outputs (image 3 keeps two candidates with score 0.9995566 whose order
depends on the reference's unstable argsort at the 30 000 cap), so the fixture stores the reference's kept rows AND their candidate ids,
and tests compare (a) the kept SET exactly and (b) the ORDER up to permutations inside groups of exactly equal scores.

Writes tests/golden/yolov5s_batch640.npz:  z_sub [8, 197, 85] (every 128th anchor row), det_i [n_i, 6], idx_i [n_i] (anchor*80+cls of each
reference row, recovered by matching the row against the reference's own candidate table), tie_groups_i = number of rows in exact-score ties.
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
N_IMG = 8


def candidate_ids_of_rows(z_img, rows, conf=0.001):
    """Recovers anchor*nc + cls of every reference-kept row: (box, score, class) identifies the candidate (first match in row-major order)."""
    x = z_img.astype(np.float32)
    nc = x.shape[1] - 5
    sel = np.nonzero(x[:, 4] > np.float32(conf))[0]
    xs = x[sel].copy()
    xs[:, 5:] *= xs[:, 4:5]
    box = NO.xywh2xyxy(xs[:, :4])
    ids = np.zeros(rows.shape[0], np.int64)
    for r, row in enumerate(rows):
        c = int(row[5])
        m = np.nonzero((xs[:, 5 + c] == row[4]) & (box == row[:4]).all(1))[0]
        assert m.size >= 1, ('reference row not found among the candidates', r, row)
        ids[r] = int(sel[m[0]]) * nc + c
    return ids


def main():
    torch.set_num_threads(8)
    bb, nk, dt, ref_nms = ref_shim.build_yolov5s()
    sd = synth.yolov5s_state_dict(calibrated=True)
    bb.load_state_dict(synth.split_prefix(sd, 'backbone.'), strict=True)
    nk.load_state_dict(synth.split_prefix(sd, 'neck.'), strict=True)
    dt.load_state_dict(synth.split_prefix(sd, 'detect.'), strict=True)
    bb.eval(); nk.eval(); dt.eval()
    torch.manual_seed(1029)  # bench.py: synthetic_frames(64, seed=1029); the first 8 images of that batch
    x = torch.randn(64, 3, 640, 640)[:N_IMG].contiguous()
    with torch.no_grad():
        z, _ = dt(list(nk(bb(x))))
    zo, _ = YO.forward(x, sd)
    print('oracle vs reference z: rel err', YO.rel_err(zo, z), 'bit-identical:', bool(torch.equal(zo, z)))
    dets = ref_nms(z.clone(), 0.001, 0.6, multi_label=True)
    odet = NO.non_max_suppression(z.numpy(), 0.001, 0.6, multi_label=True)
    out = {'z_sub': z[:, ::128].numpy()}
    for i in range(N_IMG):
        rd = dets[i].numpy()
        ids = candidate_ids_of_rows(z[i].numpy(), rd)
        od, oi = odet[i]
        same_set = set(ids.tolist()) == set(oi.tolist())
        same_order = np.array_equal(ids, oi)
        sc = rd[:, 4]
        ties = int(sum((sc == s).sum() > 1 for s in sc))
        n_cand = int(((z[i, :, 5:] * z[i, :, 4:5] > 0.001) & (z[i, :, 4:5] > 0.001)).sum())
        print(f'image {i}: kept {rd.shape[0]}, candidates {n_cand}, rows in exact-score ties {ties}, oracle set == reference: {same_set}, order identical: {same_order}')
        assert same_set
        out[f'det_{i}'] = rd
        out[f'idx_{i}'] = ids
    np.savez_compressed(os.path.join(GOLD, 'yolov5s_batch640.npz'), **out)
    print('written', os.path.join(GOLD, 'yolov5s_batch640.npz'), os.path.getsize(os.path.join(GOLD, 'yolov5s_batch640.npz')))


if __name__ == '__main__':
    main()
