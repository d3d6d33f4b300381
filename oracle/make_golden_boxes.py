"""ORACLE (test infrastructure) - fixture for the rotated-box IoU row (SURVEY.md 8(f)-1).

Runs the UNMODIFIED reference `get_box3d_corners_helper` (models/model_util.py:48-72) on seeded box pairs
(prediction = perturbed ground truth, the situation of models/det_base.py:488-495) and stores inputs + corners
as tests/golden/box_pairs.npz.  The IoU values themselves cannot come from the reference here (Boost.Geometry
is absent; oracle/make_golden_iou.py takes them from the reference's Python IoU instead); the fixture pins the
corner convention the IoU consumes.

    python -m oracle.make_golden_boxes          # authoring container only (needs /root/reference)
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_import  # noqa: E402


def make_pairs(M=256, seed=31):
    rng = np.random.default_rng(seed)
    ctr = np.stack([rng.uniform(-20, 20, M), rng.uniform(0.5, 2.0, M), rng.uniform(5, 60, M)], 1)
    size = np.stack([rng.uniform(3.0, 5.0, M), rng.uniform(1.4, 2.0, M), rng.uniform(1.3, 1.9, M)], 1)
    head = rng.uniform(-np.pi, np.pi, M)
    # predictions: from near-perfect to disjoint
    scale = rng.choice([0.02, 0.2, 1.0, 4.0], M)[:, None]
    pctr = ctr + rng.standard_normal((M, 3)) * scale * np.array([1.0, 0.3, 1.0])
    psize = size * np.exp(rng.standard_normal((M, 3)) * 0.1 * np.minimum(scale, 1.0))
    phead = head + rng.standard_normal(M) * 0.3 * np.minimum(scale[:, 0], 1.0)
    # exact special cases up front: identical boxes, pure translation, 90 degree turn, far apart
    pctr[0], psize[0], phead[0] = ctr[0], size[0], head[0]
    pctr[1], psize[1], phead[1] = ctr[1] + np.array([0.5, 0.0, 0.0]), size[1], head[1]
    pctr[2], psize[2], phead[2] = ctr[2], size[2], head[2] + np.pi / 2
    pctr[3], psize[3], phead[3] = ctr[3] + np.array([100.0, 0.0, 0.0]), size[3], head[3]
    f = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    return f(ctr), f(head), f(size), f(pctr), f(phead), f(psize)


if __name__ == "__main__":
    assert ref_import.reference_available(), "needs /root/reference (authoring container only)"
    ref_import._install_shims()
    from models.model_util import get_box3d_corners_helper
    ctr, head, size, pctr, phead, psize = make_pairs()
    t = torch.from_numpy
    gt = get_box3d_corners_helper(t(ctr), t(head), t(size)).numpy()
    pr = get_box3d_corners_helper(t(pctr), t(phead), t(psize)).numpy()
    path = os.path.join(ROOT, "tests", "golden", "box_pairs.npz")
    np.savez_compressed(path, gt_center=ctr, gt_heading=head, gt_size=size, pr_center=pctr, pr_heading=phead,
                        pr_size=psize, gt_corners=gt, pr_corners=pr)
    print(path, "%.1f KB" % (os.path.getsize(path) / 1024))
