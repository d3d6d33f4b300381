"""ORACLE (test infrastructure) - reference IoU fixture for the rotated-box IoU row (SURVEY.md 8(f)-1) and, through
it, the 3-D NMS (f-4).

The reference computes the train metric with Boost.Geometry (ops/pybind11/box_ops.h:173-260), which is not
available here, but it also ships the same metric in pure Python: utils/box_util.py (`polygon_clip`,
`box3d_iou`, `box3d_iou_pair`; models/det_base.py:28 names it as the alternative).  This script imports that
UNMODIFIED file from the reference checkout and writes tests/golden/iou_ref.npz:

    pr_corners, gt_corners   (n, 8, 3) float32   corners of get_box3d_corners_helper (oracle.box_iou.box3d_corners)
    iou                      (n, 2)    float64   box_util.box3d_iou_pair on those float32 corners: [BEV, 3-D]
    group                    (n,)      int32     index into group_names
    group_names, excluded_reasons, excluded_counts

Inputs: the pairs of tests/golden/box_pairs.npz plus seeded valid pairs in named groups.  Pairs where box_util is
not a valid reference are left out and counted per reason:
  * `touching_edges`: an edge of one footprint lies on the line of an edge of the other (coincident or collinear
    edges): the strict `>` inside test and the 1/(...) line intersection of polygon_clip break down there (two
    coincident boxes give 0.935 instead of 1);
  * `hull_error`: scipy's ConvexHull raises on the clipped polygon (fewer than 3 points, or all collinear).

    python -m oracle.make_golden_iou          # needs the reference checkout; rerunning reproduces the file
"""
import importlib.util
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import box_iou as ob  # noqa: E402
from oracle import ref_import  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "iou_ref.npz")
GROUPS = ("box_pairs", "translation", "rotation_0", "rotation_half_pi", "rotation_pi", "inside", "tiny", "large",
          "far", "heights_disjoint", "heights_partial", "near_miss")
PER_GROUP = 180


def _car(rng, m, scale=1.0):
    ctr = np.stack([rng.uniform(-20, 20, m), rng.uniform(0.5, 2.0, m), rng.uniform(5, 60, m)], 1)
    size = np.stack([rng.uniform(3.0, 5.0, m), rng.uniform(1.4, 2.0, m), rng.uniform(1.3, 1.9, m)], 1) * scale
    return ctr, rng.uniform(-np.pi, np.pi, m), size


def make_group(name, rng, m=PER_GROUP):
    """(ctr, head, size) of the box and of its partner for one group."""
    ctr, head, size = _car(rng, m)
    pc, ph, ps = ctr.copy(), head.copy(), size * np.exp(rng.normal(0, 0.1, (m, 3)))
    if name == "translation":                       # same heading, shifted in the ground plane and in height
        ps = size.copy()
        pc = ctr + rng.normal(0, 1.0, (m, 3)) * [1.0, 0.2, 1.0]
    elif name.startswith("rotation"):               # same centre, heading differences near 0, pi/2, pi
        base = {"rotation_0": 0.0, "rotation_half_pi": np.pi / 2, "rotation_pi": np.pi}[name]
        ph = head + base + rng.choice([-1, 1], m) * rng.uniform(1e-3, 0.2, m)
        pc = ctr + rng.normal(0, 0.2, (m, 3)) * [1.0, 0.1, 1.0]
    elif name == "inside":                          # the partner lies fully inside the box (BEV and height)
        ps = size * rng.uniform(0.2, 0.6, (m, 3))
        ph = head + rng.uniform(-np.pi, np.pi, m)
        pc = ctr + rng.uniform(-0.1, 0.1, (m, 3)) * size
    elif name in ("tiny", "large"):                 # 0.1 m and 20 m boxes, relative overlap as for cars
        s = 0.1 if name == "tiny" else 20.0
        if name == "tiny":                          # near the origin, where fp32 resolves a 0.1 m box to ~1e-6
            ctr = rng.uniform(-1.0, 1.0, (m, 3))
        size = np.full((m, 3), s) * rng.uniform(0.8, 1.2, (m, 3))
        ps = size * np.exp(rng.normal(0, 0.1, (m, 3)))
        pc = ctr + rng.normal(0, 0.3 * s, (m, 3)) * [1.0, 0.3, 1.0]
        ph = head + rng.normal(0, 0.3, m)
    elif name == "far":                             # z ~ 70 m: fp32 corners there carry ~4e-6 m of rounding
        ctr[:, 2] = rng.uniform(65, 75, m)
        pc = ctr + rng.normal(0, 0.5, (m, 3)) * [1.0, 0.2, 1.0]
        ph = head + rng.normal(0, 0.2, m)
    elif name in ("heights_disjoint", "heights_partial"):
        pc = ctr + rng.normal(0, 0.5, (m, 3)) * [1.0, 0.0, 1.0]
        ph = head + rng.normal(0, 0.2, m)
        hh = (size[:, 2] + ps[:, 2]) / 2
        f = rng.uniform(1.05, 2.0, m) if name == "heights_disjoint" else rng.uniform(0.1, 0.9, m)
        pc[:, 1] = ctr[:, 1] + rng.choice([-1, 1], m) * hh * f
    elif name == "near_miss":                       # footprints just apart or just overlapping along the length
        ph = head + rng.choice([-1, 1], m) * rng.uniform(0.01, 0.05, m)
        gap = rng.choice([-1, 1], m) * rng.uniform(1e-3, 0.05, m)
        along = (size[:, 0] + ps[:, 0]) / 2 + gap
        pc = ctr + np.stack([np.cos(head) * along, np.zeros(m), -np.sin(head) * along], 1)
    else:
        raise ValueError(name)
    return (ctr, head, size), (pc, ph, ps)


def _bev_ccw(c):
    """the reference's footprint ring: corners 3, 2, 1, 0 in (x, z) (box_util.box3d_iou)"""
    return [(c[i, 0], c[i, 2]) for i in range(3, -1, -1)]


def touching_edges(c1, c2, tol=1e-6):
    """an edge of one footprint lies on the line of an edge of the other (parallel and at distance <= tol *
    the larger box extent)"""
    p, q = np.array(_bev_ccw(c1)), np.array(_bev_ccw(c2))
    scale = max(np.ptp(p, 0).max(), np.ptp(q, 0).max())
    for a in range(4):
        u0, u1 = p[a], p[(a + 1) % 4]
        du = u1 - u0
        nu = np.hypot(*du)
        for b in range(4):
            v0, v1 = q[b], q[(b + 1) % 4]
            dv = v1 - v0
            par = abs(du[0] * dv[1] - du[1] * dv[0]) / (nu * np.hypot(*dv))
            dist = abs(du[0] * (v0[1] - u0[1]) - du[1] * (v0[0] - u0[0])) / nu
            if par <= tol and dist <= tol * scale:
                return True
    return False


def build(box_util):
    rng = np.random.default_rng(2024)
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "box_pairs.npz")))
    prs, gts, groups = [g["pr_corners"]], [g["gt_corners"]], [np.zeros(len(g["gt_corners"]), np.int32)]
    for k, name in enumerate(GROUPS[1:], 1):
        (c, h, s), (pc, ph, ps) = make_group(name, rng)
        gts.append(ob.box3d_corners(c, h, s).astype(np.float32))
        prs.append(ob.box3d_corners(pc, ph, ps).astype(np.float32))
        groups.append(np.full(len(c), k, np.int32))
    pr, gt, group = np.concatenate(prs), np.concatenate(gts), np.concatenate(groups)
    reasons = ("touching_edges", "hull_error")
    excluded = np.zeros(len(reasons), np.int64)
    keep, ious = [], []
    for n in range(len(pr)):
        c1, c2 = pr[n].astype(np.float64), gt[n].astype(np.float64)
        if touching_edges(c1, c2):
            excluded[0] += 1
            continue
        try:
            iou = box_util.box3d_iou_pair(c1[None], c2[None])[0]
        except Exception as e:                       # scipy.spatial.QhullError (a ValueError subclass)
            if "Qhull" not in type(e).__name__ and "QH" not in str(e):
                raise
            excluded[1] += 1
            continue
        keep.append(n)
        ious.append(iou)
    keep = np.asarray(keep)
    return dict(pr_corners=pr[keep], gt_corners=gt[keep], iou=np.asarray(ious, np.float64),
                group=group[keep], group_names=np.array(GROUPS), excluded_reasons=np.array(reasons),
                excluded_counts=excluded)


def load_box_util():
    path = os.path.join(ref_import.REF, "utils", "box_util.py")
    spec = importlib.util.spec_from_file_location("reference_box_util", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    assert ref_import.reference_available(), "needs the reference checkout"
    out = build(load_box_util())
    np.savez_compressed(OUT, **out)
    print(OUT, "%d pairs, %.1f KB; excluded %s" % (len(out["iou"]), os.path.getsize(OUT) / 1024,
                                                   dict(zip(out["excluded_reasons"], out["excluded_counts"]))))
