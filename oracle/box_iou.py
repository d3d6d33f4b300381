"""TEST INFRASTRUCTURE ONLY - CPU restatement of the pairwise rotated-box IoU train metric (SURVEY.md 8(f)-1).

Follows `rbbox_iou_3d_pair` of the reference (ops/pybind11/box_ops.h:173-260, called from
models/det_base.py:494-503 on the corners of models/model_util.py:48-72):

  * per pair n, the bird's-eye-view polygons are the (x, z) coordinates of corners 6, 7, 4, 5 (box_ops.h:206-224;
    clockwise for boxes built by get_box3d_corners_helper, i.e. positive area in Boost's default convention);
  * `inter_area` = area of their intersection, `union_area` = area of their union (box_ops.h:226-231);
  * `ymax = min(c[0].y, q[0].y)`, `ymin = max(c[4].y, q[4].y)`, `h = c[0].y - c[4].y` (box_ops.h:233-237);
  * `inter_vol = inter_area * max(0, ymax - ymin)`, `vol = max(0, area * h)` (box_ops.h:242-245);
  * out[n] = (inter_area / union_area, inter_vol / (vol + qvol - inter_vol)); pairs without intersection keep
    the zero initialisation (box_ops.h:199,226,247-248); N != K or N == 0 returns zeros (box_ops.h:201-203).

PINNED to the reference's Python IoU for convex, non-degenerate boxes.  The reference delegates the polygon
clipping to Boost.Geometry (an unversioned system dependency, not available here), but it also ships the same
metric in pure Python, utils/box_util.py (polygon_clip + ConvexHull; models/det_base.py:28).  This file restates
the published algorithm for two CONVEX polygons (Sutherland-Hodgman clipping + shoelace area; the union of two
overlapping convex polygons is one polygon of area a + b - inter) in float64; tests/test_box_iou_cpu.py checks it
against tests/golden/iou_ref.npz, box_util's values on ~2 200 pairs in named groups written by
oracle/make_golden_iou.py (BEV to 1e-9; 3-D to 4e-6, the gap between box_util's edge-length volume and Boost's
area * height on float32 corners), and against closed-form cases and an independent point-sampling estimate.

DEGENERATE RINGS (decision of round 2, pinned by tests/test_box_iou_cpu.py::test_degenerate_boxes): the reference
appends the four BEV corners without `bg::correct` (box_ops.h:206-224).  A decoded box with exactly ONE negative
footprint size (size_decode of untrained weights can produce it) gives a counter-clockwise ring, i.e. a polygon
that violates Boost's concept (clockwise, closed); `bg::intersection`/`bg::union_` are unspecified on such
input, so there is no reference value to match.  Such a pair scores (0, 0) here and in csrc/box_iou.cuh: an
invalid box gets no overlap credit, and 0 <= IoU_3D <= IoU_2D <= 1 holds for every input.  Two negative
footprint sizes are a valid box rotated by pi (orientation preserved); a negative HEIGHT needs no special
case (`vol = max(0, area*h)`, `max(0, ymax - ymin)` already give IoU_3D = 0 with the reference's own formulas).
"""
import numpy as np

BEV_ORDER = (6, 7, 4, 5)


def _shoelace_ccw(poly):
    """Signed area, counter-clockwise positive."""
    x, y = poly[:, 0], poly[:, 1]
    return 0.5 * float(np.sum(x * np.roll(y, -1) - np.roll(x, -1) * y))


def _clip_convex(subject, clip):
    """Sutherland-Hodgman: part of `subject` inside the convex polygon `clip` (either orientation)."""
    sgn = 1.0 if _shoelace_ccw(clip) >= 0 else -1.0
    out = [tuple(p) for p in subject]
    m = len(clip)
    for i in range(m):
        if not out:
            break
        a, b = clip[i], clip[(i + 1) % m]
        ex, ey = b[0] - a[0], b[1] - a[1]
        side = lambda p: sgn * (ex * (p[1] - a[1]) - ey * (p[0] - a[0]))
        inp, out = out, []
        for j in range(len(inp)):
            p, q = inp[j], inp[(j + 1) % len(inp)]
            sp, sq = side(p), side(q)
            if sp >= 0:
                out.append(p)
            if (sp >= 0) != (sq >= 0):
                t = sp / (sp - sq)
                out.append((p[0] + t * (q[0] - p[0]), p[1] + t * (q[1] - p[1])))
    return np.asarray(out, dtype=np.float64).reshape(-1, 2)


def rbbox_iou_3d_pair(box_corners, qbox_corners):
    """(N,8,3), (N,8,3) -> (N,2) float64: [:,0] BEV IoU, [:,1] 3-D IoU (box_ops.h:173-260)."""
    c = np.asarray(box_corners, dtype=np.float64)
    q = np.asarray(qbox_corners, dtype=np.float64)
    N, K = c.shape[0], q.shape[0]
    out = np.zeros((N, 2), dtype=np.float64)
    if N == 0 or K == 0 or N != K:
        return out
    for n in range(N):
        poly = c[n][list(BEV_ORDER)][:, [0, 2]]
        qpoly = q[n][list(BEV_ORDER)][:, [0, 2]]
        area, qarea = -_shoelace_ccw(poly), -_shoelace_ccw(qpoly)   # Boost: clockwise positive
        if not (area > 0.0 and qarea > 0.0):
            continue   # DEGENERATE RING (see the header): pinned decision, the pair scores (0, 0)
        inter = _clip_convex(poly, qpoly)
        inter_area = abs(_shoelace_ccw(inter)) if len(inter) >= 3 else 0.0
        if inter_area <= 0.0:
            continue
        union_area = area + qarea - inter_area
        ymax = min(c[n, 0, 1], q[n, 0, 1])
        ymin = max(c[n, 4, 1], q[n, 4, 1])
        h, qh = c[n, 0, 1] - c[n, 4, 1], q[n, 0, 1] - q[n, 4, 1]
        inter_vol = inter_area * max(0.0, ymax - ymin)
        vol, qvol = max(0.0, area * h), max(0.0, qarea * qh)
        out[n, 0] = inter_area / union_area
        out[n, 1] = inter_vol / (vol + qvol - inter_vol)
    return out


def box3d_corners(centers, headings, sizes):
    """numpy restatement of get_box3d_corners_helper (models/model_util.py:48-72): (N,3),(N,),(N,3) -> (N,8,3)."""
    centers = np.asarray(centers, dtype=np.float64)
    headings = np.asarray(headings, dtype=np.float64)
    sizes = np.asarray(sizes, dtype=np.float64)
    l, w, h = sizes[:, 0], sizes[:, 1], sizes[:, 2]
    xs = np.stack([l / 2, l / 2, -l / 2, -l / 2, l / 2, l / 2, -l / 2, -l / 2], 1)
    ys = np.stack([h / 2, h / 2, h / 2, h / 2, -h / 2, -h / 2, -h / 2, -h / 2], 1)
    zs = np.stack([w / 2, -w / 2, -w / 2, w / 2, w / 2, -w / 2, -w / 2, w / 2], 1)
    cs, sn = np.cos(headings)[:, None], np.sin(headings)[:, None]
    x = cs * xs + sn * zs + centers[:, 0:1]
    y = ys + centers[:, 1:2]
    z = -sn * xs + cs * zs + centers[:, 2:3]
    return np.stack([x, y, z], 2)
