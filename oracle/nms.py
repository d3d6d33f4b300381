"""TEST INFRASTRUCTURE ONLY - CPU restatement of the reference's rotated 3-D NMS (SURVEY.md 8(f)-4).

Follows ``rotate_nms_3d_cc`` (ops/pybind11/rbbox_iou.py:294-311): order = scores.argsort()[::-1]; corners by
``boxes3d2corners`` (:121-148); ``standup_iou`` = 3-D IoU of the axis-aligned bounding cubes (:62-96); then
``rotate_non_max_suppression_3d_cpu`` (ops/pybind11/nms_cpu.h:148-240): greedy in score order, box j is
suppressed by a kept box i when standup_iou(i, j) > 0 and the rotated 3-D IoU is >= thresh; ``keep[:top_k]``.

The rotated IoU itself is ``oracle.box_iou``, pinned to the reference's Python IoU (utils/box_util.py) for
convex, non-degenerate boxes by tests/golden/iou_ref.npz (see its header; the degenerate-ring decision documented
there applies here too).  A box with NaN geometry has NaN cube extents, fails the standup test and so is never
suppressed and suppresses nothing.  Ties in the score order: numpy's default
``argsort`` is not stable, so the reference leaves them unspecified; this restatement (and the kernel) use the
reverse of a STABLE ascending sort, i.e. among equal scores the larger index comes first."""
import numpy as np

from . import box_iou as ob


def boxes3d2corners(boxes):
    b = np.asarray(boxes, dtype=np.float64)
    return ob.box3d_corners(b[:, 0:3], b[:, 6], b[:, 3:6])      # sizes (l, w, h), same corner order


def rotate_nms_3d_cc(dets, thresh, top_k=300):
    dets = np.asarray(dets, dtype=np.float64)
    n = dets.shape[0]
    if n == 0:
        return []
    order = np.argsort(dets[:, 7], kind="stable")[::-1]
    corners = boxes3d2corners(dets)
    mn, mx = corners.min(1), corners.max(1)
    suppressed = np.zeros(n, dtype=bool)
    keep = []
    for a in range(n):
        i = order[a]
        if suppressed[i]:
            continue
        keep.append(int(i))
        # the later boxes still alive whose standup IoU with box i is > 0 (nms_cpu.h:192); a NaN extent fails
        rest = order[a + 1:]
        rest = rest[~suppressed[rest]]
        with np.errstate(invalid="ignore"):
            ext = np.minimum(mx[i], mx[rest]) - np.maximum(mn[i], mn[rest])
            rest = rest[(ext > 0).all(1)]
        for j in rest:
            iou3d = ob.rbbox_iou_3d_pair(corners[i:i + 1], corners[j:j + 1])[0, 1]
            if iou3d >= thresh:
                suppressed[j] = True
    return keep[:top_k]


def cube_overlap_pairs(dets):
    """(i, j), i < j, of the pairs whose bounding cubes overlap (the only pairs whose IoU NMS evaluates) and the
    smallest |extent| of each pair's cube intersection; NaN boxes overlap nothing."""
    c = boxes3d2corners(dets)
    mn, mx = c.min(1), c.max(1)
    i, j = np.triu_indices(len(c), 1)
    with np.errstate(invalid="ignore"):
        ext = np.minimum(mx[i], mx[j]) - np.maximum(mn[i], mn[j])
        close = np.abs(ext).min(1)
        hit = (ext > -1e-4).all(1)
    return i[hit], j[hit], close[hit], c


def pair_iou_margins(dets, thresh):
    """Per pair whose bounding cubes overlap or nearly touch: (i, j, margin), margin = the smaller of
    |IoU_3D - thresh| and |cube extent|, i.e. how far the pair is from flipping either NMS decision."""
    i, j, close, c = cube_overlap_pairs(np.asarray(dets, dtype=np.float64))
    iou = ob.rbbox_iou_3d_pair(c[i], c[j])[:, 1] if len(i) else np.zeros(0)
    return i, j, np.minimum(np.abs(iou - thresh), close)


def pair_margins(dets, thresh):
    """min over pairs of the distance to a flipped NMS decision: tests use it to skip numerically ambiguous
    inputs.  Pairs whose bounding cubes are apart by more than 1e-4 cannot flip and are not evaluated."""
    m = pair_iou_margins(dets, thresh)[2]
    return float(m.min()) if len(m) else np.inf
