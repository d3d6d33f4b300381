"""Rotated 3-D NMS row (SURVEY.md 8(f)-4) on the CPU: known answers for the oracle restatement of
rotate_nms_3d_cc (ops/pybind11/rbbox_iou.py:294-311, nms_cpu.h:148-240)."""
import numpy as np

from oracle import nms as onms


def _det(cx, cz, l, w, h, ry, score, cy=1.0):
    return [cx, cy, cz, l, w, h, ry, score]


def test_known_answers():
    # three identical boxes: only the best-scored survives; a far box is untouched
    d = np.array([_det(0, 10, 4, 2, 1.5, 0.1, 0.5), _det(0, 10, 4, 2, 1.5, 0.1, 0.9), _det(0, 10, 4, 2, 1.5, 0.1, 0.7),
                  _det(30, 40, 4, 2, 1.5, 0.3, 0.2)])
    assert onms.rotate_nms_3d_cc(d, 0.5) == [1, 3]
    # shifted by half a length: 3-D IoU = 1/3 -> kept at thresh 0.5, suppressed at thresh 0.3
    d = np.array([_det(0, 10, 4, 2, 1.5, 0.0, 0.9), _det(2, 10, 4, 2, 1.5, 0.0, 0.8)])
    assert onms.rotate_nms_3d_cc(d, 0.5) == [0, 1]
    assert onms.rotate_nms_3d_cc(d, 0.3) == [0]
    # no height overlap: BEV identical but 3-D IoU 0
    d = np.array([_det(0, 10, 4, 2, 1.5, 0.0, 0.9, cy=0.0), _det(0, 10, 4, 2, 1.5, 0.0, 0.8, cy=5.0)])
    assert onms.rotate_nms_3d_cc(d, 0.1) == [0, 1]
    # chain: A suppresses B, B would suppress C but is gone -> C survives (greedy semantics)
    d = np.array([_det(0.0, 10, 4, 2, 1.5, 0.0, 0.9), _det(1.2, 10, 4, 2, 1.5, 0.0, 0.8), _det(2.4, 10, 4, 2, 1.5, 0.0, 0.7)])
    assert onms.rotate_nms_3d_cc(d, 0.5) == [0, 2]
    # top_k, empty, ties (larger index first among equal scores)
    assert onms.rotate_nms_3d_cc(d, 0.5, top_k=1) == [0]
    assert onms.rotate_nms_3d_cc(np.zeros((0, 8)), 0.5) == []
    d = np.array([_det(0, 10, 4, 2, 1.5, 0.0, 0.5), _det(50, 10, 4, 2, 1.5, 0.0, 0.5)])
    assert onms.rotate_nms_3d_cc(d, 0.5) == [1, 0]


def test_order_and_subset_properties():
    rng = np.random.default_rng(3)
    for _ in range(5):
        n = 40
        d = np.concatenate([rng.normal([0, 1, 20], [3, 0.2, 3], (n, 3)), rng.uniform([3, 1.4, 1.3], [4.5, 1.9, 1.8], (n, 3)),
                            rng.uniform(-np.pi, np.pi, (n, 1)), rng.random((n, 1))], 1)
        keep = onms.rotate_nms_3d_cc(d, 0.25)
        assert len(set(keep)) == len(keep) and keep[0] == int(np.argmax(d[:, 7]))
        assert all(d[keep[i], 7] >= d[keep[i + 1], 7] for i in range(len(keep) - 1))
        # no two kept boxes overlap above the threshold
        c = onms.boxes3d2corners(d)
        from oracle import box_iou as ob
        for a in range(len(keep)):
            for b in range(a + 1, len(keep)):
                assert ob.rbbox_iou_3d_pair(c[keep[a]:keep[a] + 1], c[keep[b]:keep[b] + 1])[0, 1] < 0.25


ORDER_HARNESS = r'''
#include "%s"
extern "C" void host_nms_ranks(int n, const float* s, int* rank) {
    for (int i = 0; i < n; ++i) {
        int r = 0;
        for (int j = 0; j < n; ++j) r += fcn::nms_ranks_above(s[j], j, s[i], i) ? 1 : 0;
        rank[i] = r;
    }
}
extern "C" void host_nms_cubes(int n, const float* corners, float* cubes, int* overlap) {
    for (int i = 0; i < n; ++i) fcn::nms_bounding_cube(corners + 24 * i, cubes + 6 * i);
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) overlap[i * n + j] = fcn::nms_cubes_overlap(cubes + 6 * i, cubes + 6 * j);
}
'''


def _order_lib(tmp_path):
    import ctypes
    import os
    import subprocess
    hdr = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "frustum_convnet_b200", "csrc",
                       "nms_order.cuh")
    src = tmp_path / "order.cpp"
    src.write_text(ORDER_HARNESS % hdr)
    so = tmp_path / "liborder.so"
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-ffp-contract=off", "-o", str(so), str(src)])
    return ctypes.CDLL(str(so))


def _host_ranks(lib, s):
    import ctypes
    s = np.ascontiguousarray(s, dtype=np.float32)
    rank = np.full(len(s), -1, dtype=np.int32)
    lib.host_nms_ranks(ctypes.c_int(len(s)), ctypes.c_void_p(s.ctypes.data), ctypes.c_void_p(rank.ctypes.data))
    return rank


def test_device_score_order_is_a_permutation_matching_numpy(tmp_path):
    """csrc/nms_order.cuh (the rank comparison both NMS kernels use) compiled with g++: on NaN, +-inf, +-0 and long
    runs of ties the ranks form a permutation equal to np.argsort(kind="stable")[::-1], the oracle's order."""
    lib = _order_lib(tmp_path)
    nan, inf = np.float32(np.nan), np.float32(np.inf)
    rng = np.random.default_rng(17)
    cases = [
        np.array([0.5, nan, 0.5, -inf, inf, 0.0, -0.0, nan, 0.5, inf], np.float32),
        np.full(40, 0.25, np.float32),                                        # > 16 tied scores
        np.array([-0.0, 0.0, -0.0, 0.0, 0.0, -0.0] * 4, np.float32),          # -0.0 == +0.0: ties
        np.full(7, nan, np.float32),
        np.array([1.0], np.float32),
        rng.choice(np.float32([nan, inf, -inf, 0.0, -0.0, 0.3, 0.7, 1e-30, -1e30]), 600),
        rng.random(700).astype(np.float32),
    ]
    s = rng.random(2000).astype(np.float32)
    s[rng.choice(2000, 600, replace=False)] = 0.5                             # 600 equal scores
    s[rng.choice(2000, 50, replace=False)] = nan
    cases.append(s)
    for s in cases:
        rank = _host_ranks(lib, s)
        assert sorted(rank.tolist()) == list(range(len(s))), s              # a permutation of 0..n-1
        want = np.empty(len(s), np.int64)
        want[np.argsort(s, kind="stable")[::-1]] = np.arange(len(s))
        assert (rank == want).all(), (s, rank, want)
    # NaN first, then +inf; among the tied 0.5 scores the larger index first
    r = _host_ranks(lib, cases[0])
    assert r[7] == 0 and r[1] == 1 and r[9] == 2 and r[4] == 3 and r[8] < r[2] < r[0]


def test_bounding_cube_rule_for_nan_boxes(tmp_path):
    """A box with NaN geometry gets an empty bounding cube, so it overlaps nothing (the oracle's NaN extent fails
    its `> 0` test too); finite boxes overlap exactly when the oracle's cube extents are all positive."""
    import ctypes
    lib = _order_lib(tmp_path)
    rng = np.random.default_rng(19)
    n = 60
    d = np.concatenate([rng.normal([0, 1, 20], [3, 0.2, 3], (n, 3)), rng.uniform([3, 1.4, 1.3], [4.5, 1.9, 1.8], (n, 3)),
                        rng.uniform(-np.pi, np.pi, (n, 1)), rng.random((n, 1))], 1).astype(np.float32)
    d[[3, 17], 0] = np.nan
    d[29, 6] = np.nan
    c = np.ascontiguousarray(onms.boxes3d2corners(d), dtype=np.float32)
    cubes = np.zeros((n, 6), np.float32)
    ov = np.zeros((n, n), np.int32)
    lib.host_nms_cubes(ctypes.c_int(n), ctypes.c_void_p(c.ctypes.data), ctypes.c_void_p(cubes.ctypes.data),
                       ctypes.c_void_p(ov.ctypes.data))
    c64 = c.astype(np.float64)
    mn, mx = c64.min(1), c64.max(1)
    ext = np.minimum(mx[:, None], mx[None]) - np.maximum(mn[:, None], mn[None])
    with np.errstate(invalid="ignore"):
        want = (ext > 0).all(-1)
    assert (ov.astype(bool) == want).all()
    for i in (3, 17, 29):
        assert not ov[i].any() and not ov[:, i].any()
    assert want.sum() > 2 * n                                               # the finite boxes do overlap
    # the oracle keeps every NaN-geometry box and never lets one suppress another
    keep = onms.rotate_nms_3d_cc(d, 0.1, top_k=n)
    assert {3, 17, 29} <= set(keep)
