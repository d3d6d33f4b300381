"""Rotated-box IoU row (SURVEY.md 8(f)-1) on the CPU: the oracle against closed forms, an independent sampling
estimate, the reference-generated corner fixture and the reference's own Python IoU (utils/box_util.py, held in
tests/golden/iou_ref.npz: the oracle is pinned to it for convex, non-degenerate boxes); and the DEVICE
arithmetic (csrc/box_iou.cuh, the very functions the CUDA kernel calls) compiled for the host with g++ against
the oracle and the reference values."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import box_iou as ob

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _pairs():
    return dict(np.load(os.path.join(ROOT, "tests", "golden", "box_pairs.npz")))


def _boxes(ctr, head, size):
    return ob.box3d_corners(np.asarray(ctr, float), np.asarray(head, float), np.asarray(size, float))


def test_corner_restatement_matches_reference_fixture():
    g = _pairs()
    for p in ("gt", "pr"):
        mine = ob.box3d_corners(g[p + "_center"], g[p + "_heading"], g[p + "_size"])
        assert np.abs(mine - g[p + "_corners"]).max() <= 2e-5      # fp32 reference vs float64 restatement
    # bird's-eye-view polygon (corners 6,7,4,5) is clockwise == positive area in Boost's convention
    poly = g["gt_corners"][:, list(ob.BEV_ORDER)][:, :, [0, 2]].astype(np.float64)
    area = np.array([-ob._shoelace_ccw(p) for p in poly])
    assert np.allclose(area, g["gt_size"][:, 0] * g["gt_size"][:, 1], rtol=1e-4)


def test_oracle_closed_forms():
    size = np.array([[4.0, 2.0, 1.5]])
    base = _boxes([[1.0, 1.0, 10.0]], [0.0], size)
    iou = lambda q: ob.rbbox_iou_3d_pair(base, q)[0]
    assert np.allclose(iou(base), [1.0, 1.0])
    assert np.allclose(iou(_boxes([[2.0, 1.0, 10.0]], [0.0], size)), [0.6, 0.6])             # 6 / (16 - 6)
    assert np.allclose(iou(_boxes([[2.0, 1.5, 10.0]], [0.0], size)), [0.6, 6.0 / 18.0])       # heights overlap 1.0
    assert np.allclose(iou(_boxes([[1.0, 1.0, 10.0]], [np.pi / 2], size)), [1 / 3, 1 / 3])    # 4 / (16 - 4)
    assert np.allclose(iou(_boxes([[9.0, 1.0, 10.0]], [0.0], size)), [0.0, 0.0])
    assert np.allclose(iou(_boxes([[1.0, 4.0, 10.0]], [0.0], size)), [1.0, 0.0])              # no height overlap
    sq = np.array([[2.0, 2.0, 1.0]])
    a = _boxes([[0.0, 0.0, 5.0]], [0.0], sq)
    b = _boxes([[0.0, 0.0, 5.0]], [np.pi / 4], sq)
    oct_area = 8.0 * (np.sqrt(2.0) - 1.0)
    assert np.allclose(ob.rbbox_iou_3d_pair(a, b)[0, 0], oct_area / (8.0 - oct_area))
    # size mismatch / empty input return zeros (box_ops.h:201-203)
    assert ob.rbbox_iou_3d_pair(base, np.zeros((0, 8, 3))).shape == (1, 2)
    assert not ob.rbbox_iou_3d_pair(np.concatenate([base, base]), base).any()


def _inside(poly, pts):
    """points inside a clockwise convex polygon"""
    ok = np.ones(len(pts), dtype=bool)
    for i in range(len(poly)):
        a, b = poly[i], poly[(i + 1) % len(poly)]
        ok &= ((b[0] - a[0]) * (pts[:, 1] - a[1]) - (b[1] - a[1]) * (pts[:, 0] - a[0])) <= 0
    return ok


def test_oracle_against_independent_sampling_estimate():
    g = _pairs()
    gt, pr = g["gt_corners"].astype(np.float64), g["pr_corners"].astype(np.float64)
    want = ob.rbbox_iou_3d_pair(pr, gt)
    rng = np.random.default_rng(5)
    for n in range(0, 64):
        P = pr[n][list(ob.BEV_ORDER)][:, [0, 2]]
        Q = gt[n][list(ob.BEV_ORDER)][:, [0, 2]]
        lo, hi = np.minimum(P.min(0), Q.min(0)), np.maximum(P.max(0), Q.max(0))
        pts = lo + rng.random((200000, 2)) * (hi - lo)
        box = float(np.prod(hi - lo))
        inP, inQ = _inside(P, pts), _inside(Q, pts)
        inter = box * np.mean(inP & inQ)
        union = box * np.mean(inP | inQ)
        est = inter / union if union > 0 else 0.0
        assert abs(est - want[n, 0]) <= 0.01, (n, est, want[n])
    assert want[0, 0] == pytest.approx(1.0) and want[0, 1] == pytest.approx(1.0)
    assert not want[3].any()                                   # 100 m apart
    assert ((want >= 0) & (want <= 1 + 1e-12)).all() and (want[:, 1] <= want[:, 0] + 1e-12).all()


HARNESS = r'''
#include "%s"
extern "C" void host_rbbox_iou(int M, const float* c, const float* q, float* out) {
    for (int n = 0; n < M; ++n) fcn::rbbox_iou_pair(c + 24 * n, q + 24 * n, out + 2 * n);
}
'''


def test_device_arithmetic_compiled_for_the_host_matches_oracle(tmp_path):
    """csrc/box_iou.cuh is plain C++ behind FCN_HD: build it with g++ and run the kernel's math on the CPU."""
    hdr = os.path.join(ROOT, "frustum_convnet_b200", "csrc", "box_iou.cuh")
    src = tmp_path / "harness.cpp"
    src.write_text(HARNESS % hdr)
    so = tmp_path / "libiou_host.so"
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-ffp-contract=off", "-o", str(so), str(src)])
    lib = ctypes.CDLL(str(so))
    g = _pairs()
    rng = np.random.default_rng(9)
    gt, pr = g["gt_corners"], g["pr_corners"]
    # plus degenerate inputs: identical, mirrored order, zero-size, touching edges
    extra_gt = np.stack([gt[5], gt[6], np.zeros((8, 3), np.float32), gt[8]])
    extra_pr = np.stack([gt[5], pr[6][::-1].copy(), np.zeros((8, 3), np.float32),
                         gt[8] + np.float32([100, 0, 0])])
    gt = np.ascontiguousarray(np.concatenate([gt, extra_gt]), dtype=np.float32)
    pr = np.ascontiguousarray(np.concatenate([pr, extra_pr]), dtype=np.float32)
    M = gt.shape[0]
    out = np.full((M, 2), -1.0, dtype=np.float32)
    P = ctypes.c_void_p
    lib.host_rbbox_iou(ctypes.c_int(M), P(pr.ctypes.data), P(gt.ctypes.data), P(out.ctypes.data))
    want = ob.rbbox_iou_3d_pair(pr, gt)
    ok = np.ones(M, dtype=bool)
    ok[256 + 1] = False          # reversed corner order is outside the function's contract (clockwise boxes)
    assert np.isfinite(out[ok]).all()
    assert np.abs(out[ok] - want[ok]).max() <= 2e-5, np.abs(out[ok] - want[ok]).max()
    assert out[256].tolist() == pytest.approx([1.0, 1.0], abs=1e-6)
    assert not out[258].any() and not out[259].any()


def _host_iou(tmp_path, pr, gt):
    hdr = os.path.join(ROOT, "frustum_convnet_b200", "csrc", "box_iou.cuh")
    src = tmp_path / "harness2.cpp"
    src.write_text(HARNESS % hdr)
    so = tmp_path / "libiou_host2.so"
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-ffp-contract=off", "-o", str(so), str(src)])
    lib = ctypes.CDLL(str(so))
    pr = np.ascontiguousarray(pr, dtype=np.float32)
    gt = np.ascontiguousarray(gt, dtype=np.float32)
    out = np.full((pr.shape[0], 2), -1.0, dtype=np.float32)
    P = ctypes.c_void_p
    lib.host_rbbox_iou(ctypes.c_int(pr.shape[0]), P(pr.ctypes.data), P(gt.ctypes.data), P(out.ctypes.data))
    return out


def test_degenerate_boxes(tmp_path):
    """Decoded boxes with negative sizes (untrained weights; the round-1 GPU failure): the pinned decision of
    oracle/box_iou.py - a counter-clockwise (invalid) BEV ring scores (0, 0); two negative footprint sizes are
    a valid box rotated by pi; a negative height gives IoU_3D = 0 through the reference's own max(0, .) terms -
    and the invariants 0 <= IoU_3D <= IoU_2D <= 1 on random decoded boxes, for oracle AND device arithmetic."""
    ctr, head = [[0.3, 0.1, 8.0]], [0.2]
    gt = _boxes(ctr, head, [[3.9, 1.6, 1.5]])
    good = ob.rbbox_iou_3d_pair(_boxes(ctr, head, [[3.9, 1.6, 1.5]]), gt)[0]
    assert np.allclose(good, [1.0, 1.0])
    for sz in ([-3.9, 1.6, 1.5], [3.9, -1.6, 1.5]):                       # one negative footprint size
        assert not ob.rbbox_iou_3d_pair(_boxes(ctr, head, [sz]), gt).any()
        assert not ob.rbbox_iou_3d_pair(gt, _boxes(ctr, head, [sz])).any()
    both = ob.rbbox_iou_3d_pair(_boxes(ctr, head, [[-3.9, -1.6, 1.5]]), gt)[0]
    assert np.allclose(both, [1.0, 1.0])                                  # rotated by pi: the same box
    negh = ob.rbbox_iou_3d_pair(_boxes(ctr, head, [[3.9, 1.6, -1.5]]), gt)[0]
    assert negh[0] == pytest.approx(1.0) and negh[1] == 0.0
    rng = np.random.default_rng(11)
    M = 512
    c = rng.normal(0, 0.5, (M, 3)) + [0, 0, 8.0]
    h = rng.uniform(-np.pi, np.pi, M)
    s = rng.normal(0.5, 2.0, (M, 3))                                      # ~40 % negative entries
    pr = _boxes(c, h, s)
    gtb = _boxes(np.tile([[0.0, 0.0, 8.0]], (M, 1)), np.zeros(M), np.tile([[3.9, 1.6, 1.5]], (M, 1)))
    want = ob.rbbox_iou_3d_pair(pr, gtb)
    bad = (s[:, 0] * s[:, 1]) <= 0
    assert bad.sum() > 50 and not want[bad].any()
    assert ((want >= 0) & (want <= 1 + 1e-9)).all() and (want[:, 1] <= want[:, 0] + 1e-9).all()
    got = _host_iou(tmp_path, pr, gtb)
    assert np.isfinite(got).all() and np.abs(got - want).max() <= 5e-5
    assert not got[bad].any()
    assert ((got >= 0) & (got <= 1 + 1e-5)).all() and (got[:, 1] <= got[:, 0] + 1e-5).all()


def _iou_ref():
    return dict(np.load(os.path.join(ROOT, "tests", "golden", "iou_ref.npz")))


def test_iou_fixture_covers_every_group():
    """tests/golden/iou_ref.npz (oracle/make_golden_iou.py: the reference's own utils/box_util.py IoU): every
    named group is present, most pairs overlap partly in 3-D, and the exclusions are recorded."""
    g = _iou_ref()
    names = [str(n) for n in g["group_names"]]
    counts = np.bincount(g["group"], minlength=len(names))
    assert len(names) == 12 and (counts >= 150).all(), dict(zip(names, counts))
    assert len(g["iou"]) >= 2000 and g["iou"].dtype == np.float64 and g["pr_corners"].dtype == np.float32
    i3 = g["iou"][:, 1]
    assert ((i3 > 0) & (i3 < 1)).mean() > 0.8
    assert (i3[g["group"] == names.index("heights_disjoint")] == 0).all()
    assert (g["iou"][g["group"] == names.index("near_miss"), 0] == 0).sum() >= 20      # both sides of touching
    assert [str(r) for r in g["excluded_reasons"]] == ["touching_edges", "hull_error"]
    assert int(g["excluded_counts"].sum()) >= 1                           # box_pairs pair 0: coincident boxes


def test_oracle_matches_reference_python_iou():
    """The BEV clip of oracle/box_iou.py equals the reference's polygon_clip + ConvexHull to float64 rounding.  The
    3-D column differs by the volume formula alone: box_util multiplies three corner-to-corner edge lengths, Boost
    (and this oracle) the footprint area by the height; on float32 corners 70 m out the two differ by <= 2.2e-6."""
    g = _iou_ref()
    want = ob.rbbox_iou_3d_pair(g["pr_corners"], g["gt_corners"])
    err = np.abs(want - g["iou"]).max(0)
    print("oracle vs reference IoU: worst BEV %.2e, 3-D %.2e" % tuple(err))
    assert err[0] <= 1e-9 and err[1] <= 4e-6, err


def test_device_arithmetic_matches_reference_python_iou(tmp_path):
    """csrc/box_iou.cuh compiled with g++ against the reference-held values, group by group."""
    g = _iou_ref()
    got = _host_iou(tmp_path, g["pr_corners"], g["gt_corners"])
    err = np.abs(got - g["iou"])
    print("g++ box_iou.cuh vs reference IoU: worst BEV %.2e, 3-D %.2e" % tuple(err.max(0)))
    assert np.isfinite(got).all() and err.max() <= 2e-5, err.max(0)
    for k, name in enumerate(g["group_names"]):
        assert err[g["group"] == k].max() <= 2e-5, name
