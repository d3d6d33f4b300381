"""GPU: batched rotated 3-D NMS (csrc/nms3d.cu, ``fcn_rotate_nms_3d``) against the oracle (oracle/nms.py).
The keep lists are index sets, so parity is EXACT wherever no pair sits within 1e-4 of the IoU threshold (fp32
kernel vs float64 oracle); inputs with such a pair are regenerated."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _dets(rng, n, spread):
    return np.concatenate([rng.normal([0, 1, 20], [spread, 0.2, spread], (n, 3)),
                           rng.uniform([3, 1.4, 1.3], [4.5, 1.9, 1.8], (n, 3)),
                           rng.uniform(-np.pi, np.pi, (n, 1)), rng.random((n, 1))], 1).astype(np.float32)


def test_single_list_matches_oracle_and_reference_contract():
    from frustum_convnet_b200.nms import cube_nms, rotate_nms_3d_cc
    from oracle import nms as onms
    rng = np.random.default_rng(1)
    done = 0
    while done < 12:
        n = int(rng.integers(2, 90))
        d = _dets(rng, n, spread=float(rng.uniform(1.0, 6.0)))
        thr = float(rng.choice([0.1, 0.25, 0.5, 0.7]))
        if onms.pair_margins(d, thr) < 1e-4:
            continue
        want = onms.rotate_nms_3d_cc(d, thr)
        got = rotate_nms_3d_cc(torch.from_numpy(d).cuda(), thr)
        assert got == want, (n, thr)
        done += 1
    assert cube_nms(torch.zeros((0, 8), device="cuda"), 0.5) == []
    one = torch.from_numpy(_dets(rng, 1, 1.0)).cuda()
    assert cube_nms(one, 0.5) == [0]
    with pytest.raises(RuntimeError):
        cube_nms(one.cpu(), 0.5)


def test_batched_segments_top_k_and_ties():
    from frustum_convnet_b200.nms import rotate_nms_3d_batched
    from oracle import nms as onms
    rng = np.random.default_rng(2)
    segs, lens = [], [0, 1, 37, 120, 300, 5]
    for n in lens:
        while True:
            d = _dets(rng, n, spread=3.0)
            if n < 2 or onms.pair_margins(d, 0.3) >= 1e-4:
                break
        segs.append(d)
    segs[5][:, 7] = 0.5                                   # all-equal scores: larger index first
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    dets = torch.from_numpy(np.concatenate(segs)).cuda()
    keep, cnt = rotate_nms_3d_batched(dets, torch.from_numpy(off), 0.3, top_k=40)
    keep, cnt = keep.cpu().numpy(), cnt.cpu().numpy()
    for s, d in enumerate(segs):
        want = [off[s] + k for k in onms.rotate_nms_3d_cc(d, 0.3, top_k=40)]
        assert cnt[s] == len(want) and keep[s, :cnt[s]].tolist() == want, s
        assert (keep[s, cnt[s]:] == -1).all()


# ---- lists longer than the 512-box shared-memory path -------------------------------------------------------
LONG_THR = 0.25


def _scene(rng, n, area=70.0):
    """n car-like boxes spread over an area x area m ground patch (a few hundred overlapping pairs per 1000 boxes),
    scores ascending along the list so that the best boxes sit in its tail."""
    d = np.concatenate([rng.uniform([-area / 2, 0.8, 5.0], [area / 2, 1.2, 5.0 + area], (n, 3)),
                        rng.uniform([3, 1.4, 1.3], [4.5, 1.9, 1.8], (n, 3)),
                        rng.uniform(-np.pi, np.pi, (n, 1)), np.sort(rng.random((n, 1)), 0)], 1).astype(np.float32)
    return d


def _unambiguous(rng, d, thr, margin=1e-4):
    """Re-draw the position of one box of every pair within `margin` of flipping an NMS decision (IoU near the
    threshold or bounding cubes just touching) until no such pair is left: then fp32 kernel and float64 oracle
    must produce the same keep lists exactly."""
    from oracle import nms as onms
    for _ in range(50):
        i, j, m = onms.pair_iou_margins(d, thr)
        bad = np.unique(j[m < margin])
        if not len(bad):
            return d
        ok = np.isfinite(d[bad, :7]).all(1)
        bad = bad[ok]
        d[bad, 0] += rng.uniform(-0.3, 0.3, len(bad)).astype(np.float32)
        d[bad, 2] += rng.uniform(-0.3, 0.3, len(bad)).astype(np.float32)
    raise AssertionError("could not separate the pairs from the threshold")


@pytest.mark.parametrize("n", [513, 700, 2000])
def test_long_single_list_matches_oracle(n):
    """Lists past the shared-memory path are processed whole: the best boxes sit past row 512, so the answer on
    the first 512 rows (what truncation would give) differs from the full one, and the kernel must give the full
    one, with the default top_k and with an unlimited one."""
    from frustum_convnet_b200.nms import rotate_nms_3d_cc
    from oracle import nms as onms
    rng = np.random.default_rng(100 + n)
    d = _unambiguous(rng, _scene(rng, n), LONG_THR)
    full = onms.rotate_nms_3d_cc(d, LONG_THR, top_k=n)
    first512 = onms.rotate_nms_3d_cc(d[:512], LONG_THR, top_k=n)
    assert full != first512 and full[0] == n - 1                           # the case discriminates truncation
    assert len(full) > 300 or n < 700
    dd = torch.from_numpy(d).cuda()
    for top_k in (300, n):
        got = rotate_nms_3d_cc(dd, LONG_THR, top_k=top_k)
        assert got == full[:top_k], (n, top_k, len(got), len(full))
    print("n=%d: kept %d of %d (first 512 rows alone: %d)" % (n, len(full), n, len(first512)))


def test_batched_long_short_nan_inf_and_ties():
    """One call over segment lengths [0, 1, 511, 512, 513, 37, 2000]: both paths in one launch sequence, 600 equal
    scores, NaN / +-inf scores, NaN box geometry (never suppressed, suppresses nothing), counts and -1 padding."""
    from frustum_convnet_b200.nms import rotate_nms_3d_batched
    from oracle import nms as onms
    rng = np.random.default_rng(7)
    lens = [0, 1, 511, 512, 513, 37, 2000]
    segs = []
    for n in lens:
        d = _scene(rng, n, area=70.0 if n > 100 else 12.0)
        d[:, 7] = rng.permutation(d[:, 7])
        segs.append(d)
    big = segs[6]
    big[rng.choice(2000, 600, replace=False), 7] = 0.5                     # 600 equal scores
    for s, nan_rows in ((2, 5), (4, 7), (6, 20)):
        r = rng.choice(lens[s], nan_rows, replace=False)
        segs[s][r, 7] = np.nan
    for s in (3, 4, 6):
        segs[s][rng.choice(lens[s], 3, replace=False), 7] = np.inf
        segs[s][rng.choice(lens[s], 3, replace=False), 7] = -np.inf
    for s, rows in ((4, [0, 100, 512]), (5, [3]), (6, [10, 999, 1500]), (3, [511])):
        segs[s][rows, 0] = np.nan                                            # NaN geometry
    segs = [_unambiguous(rng, d, LONG_THR) if len(d) > 1 else d for d in segs]
    top_k = 700
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    dets = torch.from_numpy(np.concatenate(segs)).cuda()
    keep, cnt = rotate_nms_3d_batched(dets, torch.from_numpy(off).cuda(), LONG_THR, top_k=top_k)
    keep, cnt = keep.cpu().numpy(), cnt.cpu().numpy()
    assert keep.shape == (len(lens), top_k)
    for s, d in enumerate(segs):
        want = [int(off[s]) + k for k in onms.rotate_nms_3d_cc(d, LONG_THR, top_k=top_k)]
        assert cnt[s] == len(want) and keep[s, :cnt[s]].tolist() == want, (s, cnt[s], len(want))
        assert (keep[s, cnt[s]:] == -1).all()
        nan_geo = np.flatnonzero(np.isnan(d[:, 0]))
        assert set((off[s] + nan_geo).tolist()) <= set(want) or len(want) == top_k, s
    assert cnt[6] == top_k and cnt[0] == 0 and cnt[1] == 1
    # NaN scores first (larger index first among them), then +inf
    nan6 = np.flatnonzero(np.isnan(segs[6][:, 7]))
    assert keep[6, :len(nan6)].tolist() == (off[6] + nan6[::-1]).tolist()


def test_long_list_errors_instead_of_truncating():
    """A segment the library was not told about is flagged, never truncated: the wrapper raises."""
    from frustum_convnet_b200 import _lib
    rng = np.random.default_rng(8)
    d = torch.from_numpy(_scene(rng, 600)).cuda()
    off = torch.tensor([0, 600], dtype=torch.int32, device="cuda")
    keep = torch.full((1, 8), -1, dtype=torch.int32, device="cuda")
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    _lib.call("fcn_rotate_nms_3d", 1, d.data_ptr(), off.data_ptr(), 512, 0.25, 8, keep.data_ptr(), cnt.data_ptr(), 8,
              None, 0, stream)
    assert int(cnt[0]) == -1 and (keep == -1).all()
