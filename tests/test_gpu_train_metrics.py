"""GPU: pairwise rotated-box IoU of the train metrics (SURVEY.md 8(f)-1) through the C ABI against the oracle
(oracle/box_iou.py) and against the reference's own Python IoU (utils/box_util.py, held in
tests/golden/iou_ref.npz): pinned to the reference for convex, non-degenerate boxes.
Tolerance: 1e-4 absolute on IoU values in [0, 1] (fp32 kernel with FMA contraction vs float64 values)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR

pytestmark = pytest.mark.gpu

TOL = 1e-4


def _pairs():
    return dict(np.load(os.path.join(GOLDEN_DIR, "box_pairs.npz")))


def test_iou_matches_oracle_on_reference_generated_corners():
    from frustum_convnet_b200.box_iou import rbbox_iou_3d_pair
    from oracle import box_iou as ob
    g = _pairs()
    pr, gt = torch.from_numpy(g["pr_corners"]).cuda(), torch.from_numpy(g["gt_corners"]).cuda()
    out, (m2, m3, frac) = rbbox_iou_3d_pair(pr, gt, iou_thresh=0.7)
    want = ob.rbbox_iou_3d_pair(g["pr_corners"], g["gt_corners"])
    got = out.cpu().numpy()
    assert got.shape == want.shape and got.dtype == np.float32
    assert np.abs(got - want).max() <= TOL
    assert abs(float(m2) - want[:, 0].mean()) <= TOL and abs(float(m3) - want[:, 1].mean()) <= TOL
    # pairs within 1e-3 of the threshold may fall on either side
    lo = (want[:, 1] >= 0.7 + 1e-3).mean()
    hi = (want[:, 1] >= 0.7 - 1e-3).mean()
    assert lo - 1e-6 <= float(frac) <= hi + 1e-6
    assert torch.equal(rbbox_iou_3d_pair(pr, gt), out)                     # without stats: same values


def test_iou_matches_reference_python_iou():
    """fcn_rbbox_iou_3d_pair on every group of the reference-held fixture, incl. the two mean statistics."""
    from frustum_convnet_b200.box_iou import rbbox_iou_3d_pair
    g = dict(np.load(os.path.join(GOLDEN_DIR, "iou_ref.npz")))
    want = g["iou"]
    pr, gt = torch.from_numpy(g["pr_corners"]).cuda(), torch.from_numpy(g["gt_corners"]).cuda()
    out, (m2, m3, frac) = rbbox_iou_3d_pair(pr, gt, iou_thresh=0.5)
    got = out.cpu().numpy()
    err = np.abs(got - want)
    print("device vs reference IoU: worst BEV %.2e, 3-D %.2e; means %.2e %.2e" % (
        *err.max(0), abs(float(m2) - want[:, 0].mean()), abs(float(m3) - want[:, 1].mean())))
    assert np.isfinite(got).all() and err.max() <= TOL
    for k, name in enumerate(g["group_names"]):
        assert err[g["group"] == k].max() <= TOL, name
    assert abs(float(m2) - want[:, 0].mean()) <= TOL and abs(float(m3) - want[:, 1].mean()) <= TOL
    lo, hi = (want[:, 1] >= 0.5 + 1e-3).mean(), (want[:, 1] >= 0.5 - 1e-3).mean()
    assert lo - 1e-6 <= float(frac) <= hi + 1e-6


def test_iou_edge_cases_and_scale():
    from frustum_convnet_b200.box_iou import rbbox_iou_3d_pair
    from oracle import box_iou as ob
    g = _pairs()
    gt = torch.from_numpy(g["gt_corners"]).cuda()
    # identical boxes -> exactly overlapping; far apart -> zeros
    same = rbbox_iou_3d_pair(gt, gt).cpu().numpy()
    assert np.abs(same - 1.0).max() <= TOL
    far = rbbox_iou_3d_pair(gt + torch.tensor([500.0, 0.0, 0.0], device="cuda"), gt)
    assert not far.any()
    # symmetric in its arguments
    pr = torch.from_numpy(g["pr_corners"]).cuda()
    assert (rbbox_iou_3d_pair(pr, gt) - rbbox_iou_3d_pair(gt, pr)).abs().max() <= TOL
    # N != K and N == 0 return zeros (box_ops.h:201-203); stats of an empty set are zeros
    assert not rbbox_iou_3d_pair(gt[:5], gt[:4]).any()
    out, stats = rbbox_iou_3d_pair(gt[:0], gt[:0], iou_thresh=0.5)
    assert out.shape == (0, 2) and all(float(s) == 0.0 for s in stats)
    with pytest.raises(RuntimeError):
        rbbox_iou_3d_pair(gt.cpu(), gt.cpu())
    # many pairs (one training step has at most B*T2 foreground positions): tile the fixture 400x
    big_p, big_g = pr.repeat(400, 1, 1), gt.repeat(400, 1, 1)
    out, (m2, m3, _) = rbbox_iou_3d_pair(big_p, big_g, iou_thresh=0.7)
    want = ob.rbbox_iou_3d_pair(g["pr_corners"], g["gt_corners"])
    assert np.abs(out.view(400, -1, 2).cpu().numpy() - want[None]).max() <= TOL
    assert abs(float(m2) - want[:, 0].mean()) <= TOL and abs(float(m3) - want[:, 1].mean()) <= TOL


def test_train_branch_reports_device_iou_metrics_by_default():
    """The reference's train driver consumes IoU_<thresh> for best-model selection (train_net_det.py:203,378):
    the device metric is the default; untrained weights decode negative sizes -> degenerate pairs score 0."""
    from frustum_convnet_b200 import config, synth
    from frustum_convnet_b200.det_base import PointNetDet
    from frustum_convnet_b200 import train_path
    from oracle import box_iou as ob
    cfg, w = config.load_workload("refine_car")
    sd = synth.make_state_dict(w["arch"], 3, "KITTI", seed=11)
    m = PointNetDet(3, num_vec=3)
    m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
    m = m.cuda().train()
    data = {k: torch.from_numpy(v).cuda()
            for k, v in synth.make_frustums("refine_car", 4, seed=206, with_labels=True).items()}
    captured = {}
    orig = train_path._iou_metrics

    def spy(c_metric, c_gt, thresh):
        captured["pr"], captured["gt"] = c_metric.detach().cpu().numpy(), c_gt.detach().cpu().numpy()
        return orig(c_metric, c_gt, thresh)

    train_path._iou_metrics = spy
    try:
        losses, on = m(data)
    finally:
        train_path._iou_metrics = orig
    i2, i3, ig = (float(on[k]) for k in ("IoU_2D", "IoU_3D", "IoU_" + str(cfg.IOU_THRESH)))
    assert 0.0 <= i3 <= i2 + 1e-6 and i2 <= 1.0 + 1e-6 and 0.0 <= ig <= 1.0
    assert torch.isfinite(losses["total_loss"])
    want = ob.rbbox_iou_3d_pair(captured["pr"], captured["gt"])          # same boxes through the oracle
    assert abs(i2 - want[:, 0].mean()) <= TOL and abs(i3 - want[:, 1].mean()) <= TOL
    m.gpu_iou_metrics = False                                            # explicit opt-out -> NaN placeholders
    _, off = m(data)
    assert all(torch.isnan(off[k]) for k in ("IoU_2D", "IoU_3D", "IoU_" + str(cfg.IOU_THRESH)))


def test_iou_degenerate_predictions_on_device():
    """Negative decoded sizes (counter-clockwise BEV ring) score (0, 0); invariants hold on random decoded boxes."""
    from frustum_convnet_b200.box_iou import rbbox_iou_3d_pair
    from oracle import box_iou as ob
    rng = np.random.default_rng(11)
    M = 2048
    c = rng.normal(0, 0.5, (M, 3)) + [0, 0, 8.0]
    h = rng.uniform(-np.pi, np.pi, M)
    s = rng.normal(0.5, 2.0, (M, 3))
    pr = ob.box3d_corners(c, h, s).astype(np.float32)
    gt = ob.box3d_corners(np.tile([[0.0, 0.0, 8.0]], (M, 1)), np.zeros(M),
                          np.tile([[3.9, 1.6, 1.5]], (M, 1))).astype(np.float32)
    got = rbbox_iou_3d_pair(torch.from_numpy(pr).cuda(), torch.from_numpy(gt).cuda()).cpu().numpy()
    want = ob.rbbox_iou_3d_pair(pr, gt)
    assert np.isfinite(got).all() and np.abs(got - want).max() <= TOL
    bad = (s[:, 0] * s[:, 1]) <= 0
    assert not got[bad].any()
    assert ((got >= 0) & (got <= 1 + 1e-5)).all() and (got[:, 1] <= got[:, 0] + 1e-5).all()
