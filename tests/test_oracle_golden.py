"""CPU: the oracle restatement must reproduce the fixtures produced by the reference itself
(oracle/make_golden.py ran the unmodified /root/reference model).  This is what pins the oracle."""
import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES, load_golden
from oracle import model as om
from oracle import qdp

# The fixtures were written by torch on the CPU with 8 intra-op threads.  oneDNN splits convolution reductions by
# thread count, so the fp32 sums only round the same way with the same count, whatever the host's core count.
GOLDEN_THREADS = 8


@pytest.fixture
def golden_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_oracle_model_matches_reference_golden(name, golden_threads):
    g, data, sd, w, cfg = load_golden(name)
    arch = w["arch"]
    from frustum_convnet_b200.config import DATASET_INFO
    res = om.pointnet_det_eval(data, om.to_torch_state(sd), cfg.DATA.HEIGHT_HALF, arch.nsample,
                               DATASET_INFO[cfg.DATA.DATASET_NAME].MEAN_SIZE_ARRAY, return_all=True)
    for i in range(arch.num_scales):
        idx, cnt = res["groups"][i]
        assert np.array_equal(idx.numpy(), g["idx%d" % (i + 1)].astype(np.int64))
        assert np.array_equal(cnt.numpy(), g["cnt%d" % (i + 1)].astype(np.int32))
        np.testing.assert_allclose(res["feats"][i].numpy(), g["feat%d" % (i + 1)], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(res["x"].numpy(), g["x"], rtol=1e-5, atol=1e-5)
    B = data["point_cloud"].shape[0]
    cls = res["cls"].view(B, -1, 2).permute(0, 2, 1).numpy()
    reg = res["reg"].view(B, -1, res["reg"].shape[1]).permute(0, 2, 1).numpy()
    np.testing.assert_allclose(cls, g["cls"], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(reg, g["reg"], rtol=1e-5, atol=1e-5)
    for j, o in enumerate(res["out"]):
        np.testing.assert_allclose(o.numpy(), g["out%d" % j], rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("name", ["car_small_b3", "sunrgbd_full_b2", "refine_car_b4"])
def test_grouping_restatements_agree_with_golden(name):
    """C loop, numpy formulation (and the pure-python loop on a slice) all equal the fixture."""
    g, data, sd, w, cfg = load_golden(name)
    arch = w["arch"]
    pc = data["point_cloud"]
    for i in range(arch.num_scales):
        c = data["center_ref%d" % (i + 1)]
        d, k = cfg.DATA.HEIGHT_HALF[i], arch.nsample[i]
        gi, gc = g["idx%d" % (i + 1)].astype(np.int64), g["cnt%d" % (i + 1)].astype(np.int32)
        for fn in (qdp.qdp_c, qdp.qdp_numpy):
            idx, cnt = fn(pc, c, d, k)
            assert np.array_equal(idx, gi) and np.array_equal(cnt, gc)
        idx, cnt = qdp.qdp_c(pc, c, d, k, transposed_call=True)
        assert np.array_equal(idx, gi) and np.array_equal(cnt, gc)
        idx, cnt = qdp.qdp_loops(pc[:1, :, :], c[:1, :, :4], d, k)
        assert np.array_equal(idx, gi[:1, :4]) and np.array_equal(cnt, gc[:1, :4])


def test_grouping_reference_smoke_script_shape():
    """The reference's only op 'test' (ops/query_depth_point/test.py:8-28): B=2, N=50 uniform
    [-1,1], queries = first 10 points, dis_z=0.2, nsample=4; it prints a brute-force mask.
    Here the same construction is asserted instead of eyeballed."""
    rng = np.random.default_rng(5)
    xyz1 = (rng.random((2, 3, 50)) * 2 - 1).astype(np.float32)
    xyz2 = xyz1[:, :, :10].copy()
    idx, cnt = qdp.qdp_c(xyz1, xyz2, 0.2, 4)
    for b in range(2):
        for j in range(10):
            inside = np.nonzero(np.abs(xyz1[b, 2] - xyz2[b, 2, j]) < np.float32(0.2))[0]
            n = min(len(inside), 4)
            assert cnt[b, j] == n
            assert list(idx[b, j, :n]) == list(inside[:n])
            assert (idx[b, j, n:] == inside[0]).all()  # a query is always its own neighbour


def test_grouping_edge_cases():
    # empty sections -> zeros; strict '<' at the boundary; NaN never selected; duplicates kept
    z = np.array([0.0, 0.5, 0.5, np.nan, 1.0, 2.0], dtype=np.float32)
    pc = np.zeros((1, 3, 6), dtype=np.float32)
    pc[0, 2] = z
    c = np.zeros((1, 3, 4), dtype=np.float32)
    c[0, 2] = [0.5, 10.0, 1.5, np.nan]
    for fn in (qdp.qdp_c, qdp.qdp_numpy, qdp.qdp_loops):
        idx, cnt = fn(pc, c, 0.5, 3)
        assert list(cnt[0]) == [2, 0, 0, 0]          # |0.5-0|=0.5 and |1.5-1|=0.5 are NOT < 0.5
        assert list(idx[0, 0]) == [1, 2, 1]
        assert (idx[0, 1:] == 0).all()
    idx, cnt = qdp.qdp_c(pc, c, 0.5000001, 3)
    assert list(cnt[0]) == [3, 0, 2, 0] and list(idx[0, 0]) == [0, 1, 2]
