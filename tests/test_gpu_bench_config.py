"""GPU parity of EXACTLY the benchmarked configuration and of the full-size workloads (VERDICT r1, items 1b-1d).

bench.py runs: precision=1 (TF32 tcgen05), use_cuda_graph=True, copy_outputs=False, 10 forwards in flight on
10 CUDA streams (one plan + graph per stream), B=32.  Here the SAME configuration is compared with the
oracle (oracle.model.pointnet_det_eval, fp32 on the CPU) - all six outputs of det_base.py:411.

Stated TF32 tolerance (kind::tf32 operands keep a 10-bit mantissa, fp32 accumulate; <= 14 chained GEMMs):
  * LINEAR outputs - the head logits (cls, reg) and the centre OFFSETS (out1 - center_ref2: comparing the absolute
    centres would hide the error behind the 70 m depth range):
        max|a-b| <= 2.5e-3 * max(1, max|ref|)      and      rms(a-b) <= 1.5e-3 * max(rms(ref), 1e-3)
  * SOFTMAX outputs (out0, out4, out5): a softmax is 1/2-Lipschitz in the max-norm of its logits
    (sum_j |dp_i/dl_j| = 2 p_i (1 - p_i) <= 1/2), so the logit bound maps to
        max|dp| <= 0.5 * 2.5e-3 * max|logits_ref|     and      rms(dp) <= 1e-3   (probabilities live in [0, 1])
  * label-dependent outputs (heading = out2, size = out3) are compared with the linear bound where the oracle's
    arg-max is not numerically ambiguous (top-2 probability gap > 1e-2), as the fp32 test does with a 1e-3 gap.
Measured (B200, round 2): logits 1.2e-3 * max, probabilities 5e-3 max / 5e-4 rms.
"""
import numpy as np
import pytest
import torch

from test_gpu_parity import build_model, close, cuda_data, dev

pytestmark = pytest.mark.gpu

TF32_MAX, TF32_RMS = 2.5e-3, 1.5e-3


def _np(a):
    return a.detach().float().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)


def close_tf32(a, ref, what, mask=None, max_lim=None, rms_lim=None):
    a, ref = _np(a), _np(ref)
    assert a.shape == ref.shape, "%s shape %s vs %s" % (what, a.shape, ref.shape)
    if mask is not None:
        a, ref = a[mask], ref[mask]
    d = (a.astype(np.float64) - ref.astype(np.float64))
    err, rms = float(np.abs(d).max()), float(np.sqrt(np.mean(d * d)))
    lim = TF32_MAX * max(1.0, float(np.abs(ref).max())) if max_lim is None else max_lim
    rlim = TF32_RMS * max(float(np.sqrt(np.mean(ref.astype(np.float64) ** 2))), 1e-3) if rms_lim is None else rms_lim
    print("%-44s max err %.3e (lim %.3e)  rms %.3e (lim %.3e)" % (what, err, lim, rms, rlim))
    assert err <= lim, "%s: max abs err %.3e > %.3e" % (what, err, lim)
    assert rms <= rlim, "%s: rms err %.3e > %.3e" % (what, rms, rlim)


def _unambiguous(ref, gap=1e-2):
    hp, sp = np.sort(_np(ref[4]), -1), np.sort(_np(ref[5]), -1)
    return ((hp[..., -1] - hp[..., -2]) > gap) & ((sp[..., -1] - sp[..., -2]) > gap)


def _compare_all_six(out, logits, ra, center_ref2, what, nbins=12):
    """out: the 6-tuple; logits: (cls rows, reg rows) of the same forward; ra: oracle dict (return_all=True)."""
    ref = ra["out"]
    ok = _unambiguous(ref)
    assert ok.mean() > 0.8, "too many ambiguous arg-max positions (%.2f)" % ok.mean()
    cls_ref, reg_ref = _np(ra["cls"]), _np(ra["reg"])
    close_tf32(logits[0], cls_ref, what + " cls logits")
    close_tf32(logits[1], reg_ref, what + " reg logits")
    ref2 = np.transpose(np.asarray(center_ref2), (0, 2, 1))
    close_tf32(_np(out[1]) - ref2, _np(ref[1]) - ref2, what + " out1 (centre offsets)")
    ns = _np(ref[5]).shape[-1]
    groups = {0: cls_ref, 4: reg_ref[:, 3:3 + nbins], 5: reg_ref[:, 3 + 2 * nbins:3 + 2 * nbins + ns]}
    for j in (0, 4, 5):
        close_tf32(out[j], ref[j], "%s out%d (softmax)" % (what, j),
                   max_lim=0.5 * TF32_MAX * float(np.abs(groups[j]).max()), rms_lim=1e-3)
    close_tf32(out[2], ref[2], what + " out2 (heading)", mask=ok)
    close_tf32(out[3], ref[3], what + " out3 (size)", mask=ok)


def _oracle(workload, data, sd, cfg, w):
    from oracle import model as om
    from frustum_convnet_b200 import config
    return om.pointnet_det_eval(data, om.to_torch_state(sd), cfg.DATA.HEIGHT_HALF, w["arch"].nsample,
                                config.DATASET_INFO[cfg.DATA.DATASET_NAME].MEAN_SIZE_ARRAY, return_all=True)


def _plan_logits(m, data, w, stream=None):
    S = w["arch"].num_scales
    B, N = data["point_cloud"].shape[0], data["point_cloud"].shape[2]
    T = [data["center_ref%d" % (i + 1)].shape[2] for i in range(S)]
    if stream is None:
        cls, reg = m.engine().plan(B, N, T).logits()
    else:
        with torch.cuda.stream(stream):
            cls, reg = m.engine().plan(B, N, T).logits()
    return cls.clone(), reg.clone()


def test_bench_configuration_car_b32_matches_oracle():
    """TF32 + CUDA graph + zero-copy outputs + 10 streams in flight (bench.py default), B=32 car: every stream's result vs the oracle."""
    from frustum_convnet_b200 import config, synth
    cfg, w = config.load_workload("car")
    sd = synth.make_state_dict(w["arch"], 3, "KITTI", seed=7)           # bench.py's weights
    data = synth.make_frustums("car", 32, seed=1234)                     # bench.py's rank-0 batch
    ra = _oracle("car", data, sd, cfg, w)
    m = build_model(w, sd, cfg, precision=1, graph=True)
    m.copy_outputs = False
    nstream = 10
    streams = [torch.cuda.Stream(device=dev()) for _ in range(nstream)]
    keys = [k for k in data]
    # stream k processes the batch rolled by k frustums: the oracle result is the same roll (independent frustums)
    ins = [{k: torch.from_numpy(np.roll(data[k], s, axis=0)).to(dev()) for k in keys} for s in range(nstream)]
    torch.cuda.synchronize()
    outs = [None] * nstream
    for rep in range(3):                                                  # capture, then replays, all in flight
        for s, st in enumerate(streams):
            with torch.cuda.stream(st):
                outs[s] = m(ins[s])
    torch.cuda.synchronize()
    eng = m.engine()
    assert len(eng._plans) == nstream and all(p.graph is not None for p in eng._plans.values())
    for s in range(nstream):
        o = [t.roll(-s, 0) for t in outs[s]]
        if s in (0, 3, 7):
            lg = [t.view(32, -1, t.shape[1]).roll(-s, 0).reshape(-1, t.shape[1])
                  for t in _plan_logits(m, data, w, streams[s])]
            _compare_all_six(o, lg, ra, data["center_ref2"], "bench-config stream %d" % s)
        for a, b in zip(o, [t for t in outs[0]]):                         # all streams agree bit-exactly
            assert torch.equal(a, b)


@pytest.mark.parametrize("N", [1024, 512])
def test_people_full_size_grouping_bit_exact_and_forward(N):
    """cfgs/det_sample_people.yaml at its REAL shape T=(700,350,175,88) (MAX_DEPTH 70): the only workload that
    takes the bit-matrix grouping kernel to ~188 KB of shared memory.  N=1024 (yaml) and N=512 (BASELINE.json text)."""
    from oracle import qdp
    from frustum_convnet_b200 import config, synth
    from frustum_convnet_b200.query_depth_point import query_depth_point
    cfg, w = config.load_workload("people")
    B = 2
    data = synth.make_frustums("people", B, seed=501, N=N)
    T = [data["center_ref%d" % (i + 1)].shape[2] for i in range(4)]
    assert T == [700, 350, 175, 88]
    sd = synth.make_state_dict(w["arch"], 3, "KITTI", seed=9)
    d = cuda_data(data)
    # (1) the drop-in op, bit-exact idx / cnt
    cnt_ref = []
    for i in range(4):
        ri, rc = qdp.qdp_c(data["point_cloud"], data["center_ref%d" % (i + 1)], cfg.DATA.HEIGHT_HALF[i],
                           w["arch"].nsample[i])
        gi, gc = query_depth_point(cfg.DATA.HEIGHT_HALF[i], w["arch"].nsample[i], d["point_cloud"],
                                   d["center_ref%d" % (i + 1)])
        assert np.array_equal(gi.cpu().numpy(), ri) and np.array_equal(gc.cpu().numpy(), rc)
        cnt_ref.append(rc)
    # (2) the fused grouping of the engine (bit-matrix kernel): counts bit-exact, fp32 path == oracle
    ra = _oracle("people", data, sd, cfg, w)
    ref = ra["out"]
    m0 = build_model(w, sd, cfg, precision=0)
    out0 = m0(d)
    plan = m0.engine().plan(B, N, T)
    for i in range(4):
        assert np.array_equal(plan.cnt[i].cpu().numpy(), cnt_ref[i]), "fused grouping cnt, scale %d" % (i + 1)
    for j in (0, 1, 4, 5):
        close(out0[j], ref[j], tol=1e-3, what="people full-size fp32 out%d" % j)
    # (3) the benchmarked arithmetic at the same shape
    m1 = build_model(w, sd, cfg, precision=1, graph=True)
    out1 = m1(d)
    _compare_all_six(out1, _plan_logits(m1, data, w), ra, data["center_ref2"], "people full-size N=%d tf32" % N)


def test_sunrgbd_bench_configuration_matches_oracle():
    from frustum_convnet_b200 import config, synth
    cfg, w = config.load_workload("sunrgbd")
    sd = synth.make_state_dict(w["arch"], 10, "SUNRGBD", seed=7)
    data = synth.make_frustums("sunrgbd", 8, seed=1234)
    ra = _oracle("sunrgbd", data, sd, cfg, w)
    m = build_model(w, sd, cfg, precision=1, graph=True)
    m.copy_outputs = False
    out = m(cuda_data(data))
    _compare_all_six(out, _plan_logits(m, data, w), ra, data["center_ref2"], "sunrgbd tf32+graph")


def test_reference_cuda_kernel_agrees_bit_exact():
    """Secondary oracle: what the REFERENCE'S OWN kernel (query_depth_point_cuda_kernel.cu:16-65) computed on a
    B200 for these cases (tests/golden/qdp_ref.npz, written by oracle/make_golden_qdp_ref.py) vs our grouping op
    and vs the C restatement - upgrades the grouping pin from "restatement" to "the reference itself"."""
    from oracle import make_golden_qdp_ref, qdp
    from frustum_convnet_b200.query_depth_point import query_depth_point
    g = np.load(make_golden_qdp_ref.GOLDEN)
    cases = make_golden_qdp_ref.cases()
    chk = make_golden_qdp_ref.input_checksum(cases)
    assert abs(chk - float(g["input_checksum"])) <= 1e-6 * abs(chk), "inputs drifted from the golden fixture"
    for i, (pc, cen, dz, K) in enumerate(cases):
        idx, cnt = g["idx%d" % i].astype(np.int64), g["cnt%d" % i].astype(np.int32)
        gi, gc = query_depth_point(dz, K, torch.from_numpy(pc).to(dev()), torch.from_numpy(cen).to(dev()))
        assert gi.dtype == torch.int64 and gc.dtype == torch.int32
        assert np.array_equal(gi.cpu().numpy(), idx) and np.array_equal(gc.cpu().numpy(), cnt), \
            (pc.shape, cen.shape, dz, K)
        oi, oc = qdp.qdp_c(pc, cen, dz, K)
        assert np.array_equal(oi, idx) and np.array_equal(oc, cnt)


def test_reference_style_ctypes_binding():
    """The 12-line binding of INTEGRATION.md section 2 (what a maintainer drops into
    ops/query_depth_point/query_depth_point.py), executed literally."""
    import ctypes
    from frustum_convnet_b200 import _lib as L
    from oracle import qdp
    _lib = ctypes.CDLL(L.LIB_PATH)
    _lib.fcn_query_depth_point_bn3.argtypes = [ctypes.c_int] * 3 + [ctypes.c_float, ctypes.c_int] + [ctypes.c_void_p] * 5
    _lib.fcn_last_error.restype = ctypes.c_char_p

    class query_depth_point_cuda:
        @staticmethod
        def forward(b, n, m, dis_z, nsample, xyz1, xyz2, idx, pts_cnt):
            rc = _lib.fcn_query_depth_point_bn3(b, n, m, dis_z, nsample, xyz1.data_ptr(), xyz2.data_ptr(),
                                                idx.data_ptr(), pts_cnt.data_ptr(),
                                                torch.cuda.current_stream().cuda_stream)
            if rc:
                raise RuntimeError(_lib.fcn_last_error().decode())

    # the body of _query_depth_point.forward, query_depth_point.py:29-40
    rng = np.random.default_rng(5)
    xyz1 = torch.from_numpy((rng.random((3, 3, 500)) * 4).astype(np.float32)).to(dev())
    xyz2 = torch.from_numpy((rng.random((3, 3, 60)) * 4).astype(np.float32)).to(dev())
    dis_z, nsample = 0.3, 24
    b, n, m = xyz1.size(0), xyz1.size(2), xyz2.size(2)
    a, c = xyz1.permute(0, 2, 1).contiguous(), xyz2.permute(0, 2, 1).contiguous()
    idx = xyz1.new(b, m, nsample).long().zero_()
    pts_cnt = xyz1.new(b, m).int().zero_()
    query_depth_point_cuda.forward(b, n, m, dis_z, nsample, a, c, idx, pts_cnt)
    ri, rc_ = qdp.qdp_c(xyz1.cpu().numpy(), xyz2.cpu().numpy(), dis_z, nsample)
    assert np.array_equal(idx.cpu().numpy(), ri) and np.array_equal(pts_cnt.cpu().numpy(), rc_)
    with pytest.raises(RuntimeError):
        query_depth_point_cuda.forward(b, n, m, dis_z, 0, a, c, idx, pts_cnt)      # nsample must be positive


def test_stale_pack_after_parent_load_state_dict_and_inplace_update():
    """ADVICE r1: a checkpoint loaded through a PARENT module after eval(), and an in-place optimizer-style
    update, must both be served by the next eval forward (no stale BN-folded pack / graph)."""
    from frustum_convnet_b200 import config, synth
    cfg, w = config.load_workload("car")
    sd_a = synth.make_state_dict(w["arch"], 3, "KITTI", seed=31)
    sd_b = synth.make_state_dict(w["arch"], 3, "KITTI", seed=32)
    data = synth.make_frustums("car", 2, seed=5, max_depth=17.5)
    d = cuda_data(data)
    ma = build_model(w, sd_a, cfg, precision=1, graph=True)
    mb = build_model(w, sd_b, cfg, precision=1, graph=True)
    oa, ob = [o.clone() for o in ma(d)], [o.clone() for o in mb(d)]
    assert not torch.equal(oa[0], ob[0])

    class Wrapper(torch.nn.Module):
        def __init__(self, inner):
            super().__init__()
            self.module = inner

    wrap = Wrapper(ma)
    wrap.load_state_dict({"module." + k: torch.from_numpy(np.asarray(v)) for k, v in sd_b.items()})
    o2 = ma(d)
    for x, y in zip(o2, ob):
        assert torch.equal(x, y)
    with torch.no_grad():                                   # in-place update (what optimizer.step() does)
        for p_, (k, v) in zip(ma.parameters(), [(k, v) for k, v in ma.named_parameters()]):
            p_.copy_(torch.from_numpy(np.asarray(sd_a[k])).to(p_.device))
        for k, bfr in ma.named_buffers():
            bfr.copy_(torch.from_numpy(np.asarray(sd_a[k])).to(bfr.device))
    o3 = ma(d)
    for x, y in zip(o3, oa):
        assert torch.equal(x, y)
