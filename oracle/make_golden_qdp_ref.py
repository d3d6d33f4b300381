"""ORACLE (test infrastructure) - fixture of the reference's own CUDA grouping kernel.

Runs `query_depth_point_gpu` of the reference (oracle/_ref/libqdp_ref.so, built by oracle/build_ref_qdp.py where
the reference tree exists) on the seeded cases below and stores its outputs as tests/golden/qdp_ref.npz, so that
tests/test_gpu_bench_config.py compares the grouping op with what the reference computed on a B200 without
needing the reference tree.

    python -m oracle.make_golden_qdp_ref [OUT.npz]     # needs a CUDA device and oracle/_ref/libqdp_ref.so
"""
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden", "qdp_ref.npz")


def cases():
    """[(xyz1 (B,3,N) float32, xyz2 (B,3,M) float32, dis_z, nsample)]: every scale of every workload, then a
    small case with a NaN point and a centre exactly on the depth window's edge."""
    from frustum_convnet_b200 import config, synth
    out = []
    for wl, B in (("car", 4), ("people", 2), ("sunrgbd", 2), ("refine_car", 4)):
        cfg, w = config.load_workload(wl)
        data = synth.make_frustums(wl, B, seed=900)
        for i in range(w["arch"].num_scales):
            out.append((data["point_cloud"], data["center_ref%d" % (i + 1)], cfg.DATA.HEIGHT_HALF[i],
                        w["arch"].nsample[i]))
    rng = np.random.default_rng(17)
    a = (rng.random((3, 3, 333)) * 4 - 2).astype(np.float32)
    b = (rng.random((3, 3, 41)) * 4 - 2).astype(np.float32)
    a[0, 2, 5] = np.nan
    b[0, 2, 0] = a[0, 2, 1] + np.float32(0.25)
    out.append((a, b, 0.25, 16))
    return out


def input_checksum(cs):
    return float(sum(np.nansum(np.asarray(a, dtype=np.float64)) + np.nansum(np.asarray(b, dtype=np.float64))
                     + dz + K for a, b, dz, K in cs))


def run_reference(cs):
    """The reference kernel on cuda:0, called the way query_depth_point.py:29-39 calls it."""
    import torch
    from oracle import build_ref_qdp
    lib = ctypes.CDLL(build_ref_qdp.LIB)
    lib.qdp_ref_forward.argtypes = [ctypes.c_int] * 3 + [ctypes.c_float, ctypes.c_int] + [ctypes.c_void_p] * 5
    res = []
    for pc, cen, dz, K in cs:
        B, _, N = pc.shape
        M = cen.shape[2]
        x1t = torch.from_numpy(pc).cuda().permute(0, 2, 1).contiguous()
        x2t = torch.from_numpy(cen).cuda().permute(0, 2, 1).contiguous()
        idx = torch.zeros((B, M, K), dtype=torch.int64, device="cuda")
        cnt = torch.zeros((B, M), dtype=torch.int32, device="cuda")
        rc = lib.qdp_ref_forward(B, N, M, float(dz), int(K), x1t.data_ptr(), x2t.data_ptr(), idx.data_ptr(),
                                 cnt.data_ptr(), torch.cuda.current_stream().cuda_stream)
        assert rc == 0, rc
        torch.cuda.synchronize()
        res.append((idx.cpu().numpy(), cnt.cpu().numpy()))
    return res


if __name__ == "__main__":
    path = sys.argv[1] if len(sys.argv) > 1 else GOLDEN
    cs = cases()
    arrays = {"input_checksum": np.float64(input_checksum(cs))}
    for i, (idx, cnt) in enumerate(run_reference(cs)):
        assert idx.min() >= 0 and idx.max() < 2 ** 15 and cnt.max() < 2 ** 15
        arrays["idx%d" % i] = idx.astype(np.int16)            # point indices < N <= 2048
        arrays["cnt%d" % i] = cnt.astype(np.int16)
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    np.savez_compressed(path, **arrays)
    print(path, "%.1f KB" % (os.path.getsize(path) / 1024))
