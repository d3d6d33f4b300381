"""CPU: the C-ABI library builds, loads and exports every symbol declared in include/*.h
(no compute call is made without a GPU), and the host-side mirror behaves like the reference."""
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT


def _header_symbols():
    txt = open(os.path.join(ROOT, "include", "frustum_b200.h")).read()
    return sorted(set(re.findall(r"FCN_API\s+[\w\s\*]*?\b(fcn_\w+)\s*\(", txt)))


def test_library_builds_and_exports_every_header_symbol():
    from frustum_convnet_b200 import _lib, build
    build.build()
    lib = _lib.load()
    syms = _header_symbols()
    assert len(syms) >= 10
    for s in syms:
        assert hasattr(lib, s), "missing export " + s
        assert s in _lib.SIGNATURES, "ctypes signature table lacks " + s
    assert set(_lib.SIGNATURES) == set(syms)
    assert lib.fcn_version() >= 100


def test_argument_validation_without_gpu():
    """Validation happens before any CUDA call, so error codes are testable on CPU."""
    from frustum_convnet_b200 import _lib
    lib = _lib.load()
    assert lib.fcn_query_depth_point_b3n(1, 4, 4, 0.5, 0, None, None, None, None, None) == -1
    assert b"nsample" in lib.fcn_last_error()
    assert lib.fcn_query_depth_point_b3n(0, 4, 4, 0.5, 4, None, None, None, None, None) == 0  # empty batch
    assert lib.fcn_group_rows(None, None) == -1
    assert lib.fcn_decode_eval(1, 1, 1, 8, 12, 3, None, None, None, None, None, None, None, None, None, None) == -1
    with pytest.raises(RuntimeError):
        _lib.call("fcn_conv_gemm", None, None)
    # rotated-box IoU entry: size / NULL / alignment checks come before the launch
    assert lib.fcn_rbbox_iou_3d_pair(-1, None, None, None, 0.5, None, None) == -1
    assert lib.fcn_rbbox_iou_3d_pair(4, None, None, None, 0.5, None, None) == -1
    assert b"NULL" in lib.fcn_last_error()
    buf = np.zeros(64, dtype=np.float32)
    base = buf.ctypes.data + (-buf.ctypes.data) % 16          # a 16-byte aligned host address
    assert lib.fcn_rbbox_iou_3d_pair(1, base + 4, base, base, 0.5, None, None) == -1
    assert b"aligned" in lib.fcn_last_error()
    assert lib.fcn_rbbox_iou_3d_pair(0, None, None, None, 0.5, None, None) == 0   # nothing to do, no stats
    # rotated 3-D NMS: sizes, keep-row overflow and the long-list workspace are checked before any CUDA call
    nms = lib.fcn_rotate_nms_3d
    p = buf.ctypes.data
    assert nms(1, p, p, 10, 0.5, 300, p, p, 299, None, 0, None) == -1            # top_k > keep_stride
    assert b"keep_stride" in lib.fcn_last_error()
    assert nms(0, None, None, 0, 0.5, 8, None, None, 4, None, 0, None) == -1      # ... even with no segment
    assert nms(1, p, p, -1, 0.5, 8, p, p, 8, None, 0, None) == -1                # negative length
    assert b"max_seg_len" in lib.fcn_last_error()
    assert nms(1, p, p, 513, 0.5, 8, p, p, 8, None, 0, None) == -1               # long list, no workspace
    assert b"workspace" in lib.fcn_last_error()
    need = lib.fcn_rotate_nms_3d_workspace_bytes(1, 2000)
    assert need >= 2000 * (2000 // 32) * 4                                       # holds the n x n/32 bit matrix
    assert nms(1, p, p, 2000, 0.5, 8, p, p, 8, base, need - 1, None) == -1        # too small
    assert nms(1, p, p, 2000, 0.5, 8, p, p, 8, base + 4, need, None) == -1        # misaligned
    assert b"aligned" in lib.fcn_last_error()
    assert nms(1, None, p, 10, 0.5, 8, p, p, 8, None, 0, None) == -1             # NULL
    assert nms(0, None, None, 0, 0.5, 8, None, None, 8, None, 0, None) == 0       # nothing to do
    ws = lib.fcn_rotate_nms_3d_workspace_bytes
    assert ws(0, 2000) == 0 and ws(5, 512) == 0 and ws(3, 513) > 0
    assert ws(2, 2000) > ws(1, 2000) and ws(1, 4000) > 3 * ws(1, 2000)
    assert ws(-1, 600) == -1 and ws(1, -5) == -1
    assert ws(1, lib.fcn_rotate_nms_3d_max_seg_len() + 1) == -1
    assert lib.fcn_rotate_nms_3d_max_dets() == 512


def test_box_iou_wrapper_rejects_cpu_tensors_and_bad_shapes():
    from frustum_convnet_b200.box_iou import rbbox_iou_3d_pair
    with pytest.raises(RuntimeError):
        rbbox_iou_3d_pair(torch.zeros(2, 8, 3), torch.zeros(2, 8, 3))


def test_cpu_tensors_are_rejected_like_the_reference():
    """query_depth_point.py:23-24 asserts .is_cuda; there is no CPU path here either."""
    from frustum_convnet_b200.query_depth_point import QueryDepthPoint
    q = QueryDepthPoint(0.25, 8)
    with pytest.raises(AssertionError):
        q(torch.zeros(1, 3, 16), torch.zeros(1, 3, 4))


def test_state_dict_names_match_reference_layout(golden_loader):
    from frustum_convnet_b200 import config
    for name, modname in (("car_small_b3", "det_base"), ("sunrgbd_full_b2", "det_base_sunrgbd")):
        g, data, sd, w, cfg = golden_loader(name)
        mod = __import__("frustum_convnet_b200." + modname, fromlist=["PointNetDet"])
        m = mod.PointNetDet(3, num_vec=w["num_vec"])
        res = m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, strict=True)
        assert not res.missing_keys and not res.unexpected_keys
        n = sum(p.numel() for p in m.parameters())
        assert n == (3316777 if modname == "det_base" else 6667589)  # SURVEY.md 8(a7)
        with pytest.raises(RuntimeError):   # eval forward on CPU must fail loudly, not fall back
            m.eval()
            m({k: torch.from_numpy(v) for k, v in data.items()})


def test_engine_weight_pack_is_a_pure_function_of_the_state_dict(golden_loader):
    """BN folding on the host (CPU tensors here): folded 1x1 weights reproduce conv+BN."""
    from frustum_convnet_b200.engine import _fold_bn
    g, data, sd, w, cfg = golden_loader("car_small_b3")
    tsd = {k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}
    p = "feat_net.pointnet1.conv1"
    s, sh = _fold_bn(tsd, p + ".1")
    x = torch.randn(5, 3, dtype=torch.float64)
    wq = tsd[p + ".0.weight"].double()[:, :, 0, 0]
    ref = torch.nn.functional.batch_norm(
        (x @ wq.t()).float(), tsd[p + ".1.running_mean"], tsd[p + ".1.running_var"],
        tsd[p + ".1.weight"], tsd[p + ".1.bias"], False, 0.1, 1e-5)
    mine = x @ (wq * s[:, None]).t() + sh
    assert torch.allclose(ref.double(), mine, atol=1e-5)


def test_public_header_is_plain_c(tmp_path):
    """include/frustum_b200.h is the drop-in boundary: it must compile as C99 with nothing but libc headers."""
    import subprocess
    src = tmp_path / "hdr.c"
    src.write_text('#include "frustum_b200.h"\nint main(void) { (void)fcn_version; return 0; }\n')
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only",
                           "-I", os.path.join(ROOT, "include"), str(src)])
    txt = open(os.path.join(ROOT, "include", "frustum_b200.h")).read()
    includes = re.findall(r'#\s*include\s*[<"]([^>"]+)[>"]', txt)
    assert includes and all(i in ("stdint.h", "stddef.h") for i in includes), includes   # no torch / CUDA headers


def test_ctypes_mirrors_have_the_size_of_the_c_structs(tmp_path):
    """frustum_convnet_b200/_lib.py restates every argument struct of include/frustum_b200.h for ctypes: a field
    added on one side only would silently shift everything behind it.  Compare sizeof() as gcc sees the header."""
    import ctypes
    import subprocess
    from frustum_convnet_b200 import _lib
    pairs = [("fcn_group_args", _lib.GroupArgs), ("fcn_pointnet_args", _lib.PointnetArgs),
             ("fcn_conv_seg", _lib.ConvSeg), ("fcn_conv_args", _lib.ConvArgs), ("fcn_decode_out", _lib.DecodeOut),
             ("fcn_mega_seg", _lib.MegaSeg), ("fcn_mega_layer", _lib.MegaLayer), ("fcn_mega_job", _lib.MegaJob),
             ("fcn_mega_args", _lib.MegaArgs), ("fcn_train_src", _lib.TrainSrc), ("fcn_train_seg", _lib.TrainSeg),
             ("fcn_train_layer", _lib.TrainLayer), ("fcn_train_pool_args", _lib.TrainPool),
             ("fcn_loss_args", _lib.LossArgs), ("fcn_input_args", _lib.InputArgs)]
    src = tmp_path / "sizes.c"
    src.write_text('#include <stdio.h>\n#include "frustum_b200.h"\nint main(void) {\n' +
                   "".join('    printf("%s %%zu\\n", sizeof(%s));\n' % (n, n) for n, _ in pairs) + "    return 0;\n}\n")
    exe = tmp_path / "sizes"
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    sizes = dict(l.split() for l in subprocess.check_output([str(exe)], text=True).splitlines())
    for name, cls in pairs:
        assert int(sizes[name]) == ctypes.sizeof(cls), (name, sizes[name], ctypes.sizeof(cls))
