"""ctypes binding of libfrustum_b200.so (the C ABI declared in include/frustum_b200.h).

No CPU fallback: if the shared library is missing this module raises at load time, and every
entry point raises ``RuntimeError`` with ``fcn_last_error()`` on a non-zero status, mirroring
the reference where AT_ASSERTM / THCudaCheck surface as Python exceptions
(/root/reference/ops/query_depth_point/query_depth_point_cuda.cpp:5-10, ..._kernel.cu:85).
"""
from __future__ import annotations

import ctypes as C
import os

MAX_SCALES = 8
MAX_SEGS = 4

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FCN_LIB_PATH") or os.path.join(_HERE, "libfrustum_b200.so")   # override: kernel-variant experiments


class GroupArgs(C.Structure):
    _fields_ = [
        ("num_scales", C.c_int), ("B", C.c_int), ("N", C.c_int), ("num_vec", C.c_int),
        ("tile_rows", C.c_int), ("unique_rows", C.c_int),
        ("pc", C.c_void_p), ("one_hot", C.c_void_p),
        ("centers", C.c_void_p * MAX_SCALES),
        ("T", C.c_int * MAX_SCALES), ("K", C.c_int * MAX_SCALES),
        ("dis_z", C.c_float * MAX_SCALES),
        ("c3", C.c_int * MAX_SCALES), ("ld_feat", C.c_int * MAX_SCALES),
        ("row_cap", C.c_int * MAX_SCALES), ("tile_cap", C.c_int * MAX_SCALES),
        ("rows", C.c_void_p * MAX_SCALES), ("cnt", C.c_void_p * MAX_SCALES),
        ("feat", C.c_void_p * MAX_SCALES), ("tiles", C.c_void_p * MAX_SCALES),
        ("idx_scratch", C.c_void_p * MAX_SCALES),
        ("feat_pitch", C.c_int * MAX_SCALES),
        ("ntiles", C.c_void_p),
        ("force_scan", C.c_int),
    ]


class PointnetArgs(C.Structure):
    _fields_ = [
        ("C1", C.c_int), ("C2", C.c_int), ("C3", C.c_int), ("T", C.c_int), ("K", C.c_int),
        ("ld_feat", C.c_int), ("row_cap", C.c_int), ("tile_rows", C.c_int),
        ("unpooled", C.c_int), ("precision", C.c_int), ("B", C.c_int),
        ("rows", C.c_void_p), ("tiles", C.c_void_p), ("ntiles", C.c_void_p),
        ("max_tiles", C.c_int),
        ("w1t", C.c_void_p), ("b1", C.c_void_p), ("w2t", C.c_void_p), ("b2", C.c_void_p),
        ("w3t", C.c_void_p), ("b3", C.c_void_p),
        ("w2_tc", C.c_void_p), ("w3_tc", C.c_void_p),
        ("out", C.c_void_p), ("dbg_clocks", C.c_void_p), ("feat_pitch", C.c_int),
    ]


class ConvSeg(C.Structure):
    _fields_ = [("src", C.c_void_p), ("ld", C.c_int), ("C", C.c_int), ("T_src", C.c_int),
                ("tap", C.c_int), ("stride", C.c_int), ("pitch", C.c_int)]


class ConvArgs(C.Structure):
    _fields_ = [
        ("B", C.c_int), ("T_out", C.c_int), ("n_seg", C.c_int),
        ("seg", ConvSeg * MAX_SEGS),
        ("K_pad", C.c_int), ("n_cols", C.c_int), ("Cout", C.c_int), ("up", C.c_int),
        ("relu", C.c_int), ("precision", C.c_int),
        ("wt", C.c_void_p), ("bias", C.c_void_p), ("w_tc", C.c_void_p),
        ("out", C.c_void_p),
        ("ld_out", C.c_int), ("T_store", C.c_int), ("c_off", C.c_int), ("round_out", C.c_int),
        ("dbg_clocks", C.c_void_p), ("tmaps", C.c_void_p),
        ("P_m", C.c_int), ("P_store", C.c_int),
    ]


MAX_PEERS = 8
MEGA_MAX_DEPS = 4


class DecodeOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("cls_probs", "center", "heading", "size", "heading_probs", "size_probs")]


class MegaSeg(C.Structure):
    _fields_ = [("map_idx", C.c_int), ("kblocks", C.c_int), ("tap", C.c_int), ("stride", C.c_int)]


class MegaLayer(C.Structure):
    _fields_ = [
        ("n_seg", C.c_int), ("seg", MegaSeg * MAX_SEGS),
        ("n_stage", C.c_int), ("NT", C.c_int), ("n_tiles_n", C.c_int),
        ("relu", C.c_int), ("round_out", C.c_int), ("up", C.c_int), ("Cout", C.c_int),
        ("P_m", C.c_int), ("T_out", C.c_int), ("n_rows", C.c_int),
        ("ld_out", C.c_int), ("P_store", C.c_int), ("T_store", C.c_int), ("c_off", C.c_int),
        ("is_heads", C.c_int), ("flag_base", C.c_int), ("out_map", C.c_int), ("k_atoms", C.c_int),
        ("w_tc", C.c_void_p), ("bias", C.c_void_p), ("out", C.c_void_p),
    ]


class MegaDep(C.Structure):
    _fields_ = [("first", C.c_int), ("count", C.c_int), ("target", C.c_int)]


class MegaJob(C.Structure):
    _fields_ = [("layer", C.c_int), ("m_tile", C.c_int), ("n_tile", C.c_int), ("n_dep", C.c_int),
                ("dep", MegaDep * MEGA_MAX_DEPS)]


class MegaArgs(C.Structure):
    _fields_ = [
        ("n_layers", C.c_int), ("n_jobs", C.c_int), ("n_flags", C.c_int), ("grid", C.c_int),
        ("layers", C.c_void_p), ("jobs", C.c_void_p), ("tmaps", C.c_void_p), ("sync", C.c_void_p),
        ("n_maps", C.c_int), ("reserved0", C.c_int),
        ("B", C.c_int), ("T", C.c_int), ("NH", C.c_int), ("NS", C.c_int),
        ("center_ref", C.c_void_p), ("mean_size", C.c_void_p),
        ("n_out", C.c_int), ("n_flag_out", C.c_int),
        ("outs", DecodeOut * MAX_PEERS), ("flag_out", C.c_void_p * MAX_PEERS),
        ("dbg_clocks", C.c_void_p),
    ]


class TrainSrc(C.Structure):
    _fields_ = [("raw", C.c_void_p), ("grad", C.c_void_p), ("sums", C.c_void_p), ("gamma", C.c_void_p),
                ("beta", C.c_void_p), ("count", C.c_double), ("Cstat", C.c_int), ("coff", C.c_int), ("relu", C.c_int),
                ("ld", C.c_int), ("T", C.c_int), ("up", C.c_int), ("cup", C.c_int), ("c0", C.c_int)]


class TrainSeg(C.Structure):
    _fields_ = [("src", TrainSrc), ("C", C.c_int), ("tap", C.c_int), ("stride", C.c_int), ("s_ci", C.c_int),
                ("w_off", C.c_longlong)]


class TrainLayer(C.Structure):
    _fields_ = [("B", C.c_int), ("T_out", C.c_int), ("n_seg", C.c_int), ("N", C.c_int), ("Cout", C.c_int),
                ("up", C.c_int), ("s_co", C.c_int), ("s_j", C.c_int), ("has_bn", C.c_int), ("relu", C.c_int),
                ("seg", TrainSeg * MAX_SEGS),
                ("W", C.c_void_p), ("dW", C.c_void_p), ("bias", C.c_void_p), ("dbias", C.c_void_p),
                ("Y", C.c_void_p), ("dA", C.c_void_p), ("sums", C.c_void_p), ("dsums", C.c_void_p),
                ("gamma", C.c_void_p), ("beta", C.c_void_p), ("dgamma", C.c_void_p), ("dbeta", C.c_void_p),
                ("run_mean", C.c_void_p), ("run_var", C.c_void_p)]


class TrainPool(C.Structure):
    _fields_ = [("B", C.c_int), ("T", C.c_int), ("K", C.c_int), ("C", C.c_int), ("V", C.c_int), ("ld_feat", C.c_int),
                ("Y", C.c_void_p), ("cnt", C.c_void_p), ("sums", C.c_void_p), ("gamma", C.c_void_p),
                ("beta", C.c_void_p), ("one_hot", C.c_void_p), ("feat", C.c_void_p), ("argmax", C.c_void_p),
                ("dfeat", C.c_void_p), ("dA", C.c_void_p)]


class LossArgs(C.Structure):
    _fields_ = [("B", C.c_int), ("T2", C.c_int), ("NH", C.c_int), ("NS", C.c_int), ("with_iou", C.c_int),
                ("reserved0", C.c_int),
                ("cls", C.c_void_p), ("reg", C.c_void_p), ("center_ref2", C.c_void_p),
                ("cls_label", C.c_void_p), ("size_class", C.c_void_p),
                ("box3d_center", C.c_void_p), ("box3d_heading", C.c_void_p), ("box3d_size", C.c_void_p),
                ("mean_size", C.c_void_p),
                ("w_box", C.c_float), ("w_head_reg", C.c_float), ("w_size_reg", C.c_float), ("w_corner", C.c_float),
                ("iou_thresh", C.c_float), ("reserved1", C.c_float),
                ("dcls", C.c_void_p), ("dreg", C.c_void_p), ("out", C.c_void_p), ("scratch", C.c_void_p)]


class InputArgs(C.Structure):
    _fields_ = [("B", C.c_int), ("N", C.c_int), ("num_scales", C.c_int), ("num_classes", C.c_int),
                ("T", C.c_int * MAX_SCALES), ("stride", C.c_double * MAX_SCALES),
                ("points", C.c_void_p), ("point_offsets", C.c_void_p), ("choice", C.c_void_p),
                ("frustum_angle", C.c_void_p), ("box2d", C.c_void_p), ("P", C.c_void_p), ("cls_index", C.c_void_p),
                ("point_cloud", C.c_void_p), ("centers", C.c_void_p * MAX_SCALES), ("one_hot", C.c_void_p),
                ("rot_angle", C.c_void_p)]


# name -> (restype, argtypes); kept in one table so tests can check every symbol of the header
_I, _F, _P = C.c_int, C.c_float, C.c_void_p
SIGNATURES = {
    "fcn_version": (_I, []),
    "fcn_last_error": (C.c_char_p, []),
    "fcn_query_depth_point_bn3": (_I, [_I, _I, _I, _F, _I, _P, _P, _P, _P, _P]),
    "fcn_query_depth_point_b3n": (_I, [_I, _I, _I, _F, _I, _P, _P, _P, _P, _P]),
    "fcn_group_rows": (_I, [C.POINTER(GroupArgs), _P]),
    "fcn_pointnet_tiles": (_I, [C.POINTER(PointnetArgs), _P]),
    "fcn_conv_gemm": (_I, [C.POINTER(ConvArgs), _P]),
    "fcn_mega_forward": (_I, [C.POINTER(MegaArgs), _P]),
    "fcn_decode_eval": (_I, [_I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "fcn_bct_to_btc": (_I, [_I, _I, _I, _I, _I, _P, _P, _P]),
    "fcn_btc_to_bct": (_I, [_I, _I, _I, _I, _I, _P, _P, _P]),
    "fcn_selftest_umma": (_I, [_I, _I, _P, _P, _P, _P]),
    "fcn_encode_activation_map": (_I, [_P, _P, _I, _I, _I, _I]),
    "fcn_encode_store_map": (_I, [_P, _P, _I, _I]),
    "fcn_train_forward": (_I, [C.POINTER(TrainLayer), _P, C.c_longlong, _P]),
    "fcn_train_workspace_floats": (C.c_longlong, [C.POINTER(TrainLayer)]),
    "fcn_train_backward": (_I, [C.POINTER(TrainLayer), _I, _P]),
    "fcn_train_pool": (_I, [C.POINTER(TrainPool), _I, _P]),
    "fcn_train_finalize": (_I, [_P, _I, _I, _P]),
    "fcn_adam_step": (_I, [_P, _P, _P, _P, C.c_longlong, _F, _F, _F, _F, _F, _I, _F, _P]),
    "fcn_rotate_nms_3d": (_I, [_I, _P, _P, _I, _F, _I, _P, _P, _I, _P, C.c_longlong, _P]),
    "fcn_rotate_nms_3d_workspace_bytes": (C.c_longlong, [_I, _I]),
    "fcn_rotate_nms_3d_max_dets": (_I, []),
    "fcn_rotate_nms_3d_max_seg_len": (_I, []),
    "fcn_det_loss": (_I, [C.POINTER(LossArgs), _P]),
    "fcn_build_inputs": (_I, [C.POINTER(InputArgs), _P]),
    "fcn_ipc_export": (_I, [_P, _P, C.POINTER(C.c_longlong)]),
    "fcn_ipc_open": (_I, [_P, C.POINTER(C.c_void_p)]),
    "fcn_ipc_close": (_I, [_P]),
    "fcn_rbbox_iou_3d_pair": (_I, [_I, _P, _P, _P, _F, _P, _P]),
}

_lib = None


def load():
    """Load (once) and return the ctypes handle.  Raises if the library was not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libfrustum_b200.so is missing (%s). Build it with "
                "`python -m frustum_convnet_b200.build` (or __graft_entry__.build()); there is no "
                "CPU or PyTorch fallback for the frustum hot path." % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(status: int, what: str = ""):
    if status != 0:
        msg = load().fcn_last_error().decode(errors="replace")
        raise RuntimeError("libfrustum_b200 %s failed (%d): %s" % (what, status, msg))


def call(name: str, *args):
    check(getattr(load(), name)(*args), name)
