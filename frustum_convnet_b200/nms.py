"""Rotated 3-D NMS on the device - drop-in for the reference's ``cube_nms`` (= ``rotate_nms_3d_cc``,
ops/pybind11/rbbox_iou.py:294-311, imported by train/test_net_det.py:44 and called at :140).

    keep = cube_nms(dets_for_nms, threshold)                   # one list, like the reference (CUDA tensor in)
    keep, counts = rotate_nms_3d_batched(dets, offsets, thr)   # every image x class list of a batch in ONE launch

`dets`: (n, 8) rows [cx, cy, cz, l, w, h, ry, score]; lists of any length.  No CPU fallback: CPU tensors
raise."""
from __future__ import annotations

import torch

from . import _lib


def rotate_nms_3d_batched(dets: torch.Tensor, seg_offsets: torch.Tensor, thresh: float, top_k: int = 300):
    """-> (keep (S, top_k) int32 global row indices in descending-score order, counts (S,) int32).

    Lists of any length: every row of a segment is considered.  The segment lengths are read on the host (one
    device->host copy when `seg_offsets` lives on the device) to size the workspace of lists longer than
    ``fcn_rotate_nms_3d_max_dets()`` rows; counts are checked on the host afterwards (one synchronisation)."""
    if not dets.is_cuda:
        raise RuntimeError("rotate_nms_3d: CUDA tensors required (there is no CPU fallback)")
    assert dets.dim() == 2 and dets.shape[1] == 8, "dets must be (n, 8): cx, cy, cz, l, w, h, ry, score"
    d = dets.detach().to(torch.float32).contiguous()
    off_host = seg_offsets.detach().to(device="cpu", dtype=torch.int64)
    lens = off_host[1:] - off_host[:-1]
    if lens.numel() and int(lens.min()) < 0:
        raise ValueError("rotate_nms_3d: seg_offsets must be non-decreasing")
    if off_host.numel() and (int(off_host[0]) < 0 or int(off_host[-1]) > d.shape[0]):
        raise ValueError("rotate_nms_3d: seg_offsets out of range of dets")
    off = seg_offsets.to(device=d.device, dtype=torch.int32).contiguous()
    S = off.numel() - 1
    keep = torch.full((max(S, 0), top_k), -1, dtype=torch.int32, device=d.device)
    cnt = torch.zeros(max(S, 0), dtype=torch.int32, device=d.device)
    if S > 0:
        lib = _lib.load()
        max_len = int(lens.max())
        n_long = int((lens > lib.fcn_rotate_nms_3d_max_dets()).sum())
        ws_bytes = lib.fcn_rotate_nms_3d_workspace_bytes(n_long, max_len)
        if ws_bytes < 0:
            _lib.check(int(ws_bytes), "fcn_rotate_nms_3d_workspace_bytes")
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=d.device) if ws_bytes else None
        with torch.cuda.device(d.device):
            _lib.call("fcn_rotate_nms_3d", S, d.data_ptr(), off.data_ptr(), max_len, float(thresh), int(top_k),
                      keep.data_ptr(), cnt.data_ptr(), int(top_k), ws.data_ptr() if ws is not None else None,
                      ws_bytes, torch.cuda.current_stream(d.device).cuda_stream)
        bad = torch.nonzero(cnt < 0).flatten().tolist()
        if bad:
            raise RuntimeError("rotate_nms_3d: segments %s were not processed (keep_count = -1)" % bad[:8])
    return keep, cnt


def rotate_nms_3d_cc(dets: torch.Tensor, thresh: float, top_k: int = 300):
    """Same contract as the reference function of that name: indices to keep (descending score)."""
    n = dets.shape[0]
    if n == 0:
        return []
    off = torch.tensor([0, n], dtype=torch.int32)
    keep, cnt = rotate_nms_3d_batched(dets, off, thresh, top_k)
    return keep[0, : int(cnt[0])].tolist()


cube_nms = rotate_nms_3d_cc
