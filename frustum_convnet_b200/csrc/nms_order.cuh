// Score order and bounding-cube test of the rotated 3-D NMS (nms3d.cu), as plain C++ behind FCN_HD so that
// tests/test_nms_cpu.py can compile the same functions with g++ and check them against numpy without a GPU.
#pragma once

#include "box_iou.cuh"

namespace fcn {

// Box j (score sj) ranks above box i (score si).  The order is np.argsort(scores, kind="stable")[::-1], the
// order of the reference's `scores.argsort()[::-1]` made deterministic for ties: NaN scores first (numpy sorts
// them last), then descending score, then, among equal scores or among NaNs, the larger index first.  -0.0 and
// +0.0 are equal.  It is a strict total order on (NaN-ness, score, index), so counting the boxes that rank above
// box i gives every box a distinct rank in [0, n).
FCN_HD bool nms_ranks_above(float sj, int j, float si, int i) {
    const bool nj = sj != sj, ni = si != si;
    if (nj != ni) return nj;
    if (!nj && sj != si) return sj > si;
    return j > i;
}

// Axis-aligned bounding cube [min xyz, max xyz] of a box's 8 corners.  Corners containing a NaN give the EMPTY
// cube (+inf, -inf), which overlaps nothing: such a box is never suppressed and suppresses nothing, as in the
// reference, whose standup IoU of a NaN box is NaN and fails its `> 0` test (nms_cpu.h:192).
FCN_HD void nms_bounding_cube(const float *c, float *cube) {
    float mn[3] = {c[0], c[1], c[2]}, mx[3] = {c[0], c[1], c[2]};
    bool nan = false;
    for (int i = 0; i < 8; ++i) {
        for (int k = 0; k < 3; ++k) {
            const float v = c[3 * i + k];
            nan |= v != v;
            mn[k] = mn[k] < v ? mn[k] : v;
            mx[k] = mx[k] > v ? mx[k] : v;
        }
    }
    for (int k = 0; k < 3; ++k) {
        cube[k] = nan ? __builtin_huge_valf() : mn[k];
        cube[3 + k] = nan ? -__builtin_huge_valf() : mx[k];
    }
}

// standup IoU > 0 <=> the bounding cubes overlap with positive volume (rbbox_iou.py:62-96)
FCN_HD bool nms_cubes_overlap(const float *a, const float *b) {
    for (int k = 0; k < 3; ++k) {
        const float hi = a[3 + k] < b[3 + k] ? a[3 + k] : b[3 + k];
        const float lo = a[k] > b[k] ? a[k] : b[k];
        if (!(hi - lo > 0.f)) return false;
    }
    return true;
}

}  // namespace fcn
