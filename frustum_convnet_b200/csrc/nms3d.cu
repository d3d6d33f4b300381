// Rotated 3-D NMS on the device (SURVEY.md 8(f)-4): replaces the post-processing of test_net_det.py:126-152 ->
// ops/pybind11/rbbox_iou.py:294-311 `rotate_nms_3d_cc` (= the driver's `cube_nms`) -> nms_cpu.h:148-240
// `rotate_non_max_suppression_3d_cpu`, which today costs a device->host copy of every prediction, a Python loop
// per image / class and a CPU Boost polygon clip per box pair.
//
// Segments (= one image x class list of detections each) of any length; no box is ever left out:
//   1. corners of every box (boxes3d2corners, rbbox_iou.py:121-148) and its axis-aligned bounding cube;
//   2. rank by descending score (nms_order.cuh: the reference's scores.argsort()[::-1] with NaN first and ties
//      broken by the larger index, i.e. the reverse of a stable ascending sort);
//   3. suppression bit matrix in RANK order: bit (i, j) for j > i is set iff the bounding cubes overlap
//      (standup IoU > 0, nms_cpu.h:192) and the rotated 3-D IoU (box_iou.cuh, the same function as the train
//      metric, incl. its degenerate-ring rule) is >= thresh (nms_cpu.h:226-227);
//   4. greedy scan in rank order (keep i unless suppressed, then OR row i into the suppressed set);
//   5. the first top_k kept indices (rbbox_iou.py:311 `keep[:top_k]`) in rank order, count per segment.
// Short segments (<= NMS_MAX_DETS boxes) run all five steps in one CTA with everything in shared memory.  Longer
// ones take a global-memory path with a caller-provided workspace: one slot per long segment holding corners,
// cubes, the order and the n x ceil(n/32) bit matrix, built by a 2-D grid of (row block x 32-column word) CTAs,
// then scanned by one CTA per segment with the suppressed set in shared memory.
#include <algorithm>

#include "box_iou.cuh"
#include "common.cuh"
#include "nms_order.cuh"

namespace fcn {

constexpr int NMS_MAX_DETS = 512;
constexpr int NMS_WORDS = NMS_MAX_DETS / 32;
constexpr int NMS_THREADS = 256;

// corners in the reference order (rbbox_iou.py:131-147 == models/model_util.py:48-72)
__device__ __forceinline__ void box_to_corners(const float *d, float *c) {
    const float cx = d[0], cy = d[1], cz = d[2], l = d[3], w = d[4], h = d[5], r = d[6];
    const float cs = cosf(r), sn = sinf(r);
    const float xs[8] = {l / 2, l / 2, -l / 2, -l / 2, l / 2, l / 2, -l / 2, -l / 2};
    const float ys[8] = {h / 2, h / 2, h / 2, h / 2, -h / 2, -h / 2, -h / 2, -h / 2};
    const float zs[8] = {w / 2, -w / 2, -w / 2, w / 2, w / 2, -w / 2, -w / 2, w / 2};
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        c[3 * i + 0] = cs * xs[i] + sn * zs[i] + cx;
        c[3 * i + 1] = ys[i] + cy;
        c[3 * i + 2] = -sn * xs[i] + cs * zs[i] + cz;
    }
}

__global__ void __launch_bounds__(NMS_THREADS)
nms3d_kernel(const float *__restrict__ dets, const int *__restrict__ seg_offsets, int max_seg_len, float thresh,
             int top_k, int *__restrict__ keep, int *__restrict__ keep_count, int keep_stride) {
    extern __shared__ unsigned char nms_smem[];
    float *corners = (float *)nms_smem;                              // [n][24], in RANK order
    float *cube = corners + NMS_MAX_DETS * 24;                       // [n][6] min xyz, max xyz
    int *order = (int *)(cube + NMS_MAX_DETS * 6);                   // rank -> original index (inside the segment)
    unsigned *mask = (unsigned *)(order + NMS_MAX_DETS);             // [n][NMS_WORDS]
    const int seg = blockIdx.x;
    const int base = seg_offsets[seg], n = seg_offsets[seg + 1] - base;
    const int tid = threadIdx.x;
    if (n < 0 || n > max_seg_len) {                                  // never truncate: flag the segment
        if (tid == 0) keep_count[seg] = -1;
        return;
    }
    if (n > NMS_MAX_DETS) return;                                    // the global-memory path below owns it
    const float *d = dets + (size_t)base * 8;
    // ---- rank by descending score (nms_order.cuh)
    for (int i = tid; i < n; i += NMS_THREADS) {
        const float si = d[i * 8 + 7];
        int rank = 0;
        for (int j = 0; j < n; ++j) rank += nms_ranks_above(d[j * 8 + 7], j, si, i) ? 1 : 0;
        order[rank] = i;
    }
    __syncthreads();
    for (int r = tid; r < n; r += NMS_THREADS) {
        float c[24];
        box_to_corners(d + (size_t)order[r] * 8, c);
#pragma unroll
        for (int k = 0; k < 24; ++k) corners[r * 24 + k] = c[k];
        nms_bounding_cube(c, cube + r * 6);
    }
    for (int i = tid; i < n * NMS_WORDS; i += NMS_THREADS) mask[i] = 0u;
    __syncthreads();
    // ---- suppression bits for all pairs i < j (rank order)
    const int npairs = n * (n - 1) / 2;
    for (int p = tid; p < npairs; p += NMS_THREADS) {
        // p -> (i, j), i < j: row i holds n-1-i pairs
        int i = 0, rem = p;
        while (rem >= n - 1 - i) { rem -= n - 1 - i; ++i; }
        const int j = i + 1 + rem;
        if (!nms_cubes_overlap(cube + i * 6, cube + j * 6)) continue;
        float iou[2];
        rbbox_iou_pair(corners + i * 24, corners + j * 24, iou);
        if (iou[1] >= thresh) atomicOr(&mask[i * NMS_WORDS + (j >> 5)], 1u << (j & 31));
    }
    __syncthreads();
    // ---- greedy scan (one warp: lane = word of the suppressed set)
    if (tid < 32) {
        unsigned supp = 0u;                       // lane w holds word w of the suppressed bit set (n <= 512: 16 words)
        int kept = 0;
        for (int i = 0; i < n; ++i) {
            const unsigned word = __shfl_sync(0xffffffffu, supp, i >> 5);
            if ((word >> (i & 31)) & 1u) continue;
            if (kept < top_k && tid == 0) keep[(size_t)seg * keep_stride + kept] = base + order[i];
            ++kept;
            if (tid < NMS_WORDS) supp |= mask[i * NMS_WORDS + tid];
        }
        if (tid == 0) keep_count[seg] = min(kept, top_k);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Segments longer than NMS_MAX_DETS.  Workspace: long_seg[num_slots] (slot -> segment, -1 = unused), then
// num_slots slots of capacity `cap` (= the largest segment length the caller declared).
constexpr int NMS_LONG_MAX_DETS = 1 << 18;   // the scan keeps ceil(n/32) words in <= 32 KB of shared memory
constexpr int NMS_MAX_SLOTS = 65535;         // grid y/z limit
constexpr int NMS_ROW_BLOCK = 128;

__host__ __device__ inline size_t nms_align(size_t b) { return (b + 255) & ~(size_t)255; }
__host__ __device__ inline int nms_words(int cap) { return (cap + 31) / 32; }
__host__ __device__ inline size_t nms_slot_bytes(int cap) {
    return nms_align((size_t)cap * 24 * 4) + nms_align((size_t)cap * 6 * 4) + nms_align((size_t)cap * 4) +
           nms_align((size_t)cap * nms_words(cap) * 4);
}
__host__ __device__ inline size_t nms_workspace_bytes(int num_slots, int cap) {
    return nms_align((size_t)num_slots * 4) + (size_t)num_slots * nms_slot_bytes(cap);
}

struct NmsSlot {
    float *corners;    // [n][24], rank order
    float *cube;       // [n][6]
    int *order;        // rank -> index inside the segment
    unsigned *mask;    // [n][nms_words(cap)]: bit (i, j) = rank i suppresses rank j > i
};

__device__ inline NmsSlot nms_slot(unsigned char *ws, int num_slots, int cap, int k) {
    unsigned char *p = ws + nms_align((size_t)num_slots * 4) + (size_t)k * nms_slot_bytes(cap);
    NmsSlot s;
    s.corners = (float *)p;
    p += nms_align((size_t)cap * 24 * 4);
    s.cube = (float *)p;
    p += nms_align((size_t)cap * 6 * 4);
    s.order = (int *)p;
    p += nms_align((size_t)cap * 4);
    s.mask = (unsigned *)p;
    return s;
}

// One CTA: slot k of the workspace goes to the k-th segment with NMS_MAX_DETS < n <= cap (in segment order);
// a long segment that finds no slot is flagged with keep_count = -1.
__global__ void __launch_bounds__(1024)
nms3d_long_assign(const int *__restrict__ seg_offsets, int num_segments, int cap, int *__restrict__ long_seg,
                  int num_slots, int *__restrict__ keep_count) {
    __shared__ int warp_cnt[32];
    __shared__ int done;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int k = tid; k < num_slots; k += blockDim.x) long_seg[k] = -1;
    if (tid == 0) done = 0;
    __syncthreads();
    for (int s0 = 0; s0 < num_segments; s0 += blockDim.x) {
        const int s = s0 + tid;
        int n = 0;
        if (s < num_segments) n = seg_offsets[s + 1] - seg_offsets[s];
        const bool is_long = n > NMS_MAX_DETS && n <= cap;
        const unsigned bal = __ballot_sync(0xffffffffu, is_long);
        if (lane == 0) warp_cnt[warp] = __popc(bal);
        __syncthreads();
        int slot = done + __popc(bal & ((1u << lane) - 1u));
        for (int w = 0; w < warp; ++w) slot += warp_cnt[w];
        if (is_long) {
            if (slot < num_slots) long_seg[slot] = s;
            else keep_count[s] = -1;
        }
        __syncthreads();
        if (tid == 0)
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) done += warp_cnt[w];
        __syncthreads();
    }
}

// grid (ceil(cap / NMS_THREADS), num_slots): rank, corners and bounding cube of every box, stored in rank order
__global__ void __launch_bounds__(NMS_THREADS)
nms3d_long_boxes(const float *__restrict__ dets, const int *__restrict__ seg_offsets, unsigned char *ws,
                 int num_slots, int cap) {
    const int k = blockIdx.y, seg = ((const int *)ws)[k];
    if (seg < 0) return;
    const int base = seg_offsets[seg], n = seg_offsets[seg + 1] - base;
    const int i = blockIdx.x * NMS_THREADS + threadIdx.x;
    if (i >= n) return;
    const NmsSlot sl = nms_slot(ws, num_slots, cap, k);
    const float *d = dets + (size_t)base * 8;
    const float si = d[(size_t)i * 8 + 7];
    int rank = 0;
    for (int j = 0; j < n; ++j) rank += nms_ranks_above(d[(size_t)j * 8 + 7], j, si, i) ? 1 : 0;
    float c[24];
    box_to_corners(d + (size_t)i * 8, c);
#pragma unroll
    for (int q = 0; q < 24; ++q) sl.corners[(size_t)rank * 24 + q] = c[q];
    nms_bounding_cube(c, sl.cube + (size_t)rank * 6);
    sl.order[rank] = i;
}

// grid (ceil(cap / NMS_ROW_BLOCK), nms_words(cap), num_slots): word w of rows [r0, r0 + NMS_ROW_BLOCK), one
// row per thread against the 32 columns of the word staged in shared memory.  The scan reads row i from word
// i/32 on, so a CTA whose columns all lie below its first row writes nothing.
__global__ void __launch_bounds__(NMS_ROW_BLOCK)
nms3d_long_mask(const int *__restrict__ seg_offsets, unsigned char *ws, int num_slots, int cap, float thresh) {
    __shared__ float col_corners[32 * 24];
    __shared__ float col_cube[32 * 6];
    const int k = blockIdx.z, seg = ((const int *)ws)[k];
    if (seg < 0) return;
    const int n = seg_offsets[seg + 1] - seg_offsets[seg];
    const int r0 = blockIdx.x * NMS_ROW_BLOCK, w = blockIdx.y, c0 = w * 32;
    if (r0 >= n || c0 >= n || c0 + 32 <= r0) return;                // uniform per CTA
    const NmsSlot sl = nms_slot(ws, num_slots, cap, k);
    const int tid = threadIdx.x;
    for (int t = tid; t < 32 * 24; t += NMS_ROW_BLOCK)
        if (c0 + t / 24 < n) col_corners[t] = sl.corners[(size_t)c0 * 24 + t];
    for (int t = tid; t < 32 * 6; t += NMS_ROW_BLOCK)
        if (c0 + t / 6 < n) col_cube[t] = sl.cube[(size_t)c0 * 6 + t];
    __syncthreads();
    const int i = r0 + tid;
    if (i >= n) return;
    float ci[24], cb[6];
#pragma unroll
    for (int q = 0; q < 24; ++q) ci[q] = sl.corners[(size_t)i * 24 + q];
#pragma unroll
    for (int q = 0; q < 6; ++q) cb[q] = sl.cube[(size_t)i * 6 + q];
    unsigned bits = 0u;
    for (int jj = 0; jj < 32; ++jj) {
        const int j = c0 + jj;
        if (j <= i || j >= n) continue;
        if (!nms_cubes_overlap(cb, col_cube + jj * 6)) continue;
        float iou[2];
        rbbox_iou_pair(ci, col_corners + jj * 24, iou);
        if (iou[1] >= thresh) bits |= 1u << jj;
    }
    sl.mask[(size_t)i * nms_words(cap) + w] = bits;
}

// one CTA per slot: greedy scan in rank order, the suppressed set in shared memory
__global__ void __launch_bounds__(NMS_THREADS)
nms3d_long_scan(const int *__restrict__ seg_offsets, unsigned char *ws, int num_slots, int cap, int top_k,
                int *__restrict__ keep, int *__restrict__ keep_count, int keep_stride) {
    extern __shared__ unsigned nms_supp[];
    const int k = blockIdx.x, seg = ((const int *)ws)[k];
    if (seg < 0) return;
    const int base = seg_offsets[seg], n = seg_offsets[seg + 1] - base;
    const NmsSlot sl = nms_slot(ws, num_slots, cap, k);
    const int tid = threadIdx.x, words = nms_words(n), stride = nms_words(cap);
    for (int w = tid; w < words; w += NMS_THREADS) nms_supp[w] = 0u;
    __syncthreads();
    int kept = 0;
    for (int i = 0; i < n; ++i) {
        if ((nms_supp[i >> 5] >> (i & 31)) & 1u) continue;           // uniform: read after the last barrier
        if (kept < top_k && tid == 0) keep[(size_t)seg * keep_stride + kept] = base + sl.order[i];
        ++kept;
        __syncthreads();                                              // every thread has read bit i
        const unsigned *row = sl.mask + (size_t)i * stride;
        for (int w = (i >> 5) + tid; w < words; w += NMS_THREADS) nms_supp[w] |= row[w];
        __syncthreads();
    }
    if (tid == 0) keep_count[seg] = min(kept, top_k);
}

}  // namespace fcn

using namespace fcn;

extern "C" long long fcn_rotate_nms_3d_workspace_bytes(int num_long_segments, int max_seg_len) {
    FCN_REQUIRE(num_long_segments >= 0 && max_seg_len >= 0, "negative size");
    FCN_REQUIRE(max_seg_len <= NMS_LONG_MAX_DETS, "max_seg_len above fcn_rotate_nms_3d_max_seg_len()");
    if (num_long_segments == 0 || max_seg_len <= NMS_MAX_DETS) return 0;
    return (long long)nms_workspace_bytes(num_long_segments, max_seg_len);
}

extern "C" int fcn_rotate_nms_3d(int num_segments, const float *dets, const int32_t *seg_offsets, int max_seg_len,
                                 float thresh, int top_k, int32_t *keep, int32_t *keep_count, int keep_stride,
                                 void *workspace, long long workspace_bytes, fcn_stream_t stream) {
    FCN_REQUIRE(num_segments >= 0 && top_k >= 1 && keep_stride >= 1, "bad sizes");
    FCN_REQUIRE(top_k <= keep_stride, "top_k > keep_stride (keep rows would overflow)");
    FCN_REQUIRE(max_seg_len >= 0, "negative max_seg_len");
    FCN_REQUIRE(max_seg_len <= NMS_LONG_MAX_DETS, "max_seg_len above fcn_rotate_nms_3d_max_seg_len()");
    if (num_segments == 0) return FCN_OK;
    FCN_REQUIRE(dets && seg_offsets && keep && keep_count, "NULL pointer");
    int num_slots = 0;
    if (max_seg_len > NMS_MAX_DETS) {
        FCN_REQUIRE(workspace && workspace_bytes >= (long long)nms_workspace_bytes(1, max_seg_len),
                    "segments longer than fcn_rotate_nms_3d_max_dets() need a workspace "
                    "(fcn_rotate_nms_3d_workspace_bytes)");
        FCN_REQUIRE(((uintptr_t)workspace & 255u) == 0, "workspace must be 256-byte aligned");
        const long long slot = (long long)nms_slot_bytes(max_seg_len);
        num_slots = (int)std::min<long long>(std::min(num_segments, NMS_MAX_SLOTS), workspace_bytes / slot);
        while (num_slots > 0 && (long long)nms_workspace_bytes(num_slots, max_seg_len) > workspace_bytes) --num_slots;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t smem = (size_t)NMS_MAX_DETS * (24 + 6) * 4 + NMS_MAX_DETS * 4 + (size_t)NMS_MAX_DETS * NMS_WORDS * 4;
    FCN_CUDA(cudaFuncSetAttribute(nms3d_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    nms3d_kernel<<<num_segments, NMS_THREADS, smem, st>>>(dets, seg_offsets, max_seg_len, thresh, top_k, keep,
                                                          keep_count, keep_stride);
    FCN_LAUNCH_CHECK();
    if (num_slots == 0) return FCN_OK;
    unsigned char *ws = (unsigned char *)workspace;
    const int cap = max_seg_len;
    nms3d_long_assign<<<1, 1024, 0, st>>>(seg_offsets, num_segments, cap, (int *)ws, num_slots, keep_count);
    FCN_LAUNCH_CHECK();
    nms3d_long_boxes<<<dim3((cap + NMS_THREADS - 1) / NMS_THREADS, num_slots), NMS_THREADS, 0, st>>>(
        dets, seg_offsets, ws, num_slots, cap);
    FCN_LAUNCH_CHECK();
    nms3d_long_mask<<<dim3((cap + NMS_ROW_BLOCK - 1) / NMS_ROW_BLOCK, nms_words(cap), num_slots), NMS_ROW_BLOCK, 0,
                      st>>>(seg_offsets, ws, num_slots, cap, thresh);
    FCN_LAUNCH_CHECK();
    nms3d_long_scan<<<num_slots, NMS_THREADS, (size_t)nms_words(cap) * 4, st>>>(seg_offsets, ws, num_slots, cap, top_k,
                                                                               keep, keep_count, keep_stride);
    FCN_LAUNCH_CHECK();
    return FCN_OK;
}

extern "C" int fcn_rotate_nms_3d_max_dets(void) { return NMS_MAX_DETS; }
extern "C" int fcn_rotate_nms_3d_max_seg_len(void) { return NMS_LONG_MAX_DETS; }
