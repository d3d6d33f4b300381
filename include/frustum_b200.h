/*
 * frustum_b200.h — C ABI of libfrustum_b200.so (sm_100a).
 *
 * Drop-in boundary for the per-frustum hot path of Gorilla-Lab-SCUT/frustum-convnet:
 *   ops/query_depth_point  ->  models/det_base.PointNetFeat  ->  ConvFeatNet  ->  heads/decode.
 *
 * Conventions (SURVEY.md section 8(b)):
 *   - plain pointers + sizes only; every pointer is a DEVICE pointer unless the name says host;
 *   - the caller owns every buffer (the reference allocates outputs in Python and passes them
 *     in: ops/query_depth_point/query_depth_point.py:36-39); the library allocates nothing and
 *     keeps no state between calls except a thread-local error string;
 *   - `stream` is a cudaStream_t passed as void* (the reference launches on ATen's current
 *     stream: query_depth_point_cuda_kernel.cu:72); all calls are asynchronous;
 *   - return 0 on success, <0 on error (no C++ exception crosses the ABI; the reference raised
 *     through AT_ASSERTM / THCudaCheck: query_depth_point_cuda.cpp:5-10, ..._kernel.cu:85);
 *     fcn_last_error() returns the message of the last failing call on this thread.
 */
#ifndef FRUSTUM_B200_H_
#define FRUSTUM_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FCN_OK 0
#define FCN_ERR_INVALID (-1)
#define FCN_ERR_CUDA (-2)

#define FCN_MAX_SCALES 8
#define FCN_MAX_SEGS 4

#if defined(__GNUC__)
#define FCN_API __attribute__((visibility("default")))
#else
#define FCN_API
#endif

typedef void *fcn_stream_t;

FCN_API int fcn_version(void);
FCN_API const char *fcn_last_error(void);

/* ------------------------------------------------------------------------------------------
 * (1) Grouping op.  Replaces query_depth_point_cuda.forward(b,n,m,dis_z,nsample,xyz1,xyz2,idx,
 *     pts_cnt) bound at ops/query_depth_point/query_depth_point_cuda.cpp:25-50 (kernel
 *     query_depth_point_cuda_kernel.cu:16-86).  Same argument order and meaning.
 *     idx: (b,m,nsample) int64, pts_cnt: (b,m) int32; both fully written (no pre-zero needed).
 *     _bn3  : xyz1 (b,n,3), xyz2 (b,m,3)   — the layout the reference kernel receives.
 *     _b3n  : xyz1 (b,3,n), xyz2 (b,3,m)   — the layout QueryDepthPoint.forward receives
 *             (query_depth_point.py:18-19); saves the two permute().contiguous() copies (:29-30).
 * ------------------------------------------------------------------------------------------ */
FCN_API int fcn_query_depth_point_bn3(int b, int n, int m, float dis_z, int nsample, const float *xyz1,
                              const float *xyz2, int64_t *idx, int32_t *pts_cnt,
                              fcn_stream_t stream);
FCN_API int fcn_query_depth_point_b3n(int b, int n, int m, float dis_z, int nsample, const float *xyz1,
                              const float *xyz2, int64_t *idx, int32_t *pts_cnt,
                              fcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (2) Fused grouping -> row records (feeds the PointNet tile kernels; replaces
 *     QueryDepthPoint + torch.gather + "grouped_pc - new_pc", models/det_base.py:68-80,
 *     for all scales of PointNetFeat in ONE launch).
 *
 *     For every (frustum b, scale s) the T_s sections are scanned; section t contributes
 *     cnt = min(hits, K_s) rows (unique_rows=1) or exactly K_s rows with the reference's
 *     back-fill duplicates (unique_rows=0).  A row record is float4 {x-cx, y-cy, z-cz, bits(t)}
 *     (bits(t) = section index as int; sign bit set when the section is empty/masked).
 *     Rows of (b,s) are stored contiguously at rows[s] + b*row_cap[s]; tiles of `tile_rows`
 *     rows are appended to tiles[s] (int4 {b, row0, nrows, 0}) and counted in ntiles[s].
 *     Side outputs: cnt[s] (B,T_s) int32; feat[s] (B,T_s,ld_feat[s]) fp32 position-major is
 *     zero-filled and its one-hot channels [c3[s], c3[s]+num_vec) are written (det_base.py:145-157).
 *     idx_scratch[s] receives the selected point indices (the valid prefix of the reference idx).
 *     `ntiles` (int32[FCN_MAX_SCALES]) is reset by the call itself.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int num_scales, B, N, num_vec, tile_rows, unique_rows;
    const float *pc;                        /* (B,3,N) */
    const float *one_hot;                   /* (B,num_vec) or NULL */
    const float *centers[FCN_MAX_SCALES];   /* (B,3,T_s) */
    int T[FCN_MAX_SCALES], K[FCN_MAX_SCALES];
    float dis_z[FCN_MAX_SCALES];
    int c3[FCN_MAX_SCALES], ld_feat[FCN_MAX_SCALES];
    int row_cap[FCN_MAX_SCALES];            /* rows reserved per frustum (>= T_s*K_s) */
    int tile_cap[FCN_MAX_SCALES];           /* capacity of tiles[s] */
    void *rows[FCN_MAX_SCALES];             /* float4[B*row_cap] */
    int32_t *cnt[FCN_MAX_SCALES];           /* (B,T_s) */
    float *feat[FCN_MAX_SCALES];            /* (B,T_s,ld_feat) or NULL */
    void *tiles[FCN_MAX_SCALES];            /* int4[tile_cap] */
    int32_t *idx_scratch[FCN_MAX_SCALES];   /* (B,T_s,K_s) int32: first min(hits,K) point indices */
    int feat_pitch[FCN_MAX_SCALES];         /* rows per frustum of feat[s] (>= T_s; 0 means T_s) */
    int32_t *ntiles;                        /* int32[FCN_MAX_SCALES] */
    int force_scan;                         /* 1: section-scan kernel pair instead of the bit-matrix kernel (A/B) */
} fcn_group_args;
FCN_API int fcn_group_rows(const fcn_group_args *args, fcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (3) PointNet tile kernel: three folded (conv1x1 + BN + ReLU) layers on row tiles and the
 *     max over the rows of each section.  Replaces models/det_base.py:95-101 + torch.max(-1)
 *     (:134-143) for one scale.
 *     Weights are BN-folded and packed by the host side (see INTEGRATION.md):
 *       w1t (3,C1)  w2t (C1,C2)  w3t (C2,C3)  fp32 row-major [cin][cout];  b1,b2,b3 fp32.
 *     pooled   : out = feat (B,T,ld_feat) position-major, combined with atomic max (feat must be
 *                zero-initialised, which fcn_group_rows does).
 *     unpooled : out = (B,C3,T,K) channel-first un-pooled masked tensor — the return value of
 *                PointNetModule.forward (det_base.py:103); rows must come from unique_rows=0.
 *     precision: 0 = fp32 SIMT, 1 = TF32 tensor cores (tcgen05) for the C1->C2->C3 layers,
 *                2 = same on 2-CTA clusters (cta_group::2, M = 256; scales with C1 >= 128; weight images
 *                    packed with n-chunks C2 / 256, see INTEGRATION.md).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int C1, C2, C3, T, K, ld_feat, row_cap, tile_rows, unpooled, precision, B;
    const void *rows;       /* float4 records of this scale */
    const void *tiles;      /* int4 tile table */
    const int32_t *ntiles;  /* device scalar */
    int max_tiles;          /* host upper bound used to size the grid */
    const float *w1t, *b1, *w2t, *b2, *w3t, *b3;
    const void *w2_tc, *w3_tc;  /* tensor-core packed images (precision=1), else NULL */
    float *out;
    long long *dbg_clocks;  /* optional (NULL): CTA 0 dumps pipeline timestamps (diagnostics) */
    int feat_pitch;         /* rows per frustum of the pooled feature map (>= T; 0 means T) */
} fcn_pointnet_args;
FCN_API int fcn_pointnet_tiles(const fcn_pointnet_args *args, fcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (4) 1-D conv / transposed conv / 1x1 conv + folded BN + optional ReLU as an implicit GEMM on
 *     position-major activations.  Replaces every Conv1d/DeConv1d block of ConvFeatNet
 *     (models/det_base.py:167-224, factories models/common.py:38-63), the torch.cat calls
 *     (multi-segment A operand) and the two heads (det_base.py:367-368).
 *       precision: 0 fp32 SIMT | 1,2 TF32 tcgen05 with cp.async gather (N tile 128|64) |
 *                  3,4 TF32 tcgen05 fully TMA-fed (N tile 128|64, needs `tmaps`)
 *       out[b, t*up + j, c_off + co] = act( sum_seg sum_c src[b, t*stride + tap, c] * W + bias )
 *     K is the concatenation of the segments, each padded to a multiple of 32 (zero weights); K_pad
 *     is that sum, optionally rounded up to a multiple of 64 (required by the tensor-core variants).
 *     wt: [K_pad][n_cols] fp32 (n_cols = up*Cout rounded up to 64), bias: [n_cols].
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    const float *src;
    int ld, C, T_src, tap, stride;
    int pitch;   /* rows per frustum of src (>= T_src; 0 means T_src).  Padded maps (pitch > T_src, pad rows
                    kept zero) let the GEMM run over the flattened (frustum, position) rows: the kernel
                    taps then read a zero pad row instead of the neighbouring frustum. */
} fcn_conv_seg;
typedef struct {
    int B, T_out, n_seg;
    fcn_conv_seg seg[FCN_MAX_SEGS];
    int K_pad, n_cols, Cout, up, relu, precision;
    const float *wt, *bias;
    const void *w_tc;
    float *out;
    int ld_out, T_store, c_off;
    int round_out;   /* 1: round outputs to TF32 (cvt.rna) because a tensor-core GEMM consumes them */
    long long *dbg_clocks; /* optional (NULL): CTA (0,0) dumps per-K-block pipeline timestamps, 8 per K block */
    const void *tmaps;     /* HOST pointer to n_seg 128-byte tensor maps (precision 3|4), see below */
    int P_m;               /* pitch of the GEMM row space: row r = b*P_m + t, valid iff t < T_out (0: T_out) */
    int P_store;           /* rows per frustum of `out` (>= T_store; 0 means T_store) */
} fcn_conv_args;
FCN_API int fcn_conv_gemm(const fcn_conv_args *args, fcn_stream_t stream);

/* TMA descriptor of a position-major activation map (B,T,ld) fp32 for the fully TMA-fed conv GEMM
 * (precision 3 = N tile 128, 4 = N tile 64): 3-D tensor (channel, position, frustum), box
 * 32 x 128 x 1 with 128-byte swizzle, position step t_stride (1, or 2 for the stride-2 convs).
 * The kernel addresses the GEMM rows as ONE flattened sequence, so encode the map with B = 1 and
 * T = (number of frustums) x pitch of the padded activation map.
 * Writes 128 bytes to HOST memory; pass an array of them (one per segment) in fcn_conv_args.tmaps. */
FCN_API int fcn_encode_activation_map(void *out_map_128B, const float *base, int B, int T, int ld,
                                      int t_stride);

/* ------------------------------------------------------------------------------------------
 * (5) Eval decode of the head logits.  Replaces models/det_base.py:376-411 and
 *     models/box_transform.py:5-12,28-41.
 *     logits: (B, pitch >= T, ld) rows = [cls0, cls1, center(3), heading scores(NH), heading res(NH),
 *     size scores(NS), size res(NS*3)];  center_ref: (B,3,T) channel-first;  mean_size (NS,3).
 * ------------------------------------------------------------------------------------------ */
FCN_API int fcn_decode_eval(int B, int T, int pitch, int ld, int num_heading_bin, int num_size, const float *logits,
                    const float *center_ref, const float *mean_size, float *cls_probs,
                    float *center, float *heading, float *size, float *heading_probs,
                    float *size_probs, fcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (5b) Persistent FCN kernel: every fcn_conv_gemm layer of ConvFeatNet + heads (4) and the eval decode (5) of
 *      one forward in ONE launch (models/det_base.py:196-224,367-411).  The host describes the network as
 *        layers : per layer the A segments (tensor-map index, 32-channel blocks, kernel tap, stride), the
 *                 packed TF32 weight image / bias, the output slice and the index of its completion counters;
 *        jobs   : one [128 rows x NT columns] output tile each, in TOPOLOGICAL order (a job depends only on jobs
 *                 with a smaller index), with the counters (first, count, target) it has to wait for;
 *        tmaps  : HOST array of n_maps (<= 48) 128-byte tensor maps - A-operand load maps
 *                 (fcn_encode_activation_map) and epilogue store maps (fcn_encode_store_map); copied into the
 *                 kernel parameters at launch, like the HOST layer table;
 *        sync   : DEVICE int32[4 + n_flags], zero-initialised ONCE by the caller; [0] job counter, [1] finished
 *                 CTAs, [2] epoch (forwards completed), [4..] per-(layer,row-tile) completion counters.  The
 *                 kernel resets [0],[1],[4..] itself at the end of every forward.
 *      Persistent CTAs fetch jobs with an atomic counter (deadlock-free under any co-residency, see fcn_mega.cu).
 *      The heads layer (is_heads) stores the logits row and decodes it in place into `n_out` output sets:
 *      outs[0] is the local 6-tuple block, outs[1..] are peer buffers (mapped NVLink peer memory) - the
 *      multi-GPU result exchange without a collective; flag_out[i] (may be NULL) receives the epoch number when
 *      the forward is complete (system-scope release).
 * ------------------------------------------------------------------------------------------ */
#define FCN_MAX_PEERS 8
#define FCN_MEGA_MAX_DEPS 4
typedef struct {
    float *cls_probs, *center, *heading, *size, *heading_probs, *size_probs;
} fcn_decode_out;
typedef struct {
    int map_idx, kblocks, tap, stride;
} fcn_mega_seg;
typedef struct {
    int n_seg;
    fcn_mega_seg seg[FCN_MAX_SEGS];
    int n_stage;                 /* K stages per tile: K_pad / (32 * k_atoms) */
    int NT, n_tiles_n;           /* N tile (256 | 128 | 64) and their number */
    int relu, round_out, up, Cout;
    int P_m, T_out, n_rows;      /* GEMM row space: row r = b*P_m + t, valid iff t < T_out; n_rows = B*P_m */
    int ld_out, P_store, T_store, c_off;
    int is_heads, flag_base;
    int out_map;                 /* tensor map of the epilogue's TMA store (fcn_encode_store_map); unused for heads */
    int k_atoms;                 /* 32-wide K atoms per stage: 2 (NT <= 128) or 1 (NT = 256); 0 reads as 2 */
    const void *w_tc;            /* packed stage images, N-tile major */
    const float *bias;
    float *out;
} fcn_mega_layer;
typedef struct {
    int layer, m_tile, n_tile, n_dep;
    struct { int first, count, target; } dep[FCN_MEGA_MAX_DEPS];
} fcn_mega_job;
typedef struct {
    int n_layers, n_jobs, n_flags, grid;   /* grid: persistent CTAs (0 = one per SM) */
    const fcn_mega_layer *layers;          /* HOST, n_layers (<= 24) records */
    const fcn_mega_job *jobs;              /* device */
    const void *tmaps;                     /* HOST, n_maps x 128 bytes */
    int32_t *sync;                         /* device */
    int n_maps, reserved0;
    int B, T, NH, NS;                      /* decode: frustums, positions (T2), heading bins, size clusters */
    const float *center_ref, *mean_size;
    int n_out, n_flag_out;
    fcn_decode_out outs[FCN_MAX_PEERS];
    int32_t *flag_out[FCN_MAX_PEERS];
    long long *dbg_clocks;                 /* optional (NULL): CTA 0 dumps 16 timestamps per job (first 64 jobs) */
} fcn_mega_args;
FCN_API int fcn_mega_forward(const fcn_mega_args *args, fcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (5c) Multi-GPU plumbing for the result exchange by peer stores (one process per GPU): export a caller-owned
 *      device buffer as a CUDA-IPC handle (+ the byte offset of `dev_ptr` inside its allocation), map an
 *      exported buffer into this process for the current device, unmap it.  The mapped address (+ offset) is what
 *      fcn_mega_args.outs[1..] / flag_out[] take.  handle = 64 bytes of HOST memory.
 * ------------------------------------------------------------------------------------------ */
FCN_API int fcn_ipc_export(const void *dev_ptr, void *handle_64B, long long *offset_bytes);
FCN_API int fcn_ipc_open(const void *handle_64B, void **base_out);
FCN_API int fcn_ipc_close(void *base);

/* TMA descriptor for the epilogue stores of the persistent FCN kernel: a position-major map viewed as
 * (inner = up*ld floats, rows = flattened GEMM rows), box 32 x 32 with 128-byte swizzle.  For a transposed conv
 * with `up` taps the GEMM row r, tap j lands on output row r*up + j: one tensor row = `up` consecutive output
 * rows, the tap selects the inner offset j*ld.  Writes 128 bytes to HOST memory. */
FCN_API int fcn_encode_store_map(void *out_map_128B, const float *base, int rows, int inner);

/* ------------------------------------------------------------------------------------------
 * (7) Training step (config 5, cfgs/refine_car.yaml): PointNetDet in train() mode on hand-written kernels.
 *     Replaces the PyTorch/cuDNN autograd graph of models/det_base.py:62-224,367-368 (+ models/common.py:38-63
 *     BatchNorm in batch-statistics mode) and the optimizer step (train/train_net_det.py:121-128,322-323).
 *     All tensors are dense position-major fp32 [rows, channels]; rows = (frustum, position).  A layer is
 *         Y = act(X) * W (+bias)          act = the PRODUCER's BatchNorm (batch statistics) + ReLU, applied while
 *                                         the operand is loaded (no post-activation tensor exists)
 *     and its backward applies the BatchNorm/ReLU backward on the fly as well (see csrc/train.cu).
 *     Weights / gradients are addressed in the PARAMETER layout through strides:
 *         W[segment channel c, column n] = W + w_off + c*s_ci + (n % Cout)*s_co + (n / Cout)*s_j
 *     fcn_train_src: how a consumer sees a source tensor: position p of frustum b, channel c ->
 *         raw[(b*T + p/up)*ld + c0 + (p%up)*cup + c]   (up > 1: un-shuffled output of a transposed conv)
 *     `sums` (fp64 [2*Cstat]: Sum(y), Sum(y^2)) non-NULL = the source is a BN layer's raw output: apply
 *     gamma*(y-mean)*invstd+beta (channel (coff + c) % Cstat, `count` samples per channel) and ReLU if `relu`.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    const float *raw;
    float *grad;                 /* gradient w.r.t. the POST-activation values, same layout as raw (may be NULL) */
    const double *sums;
    const float *gamma, *beta;
    double count;
    int Cstat, coff, relu;
    int ld, T, up, cup, c0;
} fcn_train_src;
typedef struct {
    fcn_train_src src;
    int C, tap, stride, s_ci;
    long long w_off;
} fcn_train_seg;
typedef struct {
    int B, T_out, n_seg, N, Cout, up, s_co, s_j, has_bn, relu;
    fcn_train_seg seg[FCN_MAX_SEGS];
    const float *W;
    float *dW;
    const float *bias;           /* plain (no BN) layers only, else NULL */
    float *dbias;
    float *Y;                    /* raw output [B*T_out, N] */
    float *dA;                   /* gradient w.r.t. this layer's post-activation output [B*T_out, N] */
    double *sums;                /* [2*Cout] Sum(y), Sum(y^2): zeroed by the caller before the forward */
    double *dsums;               /* [2*Cout] Sum(dz), Sum(dz*xh): zeroed by the caller before the backward */
    const float *gamma, *beta;
    float *dgamma, *dbeta, *run_mean, *run_var;
} fcn_train_layer;
/* `workspace` (may be NULL): scratch for the K-split of skinny layers (partial sums, added in a fixed order);
 * fcn_train_workspace_floats(layer) = the size the launcher would like for this layer. */
FCN_API long long fcn_train_workspace_floats(const fcn_train_layer *layer);
FCN_API int fcn_train_forward(const fcn_train_layer *layer, float *workspace, long long workspace_floats,
                              fcn_stream_t stream);
/* backward of one layer: column reduction, dW (all segments), dX for the segments in need_dx_mask */
FCN_API int fcn_train_backward(const fcn_train_layer *layer, int need_dx_mask, fcn_stream_t stream);
/* PointNet pooling: feat[(b,t), c] = (cnt > 0) * max_k relu(bn(Y[(b,t,k), c])), one-hot columns appended
 * (det_base.py:100-101,134-157); backward scatters dfeat to the arg-max rows of a zero-filled dA. */
typedef struct {
    int B, T, K, C, V, ld_feat;
    const float *Y;
    const int32_t *cnt;
    const double *sums;
    const float *gamma, *beta, *one_hot;
    float *feat;
    int32_t *argmax;
    const float *dfeat;
    float *dA;
} fcn_train_pool_args;
FCN_API int fcn_train_pool(const fcn_train_pool_args *args, int backward, fcn_stream_t stream);
/* end of step, one launch for all layers (DEVICE copy of the layer table): running statistics (momentum 0.1,
 * unbiased variance), dgamma / dbeta / dbias from the reduction buffers */
FCN_API int fcn_train_finalize(const fcn_train_layer *layers_dev, int n_layers, int update_running,
                               fcn_stream_t stream);
/* fused Adam over one flat bucket (torch.optim.Adam semantics incl. L2 weight decay); grad_scale multiplies
 * the gradient first (1/world after a sum all-reduce) */
FCN_API int fcn_adam_step(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, long long n, float lr,
                          float beta1, float beta2, float eps, float weight_decay, int step, float grad_scale,
                          fcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (7b) Fused detection losses + gradient w.r.t. the head logits (row 8(f)-2, train half): everything of
 *      models/det_base.py:414-503 after the heads - foreground selection, focal loss (models/common.py:217-232),
 *      Huber / cross-entropy / corner losses (models/model_util.py:9-72, models/box_transform.py:5-65), accuracies
 *      and the rotated-IoU metrics - and its autograd backward, in three tiny launches.
 *      cls (B*T2, 2), reg (B*T2, 3 + 2*NH + 4*NS) rows in (frustum, position) order; labels as the reference's
 *      data dict holds them (cls_label int64 (B,T2) in {-1,0,1}, size_class int64 (B), box3d_* fp32).
 *      out[0..7] = total, cls, center, head_cls, head_res, size_cls, size_res, corners; out[8..13] = cls_acc,
 *      head_acc, size_acc, IoU_2D, IoU_3D, IoU_>=thresh; out[14..15] = #foreground, #non-ignored rows.
 *      scratch: 16 floats.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int B, T2, NH, NS, with_iou, reserved0;
    const float *cls, *reg, *center_ref2 /* (B,3,T2) */;
    const long long *cls_label, *size_class;
    const float *box3d_center, *box3d_heading, *box3d_size, *mean_size /* (NS,3) */;
    float w_box, w_head_reg, w_size_reg, w_corner, iou_thresh, reserved1;
    float *dcls, *dreg, *out /* 16 floats */, *scratch /* 16 floats */;
} fcn_loss_args;
FCN_API int fcn_det_loss(const fcn_loss_args *args, fcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (8) Inference post-processing ("next" row 8(f)-4): batched rotated 3-D NMS on the device.  Replaces
 *     `cube_nms` = rotate_nms_3d_cc (ops/pybind11/rbbox_iou.py:294-311) -> rotate_non_max_suppression_3d_cpu
 *     (ops/pybind11/nms_cpu.h:148-240), called per image and class from train/test_net_det.py:126-152.
 *     dets: (total, 8) fp32 rows [cx, cy, cz, l, w, h, ry, score]; segment s = rows
 *     [seg_offsets[s], seg_offsets[s+1]) (one image x class list; every row of it is considered, no list is
 *     truncated); keep: (num_segments, keep_stride) int32 GLOBAL row indices in descending-score order,
 *     keep_count[s] <= top_k <= keep_stride of them are valid.  A box is suppressed by a kept, higher-scored box
 *     when their axis-aligned bounding cubes overlap and the rotated 3-D IoU is >= thresh.  Score order: NaN
 *     first, then descending score, equal scores (and NaNs) larger index first = np.argsort(kind="stable")[::-1].
 *     A box with NaN geometry is never suppressed and suppresses nothing.
 *     max_seg_len: an upper bound of every segment length (<= fcn_rotate_nms_3d_max_seg_len()).  Segments of at
 *     most fcn_rotate_nms_3d_max_dets() rows run in shared memory, one launch in all; longer ones need `workspace`
 *     (256-byte aligned, device memory) of fcn_rotate_nms_3d_workspace_bytes(number of longer segments,
 *     max_seg_len) bytes, NULL otherwise.  A segment longer than max_seg_len, with a negative length, or left
 *     without a workspace slot gets keep_count[s] = -1 (an error for the caller to raise).  Returns an error,
 *     before any CUDA call, for top_k > keep_stride, a negative max_seg_len or a missing / too small workspace.
 * ------------------------------------------------------------------------------------------ */
FCN_API int fcn_rotate_nms_3d(int num_segments, const float *dets, const int32_t *seg_offsets, int max_seg_len,
                              float thresh, int top_k, int32_t *keep, int32_t *keep_count, int keep_stride,
                              void *workspace, long long workspace_bytes, fcn_stream_t stream);
FCN_API long long fcn_rotate_nms_3d_workspace_bytes(int num_long_segments, int max_seg_len);
FCN_API int fcn_rotate_nms_3d_max_dets(void);
FCN_API int fcn_rotate_nms_3d_max_seg_len(void);

/* ------------------------------------------------------------------------------------------
 * (9) Device-side input builder ("next" row 8(f)-3): ProviderDataset.__getitem__ of datasets/provider_sample.py
 *     (:133-203 resample + centre-view rotation, :291-327 generate_ref, datasets/data_utils.py:7-21,73-93) for a
 *     whole batch in one launch, from raw frustum points that stay resident in HBM.  `choice` (B,N) int32 = the
 *     caller's np.random.choice draw (indices into each frustum's own points).  float64 arithmetic with the
 *     reference's float32 casts.  Outputs have the layouts the model consumes: point_cloud (B,3,N),
 *     centers[s] (B,3,T_s), one_hot (B,num_classes) (optional), rot_angle (B) (optional).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int B, N, num_scales, num_classes;
    int T[FCN_MAX_SCALES];
    double stride[FCN_MAX_SCALES];
    const float *points;          /* (sum n_b, 3) raw frustum points, rect camera coordinates */
    const int32_t *point_offsets; /* (B+1) */
    const int32_t *choice;        /* (B, N) */
    const double *frustum_angle;  /* (B) */
    const double *box2d;          /* (B, 4) x1, y1, x2, y2 */
    const double *P;              /* (B, 12) calib P2, row-major 3x4 */
    const int32_t *cls_index;     /* (B) or NULL */
    float *point_cloud;
    float *centers[FCN_MAX_SCALES];
    float *one_hot;               /* or NULL */
    float *rot_angle;             /* or NULL */
} fcn_input_args;
FCN_API int fcn_build_inputs(const fcn_input_args *args, fcn_stream_t stream);

/* Layout helpers for the channel-first module APIs: (B,C,T) <-> (B,pitch >= T,ld) position-major. */
FCN_API int fcn_bct_to_btc(int B, int C, int T, int pitch, int ld, const float *src, float *dst,
                           fcn_stream_t stream);
FCN_API int fcn_btc_to_bct(int B, int C, int T, int pitch, int ld, const float *src, float *dst,
                           fcn_stream_t stream);

/* Self-test of the tcgen05/TMEM/bulk-copy building blocks: D (128,N) = A (128,K) * W^T with W given
 * as the pre-swizzled stage image of the host packer (engine.pack_sw128).  N in {64,128},
 * K multiple of 32 (<= 256).  Used by tests/ to pin the descriptor encodings on real hardware. */
FCN_API int fcn_selftest_umma(int N, int K, const float *A, const void *w_img, float *D,
                              fcn_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (6) Train-branch metric ("next" row 8(f)-1): pairwise rotated-box IoU on the device.  Replaces the CPU
 *     Boost.Geometry call rbbox_iou_3d_pair (ops/pybind11/box_ops.h:173-260) and the device->host copy of
 *     the boxes in front of it (models/det_base.py:494-495).
 *     corners, qcorners: (M, 8, 3) fp32 box corners in the order of get_box3d_corners_helper
 *     (models/model_util.py:48-72), 16-byte aligned;  iou: (M, 2) = [BEV IoU, 3-D IoU] per pair, zeros when
 *     the bird's-eye-view polygons do not overlap (box_ops.h:199,226);  stats (optional, may be NULL): 3 floats
 *     = mean BEV IoU, mean 3-D IoU, fraction of pairs with 3-D IoU >= iou_thresh (det_base.py:497-500),
 *     reduced in a fixed order (deterministic).  M == 0 writes zeros to stats.
 * ------------------------------------------------------------------------------------------ */
FCN_API int fcn_rbbox_iou_3d_pair(int M, const float *corners, const float *qcorners, float *iou,
                                  float iou_thresh, float *stats, fcn_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* FRUSTUM_B200_H_ */
