/*
 * yolo_b200.h -- C ABI of the B200-native tf2_YOLO anchor-grid engine.
 *
 * Every entry point replaces one Python function of samson6460/tf2_YOLO (cited
 * per function as reference file:line).  Conventions, all entry points:
 *   - every pointer is CALLER-OWNED DEVICE memory unless the name ends in _host;
 *   - the library allocates nothing persistent and keeps no global mutable
 *     state (re-entrant; safe from several host threads / streams);
 *   - every launch is asynchronous on the given stream (a cudaStream_t);
 *   - return 0 = OK, negative = invalid argument (YB_E_*), positive = the
 *     cudaError_t of the failing runtime call.  yb_status_string() names both.
 *   - there is no CPU fallback anywhere behind this interface.
 */
#ifndef YOLO_B200_H_
#define YOLO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* yb_stream_t; /* == cudaStream_t */

#define YB_ABI_VERSION 2
#define YB_MAX_BOXES 16  /* anchors per cell */
#define YB_MAX_SCALES 4  /* FPN outputs per fused loss launch */
#define YB_LOSS_TERMS 8  /* doubles per scale in terms_out */
#define YB_LOSS_METRICS 10 /* doubles per scale in metrics_out */
#define YB_MAX_PEERS 16   /* ranks of one node in a peer-memory exchange */
#define YB_FUSED_MAX_ROWS 2048 /* decode rows per image the one-launch decode+NMS holds in shared memory */
#define YB_ENCODE_MAX_BOXES 1024 /* boxes per image yb_encode_labels stages in shared memory */

enum {
    YB_OK = 0,
    YB_E_NULL = -1,      /* required pointer is NULL */
    YB_E_SHAPE = -2,     /* bad grid / box / class count */
    YB_E_PARAM = -3,     /* bad enum / version / mode */
    YB_E_WORKSPACE = -4, /* workspace too small or misaligned */
    YB_E_ALIGN = -5,     /* tensor pointer not 4-byte (f32) / 8-byte (f64) aligned */
    YB_E_CAPACITY = -6   /* output capacity too small (decode rows) */
};

int yb_abi_version(void);
const char* yb_status_string(int status);
/* "file:line" of the CUDA runtime call behind the last positive status this THREAD received. */
const char* yb_last_error_site(void);

/* Device-side alias of a page-locked HOST allocation.  Output pointers of the entry points below
 * may be such aliases where noted ("may be mapped host memory"): the kernel then writes its
 * result straight into host memory and the caller needs no sized D2H copy (and no round trip to
 * learn the size).  Returns the cudaError_t of cudaHostGetDevicePointer for pageable memory. */
int yb_mapped_host_pointer(void* host_ptr_host, void** device_ptr_host);

/* ------------------------------------------------------------------------
 * Grid losses: fused forward + gradient.
 * Replaces the closures returned by wrap_yolo_loss:
 *   v4  yolov4/losses/loss.py:64-169   (+ cal_iou/CIoU :10-61)
 *   v3  yolov3/losses/loss.py:40-164   (+ cal_iou :9-37)
 *   v2  yolov2/losses/loss.py:40-137
 *   v1  yolov1_5/losses/loss.py:40-118 (different cell layout, IoU differentiated)
 * The keyword arguments of wrap_yolo_loss become this POD struct.
 * ---------------------------------------------------------------------- */
typedef struct yb_loss_params {
    int32_t version;                 /* 1 | 2 | 3 | 4 */
    int32_t grid_h, grid_w;          /* grid_shape */
    int32_t bbox_num, class_num;
    int32_t has_anchors;             /* 0: anchors=None -> divisor 1 */
    float anchors[2 * YB_MAX_BOXES]; /* (w,h) per box, image-normalised */
    float binary_weight;
    float loss_weight[4];            /* v4: box,conf,prob ; v1-v3: xy,wh,conf,prob */
    float wh_reg_weight;             /* v4 kwarg; v2/v3 hard-code 0.01; v1 none (0) */
    float ignore_thresh;
    float truth_thresh;              /* v4 (>=1 disables) */
    float label_smooth;              /* v4 */
    float focal_gamma;               /* v4, v3 when use_focal */
    int32_t use_focal;               /* v3: use_focal_loss */
    int32_t use_scale;               /* v3: use_scale (v2: always 1) */
    int32_t from_logits;             /* v3/v4 only: y_pred holds RAW head outputs; the kernel applies the
                                        head transform of yolov4/models/__init__.py:42-60 (sigmoid xy/c/p,
                                        anchor*exp wh) and returns dL/d(raw) (SURVEY.md 8a N1) */
    double inv_batch;                /* 1 / N of reduce_mean(axis=0); N = GLOBAL batch when sharded */
} yb_loss_params;

typedef struct yb_loss_scale {
    const float* y_true; /* (n_cells, 5+C)            fp32 */
    const float* y_pred; /* (n_cells, B*(5+C)) | v1 (n_cells, 5B+C) */
    float* dpred;        /* like y_pred; NULL = forward only */
    int64_t n_cells;     /* N_local * grid_h * grid_w */
    yb_loss_params p;
} yb_loss_scale;

/* Workspace for a fused launch over n_scales scales. */
size_t yb_loss_workspace_bytes(int n_scales);

/* One launch over up to YB_MAX_SCALES scales (the three Keras outputs of one
 * train step).  loss_out[s] = loss of scale s (fp32, what yolo_loss returns);
 * terms_out (optional, may be NULL) = YB_LOSS_TERMS doubles per scale:
 * [total, term0..term4, 0, 0] already divided by N (v4: box,conf,prob,reg;
 * v2/v3: xy,wh,conf,prob,reg; v1: xy,wh,conf,prob). */
int yb_loss_fwd_bwd(const yb_loss_scale* scales_host, int n_scales, float* loss_out,
                    double* terms_out, void* workspace, size_t workspace_bytes,
                    yb_stream_t stream);

/* Same launch, plus the in-training metrics of yolov{2,3,4}/metrics/yolo_metrics.py:9-115
 * (wrap_obj_acc / wrap_mean_iou / wrap_class_acc / wrap_recall; v1 variant
 * yolov1_5/metrics/yolo_metrics.py) computed in the SAME pass over the tensors (zero extra HBM
 * traffic).  metrics_out: YB_LOSS_METRICS doubles per scale =
 * [obj_acc, mean_iou, class_acc, recall,  cells with correct objectness, sum of best IoU over
 * object cells, sum of obj, sum of class-argmax matches, recall true positives, n_cells]
 * (the raw sums let a sharded batch combine ranks). */
int yb_loss_fwd_bwd_metrics(const yb_loss_scale* scales_host, int n_scales, float* loss_out,
                            double* terms_out, double* metrics_out, double recall_iou_threshold,
                            void* workspace, size_t workspace_bytes, yb_stream_t stream);

/* Single-scale conveniences, one per reference package. */
int yb_loss_v1_fwd_bwd(const float* y_true, const float* y_pred, int64_t n_cells,
                       float* loss_out, float* dpred, const yb_loss_params* p,
                       void* workspace, size_t workspace_bytes, yb_stream_t stream);
int yb_loss_v2_fwd_bwd(const float* y_true, const float* y_pred, int64_t n_cells,
                       float* loss_out, float* dpred, const yb_loss_params* p,
                       void* workspace, size_t workspace_bytes, yb_stream_t stream);
int yb_loss_v3_fwd_bwd(const float* y_true, const float* y_pred, int64_t n_cells,
                       float* loss_out, float* dpred, const yb_loss_params* p,
                       void* workspace, size_t workspace_bytes, yb_stream_t stream);
int yb_loss_v4_fwd_bwd(const float* y_true, const float* y_pred, int64_t n_cells,
                       float* loss_out, float* dpred, const yb_loss_params* p,
                       void* workspace, size_t workspace_bytes, yb_stream_t stream);

/* The head transform of yolov4/models/__init__.py:42-60 (yolov3/models/__init__.py:36-63) on raw head
 * outputs, v3/v4 layout (B*(5+C) floats per cell): sigmoid x, y, objectness and class scores,
 * anchor * exp for w, h - the same float32 arithmetic the loss kernel applies with from_logits, so
 * decoding the result gives the rows the two-launch step gives for the raw heads.
 * p: the scale's loss parameters (version 3|4, has_anchors, bbox_num, class_num, anchors are read).
 * out may alias raw (out == raw: in place). */
int yb_activate_head(const yb_loss_params* p, const float* raw, float* out, int64_t n_cells, yb_stream_t stream);

/* Grid IoU (and CIoU) of the label box of a cell against its B predicted boxes:
 * yolov4/losses/loss.py:10-61 (cal_iou); v1-v3 loss.py:9-37.  box_true is
 * (n_cells, true_stride) with xywh at [0:4]; box_pred (n_cells, B, pred_stride).
 * iou_out / ciou_out are (n_cells, B) fp32; ciou_out may be NULL. */
int yb_grid_iou(const float* box_true, int true_stride, const float* box_pred,
                int pred_stride, int64_t n_cells, int bbox_num, int grid_h, int grid_w,
                float* iou_out, float* ciou_out, yb_stream_t stream);

/* ------------------------------------------------------------------------
 * Head decode: utils/tools.py:370-438 (decode), batched over images.
 * Input: n_scales tensors (n_img, grid_h, grid_w, B*(5+C)) [v1: 5B+C], dtype
 * f32 (model output) or f64 (labels).  Output rows [x,y,w,h,c,class,p] float64
 * in the reference's order: image-major, then scale in argument order, then
 * row-major (y, x, box, class).  row_offsets has n_img+1 entries (int64).
 * If more than row_capacity rows pass the threshold, rows beyond the capacity
 * are not written, *n_rows still holds the true total and the call reports it
 * through row_offsets; the host mirror re-runs with a larger buffer.
 * ---------------------------------------------------------------------- */
typedef struct yb_decode_params {
    int32_t version;   /* 1 | 2 | 3 | 4 */
    int32_t class_num;
    int32_t n_scales;
    int32_t is_f64;    /* 0: float inputs, 1: double inputs */
    int32_t grid_h[YB_MAX_SCALES], grid_w[YB_MAX_SCALES];
    int32_t bbox_num[YB_MAX_SCALES];
    double threshold;  /* compared in the input dtype, like numpy */
} yb_decode_params;

size_t yb_decode_workspace_bytes(const yb_decode_params* p, int64_t n_img);

int yb_decode(const void* const* preds_host /* n_scales device pointers */,
              int64_t n_img, const yb_decode_params* p, double* rows,
              int64_t row_capacity, int64_t* row_offsets, void* workspace,
              size_t workspace_bytes, yb_stream_t stream);

/* Fused evaluate-while-training step: the loss forward+gradient of yb_loss_fwd_bwd AND the
 * decode of the same head outputs (yb_decode on scales[i].y_pred, float32, all scales holding the
 * same images).  y_pred is streamed from HBM once for both: the decode counting pass runs on the
 * tiles the loss kernel already staged in shared memory; only cells with hits are touched again
 * to emit rows.  Results are identical to calling the two entry points separately.
 * With row_offsets == NULL only the counting pass runs (the counts stay in decode_workspace);
 * yb_decode_finish then scans them and emits the rows.  The rows are read back from y_pred, so
 * from_logits scales are rejected (YB_E_PARAM): activate raw heads with yb_activate_head first. */
int yb_loss_decode_fused(const yb_loss_scale* scales_host, int n_scales, float* loss_out,
                         double* terms_out, double decode_threshold, double* rows,
                         int64_t row_capacity, int64_t* row_offsets, void* loss_workspace,
                         size_t loss_workspace_bytes, void* decode_workspace,
                         size_t decode_workspace_bytes, yb_stream_t stream);

int yb_decode_finish(const void* const* preds_host, int64_t n_img, const yb_decode_params* p,
                     double* rows, int64_t row_capacity, int64_t* row_offsets, void* workspace,
                     size_t workspace_bytes, yb_stream_t stream);

/* ------------------------------------------------------------------------
 * Per-class greedy NMS / DIoU-NMS: utils/tools.py:687-733 (nms) with the
 * pairwise IoU of utils/tools.py:630-684 (cal_iou, mode 1 IoU / mode 2 DIoU),
 * batched over images.  rows: (n_rows,7) float64 as produced by yb_decode;
 * row_offsets: n_img+1 int64 (device).  keep[i] = 1 if row i survives.
 * out_rows (optional) receives the survivors in the reference's output order
 * (per image: class 0..C-1, original order inside a class), out_offsets
 * (n_img+1 int64) their per-image extents, out_seg_offsets (optional,
 * n_img*class_num+1 int64) their per-(image, class) extents.  n_rows is the
 * capacity of rows/keep; the true count is read on the device from
 * row_offsets[n_img], so a decode -> NMS chain needs no host round trip.
 * out_rows / out_offsets / out_seg_offsets are only ever written: they may be mapped host memory.
 * Ties: suppression on IoU >= threshold; equal confidences are visited
 * higher-original-index first.
 * ---------------------------------------------------------------------- */
size_t yb_nms_workspace_bytes(int64_t n_rows, int64_t n_img, int class_num);

int yb_nms(const double* rows, const int64_t* row_offsets, int64_t n_rows, int64_t n_img,
           int class_num, double nms_threshold, int iou_mode, uint8_t* keep,
           double* out_rows, int64_t* out_offsets, int64_t* out_seg_offsets,
           void* workspace, size_t workspace_bytes, yb_stream_t stream);

/* Gaussian soft-NMS: utils/tools.py:736-786 (soft_nms).  Same layout and outputs as yb_nms
 * (same workspace size).  Every visited box - deleted or not - multiplies the confidence c*p
 * of each not-yet-visited box it overlaps (IoU >= nms_threshold) by exp(-IoU^2/sigma); a box is
 * dropped once that pushes it below conf_threshold.  The visit order is fixed by the initial
 * confidences, so each box's fate is an independent product over the boxes before it. */
int yb_soft_nms(const double* rows, const int64_t* row_offsets, int64_t n_rows, int64_t n_img,
                int class_num, double nms_threshold, double conf_threshold, double sigma,
                uint8_t* keep, double* out_rows, int64_t* out_offsets, int64_t* out_seg_offsets,
                void* workspace, size_t workspace_bytes, yb_stream_t stream);

/* ------------------------------------------------------------------------
 * Decode + per-class NMS in ONE launch, one CTA per image (utils/tools.py:370-438 followed by
 * :687-733): the counting pass files the boxes with hits per image, the image's CTA builds its
 * float64 rows in shared memory, runs the greedy (D)IoU-NMS of every class on a warp and writes
 * the survivors - same rows, same order, same bits as yb_decode followed by yb_nms (out_rows /
 * out_offsets as there; they are only written and may be mapped host memory).  float32 heads,
 * class_num <= 256.  An image with more than rows_per_img_cap (32..YB_FUSED_MAX_ROWS) decode rows
 * is skipped (no survivors) and counted in *n_overflow (device, written by the call; may be
 * NULL): the caller then falls back to yb_decode + yb_nms, like a too small row_capacity there.
 * yb_loss_decode_nms_fused: the whole train-and-evaluate step in two launches - the loss
 * forward + gradient (as yb_loss_fwd_bwd) with the counting pass riding on its read of y_pred,
 * then the per-image kernel.  With out_offsets == NULL only the loss kernel runs (the buckets
 * stay in fused_workspace); yb_decode_nms_finish then launches the per-image kernel.
 * The step also takes RAW v3/v4 heads (from_logits on every scale): the counting pass applies the
 * head transform of yb_activate_head to the values it files, so the survivors are those of the
 * activated heads, and the gradient is d/d(raw).  The overflow fallback then decodes the
 * yb_activate_head output, not the raw heads.
 * ---------------------------------------------------------------------- */
size_t yb_decode_nms_workspace_bytes(const yb_decode_params* p, int64_t n_img, int rows_per_img_cap);

int yb_decode_nms(const void* const* preds_host, int64_t n_img, const yb_decode_params* p,
                  double nms_threshold, int iou_mode, int rows_per_img_cap, double* out_rows,
                  int64_t out_capacity, int64_t* out_offsets, unsigned int* n_overflow,
                  void* workspace, size_t workspace_bytes, yb_stream_t stream);

int yb_loss_decode_nms_fused(const yb_loss_scale* scales_host, int n_scales, float* loss_out,
                             double* terms_out, double decode_threshold, double nms_threshold,
                             int iou_mode, int rows_per_img_cap, double* out_rows,
                             int64_t out_capacity, int64_t* out_offsets, unsigned int* n_overflow,
                             void* loss_workspace, size_t loss_workspace_bytes, void* fused_workspace,
                             size_t fused_workspace_bytes, yb_stream_t stream);

/* yb_loss_decode_nms_fused for workspaces that the caller ZEROED ONCE (all yb_loss_workspace_bytes /
 * yb_decode_nms_workspace_bytes bytes) and has handed to nothing but this entry point since: both
 * kernels leave their control blocks zeroed, so the call is two launches and no memset - the form
 * a captured CUDA graph replays.  After a call that returned an error, zero them again. */
int yb_loss_decode_nms_fused_clean(const yb_loss_scale* scales_host, int n_scales, float* loss_out,
                                   double* terms_out, double decode_threshold, double nms_threshold,
                                   int iou_mode, int rows_per_img_cap, double* out_rows,
                                   int64_t out_capacity, int64_t* out_offsets, unsigned int* n_overflow,
                                   void* loss_workspace, size_t loss_workspace_bytes,
                                   void* fused_workspace, size_t fused_workspace_bytes, yb_stream_t stream);

int yb_decode_nms_finish(const void* const* preds_host, int64_t n_img, const yb_decode_params* p,
                         double nms_threshold, int iou_mode, int rows_per_img_cap, double* out_rows,
                         int64_t out_capacity, int64_t* out_offsets, unsigned int* n_overflow,
                         void* workspace, size_t workspace_bytes, yb_stream_t stream);

/* Pairwise IoU / DIoU matrix, utils/tools.py:630-684 on (g,1,.) x (1,d,.):
 * a: (na, stride_a) doubles, b: (nb, stride_b) doubles, out (na, nb). */
int yb_pairwise_iou(const double* a, int64_t na, int stride_a, const double* b, int64_t nb,
                    int stride_b, int iou_mode, double* out, yb_stream_t stream);

/* Same arithmetic, element by element: a (n, stride_a), b (n, stride_b) -> out (n). */
int yb_elementwise_iou(const double* a, int stride_a, const double* b, int stride_b, int64_t n,
                       int iou_mode, double* out, yb_stream_t stream);

/* ------------------------------------------------------------------------
 * Anchor k-means, one Lloyd assignment pass: utils/kmeans.py:79-90 with the
 * distances of :9-33 (iou_dist, area ratio) and :36-40 (euclidean).
 * data (M,d) float64; centers (k,d) float64.  Outputs: assign[M] (first
 * minimum, like np.argmin), sums (k,d), counts[k], all complete when the
 * stream reaches the end of the call.  assign may be NULL.
 * ---------------------------------------------------------------------- */
enum { YB_DIST_IOU = 0, YB_DIST_EUCLID = 1 };

size_t yb_kmeans_workspace_bytes(int64_t n_points, int k, int n_dim);

int yb_kmeans_assign(const double* data, int64_t n_points, int n_dim, const double* centers,
                     int k, int dist_kind, int32_t* assign, double* sums, int64_t* counts,
                     void* workspace, size_t workspace_bytes, yb_stream_t stream);

/* utils/kmeans.py:9-40 evaluated directly (the module's iou / iou_dist / euclidean_dist on
 * data-sized arrays): a (na, n_dim), b (nb, n_dim) float64.  outer != 0: out (na, nb), every a
 * against every b (the (k,1,d) x (1,M,d) broadcast of kmeans.py:79); outer == 0: na == nb, out (nb).
 * what: 0 iou (area ratio min/max), 1 iou_dist (1 - iou), 2 euclidean_dist. */
int yb_kmeans_dist(const double* a, int64_t na, const double* b, int64_t nb, int n_dim, int what,
                   int outer, double* out, yb_stream_t stream);

/* The Lloyd loop of utils/kmeans.py:78-98 WITHOUT the host in it.  One call = one iteration:
 * assignment pass over the resident boxes and - single rank, packed == NULL - the update of
 * kmeans.py:84-97 by the last CTA of the same launch: cluster means, loss = mean(dist(center,
 * new_center)) in NumPy's summation order, centres rewritten in place, the stop test
 * `loss < stop_dist or epoch > max_iternum`.  Sharded (packed != NULL): the pass leaves
 * [k*d sums | k counts as doubles] in `packed` for the caller's all-reduce on the same stream and
 * yb_kmeans_lloyd_update applies the update on every rank (identical inputs, identical centres).
 * `state` (device, yb_kmeans_state_bytes, zeroed by yb_kmeans_lloyd_init together with the
 * workspace's counter) holds 8-byte words: [0] status 0 running | 1 converged | 2 iteration cap |
 * 3 empty cluster | 4 peer exchange timed out, [1] completed updates, [4 + (e-1) % YB_KMEANS_HIST] the loss of update e
 * (double), then the k*(d+1) global sums / counts of the iteration that met an empty cluster.
 * A non-zero status FREEZES the loop: further steps return at once, so the host may queue
 * iterations in batches and look at `state` once per batch; the result does not depend on the
 * batch size.  On status 3 the centres are untouched: the host redraws the empty clusters with
 * numpy.random in the reference's order (kmeans.py:89), finishes that update and clears the status.
 * assign (optional) receives the assignments of the pass (against the centres BEFORE its update). */
#define YB_KMEANS_HIST 64
size_t yb_kmeans_state_bytes(int k, int n_dim);

int yb_kmeans_lloyd_init(int64_t* state, int k, int n_dim, void* workspace, size_t workspace_bytes,
                         yb_stream_t stream);

int yb_kmeans_lloyd_step(const double* data, int64_t n_points, int n_dim, double* centers, int k,
                         int dist_kind, double stop_dist, int64_t max_iternum, int64_t* state,
                         double* packed, int32_t* assign, void* workspace, size_t workspace_bytes,
                         yb_stream_t stream);

int yb_kmeans_lloyd_update(const double* packed, double* centers, int k, int n_dim, int dist_kind,
                           double stop_dist, int64_t max_iternum, int64_t* state, yb_stream_t stream);

/* Sharded Lloyd iteration with the all-reduce INSIDE the launch: the last CTA stores the rank's
 * k*(d+1) partial sums into every rank's mailbox (peer stores over NVLink / NVSwitch), publishes
 * them with a system-scope release, waits for all ranks' contributions in its own mailbox, adds
 * them in rank order (identical bits on every rank) and applies the update - one launch per
 * iteration, no NCCL call, no extra kernel.  mailboxes_host[r] = device pointer to rank r's mailbox
 * (yb_peer_mailbox_bytes(world) bytes, zeroed; own mailbox at [rank], the others opened from their
 * IPC handles).  All ranks must issue the same sequence of steps; a rank that never arrives ends
 * the peers' wait after 2 s with state[0] = 4 (exchange timed out) instead of hanging their GPUs.
 * state[2] counts the exchanges.
 * yb_peer_alloc is the only place this library owns device memory (IPC export needs a cudaMalloc
 * allocation): yb_peer_free releases it; yb_peer_open / yb_peer_close map a peer's allocation. */
size_t yb_peer_mailbox_bytes(int world);
int yb_peer_alloc(size_t bytes, void** dev_ptr_host, void* ipc_handle64_host);
int yb_peer_open(const void* ipc_handle64_host, void** dev_ptr_host);
int yb_peer_close(void* dev_ptr);
int yb_peer_free(void* dev_ptr);

int yb_kmeans_lloyd_step_peers(const double* data, int64_t n_points, int n_dim, double* centers, int k,
                               int dist_kind, double stop_dist, int64_t max_iternum, int64_t* state,
                               int32_t* assign, void* workspace, size_t workspace_bytes,
                               void* const* mailboxes_host, int rank, int world, yb_stream_t stream);

/* min / max over all elements of data (kmeans.py:68-69). out2 = {min,max}. */
int yb_minmax_f64(const double* data, int64_t n, double* out2, void* workspace,
                  size_t workspace_bytes, yb_stream_t stream);

/* ------------------------------------------------------------------------
 * PR-curve / mAP matching: utils/measurement.py:252-292 (PRfunc) and :104-130
 * (create_score_mat).  Per (image, class): every detection takes max/argmax
 * IoU over the ground truths of that class.
 * gt_rows / det_rows: (.,7) float64 rows in decode layout with int64 per-image
 * offsets (the true row counts are read on the device from offsets[n_img];
 * *_capacity only bound the launch).  Outputs per detection row: best_iou
 * (float64; -1 when the image has no ground truth of that class), best_gt (int32
 * index of the argmax among the image's ground truths OF THAT CLASS, first
 * maximum; -1 if none).  gt_class_counts (n_img, class_num) int32 counts ground
 * truths per image and class.
 * ---------------------------------------------------------------------- */
int yb_map_match(const double* gt_rows, const int64_t* gt_offsets, const double* det_rows,
                 const int64_t* det_offsets, int64_t n_img, int class_num, int64_t gt_capacity,
                 int64_t det_capacity, double* best_iou, int32_t* best_gt,
                 int32_t* gt_class_counts, yb_stream_t stream);

/* PR accumulation for one batch of images: utils/measurement.py:252-292 (PRfunc) and
 * :104-130 (create_score_mat).  det_rows are NMS survivors grouped by (image, class) with
 * det_seg_offsets (n_img*class_num+1, from yb_nms); best_iou / best_gt / gt_class_counts come
 * from yb_map_match.  gt_base[c] = ground truths of class c in earlier batches (the running
 * num_gts of measurement.py:256).  Outputs, grouped by class then image (capacity = number of
 * det rows): conf = c*p, gt_id = best_gt + running count, flag = best_iou >= iou_threshold,
 * cls; class_offsets has class_num+1 entries.  max_per_img > 0 keeps the top max_per_img
 * detections per (image, class) in descending-confidence order (:285-289).  score_acc
 * (3*class_num uint64, ADDED to): detections, flagged detections, distinct matched ground
 * truths per class (PP, TPP, TP of create_score_mat). */
size_t yb_map_accumulate_workspace_bytes(int64_t n_img, int class_num);

int yb_map_accumulate(const double* det_rows, const int64_t* det_seg_offsets, const double* best_iou,
                      const int32_t* best_gt, const int32_t* gt_class_counts, int64_t n_img,
                      int class_num, double iou_threshold, int64_t max_per_img,
                      const int64_t* gt_base, double* conf, int64_t* gt_id, uint8_t* flag,
                      int32_t* cls, int64_t* class_offsets, uint64_t* score_acc, void* workspace,
                      size_t workspace_bytes, yb_stream_t stream);

/* Append the records of one batch (the first *n_src entries of conf / gt_id / flag / cls as
 * yb_map_accumulate left them; n_src = its class_offsets + class_num, on the device) to the
 * caller's record arrays at position *total (device), then *total += *n_src - all on the device,
 * so a stream of batches accumulates without a host round trip.  Entries beyond dst_capacity are
 * dropped while *total keeps counting: the caller compares it with the capacity at the end.
 * counter: one uint32, zero before the first call (left zero by every call). */
int yb_map_append(const double* conf, const int64_t* gt_id, const uint8_t* flag, const int32_t* cls,
                  const int64_t* n_src, int64_t src_capacity, double* conf_dst, int64_t* gt_id_dst,
                  uint8_t* flag_dst, int32_t* cls_dst, int64_t dst_capacity, int64_t* total,
                  uint32_t* counter, yb_stream_t stream);

/* Final PR pass, utils/measurement.py:297-321: sort all triples by (class asc, confidence
 * desc, later position first), find the first occurrence of every matched ground truth and
 * return running counts.  order[i] = input index of the i-th sorted record; tp_cum / tpp_cum
 * (n_det+1 entries) = exclusive running counts of first-occurrence true positives / flagged
 * detections over the whole sorted array (subtract the value at a class start to get the
 * reference's per-prefix num_tp / num_tpp).  gt_table_base (class_num+1) = exclusive prefix of
 * the total ground-truth count per class; n_gt_total its last entry. */
size_t yb_pr_curve_workspace_bytes(int64_t n_det, int64_t n_gt_total);

int yb_pr_curve(const double* conf, const int32_t* cls, const int64_t* gt_id, const uint8_t* flag,
                int64_t n_det, const int64_t* gt_table_base, int64_t n_gt_total, int64_t* order,
                int64_t* tp_cum, int64_t* tpp_cum, void* workspace, size_t workspace_bytes,
                yb_stream_t stream);

/* Precision / recall of every prefix of every class (utils/measurement.py:302-319) from the running
 * counts of yb_pr_curve: class_start (class_num+1 int64, device) = extents of the classes in the
 * sorted array, gts (class_num int64, device) = ground truths per class (> 0 wherever a class has
 * records).  precision_mode 0: tpp/dets, 1: tp/(tp+fp), 2: tp/dets; recall = tp/gts. */
int yb_pr_points(const int64_t* tp_cum, const int64_t* tpp_cum, const int64_t* class_start,
                 const int64_t* gts, int class_num, int64_t n_det, int precision_mode,
                 double* precision, double* recall, yb_stream_t stream);

/* ------------------------------------------------------------------------
 * Label-side helpers (SURVEY.md 8f rows 3-4).
 * yb_down2x_labels: utils/tools.py:342-367 (down2xlabel): (n_img, gh, gw, channels) labels,
 * float32 or float64, -> (n_img, gh/2, gw/2, channels) float64; a 2x2 block whose maximum obj
 * flag equals 1 keeps its largest-area entry (first maximum, areas in the input dtype) with
 * xy re-expressed in the coarser cell.  Odd grids are rejected (the reference raises).
 * yb_column_sums: per-column sums of a (rows, cols) matrix in fp64 - the data-sized part of
 * utils/tools.py:592-627 (get_class_weight).
 * ---------------------------------------------------------------------- */
/* yb_encode_labels: box lists -> label grids, the `_encode_to_array` closure of
 * YoloDataSequence.__getitem__ (utils/tools.py:179-209) followed, for n_levels > 1, by
 * down2xlabel (utils/tools.py:342-367) once per extra level as _Yolov4DataSequence.__getitem__
 * does (yolov4/__init__.py:47-53) - all levels in ONE launch, nothing dense is read.
 * boxes: (n_boxes, 5) float64 [x1, y1, x2, y2, class index] in pixels of the resized image
 * (what the closure reads from imgaug's BoundingBox and its `labels` list); box_offsets
 * (n_img+1 int64, device): image i owns boxes [box_offsets[i], box_offsets[i+1]), applied in
 * list order: a later box overwrites x, y, w, h of its cell, the class bits of earlier boxes of
 * the cell stay set.  img_h, img_w = img.shape[0], img.shape[1]; grid_h x grid_w = the FINEST
 * grid.  out_levels_host[l], l = 0..n_levels-1, coarse grid first (the reference's label_list
 * order): (n_img, grid_h >> (n_levels-1-l), grid_w >> (n_levels-1-l), 5+class_num), float64
 * (out_f64 = 1, what the reader returns) or float32 (the cast Keras applies before the loss);
 * fully written (zero-filled) by the call.  Arithmetic is float64 in the reference's order with
 * Python's floored // and %.  A centre at or beyond the last column / row is skipped (:199),
 * negative cell indices wrap like NumPy's.  Inputs on which the reference raises (non-finite
 * corners, class outside [0, class_num), cell index below -grid, more than max_boxes_per_img
 * boxes in an image) are skipped and counted in *n_bad (device, ADDED to; may be NULL).
 * max_boxes_per_img <= YB_ENCODE_MAX_BOXES bounds the per-image box count (shared-memory size). */
int yb_encode_labels(const double* boxes, const int64_t* box_offsets, int64_t n_img,
                     int max_boxes_per_img, double img_h, double img_w, int grid_h, int grid_w,
                     int class_num, int n_levels, void* const* out_levels_host, int out_f64,
                     unsigned long long* n_bad, yb_stream_t stream);

int yb_down2x_labels(const void* labels, int is_f64, int64_t n_img, int grid_h, int grid_w,
                     int channels, double* out, yb_stream_t stream);

size_t yb_column_sums_workspace_bytes(int cols);

int yb_column_sums(const void* data, int is_f64, int64_t rows, int cols, double* out,
                   void* workspace, size_t workspace_bytes, yb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* YOLO_B200_H_ */
