/*
 * libmgd -- B200-native (sm_100a) detection-head grid path for MultiGridDet.
 *
 * C ABI of the drop-in boundary.  The reference (solufast-cvprojects/multigriddet)
 * is pure Python and has no FFI of its own; these entry points are what a ctypes
 * binding inside the reference's two hot-path modules calls instead of the NumPy
 * loops.  Each entry point names the reference interface it replaces (paths are
 * relative to the reference repository root).  INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - every function returns an mgd_status; on failure mgd_last_error() returns a
 *     thread-local, NUL-terminated description.  No C++ exception crosses the ABI.
 *   - tensors are dense, row-major, caller-allocated.  `memory` says where ALL
 *     tensor arguments of the call live: MGD_MEM_DEVICE (CUDA device `device`;
 *     work is enqueued on `stream`, the call returns without synchronising unless
 *     MGD_FLAG_SYNC is set) or MGD_MEM_HOST (the library stages through the GPU:
 *     H2D, kernels, D2H; the call is synchronous; pinned host memory is faster).
 *   - the library never frees or keeps caller memory; scratch comes from the CUDA
 *     stream-ordered pool of `device`, so calls are re-entrant and may be issued
 *     concurrently from several host threads on different streams.
 *   - there is no CPU fallback: without a CUDA device every compute entry point
 *     fails with MGD_ERR_NO_DEVICE.
 */
#ifndef MGD_H_
#define MGD_H_

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define MGD_API __attribute__((visibility("default")))
#else
#define MGD_API
#endif

#define MGD_VERSION 100            /* 0.1.0 */
#define MGD_MAX_LAYERS 5           /* generators.py:3423 knows strides 32,16,8,4,2 */
#define MGD_MAX_ANCHORS_PER_LAYER 8

typedef enum {
    MGD_OK = 0,
    MGD_ERR_INVALID_ARGUMENT = 1,  /* Python shim raises ValueError               */
    MGD_ERR_CLASS_RANGE = 2,       /* class id >= num_classes -> AssertionError,
                                      generators.py:3409                          */
    MGD_ERR_CUDA = 3,              /* RuntimeError                                */
    MGD_ERR_NO_DEVICE = 4,         /* RuntimeError: no CPU fallback exists        */
    MGD_ERR_UNSUPPORTED = 5        /* NotImplementedError                         */
} mgd_status;

enum { MGD_MEM_HOST = 0, MGD_MEM_DEVICE = 1 };

enum {
    MGD_FLAG_SYNC = 1,             /* synchronise `stream` before returning and
                                      report deferred device-side errors          */
    MGD_FLAG_HOST_ZEROCOPY = 4,    /* MGD_MEM_HOST calls on page-locked tensors: the
                                      kernels access the big host tensor in place over
                                      the link instead of staging it through device
                                      memory -- mgd_decode_nms reads only the sectors
                                      of the predictions its filter asks for (about a
                                      third of the bytes of a trained-looking head; a
                                      dense head is ~30 % slower this way),
                                      mgd_encode_targets writes y_true straight into
                                      host memory.  Pays off where the host's memory
                                      interface, not the link, is the limit (several
                                      GPUs on one host).  Pageable tensors ignore it.
                                      MGD_HOST_ZEROCOPY (env, bits 0 / 1) forces it on.  */
    MGD_FLAG_TF_COMPAT = 2         /* mgd_encode_targets: the semantics of the
                                      reference's TensorFlow encoder
                                      tf_preprocess_true_boxes (generators.py:
                                      2696-3390) instead of the NumPy encoder's:
                                      exact centre, unrounded IoL (+1e-7), every
                                      in-bounds cell of the 3x3 block written,
                                      highest box index wins a shared cell, xy =
                                      [-dcol + frac(cy), -drow + frac(cx)], class ids
                                      outside [0, C) light no class channel and
                                      raise no error                              */
};

enum { MGD_NMS_IOU = 0, MGD_NMS_DIOU = 1, MGD_NMS_SOFT = 2, MGD_NMS_WBF = 3 };
enum { MGD_WBF_CONF_AVG = 0, MGD_WBF_CONF_MAX = 1, MGD_WBF_CONF_BOX_AND_MODEL_AVG = 2 };

/*
 * Geometry of the detection head: what `anchors`, `num_classes`, `input_shape`
 * and `grid_shapes` carry in preprocess_true_boxes (multigriddet/data/
 * generators.py:3393) and in MultiGridDecoder.__init__ (multigriddet/postprocess/
 * multigrid_decode.py:25-30).  Layer l has grid_h[l] x grid_w[l] cells and
 * 5 + num_anchors[l] + num_classes channels per cell:
 * [tx, ty, tw, th, obj, anchor one-hot/logits..., class one-hot/logits...].
 * Only square inputs and grids are supported (the reference's index arithmetic is
 * only self-consistent there: generators.py:3438-3439,3459-3470).
 */
typedef struct {
    int num_layers;
    int num_classes;
    int input_h, input_w;
    int grid_h[MGD_MAX_LAYERS];
    int grid_w[MGD_MAX_LAYERS];
    int num_anchors[MGD_MAX_LAYERS];
    double anchors[MGD_MAX_LAYERS][MGD_MAX_ANCHORS_PER_LAYER][2];   /* (w, h) px */
    /* 0: the caller's anchors were float32 (generators.py:1446), arithmetic that
       touches them runs in float32 like NumPy does; 1: float64 anchors
       (utils/anchors.py:311 load_anchors) and float64 arithmetic.              */
    int anchors_f64;
} mgd_head_config;

/* Knobs of MultiGridDecoder.postprocess (multigrid_decode.py:347-357). */
typedef struct {
    int use_softmax;          /* multigrid_decode.py:140-145                      */
    int rescore_confidence;   /* multigrid_decode.py:166-170                      */
    double confidence;        /* keep score >= confidence, :271                   */
    double nms_threshold;     /* suppress metric >= threshold, nms.py:180         */
    int nms_method;           /* MGD_NMS_DIOU ('diou'), MGD_NMS_IOU ('standard' /
                                 'cluster') or MGD_NMS_SOFT ('soft': Gaussian
                                 SoftNMS, nms.py:234-288; nms_threshold and
                                 per_class are ignored like in the reference) or
                                 MGD_NMS_WBF (use_wbf=True: weighted boxes fusion
                                 with iou_thr = nms_threshold, wbf.py:98-218)     */
    int per_class;            /* 0: class-agnostic (the reference's NMS classes);
                                 1: candidates of different argmax class never
                                 suppress each other                              */
    int max_boxes;            /* top-k after NMS, :336-345                        */
    double soft_sigma;        /* SoftNMS sigma (nms.py:237 default 0.5); <= 0 -> 0.5  */
    double soft_score_threshold; /* SoftNMS final / skip threshold (default 0.001);
                                 < 0 -> 0.001                                      */
} mgd_post_config;

MGD_API int mgd_version(void);
MGD_API const char *mgd_last_error(void);
MGD_API int mgd_device_count(void);   /* 0 when no CUDA device / driver is usable */

/*
 * Multi-grid y_true target encoder.
 * Replaces preprocess_true_boxes (multigriddet/data/generators.py:3393-3473,
 * with best_fit_and_layer :2514-2544 and iol_common_center :2486-2494), called
 * from MultiGridDataGenerator.__getitem__ (:1756).
 *
 *   boxes   (batch, max_boxes, 5) float32  [x1, y1, x2, y2, class] pixels;
 *           rows with (x2-x1)*(y2-y1) <= 0 are padding (:3431)
 *   y_true  num_layers pointers (array itself in host memory), each
 *           (batch, grid_h, grid_w, 5+A_l+C) float32, fully overwritten
 *   stats   optional host int64[4]: valid boxes, candidate writes skipped by the
 *           occupancy rule (:3463), positive cells, reserved.  Only filled when
 *           the call synchronises (host memory or MGD_FLAG_SYNC).
 *
 * MGD_ERR_CLASS_RANGE if any class id >= num_classes (all rows, like :3409);
 * MGD_ERR_INVALID_ARGUMENT for a negative class id on a valid box (the reference
 * would silently write a wrong channel).  For device memory without
 * MGD_FLAG_SYNC these two are reported by the next synchronising call on the
 * same thread via mgd_poll_status().
 */
MGD_API int mgd_encode_targets(const mgd_head_config *cfg, const float *boxes,
                       int batch, int max_boxes, float *const *y_true,
                       int memory, int device, void *stream, int flags,
                       long long *stats);

/*
 * Dense head decode + score threshold + NMS + top-k + xyxy, per image.
 * Replaces MultiGridDecoder.postprocess (multigriddet/postprocess/
 * multigrid_decode.py:347-395 = decode_predictions :48-183, correct_boxes
 * :185-235, handle_predictions :237-345, _convert_to_xyxy :397-422) and the
 * greedy NMS classes (multigriddet/postprocess/nms.py:83-231, 320-385), called
 * per image from evaluator.py:262 and inference_engine.py:127.  A batch is B
 * independent batch-1 reference calls.
 *
 *   preds       num_layers pointers, each (batch, grid_h, grid_w, 5+A_l+C) float32
 *   image_hw    (batch, 2) int32 original image (h, w); NULL = model input size
 *   boxes_xywh  (batch, max_boxes, 4) float64 [x_min, y_min, w, h] (return_xyxy=False)
 *   boxes_xyxy  (batch, max_boxes, 4) int32, clipped and rounded (:409-420)
 *   scores      (batch, max_boxes) float64 (float32 values, like the reference)
 *   classes     (batch, max_boxes) int32
 *   index       (batch, max_boxes) int32 flat cell index of each detection in the
 *               decode_predictions concatenation order (layer, row, col)
 *   counts      (batch,) int32 detections per image; rows beyond it are 0 / -1
 *   Any output pointer except counts may be NULL.
 *   stats       optional host int64[4]: candidates >= confidence, detections,
 *               reserved, reserved (filled only when the call synchronises).
 * Detections are in descending score order; equal scores: lower cell index first.
 */
MGD_API int mgd_decode_nms(const mgd_head_config *cfg, const mgd_post_config *post,
                   const float *const *preds, int batch, const int *image_hw,
                   double *boxes_xywh, int *boxes_xyxy, double *scores,
                   int *classes, int *index, int *counts,
                   int memory, int device, void *stream, int flags,
                   long long *stats);

/*
 * Both halves of the grid path in ONE call on device tensors: mgd_encode_targets on
 * (enc_batch, max_gt_boxes) ground-truth boxes and mgd_decode_nms on dec_batch images of
 * head outputs (arguments as in the two functions above; device memory only).  The two
 * halves are independent, so the library forks inside the call: the target encoder (an
 * HBM-bound write stream) runs on an internal stream underneath the decoder and the
 * latency-bound NMS, and the caller's stream joins both before the call's work counts as
 * complete -- to the caller it behaves like one stream-ordered operation on `stream`.
 * Class-range errors of the encoder are reported through mgd_poll_status (asynchronous
 * semantics of mgd_encode_targets without MGD_FLAG_SYNC); MGD_FLAG_SYNC synchronises
 * `stream` before returning.  The reference never runs the two halves together
 * (generators.py:1756 is training-side, multigrid_decode.py:347 inference-side); this
 * entry exists for pipelines that do -- and for the benchmark's combined step.
 */
MGD_API int mgd_encode_decode_nms(const mgd_head_config *cfg, const mgd_post_config *post,
                          const float *gt_boxes, int enc_batch, int max_gt_boxes,
                          float *const *y_true,
                          const float *const *preds, int dec_batch, const int *image_hw,
                          double *boxes_xywh, int *boxes_xyxy, double *scores,
                          int *classes, int *index, int *counts,
                          int device, void *stream, int flags);

/*
 * Dense decode only.  Replaces MultiGridDecoder.decode_predictions
 * (multigrid_decode.py:48-98) and, when image_hw != NULL, correct_boxes
 * (:185-235) applied per image.
 *   out (batch, cells, 5+C) float64: [x, y, w, h, score, class probabilities...]
 */
MGD_API int mgd_decode_dense(const mgd_head_config *cfg, const mgd_post_config *post,
                     const float *const *preds, int batch, const int *image_hw,
                     double *out, int memory, int device, void *stream, int flags);

/*
 * Greedy NMS on caller-supplied boxes.  Replaces StandardNMS/DIoUNMS/ClusterNMS
 * .apply_nms and nms_boxes (multigriddet/postprocess/nms.py:86-119, 154-187,
 * 323-356, 389-399).
 *   boxes (n, 4) float64 xywh, scores (n,) float64, classes (n,) int32 or NULL
 *   keep  (n,) int32: kept positions in descending score order (ties: lower
 *         position first); *n_keep (one int32 in the same memory space) = how many.
 */
MGD_API int mgd_nms(const double *boxes, const double *scores, const int *classes, int n,
            double nms_threshold, int nms_method, int per_class, int max_keep,
            int *keep, int *n_keep, int memory, int device, void *stream, int flags);

/*
 * Gaussian SoftNMS on caller-supplied boxes.  Replaces SoftNMS.apply_nms
 * (multigriddet/postprocess/nms.py:249-288).
 *   keep        (n,) int32: surviving positions in INPUT order (like boxes[keep_mask])
 *   soft_scores (n,) float64: decayed score of keep[i]
 *   n_keep      one int32 in the same memory space
 */
/*
 * Weighted Boxes Fusion on caller-supplied boxes.  Replaces WeightedBoxesFusion.
 * fuse_boxes / weighted_boxes_fusion (multigriddet/postprocess/wbf.py:38-290) for the
 * concatenated boxes of all models.
 *   boxes (n,4) f64 xywh, scores (n,) f64, classes (n,) int32,
 *   box_weights (n,) f64 = weights[model of box] or NULL (all 1)
 *   out_boxes (n,4) f64, out_scores (n,) f64, out_classes (n,) int32: the fused clusters in
 *   (class ascending, leader score descending) order; *n_out = how many.
 */
MGD_API int mgd_wbf(const double *boxes, const double *scores, const int *classes,
            const double *box_weights, int n, double iou_thr, double skip_box_thr,
            int conf_type, double *out_boxes, double *out_scores, int *out_classes,
            int *n_out, int memory, int device, void *stream, int flags);

MGD_API int mgd_soft_nms(const double *boxes, const double *scores, int n, double sigma,
                 double score_threshold, int *keep, double *soft_scores, int *n_keep,
                 int memory, int device, void *stream, int flags);

/*
 * Detection-to-ground-truth matching for mAP: TP / FP flags of every detection at
 * several IoU thresholds.  Replaces match_predictions_to_gt_cached and
 * match_predictions_to_gt (multigriddet/evaluation/metrics.py:147-218, 73-144) with the
 * IoU they consume (calculate_iou_matrix :28-70; BoxUtils.box_iou utils/boxes.py:16-58),
 * called per (class, threshold) from calculate_map (:541-815).  Ground truth is only
 * shared inside one (image, class) group, so images are matched independently.
 *
 *   det_boxes (batch, max_dets, 4) float64, det_scores (batch, max_dets) float64,
 *   det_classes (batch, max_dets) int32, det_counts (batch,) int32 -- the padded layout
 *   mgd_decode_nms emits;  gt_boxes (batch, max_gt, 4) float64, gt_classes (batch, max_gt)
 *   int32, gt_counts (batch,) int32;  iou_thresholds: num_thresholds host doubles.
 *   iou_mode  MGD_IOU_CORNER: boxes are xyxy, a ground truth is a candidate only if its
 *             IoU beats 0 (the cached matcher, the default path of calculate_map);
 *             MGD_IOU_CENTRE: the four numbers are read as [x, y, w, h] centre format and
 *             the first maximum wins even at IoU 0 (the un-cached matcher, which the
 *             reference uses for > 10000 predictions and for the per-scale APs).
 *   tp         (num_thresholds, batch, max_dets) uint8: 1 = true positive, 0 = false
 *              positive (padding slots 0), in detection-slot order
 *   matched_gt (num_thresholds, batch, max_dets) int32 or NULL: index of the claimed
 *              ground truth, -1 for false positives
 * Detections of an image are visited in descending score; equal scores: later slot first
 * (np.argsort(scores)[::-1] of a stable sort).
 */
enum { MGD_IOU_CORNER = 0, MGD_IOU_CENTRE = 1 };
MGD_API int mgd_match_detections(const double *det_boxes, const double *det_scores,
                         const int *det_classes, const int *det_counts, int batch, int max_dets,
                         const double *gt_boxes, const int *gt_classes, const int *gt_counts,
                         int max_gt, const double *iou_thresholds, int num_thresholds,
                         int iou_mode, unsigned char *tp, int *matched_gt,
                         int memory, int device, void *stream, int flags);

/*
 * Streaming mAP on the device.  Replaces the rest of calculate_map (multigriddet/evaluation/
 * metrics.py:541-815) after the matcher: the per-(class, threshold) precision / recall /
 * AP arithmetic (compute_precision_recall :221-246, compute_average_precision :249-300) and
 * the re-matches of the area-filtered per-scale APs (:745-800), fed batch by batch with the
 * padded tensors mgd_decode_nms emits, without building the reference's lists of dicts.
 *
 * A "view" is one matcher run over all updates: MGD_MAP_VIEW_CORNER and MGD_MAP_VIEW_CENTRE
 * match every detection with the cached (corner IoU) or un-cached (centre-format IoU) matcher
 * of mgd_match_detections; MGD_MAP_VIEW_S / _M / _L match with the centre matcher only the
 * detections and ground truth whose (x2-x1)*(y2-y1) lies in [-inf, 1024), [1024, 9216) or
 * [9216, inf) -- the per-scale sub-calls of calculate_map.  `views` in the config is the set
 * of views to match (bit 1 << view); the others stay empty.
 *
 *   mgd_map_record_bytes  bytes of device memory per padded detection slot of `records`
 *   mgd_map_update        matches one batch and writes one record per padded slot at
 *                         records + slot_offset * mgd_map_record_bytes(); slot_offset is the
 *                         sum of batch * max_dets over the earlier updates, so a record's
 *                         position is the detection's global index (image-major, slot order).
 *                         Adds the ground-truth counts of every view to gt_hist
 *                         (MGD_MAP_VIEWS, num_classes) int64, which the caller zeroes once.
 *                         det_boxes (batch, max_dets, 4) f64 xyxy, det_scores (batch,
 *                         max_dets) f64 -- FINITE values, det_classes (batch, max_dets) int32,
 *                         det_counts (batch,) int32; gt_boxes (batch, max_gt, 4) f64,
 *                         gt_classes (batch, max_gt) int32, gt_counts (batch,) int32.  A class id
 *                         outside [0, num_classes) is reported as MGD_ERR_CLASS_RANGE through
 *                         mgd_poll_status (MGD_FLAG_SYNC synchronises and reports it).
 *   mgd_map_compute       sorts the first num_slots records (class ascending, score descending,
 *                         equal scores: later detection first) and computes, per view and
 *                         class, the AP at every threshold:
 *                           ap_out          (MGD_MAP_VIEWS, C, T) f64, MGD_MAP_COCO: all-point
 *                                           interpolation + trapezoid
 *                           voc_points_out  (MGD_MAP_VIEWS, C, T, 11) f64, MGD_MAP_VOC: the max
 *                                           precision at recall >= voc_recalls[k] (0 if none);
 *                                           the AP is their mean
 *                           det_hist_out    (MGD_MAP_VIEWS, C) int64 detections per view and class
 *                         The trapezoid takes the recalls in the order np.argsort gives them
 *                         with NumPy's generic (non-SIMD) introsort, which permutes runs of
 *                         equal recall, as in the reference's own numbers.
 *                         The entry left NULL is the one the method does not use.  A class
 *                         without detections or without ground truth gets 0 here: the
 *                         reference's rules for those cases are the caller's (they need the
 *                         two histograms only).  Scratch comes from the calling thread's
 *                         workspace (mgd_release_workspace).
 * Device memory only; work is enqueued on `stream`.
 */
#define MGD_MAP_MAX_THRESHOLDS 32
#define MGD_MAP_VOC_POINTS 11
enum { MGD_MAP_COCO = 0, MGD_MAP_VOC = 1 };
enum { MGD_MAP_VIEW_CORNER = 0, MGD_MAP_VIEW_CENTRE = 1, MGD_MAP_VIEW_S = 2, MGD_MAP_VIEW_M = 3,
       MGD_MAP_VIEW_L = 4, MGD_MAP_VIEWS = 5 };
typedef struct {
    int num_classes;                  /* C >= 1                                            */
    int num_thresholds;               /* T in [1, MGD_MAP_MAX_THRESHOLDS]                  */
    int method;                       /* MGD_MAP_COCO or MGD_MAP_VOC                       */
    int views;                        /* bit mask of the views to match, non-empty         */
    double iou_thresholds[MGD_MAP_MAX_THRESHOLDS];
    double voc_recalls[MGD_MAP_VOC_POINTS];   /* np.arange(0, 1.1, 0.1) as the host has it  */
} mgd_map_config;
MGD_API int mgd_map_record_bytes(void);
MGD_API int mgd_map_update(const mgd_map_config *cfg, const double *det_boxes,
                   const double *det_scores, const int *det_classes, const int *det_counts,
                   int batch, int max_dets, const double *gt_boxes, const int *gt_classes,
                   const int *gt_counts, int max_gt, long long slot_offset, void *records,
                   long long *gt_hist, int device, void *stream, int flags);
MGD_API int mgd_map_compute(const mgd_map_config *cfg, const void *records, long long num_slots,
                    const long long *gt_hist, double *ap_out, double *voc_points_out,
                    long long *det_hist_out, int device, void *stream, int flags);

/*
 * Sharded streaming mAP.  Each of `world` ranks runs mgd_map_update on its own shard of every
 * global batch; the APs of a class are then computed on the one rank that owns it.  The result
 * equals mgd_map_compute over the whole data, which orders equal scores of a class later
 * detection first in global image order, so every record carries its GLOBAL slot: for local
 * slot j of update u on rank r it is G_u + lo_r * M_u + (j - L_u), where G_u is the sum of
 * n_total * max_dets over the earlier updates, lo_r the rank's first image of the update
 * (contiguous shards), M_u its max_dets and L_u the rank's slot_offset of the update.
 *
 *   mgd_map_partition       takes the first num_slots records of this rank and the update
 *                           segments (num_segments, 2) int64 (L_u, G_u + lo_r * M_u) with L_u
 *                           ascending (updates without local images may be left out); drops
 *                           padding slots; stamps each record's global slot into the record;
 *                           writes the records grouped by destination rank owner[class]
 *                           (owner (C,) int32, values in [0, world)), each group in local order,
 *                           to out_records (room for num_slots records), and the records per
 *                           destination to out_counts (world,) int64.  global_slots is the
 *                           sum of n_total * max_dets over all updates (<= 2^32, else
 *                           MGD_ERR_UNSUPPORTED); world <= 256.  An owner entry outside
 *                           [0, world) is reported as MGD_ERR_INVALID_ARGUMENT through
 *                           mgd_poll_status.
 *   mgd_map_compute_merged  mgd_map_compute over the records a rank received (any order):
 *                           sorted by class ascending, score descending, global slot descending,
 *                           with gt_hist the SUM of every rank's ground-truth counts.  Only the
 *                           (view, class) pairs with owner[class] == rank get their AP and
 *                           det_hist; the others get exact zeros, so the element-wise sum of the
 *                           ranks' ap_out / voc_points_out / det_hist_out is mgd_map_compute's.
 * Device memory only; work is enqueued on `stream`; scratch as for mgd_map_compute.
 */
MGD_API int mgd_map_partition(const mgd_map_config *cfg, const void *records, long long num_slots,
                      const long long *segments, int num_segments, long long global_slots,
                      const int *owner, int world, void *out_records, long long *out_counts,
                      int device, void *stream, int flags);
MGD_API int mgd_map_compute_merged(const mgd_map_config *cfg, const void *records,
                      long long num_records, const long long *gt_hist, const int *owner, int rank,
                      double *ap_out, double *voc_points_out, long long *det_hist_out,
                      int device, void *stream, int flags);

/*
 * Precision-recall curves and confidence operating points of the full-set views.
 *
 *   mgd_map_compute_pr         mgd_map_compute, and for every view in pr->views (MGD_MAP_VIEW_CORNER
 *                              and / or MGD_MAP_VIEW_CENTRE, a subset of cfg->views) the curves and
 *                              operating points below
 *   mgd_map_compute_merged_pr  mgd_map_compute_merged, and the same for the classes owner[] gives
 *                              `rank`; the other classes have empty curve segments and exact zeros in
 *                              best_f1 / best_index / at_confidence, so the element-wise sum of the
 *                              ranks' tables is the unsharded one
 *
 * Curves (CSR): the records of class c are [offsets[c], offsets[c + 1]) in the sort's order (score
 * descending, equal scores later detection first), offsets[num_classes] records in all.  For
 * record k of its class (0-based), at threshold t of view view_list[i] (the i-th set bit of views):
 *   scores[offsets[c] + k]                    its score
 *   precision[(i * T + t) * capacity + offsets[c] + k] = cum_tp / ((k + 1) + 1e-8)
 *   recall   [(i * T + t) * capacity + offsets[c] + k] = cum_tp / (n_gt + 1e-8)
 * in float64 in compute_precision_recall's (metrics.py:221-246) operation order.  A class without
 * detections has an empty segment (the reference returns ([0.0], [0.0]) for it).
 * Operating points, per (i, class, threshold); f1 = 2.0 * p * r / (p + r), 0 where p + r == 0:
 *   best_f1 (V, C, T, 4)     (confidence = score[k], precision, recall, f1) at the first record k, in
 *                            descending-score order, of maximum f1 among the records that end a
 *                            run of equal scores (the only points a score >= confidence threshold
 *                            can produce); zeros if that maximum is 0 or the class has no records
 *   best_index (V, C, T)     that k, or -1 where best_f1 is zeros
 *   at_confidence (V, C, T, Q, 3)  (precision, recall, f1) at record K - 1, K the class's records
 *                            with score >= confidences[q]; zeros where K == 0.  NULL when Q == 0
 * capacity must be >= num_slots (num_records for the merged form).  confidences is HOST memory
 * (finite values, at most MGD_MAP_MAX_CONFIDENCES); every output is device memory.
 */
#define MGD_MAP_MAX_CONFIDENCES 32
typedef struct {
    int views;                        /* bit mask of MGD_MAP_VIEW_CORNER / _CENTRE, non-empty  */
    int num_confidences;              /* Q in [0, MGD_MAP_MAX_CONFIDENCES]                     */
    const double *confidences;        /* (Q,) host                                             */
    long long capacity;               /* records per curve row of scores / precision / recall  */
    long long *offsets;               /* (C + 1,) int64                                        */
    double *scores;                   /* (capacity,)                                           */
    double *precision;                /* (V, T, capacity), V = set bits of views               */
    double *recall;                   /* (V, T, capacity)                                      */
    double *best_f1;                  /* (V, C, T, 4)                                          */
    long long *best_index;            /* (V, C, T)                                             */
    double *at_confidence;            /* (V, C, T, Q, 3)                                       */
} mgd_map_pr;
MGD_API int mgd_map_compute_pr(const mgd_map_config *cfg, const void *records, long long num_slots,
                      const long long *gt_hist, double *ap_out, double *voc_points_out,
                      long long *det_hist_out, const mgd_map_pr *pr, int device, void *stream,
                      int flags);
MGD_API int mgd_map_compute_merged_pr(const mgd_map_config *cfg, const void *records,
                      long long num_records, const long long *gt_hist, const int *owner, int rank,
                      double *ap_out, double *voc_points_out, long long *det_hist_out,
                      const mgd_map_pr *pr, int device, void *stream, int flags);

/*
 * Loss-side ignore mask.  Replaces MultiGridLoss._compute_ignore_mask and
 * _compute_iou_batch (multigriddet/losses/multigrid_loss.py:494-703, 445-492), called once
 * per layer from the loss (:316).  Forward only: the reference casts the mask from a
 * boolean and wraps the two IoU maps in stop_gradient.  TensorFlow graph code: parity is
 * pinned against the two methods' own source executed over a NumPy stand-in for the tf.* /
 * K.* ops (the test suite's oracle/tf_shim.py; fixtures tests/golden/ignoremask_cases.npz),
 * reference quirks included -- see csrc/loss.cu; IoU values to 1e-5 (float32 exp / tanh).
 *
 *   y_pred, y_true  num_layers pointers, each (batch, grid_h, grid_w, 5+A_l+C) float32
 *   ignore_mask          (batch, grid_h, grid_w, 1) float32 per layer: 1 where the best IoU of
 *                        the cell's predicted boxes with the image's ground truth on that
 *                        layer exceeds ignore_thresh and the cell is not positive
 *   assigned_anchor_iou  same shape: IoU of the assigned anchor's box on positive cells, else 0
 *   max_iou_map          same shape: best IoU over the anchors
 *   eps                  Keras epsilon of the reference (1e-7)
 */
MGD_API int mgd_ignore_mask(const mgd_head_config *cfg, const float *const *y_pred,
                    const float *const *y_true, int batch, double ignore_thresh, double eps,
                    float *const *ignore_mask, float *const *assigned_anchor_iou,
                    float *const *max_iou_map, int memory, int device, void *stream, int flags);

/*
 * Target encoder and loss-side ignore mask in one call (SURVEY.md 8f-2 as specified): the
 * ignore mask is fed by the encoder's owner table and box records, so the ground truth of the
 * loss is never re-derived from the dense y_true tensor (4 bytes per cell are read instead of
 * 352) and y_true itself is optional.  Replaces preprocess_true_boxes (generators.py:3393-3473)
 * followed by MultiGridLoss._compute_ignore_mask (losses/multigrid_loss.py:494-703) on the same
 * boxes; results are identical to mgd_encode_targets + mgd_ignore_mask.  Device memory only.
 *   boxes (batch, max_boxes, 5) float32;  y_pred L x (batch, gh, gw, 5+A+C) float32;
 *   y_true L pointers or NULL (skip writing the targets);  outputs as in mgd_ignore_mask.
 * Class-range errors are reported through mgd_poll_status (MGD_FLAG_SYNC synchronises first).
 */
MGD_API int mgd_encode_ignore_mask(const mgd_head_config *cfg, const float *boxes, int batch,
                           int max_boxes, const float *const *y_pred, float *const *y_true,
                           double ignore_thresh, double eps, float *const *ignore_mask,
                           float *const *assigned_anchor_iou, float *const *max_iou_map,
                           int device, void *stream, int flags);

/*
 * Box-side pre-step of the encoder, over a batch (so the (B, N, 5) tensor mgd_encode_targets
 * consumes can be produced on the device).
 *
 * mgd_reshape_boxes replaces reshape_boxes (multigriddet/data/augmentation.py:112-164),
 * called per image from the legacy loader (data/generators.py:2435, 2463): scale into the
 * padded image and add the paste offset (boxes * padding / src + d), optional horizontal /
 * vertical flip, clip (x1, y1 >= 0; x2 <= target_w; y2 <= target_h), drop boxes whose width
 * or height is <= 1.  Survivors keep their order (the reference's np.random.shuffle of the
 * rows, :146, is the caller's business: pass the rows in the order wanted), the rest of each
 * image's N slots is zero.
 *   boxes   (batch, max_boxes, 5) [x1, y1, x2, y2, class]; MGD_BOXES_I32: int32, every
 *           stored coordinate truncated toward zero like NumPy's float -> int32 assignment
 *           (the legacy loader's dtype, generators.py:2429); MGD_BOXES_F64: float64
 *   counts  (batch,) int32 valid rows per image, or NULL = all max_boxes rows
 *   params  (batch, 10) int32: src_w, src_h, target_w, target_h, padding_w, padding_h, dx, dy,
 *           horizontal_flip, vertical_flip
 *   out     (batch, max_boxes, 5) same dtype; out_f32: optional float32 copy (the encoder's
 *           input dtype); out_counts (batch,) int32 or NULL
 *
 * mgd_mosaic_merge_boxes replaces merge_mosaic_bboxes (augmentation.py:606-667) under
 * random_mosaic_augment (:670-746): output image b takes the boxes of source images
 * params[b][0..3] (top-left, bottom-left, bottom-right, top-right), cuts them at
 * (crop_x, crop_y) = params[b][4..5], drops boxes left narrower than max(10, 1% of the
 * image), concatenates in (quadrant, row) order and keeps the first max_boxes.
 *   boxes (num_sources, max_boxes, 5) float64 (zero rows = padding); params (batch, 6) int32
 */
enum { MGD_BOXES_I32 = 0, MGD_BOXES_F64 = 1 };
MGD_API int mgd_reshape_boxes(const void *boxes, int boxes_dtype, const int *counts,
                      const int *params, int batch, int max_boxes, void *out, float *out_f32,
                      int *out_counts, int memory, int device, void *stream, int flags);
MGD_API int mgd_mosaic_merge_boxes(const double *boxes, int num_sources, int max_boxes,
                           const int *params, int batch, int height, int width, double *out,
                           float *out_f32, int *out_counts,
                           int memory, int device, void *stream, int flags);

/*
 * tf.data box pre-step: what happens to an image's boxes between the annotation parser and
 * tf_preprocess_true_boxes on the reference's DEFAULT training path (build_tf_dataset,
 * multigriddet/data/generators.py):
 *   - the letterbox / multi-scale box transform of _preprocess_image_and_boxes (:1859-1916,
 *     with tf_letterbox_resize :167-209): boxes * scale + padding offset, float32;
 *   - the optional horizontal flip of tf_random_horizontal_flip (:227-256), the coin handed
 *     in by the caller (hflip);
 *   - padded_batch to max_boxes_per_image rows (:1963-1976) and _expand_box_capacity
 *     (:1983-2034): zero rows up to max_boxes_per_image * expansion (1 / 2 / 4 / 8 for none /
 *     MixUp / Mosaic / both).
 * The crop / rotate / gridmask augmentations in between are image-space work and stay in the
 * reference.
 *   boxes   (batch, max_in, 5) float32 [x1, y1, x2, y2, class], original-image pixels
 *   counts  (batch,) int32 valid rows per image, or NULL (= max_in)
 *   params  (batch, 6) int32: src_h, src_w, scale_h, scale_w (the multi-scale shape sampled
 *           for the image, 0 0 = no multi-scale), hflip, reserved
 *   out     (batch, max_boxes_per_image * expansion, 5) float32 -- the tensor
 *           mgd_encode_targets consumes; rows beyond min(count, max_boxes_per_image) are zero
 *           (TensorFlow's padded_batch raises on a longer component; here it is truncated)
 */
MGD_API int mgd_letterbox_boxes(const float *boxes, const int *counts, const int *params,
                        int batch, int max_in, int input_h, int input_w,
                        int max_boxes_per_image, int expansion, float *out,
                        int memory, int device, void *stream, int flags);

/*
 * IoU matrix of two sets of xyxy boxes.  Replaces calculate_iou_matrix
 * (multigriddet/evaluation/metrics.py:28-70).  out (n, m) float64.
 */
MGD_API int mgd_iou_matrix(const double *boxes1, int n, const double *boxes2, int m, double *out,
                   int memory, int device, void *stream, int flags);

/*
 * Deferred device-side status of asynchronous calls issued by this thread on
 * `device` (class-range errors found by the encode kernel).  Synchronises `stream`, then
 * reads and clears the thread's status word (asynchronous calls OR their bits into one
 * persistent device word per thread and device; nothing accumulates if it is never polled).
 */
MGD_API int mgd_poll_status(int device, void *stream);

/*
 * Page-locked host memory for tensors that cross the boundary as MGD_MEM_HOST.  The
 * reference returns fresh NumPy arrays from every call (generators.py:3425-3429,
 * multigrid_decode.py:409-422); arrays in pageable memory move at ~6-11 GB/s through the
 * driver's bounce buffer, page-locked ones at the link rate (~55 GB/s), so the Python
 * shim allocates its outputs here and recycles them.  Portable across CUDA contexts.
 */
#include <stddef.h>
MGD_API int mgd_host_alloc(size_t bytes, void **ptr);
MGD_API int mgd_host_free(void *ptr);

/*
 * Detection exchange: the one exchange step of the image-sharded multi-GPU path.
 * The reference evaluates image by image on one host (evaluator.py:254-289) and owns every
 * detection afterwards; with the batch sharded over the GPUs of a node (one process per GPU),
 * each rank decodes its slice and every rank needs every image's padded rows.  An exchange
 * is `bytes` of device memory per rank, every rank's buffer mapped into every process through
 * CUDA IPC.  Detection outputs of mgd_decode_nms / mgd_encode_decode_nms that the caller
 * places inside its exchange buffer -- at the offsets they have in the whole-batch tensors --
 * are written by the NMS kernels into ALL ranks' buffers as they are produced (peer stores,
 * NVLink on a B200 box): no collective call, no packing pass.  Such a call is collective:
 * every rank of the exchange makes it, in the same order, with >= 1 image; all of its
 * output tensors (any may be NULL except counts) must lie in the buffer, the two box
 * tensors 16-byte aligned (remote rows travel as 16-byte stores); when the call's work
 * completes on `stream`, the rows of all ranks are present locally.
 * Ranks wait for each other on the device (flag words in the buffers); a peer that does not
 * arrive within 20 s is counted in mgd_exchange_timeouts instead of hanging the stream.
 *
 *   create   allocates this rank's buffer and returns its IPC handle (MGD_IPC_HANDLE_BYTES)
 *   connect  takes the handles of all ranks, (world_size, MGD_IPC_HANDLE_BYTES) in rank
 *            order (exchanged by the host: torch.distributed.all_gather, MPI, a file ...),
 *            and maps the peers' buffers; world_size == 1 needs no connect
 *   buffer   this rank's buffer (device pointer, zero-initialised)
 *   destroy  unmaps the peers and frees this rank's buffer after synchronising the device;
 *            the ranks must agree that no mirrored call is in flight any more (a barrier of
 *            the host-side job) before any of them destroys its end
 * One thread per exchange at a time: the calls on it are ordered by a per-exchange counter.
 */
#define MGD_IPC_HANDLE_BYTES 64
typedef struct mgd_exchange mgd_exchange;
MGD_API int mgd_exchange_create(int device, int world_size, int rank, size_t bytes,
                        mgd_exchange **exchange, unsigned char *handle);
MGD_API int mgd_exchange_connect(mgd_exchange *exchange, const unsigned char *handles);
MGD_API int mgd_exchange_buffer(mgd_exchange *exchange, void **base, size_t *bytes);
MGD_API int mgd_exchange_timeouts(mgd_exchange *exchange, void *stream, int *timeouts);
MGD_API int mgd_exchange_destroy(mgd_exchange *exchange);

/*
 * Host-memory calls stage through device buffers cached per (host thread, device); this
 * returns the calling thread's cached buffers to the driver.  Optional: they are reused
 * by the thread's next call and sized by the largest batch chunk (<= ~0.5 GB).
 */
MGD_API int mgd_release_workspace(void);

/*
 * Per-kernel timing for the calling thread (observability; the reference only has
 * wall-clock prints, evaluator.py:496-525).  Between begin and end every kernel
 * the library launches for this thread is bracketed by CUDA events on the
 * launching stream.  mgd_profile_end synchronises those events and returns, per
 * kernel kind, the summed device time in ms and the number of launches:
 *   [0] encode_assign  [1] encode_fill  [2] decode_compact  [3] nms  [4] other
 */
#define MGD_PROFILE_KINDS 5
MGD_API int mgd_profile_begin(void);
MGD_API int mgd_profile_end(double *ms, long long *launches);

/* ---- DLPack zero-copy variants -------------------------------------------------
 * The tensors arrive as DLTensor* (dlpack.h ABI, v0.8+): dtype, shape, strides and
 * device are validated and the call forwards to the pointer entry point above.
 * kDLCPU / kDLCUDAHost -> MGD_MEM_HOST, kDLCUDA -> MGD_MEM_DEVICE on that device.
 * The library only borrows the tensors for the duration of the call (for async
 * device calls: until `stream` reaches the enqueued work); it never calls a
 * DLManagedTensor deleter.
 */
struct DLTensor;
MGD_API int mgd_encode_targets_dlpack(const mgd_head_config *cfg, const struct DLTensor *boxes,
                              struct DLTensor *const *y_true, void *stream, int flags,
                              long long *stats);
MGD_API int mgd_decode_nms_dlpack(const mgd_head_config *cfg, const mgd_post_config *post,
                          const struct DLTensor *const *preds,
                          const struct DLTensor *image_hw,
                          struct DLTensor *boxes_xywh, struct DLTensor *boxes_xyxy,
                          struct DLTensor *scores, struct DLTensor *classes,
                          struct DLTensor *index, struct DLTensor *counts,
                          void *stream, int flags, long long *stats);

#ifdef __cplusplus
}
#endif
#endif /* MGD_H_ */
