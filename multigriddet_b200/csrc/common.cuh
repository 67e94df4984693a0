// Shared declarations of libmgd's CUDA translation units (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/mgd.h"

#define MGD_MAX_TOTAL_ANCHORS (MGD_MAX_LAYERS * MGD_MAX_ANCHORS_PER_LAYER)

// Device-side view of mgd_head_config plus derived constants.
struct HeadGeom {
    int L, C;
    int in_h, in_w;
    int gh[MGD_MAX_LAYERS], gw[MGD_MAX_LAYERS];
    int na[MGD_MAX_LAYERS];            // anchors per layer
    int D[MGD_MAX_LAYERS];             // channels per cell = 5 + A + C
    int anchor_first[MGD_MAX_LAYERS];  // global index of the layer's first anchor
    int K;                             // total anchors
    int cell_off[MGD_MAX_LAYERS];      // first cell of the layer within one image
    int cells;                         // cells per image over all layers
    int anchors_f64;
    float anc32[MGD_MAX_TOTAL_ANCHORS][2];
    double anc64[MGD_MAX_TOTAL_ANCHORS][2];
};

// ---- encode ---------------------------------------------------------------
// One record per valid ground-truth box, written by the assign kernel and read
// by the fill kernel for the (few) cells the box owns.
struct __align__(16) BoxRec {
    double fx, fy;     // fractional centre offsets inside the centre cell (f64 like NumPy)
    float tw, th;      // log size ratios to the matched anchor
    int hot_anchor;    // channel 5 + k
    int hot_class;     // channel 5 + A + class
};

struct EncodeArgs {
    HeadGeom g;
    int B, N;
    const float* boxes;               // (B, N, 5)
    float* y[MGD_MAX_LAYERS];         // (B, gh, gw, D)
    int* table;                       // layer-major owner table: [l][b][cell]
    int* big_tables;                  // (B, 2, cells) scratch when the tables exceed shared memory, else nullptr
    BoxRec* recs;                     // (B, N)
    int tf_compat;                    // 1: tf_preprocess_true_boxes semantics (MGD_FLAG_TF_COMPAT)
    int* status;                      // bit0: class >= C, bit1: negative class on a valid box
    unsigned long long* stats;        // [valid boxes, skipped writes, positive cells, -]
};

// ---- decode / NMS ---------------------------------------------------------
// One candidate (score >= confidence) as the decode kernel emits it: 32 bytes.
// The box is reconstructed from the raw logits by the NMS kernel.
struct __align__(16) Cand {
    float score;         // float32 score in the reference's operation order
    int index;           // flat cell index (layer, row, col)
    float t[4];          // raw tx, ty, tw, th
    int cls;             // argmax class
    int anchor;          // global index of the argmax anchor
};

struct __align__(16) BoxD { double x, y, w, h; };   // [x_min, y_min, w, h], image pixels

struct DecodeArgs {
    HeadGeom g;
    int B;
    const float* pred[MGD_MAX_LAYERS];
    const int* image_hw;              // (B, 2) or nullptr
    int use_softmax, rescore;
    double confidence;
    float obj_logit_min;              // conservative prefilter on the raw objectness logit
    float score_lo;                   // confidence * (1 - 1e-3): bound for the fast prefilters
    long long rows_in_layer[MGD_MAX_LAYERS];    // B * gh * gw
    unsigned long long cells_magic[MGD_MAX_LAYERS];   // floor(2^64 / (gh*gw)) + 1 (0 when gh*gw == 1): row -> image
    Cand* cand;                       // (B, cells)
    int* counts;                      // (B,)
    int chunk_blocks;                 // consecutive 32-row blocks a producer warp takes at a time
    int debug;                        // MGD_DECODE_DEBUG (measurements only): 1 scan only, 2 no level 3, 4 no level 2/3
};

#define MGD_MAX_MIRRORS 7            /* peers of a detection exchange: world size <= 8 */
struct NmsArgs {
    HeadGeom g;                       // decode mode: geometry for the box reconstruction
    int B;
    int cap;                          // candidate slots per image
    const Cand* cand;                 // decode mode: (B, cap) records; nullptr in explicit mode
    const double* in_boxes;           // explicit mode (mgd_nms, B == 1): (n,4) xywh
    const double* in_scores;          //   (n,)
    const int* in_classes;            //   (n,) or nullptr
    BoxD* boxes;                      // decode mode scratch: (B, cap) reconstructed boxes
    const int* counts;
    const int* image_hw;              // (B,2) or nullptr (then in_h, in_w)
    int in_h, in_w;
    double thr;
    int use_diou, per_class, max_boxes;
    int skip_small;                   // nms_kernel: skip images with <= this many candidates
    int soft;                         // 1: Gaussian SoftNMS (soft_nms_kernel)
    double soft_sigma, soft_thr;
    double* soft_scratch;             // soft: (B, cap) decayed scores; wbf: (B, cap, 5) fused clusters
    int wbf;                          // 1: weighted boxes fusion (wbf_kernel); thr = iou_thr,
                                      //    soft_thr = skip_box_thr
    int wbf_conf_type;                // 0 avg, 1 max, 2 mean(score * weight)
    const double* in_weights;         // explicit mode: per-box model weight or nullptr
    int* wbf_ints;                    // (B, 4, cap) int scratch
    int* next_image;                  // nms_warp_kernel: work counter (zeroed by the caller)
    unsigned long long* sort_scratch; // (B, 2*pow2(cap)) u64, used when count > smem capacity
    int sort_scratch_stride;          // elements (pairs) per image in sort_scratch
    unsigned char* kept_scratch;      // kept-box list in global memory when max_boxes is large
    size_t kept_scratch_stride;       // bytes per image
    double* out_xywh; int* out_xyxy; double* out_scores; int* out_classes; int* out_index;
    int* out_counts;
    unsigned long long* stats;        // [candidates, detections]
    // detection exchange (mgd_exchange_*): the outputs above lie in this rank's exchange buffer
    // and every store is repeated at the same offset of each peer's buffer (nms.cu: mirror_store)
    int n_mirrors;
    long long mirror_delta[MGD_MAX_MIRRORS];
    int warp_ctas_per_sm;             // host side: resident nms_warp_kernel CTAs per SM (0: all that fit)
};

// ---- detection exchange (exchange.cu, api.cu: mgd_exchange_*) ----------------------------
#define MGD_EXCHANGE_MAX_RANKS 8
#define MGD_EXCHANGE_HEADER_BYTES 512     /* flag words in front of the caller's bytes */
#define MGD_EXCHANGE_TIMEOUT_WORD 32      /* header word counting barrier timeouts */
struct ExchangeView {
    int world, rank;
    unsigned* header[MGD_EXCHANGE_MAX_RANKS];   // every rank's header as mapped in THIS process:
                                                // [kind 0 | 1][source rank] epochs, timeout word
};
enum { MGD_EXCHANGE_SIGNAL = 1, MGD_EXCHANGE_WAIT = 2 };
cudaError_t launch_exchange_barrier(const ExchangeView& v, int which, unsigned epoch, int phase,
                                    cudaStream_t stream);

// ---- mAP matching -----------------------------------------------------------
#define MGD_MAX_IOU_THRESHOLDS 16
struct MatchArgs {
    int B, M, N, T;
    const double* det_boxes;          // (B, M, 4)
    const double* det_scores;         // (B, M)
    const int* det_classes;           // (B, M)
    const int* det_counts;            // (B,)
    const double* gt_boxes;           // (B, N, 4)
    const int* gt_classes;            // (B, N)
    const int* gt_counts;             // (B,)
    double thr[MGD_MAP_MAX_THRESHOLDS];   // T <= MGD_MAX_IOU_THRESHOLDS for mgd_match_detections
    int mode;                         // 0: corner IoU, candidate must beat 0 (cached matcher);
                                      // 1: centre-format IoU, first maximum (un-cached matcher)
    int band;                         // 0: every box; 1 + b: only boxes in area band b
                                      // (map_area_band): the others are left out of the walk
                                      // like calculate_map's area filter (metrics.py:745-800)
    unsigned char* tp;                // (T, B, M)
    int* matched;                     // (T, B, M) or nullptr
    int* next_image;                  // work counter, zeroed by the caller
};

// ---- detection confusion matrix (match.cu: confusion_kernel) ---------------------------
// Stage 1 is one match_kernel walk at `thr` (T = 1, no band); confusion_kernel takes its claims
// and runs the cross-class stage for every confidence.
struct ConfusionArgs {
    int B, M, N, C, Q;
    int mode;                         // MGD_IOU_CORNER / MGD_IOU_CENTRE, as for stage 1
    double thr;
    double conf[MGD_MAP_MAX_CONFIDENCES];
    const double* det_boxes; const double* det_scores; const int* det_classes; const int* det_counts;
    const double* gt_boxes; const int* gt_classes; const int* gt_counts;
    const int* matched;               // (B, M) stage-1 claim of each detection, -1 = none
    unsigned long long* matrix;       // (Q, C+1, C+1) counts, added to
    int* next_image;                  // work counter, zeroed by the caller
    int* status;                      // bit 4: class id outside [0, C)
};
cudaError_t launch_confusion(const ConfusionArgs& a, int num_sms, cudaStream_t stream);

// Area band of an xyxy box for the per-scale APs: 0 = S (-inf, 1024), 1 = M [1024, 9216),
// 2 = L [9216, inf), 3 = none (NaN area).  The area is (x2-x1)*(y2-y1) in float64
// (metrics.py:_box_area) and the bounds are compared as _filter_by_area does.
__device__ __forceinline__ int map_area_band(const double* b)
{
    const double area = __dmul_rn(__dsub_rn(b[2], b[0]), __dsub_rn(b[3], b[1]));
    if (area < 1024.0) return 0;
    if (area >= 1024.0 && area < 9216.0) return 1;
    if (area >= 9216.0) return 2;
    return 3;
}

// ---- streaming mAP (map.cu) ---------------------------------------------------------------
// One record per padded detection slot, written by map_update and sorted by map_compute.
struct __align__(8) MapRec {
    double score;                     // as given (scores are finite)
    int cls;                          // -1: padding slot (or a class id reported out of range)
    int band;                         // map_area_band of the detection
    unsigned bits[MGD_MAP_VIEWS];     // bit t: true positive at threshold t in that view
    unsigned pad;
};
static_assert(sizeof(MapRec) == 40, "MapRec is the record format of mgd_map_record_bytes");

struct MapWriteArgs {
    int B, M, N, T, C, views;
    const double* det_boxes; const double* det_scores; const int* det_classes; const int* det_counts;
    const double* gt_boxes; const int* gt_classes; const int* gt_counts;
    const unsigned char* tp[MGD_MAP_VIEWS];   // (T, B, M) flags of each matched view, else nullptr
    MapRec* recs;                     // the update's first record
    unsigned long long* gt_hist;      // (MGD_MAP_VIEWS, C)
    int* status;                      // bit 2: class id outside [0, C)
};
cudaError_t launch_map_write(const MapWriteArgs& a, cudaStream_t stream);

// average recall (recall.cu: map_recall_kernel, mgd_map_recall_update): reads one update's
// records only
struct MapRecallArgs {
    int B, M, C, T, K, views;
    int limits[MGD_MAP_MAX_RECALL_LIMITS];    // strictly increasing, >= 1
    const MapRec* recs;               // the update's first record, (B, M)
    unsigned long long* tp;           // (MGD_MAP_VIEWS, C, T, K) counts, added to
    int* next_image;                  // work counter, zeroed by the caller
};
cudaError_t launch_map_recall(const MapRecallArgs& a, int num_sms, cudaStream_t stream);

// ---- detection error analysis (match.cu: tide_kernel, mgd_tide_update) -------------------
// The base is one match_kernel walk at t_f (T = 1, no band); tide_kernel types the false positives
// and misses and writes the records of every fixed set.
struct TideArgs {
    int B, M, N, C;
    int mode;                         // MGD_IOU_CORNER / MGD_IOU_CENTRE, as for the base walk
    double t_f, t_b;
    const double* det_boxes; const double* det_scores; const int* det_classes; const int* det_counts;
    const double* gt_boxes; const int* gt_classes; const int* gt_counts;
    const int* matched;               // (B, M) base claim of each detection, -1 = none
    MapRec* recs;                     // the update's first record: (B, MGD_TIDE_SETS, M)
    unsigned long long* gt_hist;      // (MGD_TIDE_SETS * C) the CORNER row, added to
    unsigned long long* counts;       // (C, MGD_TIDE_ERRORS), added to
    int* next_image;                  // work counter, zeroed by the caller
    int* status;                      // bit 5: class id outside [0, C)
};
cudaError_t launch_tide(const TideArgs& a, int num_sms, cudaStream_t stream);

// scratch of map_compute (bytes), and the enqueue of sort + AP kernels; with `pr` (validated by
// the caller) also the curves and operating points of mgd_map_compute_pr
size_t map_compute_scratch_bytes(long long n, int T);
cudaError_t launch_map_compute(const mgd_map_config& cfg, const MapRec* recs, long long n,
                               const unsigned long long* gt_hist, double* ap, double* voc,
                               unsigned long long* det_hist, void* scratch, cudaStream_t stream,
                               const mgd_map_pr* pr = nullptr);
// the same over records stamped by map_partition (ties broken by the global slot, descending);
// only the classes `owner` gives to `rank` get APs, the others exact zeros
cudaError_t launch_map_compute_merged(const mgd_map_config& cfg, const MapRec* recs, long long n,
                                      const unsigned long long* gt_hist, const int* owner, int rank,
                                      double* ap, double* voc, unsigned long long* det_hist, void* scratch,
                                      cudaStream_t stream, const mgd_map_pr* pr = nullptr);

// mgd_map_partition: the records grouped by the rank that owns their class, in local order,
// padding dropped, each stamped with its global slot (MapRec::pad)
struct MapPartitionArgs {
    const MapRec* recs; long long n;  // the rank's first n records
    int C;
    const long long* segs;            // (num_segs, 2): first local slot of an update, its global slot
    int num_segs;
    const int* owner;                 // (C,) rank that owns each class
    int world;                        // <= 256 (one radix digit)
    MapRec* out;                      // (n,) records, rank by rank
    long long* counts;                // (world,) records per rank
    int* status;                      // bit 3: owner entry outside [0, world)
};
size_t map_partition_scratch_bytes(long long n);
cudaError_t launch_map_partition(const MapPartitionArgs& a, void* scratch, cudaStream_t stream);

// ---- box-side pre-step of the encoder (reshape_boxes / merge_mosaic_bboxes) ---
struct BoxOpArgs {
    int B, N;                         // output images, box slots per image
    const void* in;                   // reshape: (B, N, 5) int32 | float64; mosaic: (n_src, N, 5) float64
    const int* counts;                // reshape: valid rows per image or nullptr (= N)
    const int* params;                // reshape: (B, 10); mosaic: (B, 6)
    int n_src, height, width;         // mosaic: source images, mosaic image size
    void* out;                        // (B, N, 5) in the input dtype
    float* out_f32;                   // optional float32 copy (what the encoder consumes)
    int* out_counts;                  // (B,) or nullptr
};

// ---- loss-side ignore mask (multigrid_loss.py:494-703) ------------------------
struct LossArgs {
    HeadGeom g;
    int B;
    const float* y_pred[MGD_MAX_LAYERS];   // (B, gh, gw, D) raw head outputs
    const float* y_true[MGD_MAX_LAYERS];   // (B, gh, gw, D) encoder targets
    float ignore_thresh, eps;
    float* ignore[MGD_MAX_LAYERS];         // (B, gh, gw, 1)
    float* assigned[MGD_MAX_LAYERS];       // (B, gh, gw, 1) IoU of the assigned anchor, 0 on negatives
    float* max_iou[MGD_MAX_LAYERS];        // (B, gh, gw, 1) best IoU over anchors
    void* gt_boxes;                        // scratch: (B, cells, 2) x 16 B corner boxes (raw | unique)
    float* gt_area;                        // scratch: (B, cells, 2)
    int* gt_count;                         // scratch: (B, L) unique ground-truth boxes
    // fed by the target encoder instead of a dense y_true (mgd_encode_ignore_mask): the assign
    // kernel's owner table (layer-major, [l][b][cell]: -1 or box record * 16 + neighbour id) and
    // its box records; y_true[] is then unused
    const int* table;
    const BoxRec* recs;
};

// NVTX ranges (header-only NVTX3: no link dependency; a no-op unless a profiler injects
// itself) around every C-ABI entry point and every kernel launch group, so nsys / ncu
// attribute GPU time to the reference function each kernel replaces.
#include <nvtx3/nvToolsExt.h>
struct nvtx_range {
    explicit nvtx_range(const char* name) { nvtxRangePushA(name); }
    ~nvtx_range() { nvtxRangePop(); }
    nvtx_range(const nvtx_range&) = delete;
    nvtx_range& operator=(const nvtx_range&) = delete;
};

// per-kernel CUDA-event timing (mgd_profile_begin / mgd_profile_end)
enum ProfKind { PROF_ENCODE_ASSIGN = 0, PROF_ENCODE_FILL = 1, PROF_DECODE_COMPACT = 2,
                PROF_NMS = 3, PROF_OTHER = 4, PROF_KINDS = 5 };
void prof_mark_begin(int kind, cudaStream_t stream);
void prof_mark_end(int kind, cudaStream_t stream);
void prof_group_begin(int kind, cudaStream_t stream);   // one event pair around several launches of `kind`
void prof_group_end(int kind, cudaStream_t stream);

// launchers (each enqueues on `stream` and returns the launch error, if any)
cudaError_t launch_encode(const EncodeArgs& a, int num_sms, cudaStream_t stream);
cudaError_t launch_encode_assign(const EncodeArgs& a, cudaStream_t stream,
                                 bool overlap_previous = false);                 // owner tables + box records
cudaError_t launch_encode_fill(const EncodeArgs& a, int num_sms, cudaStream_t stream,
                               bool overlap_previous = false);                   // the y_true writer
cudaError_t launch_decode(const DecodeArgs& a, int num_sms, cudaStream_t stream);
cudaError_t launch_nms(const NmsArgs& a, int num_sms, cudaStream_t stream);
size_t encode_assign_smem_bytes(const HeadGeom& g, int N);
bool encode_needs_big_tables(const HeadGeom& g, int N);
int nms_smem_capacity();
size_t nms_kept_bytes(int max_boxes);
cudaError_t launch_decode_dense(const DecodeArgs& a, const int* image_hw, double* out,
                                cudaStream_t stream);
cudaError_t launch_match(const MatchArgs& a, int num_sms, cudaStream_t stream);
cudaError_t launch_iou_matrix(const double* b1, int n, const double* b2, int m, double* out,
                              cudaStream_t stream);
cudaError_t launch_reshape_boxes(const BoxOpArgs& a, int boxes_i32, cudaStream_t stream);
cudaError_t launch_mosaic_merge(const BoxOpArgs& a, cudaStream_t stream);
cudaError_t launch_letterbox_boxes(const float* in, const int* counts, const int* params, int B,
                                   int n_in, int n_keep, int capacity, int input_h, int input_w,
                                   float* out, cudaStream_t stream);
cudaError_t launch_ignore_mask(const LossArgs& a, cudaStream_t stream);
cudaError_t launch_keep_from_index(const int* index, const int* counts, int max_keep, int* keep,
                                   int* n_keep, cudaStream_t stream);
