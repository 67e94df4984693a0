// Detection-to-ground-truth matching for mAP, sm_100a.
//
// Replaces the Python loops of match_predictions_to_gt / match_predictions_to_gt_cached
// (reference multigriddet/evaluation/metrics.py:73-144, 147-218) and the IoU matrix they
// consume (calculate_iou_matrix :28-70, BoxUtils.box_iou utils/boxes.py:16-58).
//
// The reference sorts all predictions of a class by score and walks them once, each
// claiming the best still-unmatched ground truth of its class in its image.  Ground
// truth is only shared inside one (image, class) group, so the walk decomposes by image:
// one warp per image visits that image's detections in descending score (ties: later
// slot first, the order of a reversed stable argsort) and the 32 lanes scan the image's
// ground-truth boxes.  Every IoU threshold is an independent walk over the same boxes.
// float64 IoU in the reference's operation order (-fmad=false), so `iou >= threshold`
// decides identically.  An optional area band (MatchArgs::band) restricts the walk to the
// boxes calculate_map's per-scale filter keeps, which is the filtered lists' result: their
// relative visiting order and ground-truth index order are those of the full lists.
// confusion_kernel extends one such walk with a cross-class stage (mgd_confusion_update), and
// tide_kernel types its errors and writes the error-fixed record sets (mgd_tide_update).
#include <math.h>
#include "common.cuh"

namespace {

constexpr int kMatchWarps = 4;

// calculate_iou_matrix (metrics.py:54-68): xyxy corners
__device__ __forceinline__ double iou_corner(const double* p, const double* g)
{
    const double x1 = fmax(p[0], g[0]), y1 = fmax(p[1], g[1]);
    const double x2 = fmin(p[2], g[2]), y2 = fmin(p[3], g[3]);
    const double inter = __dmul_rn(fmax(0.0, __dsub_rn(x2, x1)), fmax(0.0, __dsub_rn(y2, y1)));
    const double a1 = __dmul_rn(__dsub_rn(p[2], p[0]), __dsub_rn(p[3], p[1]));
    const double a2 = __dmul_rn(__dsub_rn(g[2], g[0]), __dsub_rn(g[3], g[1]));
    const double uni = __dsub_rn(__dadd_rn(a1, a2), inter);
    return uni > 0.0 ? __ddiv_rn(inter, uni) : 0.0;
}

// BoxUtils.box_iou (utils/boxes.py:28-58) as the un-cached matcher calls it: the four
// numbers are read as [x, y, w, h] centre format
__device__ __forceinline__ double iou_centre(const double* p, const double* g)
{
    const double hw1 = __ddiv_rn(p[2], 2.0), hh1 = __ddiv_rn(p[3], 2.0);
    const double hw2 = __ddiv_rn(g[2], 2.0), hh2 = __ddiv_rn(g[3], 2.0);
    const double ix0 = fmax(__dsub_rn(p[0], hw1), __dsub_rn(g[0], hw2));
    const double iy0 = fmax(__dsub_rn(p[1], hh1), __dsub_rn(g[1], hh2));
    const double ix1 = fmin(__dadd_rn(p[0], hw1), __dadd_rn(g[0], hw2));
    const double iy1 = fmin(__dadd_rn(p[1], hh1), __dadd_rn(g[1], hh2));
    if (ix1 <= ix0 || iy1 <= iy0) return 0.0;
    const double inter = __dmul_rn(__dsub_rn(ix1, ix0), __dsub_rn(iy1, iy0));
    const double uni = __dsub_rn(__dadd_rn(__dmul_rn(p[2], p[3]), __dmul_rn(g[2], g[3])), inter);
    return uni > 0.0 ? __ddiv_rn(inter, uni) : 0.0;
}

// kBand: a.band != 0 (a separate instantiation, so the plain matcher keeps its registers)
template <bool kBand>
__global__ void __launch_bounds__(kMatchWarps * 32)
match_kernel(const __grid_constant__ MatchArgs a)
{
    extern __shared__ __align__(16) unsigned char dyn[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t per_warp = (size_t)a.M * 2 + (size_t)((a.N + 31) / 32) * 4 + 16;
    unsigned short* order = reinterpret_cast<unsigned short*>(dyn + warp * ((per_warp + 15) & ~(size_t)15));
    unsigned* taken = reinterpret_cast<unsigned*>(order + ((a.M + 1) & ~1));
    const int words = (a.N + 31) / 32;

    for (;;) {
        int b = 0;
        if (lane == 0) b = atomicAdd(a.next_image, 1);
        b = __shfl_sync(0xffffffffu, b, 0);
        if (b >= a.B) break;
        const int n = min(max(a.det_counts[b], 0), a.M);
        const int g = min(max(a.gt_counts[b], 0), a.N);
        const double* dbox = a.det_boxes + (size_t)b * a.M * 4;
        const double* dsc = a.det_scores + (size_t)b * a.M;
        const int* dcl = a.det_classes + (size_t)b * a.M;
        const double* gbox = a.gt_boxes + (size_t)b * a.N * 4;
        const int* gcl = a.gt_classes + (size_t)b * a.N;

        // visiting order: score descending, equal scores: later slot first (metrics.py:93
        // with a stable argsort).  Rank by counting; n is a per-image detection count.
        for (int i = lane; i < n; i += 32) {
            const double si = dsc[i];
            int rank = 0;
            for (int j = 0; j < n; ++j) {
                const double sj = dsc[j];
                rank += (sj > si) || (sj == si && j > i);
            }
            order[rank] = (unsigned short)i;
        }
        __syncwarp();

        for (int t = 0; t < a.T; ++t) {
            const double thr = a.thr[t];
            // ground truth outside the area band starts the walk as already claimed
            for (int w = lane; w < words; w += 32) {
                unsigned m = 0u;
                if (kBand)
                    for (int j = 32 * w; j < g && j < 32 * w + 32; ++j)
                        if (map_area_band(gbox + 4 * j) != a.band - 1) m |= 1u << (j & 31);
                taken[w] = m;
            }
            __syncwarp();
            unsigned char* tp = a.tp + ((size_t)t * a.B + b) * a.M;
            int* who = a.matched ? a.matched + ((size_t)t * a.B + b) * a.M : nullptr;
            for (int k = 0; k < n; ++k) {
                const int d = order[k];
                // a detection outside the band is not in the filtered list: no claim, tp = 0;
                // the visiting order of the others is unchanged
                if (kBand && map_area_band(dbox + 4 * d) != a.band - 1) {
                    if (lane == 0) {
                        tp[d] = 0;
                        if (who) who[d] = -1;
                    }
                    continue;
                }
                const int cls = dcl[d];
                const double p[4] = {dbox[4 * d], dbox[4 * d + 1], dbox[4 * d + 2], dbox[4 * d + 3]};
                double best = 0.0;
                int best_j = -1;
                for (int j = lane; j < g; j += 32) {
                    if (gcl[j] != cls || ((taken[j >> 5] >> (j & 31)) & 1u)) continue;
                    const double q[4] = {gbox[4 * j], gbox[4 * j + 1], gbox[4 * j + 2], gbox[4 * j + 3]};
                    const double v = a.mode ? iou_centre(p, q) : iou_corner(p, q);
                    // cached matcher: a candidate must beat 0.0 (:196-199); un-cached:
                    // np.argmax over every candidate, first maximum (:133-135)
                    if (a.mode ? (best_j < 0 || v > best) : (v > best)) { best = v; best_j = j; }
                }
                #pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ov = __shfl_xor_sync(0xffffffffu, best, o);
                    const int oj = __shfl_xor_sync(0xffffffffu, best_j, o);
                    const bool take = oj >= 0 && (best_j < 0 || ov > best || (ov == best && oj < best_j));
                    if (take) { best = ov; best_j = oj; }
                }
                const bool hit = best_j >= 0 && best >= thr;
                if (lane == 0) {
                    tp[d] = hit ? 1 : 0;
                    if (who) who[d] = hit ? best_j : -1;
                    if (hit) taken[best_j >> 5] |= 1u << (best_j & 31);
                }
                __syncwarp();
            }
            for (int i = n + lane; i < a.M; i += 32) {
                tp[i] = 0;
                if (who) who[i] = -1;
            }
        }
        __syncwarp();
    }
}

// Detection confusion matrix at each confidence conf[q] (mgd_confusion_update), one warp per
// image.  The kept detections (score >= conf[q]) are a prefix of match_kernel's visiting order:
// equal scores are never split by the filter, and the greedy walk never looks ahead, so stage 1
// on the kept set is the full walk's claims (a.matched) restricted to that prefix.
//   stage 1: each claim of a kept detection counts [c, c];
//   stage 2: the kept detections stage 1 left unmatched, in the same order, each claim the
//            unclaimed ground truth of ANY class with the highest IoU (equal IoU: lowest index)
//            when it is >= thr, counted [gt class, det class].  Such a pair is never of one
//            class: at the detection's stage-1 turn every unclaimed ground truth of its class had
//            IoU < thr, and the unclaimed set has only shrunk since;
//   the kept detections still unmatched count [C, det class] (background row), the ground truth
//   still unclaimed [gt class, C] (background column).
// The shared memory per warp is match_kernel's: the visiting order and the claimed bitmap.
__global__ void __launch_bounds__(kMatchWarps * 32)
confusion_kernel(const __grid_constant__ ConfusionArgs a)
{
    extern __shared__ __align__(16) unsigned char dyn[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t per_warp = (size_t)a.M * 2 + (size_t)((a.N + 31) / 32) * 4 + 16;
    unsigned short* order = reinterpret_cast<unsigned short*>(dyn + warp * ((per_warp + 15) & ~(size_t)15));
    unsigned* taken = reinterpret_cast<unsigned*>(order + ((a.M + 1) & ~1));
    const int words = (a.N + 31) / 32;
    const long long C1 = (long long)a.C + 1;

    for (;;) {
        int b = 0;
        if (lane == 0) b = atomicAdd(a.next_image, 1);
        b = __shfl_sync(0xffffffffu, b, 0);
        if (b >= a.B) break;
        const int n = min(max(a.det_counts[b], 0), a.M);
        const int g = min(max(a.gt_counts[b], 0), a.N);
        const double* dbox = a.det_boxes + (size_t)b * a.M * 4;
        const double* dsc = a.det_scores + (size_t)b * a.M;
        const int* dcl = a.det_classes + (size_t)b * a.M;
        const double* gbox = a.gt_boxes + (size_t)b * a.N * 4;
        const int* gcl = a.gt_classes + (size_t)b * a.N;
        const int* who = a.matched + (size_t)b * a.M;

        // class ids of the real slots; a cell with an id out of range is never counted
        bool bad = false;
        for (int i = lane; i < n; i += 32) bad |= (unsigned)dcl[i] >= (unsigned)a.C;
        for (int j = lane; j < g; j += 32) bad |= (unsigned)gcl[j] >= (unsigned)a.C;
        if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(a.status, 16);

        // match_kernel's visiting order: score descending, equal scores later slot first
        for (int i = lane; i < n; i += 32) {
            const double si = dsc[i];
            int rank = 0;
            for (int j = 0; j < n; ++j) {
                const double sj = dsc[j];
                rank += (sj > si) || (sj == si && j > i);
            }
            order[rank] = (unsigned short)i;
        }
        __syncwarp();

        for (int q = 0; q < a.Q; ++q) {
            unsigned long long* mat = a.matrix + (size_t)q * C1 * C1;
            const double conf = a.conf[q];
            int K = 0;                                  // kept detections: order[0, K)
            for (int i = lane; i < n; i += 32) K += dsc[i] >= conf;
            #pragma unroll
            for (int o = 16; o > 0; o >>= 1) K += __shfl_xor_sync(0xffffffffu, K, o);

            // stage 1
            for (int w = lane; w < words; w += 32) taken[w] = 0u;
            __syncwarp();
            for (int k = lane; k < K; k += 32) {
                const int d = order[k];
                const int j = who[d];
                if (j < 0) continue;
                atomicOr(&taken[j >> 5], 1u << (j & 31));
                const int c = dcl[d];
                if ((unsigned)c < (unsigned)a.C) atomicAdd(mat + c * C1 + c, 1ull);
            }
            __syncwarp();

            // stage 2 and the background row
            for (int k = 0; k < K; ++k) {
                const int d = order[k];
                if (who[d] >= 0) continue;
                const double p[4] = {dbox[4 * d], dbox[4 * d + 1], dbox[4 * d + 2], dbox[4 * d + 3]};
                double best = 0.0;                      // thr > 0: an IoU of 0 never claims
                int best_j = -1;
                for (int j = lane; j < g; j += 32) {
                    if ((taken[j >> 5] >> (j & 31)) & 1u) continue;
                    const double qb[4] = {gbox[4 * j], gbox[4 * j + 1], gbox[4 * j + 2], gbox[4 * j + 3]};
                    const double v = a.mode ? iou_centre(p, qb) : iou_corner(p, qb);
                    if (v > best) { best = v; best_j = j; }
                }
                // most unmatched detections have no candidate at all: skip the reduction
                const bool hit = __any_sync(0xffffffffu, best_j >= 0 && best >= a.thr);
                if (hit) {
                    #pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        const double ov = __shfl_xor_sync(0xffffffffu, best, o);
                        const int oj = __shfl_xor_sync(0xffffffffu, best_j, o);
                        const bool take = oj >= 0 && (best_j < 0 || ov > best || (ov == best && oj < best_j));
                        if (take) { best = ov; best_j = oj; }
                    }
                }
                if (lane == 0) {
                    const int c = dcl[d];
                    int row = a.C;
                    if (hit) {                              // the maximum is >= thr
                        taken[best_j >> 5] |= 1u << (best_j & 31);
                        row = gcl[best_j];
                    }
                    if ((unsigned)c < (unsigned)a.C && (unsigned)row <= (unsigned)a.C)
                        atomicAdd(mat + row * C1 + c, 1ull);
                }
                __syncwarp();
            }

            // background column
            for (int j = lane; j < g; j += 32) {
                const int c = gcl[j];
                if (!((taken[j >> 5] >> (j & 31)) & 1u) && (unsigned)c < (unsigned)a.C)
                    atomicAdd(mat + c * C1 + a.C, 1ull);
            }
            __syncwarp();
        }
    }
}

// Detection error analysis (mgd_tide_update), one warp per image, after the base walk at t_f
// (a.matched).  The visiting order and the base's claimed bitmap are confusion_kernel's; two more
// bitmaps hold the claims of the Cls fix and of the Loc fix, each starting from the base's.  The
// detections are taken in visiting order: a TP keeps its record in every set; a false positive is
// typed from its best same-class IoU s and best other-class IoU o over every ground truth of the
// image (claimed or not, so the type does not depend on the order), and only the Cls / Loc claims
// do.  A ground truth named by a Cls or Loc error lies in that fix's bitmap afterwards (claimed by
// that error or by an earlier one of the same type), so Miss = in none of the three bitmaps.
// Record of set f: class f * C + c, TP flag in bits[MGD_MAP_VIEW_CORNER] bit 0; dropped: class -1.
__global__ void __launch_bounds__(kMatchWarps * 32)
tide_kernel(const __grid_constant__ TideArgs a)
{
    extern __shared__ __align__(16) unsigned char dyn[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int words = (a.N + 31) / 32;
    const size_t per_warp = (size_t)a.M * 2 + (size_t)words * 12 + 16;
    unsigned short* order = reinterpret_cast<unsigned short*>(dyn + warp * ((per_warp + 15) & ~(size_t)15));
    unsigned* taken = reinterpret_cast<unsigned*>(order + ((a.M + 1) & ~1));   // base claims
    unsigned* fix_cls = taken + words;                                         // Cls fix claims
    unsigned* fix_loc = fix_cls + words;                                       // Loc fix claims

    for (;;) {
        int b = 0;
        if (lane == 0) b = atomicAdd(a.next_image, 1);
        b = __shfl_sync(0xffffffffu, b, 0);
        if (b >= a.B) break;
        const int n = min(max(a.det_counts[b], 0), a.M);
        const int g = min(max(a.gt_counts[b], 0), a.N);
        const double* dbox = a.det_boxes + (size_t)b * a.M * 4;
        const double* dsc = a.det_scores + (size_t)b * a.M;
        const int* dcl = a.det_classes + (size_t)b * a.M;
        const double* gbox = a.gt_boxes + (size_t)b * a.N * 4;
        const int* gcl = a.gt_classes + (size_t)b * a.N;
        const int* who = a.matched + (size_t)b * a.M;
        MapRec* recs = a.recs + (size_t)b * MGD_TIDE_SETS * a.M;

        bool bad = false;
        for (int i = lane; i < n; i += 32) bad |= (unsigned)dcl[i] >= (unsigned)a.C;
        for (int j = lane; j < g; j += 32) bad |= (unsigned)gcl[j] >= (unsigned)a.C;
        if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(a.status, 32);

        // match_kernel's visiting order: score descending, equal scores later slot first
        for (int i = lane; i < n; i += 32) {
            const double si = dsc[i];
            int rank = 0;
            for (int j = 0; j < n; ++j) {
                const double sj = dsc[j];
                rank += (sj > si) || (sj == si && j > i);
            }
            order[rank] = (unsigned short)i;
        }
        for (int w = lane; w < 3 * words; w += 32) taken[w] = 0u;
        __syncwarp();
        for (int i = lane; i < n; i += 32) {
            const int j = who[i];
            if (j >= 0) atomicOr(&taken[j >> 5], 1u << (j & 31));
        }
        __syncwarp();
        for (int w = lane; w < words; w += 32) fix_cls[w] = fix_loc[w] = taken[w];
        // padding slots: class -1 in every set
        for (int k = lane; k < (a.M - n) * MGD_TIDE_SETS; k += 32) {
            const int f = k / (a.M - n), i = n + k % (a.M - n);
            MapRec r;
            r.score = dsc[i]; r.cls = -1; r.band = 3; r.pad = 0u;
            for (int v = 0; v < MGD_MAP_VIEWS; ++v) r.bits[v] = 0u;
            recs[(size_t)f * a.M + i] = r;
        }
        __syncwarp();

        for (int k = 0; k < n; ++k) {
            const int d = order[k];
            const int c = dcl[d];
            const bool ok = (unsigned)c < (unsigned)a.C;
            // kind: -1 TP, else the mgd_tide_error type; to: the target's class (Cls fix) or c
            int kind = -1, fixed = -1;
            if (who[d] < 0) {
                const double p[4] = {dbox[4 * d], dbox[4 * d + 1], dbox[4 * d + 2], dbox[4 * d + 3]};
                double s = 0.0, o = 0.0;
                int sj = -1, oj = -1;
                for (int j = lane; j < g; j += 32) {
                    const double q[4] = {gbox[4 * j], gbox[4 * j + 1], gbox[4 * j + 2], gbox[4 * j + 3]};
                    const double v = a.mode ? iou_centre(p, q) : iou_corner(p, q);
                    if (gcl[j] == c) { if (v > s) { s = v; sj = j; } }
                    else if (v > o) { o = v; oj = j; }
                }
                #pragma unroll
                for (int w = 16; w > 0; w >>= 1) {
                    const double os = __shfl_xor_sync(0xffffffffu, s, w);
                    const int osj = __shfl_xor_sync(0xffffffffu, sj, w);
                    const double oo = __shfl_xor_sync(0xffffffffu, o, w);
                    const int ooj = __shfl_xor_sync(0xffffffffu, oj, w);
                    if (osj >= 0 && (sj < 0 || os > s || (os == s && osj < sj))) { s = os; sj = osj; }
                    if (ooj >= 0 && (oj < 0 || oo > o || (oo == o && ooj < oj))) { o = oo; oj = ooj; }
                }
                // every lane holds the same s, o and targets
                int target = -1;
                unsigned* fix = nullptr;
                if (fmax(s, o) < a.t_b) kind = MGD_TIDE_BKG;
                else if (o >= a.t_f) { kind = MGD_TIDE_CLS; target = oj; fix = fix_cls; }
                else if (s >= a.t_f) kind = MGD_TIDE_DUPE;
                else if (s >= a.t_b) { kind = MGD_TIDE_LOC; target = sj; fix = fix_loc; }
                else kind = MGD_TIDE_BOTH;
                if (fix) {
                    const int tc = kind == MGD_TIDE_CLS ? gcl[target] : c;
                    if (!((fix[target >> 5] >> (target & 31)) & 1u) && (unsigned)tc < (unsigned)a.C) fixed = tc;
                    __syncwarp();
                    if (lane == 0 && fixed >= 0) fix[target >> 5] |= 1u << (target & 31);
                    __syncwarp();
                }
                if (lane == 0 && ok) atomicAdd(a.counts + (size_t)c * MGD_TIDE_ERRORS + kind, 1ull);
            }
            // lane f writes set f's record
            if (lane < MGD_TIDE_SETS) {
                const int f = lane;
                int cls = c, tp = kind < 0;
                if (kind >= 0) {
                    if (f == MGD_TIDE_FIX_FP) cls = -1;
                    else if (f == MGD_TIDE_FIX_CLS && kind == MGD_TIDE_CLS) { cls = fixed; tp = 1; }
                    else if (f == MGD_TIDE_FIX_LOC && kind == MGD_TIDE_LOC) { cls = fixed; tp = 1; }
                    else if ((f == MGD_TIDE_FIX_BOTH && kind == MGD_TIDE_BOTH) ||
                             (f == MGD_TIDE_FIX_DUPE && kind == MGD_TIDE_DUPE) ||
                             (f == MGD_TIDE_FIX_BKG && kind == MGD_TIDE_BKG)) cls = -1;
                }
                MapRec r;
                r.score = dsc[d];
                r.cls = ok && cls >= 0 ? f * a.C + cls : -1;
                r.band = r.cls >= 0 ? map_area_band(dbox + 4 * d) : 3;
                r.pad = 0u;
                for (int v = 0; v < MGD_MAP_VIEWS; ++v) r.bits[v] = 0u;
                r.bits[MGD_MAP_VIEW_CORNER] = r.cls >= 0 ? (unsigned)tp : 0u;
                recs[(size_t)f * a.M + d] = r;
            }
        }
        __syncwarp();

        // ground-truth counts of every set, and the misses
        for (int j = lane; j < g; j += 32) {
            const int c = gcl[j];
            if ((unsigned)c >= (unsigned)a.C) continue;
            const unsigned bit = 1u << (j & 31);
            const bool claimed = taken[j >> 5] & bit;
            const bool miss = !claimed && !(fix_cls[j >> 5] & bit) && !(fix_loc[j >> 5] & bit);
            for (int f = 0; f < MGD_TIDE_SETS; ++f) {
                if ((f == MGD_TIDE_FIX_MISS && miss) || (f == MGD_TIDE_FIX_FN && !claimed)) continue;
                atomicAdd(a.gt_hist + f * (long long)a.C + c, 1ull);
            }
            if (miss) atomicAdd(a.counts + (size_t)c * MGD_TIDE_ERRORS + MGD_TIDE_MISS, 1ull);
        }
        __syncwarp();
    }
}

__global__ void iou_matrix_kernel(const double* b1, int n, const double* b2, int m, double* out)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)n * m) return;
    const int i = (int)(idx / m), j = (int)(idx - (long long)i * m);
    out[idx] = iou_corner(b1 + 4 * (size_t)i, b2 + 4 * (size_t)j);
}

}  // namespace

cudaError_t launch_match(const MatchArgs& a, int num_sms, cudaStream_t stream)
{
    const size_t per_warp = ((size_t)a.M * 2 + (size_t)((a.N + 31) / 32) * 4 + 16 + 15) & ~(size_t)15;
    const size_t smem = per_warp * kMatchWarps;
    auto kernel = a.band ? match_kernel<true> : match_kernel<false>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    long long grid = ((long long)a.B + kMatchWarps - 1) / kMatchWarps;
    if (grid > (long long)num_sms * 8) grid = (long long)num_sms * 8;
    if (grid < 1) grid = 1;
    prof_mark_begin(PROF_OTHER, stream);
    kernel<<<(unsigned)grid, kMatchWarps * 32, smem, stream>>>(a);
    prof_mark_end(PROF_OTHER, stream);
    return cudaGetLastError();
}

cudaError_t launch_confusion(const ConfusionArgs& a, int num_sms, cudaStream_t stream)
{
    const size_t per_warp = ((size_t)a.M * 2 + (size_t)((a.N + 31) / 32) * 4 + 16 + 15) & ~(size_t)15;
    const size_t smem = per_warp * kMatchWarps;
    cudaError_t e = cudaFuncSetAttribute(confusion_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    long long grid = ((long long)a.B + kMatchWarps - 1) / kMatchWarps;
    if (grid > (long long)num_sms * 8) grid = (long long)num_sms * 8;
    if (grid < 1) grid = 1;
    prof_mark_begin(PROF_OTHER, stream);
    confusion_kernel<<<(unsigned)grid, kMatchWarps * 32, smem, stream>>>(a);
    prof_mark_end(PROF_OTHER, stream);
    return cudaGetLastError();
}

cudaError_t launch_tide(const TideArgs& a, int num_sms, cudaStream_t stream)
{
    const size_t per_warp = ((size_t)a.M * 2 + (size_t)((a.N + 31) / 32) * 12 + 16 + 15) & ~(size_t)15;
    const size_t smem = per_warp * kMatchWarps;
    cudaError_t e = cudaFuncSetAttribute(tide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    long long grid = ((long long)a.B + kMatchWarps - 1) / kMatchWarps;
    if (grid > (long long)num_sms * 8) grid = (long long)num_sms * 8;
    if (grid < 1) grid = 1;
    prof_mark_begin(PROF_OTHER, stream);
    tide_kernel<<<(unsigned)grid, kMatchWarps * 32, smem, stream>>>(a);
    prof_mark_end(PROF_OTHER, stream);
    return cudaGetLastError();
}

cudaError_t launch_iou_matrix(const double* b1, int n, const double* b2, int m, double* out,
                              cudaStream_t stream)
{
    const long long total = (long long)n * m;
    if (total == 0) return cudaSuccess;
    iou_matrix_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(b1, n, b2, m, out);
    return cudaGetLastError();
}
