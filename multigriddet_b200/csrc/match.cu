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

cudaError_t launch_iou_matrix(const double* b1, int n, const double* b2, int m, double* out,
                              cudaStream_t stream)
{
    const long long total = (long long)n * m;
    if (total == 0) return cudaSuccess;
    iou_matrix_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(b1, n, b2, m, out);
    return cudaGetLastError();
}
