// Average recall at detection limits (mgd_map_recall_update), sm_100a.
//
// pycocotools' AR@maxDets keeps, per (image, class), the first maxDets detections and counts
// the true positives among them.  The reference's greedy matcher (match.cu) visits an image's
// detections of one class by descending score, equal scores later slot first, and never looks
// ahead, so matching only the first k of them makes the claims the full walk made on those k.
// The TP bits mgd_map_update already wrote into the records are therefore the truncated
// evaluation's flags, and the count only needs each record's rank in that visiting order.
//
//   map_recall_kernel  one warp per image of the update, images handed out by an atomic
//                      counter.  Each lane ranks its records by comparison with the image's
//                      other records (same class; in a band view also the same band) and adds
//                      each TP bit once, in the first limit bucket above the rank; the caller
//                      takes the prefix sum over the limits.
#include "common.cuh"

namespace {

constexpr int kRecallWarps = 8;

__global__ void __launch_bounds__(kRecallWarps * 32) map_recall_kernel(const __grid_constant__ MapRecallArgs a)
{
    const int lane = threadIdx.x & 31;
    const unsigned tmask = a.T >= 32 ? 0xffffffffu : (1u << a.T) - 1u;
    for (;;) {
        int b = 0;
        if (lane == 0) b = atomicAdd(a.next_image, 1);
        b = __shfl_sync(0xffffffffu, b, 0);
        if (b >= a.B) break;
        const MapRec* r = a.recs + (size_t)b * a.M;
        for (int i = lane; i < a.M; i += 32) {
            const int c = r[i].cls;
            // padding (-1); ids of records written under another configuration are not counted
            if ((unsigned)c >= (unsigned)a.C) continue;
            const double s = r[i].score;
            const int band = r[i].band;
            int rank = 0, band_rank = 0;
            for (int j = 0; j < a.M; ++j) {
                const double sj = r[j].score;
                const bool ahead = r[j].cls == c && (sj > s || (sj == s && j > i));
                rank += ahead;
                band_rank += ahead && r[j].band == band;
            }
            for (int v = 0; v < MGD_MAP_VIEWS; ++v) {
                if (!((a.views >> v) & 1)) continue;
                if (v >= MGD_MAP_VIEW_S && band != v - MGD_MAP_VIEW_S) continue;
                unsigned bits = r[i].bits[v] & tmask;
                if (!bits) continue;
                const int rk = v >= MGD_MAP_VIEW_S ? band_rank : rank;
                int k = 0;
                while (k < a.K && rk >= a.limits[k]) ++k;
                if (k == a.K) continue;
                unsigned long long* row = a.tp + ((size_t)v * a.C + c) * a.T * a.K + k;
                for (; bits; bits &= bits - 1u)
                    atomicAdd(row + (size_t)(__ffs(bits) - 1) * a.K, 1ull);
            }
        }
    }
}

}  // namespace

cudaError_t launch_map_recall(const MapRecallArgs& a, int num_sms, cudaStream_t stream)
{
    long long grid = ((long long)a.B + kRecallWarps - 1) / kRecallWarps;
    if (grid > (long long)num_sms * 8) grid = (long long)num_sms * 8;
    if (grid < 1) grid = 1;
    prof_mark_begin(PROF_OTHER, stream);
    map_recall_kernel<<<(unsigned)grid, kRecallWarps * 32, 0, stream>>>(a);
    prof_mark_end(PROF_OTHER, stream);
    return cudaGetLastError();
}
