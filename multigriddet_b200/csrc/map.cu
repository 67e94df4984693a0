// Streaming mAP on the device (mgd_map_update / mgd_map_compute), sm_100a.
//
// Replaces what calculate_map (reference multigriddet/evaluation/metrics.py:541-815) does after
// the matcher: per class, sort the detections by score (np.argsort(scores, kind="stable")[::-1]
// in the drop-in, i.e. equal scores later detection first), cumulative TP / FP, precision and
// recall (compute_precision_recall :221-246) and the AP (compute_average_precision :249-300).
//
//   map_write_kernel      one 40-byte MapRec per padded detection slot: score, class, area band
//                         and the TP bits of every matched view (match_kernel's flags, bit t =
//                         threshold t); ground-truth counts per (view, class)
//   map_hist_kernel ..    stable LSD radix sort of record indices, 8-bit digits of the key
//   map_scatter_kernel    (class ascending, score descending); the first pass reads the input
//                         backwards so equal keys end up later index first; passes whose digit
//                         is the same for every key are skipped (decided on the device from
//                         the histograms of all digits, built in one pass)
//   map_ap_kernel         one CTA per (view, class): compacts the view's records of the class
//                         and walks them backwards once per threshold: suffix count of TP ->
//                         cum_tp, p and r in float64 in the reference's operation order, suffix
//                         max of p (np.maximum.accumulate(p[::-1])[::-1]) and the trapezoid, or
//                         the 11 VOC maxima
// Sharded (mgd_map_partition / mgd_map_compute_merged): the tile kernels of the sort, with the
// owner rank of each record's class as the digit, group a rank's records by destination and
// stamp each with its global slot; the merged sort takes four more digits from that slot
// (descending, so equal scores stay later detection first in global image order), and
// map_ap_kernel walks only the classes the rank owns.
// map_pr_kernel (mgd_map_compute_pr / _merged_pr): one CTA per (class, threshold, full-set view)
// over the same sorted order writes the precision-recall curve and the F1 / confidence
// operating points; map_ap_kernel and its launch are unchanged.
//
// compute_average_precision sorts the recalls with np.argsort (metrics.py:285) before the
// trapezoid.  They are non-decreasing already, but the sort is NumPy's unstable introsort
// (without SIMD dispatch, the NumPy the reference's numbers were produced with), which permutes
// runs of equal recall.  Only the element it leaves at the END of a run enters the AP (it sets
// the interpolated precision at the run's last point; every other term has r[i+1] == r[i]), so
// the walk takes the records in sorted order and asks np_aquicksort, a restatement of NumPy's
// aquicksort_, which record of the run that is.
#include <math.h>
#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kTileItems = 8 * kThreads;     // sort tile: 8 sub-tiles of one item per thread
constexpr int kDigits = 12;                  // 8 score bytes, then 4 class bytes (LSD order)
constexpr int kSlotDigits = 4;               // merged sort: 4 global-slot bytes below the score
constexpr int kMaxDigits = kDigits + kSlotDigits;

struct MapPlan {
    int active[kMaxDigits];                  // pass runs (its digit is not the same for all keys)
    int first[kMaxDigits];                   // first pass: reads the input (backwards without slot digits)
    int src[kMaxDigits], dst[kMaxDigits];    // index buffers
    int final_buf;
};

// Order-preserving transform of the score for a DESCENDING sort: -0.0 is taken as +0.0 first
// (NumPy compares them equal, so they must tie)
__device__ __forceinline__ unsigned long long score_key(double s)
{
    s = (s == 0.0) ? 0.0 : s;
    unsigned long long b = (unsigned long long)__double_as_longlong(s);
    b = (b >> 63) ? ~b : (b | 0x8000000000000000ull);
    return ~b;
}

// padding slots sort behind every class
__device__ __forceinline__ unsigned class_key(int cls, int C) { return cls < 0 ? (unsigned)C : (unsigned)cls; }

// digit p of a record's key; S = kSlotDigits in the merged sort, whose least significant digits
// are the global slot stamped into MapRec::pad, descending (later detection first)
template <int S>
__device__ __forceinline__ unsigned rec_digit(const MapRec& r, int p, int C)
{
    if (p < S) return (~r.pad >> (8 * p)) & 255u;
    p -= S;
    if (p < 8) return (unsigned)(score_key(r.score) >> (8 * p)) & 255u;
    return (class_key(r.cls, C) >> (8 * (p - 8))) & 255u;
}

// inclusive scan over the 256 threads of a CTA; *total = the CTA's reduction
template <typename T, typename Op>
__device__ __forceinline__ T block_scan(T v, Op op, T identity, T* total)
{
    __shared__ T warp_part[kThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    #pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T y = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v = op(y, v);
    }
    if (lane == 31) warp_part[warp] = v;
    __syncthreads();
    if (warp == 0) {
        T w = lane < kThreads / 32 ? warp_part[lane] : identity;
        #pragma unroll
        for (int o = 1; o < kThreads / 32; o <<= 1) {
            const T y = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w = op(y, w);
        }
        if (lane < kThreads / 32) warp_part[lane] = w;
    }
    __syncthreads();
    if (warp > 0) v = op(warp_part[warp - 1], v);
    *total = warp_part[kThreads / 32 - 1];
    __syncthreads();
    return v;
}

struct AddU { __device__ unsigned operator()(unsigned a, unsigned b) const { return a + b; } };
struct AddD { __device__ double operator()(double a, double b) const { return a + b; } };
struct MaxD { __device__ double operator()(double a, double b) const { return fmax(a, b); } };

// ---- record writer -------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) map_write_kernel(const __grid_constant__ MapWriteArgs a)
{
    const long long nd = (long long)a.B * a.M, ng = (long long)a.B * a.N;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nd + ng;
         i += (long long)gridDim.x * blockDim.x) {
        if (i < nd) {
            const int b = (int)(i / a.M), m = (int)(i - (long long)b * a.M);
            MapRec r;
            r.score = a.det_scores[i];
            r.cls = -1;
            r.band = 3;
            r.pad = 0u;
            for (int v = 0; v < MGD_MAP_VIEWS; ++v) r.bits[v] = 0u;
            if (m < min(max(a.det_counts[b], 0), a.M)) {
                const int c = a.det_classes[i];
                if (c < 0 || c >= a.C) {
                    atomicOr(a.status, 4);
                } else {
                    r.cls = c;
                    r.band = map_area_band(a.det_boxes + 4 * i);
                    for (int v = 0; v < MGD_MAP_VIEWS; ++v) {
                        if (!a.tp[v]) continue;
                        unsigned bits = 0u;
                        for (int t = 0; t < a.T; ++t)
                            bits |= (unsigned)(a.tp[v][(long long)t * nd + i] != 0) << t;
                        r.bits[v] = bits;
                    }
                }
            }
            a.recs[i] = r;
        } else {
            const long long j = i - nd;
            const int b = (int)(j / a.N), k = (int)(j - (long long)b * a.N);
            if (k >= min(max(a.gt_counts[b], 0), a.N)) continue;
            const int c = a.gt_classes[j];
            if (c < 0 || c >= a.C) { atomicOr(a.status, 4); continue; }
            const int band = map_area_band(a.gt_boxes + 4 * j);
            for (int v = 0; v < MGD_MAP_VIEWS; ++v)
                if (((a.views >> v) & 1) && (v < MGD_MAP_VIEW_S || band == v - MGD_MAP_VIEW_S))
                    atomicAdd(a.gt_hist + (size_t)v * a.C + c, 1ull);
        }
    }
}

// ---- radix sort ------------------------------------------------------------------------------
// histograms of all 12 + S digits in one pass (warp-aggregated: most digits are one value)
template <int S>
__global__ void __launch_bounds__(kThreads) map_hist_kernel(const MapRec* recs, unsigned n, int C, unsigned* hist)
{
    constexpr int nd = kDigits + S;
    __shared__ unsigned h[nd * 256];
    for (int k = threadIdx.x; k < nd * 256; k += blockDim.x) h[k] = 0u;
    __syncthreads();
    const unsigned lane_lt = (1u << (threadIdx.x & 31)) - 1u;
    const unsigned stride = gridDim.x * blockDim.x;
    for (unsigned base = blockIdx.x * blockDim.x; base < n; base += stride) {
        const unsigned i = base + threadIdx.x;
        const bool valid = i < n;
        MapRec r;
        if (valid) { r.score = recs[i].score; r.cls = recs[i].cls; if (S) r.pad = recs[i].pad; }
        for (int p = 0; p < nd; ++p) {
            const unsigned d = valid ? rec_digit<S>(r, p, C) : 256u;
            const unsigned peers = __match_any_sync(0xffffffffu, d);
            if (valid && (peers & lane_lt) == 0u) atomicAdd(&h[p * 256 + d], (unsigned)__popc(peers));
        }
    }
    __syncthreads();
    for (int k = threadIdx.x; k < nd * 256; k += blockDim.x)
        if (h[k]) atomicAdd(hist + k, h[k]);
}

// which passes run, and their buffers
template <int S>
__global__ void map_plan_kernel(const unsigned* hist, unsigned n, MapPlan* plan)
{
    constexpr int nd = kDigits + S;
    __shared__ int active[nd];
    const int p = threadIdx.x;
    if (p < nd) {
        int a = 1;
        for (int d = 0; d < 256; ++d) if (hist[p * 256 + d] == n) a = 0;
        active[p] = a;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    int any = 0;
    for (int q = 0; q < nd; ++q) any |= active[q];
    if (!any) active[nd - 1] = 1;           // all keys equal: one pass still reverses the input
    int cur = -1;
    for (int q = 0; q < nd; ++q) {
        plan->active[q] = active[q];
        plan->first[q] = active[q] && cur < 0;
        plan->src[q] = cur < 0 ? 0 : cur;
        if (active[q]) cur = cur < 0 ? 0 : (cur ^ 1);
        plan->dst[q] = cur < 0 ? 0 : cur;
    }
    plan->final_buf = cur;
}

// the first pass reads the records backwards so that equal keys end up later index first; with
// the global slot in the key (S > 0) no two keys are equal and it reads them in order
template <int S>
__device__ __forceinline__ unsigned pass_input(const MapPlan& pl, int p, const unsigned* bufs, unsigned n, unsigned i)
{
    return pl.first[p] ? (S ? i : n - 1u - i) : bufs[(size_t)pl.src[p] * n + i];
}

// The tile machinery below (per-tile digit counts, tile offsets, stable scatter) is shared by
// the sort passes and by the rank partition of mgd_map_partition.  A Pass says whether it runs,
// which item sits at input position i, the item's digit (256: the item is dropped) and where the
// item goes once its output position is known.

// one pass of the sort: items are record indices, the output is the pass's index buffer
template <int S>
struct SortPass {
    const MapPlan* plan; int p; const MapRec* recs; unsigned n; int C; unsigned* bufs;
    __device__ bool active() const { return plan->active[p]; }
    __device__ unsigned item(unsigned i) const { return pass_input<S>(*plan, p, bufs, n, i); }
    __device__ unsigned digit(unsigned it) const { return rec_digit<S>(recs[it], p, C); }
    __device__ void put(unsigned pos, unsigned it) const { bufs[(size_t)plan->dst[p] * n + pos] = it; }
};

// the rank partition: items are record indices, the digit is the rank that owns the record's
// class (padding slots are dropped), the output is the record with its global slot stamped in
struct PartitionPass {
    const MapRec* recs; int C; const int* owner; int world;
    const long long* segs; int num_segs;          // (num_segs, 2): first local slot, its global slot
    MapRec* out; int* status;
    __device__ bool active() const { return true; }
    __device__ unsigned item(unsigned i) const { return i; }
    __device__ unsigned digit(unsigned it) const
    {
        const int c = recs[it].cls;
        if (c < 0 || c >= C) return 256u;
        const int o = owner[c];
        if (o < 0 || o >= world) { atomicOr(status, 8); return 256u; }
        return (unsigned)o;
    }
    __device__ void put(unsigned pos, unsigned it) const
    {
        int lo = 0, hi = num_segs - 1;                    // the last segment starting at or before it
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (segs[2 * mid] <= (long long)it) lo = mid; else hi = mid - 1;
        }
        MapRec r = recs[it];
        r.pad = (unsigned)(segs[2 * lo + 1] + ((long long)it - segs[2 * lo]));
        out[pos] = r;
    }
};

// digit counts per tile: tile_counts[tile][digit]
template <class Pass>
__global__ void __launch_bounds__(kThreads) map_tile_count_kernel(const Pass pass, unsigned n, unsigned* tile_counts)
{
    __shared__ unsigned cnt[256];
    if (!pass.active()) return;
    cnt[threadIdx.x] = 0u;
    __syncthreads();
    for (int s = 0; s < kTileItems / kThreads; ++s) {
        const unsigned i = blockIdx.x * (unsigned)kTileItems + s * kThreads + threadIdx.x;
        if (i < n) {
            const unsigned d = pass.digit(pass.item(i));
            if (d < 256u) atomicAdd(&cnt[d], 1u);
        }
    }
    __syncthreads();
    tile_counts[(size_t)blockIdx.x * 256 + threadIdx.x] = cnt[threadIdx.x];
}

// tile counts -> first output position of each (tile, digit), in place.  digit_totals: the
// pass's histogram, or nullptr to sum it from the tile counts and store its first num_totals
// entries to totals_out
template <class Pass>
__global__ void __launch_bounds__(kThreads) map_tile_offsets_kernel(const Pass pass, const unsigned* digit_totals,
                                                                     unsigned tiles, unsigned* tile_counts,
                                                                     long long* totals_out, int num_totals)
{
    if (!pass.active()) return;
    const unsigned d = threadIdx.x;
    unsigned h = 0u;
    if (digit_totals) {
        h = digit_totals[d];
    } else {
        for (unsigned t = 0; t < tiles; ++t) h += tile_counts[(size_t)t * 256 + d];
        if ((int)d < num_totals) totals_out[d] = h;
    }
    unsigned total;
    unsigned base = block_scan(h, AddU(), 0u, &total) - h;
    for (unsigned t = 0; t < tiles; ++t) {
        unsigned* c = tile_counts + (size_t)t * 256 + d;
        const unsigned v = *c;
        *c = base;
        base += v;
    }
}

// stable scatter of one tile: sub-tile by sub-tile, rank = earlier items of the same digit
template <class Pass>
__global__ void __launch_bounds__(kThreads) map_scatter_kernel(const Pass pass, unsigned n, const unsigned* tile_offsets)
{
    __shared__ unsigned run[256];
    __shared__ unsigned wcnt[kThreads / 32][256];
    if (!pass.active()) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lane_lt = (1u << lane) - 1u;
    run[threadIdx.x] = tile_offsets[(size_t)blockIdx.x * 256 + threadIdx.x];
    for (int s = 0; s < kTileItems / kThreads; ++s) {
        for (int w = 0; w < kThreads / 32; ++w) wcnt[w][threadIdx.x] = 0u;
        __syncthreads();
        const unsigned i = blockIdx.x * (unsigned)kTileItems + s * kThreads + threadIdx.x;
        const bool valid = i < n;
        const unsigned it = valid ? pass.item(i) : 0u;
        const unsigned d = valid ? pass.digit(it) : 256u;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const unsigned rank = __popc(peers & lane_lt);
        if (d < 256u && rank == 0u) wcnt[warp][d] = __popc(peers);
        __syncthreads();
        unsigned sum = 0u;                                   // column of digit threadIdx.x
        for (int w = 0; w < kThreads / 32; ++w) {
            const unsigned c = wcnt[w][threadIdx.x];
            wcnt[w][threadIdx.x] = sum;
            sum += c;
        }
        __syncthreads();
        if (d < 256u) pass.put(run[d] + wcnt[warp][d] + rank, it);
        __syncthreads();
        run[threadIdx.x] += sum;
    }
}

// ---- np.argsort of the recalls ------------------------------------------------------------------
// NumPy's aquicksort_ / aheapsort_ (numpy/_core/src/npysort/quicksort.cpp, heapsort.cpp) on
// (cum_tp << 32 | position) pairs compared by cum_tp, which orders like the recalls: the
// permutation np.argsort(recalls) returns.  One thread per (view, class, threshold).
__device__ __forceinline__ bool key_less(unsigned long long a, unsigned long long b) { return (a >> 32) < (b >> 32); }

__device__ void np_aheapsort(unsigned long long* t, int n)
{
    unsigned long long* a = t - 1;                          // 1-based like NumPy
    unsigned long long tmp;
    int i, j, l;
    for (l = n >> 1; l > 0; --l) {
        tmp = a[l];
        for (i = l, j = l << 1; j <= n;) {
            if (j < n && key_less(a[j], a[j + 1])) j += 1;
            if (key_less(tmp, a[j])) { a[i] = a[j]; i = j; j += j; }
            else break;
        }
        a[i] = tmp;
    }
    for (; n > 1;) {
        tmp = a[n];
        a[n] = a[1];
        n -= 1;
        for (i = 1, j = 2; j <= n;) {
            if (j < n && key_less(a[j], a[j + 1])) j += 1;
            if (key_less(tmp, a[j])) { a[i] = a[j]; i = j; j += j; }
            else break;
        }
        a[i] = tmp;
    }
}

__device__ void np_aquicksort(unsigned long long* t, int num)
{
    constexpr int kSmall = 15;                              // SMALL_QUICKSORT
    int stack[128], depth[64];                              // larger partition pushed: <= 31 levels
    int sp = 0, dp = 0;
    int pl = 0, pr = num - 1;
    int cdepth = 0;
    for (unsigned u = (unsigned)num; u >>= 1;) ++cdepth;    // npy_get_msb
    cdepth *= 2;
    if (num <= 1) return;
    for (;;) {
        if (cdepth < 0) {
            np_aheapsort(t + pl, pr - pl + 1);
        } else {
            while (pr - pl > kSmall) {
                int pm = pl + ((pr - pl) >> 1);
                unsigned long long x;
                if (key_less(t[pm], t[pl])) { x = t[pm]; t[pm] = t[pl]; t[pl] = x; }
                if (key_less(t[pr], t[pm])) { x = t[pr]; t[pr] = t[pm]; t[pm] = x; }
                if (key_less(t[pm], t[pl])) { x = t[pm]; t[pm] = t[pl]; t[pl] = x; }
                const unsigned long long vp = t[pm];
                int pi = pl, pj = pr - 1;
                x = t[pm]; t[pm] = t[pj]; t[pj] = x;
                for (;;) {
                    do { ++pi; } while (key_less(t[pi], vp));
                    do { --pj; } while (key_less(vp, t[pj]));
                    if (pi >= pj) break;
                    x = t[pi]; t[pi] = t[pj]; t[pj] = x;
                }
                const int pk = pr - 1;
                x = t[pi]; t[pi] = t[pk]; t[pk] = x;
                if (pi - pl < pr - pi) { stack[sp++] = pi + 1; stack[sp++] = pr; pr = pi - 1; }
                else { stack[sp++] = pl; stack[sp++] = pi - 1; pl = pi + 1; }
                depth[dp++] = --cdepth;
            }
            for (int pi = pl + 1; pi <= pr; ++pi) {         // insertion sort
                const unsigned long long vi = t[pi];
                int pj = pi, pk = pi - 1;
                while (pj > pl && key_less(vi, t[pk])) t[pj--] = t[pk--];
                t[pj] = vi;
            }
        }
        if (sp == 0) break;
        pr = stack[--sp];
        pl = stack[--sp];
        cdepth = depth[--dp];
    }
}

// ---- AP ---------------------------------------------------------------------------------------
struct ApArgs {
    int C, T, method, views;
    double voc_x[MGD_MAP_VOC_POINTS];
    const MapRec* recs;
    unsigned n;
    const MapPlan* plan;
    const unsigned* bufs;
    const unsigned long long* gt_hist;
    unsigned* lists;                  // (MGD_MAP_VIEWS, n) compacted TP bits
    unsigned long long* perm;         // (MGD_MAP_VIEWS, T, n) np.argsort of each class's recalls
    double* ap;                       // (V, C, T) or nullptr
    double* voc;                      // (V, C, T, 11) or nullptr
    unsigned long long* det_hist;     // (V, C)
    const int* owner;                 // (C,) merged compute: only classes with owner[c] == rank,
    int rank;                         // the others get exact zeros; nullptr: every class
};

__global__ void __launch_bounds__(kThreads) map_ap_kernel(const __grid_constant__ ApArgs a)
{
    __shared__ unsigned seg[2];
    __shared__ double r_s[kThreads], in_s[kThreads];
    __shared__ double carry[2];                             // interp and r of the later chunk's first record
    const int c = blockIdx.x, v = blockIdx.y, tid = threadIdx.x;
    const size_t vc = (size_t)v * a.C + c;
    if (((a.views >> v) & 1) == 0 || a.n == 0u || (a.owner && a.owner[c] != a.rank)) {
        if (tid == 0) a.det_hist[vc] = 0ull;
        for (int t = tid; t < a.T; t += kThreads) if (a.ap) a.ap[vc * a.T + t] = 0.0;
        for (int k = tid; k < a.T * MGD_MAP_VOC_POINTS; k += kThreads)
            if (a.voc) a.voc[vc * a.T * MGD_MAP_VOC_POINTS + k] = 0.0;
        return;
    }
    const unsigned* sorted = a.bufs + (size_t)a.plan->final_buf * a.n;
    if (tid < 2) {                                          // class segment: lower bounds of c, c + 1
        const unsigned want = (unsigned)c + tid;
        unsigned lo = 0u, hi = a.n;
        while (lo < hi) {
            const unsigned mid = lo + (hi - lo) / 2;
            if (class_key(a.recs[sorted[mid]].cls, a.C) < want) lo = mid + 1; else hi = mid;
        }
        seg[tid] = lo;
    }
    __syncthreads();
    const unsigned s0 = seg[0], s1 = seg[1];
    // the view's records of class c, in sorted order
    unsigned* list = a.lists + (size_t)v * a.n + s0;
    unsigned n = 0u;
    for (unsigned base = s0; base < s1; base += kThreads) {
        const unsigned i = base + tid;
        unsigned member = 0u, bits = 0u;
        if (i < s1) {
            const MapRec& r = a.recs[sorted[i]];
            member = v < MGD_MAP_VIEW_S || r.band == v - MGD_MAP_VIEW_S;
            bits = r.bits[v];
        }
        unsigned total;
        const unsigned pos = block_scan(member, AddU(), 0u, &total) - member;
        if (member) list[n + pos] = bits;
        n += total;
    }
    __syncthreads();
    const unsigned long long n_gt = a.gt_hist[vc];
    if (tid == 0) a.det_hist[vc] = n;
    const double r_den = (double)n_gt + 1e-8;
    // np.argsort of the recalls, per threshold by lane 0 of a warp (the sorts diverge)
    if (a.ap && n > 1u && n_gt > 0ull && (tid & 31) == 0) {
        for (int t = tid >> 5; t < a.T; t += kThreads / 32) {
            unsigned long long* perm = a.perm + ((size_t)v * a.T + t) * a.n + s0;
            unsigned long long cum_tp = 0ull;
            for (unsigned k = 0; k < n; ++k) {
                cum_tp += (list[k] >> t) & 1u;
                perm[k] = (cum_tp << 32) | k;
            }
            np_aquicksort(perm, (int)n);
        }
    }
    __syncthreads();
    for (int t = 0; t < a.T; ++t) {
        if (n == 0u || n_gt == 0ull) {                      // the caller's special cases
            if (tid == 0 && a.ap) a.ap[vc * a.T + t] = 0.0;
            if (tid < MGD_MAP_VOC_POINTS && a.voc) a.voc[(vc * a.T + t) * MGD_MAP_VOC_POINTS + tid] = 0.0;
            continue;
        }
        unsigned tp_total = 0u;
        for (unsigned i = tid; i < n; i += kThreads) tp_total += (list[i] >> t) & 1u;
        unsigned all_tp;
        block_scan(tp_total, AddU(), 0u, &all_tp);
        // backwards over the records: thread tid takes position e - 1 - tid of the chunk [e - 256, e)
        unsigned later_tp = 0u;                             // TP flags at positions >= e
        double acc = 0.0;
        double vmax[MGD_MAP_VOC_POINTS];
        #pragma unroll
        for (int k = 0; k < MGD_MAP_VOC_POINTS; ++k) vmax[k] = 0.0;
        if (tid == 0) { carry[0] = -1.0; carry[1] = 0.0; }
        __syncthreads();
        for (long long e = n; e > 0; e -= kThreads) {
            const long long i = e - 1 - tid;
            const bool valid = i >= 0;
            const unsigned f = valid ? (list[i] >> t) & 1u : 0u;
            unsigned chunk_tp;
            const unsigned incl = block_scan(f, AddU(), 0u, &chunk_tp);
            const unsigned cum_tp = all_tp - later_tp - incl + f;          // np.cumsum(tp)[i]
            // compute_precision_recall: cum_tp / (cum_tp + cum_fp + 1e-8), cum_tp / (num_gt + 1e-8)
            const double p = (double)cum_tp / ((double)(i + 1) + 1e-8);
            const double r = (double)cum_tp / r_den;
            double chunk_max;
            const double interp = fmax(carry[0], block_scan(valid ? p : -1.0, MaxD(), -1.0, &chunk_max));
            r_s[tid] = r;
            in_s[tid] = interp;
            __syncthreads();
            if (valid && a.ap && i + 1 < (long long)n) {
                // the trapezoid in np.argsort(recalls) order: a term is non-zero only where the
                // recall steps up, i.e. at the end of a run, whose interpolated precision takes the
                // precision of the record the sort left there; interp[i + 1] is a maximum over
                // the records after the run and does not depend on their order
                const double r1 = tid > 0 ? r_s[tid - 1] : carry[1];
                const double in1 = tid > 0 ? in_s[tid - 1] : carry[0];
                if (r1 != r) {
                    const unsigned j = (unsigned)a.perm[((size_t)v * a.T + t) * a.n + s0 + (size_t)i];
                    const double q = (double)cum_tp / ((double)(j + 1u) + 1e-8);
                    acc += (r1 - r) * (in1 + fmax(q, in1)) / 2.0;
                }
            }
            if (valid && a.voc) {
                #pragma unroll
                for (int k = 0; k < MGD_MAP_VOC_POINTS; ++k)
                    if (r >= a.voc_x[k]) vmax[k] = fmax(vmax[k], p);
            }
            if (n == 1u && tid == 0 && a.ap) a.ap[vc * a.T + t] = interp * r;
            __syncthreads();
            const int last = (int)(e < kThreads ? e : kThreads) - 1;
            if (tid == 0) { carry[0] = in_s[last]; carry[1] = r_s[last]; }
            later_tp += chunk_tp;
            __syncthreads();
        }
        if (a.ap && n > 1u) {
            double sum;
            block_scan(acc, AddD(), 0.0, &sum);
            if (tid == 0) a.ap[vc * a.T + t] = sum;
        }
        if (a.voc) {
            for (int k = 0; k < MGD_MAP_VOC_POINTS; ++k) {
                double m;
                block_scan(vmax[k], MaxD(), 0.0, &m);
                if (tid == 0) a.voc[(vc * a.T + t) * MGD_MAP_VOC_POINTS + k] = m;
            }
        }
    }
}

// ---- precision-recall curves and operating points -------------------------------------------
struct PrArgs {
    int C, T, Q;
    int view[2];                      // view of output slot blockIdx.z (corner / centre)
    double conf[MGD_MAP_MAX_CONFIDENCES];
    const MapRec* recs;
    unsigned n;
    const MapPlan* plan;
    const unsigned* bufs;
    const unsigned long long* gt_hist;
    const int* owner;                 // as in ApArgs: the others get exact zeros
    int rank;
    long long cap;                    // row length of precision / recall
    long long* offsets;               // (C + 1,)
    double* scores;                   // (cap,)
    double* precision;                // (V, T, cap)
    double* recall;                   // (V, T, cap)
    double* best_f1;                  // (V, C, T, 4)
    long long* best_index;            // (V, C, T)
    double* at_conf;                  // (V, C, T, Q, 3)
};

__device__ __forceinline__ double f1_of(double p, double r) { return p + r == 0.0 ? 0.0 : 2.0 * p * r / (p + r); }

// One CTA per (class, threshold, view): walks the class's segment of the sorted order forwards,
// writes p and r at every record (the segment starts at offsets[c], so a record's sorted
// position is its curve position), keeps the first maximum F1 among records that end a run of
// equal scores, then finds each confidence's cut by binary search over the descending scores.
__global__ void __launch_bounds__(kThreads) map_pr_kernel(const __grid_constant__ PrArgs a)
{
    __shared__ unsigned seg[2];
    const int c = blockIdx.x, t = blockIdx.y, vi = blockIdx.z, v = a.view[vi], tid = threadIdx.x;
    const size_t vct = ((size_t)vi * a.C + c) * a.T + t;
    const unsigned* sorted = a.n ? a.bufs + (size_t)a.plan->final_buf * a.n : nullptr;
    if (tid < 2) {                                          // class segment, as in map_ap_kernel
        const unsigned want = (unsigned)c + tid;
        unsigned lo = 0u, hi = a.n;
        while (lo < hi) {
            const unsigned mid = lo + (hi - lo) / 2;
            if (class_key(a.recs[sorted[mid]].cls, a.C) < want) lo = mid + 1; else hi = mid;
        }
        seg[tid] = lo;
    }
    __syncthreads();
    const unsigned s0 = seg[0], s1 = seg[1];                // empty for a class another rank owns
    if (t == 0 && vi == 0 && tid == 0) {
        a.offsets[c] = s0;
        if (c == a.C - 1) a.offsets[a.C] = s1;
    }
    const size_t row = ((size_t)vi * a.T + t) * (size_t)a.cap;
    const double r_den = (double)a.gt_hist[(size_t)v * a.C + c] + 1e-8;
    unsigned carry = 0u, best_k = 0xffffffffu;
    double best = 0.0;
    for (unsigned base = s0; base < s1; base += kThreads) {
        const unsigned i = base + tid;
        const bool valid = i < s1;
        unsigned f = 0u;
        double s = 0.0;
        if (valid) {
            const MapRec& r = a.recs[sorted[i]];
            f = (r.bits[v] >> t) & 1u;
            s = r.score;
        }
        unsigned total;
        const unsigned cum_tp = carry + block_scan(f, AddU(), 0u, &total);
        if (valid) {
            const unsigned k = i - s0;
            // compute_precision_recall: cum_tp / (cum_tp + cum_fp + 1e-8), cum_tp / (num_gt + 1e-8)
            const double p = (double)cum_tp / ((double)(k + 1u) + 1e-8);
            const double r = (double)cum_tp / r_den;
            a.precision[row + i] = p;
            a.recall[row + i] = r;
            if (t == 0 && vi == 0) a.scores[i] = s;
            if (i + 1u == s1 || a.recs[sorted[i + 1u]].score != s) {     // a threshold can stop here
                const double f1 = f1_of(p, r);
                if (f1 > best) { best = f1; best_k = k; }   // k ascends per thread: the first maximum
            }
        }
        carry += total;
    }
    double m;
    block_scan(best, MaxD(), 0.0, &m);
    double neg_k;                                           // the smallest k that reaches m, as -k
    block_scan(m > 0.0 && best == m ? -(double)best_k : -4294967295.0, MaxD(), -4294967295.0, &neg_k);
    const unsigned k_first = (unsigned)-neg_k;
    // block_scan ended in __syncthreads: every p and r of the segment is visible to the CTA
    if (tid == 0) {
        double* o = a.best_f1 + vct * 4;
        if (k_first == 0xffffffffu) {
            o[0] = o[1] = o[2] = o[3] = 0.0;
            a.best_index[vct] = (a.owner && a.owner[c] != a.rank) ? 0 : -1;
        } else {
            const unsigned i = s0 + k_first;
            o[0] = a.recs[sorted[i]].score;
            o[1] = a.precision[row + i];
            o[2] = a.recall[row + i];
            o[3] = m;
            a.best_index[vct] = k_first;
        }
    }
    for (int q = tid; q < a.Q; q += kThreads) {
        unsigned lo = s0, hi = s1;                          // first record with score < conf[q]
        while (lo < hi) {
            const unsigned mid = lo + (hi - lo) / 2;
            if (a.recs[sorted[mid]].score >= a.conf[q]) lo = mid + 1; else hi = mid;
        }
        double* o = a.at_conf + (vct * a.Q + q) * 3;
        if (lo == s0) {
            o[0] = o[1] = o[2] = 0.0;
        } else {
            const double p = a.precision[row + lo - 1], r = a.recall[row + lo - 1];
            o[0] = p;
            o[1] = r;
            o[2] = f1_of(p, r);
        }
    }
}

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

}  // namespace

cudaError_t launch_map_write(const MapWriteArgs& a, cudaStream_t stream)
{
    const long long total = (long long)a.B * a.M + (long long)a.B * a.N;
    if (total == 0) return cudaSuccess;
    long long grid = (total + kThreads - 1) / kThreads;
    if (grid > 4096) grid = 4096;
    prof_mark_begin(PROF_OTHER, stream);
    map_write_kernel<<<(unsigned)grid, kThreads, 0, stream>>>(a);
    prof_mark_end(PROF_OTHER, stream);
    return cudaGetLastError();
}

// scratch: [histograms | plan | tile counts | 2 index buffers | per-view lists | recall sorts]
size_t map_compute_scratch_bytes(long long n, int T)
{
    const size_t tiles = (size_t)((n + kTileItems - 1) / kTileItems);
    return align256(kMaxDigits * 256 * 4) + align256(sizeof(MapPlan)) + align256(tiles * 256 * 4) +
           align256((size_t)n * 4 * 2) + align256((size_t)n * 4 * MGD_MAP_VIEWS) +
           (size_t)n * 8 * T * MGD_MAP_VIEWS;
}

namespace {

// S = 0: mgd_map_compute (equal keys later record first); S = kSlotDigits: the merged compute
// over records stamped with their global slot, APs of the classes `owner` gives to `rank` only
template <int S>
cudaError_t map_compute_impl(const mgd_map_config& cfg, const MapRec* recs, long long n_,
                             const unsigned long long* gt_hist, const int* owner, int rank, double* ap,
                             double* voc, unsigned long long* det_hist, void* scratch, cudaStream_t stream,
                             const mgd_map_pr* pr)
{
    constexpr int nd = kDigits + S;
    const unsigned n = (unsigned)n_;
    const unsigned tiles = (unsigned)((n_ + kTileItems - 1) / kTileItems);
    char* s = static_cast<char*>(scratch);
    unsigned* hist = reinterpret_cast<unsigned*>(s);
    s += align256(kMaxDigits * 256 * 4);
    MapPlan* plan = reinterpret_cast<MapPlan*>(s);
    s += align256(sizeof(MapPlan));
    unsigned* tile_counts = reinterpret_cast<unsigned*>(s);
    s += align256((size_t)tiles * 256 * 4);
    unsigned* bufs = reinterpret_cast<unsigned*>(s);
    s += align256((size_t)n * 4 * 2);
    unsigned* lists = reinterpret_cast<unsigned*>(s);
    s += align256((size_t)n * 4 * MGD_MAP_VIEWS);
    unsigned long long* perm = reinterpret_cast<unsigned long long*>(s);
    cudaError_t e;
    prof_mark_begin(PROF_OTHER, stream);
    if (n > 0) {
        if ((e = cudaMemsetAsync(hist, 0, nd * 256 * 4, stream)) != cudaSuccess) return e;
        unsigned grid = (n + kThreads - 1) / kThreads;
        if (grid > 1184) grid = 1184;
        map_hist_kernel<S><<<grid, kThreads, 0, stream>>>(recs, n, cfg.num_classes, hist);
        map_plan_kernel<S><<<1, 32, 0, stream>>>(hist, n, plan);
        for (int p = 0; p < nd; ++p) {
            const SortPass<S> pass{plan, p, recs, n, cfg.num_classes, bufs};
            map_tile_count_kernel<<<tiles, kThreads, 0, stream>>>(pass, n, tile_counts);
            map_tile_offsets_kernel<<<1, kThreads, 0, stream>>>(pass, hist + p * 256, tiles, tile_counts, nullptr, 0);
            map_scatter_kernel<<<tiles, kThreads, 0, stream>>>(pass, n, tile_counts);
        }
    }
    ApArgs a;
    a.C = cfg.num_classes; a.T = cfg.num_thresholds; a.method = cfg.method; a.views = cfg.views;
    for (int k = 0; k < MGD_MAP_VOC_POINTS; ++k) a.voc_x[k] = cfg.voc_recalls[k];
    a.recs = recs; a.n = n; a.plan = plan; a.bufs = bufs; a.gt_hist = gt_hist; a.lists = lists; a.perm = perm;
    a.ap = cfg.method == MGD_MAP_COCO ? ap : nullptr;
    a.voc = cfg.method == MGD_MAP_VOC ? voc : nullptr;
    a.det_hist = det_hist;
    a.owner = owner; a.rank = rank;
    map_ap_kernel<<<dim3((unsigned)cfg.num_classes, MGD_MAP_VIEWS), kThreads, 0, stream>>>(a);
    if (pr) {
        PrArgs q;
        q.C = cfg.num_classes; q.T = cfg.num_thresholds; q.Q = pr->num_confidences;
        int nv = 0;
        for (int v = MGD_MAP_VIEW_CORNER; v <= MGD_MAP_VIEW_CENTRE; ++v)
            if ((pr->views >> v) & 1) q.view[nv++] = v;
        for (int k = 0; k < MGD_MAP_MAX_CONFIDENCES; ++k) q.conf[k] = k < q.Q ? pr->confidences[k] : 0.0;
        q.recs = recs; q.n = n; q.plan = plan; q.bufs = bufs; q.gt_hist = gt_hist;
        q.owner = owner; q.rank = rank;
        q.cap = pr->capacity; q.offsets = pr->offsets; q.scores = pr->scores;
        q.precision = pr->precision; q.recall = pr->recall;
        q.best_f1 = pr->best_f1; q.best_index = pr->best_index; q.at_conf = pr->at_confidence;
        map_pr_kernel<<<dim3((unsigned)cfg.num_classes, (unsigned)cfg.num_thresholds, (unsigned)nv), kThreads, 0,
                        stream>>>(q);
    }
    prof_mark_end(PROF_OTHER, stream);
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_map_compute(const mgd_map_config& cfg, const MapRec* recs, long long n,
                               const unsigned long long* gt_hist, double* ap, double* voc,
                               unsigned long long* det_hist, void* scratch, cudaStream_t stream,
                               const mgd_map_pr* pr)
{
    return map_compute_impl<0>(cfg, recs, n, gt_hist, nullptr, 0, ap, voc, det_hist, scratch, stream, pr);
}

cudaError_t launch_map_compute_merged(const mgd_map_config& cfg, const MapRec* recs, long long n,
                                      const unsigned long long* gt_hist, const int* owner, int rank,
                                      double* ap, double* voc, unsigned long long* det_hist, void* scratch,
                                      cudaStream_t stream, const mgd_map_pr* pr)
{
    return map_compute_impl<kSlotDigits>(cfg, recs, n, gt_hist, owner, rank, ap, voc, det_hist, scratch, stream,
                                         pr);
}

size_t map_partition_scratch_bytes(long long n)
{
    return (size_t)((n + kTileItems - 1) / kTileItems) * 256 * 4;
}

cudaError_t launch_map_partition(const MapPartitionArgs& a, void* scratch, cudaStream_t stream)
{
    if (a.n == 0)
        return cudaMemsetAsync(a.counts, 0, (size_t)a.world * sizeof(long long), stream);
    const unsigned n = (unsigned)a.n;
    const unsigned tiles = (unsigned)((a.n + kTileItems - 1) / kTileItems);
    unsigned* tile_counts = static_cast<unsigned*>(scratch);
    const PartitionPass pass{a.recs, a.C, a.owner, a.world, a.segs, a.num_segs, a.out, a.status};
    prof_mark_begin(PROF_OTHER, stream);
    map_tile_count_kernel<<<tiles, kThreads, 0, stream>>>(pass, n, tile_counts);
    map_tile_offsets_kernel<<<1, kThreads, 0, stream>>>(pass, nullptr, tiles, tile_counts, a.counts, a.world);
    map_scatter_kernel<<<tiles, kThreads, 0, stream>>>(pass, n, tile_counts);
    prof_mark_end(PROF_OTHER, stream);
    return cudaGetLastError();
}
