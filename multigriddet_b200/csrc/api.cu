// C ABI of libmgd (include/mgd.h): validation, scratch management, batching,
// host staging and DLPack adapters around the kernels in encode.cu / decode.cu /
// nms.cu.  No compute happens on the host and there is no CPU fallback.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <chrono>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"
#include "dlpack_abi.h"

namespace {

thread_local std::string t_error;

int fail(int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    t_error = buf;
    return code;
}

// MGD_TRACE=1: print host-side timestamps of the staging path to stderr
static bool trace_on()
{
    const char* e = getenv("MGD_TRACE");
    return e && atoi(e);
}
struct Tracer {
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    const char* what;
    explicit Tracer(const char* w) : what(w) {}
    void mark(const char* stage)
    {
        if (!trace_on()) return;
        const auto t = std::chrono::steady_clock::now();
        fprintf(stderr, "[mgd %s] %-18s +%.1f us (abs %.3f ms)\n", what, stage,
                std::chrono::duration<double, std::micro>(t - t0).count(),
                std::chrono::duration<double, std::milli>(t.time_since_epoch()).count());
        t0 = t;
    }
};

#define CUDA_TRY(expr)                                                                   \
    do {                                                                                 \
        cudaError_t e__ = (expr);                                                        \
        if (e__ != cudaSuccess)                                                          \
            return fail(MGD_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e__)); \
    } while (0)

// ---- per-kernel event timing (observability; off unless mgd_profile_begin) -------
struct ProfSpan { int kind; int launches; cudaEvent_t t0, t1; };
thread_local bool t_prof_on = false;
thread_local std::vector<ProfSpan> t_prof_spans;
thread_local cudaEvent_t t_prof_open = nullptr;
// A group: ONE pair of events around several back-to-back launches of one kind (the per-chunk
// kernels of mgd_encode_decode_nms, which overlap head to tail through programmatic dependent
// launch -- an event record between two of them would serialise them again).  Inside a group
// the per-launch marks of that kind only count.
thread_local int t_prof_group_kind = -1;
thread_local int t_prof_group_launches = 0;
thread_local cudaEvent_t t_prof_group_open = nullptr;

}  // namespace

void prof_mark_begin(int kind, cudaStream_t stream)
{
    if (!t_prof_on) return;
    if (kind == t_prof_group_kind) return;
    cudaEventCreate(&t_prof_open);
    cudaEventRecord(t_prof_open, stream);
}

void prof_mark_end(int kind, cudaStream_t stream)
{
    if (!t_prof_on) return;
    if (kind == t_prof_group_kind) { ++t_prof_group_launches; return; }
    if (!t_prof_open) return;
    ProfSpan s;
    s.kind = kind;
    s.launches = 1;
    s.t0 = t_prof_open;
    cudaEventCreate(&s.t1);
    cudaEventRecord(s.t1, stream);
    t_prof_spans.push_back(s);
    t_prof_open = nullptr;
}

void prof_group_begin(int kind, cudaStream_t stream)
{
    if (!t_prof_on || t_prof_group_kind >= 0) return;
    t_prof_group_kind = kind;
    t_prof_group_launches = 0;
    cudaEventCreate(&t_prof_group_open);
    cudaEventRecord(t_prof_group_open, stream);
}

void prof_group_end(int kind, cudaStream_t stream)
{
    if (!t_prof_on || t_prof_group_kind != kind) return;
    if (t_prof_group_launches > 0) {
        ProfSpan s;
        s.kind = kind;
        s.launches = t_prof_group_launches;
        s.t0 = t_prof_group_open;
        cudaEventCreate(&s.t1);
        cudaEventRecord(s.t1, stream);
        t_prof_spans.push_back(s);
    } else {
        cudaEventDestroy(t_prof_group_open);
    }
    t_prof_group_open = nullptr;
    t_prof_group_kind = -1;
}

namespace {

// ---- per-device state -----------------------------------------------------------
// All scratch and staging memory comes from a library-owned stream-ordered pool per
// device (the application's default pool is left alone).  The pool never inserts
// cross-stream dependencies to reuse a block: a block freed behind a long D2H copy on
// one stream must not make another stream's H2D wait for that copy (with the default
// policy concurrent host-memory calls serialised their PCIe directions this way).
struct DeviceInfo {
    bool ready = false;
    int num_sms = 0;
    cudaMemPool_t pool = nullptr;
};
std::mutex g_mutex;
DeviceInfo g_dev[64];
thread_local cudaMemPool_t t_pool = nullptr;     // pool of the device the current call runs on

template <typename T> cudaError_t pool_malloc(T** p, size_t bytes, cudaStream_t stream)
{
    return cudaMallocFromPoolAsync(reinterpret_cast<void**>(p), bytes ? bytes : 16, t_pool, stream);
}

// Grow-only bump arena for the host-memory entry points: their staging buffers and
// per-chunk scratch are carved from memory cached per (host thread, device, stream slot),
// so a steady-state call performs no allocation at all.  (Per-chunk cudaMallocAsync /
// cudaFreeAsync made a second host thread's enqueue loop block until the first thread's
// call had drained, which serialised the two PCIe directions of concurrent calls.)
// reset() at the start of a chunk is safe because the arena is only ever used by work
// enqueued on one stream: stream order separates the chunks that share the memory.
struct Arena {
    struct Block { char* p; size_t cap; };
    std::vector<Block> blocks;
    size_t cur = 0, used = 0;
    void reset() { cur = 0; used = 0; }
    struct Mark { size_t cur, used; };
    Mark mark() const { return Mark{cur, used}; }
    void rewind(const Mark& m) { cur = m.cur; used = m.used; }
    cudaError_t take(void** out, size_t bytes)
    {
        bytes = (bytes + 255) & ~(size_t)255;
        if (bytes == 0) bytes = 256;
        for (; cur < blocks.size(); ++cur, used = 0)
            if (used + bytes <= blocks[cur].cap) {
                *out = blocks[cur].p + used;
                used += bytes;
                return cudaSuccess;
            }
        Block b;
        b.cap = bytes > (32u << 20) ? bytes : (32u << 20);
        cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&b.p), b.cap);
        if (e != cudaSuccess) return e;
        blocks.push_back(b);
        cur = blocks.size() - 1;
        used = bytes;
        *out = b.p;
        return cudaSuccess;
    }
    // after the call has synchronised: merge a fragmented arena into one block so the
    // next call of the same shape fits without growing
    void consolidate()
    {
        if (blocks.size() < 2) return;
        size_t total = 0;
        for (Block& b : blocks) { total += b.cap; cudaFree(b.p); }
        blocks.clear();
        Block b;
        b.cap = total;
        if (cudaMalloc(reinterpret_cast<void**>(&b.p), total) == cudaSuccess) blocks.push_back(b);
        else cudaGetLastError();
        reset();
    }
    void release()
    {
        for (Block& b : blocks) cudaFree(b.p);
        blocks.clear();
        reset();
    }
};

// where a kernel driver takes its scratch from: the stream-ordered pool (device-memory
// calls: freed back in stream order) or a bump arena (host-memory calls: nothing to free)
struct Alloc {
    Arena* arena;
    cudaStream_t stream;
    template <typename T> cudaError_t get(T** p, size_t bytes) const
    {
        if (arena) return arena->take(reinterpret_cast<void**>(p), bytes);
        return pool_malloc(p, bytes, stream);
    }
    cudaError_t put(void* p) const { return arena || !p ? cudaSuccess : cudaFreeAsync(p, stream); }
    // arena mode: scratch of one internal chunk is recycled by the next (same stream)
    Arena::Mark mark() const { return arena ? arena->mark() : Arena::Mark{0, 0}; }
    void rewind(const Arena::Mark& m) const { if (arena) arena->rewind(m); }
};

int device_count_quiet()
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// Entry points run on `device` and put the caller's current device back on exit: the
// library must not change the application's (or torch's) notion of the current device.
struct DeviceScope {
    int prev = -1;
    ~DeviceScope()
    {
        if (prev >= 0 && cudaSetDevice(prev) != cudaSuccess) cudaGetLastError();
    }
};

int prepare_device(int device, int* num_sms, DeviceScope* scope)
{
    const int n = device_count_quiet();
    if (n == 0)
        return fail(MGD_ERR_NO_DEVICE,
                    "no CUDA device available: libmgd has no CPU fallback (sm_100a kernels only)");
    if (device < 0 || device >= n || device >= 64)
        return fail(MGD_ERR_INVALID_ARGUMENT, "device %d out of range (have %d)", device, n);
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess) { cudaGetLastError(); cur = -1; }
    if (cur != device) {
        CUDA_TRY(cudaSetDevice(device));
        if (scope && scope->prev < 0) scope->prev = cur;
    }
    std::lock_guard<std::mutex> lock(g_mutex);
    DeviceInfo& d = g_dev[device];
    if (!d.ready) {
        cudaDeviceProp prop;
        CUDA_TRY(cudaGetDeviceProperties(&prop, device));
        if (prop.major != 10)
            return fail(MGD_ERR_NO_DEVICE,
                        "device %d is sm_%d%d; libmgd is built for sm_100a (B200) only",
                        device, prop.major, prop.minor);
        d.num_sms = prop.multiProcessorCount;
        cudaMemPoolProps pp;
        memset(&pp, 0, sizeof(pp));
        pp.allocType = cudaMemAllocationTypePinned;
        pp.handleTypes = cudaMemHandleTypeNone;
        pp.location.type = cudaMemLocationTypeDevice;
        pp.location.id = device;
        CUDA_TRY(cudaMemPoolCreate(&d.pool, &pp));
        // keep freed scratch in the pool instead of returning it to the OS
        unsigned long long keep = ~0ull;
        CUDA_TRY(cudaMemPoolSetAttribute(d.pool, cudaMemPoolAttrReleaseThreshold, &keep));
        int off = 0;
        CUDA_TRY(cudaMemPoolSetAttribute(d.pool, cudaMemPoolReuseAllowInternalDependencies, &off));
        d.ready = true;
    }
    t_pool = d.pool;
    *num_sms = d.num_sms;
    return MGD_OK;
}

// ---- geometry --------------------------------------------------------------------
int build_geom(const mgd_head_config* cfg, HeadGeom* g)
{
    if (!cfg) return fail(MGD_ERR_INVALID_ARGUMENT, "cfg is NULL");
    if (cfg->num_layers < 1 || cfg->num_layers > MGD_MAX_LAYERS)
        return fail(MGD_ERR_INVALID_ARGUMENT, "num_layers must be in [1, %d], got %d",
                    MGD_MAX_LAYERS, cfg->num_layers);
    if (cfg->num_classes < 1)
        return fail(MGD_ERR_INVALID_ARGUMENT, "num_classes must be >= 1, got %d", cfg->num_classes);
    if (cfg->input_h < 1 || cfg->input_w < 1)
        return fail(MGD_ERR_INVALID_ARGUMENT, "input shape must be positive");
    if (cfg->input_h != cfg->input_w)
        return fail(MGD_ERR_UNSUPPORTED,
                    "non-square input %dx%d: the reference's cell arithmetic is only "
                    "self-consistent for square inputs (generators.py:3438-3470)",
                    cfg->input_h, cfg->input_w);
    memset(g, 0, sizeof(*g));
    g->L = cfg->num_layers;
    g->C = cfg->num_classes;
    g->in_h = cfg->input_h;
    g->in_w = cfg->input_w;
    g->anchors_f64 = cfg->anchors_f64 ? 1 : 0;
    int k = 0;
    long long cells = 0;
    for (int l = 0; l < g->L; ++l) {
        if (cfg->grid_h[l] < 1 || cfg->grid_w[l] < 1 || cfg->grid_h[l] > 8192)
            return fail(MGD_ERR_INVALID_ARGUMENT, "grid of layer %d must be in [1, 8192]", l);
        if (cfg->grid_h[l] != cfg->grid_w[l])
            return fail(MGD_ERR_UNSUPPORTED, "non-square grid %dx%d on layer %d",
                        cfg->grid_h[l], cfg->grid_w[l], l);
        if (cfg->num_anchors[l] < 1 || cfg->num_anchors[l] > MGD_MAX_ANCHORS_PER_LAYER)
            return fail(MGD_ERR_INVALID_ARGUMENT, "layer %d: anchors per layer must be in [1, %d]",
                        l, MGD_MAX_ANCHORS_PER_LAYER);
        g->gh[l] = cfg->grid_h[l];
        g->gw[l] = cfg->grid_w[l];
        g->na[l] = cfg->num_anchors[l];
        g->D[l] = 5 + g->na[l] + g->C;
        g->anchor_first[l] = k;
        g->cell_off[l] = (int)cells;
        for (int i = 0; i < g->na[l]; ++i, ++k) {
            const double w = cfg->anchors[l][i][0], h = cfg->anchors[l][i][1];
            if (!(w > 0.0) || !(h > 0.0))
                return fail(MGD_ERR_INVALID_ARGUMENT, "anchor %d of layer %d is not positive", i, l);
            g->anc64[k][0] = w; g->anc64[k][1] = h;
            g->anc32[k][0] = (float)w; g->anc32[k][1] = (float)h;
        }
        cells += (long long)g->gh[l] * g->gw[l];
    }
    if (cells > (1 << 24))
        return fail(MGD_ERR_UNSUPPORTED, "%lld cells per image exceeds the supported 2^24", cells);
    g->K = k;
    g->cells = (int)cells;
    return MGD_OK;
}

int check_memory_arg(int memory)
{
    if (memory != MGD_MEM_HOST && memory != MGD_MEM_DEVICE)
        return fail(MGD_ERR_INVALID_ARGUMENT, "memory must be MGD_MEM_HOST or MGD_MEM_DEVICE");
    return MGD_OK;
}

int env_chunk(const char* name)
{
    const char* e = getenv(name);            // (read per call: tests shrink the chunks)
    return e ? atoi(e) : 0;
}

// images per internal chunk: keeps the per-chunk scratch (owner table / candidate
// lists) around 32 MB so it stays L2-resident between the two kernels that share it
int chunk_images(const HeadGeom& g, int batch)
{
    long long n = (32ll << 20) / ((long long)g.cells * 4);
    if (const int e = env_chunk("MGD_ENCODE_CHUNK_IMAGES")) n = e;
    if (n < 1) n = 1;
    if (n > batch) n = batch;
    return (int)n;
}

// decode + NMS: one NMS launch should see thousands of images (a warp per image), so the
// chunk is bounded by the candidate scratch (<= 1 GiB of 32-byte slots) instead
int decode_chunk_images(const HeadGeom& g, int batch)
{
    long long n = (1ll << 30) / ((long long)g.cells * (long long)sizeof(Cand));
    if (const int e = env_chunk("MGD_DECODE_CHUNK_IMAGES")) n = e;
    if (n < 1) n = 1;
    if (n > batch) n = batch;
    return (int)n;
}

// ---- deferred device-side status of asynchronous encode calls ---------------------
// One persistent device word per (host thread, device): every asynchronous call ORs its
// status bits into it (atomicOr in the assign kernel), mgd_poll_status reads it back and
// clears it.  Nothing is allocated per call and nothing accumulates if the caller never
// polls.
struct DeferredStatus {
    int* word[64] = {};
    ~DeferredStatus()
    {
        for (int d = 0; d < 64; ++d) if (word[d]) cudaFree(word[d]);
        cudaGetLastError();
    }
};
thread_local DeferredStatus t_deferred;

int deferred_status_word(int device, int** out)
{
    if (!t_deferred.word[device]) {
        CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&t_deferred.word[device]), 256));
        CUDA_TRY(cudaMemset(t_deferred.word[device], 0, 256));
    }
    *out = t_deferred.word[device];
    return MGD_OK;
}

int status_to_error(int st)
{
    if (st & 1) return fail(MGD_ERR_CLASS_RANGE, "class id must be less than num_classes");
    if (st & 2)
        return fail(MGD_ERR_INVALID_ARGUMENT,
                    "negative class id on a valid box (the reference would write a wrong channel)");
    if (st & 4) return fail(MGD_ERR_CLASS_RANGE, "mAP update: class id outside [0, num_classes)");
    if (st & 8) return fail(MGD_ERR_INVALID_ARGUMENT, "mAP partition: owner table entry outside [0, world)");
    return MGD_OK;
}

// ---- encode ------------------------------------------------------------------------
struct EncodeScratch { int* table; BoxRec* recs; };

// The fused entry (mgd_encode_decode_nms) runs the encoder in two phases.  The assign kernel
// needs ~60 KB of shared memory per CTA and cannot share an SM with the decoder's persistent
// CTAs, and the y_true writer and the decoder are both DRAM-bound (run together they take longer
// than one after the other: 4.6 ms against 3.6 ms per 4 096 images); the NMS that follows the
// decoder is latency-bound and leaves the memory system idle.  So: every chunk's assign kernel
// first, then the decoder, then the writer on a second stream underneath the NMS.
// MGD_STEP_PDL=0: plain launches instead of programmatic dependent launches between the
// independent per-chunk kernels of mgd_encode_decode_nms (measurements)
bool step_pdl()
{
    static int v = -1;
    if (v < 0) { const char* e = getenv("MGD_STEP_PDL"); v = e ? atoi(e) : 1; }
    return v != 0;
}

int encode_assign_all(const HeadGeom& g, const float* boxes, int batch, int N, float* const* y,
                      cudaStream_t stream, int* d_status, int tf_compat, std::vector<EncodeArgs>* chunks)
{
    nvtx_range nv("mgd:encode assign (preprocess_true_boxes)");
    const Alloc al{nullptr, stream};
    const int step = chunk_images(g, batch);
    // scratch of every chunk first, then the kernels back to back (nothing between two launches:
    // they overlap head to tail through programmatic dependent launch)
    for (int b0 = 0; b0 < batch; b0 += step) {
        const int nb = batch - b0 < step ? batch - b0 : step;
        EncodeArgs a;
        a.g = g;
        a.B = nb;
        a.N = N;
        a.boxes = boxes + (size_t)b0 * N * 5;
        for (int l = 0; l < g.L; ++l)
            a.y[l] = y[l] + (size_t)b0 * g.gh[l] * g.gw[l] * g.D[l];
        a.tf_compat = tf_compat;
        a.status = d_status;
        a.stats = nullptr;
        a.big_tables = nullptr;
        a.table = nullptr;
        a.recs = nullptr;
        chunks->push_back(a);                    // (first, so that a failure below still frees it)
        EncodeArgs& c = chunks->back();
        if (encode_needs_big_tables(g, N))
            CUDA_TRY(al.get(&c.big_tables, (size_t)nb * 2 * g.cells * sizeof(int)));
        CUDA_TRY(al.get(&c.table, (size_t)nb * g.cells * sizeof(int)));
        CUDA_TRY(al.get(&c.recs, (size_t)nb * (N > 0 ? N : 1) * sizeof(BoxRec)));
    }
    struct Group {                                   // one event pair around the chunk launches
        cudaStream_t st;
        explicit Group(cudaStream_t s) : st(s) { prof_group_begin(PROF_ENCODE_ASSIGN, st); }
        ~Group() { prof_group_end(PROF_ENCODE_ASSIGN, st); }
    } group(stream);
    // (each chunk has its own tables here, alive until encode_free_all: the assign kernels of
    //  consecutive chunks are independent)
    for (size_t k = 0; k < chunks->size(); ++k)
        CUDA_TRY(launch_encode_assign((*chunks)[k], stream, k > 0 && step_pdl()));
    return MGD_OK;
}

// the writer of every chunk on `stream` (which must already be ordered behind the assigns)
int encode_fill_all(std::vector<EncodeArgs>& chunks, int num_sms, cudaStream_t stream)
{
    nvtx_range nv("mgd:encode fill (preprocess_true_boxes)");
    const bool env_pdl = step_pdl();
    bool first = true;
    prof_group_begin(PROF_ENCODE_FILL, stream);
    struct GroupEnd { cudaStream_t st; ~GroupEnd() { prof_group_end(PROF_ENCODE_FILL, st); } } group_end{stream};
    for (EncodeArgs& a : chunks) {
        // every chunk's tables are alive until the caller frees them: consecutive writers are
        // independent and may overlap head to tail
        const cudaError_t e = launch_encode_fill(a, num_sms, stream, env_pdl && !first);
        if (e != cudaSuccess) return fail(MGD_ERR_CUDA, "y_true writer launch failed: %s", cudaGetErrorString(e));
        first = false;
    }
    return MGD_OK;
}

// Scratch goes back to the pool on the stream it was allocated on (once that stream is ordered
// behind every user): a block freed on another stream is not reused by this stream's next
// allocation -- the pool grew by the owner tables (125 MB per 4 096 images) every step.
void encode_free_all(std::vector<EncodeArgs>& chunks, cudaStream_t stream)
{
    const Alloc al{nullptr, stream};
    for (EncodeArgs& a : chunks) {
        al.put(a.table); al.put(a.recs); al.put(a.big_tables);
        a.table = nullptr; a.recs = nullptr; a.big_tables = nullptr;
    }
    cudaGetLastError();
}

int encode_device(const HeadGeom& g, const float* boxes, int batch, int N, float* const* y,
                  int num_sms, cudaStream_t stream, int* d_status, unsigned long long* d_stats,
                  const Alloc& al, int tf_compat)
{
    nvtx_range nv("mgd:encode (preprocess_true_boxes)");
    const int step = chunk_images(g, batch);
    for (int b0 = 0; b0 < batch; b0 += step) {
        const int nb = batch - b0 < step ? batch - b0 : step;
        const Arena::Mark mk = al.mark();
        EncodeArgs a;
        a.g = g;
        a.B = nb;
        a.N = N;
        a.boxes = boxes + (size_t)b0 * N * 5;
        for (int l = 0; l < g.L; ++l)
            a.y[l] = y[l] + (size_t)b0 * g.gh[l] * g.gw[l] * g.D[l];
        a.tf_compat = tf_compat;
        a.status = d_status;
        a.stats = d_stats;
        a.big_tables = nullptr;
        if (encode_needs_big_tables(g, N))
            CUDA_TRY(al.get(&a.big_tables, (size_t)nb * 2 * g.cells * sizeof(int)));
        CUDA_TRY(al.get(&a.table, (size_t)nb * g.cells * sizeof(int)));
        CUDA_TRY(al.get(&a.recs, (size_t)nb * (N > 0 ? N : 1) * sizeof(BoxRec)));
        CUDA_TRY(launch_encode(a, num_sms, stream));
        CUDA_TRY(al.put(a.table));
        CUDA_TRY(al.put(a.recs));
        CUDA_TRY(al.put(a.big_tables));
        al.rewind(mk);
    }
    return MGD_OK;
}

// ---- detection exchange (mgd_exchange_*) -------------------------------------------
// A buffer of device memory per rank, every rank's buffer mapped into every process of the
// job through CUDA IPC.  Detection outputs that lie in the local buffer are mirrored into the
// peers' buffers by the NMS kernels themselves (nms.cu: mirror_store); exchange.cu orders it.
}  // namespace (the handle type is part of the ABI: declared in mgd.h as an opaque struct)

struct mgd_exchange {
    int device = 0, world = 1, rank = 0;
    size_t bytes = 0;                                   // caller-visible bytes (after the header)
    char* alloc[MGD_EXCHANGE_MAX_RANKS] = {};           // every rank's allocation in this process
    bool connected = false;
    unsigned epoch = 0;                                 // collective calls made so far
    cudaIpcMemHandle_t handle;
};

namespace {

std::mutex g_exchange_mutex;
std::vector<mgd_exchange*> g_exchanges;

// the connected exchange whose local caller-visible bytes contain p, or nullptr
mgd_exchange* exchange_of(const void* p, int device)
{
    std::lock_guard<std::mutex> lock(g_exchange_mutex);
    const char* c = static_cast<const char*>(p);
    for (mgd_exchange* ex : g_exchanges) {
        const char* lo = ex->alloc[ex->rank] + MGD_EXCHANGE_HEADER_BYTES;
        if (ex->device == device && c >= lo && c < lo + ex->bytes) return ex;
    }
    return nullptr;
}

bool exchange_holds(const mgd_exchange* ex, const void* p, size_t nbytes)
{
    const char* c = static_cast<const char*>(p);
    const char* lo = ex->alloc[ex->rank] + MGD_EXCHANGE_HEADER_BYTES;
    return c >= lo && c + nbytes <= lo + ex->bytes;
}

ExchangeView exchange_view(const mgd_exchange* ex)
{
    ExchangeView v;
    memset(&v, 0, sizeof(v));
    v.world = ex->world;
    v.rank = ex->rank;
    for (int r = 0; r < ex->world; ++r) v.header[r] = reinterpret_cast<unsigned*>(ex->alloc[r]);
    return v;
}

// ---- decode + nms -------------------------------------------------------------------
float objectness_prefilter(const mgd_post_config& post)
{
    // score <= sigmoid(obj): a row with sigmoid(obj) < confidence can never pass.
    // Compare raw logits against logit(confidence) minus a margin that dwarfs any
    // float32 rounding in the reference's sigmoid (relative 1e-4 vs 1e-7).
    const double c = post.confidence;
    if (!(c > 0.0)) return -INFINITY;
    if (c >= 1.0) return 15.0f;            // sigmoid_f32(x) reaches 1.0f only for x > 17.3
    const double logit = log(c / (1.0 - c));
    return (float)(logit - 1e-3 - 1e-4 * fabs(logit));
}

int decode_nms_device(const HeadGeom& g, const mgd_post_config& post, const float* const* preds,
                      int batch, const int* image_hw, double* xywh, int* xyxy, double* scores,
                      int* classes, int* index, int* counts, int num_sms, cudaStream_t stream,
                      unsigned long long* d_stats, const Alloc& al,
                      const std::function<int()>* after_first_decode = nullptr)
{
    nvtx_range nv("mgd:decode+nms (MultiGridDecoder.postprocess)");
    const int step = decode_chunk_images(g, batch);
    const int M = post.max_boxes;
    int pow2 = 2;
    while (pow2 < g.cells) pow2 <<= 1;
    const bool big_sort = g.cells > nms_smem_capacity();
    const bool big_keep = nms_kept_bytes(M) > 64 * 1024;
    // Outputs inside a connected detection exchange are mirrored to every peer rank by the
    // NMS kernels; the call is then collective (every rank of the exchange makes it).
    int cur_dev = 0;
    CUDA_TRY(cudaGetDevice(&cur_dev));
    mgd_exchange* ex = al.arena ? nullptr : exchange_of(counts, cur_dev);
    if (ex) {
        const struct { const void* p; size_t n; const char* name; } outs[] = {
            {xywh, (size_t)batch * M * 4 * sizeof(double), "boxes_xywh"},
            {xyxy, (size_t)batch * M * 4 * sizeof(int), "boxes_xyxy"},
            {scores, (size_t)batch * M * sizeof(double), "scores"},
            {classes, (size_t)batch * M * sizeof(int), "classes"},
            {index, (size_t)batch * M * sizeof(int), "index"},
            {counts, (size_t)batch * sizeof(int), "counts"}};
        for (const auto& o : outs) {
            if (!o.p) continue;
            if (!exchange_holds(ex, o.p, o.n))
                return fail(MGD_ERR_INVALID_ARGUMENT, "counts lies in a detection exchange but %s does "
                            "not (all outputs of a mirrored call must come from the same exchange)", o.name);
            if ((reinterpret_cast<uintptr_t>(o.p) & 15) && (o.p == (const void*)xywh || o.p == (const void*)xyxy))
                return fail(MGD_ERR_INVALID_ARGUMENT, "%s inside a detection exchange must be 16-byte aligned", o.name);
        }
        ++ex->epoch;
        // "ready", first half: this rank no longer reads the rows the call is about to overwrite
        if (ex->world > 1)
            CUDA_TRY(launch_exchange_barrier(exchange_view(ex), 0, ex->epoch, MGD_EXCHANGE_SIGNAL, stream));
    }
    for (int b0 = 0; b0 < batch; b0 += step) {
        const int nb = batch - b0 < step ? batch - b0 : step;
        const Arena::Mark mk = al.mark();
        DecodeArgs d;
        memset(&d, 0, sizeof(d));
        d.g = g;
        d.B = nb;
        for (int l = 0; l < g.L; ++l)
            d.pred[l] = preds[l] + (size_t)b0 * g.gh[l] * g.gw[l] * g.D[l];
        d.image_hw = image_hw ? image_hw + 2 * (size_t)b0 : nullptr;
        d.use_softmax = post.use_softmax;
        d.rescore = post.rescore_confidence;
        d.confidence = post.confidence;
        d.obj_logit_min = objectness_prefilter(post);
        d.score_lo = post.confidence > 0.0 ? (float)(post.confidence * (1.0 - 1e-3)) : -1.0f;
        CUDA_TRY(al.get(&d.cand, (size_t)nb * g.cells * sizeof(Cand)));
        // counts[nb], counts[nb+1]: the work counters of the two warp-per-image NMS launches
        CUDA_TRY(al.get(&d.counts, (size_t)(nb + 2) * sizeof(int)));
        CUDA_TRY(cudaMemsetAsync(d.counts, 0, (size_t)(nb + 2) * sizeof(int), stream));
        {
            const cudaError_t e = launch_decode(d, num_sms, stream);
            if (e == cudaErrorInvalidConfiguration) {
                cudaGetLastError();
                return fail(MGD_ERR_UNSUPPORTED, "head too wide for the decode kernel: %d channels per "
                            "cell (at most ~1750 are supported)", g.D[0]);
            }
            CUDA_TRY(e);
        }
        if (after_first_decode && b0 == 0) {
            const int hook_rc = (*after_first_decode)();
            if (hook_rc) return hook_rc;
        }

        NmsArgs n;
        memset(&n, 0, sizeof(n));
        n.g = g;
        n.B = nb;
        n.cap = g.cells;
        n.cand = d.cand;
        CUDA_TRY(al.get(&n.boxes, (size_t)nb * g.cells * sizeof(BoxD)));
        n.counts = d.counts;
        n.next_image = d.counts + nb;
        n.image_hw = d.image_hw;
        n.in_h = g.in_h; n.in_w = g.in_w;
        n.thr = post.nms_threshold;
        n.use_diou = post.nms_method == MGD_NMS_DIOU;
        n.per_class = post.per_class;
        n.max_boxes = M;
        if (post.nms_method == MGD_NMS_SOFT) {
            n.soft = 1;
            n.soft_sigma = post.soft_sigma > 0.0 ? post.soft_sigma : 0.5;
            n.soft_thr = post.soft_score_threshold >= 0.0 ? post.soft_score_threshold : 0.001;
            CUDA_TRY(al.get(&n.soft_scratch, (size_t)nb * g.cells * sizeof(double)));
        }
        if (post.nms_method == MGD_NMS_WBF) {
            if (g.C > 65535) return fail(MGD_ERR_UNSUPPORTED, "WBF supports up to 65535 classes");
            n.wbf = 1;
            n.wbf_conf_type = MGD_WBF_CONF_AVG;            // handle_predictions: WeightedBoxesFusion(iou_thr=...)
            n.soft_thr = 0.0;                              // skip_box_thr default
            CUDA_TRY(al.get(&n.soft_scratch, (size_t)nb * g.cells * 5 * sizeof(double)));
            CUDA_TRY(al.get(&n.wbf_ints, (size_t)nb * g.cells * 4 * sizeof(int)));
        }
        if (n.wbf || big_sort) {                         // one allocation serves both users
            n.sort_scratch_stride = pow2;
            CUDA_TRY(al.get(&n.sort_scratch, (size_t)nb * 2 * pow2 * sizeof(unsigned long long)));
        }
        if (big_keep) {
            n.kept_scratch_stride = (nms_kept_bytes(M) + 15) & ~(size_t)15;
            CUDA_TRY(al.get(&n.kept_scratch, (size_t)nb * n.kept_scratch_stride));
        }
        n.out_xywh = xywh ? xywh + (size_t)b0 * M * 4 : nullptr;
        n.out_xyxy = xyxy ? xyxy + (size_t)b0 * M * 4 : nullptr;
        n.out_scores = scores ? scores + (size_t)b0 * M : nullptr;
        n.out_classes = classes ? classes + (size_t)b0 * M : nullptr;
        n.out_index = index ? index + (size_t)b0 * M : nullptr;
        n.out_counts = counts + b0;
        n.stats = d_stats;
        // With the y_true writer running underneath (mgd_encode_decode_nms), 4 resident NMS CTAs
        // per SM instead of the 7 that fit: the NMS gets slower (0.55 -> 0.8 ms per 4 096 images)
        // but stays hidden, and the writer keeps more of the SM (step 3.04 -> 2.94 ms).
        if (after_first_decode) n.warp_ctas_per_sm = 4;
        if (ex && ex->world > 1) {
            for (int r = 0; r < ex->world; ++r)
                if (r != ex->rank)
                    n.mirror_delta[n.n_mirrors++] = (long long)(ex->alloc[r] - ex->alloc[ex->rank]);
            // "ready", second half: every peer has entered its call (it may still be decoding)
            if (b0 == 0) CUDA_TRY(launch_exchange_barrier(exchange_view(ex), 0, ex->epoch, MGD_EXCHANGE_WAIT, stream));
        }
        CUDA_TRY(launch_nms(n, num_sms, stream));
        // "complete": every rank's rows of this call have landed everywhere
        if (ex && ex->world > 1 && b0 + nb >= batch)
            CUDA_TRY(launch_exchange_barrier(exchange_view(ex), 1, ex->epoch,
                                             MGD_EXCHANGE_SIGNAL | MGD_EXCHANGE_WAIT, stream));
        CUDA_TRY(al.put(n.sort_scratch));
        CUDA_TRY(al.put(n.kept_scratch));
        CUDA_TRY(al.put(n.soft_scratch));
        CUDA_TRY(al.put(n.wbf_ints));
        CUDA_TRY(al.put(n.boxes));
        CUDA_TRY(al.put(d.cand));
        CUDA_TRY(al.put(d.counts));
        al.rewind(mk);
    }
    return MGD_OK;
}

int check_post(const mgd_post_config* post)
{
    if (!post) return fail(MGD_ERR_INVALID_ARGUMENT, "post config is NULL");
    if (post->max_boxes < 1 || post->max_boxes > (1 << 20))
        return fail(MGD_ERR_INVALID_ARGUMENT, "max_boxes must be in [1, 2^20], got %d", post->max_boxes);
    if (post->nms_method < MGD_NMS_IOU || post->nms_method > MGD_NMS_WBF)
        return fail(MGD_ERR_UNSUPPORTED, "nms_method %d is not built", post->nms_method);
    if (post->confidence != post->confidence || post->nms_threshold != post->nms_threshold)
        return fail(MGD_ERR_INVALID_ARGUMENT, "confidence / nms_threshold is NaN");
    return MGD_OK;
}

// streams used for host-memory calls, one pair per host thread and device
struct HostStreams {
    cudaStream_t s[2] = {nullptr, nullptr};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    Arena chunk[2];          // staging + scratch of the chunk in flight on s[i]
    Arena call;              // per-call tensors (boxes, output slab, status words)
    // scratch of the mAP entry points (device-memory calls on the caller's stream): the next
    // call, on whatever stream, first waits for map_done, recorded behind the previous one
    Arena map;
    cudaEvent_t map_done = nullptr;
    // page-locked bounce buffers for PAGEABLE caller memory: the driver's own pageable
    // path is one memcpy thread (~11 GB/s); several threads filling a page-locked chunk
    // while the previous chunk is on the link reach ~3x that
    unsigned char* bounce[2] = {nullptr, nullptr};
    size_t bounce_cap[2] = {0, 0};
    cudaEvent_t bounce_done[2] = {nullptr, nullptr};
    bool bounce_busy[2] = {false, false};
    // a host thread that ends gives its staging back (errors ignored: at process exit the
    // CUDA runtime may already be gone)
    ~HostStreams()
    {
        if (!s[0] && !s[1] && chunk[0].blocks.empty() && chunk[1].blocks.empty() &&
            call.blocks.empty() && map.blocks.empty() && !map_done && !bounce[0] && !bounce[1]) return;
        for (int i = 0; i < 2; ++i) if (s[i]) cudaStreamSynchronize(s[i]);
        if (map_done) { cudaEventSynchronize(map_done); cudaEventDestroy(map_done); }
        chunk[0].release(); chunk[1].release(); call.release(); map.release();
        for (int i = 0; i < 2; ++i) {
            if (bounce[i]) cudaFreeHost(bounce[i]);
            if (bounce_done[i]) cudaEventDestroy(bounce_done[i]);
            if (ev[i]) cudaEventDestroy(ev[i]);
            if (s[i]) cudaStreamDestroy(s[i]);
        }
        cudaGetLastError();
    }
};
thread_local HostStreams t_streams[64];

int host_streams(int device, cudaStream_t** out, cudaEvent_t** ev, HostStreams** self = nullptr)
{
    HostStreams& hs = t_streams[device];
    if (self) *self = &hs;
    for (int i = 0; i < 2; ++i) {
        if (!hs.s[i]) CUDA_TRY(cudaStreamCreateWithFlags(&hs.s[i], cudaStreamNonBlocking));
        if (!hs.ev[i]) CUDA_TRY(cudaEventCreateWithFlags(&hs.ev[i], cudaEventDisableTiming));
    }
    *out = hs.s;
    if (ev) *ev = hs.ev;
    return MGD_OK;
}

// true when the driver knows nothing about p: ordinary pageable host memory
bool is_pageable(const void* p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return at.type == cudaMemoryTypeUnregistered;
}

int host_copy_threads()
{
    static int n = -1;
    if (n < 0) {
        const char* e = getenv("MGD_HOST_COPY_THREADS");
        const int hw = (int)std::thread::hardware_concurrency();
        n = e ? atoi(e) : (hw >= 32 ? 8 : (hw >= 8 ? hw / 4 : 2));   // a quarter of the cores, 2..8
        if (hw > 0 && n > hw) n = hw;
        if (n < 1) n = 1;
    }
    return n;
}

void parallel_copy(void* dst, const void* src, size_t bytes)
{
    const int n = bytes < (8u << 20) ? 1 : host_copy_threads();
    if (n == 1) { memcpy(dst, src, bytes); return; }
    const size_t part = ((bytes / n) + 4095) & ~(size_t)4095;
    std::vector<std::thread> workers;
    for (int i = 1; i < n; ++i) {
        const size_t off = (size_t)i * part;
        if (off >= bytes) break;
        const size_t len = off + part < bytes ? part : bytes - off;
        workers.emplace_back([=] { memcpy(static_cast<char*>(dst) + off, static_cast<const char*>(src) + off, len); });
    }
    memcpy(dst, src, part < bytes ? part : bytes);
    for (std::thread& t : workers) t.join();
}

// page-locked bounce slot of at least `bytes`, idle (its previous H2D has completed)
int bounce_slot(HostStreams* hs, int slot, size_t bytes, unsigned char** out)
{
    if (hs->bounce_busy[slot]) {
        CUDA_TRY(cudaEventSynchronize(hs->bounce_done[slot]));
        hs->bounce_busy[slot] = false;
    }
    if (hs->bounce_cap[slot] < bytes) {
        if (hs->bounce[slot]) CUDA_TRY(cudaFreeHost(hs->bounce[slot]));
        hs->bounce[slot] = nullptr; hs->bounce_cap[slot] = 0;
        CUDA_TRY(cudaHostAlloc(reinterpret_cast<void**>(&hs->bounce[slot]), bytes, cudaHostAllocPortable));
        hs->bounce_cap[slot] = bytes;
    }
    if (!hs->bounce_done[slot]) CUDA_TRY(cudaEventCreateWithFlags(&hs->bounce_done[slot], cudaEventDisableTiming));
    *out = hs->bounce[slot];
    return MGD_OK;
}

// A host pointer the GPU can address in place (cudaHostAlloc / cudaHostRegister /
// torch pin_memory under UVA): returns its device alias, nullptr for pageable memory.
template <typename T> T* mapped_alias(T* p, size_t bytes)
{
    if (!p || bytes == 0) return nullptr;
    const unsigned char* ends[2] = {reinterpret_cast<const unsigned char*>(p),
                                    reinterpret_cast<const unsigned char*>(p) + bytes - 1};
    void* dev = nullptr;
    for (int i = 0; i < 2; ++i) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, ends[i]) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        if (at.type != cudaMemoryTypeHost || !at.devicePointer) return nullptr;
        if (i == 0) dev = at.devicePointer;
    }
    return reinterpret_cast<T*>(dev);
}

// MGD_HOST_ZEROCOPY: bit 0 = decode reads pinned predictions in place over PCIe (only the
// sectors the three-level filter asks for cross the link), bit 1 = encode writes pinned
// y_true in place.  Pageable memory always takes the staged path.
int zerocopy_mode()
{
    static int v = -1;
    if (v < 0) { const char* e = getenv("MGD_HOST_ZEROCOPY"); v = e ? atoi(e) : 0; }
    return v;
}

int host_chunk(const HeadGeom& g, int batch)
{
    // ~128 MB of y_true / predictions per chunk (2.3 ms on a Gen5 x16 link): long enough
    // to run the link at speed, short enough that (a) the two streams overlap H2D, kernels
    // and D2H within a call and (b) concurrent calls from other host threads interleave on
    // the copy engines instead of queueing behind a near-gigabyte transfer
    static long long mb = -1;
    if (mb < 0) { const char* e = getenv("MGD_HOST_CHUNK_MB"); mb = e && atoll(e) > 0 ? atoll(e) : 128; }
    long long per_image = 0;
    for (int l = 0; l < g.L; ++l) per_image += (long long)g.gh[l] * g.gw[l] * g.D[l] * 4;
    long long n = (mb << 20) / (per_image > 0 ? per_image : 1);
    if (n < 1) n = 1;
    if (n > batch) n = batch;
    return (int)n;
}

}  // namespace

extern "C" {

int mgd_version(void) { return MGD_VERSION; }

const char* mgd_last_error(void) { return t_error.c_str(); }

int mgd_device_count(void) { return device_count_quiet(); }

int mgd_host_alloc(size_t bytes, void** ptr)
{
    if (!ptr) return fail(MGD_ERR_INVALID_ARGUMENT, "ptr is NULL");
    *ptr = nullptr;
    if (device_count_quiet() == 0)
        return fail(MGD_ERR_NO_DEVICE, "no CUDA device: page-locked memory is not available");
    CUDA_TRY(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocPortable));
    return MGD_OK;
}

int mgd_host_free(void* ptr)
{
    if (ptr) CUDA_TRY(cudaFreeHost(ptr));
    return MGD_OK;
}

int mgd_exchange_create(int device, int world_size, int rank, size_t bytes, mgd_exchange** out,
                        unsigned char* handle)
{
    if (!out || !handle) return fail(MGD_ERR_INVALID_ARGUMENT, "NULL argument");
    *out = nullptr;
    if (world_size < 1 || world_size > MGD_EXCHANGE_MAX_RANKS)
        return fail(MGD_ERR_UNSUPPORTED, "a detection exchange spans 1..%d ranks (one node), got %d",
                    MGD_EXCHANGE_MAX_RANKS, world_size);
    if (rank < 0 || rank >= world_size) return fail(MGD_ERR_INVALID_ARGUMENT, "rank %d outside [0, %d)", rank, world_size);
    if (bytes == 0) return fail(MGD_ERR_INVALID_ARGUMENT, "bytes must be > 0");
    int num_sms;
    DeviceScope dev_scope;
    int rc = prepare_device(device, &num_sms, &dev_scope);
    if (rc) return rc;
    static_assert(sizeof(cudaIpcMemHandle_t) == MGD_IPC_HANDLE_BYTES, "IPC handle size");
    mgd_exchange* ex = new mgd_exchange();
    ex->device = device;
    ex->world = world_size;
    ex->rank = rank;
    ex->bytes = (bytes + 255) & ~(size_t)255;
    // cudaMalloc, not the stream-ordered pool: only plain allocations can be exported over IPC
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, MGD_EXCHANGE_HEADER_BYTES + ex->bytes);
    if (e == cudaSuccess) e = cudaMemset(p, 0, MGD_EXCHANGE_HEADER_BYTES + ex->bytes);
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&ex->handle, p);
    if (e != cudaSuccess) {
        if (p) cudaFree(p);
        delete ex;
        cudaGetLastError();
        return fail(MGD_ERR_CUDA, "exchange allocation failed: %s", cudaGetErrorString(e));
    }
    ex->alloc[rank] = static_cast<char*>(p);
    memcpy(handle, &ex->handle, MGD_IPC_HANDLE_BYTES);
    if (world_size == 1) {
        ex->connected = true;
        std::lock_guard<std::mutex> lock(g_exchange_mutex);
        g_exchanges.push_back(ex);
    }
    *out = ex;
    return MGD_OK;
}

int mgd_exchange_connect(mgd_exchange* ex, const unsigned char* handles)
{
    if (!ex || !handles) return fail(MGD_ERR_INVALID_ARGUMENT, "NULL argument");
    if (ex->connected) return MGD_OK;
    int num_sms;
    DeviceScope dev_scope;
    int rc = prepare_device(ex->device, &num_sms, &dev_scope);
    if (rc) return rc;
    for (int r = 0; r < ex->world; ++r) {
        if (r == ex->rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + (size_t)r * MGD_IPC_HANDLE_BYTES, MGD_IPC_HANDLE_BYTES);
        void* p = nullptr;
        const cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            for (int q = 0; q < r; ++q)
                if (q != ex->rank && ex->alloc[q]) { cudaIpcCloseMemHandle(ex->alloc[q]); ex->alloc[q] = nullptr; }
            cudaGetLastError();
            return fail(MGD_ERR_CUDA, "cannot map the exchange buffer of rank %d: %s (peer access over "
                        "NVLink / PCIe between the two devices is required)", r, cudaGetErrorString(e));
        }
        ex->alloc[r] = static_cast<char*>(p);
    }
    ex->connected = true;
    std::lock_guard<std::mutex> lock(g_exchange_mutex);
    g_exchanges.push_back(ex);
    return MGD_OK;
}

int mgd_exchange_buffer(mgd_exchange* ex, void** base, size_t* bytes)
{
    if (!ex || !base) return fail(MGD_ERR_INVALID_ARGUMENT, "NULL argument");
    *base = ex->alloc[ex->rank] + MGD_EXCHANGE_HEADER_BYTES;
    if (bytes) *bytes = ex->bytes;
    return MGD_OK;
}

int mgd_exchange_timeouts(mgd_exchange* ex, void* stream, int* timeouts)
{
    if (!ex || !timeouts) return fail(MGD_ERR_INVALID_ARGUMENT, "NULL argument");
    int num_sms;
    DeviceScope dev_scope;
    int rc = prepare_device(ex->device, &num_sms, &dev_scope);
    if (rc) return rc;
    unsigned v = 0;
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    CUDA_TRY(cudaMemcpy(&v, reinterpret_cast<unsigned*>(ex->alloc[ex->rank]) + MGD_EXCHANGE_TIMEOUT_WORD,
                        sizeof(v), cudaMemcpyDeviceToHost));
    *timeouts = (int)v;
    return MGD_OK;
}

int mgd_exchange_destroy(mgd_exchange* ex)
{
    if (!ex) return MGD_OK;
    {
        std::lock_guard<std::mutex> lock(g_exchange_mutex);
        for (size_t i = 0; i < g_exchanges.size(); ++i)
            if (g_exchanges[i] == ex) { g_exchanges.erase(g_exchanges.begin() + i); break; }
    }
    int num_sms;
    DeviceScope dev_scope;
    if (prepare_device(ex->device, &num_sms, &dev_scope) == MGD_OK) {
        cudaDeviceSynchronize();
        for (int r = 0; r < ex->world; ++r) {
            if (!ex->alloc[r]) continue;
            if (r == ex->rank) cudaFree(ex->alloc[r]);
            else cudaIpcCloseMemHandle(ex->alloc[r]);
        }
        cudaGetLastError();
    }
    delete ex;
    return MGD_OK;
}

int mgd_release_workspace(void)
{
    // staging arenas of the calling thread (host-memory entry points), all devices
    int cur = 0;
    const bool have = cudaGetDevice(&cur) == cudaSuccess;
    for (int d = 0; d < 64; ++d) {
        HostStreams& hs = t_streams[d];
        if (hs.chunk[0].blocks.empty() && hs.chunk[1].blocks.empty() && hs.call.blocks.empty() &&
            hs.map.blocks.empty() && !hs.bounce[0] && !hs.bounce[1]) continue;
        if (cudaSetDevice(d) != cudaSuccess) { cudaGetLastError(); continue; }
        for (int i = 0; i < 2; ++i) if (hs.s[i]) cudaStreamSynchronize(hs.s[i]);
        if (hs.map_done) cudaEventSynchronize(hs.map_done);
        hs.chunk[0].release(); hs.chunk[1].release(); hs.call.release(); hs.map.release();
        for (int i = 0; i < 2; ++i) {
            if (hs.bounce[i]) cudaFreeHost(hs.bounce[i]);
            hs.bounce[i] = nullptr; hs.bounce_cap[i] = 0; hs.bounce_busy[i] = false;
        }
    }
    if (have) cudaSetDevice(cur);
    cudaGetLastError();
    return MGD_OK;
}

int mgd_profile_begin(void)
{
    for (ProfSpan& s : t_prof_spans) { cudaEventDestroy(s.t0); cudaEventDestroy(s.t1); }
    t_prof_spans.clear();
    t_prof_on = true;
    return MGD_OK;
}

int mgd_profile_end(double* ms, long long* launches)
{
    t_prof_on = false;
    for (int k = 0; k < PROF_KINDS; ++k) { if (ms) ms[k] = 0.0; if (launches) launches[k] = 0; }
    int rc = MGD_OK;
    for (ProfSpan& s : t_prof_spans) {
        float t = 0.f;
        cudaError_t e = cudaEventSynchronize(s.t1);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&t, s.t0, s.t1);
        if (e != cudaSuccess) rc = fail(MGD_ERR_CUDA, "profile: %s", cudaGetErrorString(e));
        else { if (ms) ms[s.kind] += t; if (launches) launches[s.kind] += s.launches; }
        cudaEventDestroy(s.t0);
        cudaEventDestroy(s.t1);
    }
    t_prof_spans.clear();
    return rc;
}

int mgd_poll_status(int device, void* stream)
{
    int num_sms;
    DeviceScope dev_scope;
    int rc = prepare_device(device, &num_sms, &dev_scope);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    int st = 0;
    if (t_deferred.word[device]) {
        CUDA_TRY(cudaMemcpy(&st, t_deferred.word[device], sizeof(int), cudaMemcpyDeviceToHost));
        if (st) CUDA_TRY(cudaMemset(t_deferred.word[device], 0, sizeof(int)));
    }
    return status_to_error(st);
}

int mgd_encode_targets(const mgd_head_config* cfg, const float* boxes, int batch, int max_boxes,
                       float* const* y_true, int memory, int device, void* stream, int flags,
                       long long* stats)
{
    nvtx_range nv_api("mgd_encode_targets");
    HeadGeom g;
    int rc = build_geom(cfg, &g);
    if (rc) return rc;
    if ((rc = check_memory_arg(memory))) return rc;
    if (batch < 0 || max_boxes < 0)
        return fail(MGD_ERR_INVALID_ARGUMENT, "batch and max_boxes must be >= 0");
    if (!y_true) return fail(MGD_ERR_INVALID_ARGUMENT, "y_true is NULL");
    for (int l = 0; l < g.L; ++l)
        if (!y_true[l] && batch > 0) return fail(MGD_ERR_INVALID_ARGUMENT, "y_true[%d] is NULL", l);
    if (!boxes && (long long)batch * max_boxes > 0)
        return fail(MGD_ERR_INVALID_ARGUMENT, "boxes is NULL");
    if (max_boxes > 65000)
        return fail(MGD_ERR_UNSUPPORTED, "max_boxes per image must be <= 65000, got %d", max_boxes);
    if ((long long)chunk_images(g, batch > 0 ? batch : 1) * max_boxes >= (1ll << 27))
        return fail(MGD_ERR_UNSUPPORTED, "batch chunk x max_boxes too large");
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    if (stats) memset(stats, 0, 4 * sizeof(long long));
    if (batch == 0) return MGD_OK;

    if (memory == MGD_MEM_DEVICE && !(flags & MGD_FLAG_SYNC)) {
        // asynchronous: status bits go to the thread's persistent word (mgd_poll_status)
        cudaStream_t st = (cudaStream_t)stream;
        int* d_flag;
        if ((rc = deferred_status_word(device, &d_flag))) return rc;
        return encode_device(g, boxes, batch, max_boxes, y_true, num_sms, st, d_flag, nullptr,
                             Alloc{nullptr, st}, (flags & MGD_FLAG_TF_COMPAT) != 0);
    }
    if (memory == MGD_MEM_DEVICE) {
        cudaStream_t st = (cudaStream_t)stream;
        int* d_status;
        unsigned long long* d_stats = nullptr;
        CUDA_TRY(pool_malloc(&d_status, sizeof(int) + 4 * sizeof(unsigned long long), st));
        CUDA_TRY(cudaMemsetAsync(d_status, 0, sizeof(int) + 4 * sizeof(unsigned long long), st));
        // keep the 8-byte counters aligned: status word sits after them
        d_stats = reinterpret_cast<unsigned long long*>(d_status);
        int* d_flag = reinterpret_cast<int*>(d_stats + 4);
        rc = encode_device(g, boxes, batch, max_boxes, y_true, num_sms, st, d_flag, d_stats,
                           Alloc{nullptr, st}, (flags & MGD_FLAG_TF_COMPAT) != 0);
        if (rc) return rc;
        if (flags & MGD_FLAG_SYNC) {
            unsigned long long h[5] = {0, 0, 0, 0, 0};
            CUDA_TRY(cudaMemcpyAsync(h, d_status, sizeof(int) + 4 * sizeof(unsigned long long),
                                     cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaFreeAsync(d_status, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            if (stats) for (int i = 0; i < 4; ++i) stats[i] = (long long)h[i];
            return status_to_error((int)(h[4] & 0xffffffffu));
        }
        CUDA_TRY(cudaFreeAsync(d_status, st));
        return MGD_OK;
    }

    // host memory: stage through the GPU in chunks, two streams so that the D2H of one
    // chunk overlaps the kernels of the next.  The (small) box tensor goes up once, ahead
    // of the chunks, so no chunk waits on the H2D engine behind another call's bulk copy.
    Tracer tr("encode/host");
    cudaStream_t* ss;
    cudaEvent_t* ev;
    HostStreams* hs;
    if ((rc = host_streams(device, &ss, &ev, &hs))) return rc;
    hs->call.reset();
    unsigned long long* d_meta;      // [4 stats][status]
    CUDA_TRY(hs->call.take(reinterpret_cast<void**>(&d_meta), 5 * sizeof(unsigned long long)));
    CUDA_TRY(cudaMemsetAsync(d_meta, 0, 5 * sizeof(unsigned long long), ss[0]));
    float* d_boxes;
    const size_t box_bytes = (size_t)batch * max_boxes * 5 * sizeof(float);
    CUDA_TRY(hs->call.take(reinterpret_cast<void**>(&d_boxes), box_bytes));
    if (box_bytes) CUDA_TRY(cudaMemcpyAsync(d_boxes, boxes, box_bytes, cudaMemcpyHostToDevice, ss[0]));
    CUDA_TRY(cudaEventRecord(ev[0], ss[0]));
    CUDA_TRY(cudaStreamWaitEvent(ss[1], ev[0], 0));
    int step = host_chunk(g, batch);
    float* z_y[MGD_MAX_LAYERS];
    bool zero_copy = (zerocopy_mode() & 2) != 0 || (flags & MGD_FLAG_HOST_ZEROCOPY) != 0;
    for (int l = 0; l < g.L && zero_copy; ++l) {
        z_y[l] = mapped_alias(y_true[l], (size_t)batch * g.gh[l] * g.gw[l] * g.D[l] * 4);
        zero_copy = z_y[l] != nullptr;
    }
    if (zero_copy) step = batch;
    // pageable y_true (the caller's own unpinned arrays): D2H into page-locked bounce chunks,
    // then several threads copy a finished chunk out while the next one is on the link
    bool pageable = !zero_copy && host_copy_threads() > 1 &&
                    (size_t)batch * g.cells * g.D[0] * 4 >= (32u << 20);
    for (int l = 0; l < g.L && pageable; ++l) pageable = is_pageable(y_true[l]);
    struct CopyOut { bool live = false; size_t off[MGD_MAX_LAYERS], bytes[MGD_MAX_LAYERS]; float* dst[MGD_MAX_LAYERS]; };
    CopyOut pending[2];
    auto drain = [&](int slot) -> int {
        CopyOut& c = pending[slot];
        if (!c.live) return MGD_OK;
        CUDA_TRY(cudaEventSynchronize(hs->bounce_done[slot]));
        hs->bounce_busy[slot] = false;
        for (int l = 0; l < g.L; ++l) parallel_copy(c.dst[l], hs->bounce[slot] + c.off[l], c.bytes[l]);
        c.live = false;
        return MGD_OK;
    };
    int k = 0;
    for (int b0 = 0; b0 < batch; b0 += step, ++k) {
        const int nb = batch - b0 < step ? batch - b0 : step;
        cudaStream_t st = ss[k & 1];
        Arena& ar = hs->chunk[k & 1];
        ar.reset();
        float* d_y[MGD_MAX_LAYERS];
        for (int l = 0; l < g.L; ++l) {
            if (zero_copy) d_y[l] = z_y[l];
            else CUDA_TRY(ar.take(reinterpret_cast<void**>(&d_y[l]), (size_t)nb * g.gh[l] * g.gw[l] * g.D[l] * 4));
        }
        rc = encode_device(g, d_boxes + (size_t)b0 * max_boxes * 5, nb, max_boxes, d_y, num_sms, st,
                           reinterpret_cast<int*>(d_meta + 4), d_meta, Alloc{&ar, st},
                           (flags & MGD_FLAG_TF_COMPAT) != 0);
        if (rc) return rc;
        unsigned char* bounce = nullptr;
        if (pageable) {
            if ((rc = drain(k & 1))) return rc;
            size_t need = 0;
            for (int l = 0; l < g.L; ++l) need += (((size_t)nb * g.gh[l] * g.gw[l] * g.D[l] * 4) + 255) & ~(size_t)255;
            if ((rc = bounce_slot(hs, k & 1, need, &bounce))) return rc;
        }
        size_t bounce_off = 0;
        for (int l = 0; l < g.L && !zero_copy; ++l) {
            const size_t per = (size_t)g.gh[l] * g.gw[l] * g.D[l];
            const size_t bytes = (size_t)nb * per * 4;
            float* dst = y_true[l] + (size_t)b0 * per;
            if (bounce) {
                CopyOut& c = pending[k & 1];
                c.off[l] = bounce_off; c.bytes[l] = bytes; c.dst[l] = dst;
                dst = reinterpret_cast<float*>(bounce + bounce_off);
                bounce_off += (bytes + 255) & ~(size_t)255;
            }
            CUDA_TRY(cudaMemcpyAsync(dst, d_y[l], bytes, cudaMemcpyDeviceToHost, st));
        }
        if (bounce) {
            CUDA_TRY(cudaEventRecord(hs->bounce_done[k & 1], st));
            hs->bounce_busy[k & 1] = true;
            pending[k & 1].live = true;
        }
    }
    if (pageable) {
        if ((rc = drain(k & 1))) return rc;           // the older of the two chunks in flight first
        if ((rc = drain((k + 1) & 1))) return rc;
    }
    tr.mark("chunks enqueued");
    CUDA_TRY(cudaEventRecord(ev[1], ss[1]));
    CUDA_TRY(cudaStreamWaitEvent(ss[0], ev[1], 0));
    // drain first, read back after: a copy into pageable memory (this stack word, or the
    // caller's unpinned arrays) waits for the stream INSIDE the driver, and other host
    // threads' launches stall behind it for the whole transfer
    CUDA_TRY(cudaStreamSynchronize(ss[0]));
    unsigned long long h[5];
    CUDA_TRY(cudaMemcpy(h, d_meta, sizeof(h), cudaMemcpyDeviceToHost));
    tr.mark("synchronised");
    hs->chunk[0].consolidate(); hs->chunk[1].consolidate(); hs->call.consolidate();
    if (stats) for (int i = 0; i < 4; ++i) stats[i] = (long long)h[i];
    return status_to_error((int)(h[4] & 0xffffffffu));
}

int mgd_decode_nms(const mgd_head_config* cfg, const mgd_post_config* post,
                   const float* const* preds, int batch, const int* image_hw,
                   double* boxes_xywh, int* boxes_xyxy, double* scores, int* classes, int* index,
                   int* counts, int memory, int device, void* stream, int flags, long long* stats)
{
    nvtx_range nv_api("mgd_decode_nms");
    HeadGeom g;
    int rc = build_geom(cfg, &g);
    if (rc) return rc;
    if ((rc = check_post(post))) return rc;
    if ((rc = check_memory_arg(memory))) return rc;
    if (batch < 0) return fail(MGD_ERR_INVALID_ARGUMENT, "batch must be >= 0");
    if (!preds) return fail(MGD_ERR_INVALID_ARGUMENT, "preds is NULL");
    for (int l = 0; l < g.L; ++l)
        if (!preds[l] && batch > 0) return fail(MGD_ERR_INVALID_ARGUMENT, "preds[%d] is NULL", l);
    if (!counts && batch > 0) return fail(MGD_ERR_INVALID_ARGUMENT, "counts is NULL");
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    if (stats) memset(stats, 0, 4 * sizeof(long long));
    if (batch == 0) return MGD_OK;
    const int M = post->max_boxes;

    if (memory == MGD_MEM_DEVICE) {
        cudaStream_t st = (cudaStream_t)stream;
        unsigned long long* d_stats = nullptr;
        const bool want_stats = stats && (flags & MGD_FLAG_SYNC);
        if (want_stats) {
            CUDA_TRY(pool_malloc(&d_stats, 4 * sizeof(unsigned long long), st));
            CUDA_TRY(cudaMemsetAsync(d_stats, 0, 4 * sizeof(unsigned long long), st));
        }
        rc = decode_nms_device(g, *post, preds, batch, image_hw, boxes_xywh, boxes_xyxy, scores,
                               classes, index, counts, num_sms, st, d_stats, Alloc{nullptr, st});
        if (rc) return rc;
        if (flags & MGD_FLAG_SYNC) {
            unsigned long long h[4] = {0, 0, 0, 0};
            if (want_stats) {
                CUDA_TRY(cudaMemcpyAsync(h, d_stats, sizeof(h), cudaMemcpyDeviceToHost, st));
                CUDA_TRY(cudaFreeAsync(d_stats, st));
            }
            CUDA_TRY(cudaStreamSynchronize(st));
            if (stats) for (int i = 0; i < 4; ++i) stats[i] = (long long)h[i];
        }
        return MGD_OK;
    }

    // host memory: predictions go up in chunks on two streams (H2D of one chunk overlaps the
    // kernels of the previous one); image shapes go up once ahead of the chunks and all
    // detections come back in one slab at the end, so the small copies never queue behind
    // another call's bulk transfer more than once.
    Tracer tr("decode_nms/host");
    cudaStream_t* ss;
    cudaEvent_t* ev;
    HostStreams* hs;
    if ((rc = host_streams(device, &ss, &ev, &hs))) return rc;
    tr.mark("streams");
    // one output slab: stats u64[4] | xywh f64 | scores f64 | xyxy i32 | classes i32 | index i32 | counts i32 | hw i32
    const size_t n_det = (size_t)batch * M;
    const size_t off_xywh = 4 * sizeof(unsigned long long);
    const size_t off_scores = off_xywh + n_det * 4 * sizeof(double);
    const size_t off_xyxy = off_scores + n_det * sizeof(double);
    const size_t off_cls = off_xyxy + n_det * 4 * sizeof(int);
    const size_t off_idx = off_cls + n_det * sizeof(int);
    const size_t off_cnt = off_idx + n_det * sizeof(int);
    const size_t off_hw = off_cnt + (size_t)batch * sizeof(int);
    const size_t slab = off_hw + (size_t)batch * 2 * sizeof(int);
    unsigned char* d_out;
    hs->call.reset();
    CUDA_TRY(hs->call.take(reinterpret_cast<void**>(&d_out), slab));
    unsigned long long* d_stats = reinterpret_cast<unsigned long long*>(d_out);
    CUDA_TRY(cudaMemsetAsync(d_stats, 0, 4 * sizeof(unsigned long long), ss[0]));
    int* d_hw = nullptr;
    if (image_hw) {
        d_hw = reinterpret_cast<int*>(d_out + off_hw);
        CUDA_TRY(cudaMemcpyAsync(d_hw, image_hw, (size_t)batch * 2 * sizeof(int), cudaMemcpyHostToDevice, ss[0]));
    }
    CUDA_TRY(cudaEventRecord(ev[0], ss[0]));
    CUDA_TRY(cudaStreamWaitEvent(ss[1], ev[0], 0));
    tr.mark("slab");
    int step = host_chunk(g, batch);
    // pinned predictions: the decode kernel can read them in place
    const float* z_pred[MGD_MAX_LAYERS];
    bool zero_copy = (zerocopy_mode() & 1) != 0 || (flags & MGD_FLAG_HOST_ZEROCOPY) != 0;
    for (int l = 0; l < g.L && zero_copy; ++l) {
        z_pred[l] = mapped_alias(preds[l], (size_t)batch * g.gh[l] * g.gw[l] * g.D[l] * 4);
        zero_copy = z_pred[l] != nullptr;
    }
    // (still chunked: kernels of other calls get onto the SMs between the chunks)
    // pageable predictions: bounce through page-locked chunks filled by several threads
    bool pageable = !zero_copy && host_copy_threads() > 1 &&
                    (size_t)batch * g.cells * g.D[0] * 4 >= (32u << 20);
    for (int l = 0; l < g.L && pageable; ++l) pageable = is_pageable(preds[l]);
    int k = 0;
    for (int b0 = 0; b0 < batch; b0 += step, ++k) {
        const int nb = batch - b0 < step ? batch - b0 : step;
        cudaStream_t st = ss[k & 1];
        Arena& ar = hs->chunk[k & 1];
        ar.reset();
        float* d_pred[MGD_MAX_LAYERS];
        unsigned char* bounce = nullptr;
        size_t bounce_off = 0;
        if (pageable) {
            size_t need = 0;
            for (int l = 0; l < g.L; ++l) need += (((size_t)nb * g.gh[l] * g.gw[l] * g.D[l] * 4) + 255) & ~(size_t)255;
            if ((rc = bounce_slot(hs, k & 1, need, &bounce))) return rc;
        }
        for (int l = 0; l < g.L; ++l) {
            const size_t per = (size_t)g.gh[l] * g.gw[l] * g.D[l];
            if (zero_copy) { d_pred[l] = const_cast<float*>(z_pred[l]) + (size_t)b0 * per; continue; }
            const size_t bytes = (size_t)nb * per * 4;
            CUDA_TRY(ar.take(reinterpret_cast<void**>(&d_pred[l]), bytes));
            const void* src = preds[l] + (size_t)b0 * per;
            if (bounce) {
                parallel_copy(bounce + bounce_off, src, bytes);
                src = bounce + bounce_off;
                bounce_off += (bytes + 255) & ~(size_t)255;
            }
            CUDA_TRY(cudaMemcpyAsync(d_pred[l], src, bytes, cudaMemcpyHostToDevice, st));
        }
        if (bounce) {
            CUDA_TRY(cudaEventRecord(hs->bounce_done[k & 1], st));
            hs->bounce_busy[k & 1] = true;
        }
        rc = decode_nms_device(g, *post, d_pred, nb, d_hw ? d_hw + 2 * (size_t)b0 : nullptr,
                               reinterpret_cast<double*>(d_out + off_xywh) + (size_t)b0 * M * 4,
                               reinterpret_cast<int*>(d_out + off_xyxy) + (size_t)b0 * M * 4,
                               reinterpret_cast<double*>(d_out + off_scores) + (size_t)b0 * M,
                               reinterpret_cast<int*>(d_out + off_cls) + (size_t)b0 * M,
                               reinterpret_cast<int*>(d_out + off_idx) + (size_t)b0 * M,
                               reinterpret_cast<int*>(d_out + off_cnt) + b0, num_sms, st, d_stats,
                               Alloc{&ar, st});
        if (rc) return rc;
    }
    tr.mark("chunks enqueued");
    CUDA_TRY(cudaEventRecord(ev[1], ss[1]));
    CUDA_TRY(cudaStreamWaitEvent(ss[0], ev[1], 0));
    cudaStream_t st = ss[0];
    // drain first, read back after (see mgd_encode_targets): the detection arrays are
    // usually pageable, and a pageable copy that has to wait for the stream blocks the
    // launches of every other host thread meanwhile
    CUDA_TRY(cudaStreamSynchronize(st));
    unsigned long long h[4];
    CUDA_TRY(cudaMemcpyAsync(h, d_stats, sizeof(h), cudaMemcpyDeviceToHost, st));
    if (boxes_xywh)
        CUDA_TRY(cudaMemcpyAsync(boxes_xywh, d_out + off_xywh, n_det * 4 * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (scores)
        CUDA_TRY(cudaMemcpyAsync(scores, d_out + off_scores, n_det * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (boxes_xyxy)
        CUDA_TRY(cudaMemcpyAsync(boxes_xyxy, d_out + off_xyxy, n_det * 4 * sizeof(int), cudaMemcpyDeviceToHost, st));
    if (classes)
        CUDA_TRY(cudaMemcpyAsync(classes, d_out + off_cls, n_det * sizeof(int), cudaMemcpyDeviceToHost, st));
    if (index)
        CUDA_TRY(cudaMemcpyAsync(index, d_out + off_idx, n_det * sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(counts, d_out + off_cnt, (size_t)batch * sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    tr.mark("synchronised");
    hs->chunk[0].consolidate(); hs->chunk[1].consolidate(); hs->call.consolidate();
    if (stats) for (int i = 0; i < 4; ++i) stats[i] = (long long)h[i];
    return MGD_OK;
}

// side stream + fork / join events of the fused entry, one set per (host thread, device)
struct ForkStreams {
    cudaStream_t side = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
    ~ForkStreams()
    {
        if (fork) cudaEventDestroy(fork);
        if (join) cudaEventDestroy(join);
        if (side) cudaStreamDestroy(side);
        cudaGetLastError();
    }
};
thread_local ForkStreams t_fork[64];

int mgd_encode_decode_nms(const mgd_head_config* cfg, const mgd_post_config* post,
                          const float* gt_boxes, int enc_batch, int max_gt_boxes,
                          float* const* y_true,
                          const float* const* preds, int dec_batch, const int* image_hw,
                          double* boxes_xywh, int* boxes_xyxy, double* scores,
                          int* classes, int* index, int* counts,
                          int device, void* stream, int flags)
{
    nvtx_range nv_api("mgd_encode_decode_nms");
    HeadGeom g;
    int rc = build_geom(cfg, &g);
    if (rc) return rc;
    if ((rc = check_post(post))) return rc;
    if (enc_batch < 0 || dec_batch < 0 || max_gt_boxes < 0)
        return fail(MGD_ERR_INVALID_ARGUMENT, "batch sizes and max_gt_boxes must be >= 0");
    if (enc_batch > 0) {
        if (!y_true) return fail(MGD_ERR_INVALID_ARGUMENT, "y_true is NULL");
        for (int l = 0; l < g.L; ++l)
            if (!y_true[l]) return fail(MGD_ERR_INVALID_ARGUMENT, "y_true[%d] is NULL", l);
        if (!gt_boxes && max_gt_boxes > 0) return fail(MGD_ERR_INVALID_ARGUMENT, "gt_boxes is NULL");
        if (max_gt_boxes > 65000)
            return fail(MGD_ERR_UNSUPPORTED, "max_boxes per image must be <= 65000, got %d", max_gt_boxes);
        if ((long long)chunk_images(g, enc_batch) * max_gt_boxes >= (1ll << 27))
            return fail(MGD_ERR_UNSUPPORTED, "batch chunk x max_boxes too large");
    }
    if (dec_batch > 0) {
        if (!preds) return fail(MGD_ERR_INVALID_ARGUMENT, "preds is NULL");
        for (int l = 0; l < g.L; ++l)
            if (!preds[l]) return fail(MGD_ERR_INVALID_ARGUMENT, "preds[%d] is NULL", l);
        if (!counts) return fail(MGD_ERR_INVALID_ARGUMENT, "counts is NULL");
    }
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    ForkStreams& fk = t_fork[device];
    if (!fk.side) {
        // lowest priority: decode / NMS blocks are placed first, the writer takes what is left
        int lo = 0, hi = 0;
        CUDA_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        const char* pe = getenv("MGD_STEP_PRIORITY");          // measurements: -1 low, 0 default, 1 high
        const int want = pe ? atoi(pe) : -1;
        CUDA_TRY(cudaStreamCreateWithPriority(&fk.side, cudaStreamNonBlocking, want < 0 ? lo : (want > 0 ? hi : 0)));
        CUDA_TRY(cudaEventCreateWithFlags(&fk.fork, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&fk.join, cudaEventDisableTiming));
    }
    std::vector<EncodeArgs> chunks;
    if (enc_batch > 0) {
        int* d_flag;
        if ((rc = deferred_status_word(device, &d_flag))) return rc;
        rc = encode_assign_all(g, gt_boxes, enc_batch, max_gt_boxes, y_true, st, d_flag,
                               (flags & MGD_FLAG_TF_COMPAT) != 0, &chunks);
        if (rc) { encode_free_all(chunks, st); return rc; }
    }
    if (dec_batch == 0) {
        rc = encode_fill_all(chunks, num_sms, st);
        encode_free_all(chunks, st);
        if (rc) return rc;
        if (flags & MGD_FLAG_SYNC) CUDA_TRY(cudaStreamSynchronize(st));
        return MGD_OK;
    }
    bool forked = false;
    const std::function<int()> fork_writer = [&]() -> int {
        if (chunks.empty()) return MGD_OK;
        CUDA_TRY(cudaEventRecord(fk.fork, st));                  // behind the assigns and the decoder
        CUDA_TRY(cudaStreamWaitEvent(fk.side, fk.fork, 0));
        forked = true;
        const int frc = encode_fill_all(chunks, num_sms, fk.side);
        CUDA_TRY(cudaEventRecord(fk.join, fk.side));
        return frc;
    };
    rc = decode_nms_device(g, *post, preds, dec_batch, image_hw, boxes_xywh, boxes_xyxy, scores,
                           classes, index, counts, num_sms, st, nullptr, Alloc{nullptr, st}, &fork_writer);
    if (forked) {
        const cudaError_t e = cudaStreamWaitEvent(st, fk.join, 0);
        if (e != cudaSuccess && rc == MGD_OK) rc = fail(MGD_ERR_CUDA, "join failed: %s", cudaGetErrorString(e));
    }
    encode_free_all(chunks, st);                                 // st is behind the writer now
    if (rc) return rc;
    if (flags & MGD_FLAG_SYNC) CUDA_TRY(cudaStreamSynchronize(st));
    return MGD_OK;
}

int mgd_decode_dense(const mgd_head_config* cfg, const mgd_post_config* post,
                     const float* const* preds, int batch, const int* image_hw, double* out,
                     int memory, int device, void* stream, int flags)
{
    nvtx_range nv_api("mgd_decode_dense");
    HeadGeom g;
    int rc = build_geom(cfg, &g);
    if (rc) return rc;
    if (!post) return fail(MGD_ERR_INVALID_ARGUMENT, "post config is NULL");
    if ((rc = check_memory_arg(memory))) return rc;
    if (batch < 0) return fail(MGD_ERR_INVALID_ARGUMENT, "batch must be >= 0");
    if (batch > 0 && (!preds || !out)) return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor");
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    if (batch == 0) return MGD_OK;
    DecodeArgs d;
    memset(&d, 0, sizeof(d));
    d.g = g;
    d.use_softmax = post->use_softmax;
    d.rescore = post->rescore_confidence;
    const size_t out_per = (size_t)g.cells * (5 + g.C);
    if (memory == MGD_MEM_DEVICE) {
        cudaStream_t st = (cudaStream_t)stream;
        d.B = batch;
        for (int l = 0; l < g.L; ++l) d.pred[l] = preds[l];
        CUDA_TRY(launch_decode_dense(d, image_hw, out, st));
        if (flags & MGD_FLAG_SYNC) CUDA_TRY(cudaStreamSynchronize(st));
        return MGD_OK;
    }
    cudaStream_t* ss;
    if ((rc = host_streams(device, &ss, nullptr))) return rc;
    cudaStream_t st = ss[0];
    long long per_image = (long long)out_per * 8;
    int step = (int)((512ll << 20) / per_image);
    if (step < 1) step = 1;
    for (int b0 = 0; b0 < batch; b0 += step) {
        const int nb = batch - b0 < step ? batch - b0 : step;
        float* d_pred[MGD_MAX_LAYERS];
        d.B = nb;
        for (int l = 0; l < g.L; ++l) {
            const size_t per = (size_t)g.gh[l] * g.gw[l] * g.D[l];
            CUDA_TRY(pool_malloc(&d_pred[l], (size_t)nb * per * 4, st));
            CUDA_TRY(cudaMemcpyAsync(d_pred[l], preds[l] + (size_t)b0 * per, (size_t)nb * per * 4,
                                     cudaMemcpyHostToDevice, st));
            d.pred[l] = d_pred[l];
        }
        int* d_hw = nullptr;
        if (image_hw) {
            CUDA_TRY(pool_malloc(&d_hw, (size_t)nb * 2 * sizeof(int), st));
            CUDA_TRY(cudaMemcpyAsync(d_hw, image_hw + 2 * (size_t)b0, (size_t)nb * 2 * sizeof(int),
                                     cudaMemcpyHostToDevice, st));
        }
        double* d_out;
        CUDA_TRY(pool_malloc(&d_out, (size_t)nb * out_per * 8, st));
        CUDA_TRY(launch_decode_dense(d, d_hw, d_out, st));
        CUDA_TRY(cudaMemcpyAsync(out + (size_t)b0 * out_per, d_out, (size_t)nb * out_per * 8,
                                 cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaFreeAsync(d_out, st));
        if (d_hw) CUDA_TRY(cudaFreeAsync(d_hw, st));
        for (int l = 0; l < g.L; ++l) CUDA_TRY(cudaFreeAsync(d_pred[l], st));
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    return MGD_OK;
}

int mgd_nms(const double* boxes, const double* scores, const int* classes, int n,
            double nms_threshold, int nms_method, int per_class, int max_keep, int* keep,
            int* n_keep, int memory, int device, void* stream, int flags)
{
    nvtx_range nv_api("mgd_nms");
    int rc;
    if ((rc = check_memory_arg(memory))) return rc;
    if (n < 0) return fail(MGD_ERR_INVALID_ARGUMENT, "n must be >= 0");
    if (nms_method != MGD_NMS_IOU && nms_method != MGD_NMS_DIOU)
        return fail(MGD_ERR_UNSUPPORTED, "nms_method %d not built", nms_method);
    if (!n_keep) return fail(MGD_ERR_INVALID_ARGUMENT, "n_keep is NULL");
    if (n > 0 && (!boxes || !scores || !keep)) return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor");
    if (max_keep <= 0 || max_keep > n) max_keep = n;
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    const bool host = memory == MGD_MEM_HOST;
    cudaStream_t st = (cudaStream_t)stream;
    if (host) {
        cudaStream_t* ss;
        if ((rc = host_streams(device, &ss, nullptr))) return rc;
        st = ss[0];
    }
    if (n == 0) {
        if (host) { *n_keep = 0; return MGD_OK; }
        CUDA_TRY(cudaMemsetAsync(n_keep, 0, sizeof(int), st));
        if (flags & MGD_FLAG_SYNC) CUDA_TRY(cudaStreamSynchronize(st));
        return MGD_OK;
    }
    const double* d_boxes = boxes; const double* d_scores = scores; const int* d_classes = classes;
    int* d_keep = keep; int* d_nkeep = n_keep;
    void* staged = nullptr;
    if (host) {
        const size_t bytes = (size_t)n * (4 * 8 + 8 + 4 + 4) + 16;
        CUDA_TRY(pool_malloc(&staged, bytes, st));
        double* p = reinterpret_cast<double*>(staged);
        CUDA_TRY(cudaMemcpyAsync(p, boxes, (size_t)n * 32, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(p + 4 * (size_t)n, scores, (size_t)n * 8, cudaMemcpyHostToDevice, st));
        int* q = reinterpret_cast<int*>(p + 5 * (size_t)n);
        if (classes) CUDA_TRY(cudaMemcpyAsync(q, classes, (size_t)n * 4, cudaMemcpyHostToDevice, st));
        d_boxes = p; d_scores = p + 4 * (size_t)n; d_classes = classes ? q : nullptr;
        d_keep = q + n; d_nkeep = q + 2 * (size_t)n;
    }
    int* count; int* d_index; int* d_counts;
    CUDA_TRY(pool_malloc(&count, 2 * sizeof(int) + (size_t)max_keep * sizeof(int), st));
    d_counts = count + 1;
    d_index = count + 2;
    CUDA_TRY(cudaMemcpyAsync(count, &n, sizeof(int), cudaMemcpyHostToDevice, st));
    NmsArgs a;
    memset(&a, 0, sizeof(a));
    a.B = 1; a.cap = n; a.counts = count;
    a.in_boxes = d_boxes; a.in_scores = d_scores; a.in_classes = d_classes;
    a.thr = nms_threshold; a.use_diou = nms_method == MGD_NMS_DIOU; a.per_class = per_class;
    a.max_boxes = max_keep;
    int pow2 = 2;
    while (pow2 < n) pow2 <<= 1;
    if (n > nms_smem_capacity()) {
        a.sort_scratch_stride = pow2;
        CUDA_TRY(pool_malloc(&a.sort_scratch, (size_t)2 * pow2 * sizeof(unsigned long long), st));
    }
    if (nms_kept_bytes(max_keep) > 64 * 1024) {
        a.kept_scratch_stride = (nms_kept_bytes(max_keep) + 15) & ~(size_t)15;
        CUDA_TRY(pool_malloc(&a.kept_scratch, a.kept_scratch_stride, st));
    }
    a.out_index = d_index;
    a.out_counts = d_counts;
    CUDA_TRY(launch_nms(a, num_sms, st));
    CUDA_TRY(launch_keep_from_index(d_index, d_counts, max_keep, d_keep, d_nkeep, st));
    if (host) {
        CUDA_TRY(cudaMemcpyAsync(n_keep, d_nkeep, sizeof(int), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(keep, d_keep, (size_t)max_keep * sizeof(int), cudaMemcpyDeviceToHost, st));
    }
    if (a.sort_scratch) CUDA_TRY(cudaFreeAsync(a.sort_scratch, st));
    if (a.kept_scratch) CUDA_TRY(cudaFreeAsync(a.kept_scratch, st));
    CUDA_TRY(cudaFreeAsync(count, st));
    if (staged) CUDA_TRY(cudaFreeAsync(staged, st));
    if (host || (flags & MGD_FLAG_SYNC)) CUDA_TRY(cudaStreamSynchronize(st));
    return MGD_OK;
}

int mgd_wbf(const double* boxes, const double* scores, const int* classes,
            const double* box_weights, int n, double iou_thr, double skip_box_thr, int conf_type,
            double* out_boxes, double* out_scores, int* out_classes, int* n_out, int memory,
            int device, void* stream, int flags)
{
    nvtx_range nv_api("mgd_wbf");
    int rc;
    if ((rc = check_memory_arg(memory))) return rc;
    if (n < 0) return fail(MGD_ERR_INVALID_ARGUMENT, "n must be >= 0");
    if (!n_out) return fail(MGD_ERR_INVALID_ARGUMENT, "n_out is NULL");
    if (n > 0 && (!boxes || !scores || !classes || !out_boxes || !out_scores || !out_classes))
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor");
    if (conf_type < 0 || conf_type > 2) return fail(MGD_ERR_INVALID_ARGUMENT, "bad conf_type");
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    const bool host = memory == MGD_MEM_HOST;
    cudaStream_t st = (cudaStream_t)stream;
    if (host) {
        cudaStream_t* ss;
        if ((rc = host_streams(device, &ss, nullptr))) return rc;
        st = ss[0];
    }
    if (n == 0) {
        if (host) { *n_out = 0; return MGD_OK; }
        CUDA_TRY(cudaMemsetAsync(n_out, 0, sizeof(int), st));
        if (flags & MGD_FLAG_SYNC) CUDA_TRY(cudaStreamSynchronize(st));
        return MGD_OK;
    }
    const size_t nn = (size_t)n;
    int pow2 = 2;
    while (pow2 < n) pow2 <<= 1;
    // staging: boxes 4n | scores n | weights n | fused 5n | out_boxes 4n | out_scores n  (f64)
    //          sort 2*pow2 (u64) | classes n | out_classes n | ints 4n | counts 2        (i32)
    unsigned char* buf;
    const size_t f64s = nn * (4 + 1 + 1 + 5 + 4 + 1);
    CUDA_TRY(pool_malloc(&buf, f64s * 8 + (size_t)2 * pow2 * 8 + nn * 6 * 4 + 64, st));
    double* d_boxes = reinterpret_cast<double*>(buf);
    double* d_scores = d_boxes + 4 * nn;
    double* d_w = d_scores + nn;
    double* d_fused = d_w + nn;
    double* d_ob = d_fused + 5 * nn;
    double* d_os = d_ob + 4 * nn;
    unsigned long long* d_sort = reinterpret_cast<unsigned long long*>(d_os + nn);
    int* d_cls = reinterpret_cast<int*>(d_sort + 2 * (size_t)pow2);
    int* d_oc = d_cls + nn;
    int* d_ints = d_oc + nn;
    int* d_cnt = d_ints + 4 * nn;
    const cudaMemcpyKind in_kind = host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    CUDA_TRY(cudaMemcpyAsync(d_boxes, boxes, nn * 32, in_kind, st));
    CUDA_TRY(cudaMemcpyAsync(d_scores, scores, nn * 8, in_kind, st));
    CUDA_TRY(cudaMemcpyAsync(d_cls, classes, nn * 4, in_kind, st));
    if (box_weights) CUDA_TRY(cudaMemcpyAsync(d_w, box_weights, nn * 8, in_kind, st));
    CUDA_TRY(cudaMemcpyAsync(d_cnt, &n, sizeof(int), cudaMemcpyHostToDevice, st));
    NmsArgs a;
    memset(&a, 0, sizeof(a));
    a.B = 1; a.cap = n; a.counts = d_cnt;
    a.in_boxes = d_boxes; a.in_scores = d_scores; a.in_classes = d_cls;
    a.in_weights = box_weights ? d_w : nullptr;
    a.max_boxes = n;
    a.wbf = 1; a.wbf_conf_type = conf_type; a.thr = iou_thr; a.soft_thr = skip_box_thr;
    a.soft_scratch = d_fused; a.wbf_ints = d_ints;
    a.sort_scratch = d_sort; a.sort_scratch_stride = pow2;
    a.out_xywh = d_ob; a.out_scores = d_os; a.out_classes = d_oc; a.out_counts = d_cnt + 1;
    CUDA_TRY(launch_nms(a, num_sms, st));
    const cudaMemcpyKind out_kind = host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    CUDA_TRY(cudaMemcpyAsync(out_boxes, d_ob, nn * 32, out_kind, st));
    CUDA_TRY(cudaMemcpyAsync(out_scores, d_os, nn * 8, out_kind, st));
    CUDA_TRY(cudaMemcpyAsync(out_classes, d_oc, nn * 4, out_kind, st));
    CUDA_TRY(cudaMemcpyAsync(n_out, d_cnt + 1, sizeof(int), out_kind, st));
    CUDA_TRY(cudaFreeAsync(buf, st));
    if (host || (flags & MGD_FLAG_SYNC)) CUDA_TRY(cudaStreamSynchronize(st));
    return MGD_OK;
}

int mgd_soft_nms(const double* boxes, const double* scores, int n, double sigma,
                 double score_threshold, int* keep, double* soft_scores, int* n_keep, int memory,
                 int device, void* stream, int flags)
{
    nvtx_range nv_api("mgd_soft_nms");
    int rc;
    if ((rc = check_memory_arg(memory))) return rc;
    if (n < 0) return fail(MGD_ERR_INVALID_ARGUMENT, "n must be >= 0");
    if (!n_keep) return fail(MGD_ERR_INVALID_ARGUMENT, "n_keep is NULL");
    if (n > 0 && (!boxes || !scores || !keep || !soft_scores))
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor");
    if (!(sigma > 0.0)) return fail(MGD_ERR_INVALID_ARGUMENT, "sigma must be positive");
    if (score_threshold != score_threshold)
        return fail(MGD_ERR_INVALID_ARGUMENT, "score_threshold is NaN");
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    const bool host = memory == MGD_MEM_HOST;
    cudaStream_t st = (cudaStream_t)stream;
    if (host) {
        cudaStream_t* ss;
        if ((rc = host_streams(device, &ss, nullptr))) return rc;
        st = ss[0];
    }
    if (n == 0) {
        if (host) { *n_keep = 0; return MGD_OK; }
        CUDA_TRY(cudaMemsetAsync(n_keep, 0, sizeof(int), st));
        if (flags & MGD_FLAG_SYNC) CUDA_TRY(cudaStreamSynchronize(st));
        return MGD_OK;
    }
    // device staging: boxes (4n f64) | scores (n f64) | soft out (n f64) | keep (n i32) | counts (2 i32)
    const size_t nn = (size_t)n;
    unsigned char* buf;
    CUDA_TRY(pool_malloc(&buf, nn * (32 + 8 + 8 + 8 + 4) + 64, st));
    double* d_boxes = reinterpret_cast<double*>(buf);
    double* d_scores = d_boxes + 4 * nn;
    double* d_soft_out = d_scores + nn;
    double* d_soft = d_soft_out + nn;
    int* d_keep = reinterpret_cast<int*>(d_soft + nn);
    int* d_cnt = d_keep + nn;
    const cudaMemcpyKind in_kind = host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    CUDA_TRY(cudaMemcpyAsync(d_boxes, boxes, nn * 32, in_kind, st));
    CUDA_TRY(cudaMemcpyAsync(d_scores, scores, nn * 8, in_kind, st));
    CUDA_TRY(cudaMemcpyAsync(d_cnt, &n, sizeof(int), cudaMemcpyHostToDevice, st));
    NmsArgs a;
    memset(&a, 0, sizeof(a));
    a.B = 1; a.cap = n; a.counts = d_cnt;
    a.in_boxes = d_boxes; a.in_scores = d_scores;
    a.max_boxes = n;
    a.soft = 1; a.soft_sigma = sigma; a.soft_thr = score_threshold; a.soft_scratch = d_soft;
    int pow2 = 2;
    while (pow2 < n) pow2 <<= 1;
    if (n > nms_smem_capacity()) {
        a.sort_scratch_stride = pow2;
        CUDA_TRY(pool_malloc(&a.sort_scratch, (size_t)2 * pow2 * sizeof(unsigned long long), st));
    }
    a.out_index = d_keep; a.out_scores = d_soft_out; a.out_counts = d_cnt + 1;
    CUDA_TRY(launch_nms(a, num_sms, st));
    const cudaMemcpyKind out_kind = host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    CUDA_TRY(cudaMemcpyAsync(keep, d_keep, nn * sizeof(int), out_kind, st));
    CUDA_TRY(cudaMemcpyAsync(soft_scores, d_soft_out, nn * sizeof(double), out_kind, st));
    CUDA_TRY(cudaMemcpyAsync(n_keep, d_cnt + 1, sizeof(int), out_kind, st));
    if (a.sort_scratch) CUDA_TRY(cudaFreeAsync(a.sort_scratch, st));
    CUDA_TRY(cudaFreeAsync(buf, st));
    if (host || (flags & MGD_FLAG_SYNC)) CUDA_TRY(cudaStreamSynchronize(st));
    return MGD_OK;
}

int mgd_match_detections(const double* det_boxes, const double* det_scores, const int* det_classes,
                         const int* det_counts, int batch, int max_dets, const double* gt_boxes,
                         const int* gt_classes, const int* gt_counts, int max_gt,
                         const double* iou_thresholds, int num_thresholds, int iou_mode,
                         unsigned char* tp, int* matched_gt, int memory, int device, void* stream,
                         int flags)
{
    nvtx_range nv_api("mgd_match_detections");
    int rc;
    if ((rc = check_memory_arg(memory))) return rc;
    if (batch < 0 || max_dets < 0 || max_gt < 0)
        return fail(MGD_ERR_INVALID_ARGUMENT, "batch, max_dets and max_gt must be >= 0");
    if (num_thresholds < 1 || num_thresholds > MGD_MAX_IOU_THRESHOLDS || !iou_thresholds)
        return fail(MGD_ERR_INVALID_ARGUMENT, "num_thresholds must be in [1, %d]", MGD_MAX_IOU_THRESHOLDS);
    if (iou_mode != MGD_IOU_CORNER && iou_mode != MGD_IOU_CENTRE)
        return fail(MGD_ERR_INVALID_ARGUMENT, "iou_mode must be MGD_IOU_CORNER or MGD_IOU_CENTRE");
    if (max_dets > 65535) return fail(MGD_ERR_UNSUPPORTED, "max_dets per image must be <= 65535");
    if ((size_t)max_dets * 2 + (size_t)max_gt / 8 > 48 * 1024)
        return fail(MGD_ERR_UNSUPPORTED, "max_dets / max_gt too large for one warp's shared memory");
    if (batch > 0 && (!det_counts || !gt_counts || !tp))
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor");
    if ((long long)batch * max_dets > 0 && (!det_boxes || !det_scores || !det_classes))
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL detection tensor");
    if ((long long)batch * max_gt > 0 && (!gt_boxes || !gt_classes))
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL ground-truth tensor");
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    if (batch == 0) return MGD_OK;
    const bool host = memory == MGD_MEM_HOST;
    cudaStream_t st = (cudaStream_t)stream;
    if (host) {
        cudaStream_t* ss;
        if ((rc = host_streams(device, &ss, nullptr))) return rc;
        st = ss[0];
    }
    MatchArgs a;
    memset(&a, 0, sizeof(a));
    a.B = batch; a.M = max_dets; a.N = max_gt; a.T = num_thresholds; a.mode = iou_mode;
    for (int t = 0; t < num_thresholds; ++t) a.thr[t] = iou_thresholds[t];
    const size_t nd = (size_t)batch * max_dets, ng = (size_t)batch * max_gt;
    const size_t n_out = (size_t)num_thresholds * nd;
    // staging (host memory) / scratch: one block, 8-byte fields first
    const size_t off_dsc = nd * 32, off_gbox = off_dsc + nd * 8, off_who = off_gbox + ng * 32;
    const size_t off_dcl = off_who + n_out * 4, off_gcl = off_dcl + nd * 4, off_dcn = off_gcl + ng * 4;
    const size_t off_gcn = off_dcn + (size_t)batch * 4, off_ctr = off_gcn + (size_t)batch * 4;
    const size_t off_tp = off_ctr + 16, total = off_tp + n_out;
    unsigned char* buf;
    CUDA_TRY(pool_malloc(&buf, host ? total : 64, st));
    int* d_ctr = reinterpret_cast<int*>(host ? buf + off_ctr : buf);
    CUDA_TRY(cudaMemsetAsync(d_ctr, 0, sizeof(int), st));
    if (host) {
        auto up = [&](size_t off, const void* src, size_t bytes) -> cudaError_t {
            return bytes ? cudaMemcpyAsync(buf + off, src, bytes, cudaMemcpyHostToDevice, st) : cudaSuccess;
        };
        CUDA_TRY(up(0, det_boxes, nd * 32));
        CUDA_TRY(up(off_dsc, det_scores, nd * 8));
        CUDA_TRY(up(off_gbox, gt_boxes, ng * 32));
        CUDA_TRY(up(off_dcl, det_classes, nd * 4));
        CUDA_TRY(up(off_gcl, gt_classes, ng * 4));
        CUDA_TRY(up(off_dcn, det_counts, (size_t)batch * 4));
        CUDA_TRY(up(off_gcn, gt_counts, (size_t)batch * 4));
        a.det_boxes = reinterpret_cast<const double*>(buf);
        a.det_scores = reinterpret_cast<const double*>(buf + off_dsc);
        a.gt_boxes = reinterpret_cast<const double*>(buf + off_gbox);
        a.det_classes = reinterpret_cast<const int*>(buf + off_dcl);
        a.gt_classes = reinterpret_cast<const int*>(buf + off_gcl);
        a.det_counts = reinterpret_cast<const int*>(buf + off_dcn);
        a.gt_counts = reinterpret_cast<const int*>(buf + off_gcn);
        a.tp = buf + off_tp;
        a.matched = matched_gt ? reinterpret_cast<int*>(buf + off_who) : nullptr;
    } else {
        a.det_boxes = det_boxes; a.det_scores = det_scores; a.det_classes = det_classes;
        a.det_counts = det_counts; a.gt_boxes = gt_boxes; a.gt_classes = gt_classes;
        a.gt_counts = gt_counts; a.tp = tp; a.matched = matched_gt;
    }
    a.next_image = d_ctr;
    CUDA_TRY(launch_match(a, num_sms, st));
    if (host) {
        CUDA_TRY(cudaStreamSynchronize(st));
        if (n_out) CUDA_TRY(cudaMemcpy(tp, buf + off_tp, n_out, cudaMemcpyDeviceToHost));
        if (matched_gt && n_out) CUDA_TRY(cudaMemcpy(matched_gt, buf + off_who, n_out * 4, cudaMemcpyDeviceToHost));
    }
    CUDA_TRY(cudaFreeAsync(buf, st));
    if (!host && (flags & MGD_FLAG_SYNC)) CUDA_TRY(cudaStreamSynchronize(st));
    return MGD_OK;
}

namespace {

int check_map_config(const mgd_map_config* cfg)
{
    if (!cfg) return fail(MGD_ERR_INVALID_ARGUMENT, "cfg is NULL");
    if (cfg->num_classes < 1)
        return fail(MGD_ERR_INVALID_ARGUMENT, "num_classes must be >= 1, got %d", cfg->num_classes);
    if (cfg->num_thresholds < 1 || cfg->num_thresholds > MGD_MAP_MAX_THRESHOLDS)
        return fail(MGD_ERR_INVALID_ARGUMENT, "num_thresholds must be in [1, %d], got %d",
                    MGD_MAP_MAX_THRESHOLDS, cfg->num_thresholds);
    if (cfg->method != MGD_MAP_COCO && cfg->method != MGD_MAP_VOC)
        return fail(MGD_ERR_INVALID_ARGUMENT, "method must be MGD_MAP_COCO or MGD_MAP_VOC, got %d", cfg->method);
    if (cfg->views < 1 || cfg->views >= (1 << MGD_MAP_VIEWS))
        return fail(MGD_ERR_INVALID_ARGUMENT, "views must be a non-empty mask of MGD_MAP_VIEW_* bits");
    return MGD_OK;
}

// the calling thread's mAP scratch on `device`, ordered behind its previous use
int map_workspace(int device, cudaStream_t st, Arena** out)
{
    HostStreams& hs = t_streams[device];
    if (!hs.map_done) CUDA_TRY(cudaEventCreateWithFlags(&hs.map_done, cudaEventDisableTiming));
    CUDA_TRY(cudaStreamWaitEvent(st, hs.map_done, 0));
    hs.map.reset();
    *out = &hs.map;
    return MGD_OK;
}

int map_workspace_done(int device, cudaStream_t st)
{
    CUDA_TRY(cudaEventRecord(t_streams[device].map_done, st));
    return MGD_OK;
}

}  // namespace

int mgd_map_record_bytes(void)
{
    return (int)sizeof(MapRec);
}

int mgd_map_update(const mgd_map_config* cfg, const double* det_boxes, const double* det_scores,
                   const int* det_classes, const int* det_counts, int batch, int max_dets,
                   const double* gt_boxes, const int* gt_classes, const int* gt_counts, int max_gt,
                   long long slot_offset, void* records, long long* gt_hist, int device, void* stream,
                   int flags)
{
    nvtx_range nv_api("mgd_map_update");
    int rc;
    if ((rc = check_map_config(cfg))) return rc;
    if (batch < 0 || max_dets < 0 || max_gt < 0 || slot_offset < 0)
        return fail(MGD_ERR_INVALID_ARGUMENT, "batch, max_dets, max_gt and slot_offset must be >= 0");
    if (slot_offset + (long long)batch * max_dets > 0x7fffffffll)
        return fail(MGD_ERR_UNSUPPORTED, "more than 2^31 - 1 detection slots in one evaluation");
    if (max_dets > 65535) return fail(MGD_ERR_UNSUPPORTED, "max_dets per image must be <= 65535");
    if ((size_t)max_dets * 2 + (size_t)max_gt / 8 > 48 * 1024)
        return fail(MGD_ERR_UNSUPPORTED, "max_dets / max_gt too large for one warp's shared memory");
    if (batch > 0 && (!det_counts || !gt_counts || !gt_hist))
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor");
    if ((long long)batch * max_dets > 0 && (!det_boxes || !det_scores || !det_classes || !records))
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL detection tensor");
    if ((long long)batch * max_gt > 0 && (!gt_boxes || !gt_classes))
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL ground-truth tensor");
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    if (batch == 0) return MGD_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int* d_status;
    if ((rc = deferred_status_word(device, &d_status))) return rc;
    Arena* ws;
    if ((rc = map_workspace(device, st, &ws))) return rc;
    const size_t flags_bytes = (size_t)cfg->num_thresholds * batch * max_dets;
    int* counters;
    CUDA_TRY(ws->take(reinterpret_cast<void**>(&counters), MGD_MAP_VIEWS * sizeof(int)));
    CUDA_TRY(cudaMemsetAsync(counters, 0, MGD_MAP_VIEWS * sizeof(int), st));
    MapWriteArgs w;
    memset(&w, 0, sizeof(w));
    // one match_kernel walk per view: corner / centre IoU over everything, centre IoU per band
    for (int v = 0; v < MGD_MAP_VIEWS; ++v) {
        if (!((cfg->views >> v) & 1)) continue;
        MatchArgs a;
        memset(&a, 0, sizeof(a));
        a.B = batch; a.M = max_dets; a.N = max_gt; a.T = cfg->num_thresholds;
        for (int t = 0; t < a.T; ++t) a.thr[t] = cfg->iou_thresholds[t];
        a.mode = v == MGD_MAP_VIEW_CORNER ? MGD_IOU_CORNER : MGD_IOU_CENTRE;
        a.band = v >= MGD_MAP_VIEW_S ? 1 + v - MGD_MAP_VIEW_S : 0;
        a.det_boxes = det_boxes; a.det_scores = det_scores; a.det_classes = det_classes;
        a.det_counts = det_counts; a.gt_boxes = gt_boxes; a.gt_classes = gt_classes;
        a.gt_counts = gt_counts;
        unsigned char* tp;
        CUDA_TRY(ws->take(reinterpret_cast<void**>(&tp), flags_bytes));
        a.tp = tp;
        a.next_image = counters + v;
        if (flags_bytes) CUDA_TRY(launch_match(a, num_sms, st));
        w.tp[v] = tp;
    }
    w.B = batch; w.M = max_dets; w.N = max_gt; w.T = cfg->num_thresholds; w.C = cfg->num_classes;
    w.views = cfg->views;
    w.det_boxes = det_boxes; w.det_scores = det_scores; w.det_classes = det_classes;
    w.det_counts = det_counts; w.gt_boxes = gt_boxes; w.gt_classes = gt_classes; w.gt_counts = gt_counts;
    w.recs = static_cast<MapRec*>(records) + slot_offset;
    w.gt_hist = reinterpret_cast<unsigned long long*>(gt_hist);
    w.status = d_status;
    CUDA_TRY(launch_map_write(w, st));
    if ((rc = map_workspace_done(device, st))) return rc;
    if (flags & MGD_FLAG_SYNC) return mgd_poll_status(device, stream);
    return MGD_OK;
}

int mgd_map_compute(const mgd_map_config* cfg, const void* records, long long num_slots,
                    const long long* gt_hist, double* ap_out, double* voc_points_out,
                    long long* det_hist_out, int device, void* stream, int flags)
{
    nvtx_range nv_api("mgd_map_compute");
    int rc;
    if ((rc = check_map_config(cfg))) return rc;
    if (num_slots < 0 || num_slots > 0x7fffffffll)
        return fail(MGD_ERR_INVALID_ARGUMENT, "num_slots must be in [0, 2^31 - 1]");
    if ((num_slots > 0 && !records) || !gt_hist || !det_hist_out)
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor");
    if (cfg->method == MGD_MAP_COCO ? !ap_out : !voc_points_out)
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL output of the configured method");
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    Arena* ws;
    if ((rc = map_workspace(device, st, &ws))) return rc;
    void* scratch;
    CUDA_TRY(ws->take(&scratch, map_compute_scratch_bytes(num_slots, cfg->num_thresholds)));
    CUDA_TRY(launch_map_compute(*cfg, static_cast<const MapRec*>(records), num_slots,
                                reinterpret_cast<const unsigned long long*>(gt_hist), ap_out, voc_points_out,
                                reinterpret_cast<unsigned long long*>(det_hist_out), scratch, st));
    if ((rc = map_workspace_done(device, st))) return rc;
    if (flags & MGD_FLAG_SYNC) CUDA_TRY(cudaStreamSynchronize(st));
    return MGD_OK;
}

int mgd_map_partition(const mgd_map_config* cfg, const void* records, long long num_slots,
                      const long long* segments, int num_segments, long long global_slots, const int* owner,
                      int world, void* out_records, long long* out_counts, int device, void* stream, int flags)
{
    nvtx_range nv_api("mgd_map_partition");
    int rc;
    if ((rc = check_map_config(cfg))) return rc;
    if (num_slots < 0 || num_slots > 0x7fffffffll)
        return fail(MGD_ERR_INVALID_ARGUMENT, "num_slots must be in [0, 2^31 - 1]");
    if (num_segments < 0 || (num_slots > 0 && num_segments < 1))
        return fail(MGD_ERR_INVALID_ARGUMENT, "num_segments must be >= 1 when there are records");
    if (global_slots < num_slots)
        return fail(MGD_ERR_INVALID_ARGUMENT, "global_slots must be >= num_slots");
    if (global_slots > (1ll << 32))
        return fail(MGD_ERR_UNSUPPORTED, "more than 2^32 global detection slots in one evaluation");
    if (world < 1) return fail(MGD_ERR_INVALID_ARGUMENT, "world must be >= 1, got %d", world);
    if (world > 256) return fail(MGD_ERR_UNSUPPORTED, "world must be <= 256, got %d", world);
    if (!owner || !out_counts) return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor");
    if (num_slots > 0 && (!records || !segments || !out_records))
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor");
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    MapPartitionArgs a;
    a.recs = static_cast<const MapRec*>(records); a.n = num_slots; a.C = cfg->num_classes;
    a.segs = segments; a.num_segs = num_segments; a.owner = owner; a.world = world;
    a.out = static_cast<MapRec*>(out_records); a.counts = out_counts;
    if ((rc = deferred_status_word(device, &a.status))) return rc;
    Arena* ws;
    if ((rc = map_workspace(device, st, &ws))) return rc;
    void* scratch;
    CUDA_TRY(ws->take(&scratch, map_partition_scratch_bytes(num_slots)));
    CUDA_TRY(launch_map_partition(a, scratch, st));
    if ((rc = map_workspace_done(device, st))) return rc;
    if (flags & MGD_FLAG_SYNC) return mgd_poll_status(device, stream);
    return MGD_OK;
}

int mgd_map_compute_merged(const mgd_map_config* cfg, const void* records, long long num_records,
                           const long long* gt_hist, const int* owner, int rank, double* ap_out,
                           double* voc_points_out, long long* det_hist_out, int device, void* stream, int flags)
{
    nvtx_range nv_api("mgd_map_compute_merged");
    int rc;
    if ((rc = check_map_config(cfg))) return rc;
    if (num_records < 0 || num_records > 0x7fffffffll)
        return fail(MGD_ERR_INVALID_ARGUMENT, "num_records must be in [0, 2^31 - 1]");
    if ((num_records > 0 && !records) || !gt_hist || !owner || !det_hist_out)
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor");
    if (cfg->method == MGD_MAP_COCO ? !ap_out : !voc_points_out)
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL output of the configured method");
    if (rank < 0) return fail(MGD_ERR_INVALID_ARGUMENT, "rank must be >= 0, got %d", rank);
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    Arena* ws;
    if ((rc = map_workspace(device, st, &ws))) return rc;
    void* scratch;
    CUDA_TRY(ws->take(&scratch, map_compute_scratch_bytes(num_records, cfg->num_thresholds)));
    CUDA_TRY(launch_map_compute_merged(*cfg, static_cast<const MapRec*>(records), num_records,
                                       reinterpret_cast<const unsigned long long*>(gt_hist), owner, rank,
                                       ap_out, voc_points_out, reinterpret_cast<unsigned long long*>(det_hist_out),
                                       scratch, st));
    if ((rc = map_workspace_done(device, st))) return rc;
    if (flags & MGD_FLAG_SYNC) CUDA_TRY(cudaStreamSynchronize(st));
    return MGD_OK;
}

namespace {

// the curve / operating-point outputs of mgd_map_compute_pr and _merged_pr; n: records in
int check_map_pr(const mgd_map_config* cfg, const mgd_map_pr* pr, long long n)
{
    const int full = (1 << MGD_MAP_VIEW_CORNER) | (1 << MGD_MAP_VIEW_CENTRE);
    if (!pr) return fail(MGD_ERR_INVALID_ARGUMENT, "pr is NULL");
    if (pr->views == 0 || (pr->views & ~full))
        return fail(MGD_ERR_INVALID_ARGUMENT, "pr->views must be a non-empty mask of MGD_MAP_VIEW_CORNER / _CENTRE");
    if (pr->views & ~cfg->views)
        return fail(MGD_ERR_INVALID_ARGUMENT, "pr->views holds a view cfg->views does not match");
    if (pr->num_confidences < 0 || pr->num_confidences > MGD_MAP_MAX_CONFIDENCES)
        return fail(MGD_ERR_INVALID_ARGUMENT, "num_confidences must be in [0, %d], got %d",
                    MGD_MAP_MAX_CONFIDENCES, pr->num_confidences);
    if (pr->num_confidences > 0 && (!pr->confidences || !pr->at_confidence))
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL confidences or at_confidence");
    for (int q = 0; q < pr->num_confidences; ++q)
        if (!isfinite(pr->confidences[q]))
            return fail(MGD_ERR_INVALID_ARGUMENT, "confidences[%d] is not finite", q);
    if (pr->capacity < n)
        return fail(MGD_ERR_INVALID_ARGUMENT, "capacity (%lld) is below the record count (%lld)", pr->capacity, n);
    if (!pr->offsets || !pr->best_f1 || !pr->best_index)
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL operating-point output");
    if (pr->capacity > 0 && (!pr->scores || !pr->precision || !pr->recall))
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL curve output");
    return MGD_OK;
}

}  // namespace

int mgd_map_compute_pr(const mgd_map_config* cfg, const void* records, long long num_slots,
                       const long long* gt_hist, double* ap_out, double* voc_points_out,
                       long long* det_hist_out, const mgd_map_pr* pr, int device, void* stream, int flags)
{
    nvtx_range nv_api("mgd_map_compute_pr");
    int rc;
    if ((rc = check_map_config(cfg))) return rc;
    if (num_slots < 0 || num_slots > 0x7fffffffll)
        return fail(MGD_ERR_INVALID_ARGUMENT, "num_slots must be in [0, 2^31 - 1]");
    if ((num_slots > 0 && !records) || !gt_hist || !det_hist_out)
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor");
    if (cfg->method == MGD_MAP_COCO ? !ap_out : !voc_points_out)
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL output of the configured method");
    if ((rc = check_map_pr(cfg, pr, num_slots))) return rc;
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    Arena* ws;
    if ((rc = map_workspace(device, st, &ws))) return rc;
    void* scratch;
    CUDA_TRY(ws->take(&scratch, map_compute_scratch_bytes(num_slots, cfg->num_thresholds)));
    CUDA_TRY(launch_map_compute(*cfg, static_cast<const MapRec*>(records), num_slots,
                                reinterpret_cast<const unsigned long long*>(gt_hist), ap_out, voc_points_out,
                                reinterpret_cast<unsigned long long*>(det_hist_out), scratch, st, pr));
    if ((rc = map_workspace_done(device, st))) return rc;
    if (flags & MGD_FLAG_SYNC) CUDA_TRY(cudaStreamSynchronize(st));
    return MGD_OK;
}

int mgd_map_compute_merged_pr(const mgd_map_config* cfg, const void* records, long long num_records,
                              const long long* gt_hist, const int* owner, int rank, double* ap_out,
                              double* voc_points_out, long long* det_hist_out, const mgd_map_pr* pr, int device,
                              void* stream, int flags)
{
    nvtx_range nv_api("mgd_map_compute_merged_pr");
    int rc;
    if ((rc = check_map_config(cfg))) return rc;
    if (num_records < 0 || num_records > 0x7fffffffll)
        return fail(MGD_ERR_INVALID_ARGUMENT, "num_records must be in [0, 2^31 - 1]");
    if ((num_records > 0 && !records) || !gt_hist || !owner || !det_hist_out)
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor");
    if (cfg->method == MGD_MAP_COCO ? !ap_out : !voc_points_out)
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL output of the configured method");
    if (rank < 0) return fail(MGD_ERR_INVALID_ARGUMENT, "rank must be >= 0, got %d", rank);
    if ((rc = check_map_pr(cfg, pr, num_records))) return rc;
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    Arena* ws;
    if ((rc = map_workspace(device, st, &ws))) return rc;
    void* scratch;
    CUDA_TRY(ws->take(&scratch, map_compute_scratch_bytes(num_records, cfg->num_thresholds)));
    CUDA_TRY(launch_map_compute_merged(*cfg, static_cast<const MapRec*>(records), num_records,
                                       reinterpret_cast<const unsigned long long*>(gt_hist), owner, rank,
                                       ap_out, voc_points_out, reinterpret_cast<unsigned long long*>(det_hist_out),
                                       scratch, st, pr));
    if ((rc = map_workspace_done(device, st))) return rc;
    if (flags & MGD_FLAG_SYNC) CUDA_TRY(cudaStreamSynchronize(st));
    return MGD_OK;
}

int mgd_ignore_mask(const mgd_head_config* cfg, const float* const* y_pred,
                    const float* const* y_true, int batch, double ignore_thresh, double eps,
                    float* const* ignore_mask, float* const* assigned_anchor_iou,
                    float* const* max_iou_map, int memory, int device, void* stream, int flags)
{
    nvtx_range nv_api("mgd_ignore_mask");
    HeadGeom g;
    int rc = build_geom(cfg, &g);
    if (rc) return rc;
    if ((rc = check_memory_arg(memory))) return rc;
    if (batch < 0) return fail(MGD_ERR_INVALID_ARGUMENT, "batch must be >= 0");
    if (!y_pred || !y_true || !ignore_mask || !assigned_anchor_iou || !max_iou_map)
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor list");
    for (int l = 0; l < g.L && batch > 0; ++l)
        if (!y_pred[l] || !y_true[l] || !ignore_mask[l] || !assigned_anchor_iou[l] || !max_iou_map[l])
            return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor for layer %d", l);
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    if (batch == 0) return MGD_OK;
    const bool host = memory == MGD_MEM_HOST;
    cudaStream_t st = (cudaStream_t)stream;
    if (host) {
        cudaStream_t* ss;
        if ((rc = host_streams(device, &ss, nullptr))) return rc;
        st = ss[0];
    }
    LossArgs a;
    memset(&a, 0, sizeof(a));
    a.g = g; a.B = batch; a.ignore_thresh = (float)ignore_thresh; a.eps = (float)eps;
    // scratch: ground-truth lists; host memory: staged tensors as well
    const size_t n_gt = (size_t)batch * g.cells * 2;
    size_t in_floats = 0, out_floats = 0;
    for (int l = 0; l < g.L; ++l) {
        in_floats += (size_t)batch * g.gh[l] * g.gw[l] * g.D[l];
        out_floats += (size_t)batch * g.gh[l] * g.gw[l];
    }
    const size_t off_area = n_gt * 16, off_cnt = off_area + n_gt * 4;
    const size_t off_in = (off_cnt + (size_t)batch * g.L * 4 + 15) & ~(size_t)15;
    const size_t total = off_in + (host ? (2 * in_floats + 3 * out_floats) * 4 : 0);
    unsigned char* buf;
    CUDA_TRY(pool_malloc(&buf, total, st));
    a.gt_boxes = buf;
    a.gt_area = reinterpret_cast<float*>(buf + off_area);
    a.gt_count = reinterpret_cast<int*>(buf + off_cnt);
    float* cursor = reinterpret_cast<float*>(buf + off_in);
    for (int l = 0; l < g.L; ++l) {
        const size_t n_in = (size_t)batch * g.gh[l] * g.gw[l] * g.D[l];
        const size_t n_out = (size_t)batch * g.gh[l] * g.gw[l];
        if (host) {
            CUDA_TRY(cudaMemcpyAsync(cursor, y_pred[l], n_in * 4, cudaMemcpyHostToDevice, st));
            a.y_pred[l] = cursor; cursor += n_in;
            CUDA_TRY(cudaMemcpyAsync(cursor, y_true[l], n_in * 4, cudaMemcpyHostToDevice, st));
            a.y_true[l] = cursor; cursor += n_in;
            a.ignore[l] = cursor; cursor += n_out;
            a.assigned[l] = cursor; cursor += n_out;
            a.max_iou[l] = cursor; cursor += n_out;
        } else {
            a.y_pred[l] = y_pred[l]; a.y_true[l] = y_true[l];
            a.ignore[l] = ignore_mask[l]; a.assigned[l] = assigned_anchor_iou[l]; a.max_iou[l] = max_iou_map[l];
        }
    }
    CUDA_TRY(launch_ignore_mask(a, st));
    if (host) {
        CUDA_TRY(cudaStreamSynchronize(st));
        for (int l = 0; l < g.L; ++l) {
            const size_t n_out = (size_t)batch * g.gh[l] * g.gw[l] * 4;
            CUDA_TRY(cudaMemcpy(ignore_mask[l], a.ignore[l], n_out, cudaMemcpyDeviceToHost));
            CUDA_TRY(cudaMemcpy(assigned_anchor_iou[l], a.assigned[l], n_out, cudaMemcpyDeviceToHost));
            CUDA_TRY(cudaMemcpy(max_iou_map[l], a.max_iou[l], n_out, cudaMemcpyDeviceToHost));
        }
    }
    CUDA_TRY(cudaFreeAsync(buf, st));
    if (!host && (flags & MGD_FLAG_SYNC)) CUDA_TRY(cudaStreamSynchronize(st));
    return MGD_OK;
}

int mgd_reshape_boxes(const void* boxes, int boxes_dtype, const int* counts, const int* params,
                      int batch, int max_boxes, void* out, float* out_f32, int* out_counts,
                      int memory, int device, void* stream, int flags)
{
    nvtx_range nv_api("mgd_reshape_boxes");
    int rc;
    if ((rc = check_memory_arg(memory))) return rc;
    if (batch < 0 || max_boxes < 0) return fail(MGD_ERR_INVALID_ARGUMENT, "batch and max_boxes must be >= 0");
    if (boxes_dtype != MGD_BOXES_I32 && boxes_dtype != MGD_BOXES_F64)
        return fail(MGD_ERR_INVALID_ARGUMENT, "boxes_dtype must be MGD_BOXES_I32 or MGD_BOXES_F64");
    const size_t n = (size_t)batch * max_boxes * 5;
    if (batch > 0 && !params) return fail(MGD_ERR_INVALID_ARGUMENT, "params is NULL");
    if (n > 0 && (!boxes || !out)) return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor");
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    if (batch == 0) return MGD_OK;
    const size_t esz = boxes_dtype == MGD_BOXES_I32 ? 4 : 8;
    BoxOpArgs a;
    memset(&a, 0, sizeof(a));
    a.B = batch; a.N = max_boxes;
    if (memory == MGD_MEM_DEVICE) {
        cudaStream_t st = (cudaStream_t)stream;
        a.in = boxes; a.counts = counts; a.params = params; a.out = out; a.out_f32 = out_f32;
        a.out_counts = out_counts;
        CUDA_TRY(launch_reshape_boxes(a, boxes_dtype == MGD_BOXES_I32, st));
        if (flags & MGD_FLAG_SYNC) CUDA_TRY(cudaStreamSynchronize(st));
        return MGD_OK;
    }
    cudaStream_t* ss;
    if ((rc = host_streams(device, &ss, nullptr))) return rc;
    cudaStream_t st = ss[0];
    // staging: in | out (8-byte fields first) | out_f32 | params | counts | out_counts
    const size_t off_out = (n * esz + 7) & ~(size_t)7, off_f32 = off_out + ((n * esz + 7) & ~(size_t)7);
    const size_t off_par = off_f32 + n * 4, off_cnt = off_par + (size_t)batch * 40;
    const size_t off_ocn = off_cnt + (size_t)batch * 4, total = off_ocn + (size_t)batch * 4;
    unsigned char* buf;
    CUDA_TRY(pool_malloc(&buf, total, st));
    if (n) CUDA_TRY(cudaMemcpyAsync(buf, boxes, n * esz, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(buf + off_par, params, (size_t)batch * 40, cudaMemcpyHostToDevice, st));
    if (counts) CUDA_TRY(cudaMemcpyAsync(buf + off_cnt, counts, (size_t)batch * 4, cudaMemcpyHostToDevice, st));
    a.in = buf; a.out = buf + off_out; a.out_f32 = reinterpret_cast<float*>(buf + off_f32);
    a.params = reinterpret_cast<const int*>(buf + off_par);
    a.counts = counts ? reinterpret_cast<const int*>(buf + off_cnt) : nullptr;
    a.out_counts = reinterpret_cast<int*>(buf + off_ocn);
    CUDA_TRY(launch_reshape_boxes(a, boxes_dtype == MGD_BOXES_I32, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (n) CUDA_TRY(cudaMemcpy(out, buf + off_out, n * esz, cudaMemcpyDeviceToHost));
    if (out_f32 && n) CUDA_TRY(cudaMemcpy(out_f32, buf + off_f32, n * 4, cudaMemcpyDeviceToHost));
    if (out_counts) CUDA_TRY(cudaMemcpy(out_counts, buf + off_ocn, (size_t)batch * 4, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaFreeAsync(buf, st));
    return MGD_OK;
}

int mgd_encode_ignore_mask(const mgd_head_config* cfg, const float* boxes, int batch, int max_boxes,
                           const float* const* y_pred, float* const* y_true, double ignore_thresh,
                           double eps, float* const* ignore_mask, float* const* assigned_anchor_iou,
                           float* const* max_iou_map, int device, void* stream, int flags)
{
    nvtx_range nv_api("mgd_encode_ignore_mask");
    HeadGeom g;
    int rc = build_geom(cfg, &g);
    if (rc) return rc;
    if (batch < 0 || max_boxes < 0) return fail(MGD_ERR_INVALID_ARGUMENT, "batch and max_boxes must be >= 0");
    if (!y_pred || !ignore_mask || !assigned_anchor_iou || !max_iou_map)
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor list");
    for (int l = 0; l < g.L && batch > 0; ++l)
        if (!y_pred[l] || !ignore_mask[l] || !assigned_anchor_iou[l] || !max_iou_map[l] || (y_true && !y_true[l]))
            return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor for layer %d", l);
    if (!boxes && (long long)batch * max_boxes > 0) return fail(MGD_ERR_INVALID_ARGUMENT, "boxes is NULL");
    if (max_boxes > 65000)
        return fail(MGD_ERR_UNSUPPORTED, "max_boxes per image must be <= 65000, got %d", max_boxes);
    if ((long long)chunk_images(g, batch > 0 ? batch : 1) * max_boxes >= (1ll << 27))
        return fail(MGD_ERR_UNSUPPORTED, "batch chunk x max_boxes too large");
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    if (batch == 0) return MGD_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int* d_flag;
    if ((rc = deferred_status_word(device, &d_flag))) return rc;
    const Alloc al{nullptr, st};
    const int step = chunk_images(g, batch);
    for (int b0 = 0; b0 < batch; b0 += step) {
        const int nb = batch - b0 < step ? batch - b0 : step;
        EncodeArgs e;
        e.g = g; e.B = nb; e.N = max_boxes;
        e.boxes = boxes + (size_t)b0 * max_boxes * 5;
        for (int l = 0; l < g.L; ++l)
            e.y[l] = y_true ? y_true[l] + (size_t)b0 * g.gh[l] * g.gw[l] * g.D[l] : nullptr;
        e.tf_compat = (flags & MGD_FLAG_TF_COMPAT) != 0;
        e.status = d_flag; e.stats = nullptr;
        e.big_tables = nullptr; e.table = nullptr; e.recs = nullptr;
        unsigned char* scratch = nullptr;
        auto release = [&]() { al.put(e.table); al.put(e.recs); al.put(e.big_tables); al.put(scratch); };
        cudaError_t ce = cudaSuccess;
        if (encode_needs_big_tables(g, max_boxes))
            ce = al.get(&e.big_tables, (size_t)nb * 2 * g.cells * sizeof(int));
        if (ce == cudaSuccess) ce = al.get(&e.table, (size_t)nb * g.cells * sizeof(int));
        if (ce == cudaSuccess) ce = al.get(&e.recs, (size_t)nb * (max_boxes > 0 ? max_boxes : 1) * sizeof(BoxRec));
        const size_t n_gt = (size_t)nb * g.cells * 2;
        const size_t off_area = n_gt * 16, off_cnt = off_area + n_gt * 4;
        if (ce == cudaSuccess) ce = al.get(&scratch, off_cnt + (size_t)nb * g.L * 4);
        if (ce == cudaSuccess) ce = launch_encode_assign(e, st);
        if (ce == cudaSuccess && y_true) ce = launch_encode_fill(e, num_sms, st);
        if (ce == cudaSuccess) {
            LossArgs a;
            memset(&a, 0, sizeof(a));
            a.g = g; a.B = nb; a.ignore_thresh = (float)ignore_thresh; a.eps = (float)eps;
            a.table = e.table; a.recs = e.recs;
            a.gt_boxes = scratch;
            a.gt_area = reinterpret_cast<float*>(scratch + off_area);
            a.gt_count = reinterpret_cast<int*>(scratch + off_cnt);
            for (int l = 0; l < g.L; ++l) {
                const size_t cells_b0 = (size_t)b0 * g.gh[l] * g.gw[l];
                a.y_pred[l] = y_pred[l] + cells_b0 * g.D[l];
                a.ignore[l] = ignore_mask[l] + cells_b0;
                a.assigned[l] = assigned_anchor_iou[l] + cells_b0;
                a.max_iou[l] = max_iou_map[l] + cells_b0;
            }
            ce = launch_ignore_mask(a, st);
        }
        release();
        CUDA_TRY(ce);
    }
    if (flags & MGD_FLAG_SYNC) {
        CUDA_TRY(cudaStreamSynchronize(st));
        return mgd_poll_status(device, stream);
    }
    return MGD_OK;
}

int mgd_letterbox_boxes(const float* boxes, const int* counts, const int* params, int batch,
                        int max_in, int input_h, int input_w, int max_boxes_per_image, int expansion,
                        float* out, int memory, int device, void* stream, int flags)
{
    nvtx_range nv_api("mgd_letterbox_boxes");
    int rc;
    if ((rc = check_memory_arg(memory))) return rc;
    if (batch < 0 || max_in < 0 || max_boxes_per_image < 1)
        return fail(MGD_ERR_INVALID_ARGUMENT, "batch, max_in >= 0 and max_boxes_per_image >= 1 required");
    if (expansion != 1 && expansion != 2 && expansion != 4 && expansion != 8)
        return fail(MGD_ERR_INVALID_ARGUMENT, "expansion must be 1, 2, 4 or 8 (generators.py:2008-2017)");
    if (input_h < 1 || input_w < 1) return fail(MGD_ERR_INVALID_ARGUMENT, "input shape must be positive");
    const long long cap = (long long)max_boxes_per_image * expansion;
    if (cap > (1 << 20)) return fail(MGD_ERR_UNSUPPORTED, "capacity too large");
    if (batch > 0 && (!params || !out || (max_in > 0 && !boxes)))
        return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor");
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    if (batch == 0) return MGD_OK;
    if (memory == MGD_MEM_DEVICE) {
        cudaStream_t st = (cudaStream_t)stream;
        CUDA_TRY(launch_letterbox_boxes(boxes, counts, params, batch, max_in, max_boxes_per_image,
                                        (int)cap, input_h, input_w, out, st));
        if (flags & MGD_FLAG_SYNC) CUDA_TRY(cudaStreamSynchronize(st));
        return MGD_OK;
    }
    cudaStream_t* ss;
    if ((rc = host_streams(device, &ss, nullptr))) return rc;
    cudaStream_t st = ss[0];
    const size_t n_in = (size_t)batch * max_in * 5 * 4, n_out = (size_t)batch * cap * 5 * 4;
    const size_t off_out = (n_in + 15) & ~(size_t)15, off_par = off_out + ((n_out + 15) & ~(size_t)15);
    const size_t off_cnt = off_par + (size_t)batch * 24, total = off_cnt + (size_t)batch * 4;
    unsigned char* buf;
    CUDA_TRY(pool_malloc(&buf, total, st));
    if (n_in) CUDA_TRY(cudaMemcpyAsync(buf, boxes, n_in, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(buf + off_par, params, (size_t)batch * 24, cudaMemcpyHostToDevice, st));
    if (counts) CUDA_TRY(cudaMemcpyAsync(buf + off_cnt, counts, (size_t)batch * 4, cudaMemcpyHostToDevice, st));
    cudaError_t e = launch_letterbox_boxes(reinterpret_cast<const float*>(buf),
                                           counts ? reinterpret_cast<const int*>(buf + off_cnt) : nullptr,
                                           reinterpret_cast<const int*>(buf + off_par), batch, max_in,
                                           max_boxes_per_image, (int)cap, input_h, input_w,
                                           reinterpret_cast<float*>(buf + off_out), st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaMemcpy(out, buf + off_out, n_out, cudaMemcpyDeviceToHost);
    cudaFreeAsync(buf, st);
    CUDA_TRY(e);
    return MGD_OK;
}

int mgd_mosaic_merge_boxes(const double* boxes, int num_sources, int max_boxes, const int* params,
                           int batch, int height, int width, double* out, float* out_f32,
                           int* out_counts, int memory, int device, void* stream, int flags)
{
    nvtx_range nv_api("mgd_mosaic_merge_boxes");
    int rc;
    if ((rc = check_memory_arg(memory))) return rc;
    if (batch < 0 || max_boxes < 0 || num_sources < 0)
        return fail(MGD_ERR_INVALID_ARGUMENT, "batch, num_sources and max_boxes must be >= 0");
    const size_t n_in = (size_t)num_sources * max_boxes * 5, n = (size_t)batch * max_boxes * 5;
    if (batch > 0 && !params) return fail(MGD_ERR_INVALID_ARGUMENT, "params is NULL");
    if (n > 0 && (!out || (n_in > 0 && !boxes))) return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor");
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    if (batch == 0) return MGD_OK;
    BoxOpArgs a;
    memset(&a, 0, sizeof(a));
    a.B = batch; a.N = max_boxes; a.n_src = num_sources; a.height = height; a.width = width;
    if (memory == MGD_MEM_DEVICE) {
        cudaStream_t st = (cudaStream_t)stream;
        a.in = boxes; a.params = params; a.out = out; a.out_f32 = out_f32; a.out_counts = out_counts;
        CUDA_TRY(launch_mosaic_merge(a, st));
        if (flags & MGD_FLAG_SYNC) CUDA_TRY(cudaStreamSynchronize(st));
        return MGD_OK;
    }
    cudaStream_t* ss;
    if ((rc = host_streams(device, &ss, nullptr))) return rc;
    cudaStream_t st = ss[0];
    const size_t off_out = n_in * 8, off_f32 = off_out + n * 8, off_par = off_f32 + n * 4;
    const size_t off_ocn = off_par + (size_t)batch * 24, total = off_ocn + (size_t)batch * 4;
    unsigned char* buf;
    CUDA_TRY(pool_malloc(&buf, total, st));
    if (n_in) CUDA_TRY(cudaMemcpyAsync(buf, boxes, n_in * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(buf + off_par, params, (size_t)batch * 24, cudaMemcpyHostToDevice, st));
    a.in = buf; a.out = buf + off_out; a.out_f32 = reinterpret_cast<float*>(buf + off_f32);
    a.params = reinterpret_cast<const int*>(buf + off_par);
    a.out_counts = reinterpret_cast<int*>(buf + off_ocn);
    CUDA_TRY(launch_mosaic_merge(a, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (n) CUDA_TRY(cudaMemcpy(out, buf + off_out, n * 8, cudaMemcpyDeviceToHost));
    if (out_f32 && n) CUDA_TRY(cudaMemcpy(out_f32, buf + off_f32, n * 4, cudaMemcpyDeviceToHost));
    if (out_counts) CUDA_TRY(cudaMemcpy(out_counts, buf + off_ocn, (size_t)batch * 4, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaFreeAsync(buf, st));
    return MGD_OK;
}

int mgd_iou_matrix(const double* boxes1, int n, const double* boxes2, int m, double* out, int memory,
                   int device, void* stream, int flags)
{
    nvtx_range nv_api("mgd_iou_matrix");
    int rc;
    if ((rc = check_memory_arg(memory))) return rc;
    if (n < 0 || m < 0) return fail(MGD_ERR_INVALID_ARGUMENT, "n and m must be >= 0");
    if ((long long)n * m > 0 && (!boxes1 || !boxes2 || !out)) return fail(MGD_ERR_INVALID_ARGUMENT, "NULL tensor");
    int num_sms;
    DeviceScope dev_scope;
    if ((rc = prepare_device(device, &num_sms, &dev_scope))) return rc;
    if ((long long)n * m == 0) return MGD_OK;
    const bool host = memory == MGD_MEM_HOST;
    cudaStream_t st = (cudaStream_t)stream;
    if (!host) {
        CUDA_TRY(launch_iou_matrix(boxes1, n, boxes2, m, out, st));
        if (flags & MGD_FLAG_SYNC) CUDA_TRY(cudaStreamSynchronize(st));
        return MGD_OK;
    }
    cudaStream_t* ss;
    if ((rc = host_streams(device, &ss, nullptr))) return rc;
    st = ss[0];
    double* buf;
    const size_t nn = (size_t)n * 4, mm = (size_t)m * 4, oo = (size_t)n * m;
    CUDA_TRY(pool_malloc(&buf, (nn + mm + oo) * 8, st));
    CUDA_TRY(cudaMemcpyAsync(buf, boxes1, nn * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(buf + nn, boxes2, mm * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(launch_iou_matrix(buf, n, buf + nn, m, buf + nn + mm, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaMemcpy(out, buf + nn + mm, oo * 8, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaFreeAsync(buf, st));
    return MGD_OK;
}

}  // extern "C"

// ---- DLPack adapters ---------------------------------------------------------------
namespace {

int dl_check(const DLTensor* t, const char* name, uint8_t code, uint8_t bits, int ndim,
             const long long* shape, int* memory, int* device)
{
    if (!t) return fail(MGD_ERR_INVALID_ARGUMENT, "%s is NULL", name);
    if (t->dtype.code != code || t->dtype.bits != bits || t->dtype.lanes != 1)
        return fail(MGD_ERR_INVALID_ARGUMENT, "%s: wrong dtype (code %d bits %d)", name,
                    (int)t->dtype.code, (int)t->dtype.bits);
    if (t->ndim != ndim) return fail(MGD_ERR_INVALID_ARGUMENT, "%s: expected %d dims, got %d", name, ndim, t->ndim);
    long long expect_stride = 1;
    for (int i = ndim - 1; i >= 0; --i) {
        if (shape[i] >= 0 && t->shape[i] != shape[i])
            return fail(MGD_ERR_INVALID_ARGUMENT, "%s: dim %d is %lld, expected %lld", name, i,
                        (long long)t->shape[i], shape[i]);
        if (t->strides && t->shape[i] > 1 && t->strides[i] != expect_stride)
            return fail(MGD_ERR_INVALID_ARGUMENT, "%s: tensor must be dense row-major", name);
        expect_stride *= t->shape[i];
    }
    int mem, dev = 0;
    if (t->device.device_type == kDLCPU || t->device.device_type == kDLCUDAHost) mem = MGD_MEM_HOST;
    else if (t->device.device_type == kDLCUDA) { mem = MGD_MEM_DEVICE; dev = t->device.device_id; }
    else return fail(MGD_ERR_INVALID_ARGUMENT, "%s: unsupported DLPack device type %d", name,
                     (int)t->device.device_type);
    if (*memory < 0) { *memory = mem; *device = dev; }
    else if (*memory != mem || (mem == MGD_MEM_DEVICE && *device != dev))
        return fail(MGD_ERR_INVALID_ARGUMENT, "%s: all tensors of a call must live in the same memory", name);
    return MGD_OK;
}

template <typename T> T* dl_ptr(const DLTensor* t)
{
    return t ? reinterpret_cast<T*>(static_cast<char*>(t->data) + t->byte_offset) : nullptr;
}

}  // namespace

extern "C" {

int mgd_encode_targets_dlpack(const mgd_head_config* cfg, const DLTensor* boxes,
                              DLTensor* const* y_true, void* stream, int flags, long long* stats)
{
    HeadGeom g;
    int rc = build_geom(cfg, &g);
    if (rc) return rc;
    int memory = -1, device = 0;
    const long long bshape[3] = {-1, -1, 5};
    if ((rc = dl_check(boxes, "boxes", kDLFloat, 32, 3, bshape, &memory, &device))) return rc;
    const long long B = boxes->shape[0], N = boxes->shape[1];
    if (!y_true) return fail(MGD_ERR_INVALID_ARGUMENT, "y_true is NULL");
    float* yp[MGD_MAX_LAYERS];
    for (int l = 0; l < g.L; ++l) {
        const long long s[4] = {B, g.gh[l], g.gw[l], g.D[l]};
        char name[32];
        snprintf(name, sizeof(name), "y_true[%d]", l);
        if ((rc = dl_check(y_true[l], name, kDLFloat, 32, 4, s, &memory, &device))) return rc;
        yp[l] = dl_ptr<float>(y_true[l]);
    }
    int cur = 0;
    if (memory == MGD_MEM_HOST) { cudaGetDevice(&cur); cudaGetLastError(); device = cur; }
    return mgd_encode_targets(cfg, dl_ptr<const float>(boxes), (int)B, (int)N, yp, memory, device,
                              stream, flags, stats);
}

int mgd_decode_nms_dlpack(const mgd_head_config* cfg, const mgd_post_config* post,
                          const DLTensor* const* preds, const DLTensor* image_hw,
                          DLTensor* boxes_xywh, DLTensor* boxes_xyxy, DLTensor* scores,
                          DLTensor* classes, DLTensor* index, DLTensor* counts, void* stream,
                          int flags, long long* stats)
{
    HeadGeom g;
    int rc = build_geom(cfg, &g);
    if (rc) return rc;
    if ((rc = check_post(post))) return rc;
    if (!preds || !preds[0]) return fail(MGD_ERR_INVALID_ARGUMENT, "preds is NULL");
    int memory = -1, device = 0;
    const long long B = preds[0]->ndim == 4 ? preds[0]->shape[0] : -1;
    const float* pp[MGD_MAX_LAYERS];
    for (int l = 0; l < g.L; ++l) {
        const long long s[4] = {B, g.gh[l], g.gw[l], g.D[l]};
        char name[32];
        snprintf(name, sizeof(name), "preds[%d]", l);
        if ((rc = dl_check(preds[l], name, kDLFloat, 32, 4, s, &memory, &device))) return rc;
        pp[l] = dl_ptr<const float>(preds[l]);
    }
    const long long M = post->max_boxes;
    const long long s_hw[2] = {B, 2}, s_b4[3] = {B, M, 4}, s_b[2] = {B, M}, s_c[1] = {B};
    if (image_hw && (rc = dl_check(image_hw, "image_hw", kDLInt, 32, 2, s_hw, &memory, &device))) return rc;
    if (boxes_xywh && (rc = dl_check(boxes_xywh, "boxes_xywh", kDLFloat, 64, 3, s_b4, &memory, &device))) return rc;
    if (boxes_xyxy && (rc = dl_check(boxes_xyxy, "boxes_xyxy", kDLInt, 32, 3, s_b4, &memory, &device))) return rc;
    if (scores && (rc = dl_check(scores, "scores", kDLFloat, 64, 2, s_b, &memory, &device))) return rc;
    if (classes && (rc = dl_check(classes, "classes", kDLInt, 32, 2, s_b, &memory, &device))) return rc;
    if (index && (rc = dl_check(index, "index", kDLInt, 32, 2, s_b, &memory, &device))) return rc;
    if ((rc = dl_check(counts, "counts", kDLInt, 32, 1, s_c, &memory, &device))) return rc;
    int cur = 0;
    if (memory == MGD_MEM_HOST) { cudaGetDevice(&cur); cudaGetLastError(); device = cur; }
    return mgd_decode_nms(cfg, post, pp, (int)B, dl_ptr<const int>(image_hw),
                          dl_ptr<double>(boxes_xywh), dl_ptr<int>(boxes_xyxy), dl_ptr<double>(scores),
                          dl_ptr<int>(classes), dl_ptr<int>(index), dl_ptr<int>(counts), memory,
                          device, stream, flags, stats);
}

}  // extern "C"
