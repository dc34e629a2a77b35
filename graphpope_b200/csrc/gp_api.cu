// gp_api.cu — library-level entry points of the C ABI: errors, device info and the one-call
// host-buffer path that stands in for get_geodesic_distance_vector + concat_into_features
// (reference utils.py:116-135).
#include "gp_msbfs.cuh"

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#if defined(__x86_64__) || defined(_M_X64)
#include <emmintrin.h>
#endif
#include <thread>
#include <vector>

#include <nvtx3/nvToolsExt.h>
#include <unistd.h>

bool gp_is_capturing();
bool gp_xcopy_tma_ok(const float *d_x, int64_t num_features, int64_t ld_x, const float *d_out, int64_t ld_out);
int gp_launch_xcopy_tma(const float *d_x, int64_t num_nodes, int64_t num_features, int64_t ld_x, float *d_out,
                        int64_t ld_out, cudaStream_t stream);
struct gp_exchange;
int gp_exchange_launch(gp_exchange *x, int parity, const float *d_x, int64_t f, int64_t ldx, float *d_out, int64_t ldo,
                       int64_t coff, cudaStream_t stream);
int gp_exchange_next_parity(gp_exchange *x);
static bool g_capturing_flag_for_count() { return gp_is_capturing(); }
void gp_count_launches(int n);

namespace {
thread_local char g_err[512] = "";
int g_sm_count = 0;
std::atomic<long long> g_launches{0};
}  // namespace

static thread_local int g_capture_count = 0;  // kernels this thread recorded into the graph it is capturing
void gp_count_launch()
{
    if (g_capturing_flag_for_count()) ++g_capture_count;
    else g_launches.fetch_add(1, std::memory_order_relaxed);
}
void gp_count_launches(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

extern "C" int64_t gp_launch_count(void) { return (int64_t)g_launches.load(); }

void gp_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int gp_sm_count()
{
    if (g_sm_count == 0) {
        int dev = 0, sms = 0;
        if (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0)
            g_sm_count = sms;
        else
            return 148;
    }
    return g_sm_count;
}

const GpEnv &gp_env()
{
    static const GpEnv env = [] {
        auto geti = [](const char *name, int dflt) {
            const char *v = getenv(name);
            return v ? atoi(v) : dflt;
        };
        GpEnv e;
        e.use_graph = geti("GP_USE_GRAPH", 1);
        e.bfs_trace = getenv("GP_BFS_TRACE") != nullptr;
        e.xchg_grid = geti("GP_XCHG_GRID", 0);
        e.xchg_debug = geti("GP_XCHG_DEBUG", 0);
        e.stage_events = geti("GP_STAGE_EVENTS", 0);
        e.pdl = geti("GP_PDL", 1);
        e.csr_trace = geti("GP_CSR_TRACE", 0);
        e.nvtx = geti("GP_NVTX", 1);
        return e;
    }();  // function-local static: initialised once, thread-safe
    return env;
}

uint64_t gp_next_uid()
{
    static std::atomic<uint64_t> next{1};
    return next.fetch_add(1, std::memory_order_relaxed);
}

GpRange::GpRange(const char *name) : on(gp_env().nvtx != 0)
{
    if (on) nvtxRangePushA(name);
}
GpRange::~GpRange()
{
    if (on) nvtxRangePop();
}

extern "C" int gp_abi_version(void) { return GP_ABI_VERSION; }

extern "C" const char *gp_last_error(void) { return g_err; }

extern "C" const char *gp_status_string(int status)
{
    switch (status) {
        case GP_OK: return "ok";
        case GP_ERR_INVALID: return "invalid argument";
        case GP_ERR_CUDA: return "CUDA runtime error";
        case GP_ERR_OOM: return "out of memory";
        case GP_ERR_INDEX_RANGE: return "index outside [0, num_nodes)";
        case GP_ERR_LEVEL_OVERFLOW: return "hop distance does not fit uint16";
        case GP_ERR_UNSUPPORTED: return "unsupported size or option";
        case GP_ERR_NOT_CONVERGED: return "power iteration failed to converge";
        case GP_ERR_NO_DEVICE: return "no usable CUDA device";
        default: return "unknown status";
    }
}

extern "C" int gp_device_info(int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor, char *name,
                              int64_t name_cap)
{
    int dev = 0, count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        cudaGetLastError();
        gp_set_error("no CUDA device is visible to this process");
        return GP_ERR_NO_DEVICE;
    }
    GP_CUDA_CHECK(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    GP_CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    if (name && name_cap > 0) {
        strncpy(name, prop.name, (size_t)name_cap - 1);
        name[name_cap - 1] = 0;
    }
    return GP_OK;
}

// ------------------------------------------------------------------------------------------
// One-call host path.  A small cache keeps the handles, device staging and the stream alive
// between calls of the same shape so repeated calls pay no allocation.
// The state of the one-call host entry lives in an explicit context the caller may own (gp_ctx_create): handles,
// device staging, a stream and the pinned ring.  Two host threads with two contexts share nothing but the device;
// gp_geodesic_embed_host without a context uses one process-wide default context behind a mutex.
struct gp_ctx {
    std::mutex mutex;
    int64_t n = -1, e_cap = -1, k_cap = -1;
    uint32_t flags = 0;
    gp_csr *csr = nullptr;
    gp_msbfs *bfs = nullptr;
    int64_t *d_edges = nullptr;
    int64_t *d_anchors = nullptr;
    float *d_feat = nullptr;
    uint16_t *d_hops = nullptr;
    cudaStream_t stream = nullptr;
    // pageable outputs: two pinned 8 MB ring slots; the GPU fills one while the host scatters the other into the
    // caller's rows (no N*K*4-byte pinned allocation, no second pass over the whole block)
    float *h_ring[2] = {nullptr, nullptr};
    cudaEvent_t ring_ev[2] = {nullptr, nullptr};

    void release()
    {
        gp_msbfs_free(bfs);
        gp_csr_free(csr);
        cudaFree(d_edges);
        cudaFree(d_anchors);
        cudaFree(d_feat);
        cudaFree(d_hops);
        bfs = nullptr;
        csr = nullptr;
        d_edges = nullptr;
        d_anchors = nullptr;
        d_feat = nullptr;
        d_hops = nullptr;
        n = e_cap = k_cap = -1;
    }
};

typedef gp_ctx HostCtx;

namespace {

HostCtx &default_ctx()
{
    static HostCtx ctx;
    return ctx;
}

int ensure_ctx(HostCtx &c, int64_t n, int64_t e, int64_t k, uint32_t flags)
{
    if (c.stream == nullptr) {
        GP_TRY(gp_device_info(nullptr, nullptr, nullptr, nullptr, 0));  // GP_ERR_NO_DEVICE, not a raw runtime error
        GP_CUDA_CHECK(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
    }
    if (c.n == n && c.flags == flags && e <= c.e_cap && k <= c.k_cap) return GP_OK;
    c.release();
    GP_TRY(gp_csr_create(n, e, flags, &c.csr));
    GP_TRY(gp_msbfs_create(c.csr, k, &c.bfs));
    GP_CUDA_CHECK(cudaMalloc(&c.d_edges, sizeof(int64_t) * (size_t)std::max<int64_t>(2 * e, 2)));
    GP_CUDA_CHECK(cudaMalloc(&c.d_anchors, sizeof(int64_t) * (size_t)std::max<int64_t>(k, 1)));
    GP_CUDA_CHECK(cudaMalloc(&c.d_feat, sizeof(float) * (size_t)std::max<int64_t>(n * k, 1)));
    GP_CUDA_CHECK(cudaMalloc(&c.d_hops, sizeof(uint16_t) * (size_t)std::max<int64_t>(n * k, 1)));
    c.n = n;
    c.e_cap = e;
    c.k_cap = k;
    c.flags = flags;
    return GP_OK;
}

// ---- host-side row copies (concat_into_features, utils.py:129-135, for host buffers) ----------------
// The copy of x into columns [0, F) of the [N, F + K] result is the longest leg of the host entry point
// (178 MB at Flickr size against 91 MB of PCIe traffic), so it runs on a persistent pool of worker
// threads (no thread creation per call) and writes with non-temporal stores (no read-for-ownership of
// the destination lines: one third less memory traffic).
class HostPool {
public:
    static HostPool &get()
    {
        static HostPool pool;
        return pool;
    }
    // fn(first_row, last_row) over [0, rows) in chunks, on all workers plus the caller
    void parallel_rows(int64_t rows, int64_t chunk, const std::function<void(int64_t, int64_t)> &fn)
    {
        // The workers exist only in the process that created them: after fork() (DataLoader workers,
        // multiprocessing) the child copies the rows itself.  A second caller does not queue behind a running
        // job either (two contexts on two threads must not serialise): it copies on its own thread.
        std::unique_lock<std::mutex> run_lock(run_mutex_, std::try_to_lock);
        if (getpid() != owner_pid_ || !run_lock.owns_lock()) {
            fn(0, rows);
            return;
        }
        {
            std::lock_guard<std::mutex> lk(m_);
            fn_ = &fn;
            rows_ = rows;
            chunk_ = chunk;
            next_.store(0);
            pending_ = (int)workers_.size();
            ++epoch_;
        }
        cv_.notify_all();
        work();
        std::unique_lock<std::mutex> lk(m_);
        done_cv_.wait(lk, [&] { return pending_ == 0; });
        fn_ = nullptr;
    }

private:
    HostPool() : owner_pid_(getpid())
    {
        int nt = (int)std::min<unsigned>(std::max(1u, std::thread::hardware_concurrency()), 16u) - 1;
        for (int t = 0; t < nt; ++t) workers_.emplace_back([this] { loop(); });
    }
    ~HostPool()
    {
        if (getpid() != owner_pid_) {  // forked child: the worker threads were never copied, nothing to join
            for (auto &t : workers_) t.detach();
            return;
        }
        {
            std::lock_guard<std::mutex> lk(m_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto &t : workers_) t.join();
    }
    void work()
    {
        for (;;) {
            const int64_t r0 = next_.fetch_add(chunk_);
            if (r0 >= rows_) break;
            (*fn_)(r0, std::min(rows_, r0 + chunk_));
        }
    }
    void loop()
    {
        uint64_t seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return stop_ || epoch_ != seen; });
                if (stop_) return;
                seen = epoch_;
            }
            work();
            {
                std::lock_guard<std::mutex> lk(m_);
                if (--pending_ == 0) done_cv_.notify_one();
            }
        }
    }
    const pid_t owner_pid_;
    std::vector<std::thread> workers_;
    std::mutex m_, run_mutex_;
    std::condition_variable cv_, done_cv_;
    const std::function<void(int64_t, int64_t)> *fn_ = nullptr;
    std::atomic<int64_t> next_{0};
    int64_t rows_ = 0, chunk_ = 1;
    int pending_ = 0;
    uint64_t epoch_ = 0;
    bool stop_ = false;
};

inline void copy_row_streaming(const float *src, float *dst, size_t n)
{
#if defined(__x86_64__) || defined(_M_X64)
    size_t i = 0;
    while (i < n && (reinterpret_cast<uintptr_t>(dst + i) & 15u)) {
        dst[i] = src[i];
        ++i;
    }
    for (; i + 16 <= n; i += 16) {
        const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i));
        const __m128i b = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i + 4));
        const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i + 8));
        const __m128i d = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i + 12));
        _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i), a);
        _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i + 4), b);
        _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i + 8), c);
        _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i + 12), d);
    }
    for (; i + 4 <= n; i += 4)
        _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i), _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i)));
    for (; i < n; ++i) dst[i] = src[i];
#else
    memcpy(dst, src, n * sizeof(float));
#endif
}

void copy_rows_parallel(const float *src, int64_t ld_src, float *dst, int64_t ld_dst, int64_t rows,
                        int64_t cols)
{
    if (rows <= 0 || cols <= 0) return;
    auto work = [=](int64_t r0, int64_t r1) {
        for (int64_t r = r0; r < r1; ++r) copy_row_streaming(src + r * ld_src, dst + r * ld_dst, (size_t)cols);
#if defined(__x86_64__) || defined(_M_X64)
        _mm_sfence();
#endif
    };
    if (rows * cols < (1 << 20)) {
        work(0, rows);
        return;
    }
    HostPool::get().parallel_rows(rows, 512, work);
}

}  // namespace

// ------------------------------------------------------------------------------------------
// Whole device pipeline as one call, replayed from a CUDA graph: csr build -> ms-bfs -> epilogue is
// ~25 small launches whose gaps rival their run time at Flickr size.  The first call with a given
// argument tuple runs eagerly, the second is stream-captured (on a private stream: the legacy
// default stream cannot capture), later calls are a single cudaGraphLaunch.
namespace {

struct PipeKey {
    uint64_t csr, bfs, xchg;  // handle uids (addresses are reused by the allocator, uids are not)
    const void *ei, *anchors, *x, *out;
    int64_t e, k, f, ldx, ldo, coff, parity;
    bool operator==(const PipeKey &o) const { return memcmp(this, &o, sizeof(PipeKey)) == 0; }
};

struct PipeEntry {
    PipeKey key;
    cudaGraphExec_t exec = nullptr;
    int seen = 0;
    int kernels = 0;  // kernel nodes in the captured graph
    bool has_events = false;  // captured with the stage-event nodes
    uint64_t stamp = 0;
};

}  // namespace

// The captured pipelines of one MS-BFS handle (the handle owns them: no process-wide cache, no global lock; a
// handle is used by one thread at a time, like a stream).
struct gp_pipe_cache {
    std::vector<PipeEntry> pipes;
    cudaStream_t capture_stream = nullptr;
    uint64_t clock = 0;
};

namespace {

thread_local bool g_capturing = false;  // a capture belongs to the thread that runs it

int run_pipeline_eager(gp_csr *csr, gp_msbfs *bfs, const int64_t *d_ei, int64_t e, const int64_t *d_anchors,
                       int64_t k, const float *d_x, int64_t f, int64_t ldx, float *d_out, int64_t ldo,
                       int64_t coff, cudaStream_t s, gp_exchange *xchg = nullptr, int parity = 0)
{
    // concat_into_features' copy of x (utils.py:133-134) stays fused in the epilogue kernel.  It depends on neither the
    // csr build nor the traversal, but run beside them on a side stream it slows them by about its own duration,
    // whatever moves the rows (profiles/r02_notes.md).
    // stage clocks of the step (gp_pipeline_stage_ms): inside a capture these become event-record nodes
    const unsigned ev_flags = gp_is_capturing() ? cudaEventRecordExternal : cudaEventRecordDefault;
    const bool stage_events = gp_stage_events_on(bfs);
    if (stage_events) GP_CUDA_CHECK(cudaEventRecordWithFlags(bfs->ev_pipe0, s, ev_flags));
    {
        GpRange r("graphpope:csr_build");
        GP_TRY(gp_csr_build(csr, d_ei, e, s));
    }
    {
        GpRange r("graphpope:msbfs");
        GP_TRY(gp_msbfs_run(bfs, d_anchors, k, s));
    }
    GpRange r(xchg != nullptr ? "graphpope:exchange_decode" : "graphpope:epilogue");
    if (xchg != nullptr) GP_TRY(gp_exchange_launch(xchg, parity, d_x, f, ldx, d_out, ldo, coff, s));
    else if (d_out != nullptr) GP_TRY(gp_msbfs_features(bfs, d_x, f, ldx, d_out, ldo, coff, s));  // NULL: empty output
    if (stage_events) GP_CUDA_CHECK(cudaEventRecordWithFlags(bfs->ev_pipe1, s, ev_flags));
    bfs->pipe_timed = stage_events;
    return GP_OK;
}

}  // namespace

bool gp_is_capturing() { return g_capturing; }

// Called when an MS-BFS handle is freed: its captured pipelines go with it.  (csr / exchange handles are referred to
// by uid, so a graph that names a freed one can never be matched again; it is dropped with its bfs handle.)
void gp_pipe_cache_free(gp_pipe_cache *pc)
{
    if (pc == nullptr) return;
    for (auto &e : pc->pipes)
        if (e.exec) cudaGraphExecDestroy(e.exec);
    if (pc->capture_stream) cudaStreamDestroy(pc->capture_stream);
    delete pc;
}

uint64_t gp_exchange_uid(const gp_exchange *x);

static int geodesic_run_impl(gp_csr_t *csr, gp_msbfs_t *bfs, const int64_t *d_edge_index, int64_t num_edges,
                             const int64_t *d_anchors, int64_t num_anchors, const float *d_x,
                             int64_t num_features, int64_t ld_x, float *d_out, int64_t ld_out,
                             int64_t col_offset, gp_stream_t stream_, gp_exchange *xchg, int parity)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    GP_REQUIRE(csr != nullptr && bfs != nullptr, GP_ERR_INVALID, "gp_geodesic_run: NULL handle");
    if (!gp_env().use_graph || csr->num_nodes == 0 || num_anchors == 0)
        return run_pipeline_eager(csr, bfs, d_edge_index, num_edges, d_anchors, num_anchors, d_x, num_features, ld_x,
                                  d_out, ld_out, col_offset, stream, xchg, parity);
    if (bfs->pipe_cache == nullptr) bfs->pipe_cache = new (std::nothrow) gp_pipe_cache();
    GP_REQUIRE(bfs->pipe_cache != nullptr, GP_ERR_OOM, "gp_geodesic_run: host allocation failed");
    gp_pipe_cache &pc = *bfs->pipe_cache;
    PipeKey key;
    memset(&key, 0, sizeof(key));
    key.csr = csr->uid; key.bfs = bfs->uid; key.ei = d_edge_index; key.anchors = d_anchors; key.x = d_x; key.out = d_out;
    key.e = num_edges; key.k = num_anchors; key.f = num_features; key.ldx = ld_x; key.ldo = ld_out; key.coff = col_offset;
    key.xchg = xchg ? gp_exchange_uid(xchg) : 0; key.parity = parity;
    PipeEntry *ent = nullptr;
    for (auto &p : pc.pipes)
        if (p.key == key) ent = &p;
    if (ent == nullptr) {
        if (pc.pipes.size() >= 8) {  // evict the least recently used graph
            size_t lru = 0;
            for (size_t i = 1; i < pc.pipes.size(); ++i)
                if (pc.pipes[i].stamp < pc.pipes[lru].stamp) lru = i;
            if (pc.pipes[lru].exec) cudaGraphExecDestroy(pc.pipes[lru].exec);
            pc.pipes.erase(pc.pipes.begin() + lru);
        }
        pc.pipes.emplace_back();
        ent = &pc.pipes.back();
        ent->key = key;
    }
    ent->stamp = ++pc.clock;
    ent->seen += 1;
    if (ent->exec == nullptr && ent->seen == 2) {
        if (pc.capture_stream == nullptr)
            GP_CUDA_CHECK(cudaStreamCreateWithFlags(&pc.capture_stream, cudaStreamNonBlocking));
        cudaGraph_t graph = nullptr;
        if (cudaStreamBeginCapture(pc.capture_stream, cudaStreamCaptureModeRelaxed) == cudaSuccess) {
            g_capturing = true;
            g_capture_count = 0;
            const int rc = run_pipeline_eager(csr, bfs, d_edge_index, num_edges, d_anchors, num_anchors, d_x,
                                              num_features, ld_x, d_out, ld_out, col_offset, pc.capture_stream, xchg,
                                              parity);
            g_capturing = false;
            ent->kernels = g_capture_count;
            ent->has_events = bfs->pipe_timed;
            const cudaError_t ce = cudaStreamEndCapture(pc.capture_stream, &graph);
            if (rc == GP_OK && ce == cudaSuccess && graph != nullptr) {
                if (cudaGraphInstantiate(&ent->exec, graph, 0) != cudaSuccess) ent->exec = nullptr;
            }
            if (graph) cudaGraphDestroy(graph);
        }
        cudaGetLastError();  // a failed capture must not poison later calls; fall back to eager launches
        if (ent->exec == nullptr) ent->seen = 1 << 20;  // do not retry
    }
    if (ent->exec != nullptr) {
        csr->in_built = false;  // the replay rebuilds the out-edge CSR from the (possibly changed) edge buffer
        csr->num_input_edges = num_edges;
        csr->built = true;
        gp_msbfs_layout(bfs, num_anchors);  // the handle may have run another anchor count since the capture
        bfs->ran = true;
        bfs->pipe_timed = bfs->kernel_timed = ent->has_events;
        gp_count_launches(ent->kernels);  // kernels inside the graph
        GpRange r("graphpope:pipeline_graph_replay");
        GP_CUDA_CHECK(cudaGraphLaunch(ent->exec, stream));
        return GP_OK;
    }
    return run_pipeline_eager(csr, bfs, d_edge_index, num_edges, d_anchors, num_anchors, d_x, num_features, ld_x,
                              d_out, ld_out, col_offset, stream, xchg, parity);
}

extern "C" int gp_geodesic_run(gp_csr_t *csr, gp_msbfs_t *bfs, const int64_t *d_edge_index, int64_t num_edges,
                               const int64_t *d_anchors, int64_t num_anchors, const float *d_x,
                               int64_t num_features, int64_t ld_x, float *d_out, int64_t ld_out,
                               int64_t col_offset, gp_stream_t stream_)
{
    GP_REQUIRE(csr != nullptr && bfs != nullptr, GP_ERR_INVALID, "gp_geodesic_run: NULL handle");
    // an empty [N, F+K] tensor may have no storage, so d_out may be NULL only when there is nothing to write
    const bool writes = csr->num_nodes > 0 && (num_anchors > 0 || (d_x != nullptr && num_features > 0));
    GP_REQUIRE(d_out != nullptr || !writes, GP_ERR_INVALID, "gp_geodesic_run: d_out is NULL");
    return geodesic_run_impl(csr, bfs, d_edge_index, num_edges, d_anchors, num_anchors, d_x, num_features, ld_x, d_out,
                             ld_out, col_offset, stream_, nullptr, 0);
}

// Sharded step as one call: csr build + MS-BFS of this rank's anchors + the fused push exchange / decode kernel
// (gp_exchange.cu), graph-replayed per step parity.  Collective: every rank of the exchange calls it once per step.
extern "C" int gp_geodesic_run_exchange(gp_csr_t *csr, gp_msbfs_t *bfs, gp_exchange_t *xchg, const int64_t *d_edge_index,
                                        int64_t num_edges, const int64_t *d_anchors, int64_t num_anchors,
                                        const float *d_x, int64_t num_features, int64_t ld_x, float *d_out,
                                        int64_t ld_out, int64_t col_offset, gp_stream_t stream_)
{
    GP_REQUIRE(xchg != nullptr && d_out != nullptr, GP_ERR_INVALID, "gp_geodesic_run_exchange: NULL argument");
    GP_REQUIRE(csr != nullptr && csr->num_nodes > 0 && num_anchors > 0, GP_ERR_INVALID,
               "gp_geodesic_run_exchange: empty graph or shard");
    return geodesic_run_impl(csr, bfs, d_edge_index, num_edges, d_anchors, num_anchors, d_x, num_features, ld_x, d_out,
                             ld_out, col_offset, stream_, xchg, gp_exchange_next_parity(xchg));
}

extern "C" int gp_concat_x(const float *d_x, int64_t num_nodes, int64_t num_features, int64_t ld_x, float *d_out,
                           int64_t ld_out, gp_stream_t stream)
{
    GP_REQUIRE(num_nodes >= 0 && num_features >= 0 && ld_x >= num_features && ld_out >= num_features, GP_ERR_INVALID,
               "gp_concat_x: inconsistent sizes");
    if (num_nodes == 0 || num_features == 0) return GP_OK;
    GP_REQUIRE(d_x != nullptr && d_out != nullptr, GP_ERR_INVALID, "gp_concat_x: NULL argument");
    if (gp_xcopy_tma_ok(d_x, num_features, ld_x, d_out, ld_out))
        return gp_launch_xcopy_tma(d_x, num_nodes, num_features, ld_x, d_out, ld_out, (cudaStream_t)stream);
    GP_CUDA_CHECK(cudaMemcpy2DAsync(d_out, (size_t)ld_out * sizeof(float), d_x, (size_t)ld_x * sizeof(float),
                                    (size_t)num_features * sizeof(float), (size_t)num_nodes,
                                    cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return GP_OK;
}

// Round 1's pull exchange was removed (its other four entry points are in gp_epilogue.cu); kept so that programs
// built against ABI version 1 still link.
extern "C" int gp_geodesic_run_packed(gp_csr_t *, gp_msbfs_t *, const int64_t *, int64_t, const int64_t *, int64_t,
                                      int32_t, gp_stream_t)
{
    GP_REQUIRE(false, GP_ERR_UNSUPPORTED, "gp_geodesic_run_packed: removed, use gp_geodesic_run_exchange");
}

extern "C" int gp_host_concat(const float *h_x, int64_t num_features, const float *h_block, int64_t block_cols,
                              int64_t num_nodes, float *h_out, int64_t ld_out)
{
    GP_REQUIRE(num_nodes >= 0 && num_features >= 0 && block_cols >= 0 && ld_out >= num_features + block_cols,
               GP_ERR_INVALID, "gp_host_concat: inconsistent sizes");
    GP_REQUIRE(h_out != nullptr || num_nodes == 0, GP_ERR_INVALID, "gp_host_concat: out is NULL");
    if (h_x != nullptr) copy_rows_parallel(h_x, num_features, h_out, ld_out, num_nodes, num_features);
    if (h_block != nullptr) copy_rows_parallel(h_block, block_cols, h_out + num_features, ld_out, num_nodes, block_cols);
    return GP_OK;
}

extern "C" int gp_block_to_host(const float *d_block, int64_t num_nodes, int64_t block_cols, float *h_out,
                                int64_t ld_out, int64_t col_offset, gp_stream_t stream_)
{
    GP_REQUIRE(num_nodes >= 0 && block_cols >= 0 && col_offset >= 0 && ld_out >= col_offset + block_cols, GP_ERR_INVALID,
               "gp_block_to_host: inconsistent sizes");
    if (num_nodes == 0 || block_cols == 0) return GP_OK;
    GP_REQUIRE(d_block != nullptr && h_out != nullptr, GP_ERR_INVALID, "gp_block_to_host: NULL argument");
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, h_out) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    GP_REQUIRE(pinned, GP_ERR_INVALID, "gp_block_to_host: h_out must be pinned host memory");
    GP_CUDA_CHECK(cudaMemcpy2DAsync(h_out + col_offset, sizeof(float) * (size_t)ld_out, d_block,
                                    sizeof(float) * (size_t)block_cols, sizeof(float) * (size_t)block_cols,
                                    (size_t)num_nodes, cudaMemcpyDeviceToHost, (cudaStream_t)stream_));
    return GP_OK;
}

extern "C" int gp_ctx_create(gp_ctx_t **out)
{
    GP_REQUIRE(out != nullptr, GP_ERR_INVALID, "gp_ctx_create: out is NULL");
    *out = new (std::nothrow) gp_ctx();
    GP_REQUIRE(*out != nullptr, GP_ERR_OOM, "gp_ctx_create: host allocation failed");
    return GP_OK;
}

extern "C" int gp_ctx_free(gp_ctx_t *ctx)
{
    if (ctx == nullptr) return GP_OK;
    ctx->release();
    for (int i = 0; i < 2; ++i) {
        if (ctx->h_ring[i]) cudaFreeHost(ctx->h_ring[i]);
        if (ctx->ring_ev[i]) cudaEventDestroy(ctx->ring_ev[i]);
    }
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return GP_OK;
}

extern "C" int gp_geodesic_embed_host(const int64_t *h_edge_index, int64_t num_edges, int64_t num_nodes,
                                      uint32_t csr_flags, const int64_t *h_anchors, int64_t num_anchors,
                                      const float *h_x, int64_t num_features, float *h_out, int64_t ld_out,
                                      int64_t col_offset, uint16_t *h_hops, gp_msbfs_stats_t *stats)
{
    return gp_geodesic_embed_host_ctx(&default_ctx(), h_edge_index, num_edges, num_nodes, csr_flags, h_anchors,
                                      num_anchors, h_x, num_features, h_out, ld_out, col_offset, h_hops, stats);
}

extern "C" int gp_geodesic_embed_host_ctx(gp_ctx_t *ctx, const int64_t *h_edge_index, int64_t num_edges,
                                          int64_t num_nodes, uint32_t csr_flags, const int64_t *h_anchors,
                                          int64_t num_anchors, const float *h_x, int64_t num_features, float *h_out,
                                          int64_t ld_out, int64_t col_offset, uint16_t *h_hops, gp_msbfs_stats_t *stats)
{
    GP_REQUIRE(ctx != nullptr, GP_ERR_INVALID, "gp_geodesic_embed_host_ctx: ctx is NULL");
    GP_REQUIRE(num_edges >= 0 && num_nodes >= 0 && num_anchors >= 0 && num_features >= 0, GP_ERR_INVALID,
               "gp_geodesic_embed_host: negative size");
    GP_REQUIRE(num_edges == 0 || h_edge_index != nullptr, GP_ERR_INVALID, "edge_index is NULL");
    GP_REQUIRE(num_anchors == 0 || h_anchors != nullptr, GP_ERR_INVALID, "anchors is NULL");
    GP_REQUIRE(h_out != nullptr || num_nodes == 0 || (num_anchors == 0 && h_x == nullptr), GP_ERR_INVALID,
               "out is NULL");
    GP_REQUIRE(col_offset >= 0 && ld_out >= col_offset + num_anchors && (h_x == nullptr || col_offset >= num_features),
               GP_ERR_INVALID, "gp_geodesic_embed_host: inconsistent ld_out / col_offset");
    HostCtx &c = *ctx;
    std::lock_guard<std::mutex> lock(c.mutex);  // a context serves one call at a time; contexts are independent
    GP_TRY(ensure_ctx(c, num_nodes, num_edges, num_anchors, csr_flags));
    GpRange range("graphpope:embed_host");
    cudaStream_t s = c.stream;
    if (num_edges > 0)
        GP_CUDA_CHECK(cudaMemcpyAsync(c.d_edges, h_edge_index, sizeof(int64_t) * 2 * (size_t)num_edges,
                                      cudaMemcpyHostToDevice, s));
    if (num_anchors > 0)
        GP_CUDA_CHECK(cudaMemcpyAsync(c.d_anchors, h_anchors, sizeof(int64_t) * (size_t)num_anchors,
                                      cudaMemcpyHostToDevice, s));
    GP_TRY(gp_csr_build(c.csr, c.d_edges, num_edges, s));
    GP_TRY(gp_msbfs_run(c.bfs, c.d_anchors, num_anchors, s));
    if (num_nodes > 0 && num_anchors > 0) {
        GP_TRY(gp_msbfs_features(c.bfs, nullptr, 0, 0, c.d_feat, num_anchors, 0, s));
        if (h_hops) GP_TRY(gp_msbfs_hops_u16(c.bfs, c.d_hops, num_anchors, 0, s));
    }
    // The feature block lands in columns [col_offset, col_offset + K).  A pinned h_out takes a
    // strided DMA directly; a pageable one goes through a pinned staging block (one contiguous DMA,
    // then a threaded row scatter) because a pageable 2-D copy degenerates into N tiny transfers.
    const bool have_block = num_nodes > 0 && num_anchors > 0;
    bool staged = false;
    if (have_block) {
        cudaPointerAttributes attr;
        const bool pinned = cudaPointerGetAttributes(&attr, h_out) == cudaSuccess && attr.type == cudaMemoryTypeHost;
        cudaGetLastError();
        if (pinned) {
            GP_CUDA_CHECK(cudaMemcpy2DAsync(h_out + col_offset, sizeof(float) * (size_t)ld_out, c.d_feat,
                                            sizeof(float) * (size_t)num_anchors, sizeof(float) * (size_t)num_anchors,
                                            (size_t)num_nodes, cudaMemcpyDeviceToHost, s));
        } else {
            staged = true;  // ring-buffered below, after the hop matrix has been queued behind the block
        }
        if (h_hops)
            GP_CUDA_CHECK(cudaMemcpyAsync(h_hops, c.d_hops, sizeof(uint16_t) * (size_t)(num_nodes * num_anchors),
                                          cudaMemcpyDeviceToHost, s));
    }
    // concat_into_features (utils.py:129-135): x goes into columns [0, F) on the host, while the
    // GPU works.
    if (staged) {
        // Pageable h_out: rows [r0, r1) of the device block go to a pinned ring slot (one contiguous DMA), the host
        // scatters the previous slot into the caller's rows meanwhile.  The copy of x runs after the first two DMAs
        // have been queued, so it overlaps them as well.
        constexpr size_t RING_BYTES = 8u << 20;
        for (int i = 0; i < 2; ++i) {
            if (c.h_ring[i] == nullptr) GP_CUDA_CHECK(cudaMallocHost((void **)&c.h_ring[i], RING_BYTES));
            if (c.ring_ev[i] == nullptr) GP_CUDA_CHECK(cudaEventCreateWithFlags(&c.ring_ev[i], cudaEventDisableTiming));
        }
        const int64_t rows_per = std::max<int64_t>(1, (int64_t)(RING_BYTES / (sizeof(float) * (size_t)num_anchors)));
        const int64_t chunks = gp_ceil_div(num_nodes, rows_per);
        auto enqueue = [&](int64_t i) -> int {
            const int64_t r0 = i * rows_per, r1 = std::min(num_nodes, r0 + rows_per);
            GP_CUDA_CHECK(cudaMemcpyAsync(c.h_ring[i & 1], c.d_feat + r0 * num_anchors,
                                          sizeof(float) * (size_t)((r1 - r0) * num_anchors), cudaMemcpyDeviceToHost, s));
            GP_CUDA_CHECK(cudaEventRecord(c.ring_ev[i & 1], s));
            return GP_OK;
        };
        GP_REQUIRE((size_t)num_anchors * sizeof(float) <= RING_BYTES, GP_ERR_UNSUPPORTED,
                   "gp_geodesic_embed_host: more than %zu anchors need a pinned output buffer", RING_BYTES / sizeof(float));
        for (int64_t i = 0; i < std::min<int64_t>(2, chunks); ++i) GP_TRY(enqueue(i));
        if (h_x != nullptr) copy_rows_parallel(h_x, num_features, h_out, ld_out, num_nodes, num_features);
        for (int64_t i = 0; i < chunks; ++i) {
            const int64_t r0 = i * rows_per, r1 = std::min(num_nodes, r0 + rows_per);
            GP_CUDA_CHECK(cudaEventSynchronize(c.ring_ev[i & 1]));
            copy_rows_parallel(c.h_ring[i & 1], num_anchors, h_out + r0 * ld_out + col_offset, ld_out, r1 - r0, num_anchors);
            if (i + 2 < chunks) GP_TRY(enqueue(i + 2));
        }
    } else if (h_x != nullptr) {
        copy_rows_parallel(h_x, num_features, h_out, ld_out, num_nodes, num_features);
    }
    gp_msbfs_stats_t local;
    GP_TRY(gp_msbfs_stats(c.bfs, stats ? stats : &local, s));  // synchronises and reports device errors
    return GP_OK;
}
