// gp_common.cuh — shared host/device helpers for the graphpope_b200 kernels (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string.h>

#include "../../include/graphpope_b200.h"

typedef unsigned long long u64;
typedef unsigned int u32;

// ---------------------------------------------------------------- host-side errors
void gp_set_error(const char *fmt, ...);

#define GP_CUDA_CHECK(expr)                                                              \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess) {                                                         \
            gp_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),         \
                         __FILE__, __LINE__);                                            \
            return (_e == cudaErrorMemoryAllocation) ? GP_ERR_OOM : GP_ERR_CUDA;         \
        }                                                                                \
    } while (0)

#define GP_REQUIRE(cond, status, ...)                                                    \
    do {                                                                                 \
        if (!(cond)) {                                                                   \
            gp_set_error(__VA_ARGS__);                                                   \
            return (status);                                                             \
        }                                                                                \
    } while (0)

#define GP_TRY(expr)                                                                     \
    do {                                                                                 \
        int _s = (expr);                                                                 \
        if (_s != GP_OK) return _s;                                                      \
    } while (0)

static inline int64_t gp_ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Device-latched error bits (status words live in handle-owned device memory).
enum : int { GP_DEV_ERR_EDGE_RANGE = 1, GP_DEV_ERR_ANCHOR_RANGE = 2, GP_DEV_ERR_LEVEL_OVERFLOW = 4 };

int gp_sm_count();  // cached multiProcessorCount of the current device

// Experiment / diagnostic switches, read from the environment ONCE per process (first use, thread-safe) and passed
// around as plain data afterwards: no getenv on any call path, no function-local caches.
struct GpEnv {
    int use_graph;       // GP_USE_GRAPH (default 1): replay the fused pipeline from a CUDA graph
    int bfs_trace;       // GP_BFS_TRACE: per-level clocks
    int xchg_grid;       // GP_XCHG_GRID: cap on the exchange kernel's grid (tests: several ranks on one GPU)
    int xchg_debug;      // GP_XCHG_DEBUG
    int stage_events;    // GP_STAGE_EVENTS (default 0): event NODES around csr / bfs / epilogue inside captured pipelines
    int pdl;             // GP_PDL (default 1): programmatic dependent launch inside the csr build
    int csr_trace;       // GP_CSR_TRACE: events after every launch of the csr build
    int nvtx;            // GP_NVTX (default 1): NVTX ranges around the stages
};
const GpEnv &gp_env();
uint64_t gp_next_uid();  // identity of a handle for the graph cache (addresses get reused, uids do not)

// NVTX range around a host-side stage (csr / bfs / exchange / epilogue / h2d / d2h); free when no tool is attached.
struct GpRange {
    explicit GpRange(const char *name);
    ~GpRange();
    bool on;
};

// Every kernel launch of the library goes through GP_LAUNCH so callers (bench.py) can report how
// many of OUR kernels ran inside a timed region (gp_launch_count in the ABI).
void gp_count_launch();
bool gp_is_capturing();            // true while gp_geodesic_run is stream-capturing the pipeline
#define GP_LAUNCH(kernel, grid, block, smem, stream, ...)                         \
    do {                                                                          \
        gp_count_launch();                                                        \
        kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);               \
    } while (0)

// Programmatic dependent launch (PDL): the kernel may be scheduled while its predecessor in the stream is still
// running (its prologue and launch latency overlap the predecessor's tail); it must call gp_pdl_wait() before it
// touches anything the predecessor wrote.  Used for the chain of small kernels of the csr build, whose run times
// rival the gaps between dependent launches.  Captured into CUDA graphs as programmatic edges.
#ifdef __CUDACC__
template <typename... KArgs, typename... Args>
static inline cudaError_t gp_launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                        Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = gp_env().pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
#define GP_LAUNCH_PDL(kernel, grid, block, smem, stream, ...)                                     \
    do {                                                                                          \
        gp_count_launch();                                                                        \
        GP_CUDA_CHECK(gp_launch_pdl(kernel, dim3(grid), dim3(block), (smem), (stream), __VA_ARGS__)); \
    } while (0)
#endif

// ---------------------------------------------------------------- device helpers
#ifdef __CUDACC__

// First statements of a kernel launched with GP_LAUNCH_PDL: let the successor be scheduled, then wait until the
// predecessor has completed and its writes are visible.  Both are no-ops for ordinary launches.
__device__ __forceinline__ void gp_pdl_enter()
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

constexpr u32 FULL_MASK = 0xFFFFFFFFu;

__device__ __forceinline__ u32 lane_id() { return threadIdx.x & 31u; }

__device__ __forceinline__ u64 shfl_xor_u64(u64 v, int m)
{
    u32 lo = (u32)v, hi = (u32)(v >> 32);
    lo = __shfl_xor_sync(FULL_MASK, lo, m);
    hi = __shfl_xor_sync(FULL_MASK, hi, m);
    return ((u64)hi << 32) | lo;
}

__device__ __forceinline__ u64 warp_or_u64(u64 v)
{
    u32 lo = __reduce_or_sync(FULL_MASK, (u32)v);
    u32 hi = __reduce_or_sync(FULL_MASK, (u32)(v >> 32));
    return ((u64)hi << 32) | lo;
}

__device__ __forceinline__ u32 ld_acquire_u32(const u32 *p)
{
    u32 v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ u32 ld_relaxed_u32(const u32 *p)
{
    u32 v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ void st_relaxed_u32(u32 *p, u32 v)
{
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

__device__ __forceinline__ void red_release_add_u32(u32 *p, u32 v)
{
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Grid-wide barrier for a cooperatively launched (co-resident) grid.  `counter`
// is a zero-initialised device word that only ever grows; `target` is the
// caller's running arrival target (per thread, all threads keep the same value).
__device__ __forceinline__ void grid_barrier(u32 *counter, u32 &target, u32 nblocks)
{
    target += nblocks;
    __syncthreads();
    if (threadIdx.x == 0) {
        red_release_add_u32(counter, 1u);
        // poll with relaxed loads (an acquire load invalidates this SM's L1 on every poll, which
        // would evict lines other CTAs on the SM are still using), then acquire once
        while (ld_relaxed_u32(counter) < target) {
        }
        (void)ld_acquire_u32(counter);
    }
    __syncthreads();
}

#endif  // __CUDACC__
