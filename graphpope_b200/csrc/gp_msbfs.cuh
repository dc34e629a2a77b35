// gp_msbfs.cuh — handle layout of the multi-source BFS (internal).
#pragma once

#include "gp_internal.h"

constexpr int GP_BFS_MAX_LANE_WORDS = 256;  // B * WB cap (K <= 16384 per GPU)
constexpr int GP_BFS_PLANES = 16;           // deep-hop distance bit planes (uint16 range)
constexpr int GP_BFS_LEVEL_ARRAYS = 15;     // hops 1..15 are recorded as write-once frontier arrays
constexpr int GP_BFS_CACHE_ITERS = 4;      // warp-iterations whose work items are cached in shared memory
constexpr int GP_BFS_MAP_SMEM_MAX = 64 * 1024;  // largest set of frontier bitmaps staged in shared memory
constexpr int GP_BFS_DONE_BATCHES = 8;     // batches that keep per-row "done" flags for cached items
constexpr int GP_MAX_RANKS = 8;             // GPUs of one NVSwitch node
constexpr int GP_BFS_RESULT_ARRAYS = 1 + GP_BFS_LEVEL_ARRAYS + GP_BFS_PLANES;  // 32
constexpr long long GP_BFS_TRACE_WORDS = 32ll * 160 * 4 * 32 * 4;  // levels * max warps * 4 slots

enum : int {
    GP_BFS_ST_MAX_LEVEL = 0,
    GP_BFS_ST_ERROR = 1,
    GP_BFS_ST_LEVELS = 2,
    GP_BFS_ST_WORDS = 8
};

struct gp_pipe_cache;  // captured pipelines of this handle (gp_api.cu)
void gp_pipe_cache_free(gp_pipe_cache *pc);

struct gp_msbfs {
    uint64_t uid = gp_next_uid();
    gp_pipe_cache *pipe_cache = nullptr;
    const gp_csr *csr = nullptr;
    int64_t num_nodes = 0;
    int64_t max_anchors = 0;
    int64_t cap_words_per_node = 0;  // lane words per node the buffers were sized for
    // configuration of the last run
    int64_t num_anchors = 0;
    int wb = 1;        // lane words per batch row (1, 2 or 4)
    int batches = 0;   // independent 64*wb-anchor batches
    bool ran = false;

    u64 *lane_buf = nullptr; // one allocation: seeds | R[0..31] | 3 deep frontiers (pointers below are set per run)
    void *scratch = nullptr; // one allocation: live | bar | counters | status | nzmap (cleared by one memset per run)
    size_t scratch_bytes = 0;
    u64 *seen = nullptr;     // result block R[0..31], each [batches][N][wb]; R[0] = reached mask (gp_msbfs.cu)
    u64 *fr_a = nullptr;     // three rotating frontiers for hops >= 16
    u64 *fr_b = nullptr;
    u64 *fr_c = nullptr;
    u64 *seeds = nullptr;    // hop-0 frontier
    u64 *live = nullptr;     // [3][GP_BFS_MAX_LANE_WORDS]
    u64 *hub_acc = nullptr;  // [batches][hub_capacity][wb] partial ORs of hub rows (zero between levels)
    u32 *hub_cnt = nullptr;  // [batches][hub_capacity] hub chunks arrived (zero between levels)
    u64 *bar = nullptr;      // grid barrier words
    u32 *nzmap = nullptr;    // [3][lane-word batches][ceil(N/32)] non-zero-row bitmaps of the last three frontiers
    int64_t nzwords = 0;     // ceil(N / 32)
    int map_smem_bytes = 0;  // shared memory the launch reserves for the maps (0: maps off for this size)
    int map_want_bytes = -1; // map size the cached launch configuration was computed for
    int64_t hub_capacity = 0;
    bool hub_zeroed = false;
    u64 *packed = nullptr;   // [2 slots][GP_PACKED_ARRAYS][cap words] exchange buffers (allocated on first pack)
    int *deep_flag = nullptr;  // device int: 1 if the last packed run had hops > 15 (packed format invalid)
    int *status = nullptr;      // [GP_BFS_ST_WORDS]
    u64 *counters = nullptr;    // [4] gathers issued, unused, %globaltimer at kernel entry and after the last level
    u64 *trace = nullptr;       // [32 levels][warps][4] phase clocks, only with GP_BFS_TRACE=1
    int grid_blocks = 0;
    int grid_cfg = -1;          // kernel variant (WB, MAPG) the cached grid size was computed for
    cudaEvent_t ev_start = nullptr, ev_stop = nullptr;  // bracket the persistent kernel alone
    cudaEvent_t ev_pipe0 = nullptr, ev_pipe1 = nullptr;  // first / last node of the last gp_geodesic_run pipeline
    bool pipe_timed = false;   // the last fused run recorded ev_pipe0 / ev_pipe1
    bool kernel_timed = false; // the last run recorded ev_start / ev_stop
    int stage_events = -1;     // event nodes inside CAPTURED pipelines: -1 = GP_STAGE_EVENTS (default off), 0 / 1 = set
};

void gp_msbfs_layout(gp_msbfs *h, int64_t num_anchors);
// Whether this launch records the stage events: always for eager launches (an event record costs ~1 us there), inside a
// stream capture only on request (an event-record NODE costs ~4 us of the replayed step: 246 -> 231 us without the four).
bool gp_stage_events_on(const gp_msbfs *h);

// Fused decode + concat epilogue over `num_ranks` plane sets (1 = local result).
struct GpDecodeParams {
    const u64 *planes0;        // result block of rank 0 (R[0..], gp_msbfs.cu), R[0] = reached mask
    long long rank_stride;     // words between consecutive ranks' result blocks
    long long plane_stride;    // words between consecutive arrays of a block
    int num_ranks;
    int num_arrays;            // leading arrays of R that are valid (1 + max hop, or 32 if deep); <0: from status
    const int *status;         // device status words (max level) when num_arrays < 0
    long long n;
    long long anchors_per_rank;
    int wb;
    const float *x;            // optional [N, ld_x]
    long long num_features, ld_x;
    float *out;
    long long ld_out, col_offset;
    // packed exchange format (gp_msbfs_pack): 5 arrays per rank = reached mask + 4 hop-index bit planes,
    // read in place from every rank's buffer (own memory or NVLink peer mappings)
    int packed;
    const u64 *rank_ptr[GP_MAX_RANKS];
};
constexpr int GP_PACKED_ARRAYS = 5;
int gp_launch_decode_features(const GpDecodeParams &p, cudaStream_t stream);
