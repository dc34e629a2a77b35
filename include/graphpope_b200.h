/*
 * graphpope_b200.h — C ABI of the B200-native GraphPOPE embedding-generation path.
 *
 * The reference (JeroendenBoef/GraphPOPE) is pure Python and has no FFI; this
 * header IS the drop-in boundary a maintainer binds from utils.py (ctypes stub in
 * INTEGRATION.md).  Each entry point cites the reference code it replaces
 * (file:line into the reference repository).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++/torch types.
 *   - Every function returns an int status (GP_OK == 0) and never throws;
 *     gp_last_error() returns a thread-local message for the last failure.
 *   - "d_" pointers are device pointers on the current CUDA device, "h_"
 *     pointers are host pointers.  The caller owns every buffer it passes in;
 *     the library owns only the opaque handles it creates.
 *   - gp_stream_t is a cudaStream_t (0 = the legacy default stream).  Calls
 *     documented "async" only enqueue work on that stream; results are valid
 *     after the stream is synchronised.  Calls documented "syncs" synchronise it.
 *   - Data-dependent failures detected on the device (edge index out of range,
 *     anchor out of range, hop distance not representable in uint16) are
 *     latched in the handle and reported by the next syncing call.
 *   - The header is strict C99; examples/embed_host.c is a complete caller of the
 *     one-call host entry with its expected rows (built and run by the test suite).
 */
#ifndef GRAPHPOPE_B200_H
#define GRAPHPOPE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GP_ABI_VERSION 1

typedef void *gp_stream_t;

enum gp_status {
    GP_OK = 0,
    GP_ERR_INVALID = 1,        /* bad argument (NULL, negative size, misuse)      */
    GP_ERR_CUDA = 2,           /* a CUDA runtime call failed                     */
    GP_ERR_OOM = 3,            /* device or host allocation failed               */
    GP_ERR_INDEX_RANGE = 4,    /* edge_index / anchor entry outside [0, N)       */
    GP_ERR_LEVEL_OVERFLOW = 5, /* a hop distance >= 65535 (uint16 sentinel)      */
    GP_ERR_UNSUPPORTED = 6,    /* size beyond what this build supports           */
    GP_ERR_NOT_CONVERGED = 7,  /* PageRank hit max_iter (networkx raises too)    */
    GP_ERR_NO_DEVICE = 8       /* no CUDA device / wrong architecture            */
};

#define GP_UNREACHABLE_U16 0xFFFFu

/* gp_csr_create flags */
#define GP_CSR_SYMMETRIZE 0x1u /* add the reverse of every edge (identity on the
                                  symmetric datasets; default off = reference
                                  DiGraph semantics, utils.py:121)                */

/* cdist modes: keys of dist_map, utils.py:158-162 */
enum gp_cdist_mode {
    GP_CDIST_COSINE_DISTANCE = 0,   /* 'distance'   -> sklearn cosine_distances   */
    GP_CDIST_COSINE_SIMILARITY = 1, /* 'similarity' -> sklearn cosine_similarity  */
    GP_CDIST_EUCLIDEAN = 2          /* 'euclidean'  -> sklearn euclidean_distances */
};

typedef struct gp_csr gp_csr_t;     /* de-duplicated digraph in CSR form          */
typedef struct gp_msbfs gp_msbfs_t; /* multi-source BFS workspace + results       */
typedef struct gp_exchange gp_exchange_t; /* exchange buffers of one rank (gp_exchange.cu) */
typedef struct gp_ctx gp_ctx_t;     /* state of the one-call host entry: handles, staging, stream */

typedef struct gp_csr_info {
    int64_t num_nodes;
    int64_t num_input_edges;  /* E columns given to gp_csr_build                 */
    int64_t num_edges;        /* directed edges after de-duplication (E')        */
    int64_t max_out_degree;
    int32_t is_symmetric;     /* 1 if every edge has its reverse                 */
    int32_t reserved;
} gp_csr_info_t;

typedef struct gp_msbfs_stats {
    int64_t num_anchors;
    int64_t lane_words;        /* uint64 lane words per node (64 anchors each)   */
    int32_t max_level;         /* largest finite hop distance                    */
    int32_t levels_run;        /* level sweeps executed                          */
    int32_t pull_levels;       /* = levels_run: every level pulls                */
    int32_t push_levels;       /* 0                                              */
    int64_t edges_examined;    /* neighbour lane-word gathers issued             */
    int64_t grid_blocks;       /* persistent grid size                           */
} gp_msbfs_stats_t;

/* ------------------------------------------------------------------ library */
int gp_abi_version(void);
const char *gp_last_error(void);
const char *gp_status_string(int status);
/* Device properties the host layer reports (SM count, name).  Syncs nothing. */
int gp_device_info(int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor, char *name, int64_t name_cap);
/* Number of kernels this library has launched in this process so far (bench.py's gpu_launches). */
int64_t gp_launch_count(void);

/* ------------------------------------------------------------------ CSR build
 * Replaces torch_geometric.utils.to_networkx(data) as called at utils.py:121
 * (and :27,33,39,45,51,57): nodes 0..N-1, parallel edges collapse, self-loops
 * kept, no symmetrisation unless GP_CSR_SYMMETRIZE.  Built on the device as a
 * counting sort by source row + a sort/unique inside every row (gp_csr.cu).     */
int gp_csr_create(int64_t num_nodes, int64_t edge_capacity, uint32_t flags, gp_csr_t **out);
/* async.  d_edge_index: int64 [2, num_edges] row-major (row 0 = src, row 1 = dst). */
int gp_csr_build(gp_csr_t *csr, const int64_t *d_edge_index, int64_t num_edges, gp_stream_t stream);
/* syncs.  Reports latched GP_ERR_INDEX_RANGE. */
int gp_csr_info(gp_csr_t *csr, gp_csr_info_t *info, gp_stream_t stream);
/* syncs.  Copies the CSR into caller device buffers: which = 0 out-edges (row u
 * lists v with u->v), 1 in-edges (row v lists u with u->v).  d_rowptr int32[N+1],
 * d_col int32[>= num_edges].  Rows are ascending and unique.                    */
int gp_csr_export(gp_csr_t *csr, int which, int32_t *d_rowptr, int32_t *d_col, gp_stream_t stream);
/* Diagnostics (GP_CSR_TRACE=1 in the environment): milliseconds of the stages of the last build (memsets, count, scan,
 * scatter, row sort, row scan, descriptors) from events recorded after every launch; *num = values written
 * (<= cap).  syncs.                                                                                          */
int gp_csr_trace_ms(gp_csr_t *csr, float *ms, int32_t cap, int32_t *num);
int gp_csr_free(gp_csr_t *csr);

/* ------------------------------------------------------------------ MS-BFS
 * Replaces shortest_path_length + all_pairs_shortest_path_length_parallel
 * (utils.py:64-81, 92-114): hops(node -> anchor_j) for every node and anchor,
 * as one multi-source BFS from the anchors over reversed edges, 64 anchors per
 * uint64 lane word, in one persistent kernel.                                   */
int gp_msbfs_create(const gp_csr_t *csr, int64_t max_anchors, gp_msbfs_t **out);
/* async.  d_anchors: int64[num_anchors] (duplicates allowed, utils.py:24). */
int gp_msbfs_run(gp_msbfs_t *bfs, const int64_t *d_anchors, int64_t num_anchors, gp_stream_t stream);
/* async.  Integer hop matrix: d_dist[node*ld + col_offset + j] = hops or 0xFFFF. */
int gp_msbfs_hops_u16(gp_msbfs_t *bfs, uint16_t *d_dist, int64_t ld, int64_t col_offset, gp_stream_t stream);
/* async.  Fused normalise / unreachable-fill / concat epilogue; replaces the
 * value convention of utils.py:73,76, the tensor conversion of utils.py:125 and
 * concat_into_features (utils.py:129-135):
 *   d_out[node*ld_out + j]                 = d_x[node*ld_x + j]      j in [0, F)   (skipped if d_x == NULL)
 *   d_out[node*ld_out + col_offset + j]    = 1/(hops+1), 0 if unreachable, j in [0, K)
 * IEEE fp32 division (bit-equal to the reference's float64 -> float32 rounding). */
int gp_msbfs_features(gp_msbfs_t *bfs, const float *d_x, int64_t num_features, int64_t ld_x,
                      float *d_out, int64_t ld_out, int64_t col_offset, gp_stream_t stream);
/* Hop 1 pulls like every other hop (a push form measured slower; profiles/r02_notes.md).  Kept for programs built
 * against ABI version 1: enable == 0 returns GP_OK, any other value GP_ERR_UNSUPPORTED.                          */
int gp_msbfs_set_push(gp_msbfs_t *bfs, int32_t enable);
/* syncs.  Reports latched GP_ERR_INDEX_RANGE / GP_ERR_LEVEL_OVERFLOW. */
int gp_msbfs_stats(gp_msbfs_t *bfs, gp_msbfs_stats_t *stats, gp_stream_t stream);
/* syncs on the kernel's own events.  Device time of the last MS-BFS kernel launch alone (CUDA
 * events recorded on the launch stream right around the persistent kernel), in milliseconds. */
int gp_msbfs_kernel_ms(gp_msbfs_t *bfs, float *ms);
/* Diagnostics (needs GP_BFS_TRACE=1 in the environment at gp_msbfs_create): per-warp SM clocks at
 * the start of each level sweep and after the hub / medium / short row phases.  syncs.        */
int gp_msbfs_trace(gp_msbfs_t *bfs, uint64_t *h_out, int64_t cap_words, int32_t *levels, int32_t *warps);
int gp_msbfs_free(gp_msbfs_t *bfs);

/* async.  gp_csr_build + gp_msbfs_run + gp_msbfs_features as ONE call.  Repeated calls with the same
 * arguments replay a captured CUDA graph (one launch instead of ~25); GP_USE_GRAPH=0 disables it.  */
int gp_geodesic_run(gp_csr_t *csr, gp_msbfs_t *bfs, const int64_t *d_edge_index, int64_t num_edges,
                    const int64_t *d_anchors, int64_t num_anchors, const float *d_x, int64_t num_features,
                    int64_t ld_x, float *d_out, int64_t ld_out, int64_t col_offset, gp_stream_t stream);

/* Stage clocks.  Eager launches always record CUDA events around the csr build, the MS-BFS kernel and the epilogue.
 * Inside the captured pipeline of gp_geodesic_run an event-record NODE costs ~4 us of the replayed step (246 -> 231 us
 * for the four at Flickr size), so they are recorded only on request: gp_msbfs_set_stage_events(bfs, 1) (the handle's
 * captured pipelines are dropped and re-captured).  gp_pipeline_stage_ms (syncs on its own events): ms3[0] = csr build
 * (+ the MS-BFS state memset), ms3[1] = the persistent MS-BFS kernel, ms3[2] = epilogue (decode + concat, pack, or
 * the exchange kernel) of the last fused run.  gp_msbfs_kernel_device_ns needs no events: the kernel stamps
 * %globaltimer at its entry and after its last level.                                                        */
int gp_msbfs_set_stage_events(gp_msbfs_t *bfs, int32_t enable);
int gp_msbfs_kernel_device_ns(gp_msbfs_t *bfs, uint64_t *ns, gp_stream_t stream);
int gp_pipeline_stage_ms(gp_msbfs_t *bfs, float *ms3);

/* async.  The x half of concat_into_features (utils.py:133-134) alone: d_out[:, 0:F] = d_x (a bulk-copy kernel for
 * 16-byte aligned rows, else one strided device-to-device transfer), for callers that want the copy on their own
 * stream; follow with gp_msbfs_features / gp_decode_peers called with d_x == NULL.  gp_geodesic_run keeps the copy
 * inside its epilogue kernel: running it beside the csr build and the MS-BFS measured slower on B200 (copy engine
 * 0.323 ms, copy kernels 0.265-0.301 ms, against 0.246 ms per step).                                           */
int gp_concat_x(const float *d_x, int64_t num_nodes, int64_t num_features, int64_t ld_x, float *d_out,
                int64_t ld_out, gp_stream_t stream);

/* Bit-sliced result planes of the last run, for the multi-GPU gather
 * (anchor-sharded ranks exchange these instead of uint16/fp32 columns):
 *   plane 0          "reached" mask;
 *   plane l, 1..15   lanes first reached at hop l (one-hot over the planes);
 *   plane 16 + q     bit q of the hop count of lanes first reached at hop 16 or later.
 * num_planes = 1 + max_level (1..16) when every hop is <= 15, else 32.  Planes at or past
 * num_planes hold stale bits of earlier runs.  Each plane is uint64
 * [batches][N][words_per_batch].  syncs (needs max_level).                      */
int gp_msbfs_planes(gp_msbfs_t *bfs, const uint64_t **d_planes, int64_t *plane_stride_words,
                    int32_t *num_planes, int32_t *batches, int32_t *words_per_batch, gp_stream_t stream);
/* async.  Decode planes gathered from `num_ranks` anchor shards (each shard laid
 * out as gp_msbfs_planes reports, shard r at d_gathered + r*rank_stride_words)
 * into columns [col_offset + r*anchors_per_rank + j] of d_out, optionally
 * copying x as gp_msbfs_features does.  num_planes is one value for all shards,
 * 1..16 or 32 (the largest any shard reported); a shard that reported fewer must
 * hold zeros in its planes up to num_planes.  GP_ERR_INVALID, before any CUDA
 * call, for other num_planes, plane_stride_words < batches*words_per_batch*N,
 * rank_stride_words < num_planes*plane_stride_words (more than one rank),
 * col_offset < 0, ld_x < num_features, or a NULL d_gathered / d_out.            */
int gp_decode_gathered(const uint64_t *d_gathered, int64_t rank_stride_words, int32_t num_ranks,
                       int64_t num_nodes, int64_t anchors_per_rank, int32_t num_planes,
                       int32_t batches, int32_t words_per_batch, int64_t plane_stride_words,
                       const float *d_x, int64_t num_features, int64_t ld_x,
                       float *d_out, int64_t ld_out, int64_t col_offset, gp_stream_t stream);

/* ---- peer-to-peer assembly (NVLink / NVSwitch): no staging buffer, no all-gather.
 * gp_msbfs_pack (async) rewrites the last result into the fixed-size exchange format (reached mask +
 * 4 hop-index bit planes, valid for hops <= 15; *d_deep_flag tells on the device if that failed) in one
 * of two slots; gp_msbfs_ipc_export / gp_ipc_open hand the buffer to the other ranks of the node as CUDA
 * IPC mappings; gp_decode_peers (async) is the fused epilogue whose loads read every rank's buffer in
 * place — its own from HBM, the peers' over NVLink — while it writes the [N, F+K] rows.               */
int gp_msbfs_pack(gp_msbfs_t *bfs, int32_t slot, const uint64_t **d_packed, int64_t *plane_stride_words,
                  int32_t *batches, int32_t *words_per_batch, const int32_t **d_deep_flag, gp_stream_t stream);
/* async.  gp_csr_build + gp_msbfs_run + gp_msbfs_pack(slot) as one graph-replayed call (a rank's share of
 * a sharded step up to the exchange).                                                                */
int gp_geodesic_run_packed(gp_csr_t *csr, gp_msbfs_t *bfs, const int64_t *d_edge_index, int64_t num_edges,
                           const int64_t *d_anchors, int64_t num_anchors, int32_t slot, gp_stream_t stream);
/* Pointers / shape of exchange slot `slot` without launching anything. */
int gp_msbfs_packed_info(gp_msbfs_t *bfs, int32_t slot, const uint64_t **d_packed, int64_t *plane_stride_words,
                         int32_t *batches, int32_t *words_per_batch, const int32_t **d_deep_flag);
int gp_msbfs_ipc_export(gp_msbfs_t *bfs, uint8_t *handle64, int64_t *slot_stride_words);
int gp_ipc_open(const uint8_t *handle64, void **d_ptr);
int gp_ipc_close(void *d_ptr);
int gp_decode_peers(const uint64_t *const *h_rank_ptrs, int32_t num_ranks, int64_t num_nodes,
                    int64_t anchors_per_rank, int32_t batches, int32_t words_per_batch, int64_t plane_stride_words,
                    const float *d_x, int64_t num_features, int64_t ld_x, float *d_out, int64_t ld_out,
                    int64_t col_offset, gp_stream_t stream);

/* ---- device exchange (gp_exchange.cu): pack -> gather from every rank -> decode as ONE cooperative kernel over
 * NVLink peer memory, no collective library call.  It replaces the result hand-back of the reference's pool
 * (utils.py:98-106) for anchor shards spread over the GPUs of one NVSwitch node: every rank packs its result into its
 * own exchange buffer and raises a flag on the peers; the row-streaming epilogue then pulls the peers' packed row
 * segments into shared memory with the bulk-copy engine (cp.async.bulk) two blocks ahead of the rows it writes.
 *   gp_exchange_create      buffers of this rank: 2 step parities x 5 packed planes, plus flags.
 *   gp_exchange_ipc_export  CUDA IPC handle of the buffer (open it in the other ranks with gp_ipc_open),
 *   gp_exchange_local_ptr   or its plain device pointer (ranks sharing one process),
 *   gp_exchange_set_peer    tell this rank where rank r's buffer is mapped.
 *   gp_geodesic_run_exchange (async, COLLECTIVE: every rank calls it once per step, in the same order)
 *                           gp_csr_build + gp_msbfs_run on this rank's `num_anchors` anchors + the fused kernel:
 *                           d_out[:, 0:F] = x, d_out[:, col_offset + r*num_anchors + j] = feature of rank r's anchor
 *                           j, for every rank r.  num_anchors must be the same multiple of 8 on every rank; d_out
 *                           16-byte aligned, ld_out and col_offset multiples of 4.  Replays a CUDA graph.
 *   gp_exchange_status      syncs.  *deep = 1 if some shard had hops > 15 in the last step (the 5-plane format
 *                           cannot hold them: redo the step through gp_msbfs_planes / gp_decode_gathered);
 *                           GP_ERR_CUDA if a peer's flag never arrived (bounded wait, ~8 s).                   */
int gp_exchange_create(gp_msbfs_t *bfs, int32_t world, int32_t rank, gp_exchange_t **out);
int gp_exchange_ipc_export(gp_exchange_t *xchg, uint8_t *handle64);
int gp_exchange_local_ptr(gp_exchange_t *xchg, void **d_ptr);
int gp_exchange_set_peer(gp_exchange_t *xchg, int32_t rank, void *d_ptr);
int gp_geodesic_run_exchange(gp_csr_t *csr, gp_msbfs_t *bfs, gp_exchange_t *xchg, const int64_t *d_edge_index,
                             int64_t num_edges, const int64_t *d_anchors, int64_t num_anchors, const float *d_x,
                             int64_t num_features, int64_t ld_x, float *d_out, int64_t ld_out, int64_t col_offset,
                             gp_stream_t stream);
/* async, COLLECTIVE.  The fused exchange / decode kernel alone, after the caller's own gp_msbfs_run. */
int gp_exchange_run(gp_exchange_t *xchg, const float *d_x, int64_t num_features, int64_t ld_x, float *d_out,
                    int64_t ld_out, int64_t col_offset, gp_stream_t stream);
int gp_exchange_status(gp_exchange_t *xchg, int32_t *deep, gp_stream_t stream);
/* Tuning / tests: cap the cooperative grid of the fused kernel (ranks sharing one GPU must all be resident at once,
 * since they wait for each other's flags); 0 = one full wave.                                                 */
int gp_exchange_set_grid(gp_exchange_t *xchg, int32_t max_blocks);
/* Diagnostics, syncs the device: globaltimer stamps (ns) of the last step: [0] block 0 starts, [1] block 0 has packed
 * its share, [2] block 0 has seen every peer's flag, [3] the last block leaves. */
int gp_exchange_trace(gp_exchange_t *xchg, uint64_t *h_stamps8);
int gp_exchange_free(gp_exchange_t *xchg);

/* ------------------------------------------------------------------ compact feature store
 * The anchor block of the [N, F+K] matrix in P bits per entry instead of 32, and the trainer's mini-batch lookup
 * x[n_id] (main.py:120,177) served from it.  A store is uint64 [N][P][W], W = ceil(K/64), one contiguous record per
 * node: plane 0 = reached mask, plane 1 + q = bit q of the hop count; column j is word j >> 6, bit j & 63 of a plane.
 * P = 1 + bit_length(max hop) (1..17).  Padding bits past K and hop bits of unreached lanes are zero.  The value of
 * column j is 1/(hops+1) in IEEE fp32 if reached, else 0 (bit-equal to gp_msbfs_features).  The caller owns the
 * store buffer.                                                                                                  */
/* syncs.  P and W of the store for the last gp_msbfs_run on bfs (bytes = N * P * W * 8). */
int gp_fstore_layout(gp_msbfs_t *bfs, int32_t *num_planes, int64_t *words_per_plane, gp_stream_t stream);
/* syncs.  Packs the last result into d_store [N][num_planes][W]; GP_ERR_INVALID if num_planes is too small (or
 * above 17).  The store does not refer to bfs afterwards (the handle may be rerun or freed).                    */
int gp_fstore_pack(gp_msbfs_t *bfs, uint64_t *d_store, int32_t num_planes, gp_stream_t stream);
/* async.  Merges anchor-shard stores into one store: d_shards is uint64 [S][N][P][Ws], shard s holding columns
 * [s*cols_per_shard, min((s+1)*cols_per_shard, K)) in the store format above with Ws >= ceil(cols_per_shard/64)
 * words per plane (tail shards may be short or empty; their words past their own columns are ignored).  Writes
 * d_store [N][P][ceil(K/64)], byte-identical to the store of one run over all K anchors packed with P planes.
 * GP_ERR_INVALID, before any CUDA call, if P is outside [1, 17], Ws < ceil(cols_per_shard/64),
 * S*cols_per_shard < K, or a pointer is NULL while N*K > 0.                                                     */
int gp_fstore_merge(const uint64_t *d_shards, int32_t num_shards, int64_t cols_per_shard, int64_t words_per_shard,
                    int64_t num_nodes, int32_t num_planes, int64_t num_anchors, uint64_t *d_store,
                    gp_stream_t stream);
/* async.  Mini-batch rows of concat_into_features(x, features) (utils.py:129-135) as main.py:120,177 index them:
 *   d_out[i*ld_out + c]              = d_x[rows[i]*ld_x + c]     c in [0, F)   (skipped if d_x == NULL)
 *   d_out[i*ld_out + col_offset + j] = value of column j of node rows[i], j in [0, K)
 * A negative id wraps once (rows[i] + N, as torch indexing does).  An id outside [-N, N) gets an all-zero output
 * row and increments *d_bad_rows (optional device int32 counter); nothing is loaded for it.                      */
int gp_fstore_gather(const uint64_t *d_store, int64_t num_nodes, int64_t num_anchors, int32_t num_planes,
                     const int64_t *d_rows, int64_t num_rows, const float *d_x, int64_t num_features, int64_t ld_x,
                     float *d_out, int64_t ld_out, int64_t col_offset, int32_t *d_bad_rows, gp_stream_t stream);

/* async.  Stand-alone epilogue from a uint16 hop matrix (utils.py:73,76,125). */
int gp_normalize_into(const uint16_t *d_dist, int64_t num_nodes, int64_t num_anchors, int64_t ld_dist,
                      float *d_out, int64_t ld_out, int64_t col_offset, gp_stream_t stream);

/* ------------------------------------------------------------------ one-call host entry
 * get_geodesic_distance_vector + concat_into_features with HOST buffers
 * (utils.py:116-135): copies edge_index/anchors to the device, builds the CSR,
 * runs the MS-BFS and the epilogue, and copies the feature block back into
 * h_out[:, col_offset:col_offset+K] (row pitch ld_out floats).  If h_x != NULL
 * its F columns are copied into h_out[:, 0:F] on the host while the GPU works.
 * h_hops (optional, may be NULL) receives the uint16 hop matrix [N, K].  syncs.
 * GP_ERR_NO_DEVICE when the process sees no CUDA device (there is no CPU fallback). */
int gp_geodesic_embed_host(const int64_t *h_edge_index, int64_t num_edges, int64_t num_nodes,
                           uint32_t csr_flags, const int64_t *h_anchors, int64_t num_anchors,
                           const float *h_x, int64_t num_features,
                           float *h_out, int64_t ld_out, int64_t col_offset,
                           uint16_t *h_hops, gp_msbfs_stats_t *stats);

/* The same with an explicit context.  A context owns everything the one-call entry keeps between calls (CSR and
 * MS-BFS handles, device staging, its stream, the pinned ring for pageable outputs); it serves one call at a time, and
 * contexts are independent: two host threads with two contexts do not serialise.  gp_geodesic_embed_host uses one
 * process-wide default context.  The library keeps no other mutable global state: captured CUDA graphs belong to the
 * MS-BFS handle they were captured for, environment switches are read once per process.                          */
int gp_ctx_create(gp_ctx_t **out);
int gp_ctx_free(gp_ctx_t *ctx);
int gp_geodesic_embed_host_ctx(gp_ctx_t *ctx, const int64_t *h_edge_index, int64_t num_edges, int64_t num_nodes,
                               uint32_t csr_flags, const int64_t *h_anchors, int64_t num_anchors,
                               const float *h_x, int64_t num_features,
                               float *h_out, int64_t ld_out, int64_t col_offset,
                               uint16_t *h_hops, gp_msbfs_stats_t *stats);

/* Host side of concat_into_features (utils.py:129-135) for results that arrive as a separate
 * [N, block_cols] block: out[:, 0:F] = x, out[:, F:F+block_cols] = block, threaded row copies.      */
int gp_host_concat(const float *h_x, int64_t num_features, const float *h_block, int64_t block_cols,
                   int64_t num_nodes, float *h_out, int64_t ld_out);
/* async.  Device block [N, block_cols] (contiguous) -> columns [col_offset, col_offset + block_cols) of
 * the PINNED host matrix h_out (leading dimension ld_out) as one strided DMA, so the host only has to
 * copy x (gp_host_concat with h_block = NULL) while the transfer runs.  GP_ERR_INVALID if h_out is
 * pageable (a pageable 2-D copy degenerates into N small transfers: stage it instead).              */
int gp_block_to_host(const float *d_block, int64_t num_nodes, int64_t block_cols, float *h_out, int64_t ld_out,
                     int64_t col_offset, gp_stream_t stream);

/* ------------------------------------------------------------------ KMeans anchors (node2vec branch)
 * attach_node2vec takes the KMeans centres of the node2vec table as anchors for every sampling_method but
 * 'stochastic' (utils.py:168-170).  Three building blocks, driven by graphpope_b200.device.kmeans:
 *   gp_kmeans_plusplus  k-means++ seeding (exact D^2 sampling by an exponential race); syncs.
 *                       d_centers float32[K, D] out, d_mind2 float32[N] scratch, d_chosen int64[K] out.
 *   gp_kmeans_assign    nearest centre of every row on the tensor cores (the pairwise kernel in arg-min
 *                       mode, nothing but the result leaves the SM); async.  d_best uint64[N]:
 *                       (float bits of the squared distance << 32) | centre index.
 *   gp_kmeans_update    centres := mean of their rows (an empty cluster keeps its centre); *d_shift2 =
 *                       sum of squared centre moves, *d_inertia = sum of squared distances; async.       */
int gp_kmeans_plusplus(const float *d_emb, int64_t num_nodes, int64_t num_centers, int64_t dim, int64_t first_index,
                       uint64_t seed, float *d_centers, float *d_mind2, int64_t *d_chosen, gp_stream_t stream);
int gp_kmeans_assign(const float *d_emb, const float *d_centers, int64_t num_nodes, int64_t num_centers, int64_t dim,
                     uint64_t *d_best, gp_stream_t stream);
int gp_kmeans_update(const float *d_emb, const uint64_t *d_best, int64_t num_nodes, int64_t num_centers, int64_t dim,
                     float *d_centers, float *d_sums, int32_t *d_counts, double *d_shift2, double *d_inertia,
                     gp_stream_t stream);

/* ------------------------------------------------------------------ samplers
 * degree_centrality (utils.py:38-42): in+out degree over de-duplicated edges
 * (a self-loop counts 2).  async.  d_degree int32[N].                           */
int gp_degree(const gp_csr_t *csr, int32_t *d_degree, gp_stream_t stream);
/* pagerank (utils.py:26-30 -> networkx _pagerank_scipy defaults): float64 power
 * iteration, uniform start/personalisation, dangling mass spread uniformly,
 * stop when the L1 change < N*tol.  syncs.  d_x float64[N].                     */
int gp_pagerank(const gp_csr_t *csr, double alpha, double tol, int32_t max_iter,
                double *d_x, int32_t *iterations, gp_stream_t stream);
/* closeness_centrality (utils.py:50-54 -> nx.closeness_centrality defaults: incoming distance,
 * Wasserman-Faust scaling): scores of ALL nodes from N/4096 passes of the MS-BFS with every node as an
 * anchor plus bit-sliced column sums; float64 in networkx's operation order (bit-equal).  syncs.
 * d_score float64[N].                                                                             */
int gp_closeness(const gp_csr_t *csr, double *d_score, gp_stream_t stream);
/* clustering_coefficient (utils.py:56-60 -> nx.clustering on the DiGraph, Fagiolo's directed clustering):
 * integer triangle and degree counts from shared-memory node bitmaps, one float64 division (bit-equal).
 * syncs.  d_score float64[N].  GP_ERR_UNSUPPORTED when two N-bit maps do not fit in shared memory.   */
int gp_clustering(const gp_csr_t *csr, double *d_score, gp_stream_t stream);
/* betweenness_centrality (utils.py:32-36 -> nx.betweenness_centrality defaults: Brandes, normalized, no
 * endpoints, on the DiGraph): 32 sources per batch, one warp lane per source, level-synchronous pull sweeps in
 * one persistent kernel (gp_betweenness.cu).  Path counts are exact; the float64 dependency sums have a fixed
 * order that differs from networkx's queue order, so scores agree to a few ulp, not bit for bit.  syncs.
 * d_score float64[N].  The workspace (~1.1 KB per node) lives in the csr handle and is reused by later calls:
 * one gp_betweenness call at a time per handle.                                                        */
int gp_betweenness(const gp_csr_t *csr, double *d_score, gp_stream_t stream);
/* eigenvector_centrality (utils.py:44-48 -> nx.eigenvector_centrality_numpy: eigenvector of A^T for the
 * largest real eigenvalue, unit L2 norm, positive): float64 power iteration on (A^T + I) until the L1 change
 * of the normalised vector is <= N * tol.  networkx uses ARPACK, so scores agree to rounding (tests: 1e-9), not
 * bit for bit; the caller checks strong connectivity first, as networkx >= 3.2 does.  syncs.  d_x float64[N].
 * GP_ERR_NOT_CONVERGED after max_iter iterations (graphs with a tiny spectral gap, e.g. long paths).    */
int gp_eigenvector(const gp_csr_t *csr, double tol, int32_t max_iter, double *d_x, int32_t *iterations,
                   gp_stream_t stream);
/* Stable top-k of utils.py:29-30 / 41-42: ascending stable sort by score, keep
 * the last k (ties keep ascending node id; output in ascending-score order).
 * async.  d_out int64[min(k, N)] (k == 0 returns all N: list[-0:] quirk).       */
int gp_topk_stable_i32(const int32_t *d_score, int64_t num_nodes, int64_t k, int64_t *d_out, gp_stream_t stream);
int gp_topk_stable_f64(const double *d_score, int64_t num_nodes, int64_t k, int64_t *d_out, gp_stream_t stream);

/* ------------------------------------------------------------------ node2vec block
 * The pairwise step + MinMaxScaler of attach_node2vec (utils.py:174-176):
 * out[:, col_offset + j] = minmax_j( f(emb_i, anchor_j) ), f per gp_cdist_mode,
 * tensor-core GEMM with split-precision operands and fp32 accumulation.
 * d_emb float32 [N, D], d_anchor_emb float32 [K, D].  async.                    */
int gp_cdist_minmax(const float *d_emb, const float *d_anchor_emb, int64_t num_nodes, int64_t num_anchors,
                    int64_t dim, int32_t mode, int32_t apply_minmax,
                    float *d_out, int64_t ld_out, int64_t col_offset, gp_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GRAPHPOPE_B200_H */
