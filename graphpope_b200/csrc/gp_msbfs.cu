// gp_msbfs.cu — multi-source BFS over bit lanes, one persistent cooperative kernel (sm_100a).
//
// Replaces the N*K nx.shortest_path calls of the reference hot loop (utils.py:69-77, fanned
// out by utils.py:92-114): hops(node -> anchor_j) for all nodes and anchors is computed as a
// level-synchronous BFS from all anchors at once, 64 anchors per uint64 lane word.
//
// Formulation.  Paths run node -> anchor (row = source, utils.py:73), so the frontier moves
// against the edge direction.  In PULL form a row u ORs the frontier words of its
// OUT-neighbours: new[u] = (OR_{u->v} frontier[v]) & ~seen[u].  Each row is finalised by exactly
// one thread group, so there are no atomics on the lane state and a level needs one grid barrier.
//
// Work decomposition.  On the named graphs the lane state (a few MB) lives in L2.  A dense level is
// bound by the rate at which an SM can gather random 32-byte rows out of L2 (~1.1 SM-cycles per row,
// tools/microbench/gather_rate.cu); every other level is bound by instruction issue and the grid
// barrier, so the kernel (a) gathers only what can matter and (b) keeps the per-slot instruction
// count small.  The CSR builder (gp_csr.cu) emits a degree-ordered list of 16-byte row descriptors;
// a row of degree d is served by G = 1,2,4,...,32 "slots" (threads) of <= 4 edges each (4G >= d), hub
// rows are cut into 128-edge chunks (G = 32, one warp) whose partial ORs meet in a small accumulator
// that the last-arriving chunk finalises (release / acquire through the arrival counter).  One slot = <= 4 column indices -> <= 4 whole frontier rows
// (one 256-bit load each at 256 anchors per batch, all issued back to back) -> shuffle-OR over the G
// slots of the row -> finalise.  Three filters cut the gathers to the ones that can matter:
//   * a per-hop bitmap of non-zero frontier rows, staged in shared memory every level: a neighbour
//     whose frontier row is zero is not gathered (the first and last levels touch almost nothing);
//   * per-row "done" flags: a row every still-live lane has reached is never gathered again;
//   * a per-word "live" mask (lanes whose frontier is non-empty anywhere).
// Tiles (32 slots of one class) are dealt round-robin to the CTAs, heaviest classes first, and the
// warps of a CTA pull them from a shared-memory queue, so hub tiles start first and no warp idles
// while another still has two tiles to go.
//
// Data layout (all uint64, node-major so one neighbour gather is one 32-byte sector at wb == 4):
//   result block R, 32 arrays of [batches][N][wb]:
//     R[0]        reached mask ("seen")
//     R[l]        l = 1..15: lanes FIRST reached at hop l.  These are simply the frontiers: level l
//                 writes its next-frontier into R[l] and nothing ever overwrites it, so recording
//                 the hop count costs no extra traffic at all on shallow graphs.
//     R[16 + q]   q = 0..15: bit q of the hop count of lanes first reached at hop >= 16 (deep
//                 graphs only; OR-ed in with fire-and-forget reductions at L2).
//   plus the seed frontier and two ping-pong frontiers used from hop 16 on.
// The uint16 / fp32 matrices are never scattered to: the epilogue (gp_epilogue.cu) decodes R row
// by row with fully coalesced stores.
#include "gp_msbfs.cuh"

#include <new>

namespace {

struct BfsParams {
    int n;
    int batches;
    int num_anchors;
    int hub_capacity;
    const int *__restrict__ col;
    const int4 *__restrict__ desc;
    const int *__restrict__ meta;   // csr meta words (class counts as running totals, slot bases)
    int desc_off[GP_NUM_CLASSES];   // first descriptor of each class's region in `desc` (fixed per csr handle)
    const long long *__restrict__ anchors;
    u64 *result;                    // R[0..31], see the layout note above
    u64 *seeds;                     // level-0 frontier (the anchors)
    u64 *fr_a;                      // three rotating frontiers for hops >= 16 (hop l lives in buffer l % 3)
    u64 *fr_b;
    u64 *fr_c;
    long long plane_stride;         // words per array = batches * n * wb
    u64 *live;                      // [3][GP_BFS_MAX_LANE_WORDS]
    u64 *hub_acc;                   // [batches][hub_capacity][wb] partial ORs of hub rows
    u32 *hub_cnt;                   // [batches][hub_capacity] chunks arrived
    u64 *bar;                       // [3] grid barrier words, rotating by level % 3 (see grid_barrier_flags)
    u32 *nzmap;                     // [3][batches][nzwords] bit u set <=> frontier row u of that hop is non-zero
    int nzwords;                    // words per batch map = ceil(n / 32)
    int map_stride;                 // words between the three rotating map sets (batches * nzwords, padded to 4)
    int map_smem_words;             // map_stride if the maps are staged in shared memory, else 0 (maps off)
    int *status;
    u64 *counters;
    u64 *trace;                     // optional per-warp phase clocks (diagnostics), else nullptr
};

template <int VW>
__device__ __forceinline__ void vload(const u64 *p, u64 (&v)[VW])
{
    if constexpr (VW == 4) {  // one 256-bit load (LDG.E.ENL2.256): a whole 256-anchor row in one request
        asm volatile("ld.global.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(v[0]), "=l"(v[1]), "=l"(v[2]), "=l"(v[3]) : "l"(p));
    } else if constexpr (VW == 2) {
        asm volatile("ld.global.v2.u64 {%0,%1}, [%2];" : "=l"(v[0]), "=l"(v[1]) : "l"(p));
    } else {
        asm volatile("ld.global.u64 %0, [%1];" : "=l"(v[0]) : "l"(p));
    }
}

template <int VW>
__device__ __forceinline__ void vstore(u64 *p, const u64 (&v)[VW])
{
    if constexpr (VW == 4) {
        asm volatile("st.global.v4.u64 [%0], {%1,%2,%3,%4};" ::"l"(p), "l"(v[0]), "l"(v[1]), "l"(v[2]), "l"(v[3]) : "memory");
    } else if constexpr (VW == 2) {
        asm volatile("st.global.v2.u64 [%0], {%1,%2};" ::"l"(p), "l"(v[0]), "l"(v[1]) : "memory");
    } else {
        asm volatile("st.global.u64 [%0], %1;" ::"l"(p), "l"(v[0]) : "memory");
    }
}

__device__ __forceinline__ void red_or_u64(u64 *p, u64 v)
{
    asm volatile("red.relaxed.gpu.global.or.b64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__device__ __forceinline__ u32 atom_add_acq_rel_u32(u32 *p, u32 v)
{
    u32 old;
    asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
    return old;
}

__device__ __forceinline__ u64 ld_relaxed_u64(const u64 *p)
{
    u64 v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ void red_or_u32(u32 *p, u32 v)
{
    asm volatile("red.relaxed.gpu.global.or.b32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Grid barrier that also tells every CTA (a) whether ANY CTA reached a new lane this level,
// (b) whether ANY CTA still owns a row that can gain lanes and (c) how many rows of the frontier
// just written are non-zero.  One 64-bit word per level, three words rotating by level % 3 (CTA 0
// clears the word two levels ahead), so every level starts from zero:
//   bits [0,12) arrivals, [12,24) CTAs reporting `any`, [24,36) CTAs reporting `notdone`,
//   [36,64) non-zero frontier rows.  (The launch keeps the grid below 4096 CTAs.)
constexpr u64 GP_BAR_FIELD = (1ull << 12) - 1ull;
__device__ __forceinline__ u64 grid_barrier_flags(u64 *bar_word, u32 nblocks, bool cta_any, bool cta_notdone,
                                                  u64 *s_bcast, int *s_any_flag, int *s_notdone_flag, int *s_nzrows,
                                                  int *s_queue, int nqueues)
{
    __syncthreads();
    if (threadIdx.x < nqueues) s_queue[threadIdx.x] = 0;  // the CTA's tile queues restart with the next level
    if (threadIdx.x == 0) {
        const u64 inc = 1ull | ((u64)(cta_any ? 1u : 0u) << 12) | ((u64)(cta_notdone ? 1u : 0u) << 24) |
                        ((u64)(u32)*s_nzrows << 36);
        *s_any_flag = 0;  // every thread has read the flags (before the sync above); next writes come after the sync below
        *s_notdone_flag = 0;
        *s_nzrows = 0;
        asm volatile("red.release.gpu.global.add.u64 [%0], %1;" ::"l"(bar_word), "l"(inc) : "memory");
        u64 v;
        do {
            v = ld_relaxed_u64(bar_word);  // relaxed polling: an acquire load would flush this SM's L1 each time
        } while ((u32)(v & GP_BAR_FIELD) < nblocks);
        u32 dummy;  // one acquire load after the relaxed polling (measured faster than fence.acq_rel here)
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(dummy) : "l"(bar_word) : "memory");
        *s_bcast = v;
    }
    __syncthreads();
    return *s_bcast;
}
__device__ __forceinline__ bool bar_any(u64 v) { return ((v >> 12) & GP_BAR_FIELD) != 0; }
__device__ __forceinline__ bool bar_notdone(u64 v) { return ((v >> 24) & GP_BAR_FIELD) != 0; }
__device__ __forceinline__ long long bar_nzrows(u64 v) { return (long long)(v >> 36); }

#define GP_TRACE(slot)                                                                             \
    do {                                                                                           \
        if (p.trace != nullptr && lane == 0 && level <= 32)                                        \
            p.trace[(((size_t)(level - 1) * total_warps + gwarp) << 2) + (slot)] = (u64)clock64(); \
    } while (0)

template <int VW>
struct LevelCtx {
    const u64 *cur;
    u64 *nxt;
    u64 *seen;
    u64 *planes;   // R[16]: deep-hop bit planes
    long long plane_stride;
    int level;
    u32 *map_w;    // non-zero-row bitmap of the frontier being written (this batch), or nullptr
};

// Owner-side update of one row's VW lane words.  The frontier array being written was zeroed one level ahead
// (see the level prologue), so a row with nothing new writes nothing at all.  Returns true if the row can still
// gain lanes (some lane that is live this level has not reached it yet).
template <int VW>
__device__ __forceinline__ bool finalize_row(const LevelCtx<VW> &c, size_t off, int row, const u64 (&acc)[VW],
                                             u64 (&seenv)[VW], u64 (&live_acc)[VW], const u64 (&lv)[VW], int &nzrows)
{
    u64 nw[VW];
    bool any = false;
#pragma unroll
    for (int i = 0; i < VW; ++i) {
        nw[i] = acc[i] & ~seenv[i];
        any |= nw[i] != 0;
    }
    if (any) {
        vstore<VW>(c.nxt + off, nw);  // for level <= 15 this IS the record "first reached at hop level"
#pragma unroll
        for (int i = 0; i < VW; ++i) {
            seenv[i] |= nw[i];
            live_acc[i] |= nw[i];
        }
        vstore<VW>(c.seen + off, seenv);
        ++nzrows;
        if (c.map_w != nullptr) red_or_u32(c.map_w + (row >> 5), 1u << (row & 31));
        if (c.level > GP_BFS_LEVEL_ARRAYS) {
            // deep graphs: OR the new lanes into every bit plane set in `level` (fire-and-forget at L2)
            for (int lb = c.level; lb; lb &= lb - 1) {
                u64 *pp = c.planes + (size_t)(__ffs(lb) - 1) * c.plane_stride + off;
#pragma unroll
                for (int i = 0; i < VW; ++i)
                    if (nw[i]) red_or_u64(pp + i, nw[i]);
            }
        }
    }
    bool incomplete = false;
#pragma unroll
    for (int i = 0; i < VW; ++i) incomplete |= (~seenv[i] & lv[i]) != 0;
    return incomplete;
}

// Launch shape: 384 threads x 2 CTAs per SM (80 registers) ties 768x1 as the fastest; fewer warps run 5% slower, more
// warps spill (profiles/r01k_notes.md).
constexpr int BFS_THREADS = 384;
constexpr int BFS_CTAS_PER_SM = 2;
constexpr int BFS_WARPS = BFS_THREADS / 32;
// Tiles of a CTA whose work items live in shared memory: GP_BFS_CACHE_ITERS per warp.
constexpr int BFS_CACHED_TILES = GP_BFS_CACHE_ITERS * BFS_WARPS;
constexpr size_t BFS_CACHE_BYTES =
    (size_t)BFS_CACHED_TILES * 32 * (2 * sizeof(int4) + GP_BFS_DONE_BATCHES) + (size_t)BFS_CACHED_TILES * GP_BFS_DONE_BATCHES;
static_assert((BFS_CACHED_TILES * GP_BFS_DONE_BATCHES) % 16 == 0, "the staged bitmaps that follow are read as uint4");

// Descriptor and column indices of the 32 slots of tile `t0 / 32` (one degree class per tile).
//   lead = {row or -1, count | chunks << 8 | first << 30, hub index, log2 G}, cols = <= 4 columns or -1.
__device__ __forceinline__ void load_tile(const BfsParams &p, const int *s_ent_base, const int *s_slot_base, int t0,
                                          int lane, int4 &lead, int4 &cols)
{
    int cls = 0;
    while (t0 >= s_slot_base[cls + 1]) ++cls;  // regions are GP_SLOT_ALIGN aligned: warp-uniform
    const int gsh = cls <= 1 ? 5 : 6 - cls;    // log2 of slots per row: 32,32,16,8,4,2,1
    const int rel = t0 - s_slot_base[cls] + lane;
    const int idx_in_class = rel >> gsh;
    const int sub = rel & ((1 << gsh) - 1);
    const bool active = idx_in_class < s_ent_base[cls + 1] - s_ent_base[cls];  // entries of the class
    const int4 d = active ? __ldg(p.desc + p.desc_off[cls] + idx_in_class) : make_int4(-1, 0, 0, -1);
    lead = make_int4(active ? d.x : -1, d.z, d.w, gsh);
    const int cnt = d.z & 0xFF;
    int c[GP_SLOT_EDGES];
#pragma unroll
    for (int i = 0; i < GP_SLOT_EDGES; ++i) {
        const int idx = sub + (i << gsh);  // consecutive slots read consecutive columns
        c[i] = (active && idx < cnt) ? __ldg(p.col + d.y + idx) : -1;
    }
    cols = make_int4(c[0], c[1], c[2], c[3]);
}

// WB lane words per node row = one thread loads a whole row (8, 16 or 32 bytes).
template <int WB, bool MAPG>
__global__ void __launch_bounds__(BFS_THREADS, BFS_CTAS_PER_SM) msbfs_kernel(BfsParams p)
{
    constexpr int VW = WB;
    constexpr int NT = BFS_THREADS;
    constexpr int WARPS = BFS_WARPS;
    constexpr int JT = BFS_CACHED_TILES;
    static_assert(GP_SLOT_EDGES == 4, "slot layout is int4");
    // Work cache: a CTA visits the same tiles every level, so the descriptors and column indices of
    // its first JT tiles are loaded ONCE into shared memory; a level then costs a single dependent
    // round trip (gathers + seen together).
    extern __shared__ __align__(16) unsigned char s_dyn[];
    int4 *s_lead = reinterpret_cast<int4 *>(s_dyn);                 // [JT][32]
    int4 *s_cols = s_lead + JT * 32;                                // [JT][32]
    unsigned char *s_done = reinterpret_cast<unsigned char *>(s_cols + JT * 32);  // [DONE_B][JT][32]
    unsigned char *s_tdone = s_done + GP_BFS_DONE_BATCHES * JT * 32;               // [DONE_B][JT] whole tile finished
    u32 *s_map = reinterpret_cast<u32 *>(s_tdone + GP_BFS_DONE_BATCHES * JT);      // [batches][nzwords] or absent
    __shared__ u32 s_live32[GP_BFS_MAX_LANE_WORDS * 2];
    __shared__ int s_ent_base[GP_NUM_CLASSES + 1];
    __shared__ int s_slot_base[GP_NUM_CLASSES + 1];
    __shared__ u64 s_bcast;
    __shared__ u64 s_lv[GP_BFS_MAX_LANE_WORDS];
    __shared__ int s_any;
    __shared__ int s_notdone;
    __shared__ int s_nzrows;
    __shared__ int s_queue[GP_BFS_MAX_LANE_WORDS];  // one tile queue per batch

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long gthreads = (long long)gridDim.x * NT;
    const long long gtid = (long long)blockIdx.x * NT + tid;
    const int gwarp = blockIdx.x * WARPS + warp, total_warps = gridDim.x * WARPS;
    const int n = p.n, lw = p.batches * WB;
    // MAPG: the per-hop bitmaps do not fit in shared memory (large graphs); the same filter then reads
    // them straight from global memory (L1 resident within a level; the barrier's acquire drops stale lines)
    const bool use_map = MAPG || p.map_smem_words > 0;
    u64 gathers = 0;

#define GP_TRACE_PRO(slot)                                                                    \
    do {                                                                                      \
        if (p.trace != nullptr && lane == 0)                                                  \
            p.trace[(((size_t)31 * total_warps + gwarp) << 2) + (slot)] = (u64)clock64();     \
    } while (0)
    GP_TRACE_PRO(0);
    if (gtid == 0) {  // device-clock stamps of the kernel (gp_msbfs_kernel_device_ns): entry, and after the last level
        u64 t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        p.counters[2] = t;
    }
    for (int i = tid; i < GP_BFS_MAX_LANE_WORDS * 2; i += NT) s_live32[i] = 0;
    if (tid <= GP_NUM_CLASSES) {
        s_ent_base[tid] = p.meta[GP_META_ENT_BASE + tid];
        s_slot_base[tid] = p.meta[GP_META_SLOT_BASE + tid];
    }
    if (tid == 0) {
        s_any = 0;
        s_notdone = 0;
        s_nzrows = 0;
    }
    if (tid < GP_BFS_MAX_LANE_WORDS) s_queue[tid] = 0;

    // ---- level 0: seed the anchors (duplicates simply set their own lane bits)
    for (long long j = gtid; j < p.num_anchors; j += gthreads) {
        const long long a = p.anchors[j];
        if (a < 0 || a >= n) {
            atomicOr(&p.status[GP_BFS_ST_ERROR], GP_DEV_ERR_ANCHOR_RANGE);
            continue;
        }
        const int b = (int)(j / (64 * WB)), w = (int)((j / 64) % WB);
        const u64 bit = 1ull << (j & 63);
        const size_t off = ((size_t)b * n + (size_t)a) * WB + w;
        atomicOr(p.result + off, bit);
        atomicOr(p.seeds + off, bit);
        atomicOr(p.live + 1 * GP_BFS_MAX_LANE_WORDS + b * WB + w, bit);
        if (use_map) atomicOr(p.nzmap + (size_t)b * p.nzwords + (size_t)(a >> 5), 1u << (a & 31));  // map of hop 0
    }
    __syncthreads();
    GP_TRACE_PRO(1);
    const int total_tiles = s_slot_base[GP_NUM_CLASSES] / 32;
    // tile j of this CTA is global tile blockIdx.x + gridDim.x * j
    const int tiles_cta = total_tiles > (int)blockIdx.x ? (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const int cached_tiles = tiles_cta < JT ? tiles_cta : JT;
    // the cached tiles of a warp are fetched together: their descriptor loads, then their column loads, are all in
    // flight at once (one tile after the other this was 2 dependent round trips per tile before the first level)
    {
        constexpr int TPW = JT / WARPS;  // cached tiles per warp
        int4 lead[TPW], cols[TPW];
#pragma unroll
        for (int q = 0; q < TPW; ++q) {
            const int j = warp + q * WARPS;
            lead[q] = make_int4(-1, 0, 0, 0);
            cols[q] = make_int4(-1, -1, -1, -1);
            if (j < cached_tiles)
                load_tile(p, s_ent_base, s_slot_base, ((int)blockIdx.x + (int)gridDim.x * j) * 32, lane, lead[q], cols[q]);
        }
#pragma unroll
        for (int q = 0; q < TPW; ++q) {
            const int j = warp + q * WARPS;
            if (j < cached_tiles) {
                s_lead[j * 32 + lane] = lead[q];
                s_cols[j * 32 + lane] = cols[q];
                for (int b = 0; b < GP_BFS_DONE_BATCHES; ++b) s_done[(b * JT + j) * 32 + lane] = lead[q].x < 0 ? 1 : 0;
            }
        }
    }
    for (int i = tid; i < GP_BFS_DONE_BATCHES * JT; i += NT) s_tdone[i] = 0;
    GP_TRACE_PRO(2);
    grid_barrier_flags(p.bar + 0, gridDim.x, false, false, &s_bcast, &s_any, &s_notdone, &s_nzrows, s_queue, p.batches);
    GP_TRACE_PRO(3);

    int level = 1, max_level = 0;
    long long nz_prev = p.num_anchors;  // non-zero rows of the frontier about to be read (hop 0: the anchors)
    while (true) {
        LevelCtx<VW> c;
        // frontier of hop l lives in R[l] for l <= 15, then in the ping-pong pair
        auto frontier = [&](int l) -> u64 * {
            if (l == 0) return p.seeds;
            if (l <= GP_BFS_LEVEL_ARRAYS) return p.result + (size_t)l * p.plane_stride;
            return l % 3 == 0 ? p.fr_a : (l % 3 == 1 ? p.fr_b : p.fr_c);
        };
        c.cur = frontier(level - 1);
        c.nxt = frontier(level);
        c.seen = p.result;
        c.planes = p.result + (size_t)(1 + GP_BFS_LEVEL_ARRAYS) * p.plane_stride;
        c.plane_stride = p.plane_stride;
        c.level = level;
        // Rows write their next-frontier words only when a lane is new, so every frontier array is cleared one
        // level AHEAD of its use, by the whole grid with coalesced stores that nobody waits for (the host clears
        // the arrays of hops 0 and 1).  The deep-hop bit planes, first needed at hop 16, are cleared at hop 15.
        {
            u64 *z = frontier(level + 1);
            for (long long i = gtid; i < p.plane_stride; i += gthreads) z[i] = 0;
            if (level == GP_BFS_LEVEL_ARRAYS) {
                u64 *pl = c.planes;
                for (long long i = gtid; i < (long long)GP_BFS_PLANES * p.plane_stride; i += gthreads) pl[i] = 0;
            }
        }
        const u64 *live_r = p.live + (level % 3) * GP_BFS_MAX_LANE_WORDS;
        u64 *live_w = p.live + ((level + 1) % 3) * GP_BFS_MAX_LANE_WORDS;
        u64 *live_z = p.live + ((level + 2) % 3) * GP_BFS_MAX_LANE_WORDS;
        if (blockIdx.x == 0 && tid < lw) live_z[tid] = 0;
        if (gtid == 0) p.bar[(level + 1) % 3] = 0;  // last used two levels ago; next used one level from now
        // maps rotate like the barrier words: hop h lives in map h % 3.  A dense frontier (most rows
        // non-zero) makes the map useless, so it is staged only when it can filter something.
        const bool map_level = use_map && nz_prev * 2 < (long long)n * p.batches;
        u32 *map_w = use_map ? p.nzmap + (size_t)(level % 3) * p.map_stride : nullptr;
        if (use_map) {
            uint4 *map_z = reinterpret_cast<uint4 *>(p.nzmap + (size_t)((level + 1) % 3) * p.map_stride);
            const int quads = p.map_stride >> 2;  // padded to a multiple of 4 words
            for (long long i = gtid; i < quads; i += gthreads) map_z[i] = make_uint4(0, 0, 0, 0);
            if (map_level && !MAPG) {
                const uint4 *map_r = reinterpret_cast<const uint4 *>(p.nzmap + (size_t)((level - 1) % 3) * p.map_stride);
                uint4 *s_map4 = reinterpret_cast<uint4 *>(s_map);
#pragma unroll 4
                for (int i = tid; i < quads; i += NT) s_map4[i] = __ldcg(map_r + i);
            }
        }
        if (tid < lw) s_lv[tid] = ld_relaxed_u64(live_r + tid);  // one L2 read per CTA instead of one per warp
        __syncthreads();
        GP_TRACE(0);

        int nzrows = 0;
        for (int b = 0; b < p.batches; ++b) {
            u64 lv[VW], live_acc[VW];
#pragma unroll
            for (int i = 0; i < VW; ++i) {
                lv[i] = s_lv[b * WB + i];
                live_acc[i] = 0;
            }
            const u64 *cur_b_rows = c.cur + (size_t)b * n * WB;
            const u32 *s_map_b = s_map + (size_t)b * p.nzwords;
            const u32 *g_map_b = p.nzmap + (size_t)((level - 1) % 3) * p.map_stride + (size_t)b * p.nzwords;
            c.map_w = use_map ? map_w + (size_t)b * p.nzwords : nullptr;
            // tile queue of this batch: every warp starts with tile `warp`, the rest are handed out on
            // demand; the index of the NEXT tile is requested before the current one is processed
            int j_next = 0;
            for (int j = warp; j < tiles_cta; j = __shfl_sync(FULL_MASK, j_next, 0)) {
                if (lane == 0) j_next = atomicAdd(&s_queue[b], 1) + WARPS;

            unsigned char *tdone = (j < JT && b < GP_BFS_DONE_BATCHES) ? s_tdone + b * JT + j : nullptr;
            if (tdone != nullptr && *tdone) continue;  // every row of the tile holds all live lanes: nothing to do
            int4 lead, cols;
            unsigned char *dflag = nullptr;
            if (j < JT) {
                lead = s_lead[j * 32 + lane];
                cols = s_cols[j * 32 + lane];
                if (b < GP_BFS_DONE_BATCHES) dflag = s_done + (b * JT + j) * 32;
            } else {
                load_tile(p, s_ent_base, s_slot_base, ((int)blockIdx.x + (int)gridDim.x * j) * 32, lane, lead, cols);
            }
            const int gsh = lead.w;
            const int sub = lane & ((1 << gsh) - 1);
            const bool leader = sub == 0 && lead.x >= 0;
            const int nch = (lead.y >> 8) & 0x3FFFFF;
            const size_t off = ((size_t)b * n + (size_t)(lead.x >= 0 ? lead.x : 0)) * WB;
            // a row is "done" once every still-live lane has reached it: it never needs gathering again
            const bool done = dflag != nullptr ? dflag[lane - sub] != 0 : lead.x < 0;
            u64 seenv[VW], acc[VW];
#pragma unroll
            for (int i = 0; i < VW; ++i) {
                seenv[i] = ~0ull;
                acc[i] = 0;
            }
            if (__all_sync(FULL_MASK, done)) {
                if (tdone != nullptr && lane == 0) *tdone = 1;
                continue;
            }
            const int v[GP_SLOT_EDGES] = {cols.x, cols.y, cols.z, cols.w};
            u32 needbits = 0;
            if (!done) {
#pragma unroll
                for (int i = 0; i < GP_SLOT_EDGES; ++i) {
                    // gather only neighbours whose frontier row is non-zero at this hop
                    const bool nz = v[i] >= 0 && (!map_level || (((MAPG ? g_map_b[v[i] >> 5] : s_map_b[v[i] >> 5]) >> (v[i] & 31)) & 1u));
                    needbits |= (u32)nz << i;
                }
            }
            const u32 bal = __ballot_sync(FULL_MASK, needbits != 0);
            const u32 gmask = gsh == 5 ? FULL_MASK : (((1u << (1 << gsh)) - 1u) << (lane - sub));
            const bool group_need = (bal & gmask) != 0;
            u64 t[GP_SLOT_EDGES][VW];
#pragma unroll
            for (int i = 0; i < GP_SLOT_EDGES; ++i) {
#pragma unroll
                for (int q = 0; q < VW; ++q) t[i][q] = 0;
                if ((needbits >> i) & 1u) vload<VW>(cur_b_rows + (size_t)(u32)v[i] * WB, t[i]);
            }
            // the finalising lane needs the reached mask; chunks of a hub row always take part in the
            // arrival protocol (every chunk reads the same mask before the last one updates it)
            const bool eval = leader && !done && (group_need || nch > 0);
            if (eval) vload<VW>(p.result + off, seenv);
#pragma unroll
            for (int i = 0; i < GP_SLOT_EDGES; ++i)
#pragma unroll
                for (int q = 0; q < VW; ++q) acc[q] |= t[i][q];
            gathers += (u64)VW * (u64)__popc(needbits);
            if (bal != 0) {
                if (gsh == 5) {
#pragma unroll
                    for (int q = 0; q < VW; ++q) acc[q] = warp_or_u64(acc[q]);
                } else {
                    for (int m = 1; m < (1 << gsh); m <<= 1)
#pragma unroll
                        for (int q = 0; q < VW; ++q) acc[q] |= shfl_xor_u64(acc[q], m);
                }
            }
            if (!leader) continue;
            if (!eval) {
                // done, or not done but no neighbour has anything new: the row's next frontier stays empty
                if (!done) s_notdone = 1;  // flags are set as soon as a row completes, so this row still lacks lanes
                continue;
            }
            bool need_row = false;
#pragma unroll
            for (int i = 0; i < VW; ++i) need_row |= (~seenv[i] & lv[i]) != 0;
            if (!need_row) {
                // nothing left to reach here (monotone: seen grows, live shrinks): remember it
                if (dflag != nullptr) dflag[lane] = 1;
                else s_notdone = 1;  // untracked rows cannot prove the end of the search
            } else if (nch == 0) {
                if (finalize_row<VW>(c, off, lead.x, acc, seenv, live_acc, lv, nzrows) || dflag == nullptr) s_notdone = 1;
                else dflag[lane] = 1;
            } else {
                // hub chunk: deposit the partial OR (fire-and-forget reductions at L2), then arrive with an
                // acq_rel add: the deposits are released by it, and the chunk that completes the count acquires
                // every earlier chunk's deposits through the counter's release sequence before it reads them.
                const size_t hidx = (size_t)b * p.hub_capacity + (size_t)lead.z;
                u64 *accp = p.hub_acc + hidx * WB;
#pragma unroll
                for (int q = 0; q < VW; ++q)
                    if (acc[q]) red_or_u64(accp + q, acc[q]);
                const u32 old = atom_add_acq_rel_u32(p.hub_cnt + hidx, 1u);
                if (old == (u32)nch - 1u) {
                    u64 comb[VW];
#pragma unroll
                    for (int q = 0; q < VW; ++q) comb[q] = atomicExch(accp + q, 0ull);
                    p.hub_cnt[hidx] = 0;
                    if (finalize_row<VW>(c, off, lead.x, comb, seenv, live_acc, lv, nzrows) || dflag == nullptr) s_notdone = 1;
                    else dflag[lane] = 1;
                } else {
                    s_notdone = 1;  // only the finalising chunk sees the updated mask
                }
            }
            }
            // ---- fold this batch's newly reached lanes into the CTA's live words
#pragma unroll
            for (int i = 0; i < VW; ++i) {
                const u64 x = warp_or_u64(live_acc[i]);
                if (lane == 0 && x) {
                    atomicOr(&s_live32[(b * WB + i) * 2], (u32)x);
                    atomicOr(&s_live32[(b * WB + i) * 2 + 1], (u32)(x >> 32));
                    s_any = 1;
                }
            }
        }
        nzrows = __reduce_add_sync(FULL_MASK, nzrows);
        if (lane == 0 && nzrows) atomicAdd(&s_nzrows, nzrows);
        GP_TRACE(3);
        __syncthreads();
        if (tid < lw) {
            const u64 x = ((u64)s_live32[tid * 2 + 1] << 32) | s_live32[tid * 2];
            if (x) atomicOr(live_w + tid, x);
            s_live32[tid * 2] = 0;
            s_live32[tid * 2 + 1] = 0;
        }
        const bool cta_any = s_any != 0, cta_notdone = s_notdone != 0;
        const u64 fl = grid_barrier_flags(p.bar + level % 3, gridDim.x, cta_any, cta_notdone, &s_bcast, &s_any,
                                          &s_notdone, &s_nzrows, s_queue, p.batches);
        nz_prev = bar_nzrows(fl);
        if (!bar_any(fl)) break;  // no lane reached a new row: the frontier just written is empty
        if (level >= (int)GP_UNREACHABLE_U16) {
            // a lane was first reached at hop 65535: not representable next to the 0xFFFF sentinel
            if (gtid == 0) atomicOr(&p.status[GP_BFS_ST_ERROR], GP_DEV_ERR_LEVEL_OVERFLOW);
            break;
        }
        max_level = level;
        if (!bar_notdone(fl)) break;  // every row already holds all live lanes: the next level cannot find anything
        ++level;
    }

    // ---- stats
    for (int m = 16; m; m >>= 1) gathers += shfl_xor_u64(gathers, m);
    if (lane == 0 && gathers) atomicAdd(p.counters, gathers);
    if (gtid == 0) {
        u64 t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        p.counters[3] = t;
        p.status[GP_BFS_ST_MAX_LEVEL] = max_level;
        p.status[GP_BFS_ST_LEVELS] = level;
    }
}

// Frontier bitmaps are staged in shared memory when they fit next to the work cache without costing a resident CTA;
// bitmaps too large for shared memory are read from global memory by the MAPG variant.
template <int WB>
int launch_bfs(gp_msbfs *h, const BfsParams &p, cudaStream_t stream)
{
    const int want_map = (int)((size_t)p.map_stride * sizeof(u32));
    const bool mapg = BFS_CACHE_BYTES + (size_t)p.map_stride * sizeof(u32) > 200 * 1024 / (size_t)BFS_CTAS_PER_SM;
    void (*const kernel)(BfsParams) = mapg ? msbfs_kernel<WB, true> : msbfs_kernel<WB, false>;
    const int key = WB * 2 + (mapg ? 1 : 0);
    if (h->grid_blocks == 0 || h->grid_cfg != key || h->map_want_bytes != want_map) {
        int occ = 0, occ_map = 0;
        cudaFuncAttributes fa;
        GP_CUDA_CHECK(cudaFuncGetAttributes(&fa, kernel));
        int smem_optin = 0, dev = 0;
        GP_CUDA_CHECK(cudaGetDevice(&dev));
        GP_CUDA_CHECK(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        const int dyn_room = smem_optin - (int)fa.sharedSizeBytes;
        const int cache_bytes = (int)BFS_CACHE_BYTES;
        int dyn_max = cache_bytes + GP_BFS_MAP_SMEM_MAX;
        if (dyn_max > dyn_room) dyn_max = dyn_room;
        GP_REQUIRE(dyn_max >= cache_bytes, GP_ERR_CUDA, "msbfs work cache does not fit in shared memory");
        GP_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_max));
        GP_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, BFS_THREADS, BFS_CACHE_BYTES));
        GP_REQUIRE(occ >= 1, GP_ERR_CUDA, "msbfs kernel does not fit on an SM");
        if (occ > BFS_CTAS_PER_SM) occ = BFS_CTAS_PER_SM;
        h->map_smem_bytes = 0;
        if (!mapg && cache_bytes + want_map <= dyn_max) {
            GP_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_map, kernel, BFS_THREADS,
                                                                        BFS_CACHE_BYTES + want_map));
            if (occ_map >= occ) h->map_smem_bytes = want_map;
        }
        h->grid_blocks = occ * gp_sm_count();
        h->grid_cfg = key;
        h->map_want_bytes = want_map;
    }
    BfsParams pp = p;
    pp.map_smem_words = h->map_smem_bytes > 0 ? p.map_stride : 0;
    void *args[] = {&pp};
    gp_count_launch();
    // inside a graph capture the timing events become event-record nodes (re-recorded on every replay)
    const unsigned ev_flags = gp_is_capturing() ? cudaEventRecordExternal : cudaEventRecordDefault;
    h->kernel_timed = gp_stage_events_on(h);
    if (h->kernel_timed) GP_CUDA_CHECK(cudaEventRecordWithFlags(h->ev_start, stream, ev_flags));
    GP_CUDA_CHECK(cudaLaunchCooperativeKernel((const void *)kernel, dim3(h->grid_blocks), dim3(BFS_THREADS), args,
                                              BFS_CACHE_BYTES + h->map_smem_bytes, stream));
    if (h->kernel_timed) GP_CUDA_CHECK(cudaEventRecordWithFlags(h->ev_stop, stream, ev_flags));
    return GP_OK;
}
}  // namespace

static void bfs_config(int64_t k, int *wb, int *batches)
{
    *wb = k <= 64 ? 1 : (k <= 128 ? 2 : 4);
    *batches = (int)gp_ceil_div(k > 0 ? k : 1, 64 * (*wb));
}

// Host view of a run with `num_anchors` anchors: lane layout and the array pointers inside lane_buf.  Also called
// when a captured pipeline is replayed, so the decode entry points see the layout of the run they follow.
void gp_msbfs_layout(gp_msbfs *h, int64_t num_anchors)
{
    int wb, batches;
    bfs_config(num_anchors, &wb, &batches);
    h->wb = wb;
    h->batches = batches;
    h->num_anchors = num_anchors;
    const size_t words = (size_t)wb * batches * (size_t)h->num_nodes;
    h->seeds = h->lane_buf;
    h->seen = h->lane_buf + words;  // R[0]; R[l] = seen + l * words
    h->fr_a = h->seen + (size_t)GP_BFS_RESULT_ARRAYS * words;
    h->fr_b = h->fr_a + words;
    h->fr_c = h->fr_b + words;
}

extern "C" int gp_msbfs_create(const gp_csr_t *csr, int64_t max_anchors, gp_msbfs_t **out)
{
    GP_REQUIRE(out != nullptr, GP_ERR_INVALID, "gp_msbfs_create: out is NULL");
    *out = nullptr;
    GP_REQUIRE(csr != nullptr, GP_ERR_INVALID, "gp_msbfs_create: csr is NULL");
    GP_REQUIRE(max_anchors >= 0, GP_ERR_INVALID, "gp_msbfs_create: negative anchor count");
    int wb, batches;
    bfs_config(max_anchors, &wb, &batches);
    GP_REQUIRE((int64_t)wb * batches <= GP_BFS_MAX_LANE_WORDS, GP_ERR_UNSUPPORTED,
               "gp_msbfs_create: %lld anchors exceed the %d-anchor limit per GPU", (long long)max_anchors,
               GP_BFS_MAX_LANE_WORDS * 64);
    gp_msbfs *h = new (std::nothrow) gp_msbfs();
    GP_REQUIRE(h != nullptr, GP_ERR_OOM, "gp_msbfs_create: host allocation failed");
    h->csr = csr;
    h->num_nodes = csr->num_nodes;
    h->max_anchors = max_anchors;
    h->cap_words_per_node = (int64_t)wb * batches;
    const size_t words = (size_t)h->cap_words_per_node * (size_t)(h->num_nodes > 0 ? h->num_nodes : 1);
    int rc = GP_OK;
    auto alloc = [&](void **ptr, size_t bytes) {
        if (rc != GP_OK) return;
        cudaError_t e = cudaMalloc(ptr, bytes > 0 ? bytes : 16);
        if (e != cudaSuccess) {
            gp_set_error("gp_msbfs_create: cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
            rc = (e == cudaErrorMemoryAllocation) ? GP_ERR_OOM : GP_ERR_CUDA;
        }
    };
    // lane state, one allocation: seed frontier, then the result block R[0..31] (reached mask, 15
    // first-reached-at-hop arrays, 16 deep-hop bit planes), then three rotating frontiers for hops >= 16.  The
    // seed frontier sits right before R[0] and R[1] so one memset clears the three arrays a run starts from.
    // The small per-run state sits right in front of them in the same allocation, so ONE memset per run clears it
    // together with those three arrays:
    //   live [3][MAX_LANE_WORDS] u64 | bar [8] u64 | counters [4] u64 | status [16] int | nzmap | pad || seeds | R[0] | ...
    h->nzwords = (h->num_nodes + 31) / 32;
    h->scratch_bytes = (size_t)(3 * GP_BFS_MAX_LANE_WORDS + 8 + 4) * sizeof(u64) + 16 * sizeof(int) +
                       3 * ((size_t)batches * (size_t)h->nzwords + 4) * sizeof(u32);
    h->scratch_bytes = (h->scratch_bytes + 255) / 256 * 256;
    alloc((void **)&h->scratch, h->scratch_bytes + (size_t)(1 + GP_BFS_RESULT_ARRAYS + 3) * words * sizeof(u64));
    h->lane_buf = h->scratch != nullptr ? reinterpret_cast<u64 *>((char *)h->scratch + h->scratch_bytes) : nullptr;
    h->hub_capacity = csr->hub_capacity;
    alloc((void **)&h->hub_acc, (size_t)h->hub_capacity * (size_t)h->cap_words_per_node * sizeof(u64));
    alloc((void **)&h->hub_cnt, (size_t)h->hub_capacity * (size_t)h->cap_words_per_node * sizeof(u32));
    if (rc == GP_OK) {
        h->live = reinterpret_cast<u64 *>(h->scratch);
        h->bar = h->live + 3 * GP_BFS_MAX_LANE_WORDS;
        h->counters = h->bar + 8;
        h->status = reinterpret_cast<int *>(h->counters + 4);
        h->nzmap = reinterpret_cast<u32 *>(h->status + 16);
    }
    if (gp_env().bfs_trace) alloc((void **)&h->trace, GP_BFS_TRACE_WORDS * sizeof(u64));
    if (rc == GP_OK && (cudaEventCreate(&h->ev_start) != cudaSuccess || cudaEventCreate(&h->ev_stop) != cudaSuccess ||
                        cudaEventCreate(&h->ev_pipe0) != cudaSuccess || cudaEventCreate(&h->ev_pipe1) != cudaSuccess)) {
        gp_set_error("gp_msbfs_create: cudaEventCreate failed");
        rc = GP_ERR_CUDA;
    }
    if (rc != GP_OK) {
        gp_msbfs_free(h);
        return rc;
    }
    *out = h;
    return GP_OK;
}

extern "C" int gp_msbfs_free(gp_msbfs_t *h)
{
    if (!h) return GP_OK;
    gp_pipe_cache_free(h->pipe_cache);
    cudaFree(h->scratch);  // the lane arrays live in the same allocation
    cudaFree(h->hub_acc);
    cudaFree(h->hub_cnt);
    cudaFree(h->packed);
    cudaFree(h->deep_flag);
    cudaFree(h->trace);
    if (h->ev_start) cudaEventDestroy(h->ev_start);
    if (h->ev_stop) cudaEventDestroy(h->ev_stop);
    if (h->ev_pipe0) cudaEventDestroy(h->ev_pipe0);
    if (h->ev_pipe1) cudaEventDestroy(h->ev_pipe1);
    delete h;
    return GP_OK;
}

extern "C" int gp_msbfs_run(gp_msbfs_t *h, const int64_t *d_anchors, int64_t num_anchors, gp_stream_t stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    GP_REQUIRE(h != nullptr, GP_ERR_INVALID, "gp_msbfs_run: handle is NULL");
    GP_REQUIRE(h->csr->built, GP_ERR_INVALID, "gp_msbfs_run: the CSR has not been built");
    GP_REQUIRE(h->csr->num_nodes == h->num_nodes, GP_ERR_INVALID, "gp_msbfs_run: CSR changed size");
    GP_REQUIRE(num_anchors >= 0 && num_anchors <= h->max_anchors, GP_ERR_INVALID,
               "gp_msbfs_run: %lld anchors exceed max_anchors %lld", (long long)num_anchors,
               (long long)h->max_anchors);
    GP_REQUIRE(num_anchors == 0 || d_anchors != nullptr, GP_ERR_INVALID, "gp_msbfs_run: anchors is NULL");
    gp_msbfs_layout(h, num_anchors);
    h->ran = false;
    const int wb = h->wb, batches = h->batches;
    const int64_t n = h->num_nodes;
    const size_t words = (size_t)wb * batches * (size_t)n;
    const int map_stride = (int)(((int64_t)batches * h->nzwords + 3) / 4 * 4);
    if (n == 0 || num_anchors == 0) {
        GP_CUDA_CHECK(cudaMemsetAsync(h->scratch, 0, h->scratch_bytes, stream));  // status / counters, read by gp_msbfs_stats
        h->ran = true;
        return GP_OK;
    }
    // ONE memset: live, bar, counters, status, maps + seeds, reached mask and the hop-1 frontier; every later frontier
    // array is cleared by the kernel one level before it is written
    GP_CUDA_CHECK(cudaMemsetAsync(h->scratch, 0, h->scratch_bytes + 3 * words * sizeof(u64), stream));
    if (!h->hub_zeroed) {
        // the kernel leaves these zeroed again (the finalising chunk resets its row's words)
        GP_CUDA_CHECK(cudaMemsetAsync(h->hub_acc, 0, (size_t)h->hub_capacity * h->cap_words_per_node * sizeof(u64), stream));
        GP_CUDA_CHECK(cudaMemsetAsync(h->hub_cnt, 0, (size_t)h->hub_capacity * h->cap_words_per_node * sizeof(u32), stream));
        h->hub_zeroed = true;
    }
    BfsParams p;
    p.n = (int)n;
    p.batches = batches;
    p.num_anchors = (int)num_anchors;
    p.hub_capacity = (int)h->hub_capacity;
    p.desc = h->csr->desc;
    for (int k = 0; k < GP_NUM_CLASSES; ++k) p.desc_off[k] = h->csr->desc_off[k];
    p.hub_acc = h->hub_acc;
    p.hub_cnt = h->hub_cnt;
    p.bar = h->bar;
    p.nzmap = h->nzmap;
    p.nzwords = (int)h->nzwords;
    p.map_stride = map_stride;
    p.map_smem_words = 0;  // decided by launch_bfs
    p.col = h->csr->col;
    p.meta = h->csr->meta;
    p.anchors = (const long long *)d_anchors;
    p.result = h->seen;
    p.seeds = h->seeds;
    p.fr_a = h->fr_a;
    p.fr_b = h->fr_b;
    p.fr_c = h->fr_c;
    p.plane_stride = (long long)words;
    p.live = h->live;
    p.status = h->status;
    p.counters = h->counters;
    p.trace = h->trace;
    GP_TRY(wb == 1 ? launch_bfs<1>(h, p, stream) : wb == 2 ? launch_bfs<2>(h, p, stream)
                                                             : launch_bfs<4>(h, p, stream));
    h->ran = true;
    return GP_OK;
}

bool gp_stage_events_on(const gp_msbfs *h)
{
    if (!gp_is_capturing()) return true;
    return (h->stage_events < 0 ? gp_env().stage_events : h->stage_events) != 0;
}

extern "C" int gp_msbfs_set_stage_events(gp_msbfs_t *h, int32_t enable)
{
    GP_REQUIRE(h != nullptr, GP_ERR_INVALID, "gp_msbfs_set_stage_events: handle is NULL");
    h->stage_events = enable ? 1 : 0;
    gp_pipe_cache_free(h->pipe_cache);  // captured pipelines were recorded with the other setting
    h->pipe_cache = nullptr;
    return GP_OK;
}

// Device-clock duration of the last MS-BFS kernel: %globaltimer at the entry of thread 0 and after the last level, in
// nanoseconds (no event nodes needed: this is what the timed loop of bench.py reads).  syncs the stream.
extern "C" int gp_msbfs_kernel_device_ns(gp_msbfs_t *h, uint64_t *ns, gp_stream_t stream_)
{
    GP_REQUIRE(h != nullptr && ns != nullptr, GP_ERR_INVALID, "gp_msbfs_kernel_device_ns: NULL argument");
    GP_REQUIRE(h->ran, GP_ERR_INVALID, "gp_msbfs_kernel_device_ns: gp_msbfs_run has not been called");
    u64 st[2] = {0, 0};
    *ns = 0;
    if (h->num_nodes == 0 || h->num_anchors == 0) return GP_OK;
    GP_CUDA_CHECK(cudaMemcpyAsync(st, h->counters + 2, sizeof(st), cudaMemcpyDeviceToHost, (cudaStream_t)stream_));
    GP_CUDA_CHECK(cudaStreamSynchronize((cudaStream_t)stream_));
    *ns = st[1] > st[0] ? st[1] - st[0] : 0;
    return GP_OK;
}

// Hop 1 always pulls; the entry point stays for programs built against ABI version 1.
extern "C" int gp_msbfs_set_push(gp_msbfs_t *h, int32_t enable)
{
    GP_REQUIRE(h != nullptr, GP_ERR_INVALID, "gp_msbfs_set_push: handle is NULL");
    GP_REQUIRE(enable == 0, GP_ERR_UNSUPPORTED, "gp_msbfs_set_push: hop 1 always pulls; push direction is not supported");
    return GP_OK;
}

extern "C" int gp_msbfs_stats(gp_msbfs_t *h, gp_msbfs_stats_t *stats, gp_stream_t stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    GP_REQUIRE(h != nullptr && stats != nullptr, GP_ERR_INVALID, "gp_msbfs_stats: NULL argument");
    GP_REQUIRE(h->ran, GP_ERR_INVALID, "gp_msbfs_stats: gp_msbfs_run has not been called");
    int st[GP_BFS_ST_WORDS];
    u64 cnt[4];
    int csr_err = 0;
    GP_CUDA_CHECK(cudaMemcpyAsync(st, h->status, sizeof(st), cudaMemcpyDeviceToHost, stream));
    GP_CUDA_CHECK(cudaMemcpyAsync(cnt, h->counters, sizeof(cnt), cudaMemcpyDeviceToHost, stream));
    GP_CUDA_CHECK(cudaMemcpyAsync(&csr_err, &h->csr->meta[GP_META_ERROR], sizeof(int), cudaMemcpyDeviceToHost,
                                  stream));
    GP_CUDA_CHECK(cudaStreamSynchronize(stream));
    stats->num_anchors = h->num_anchors;
    stats->lane_words = (int64_t)h->wb * h->batches;
    stats->max_level = st[GP_BFS_ST_MAX_LEVEL];
    stats->levels_run = st[GP_BFS_ST_LEVELS];
    stats->pull_levels = st[GP_BFS_ST_LEVELS];  // every level pulls
    stats->push_levels = 0;
    stats->edges_examined = (int64_t)cnt[0];
    stats->grid_blocks = h->grid_blocks;
    GP_REQUIRE(!(csr_err & GP_DEV_ERR_EDGE_RANGE), GP_ERR_INDEX_RANGE,
               "edge_index holds an entry outside [0, %lld)", (long long)h->num_nodes);
    GP_REQUIRE(!(st[GP_BFS_ST_ERROR] & GP_DEV_ERR_ANCHOR_RANGE), GP_ERR_INDEX_RANGE,
               "anchor index outside [0, %lld)", (long long)h->num_nodes);
    GP_REQUIRE(!(st[GP_BFS_ST_ERROR] & GP_DEV_ERR_LEVEL_OVERFLOW), GP_ERR_LEVEL_OVERFLOW,
               "a hop distance reached 65535 and does not fit the uint16 distance matrix");
    return GP_OK;
}

extern "C" int gp_msbfs_trace(gp_msbfs_t *h, uint64_t *h_out, int64_t cap_words, int32_t *levels, int32_t *warps)
{
    GP_REQUIRE(h != nullptr && h_out != nullptr && levels && warps, GP_ERR_INVALID, "gp_msbfs_trace: NULL argument");
    GP_REQUIRE(h->trace != nullptr, GP_ERR_INVALID, "gp_msbfs_trace: set GP_BFS_TRACE=1 before gp_msbfs_create");
    gp_msbfs_stats_t st;
    gp_msbfs_stats(h, &st, nullptr);
    GP_CUDA_CHECK(cudaDeviceSynchronize());
    *levels = st.levels_run < 32 ? st.levels_run : 32;
    *warps = h->grid_blocks * BFS_WARPS;
    const int64_t words = (int64_t)32 * (*warps) * 4;  // all 32 rows: row 31 holds the prologue stamps of shallow runs
    GP_REQUIRE(words <= cap_words && words <= GP_BFS_TRACE_WORDS, GP_ERR_INVALID, "gp_msbfs_trace: buffer too small");
    GP_CUDA_CHECK(cudaMemcpy(h_out, h->trace, sizeof(u64) * (size_t)words, cudaMemcpyDeviceToHost));
    return GP_OK;
}

extern "C" int gp_msbfs_kernel_ms(gp_msbfs_t *h, float *ms)
{
    GP_REQUIRE(h != nullptr && ms != nullptr, GP_ERR_INVALID, "gp_msbfs_kernel_ms: NULL argument");
    GP_REQUIRE(h->ran, GP_ERR_INVALID, "gp_msbfs_kernel_ms: gp_msbfs_run has not been called");
    GP_REQUIRE(h->kernel_timed, GP_ERR_INVALID, "gp_msbfs_kernel_ms: the last run replayed a pipeline captured without "
               "stage events (gp_msbfs_set_stage_events); gp_msbfs_kernel_device_ns needs none");
    *ms = 0.0f;
    if (h->num_nodes == 0 || h->num_anchors == 0) return GP_OK;
    GP_CUDA_CHECK(cudaEventSynchronize(h->ev_stop));
    GP_CUDA_CHECK(cudaEventElapsedTime(ms, h->ev_start, h->ev_stop));
    return GP_OK;
}

extern "C" int gp_pipeline_stage_ms(gp_msbfs_t *h, float *ms3)
{
    GP_REQUIRE(h != nullptr && ms3 != nullptr, GP_ERR_INVALID, "gp_pipeline_stage_ms: NULL argument");
    GP_REQUIRE(h->ran && h->pipe_timed && h->kernel_timed, GP_ERR_INVALID,
               "gp_pipeline_stage_ms: no fused run with stage events on this handle (gp_msbfs_set_stage_events)");
    ms3[0] = ms3[1] = ms3[2] = 0.0f;
    if (h->num_nodes == 0 || h->num_anchors == 0) return GP_OK;
    GP_CUDA_CHECK(cudaEventSynchronize(h->ev_pipe1));
    GP_CUDA_CHECK(cudaEventElapsedTime(ms3 + 0, h->ev_pipe0, h->ev_start));
    GP_CUDA_CHECK(cudaEventElapsedTime(ms3 + 1, h->ev_start, h->ev_stop));
    GP_CUDA_CHECK(cudaEventElapsedTime(ms3 + 2, h->ev_stop, h->ev_pipe1));
    return GP_OK;
}

extern "C" int gp_msbfs_planes(gp_msbfs_t *h, const uint64_t **d_planes, int64_t *plane_stride_words,
                               int32_t *num_planes, int32_t *batches, int32_t *words_per_batch,
                               gp_stream_t stream_)
{
    GP_REQUIRE(h != nullptr && d_planes && plane_stride_words && num_planes && batches && words_per_batch,
               GP_ERR_INVALID, "gp_msbfs_planes: NULL argument");
    gp_msbfs_stats_t st;
    GP_TRY(gp_msbfs_stats(h, &st, stream_));
    *d_planes = (const uint64_t *)h->seen;
    *plane_stride_words = (int64_t)h->wb * h->batches * h->num_nodes;
    *num_planes = st.max_level <= GP_BFS_LEVEL_ARRAYS ? 1 + st.max_level : GP_BFS_RESULT_ARRAYS;
    *batches = h->batches;
    *words_per_batch = h->wb;
    return GP_OK;
}
