// gp_exchange.cu — the exchange step of the anchor-sharded path as ONE kernel over NVLink peer memory:
// pack -> gather from every rank -> decode, with no collective library call and no host round trip.
//
// The reference has no device exchange: its pool workers pickle their result dicts back to the parent
// (utils.py:98-106) and every DDP rank recomputes everything (main.py:88-98).  Here the anchors are sharded over
// the GPUs of one NVSwitch node and every rank must end up with the full float32 [N, F + K] matrix.  Round 1
// packed, all-reduced a flag through NCCL (22-26 us, only there to order pack before decode) and then let the
// epilogue read the peers' packed shards with ordinary loads, one dependent NVLink round trip per output row.
// This kernel (one resident wave, launched cooperatively) does, per rank:
//   pack     rewrite the rank's result into the 5-plane exchange format (reached mask + 4 hop-index bit planes,
//            valid for hops <= 15) in its OWN exchange buffer, slot [step parity]; blocks count themselves out
//            (acq_rel counter) and the last one writes "epoch, deep bit" with st.release.sys into flag
//            [parity][this rank] of every peer;
//   wait     one thread per block polls (ld.acquire.sys, bounded) until every peer's flag shows this step's epoch:
//            their packed shards are complete and visible;
//   stream   ONE pass over the node rows in blocks of 8-64 rows.  One thread per block drives the bulk-copy engine
//            (cp.async.bulk peer global -> shared, completion on an mbarrier, three stages, two blocks ahead): the
//            5 x (G-1) packed row segments of a block arrive in shared memory while the warps stream earlier rows,
//            so the NVLink transfer is spread over the whole HBM-bound pass and costs no load/store unit work.
//            A warp writes whole output rows: x (concat_into_features, utils.py:129-135), the rank's own columns
//            decoded from the unpacked result, the peers' columns decoded from shared memory.
// Slots are double-buffered by step parity: a rank can only pack step t+2 after it has seen every peer's flag of
// step t+1, which a peer raises after finishing step t, so nobody overwrites a slot that is still being read.
// Blocks wait for other GPUs, so all blocks of all ranks must be running: the grid is one resident wave.  Waiting
// is bounded (GP_XCHG_TIMEOUT_CYCLES): a rank whose peer died reports GP_ERR_CUDA instead of hanging the GPU.
// Measured dead ends (profiles/r02_notes.md): PUSHING the packed shard with ordinary stores — posted stores to
// peer memory back-pressure the SM's local streaming stores (phase times 1.3-2x), a fence.sc.sys before the flag
// costs ~20 us behind them, dedicated pushing blocks need dynamic row hand-out whose same-address atomics cost
// ~30 us per pass.
#include "gp_msbfs.cuh"
#include "gp_tma.cuh"

#include <new>

struct gp_exchange {
    uint64_t uid = gp_next_uid();
    gp_msbfs *bfs = nullptr;
    int world = 1, rank = 0;
    size_t cap_words = 0;          // lane words per plane the slots were sized for
    size_t pk_stride = 0;          // words between packed planes (cap_words rounded up to 16-byte multiples)
    unsigned char *buf = nullptr;  // flags [2][GP_MAX_RANKS] u32 (256 B) | packed [2][5][pk_stride] u64 | pad
    unsigned char *peer[GP_MAX_RANKS] = {};  // base of every rank's buffer (own = buf)
    u32 *local = nullptr;          // [0..1] epoch of each parity, [2..3] blocks packed, [4] deep (last step), [5] timeout,
                                   // [6..7] blocks left; bytes 64..: u64 globaltimer stamps (diagnostics)
    int step = 0;
    int grid_blocks = 0;
    int grid_cap = 0;
    int smem_bytes = 0;
};

namespace {

constexpr int XCHG_THREADS = 256;
constexpr int XCHG_WARPS = XCHG_THREADS / 32;
constexpr size_t XCHG_FLAG_BYTES = 256;
constexpr int XCHG_STAGES = 3;
constexpr int XCHG_STAGE_CAP = 18 * 1024;  // bytes of peer segments per stage
constexpr long long GP_XCHG_TIMEOUT_CYCLES = 16000000000ll;  // ~8 s at 1.9 GHz

struct XchgParams {
    // local result (gp_msbfs.cu layout)
    const u64 *result;
    const int *status;
    long long plane_stride;   // words per array of the local result = wb * batches * n
    long long n;
    int wb, batches, kr;      // lanes of one shard
    int world, rank, parity;
    size_t pk_stride;
    int block_rows;           // node rows per streamed block
    int seg_stride;           // bytes of one (peer, plane, batch) segment in a stage = block_rows * wb * 8
    int stage_bytes;
    int debug;
    unsigned char *peer[GP_MAX_RANKS];
    u32 *local;
    const float *x;
    long long num_features, ld_x;
    float *out;
    long long ld_out, col_offset;
    int vec_x;
};

__device__ __forceinline__ float inv_hops_x(u32 d) { return __fdiv_rn(1.0f, __uint2float_rn(d + 1u)); }

__device__ __forceinline__ u64 *packed_ptr(const XchgParams &p, int rank)
{
    return reinterpret_cast<u64 *>(p.peer[rank] + XCHG_FLAG_BYTES) + (size_t)p.parity * GP_PACKED_ARRAYS * p.pk_stride;
}

__device__ __forceinline__ u32 *flag_ptr(const XchgParams &p, int dest, int src)
{
    return reinterpret_cast<u32 *>(p.peer[dest]) + p.parity * GP_MAX_RANKS + src;
}

__device__ __forceinline__ void copy_x_row_x(const float *xrow, float *orow, int f, int lane, int vec_x)
{
    constexpr int T = 4;
    if (vec_x) {
        const float4 *x4 = reinterpret_cast<const float4 *>(xrow);
        float4 *o4 = reinterpret_cast<float4 *>(orow);
        const int q = f >> 2;
        for (int i0 = 0; i0 < q; i0 += 32 * T) {
            float4 v[T];
#pragma unroll
            for (int t = 0; t < T; ++t) {
                const int i = i0 + lane + 32 * t;
                if (i < q) v[t] = __ldcs(x4 + i);
            }
#pragma unroll
            for (int t = 0; t < T; ++t) {
                const int i = i0 + lane + 32 * t;
                if (i < q) __stcs(o4 + i, v[t]);
            }
        }
        for (int i = (q << 2) + lane; i < f; i += 32) orow[i] = __ldcs(xrow + i);
    } else {
        for (int i = lane; i < f; i += 32) orow[i] = __ldcs(xrow + i);
    }
}

// 8 columns of one (node, rank, batch, lane byte) from the 5 packed bytes.
__device__ __forceinline__ void store8(float *dst, u32 reach, u32 m0, u32 m1, u32 m2, u32 m3, const float *s_inv)
{
    float v[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const u32 d = ((m0 >> c) & 1u) | (((m1 >> c) & 1u) << 1) | (((m2 >> c) & 1u) << 2) | (((m3 >> c) & 1u) << 3);
        v[c] = ((reach >> c) & 1u) ? s_inv[d] : 0.0f;
    }
    __stcs(reinterpret_cast<float4 *>(dst), make_float4(v[0], v[1], v[2], v[3]));
    __stcs(reinterpret_cast<float4 *>(dst) + 1, make_float4(v[4], v[5], v[6], v[7]));
}

__global__ void __launch_bounds__(XCHG_THREADS, 4) exchange_decode_kernel(XchgParams p)
{
    extern __shared__ __align__(128) unsigned char s_stage[];  // [XCHG_STAGES][stage_bytes]
    __shared__ __align__(8) u64 s_full[XCHG_STAGES];
    __shared__ float s_inv[16];
    __shared__ u32 s_epoch;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < 16) s_inv[tid] = inv_hops_x((u32)tid);
    if (tid == 0) {
        // The epoch of this step: one more than the rank's counter for this parity.  The counter is bumped by the
        // last block to LEAVE the kernel, i.e. after every block has read it here.
        s_epoch = ld_relaxed_u32(p.local + p.parity) + 1u;
        for (int s = 0; s < XCHG_STAGES; ++s) gp_mbar_init(gp_smem_addr(&s_full[s]), 1);
        gp_mbar_init_fence();
    }
    __syncthreads();
    const u32 epoch = s_epoch;
    const int ml = p.status[GP_BFS_ST_MAX_LEVEL];
    const int levels = min(ml, GP_BFS_LEVEL_ARRAYS);
    const u32 deep = ml > GP_BFS_LEVEL_ARRAYS ? 1u : 0u;
    const long long gthreads = (long long)gridDim.x * XCHG_THREADS;
    const long long gtid = (long long)blockIdx.x * XCHG_THREADS + tid;
    u64 *stamp = reinterpret_cast<u64 *>(p.local + 16);
    auto now = [] {
        u64 t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        return t;
    };
    if (gtid == 0) stamp[0] = now();

    if (p.world > 1) {
        // ---- pack: the rank's shard in the exchange format, into its own buffer
        u64 *mine = packed_ptr(p, p.rank);
        for (long long i = gtid; i < p.plane_stride; i += gthreads) {
            u64 m0 = 0, m1 = 0, m2 = 0, m3 = 0;
            const u64 reach = p.result[i];
            u64 w[GP_BFS_LEVEL_ARRAYS];
#pragma unroll
            for (int l = 1; l <= GP_BFS_LEVEL_ARRAYS; ++l)  // all level words requested together
                w[l - 1] = l <= levels ? p.result[(size_t)l * p.plane_stride + i] : 0ull;
#pragma unroll
            for (int l = 1; l <= GP_BFS_LEVEL_ARRAYS; ++l) {
                if (l & 1) m0 |= w[l - 1];
                if (l & 2) m1 |= w[l - 1];
                if (l & 4) m2 |= w[l - 1];
                if (l & 8) m3 |= w[l - 1];
            }
            mine[i] = reach;
            mine[p.pk_stride + i] = m0;
            mine[2 * p.pk_stride + i] = m1;
            mine[3 * p.pk_stride + i] = m2;
            mine[4 * p.pk_stride + i] = m3;
        }
        __syncthreads();
        if (tid == 0) {
            u32 old;  // acq_rel: this block's stores (ordered by the barrier above) are released, earlier blocks' acquired
            asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(old) : "l"(p.local + 2 + p.parity) : "memory");
            if (old == gridDim.x - 1) {
                p.local[2 + p.parity] = 0;
                for (int q = 1; q < p.world; ++q)
                    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flag_ptr(p, (p.rank + q) % p.world, p.rank)),
                                 "r"((epoch << 1) | deep)
                                 : "memory");
            }
            if (gtid == 0) stamp[1] = now();
            // ---- wait: every peer's shard is packed and visible
            u32 any_deep = deep;
            bool timed_out = false;
            for (int q = 1; q < p.world && !(p.debug & 1); ++q) {
                const u32 *fp = flag_ptr(p, p.rank, (p.rank + q) % p.world);
                const long long t0 = clock64();
                u32 f;
                for (;;) {
                    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(f) : "l"(fp) : "memory");
                    if ((f >> 1) == epoch) break;
                    if (clock64() - t0 > GP_XCHG_TIMEOUT_CYCLES) {
                        timed_out = true;
                        break;
                    }
                }
                any_deep |= f & 1u;
            }
            if (timed_out) atomicExch(p.local + 5, 1u);  // sticky: a dead peer is fatal
            // every block has seen the same flags: block 0 writes this step's deep bit (0 or 1), so a shallow step
            // after a deep one reports 0
            if (blockIdx.x == 0) p.local[4] = any_deep;
            if (gtid == 0) stamp[2] = now();
        }
        __syncthreads();
    } else if (gtid == 0) {
        p.local[4] = deep;
    }

    // ---- stream: one pass over the row blocks; thread 0 keeps the bulk-copy engine two blocks ahead
    const int RB = p.block_rows;
    const long long nblk = (p.n + RB - 1) / RB;
    const long long first = blockIdx.x, step = gridDim.x;
    const long long cnt = nblk > first ? (nblk - first + step - 1) / step : 0;
    const int row_bytes = p.wb * 8;
    const size_t plane_bytes = (size_t)p.plane_stride * 8;
    const unsigned char *own = reinterpret_cast<const unsigned char *>(p.result);
    const u32 stage0 = gp_smem_addr(s_stage);
    auto prefetch = [&](long long k) {  // thread 0 only
        const int s = (int)(k % XCHG_STAGES);
        const long long u0 = (first + k * step) * RB;
        const int rows = (int)(p.n - u0 < RB ? p.n - u0 : RB);
        const u32 seg = (u32)((rows * row_bytes + 15) & ~15);  // the buffers carry slack for the rounded-up tail
        const u32 bar = gp_smem_addr(&s_full[s]);
        gp_mbar_expect_tx(bar, seg * (u32)((p.world - 1) * GP_PACKED_ARRAYS * p.batches));
        u32 dst = stage0 + (u32)s * (u32)p.stage_bytes;
        for (int q = 1; q < p.world; ++q) {
            const unsigned char *src = reinterpret_cast<const unsigned char *>(packed_ptr(p, (p.rank + q) % p.world));
            for (int a = 0; a < GP_PACKED_ARRAYS; ++a)
                for (int b = 0; b < p.batches; ++b) {
                    gp_bulk_load(dst, src + ((size_t)a * p.pk_stride) * 8 + ((size_t)b * p.n + (size_t)u0) * row_bytes, seg, bar);
                    dst += (u32)p.seg_stride;
                }
        }
    };
    if (p.world > 1 && tid == 0)
        for (long long k = 0; k < XCHG_STAGES - 1 && k < cnt; ++k) prefetch(k);
    for (long long k = 0; k < cnt; ++k) {
        const int s = (int)(k % XCHG_STAGES);
        if (p.world > 1) {
            // stage (k + 2) % 3 was last read in iteration k - 1, which every warp left through the barrier below
            if (tid == 0 && k + XCHG_STAGES - 1 < cnt) prefetch(k + XCHG_STAGES - 1);
            gp_mbar_wait(gp_smem_addr(&s_full[s]), (u32)((k / XCHG_STAGES) & 1));
        }
        const long long u0 = (first + k * step) * RB;
        const long long u1 = u0 + RB < p.n ? u0 + RB : p.n;
        const unsigned char *st = s_stage + (size_t)s * p.stage_bytes;
        for (long long u = u0 + warp; u < u1; u += XCHG_WARPS) {
            float *orow = p.out + (size_t)u * p.ld_out;
            if (p.x != nullptr) copy_x_row_x(p.x + (size_t)u * p.ld_x, orow, (int)p.num_features, lane, p.vec_x);
            for (int b = 0; b < p.batches; ++b) {
                const int col0 = b * 64 * p.wb + lane * 8;
                if (lane >= row_bytes || col0 >= p.kr) continue;
                const unsigned char *rowp = own + ((size_t)b * p.n + (size_t)u) * row_bytes + lane;
                const u32 reach = rowp[0];
                u32 m0 = 0, m1 = 0, m2 = 0, m3 = 0;
                if (reach) {
#pragma unroll
                    for (int l = 1; l <= GP_BFS_LEVEL_ARRAYS; ++l) {
                        if (l <= levels) {
                            const u32 bl = rowp[(size_t)l * plane_bytes];
                            if (l & 1) m0 |= bl;
                            if (l & 2) m1 |= bl;
                            if (l & 4) m2 |= bl;
                            if (l & 8) m3 |= bl;
                        }
                    }
                }
                store8(orow + p.col_offset + (size_t)p.rank * p.kr + col0, reach, m0, m1, m2, m3, s_inv);
                // the peers' columns of this row: five bytes per peer out of the staged segments
                const unsigned char *sp = st + (size_t)b * p.seg_stride + (size_t)(u - u0) * row_bytes + lane;
                for (int q = 1; q < p.world; ++q) {
                    const int src = (p.rank + q) % p.world;
                    const size_t ps = (size_t)p.batches * p.seg_stride;  // stride between planes of one peer
                    const unsigned char *pp = sp + (size_t)(q - 1) * GP_PACKED_ARRAYS * ps;
                    store8(orow + p.col_offset + (size_t)src * p.kr + col0, pp[0], pp[ps], pp[2 * ps], pp[3 * ps], pp[4 * ps],
                           s_inv);
                }
            }
        }
        if (p.world > 1) __syncthreads();  // the stage may be refilled
    }
    // ---- the last block to leave publishes the epoch for the next step of this parity
    __syncthreads();
    if (tid == 0) {
        u32 old;
        asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(old) : "l"(p.local + 6 + p.parity) : "memory");
        if (old == gridDim.x - 1) {
            p.local[6 + p.parity] = 0;
            asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p.local + p.parity), "r"(epoch) : "memory");
            stamp[3] = now();
        }
    }
}

}  // namespace

extern "C" int gp_exchange_create(gp_msbfs_t *bfs, int32_t world, int32_t rank, gp_exchange_t **out)
{
    GP_REQUIRE(out != nullptr, GP_ERR_INVALID, "gp_exchange_create: out is NULL");
    *out = nullptr;
    GP_REQUIRE(bfs != nullptr && world >= 1 && world <= GP_MAX_RANKS && rank >= 0 && rank < world, GP_ERR_INVALID,
               "gp_exchange_create: bad argument (1..%d ranks)", GP_MAX_RANKS);
    gp_exchange *x = new (std::nothrow) gp_exchange();
    GP_REQUIRE(x != nullptr, GP_ERR_OOM, "gp_exchange_create: host allocation failed");
    x->bfs = bfs;
    x->world = world;
    x->rank = rank;
    x->cap_words = (size_t)bfs->cap_words_per_node * (size_t)(bfs->num_nodes > 0 ? bfs->num_nodes : 1);
    x->pk_stride = (x->cap_words + 1) & ~(size_t)1;  // planes start on 16-byte boundaries (bulk copies)
    const size_t bytes = XCHG_FLAG_BYTES + 2 * (size_t)GP_PACKED_ARRAYS * x->pk_stride * sizeof(u64) + 64;
    cudaError_t e = cudaMalloc((void **)&x->buf, bytes);
    if (e == cudaSuccess) e = cudaMemset(x->buf, 0, bytes);
    if (e == cudaSuccess) e = cudaMalloc((void **)&x->local, 256);
    if (e == cudaSuccess) e = cudaMemset(x->local, 0, 256);
    if (e != cudaSuccess) {
        gp_set_error("gp_exchange_create: allocating %zu bytes failed: %s", bytes, cudaGetErrorString(e));
        cudaFree(x->buf);
        cudaFree(x->local);
        delete x;
        return e == cudaErrorMemoryAllocation ? GP_ERR_OOM : GP_ERR_CUDA;
    }
    x->peer[rank] = x->buf;
    *out = x;
    return GP_OK;
}

extern "C" int gp_exchange_ipc_export(gp_exchange_t *x, uint8_t *handle64)
{
    GP_REQUIRE(x != nullptr && handle64 != nullptr, GP_ERR_INVALID, "gp_exchange_ipc_export: NULL argument");
    cudaIpcMemHandle_t hd;
    GP_CUDA_CHECK(cudaIpcGetMemHandle(&hd, x->buf));
    memcpy(handle64, &hd, 64);
    return GP_OK;
}

extern "C" int gp_exchange_local_ptr(gp_exchange_t *x, void **d_ptr)
{
    GP_REQUIRE(x != nullptr && d_ptr != nullptr, GP_ERR_INVALID, "gp_exchange_local_ptr: NULL argument");
    *d_ptr = x->buf;
    return GP_OK;
}

extern "C" int gp_exchange_set_peer(gp_exchange_t *x, int32_t rank, void *d_ptr)
{
    GP_REQUIRE(x != nullptr && rank >= 0 && rank < x->world && d_ptr != nullptr, GP_ERR_INVALID,
               "gp_exchange_set_peer: bad argument");
    GP_REQUIRE(rank != x->rank || d_ptr == x->buf, GP_ERR_INVALID, "gp_exchange_set_peer: own slot is fixed");
    x->peer[rank] = (unsigned char *)d_ptr;
    return GP_OK;
}

extern "C" int gp_exchange_free(gp_exchange_t *x)
{
    if (!x) return GP_OK;
    cudaFree(x->buf);
    cudaFree(x->local);
    delete x;
    return GP_OK;
}

// syncs.  *deep = 1 if some rank's shard had hops > 15 in the last step (packed format invalid: use the
// all-gather path); GP_ERR_CUDA if a peer's flag never arrived.
extern "C" int gp_exchange_status(gp_exchange_t *x, int32_t *deep, gp_stream_t stream_)
{
    GP_REQUIRE(x != nullptr, GP_ERR_INVALID, "gp_exchange_status: NULL argument");
    u32 st[2] = {0, 0};
    GP_CUDA_CHECK(cudaMemcpyAsync(st, x->local + 4, sizeof(st), cudaMemcpyDeviceToHost, (cudaStream_t)stream_));
    GP_CUDA_CHECK(cudaStreamSynchronize((cudaStream_t)stream_));
    if (deep) *deep = (int32_t)st[0];
    GP_REQUIRE(st[1] == 0, GP_ERR_CUDA, "exchange: a peer rank's result never arrived (timed out waiting for its flag)");
    return GP_OK;
}

// Diagnostics: globaltimer stamps (ns) of the last step: [0] block 0 starts, [1] block 0 has packed its share,
// [2] block 0 has seen every peer's flag, [3] the last block leaves.  syncs the device.
extern "C" int gp_exchange_trace(gp_exchange_t *x, uint64_t *h_stamps8)
{
    GP_REQUIRE(x != nullptr && h_stamps8 != nullptr, GP_ERR_INVALID, "gp_exchange_trace: NULL argument");
    GP_CUDA_CHECK(cudaDeviceSynchronize());
    GP_CUDA_CHECK(cudaMemcpy(h_stamps8, x->local + 16, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return GP_OK;
}

uint64_t gp_exchange_uid(const gp_exchange *x) { return x->uid; }

// Tuning / tests: cap the cooperative grid (several ranks sharing one GPU must all be resident at once).  Takes
// effect at the next launch; 0 restores one full wave.
extern "C" int gp_exchange_set_grid(gp_exchange_t *x, int32_t max_blocks)
{
    GP_REQUIRE(x != nullptr && max_blocks >= 0, GP_ERR_INVALID, "gp_exchange_set_grid: bad argument");
    x->grid_cap = max_blocks;
    x->grid_blocks = 0;
    return GP_OK;
}

int gp_exchange_next_parity(gp_exchange *x) { return (x->step++) & 1; }

int gp_exchange_launch(gp_exchange *x, int parity, const float *d_x, int64_t f, int64_t ldx, float *d_out, int64_t ldo,
                       int64_t coff, cudaStream_t stream)
{
    gp_msbfs *h = x->bfs;
    GP_REQUIRE(h->ran, GP_ERR_INVALID, "exchange: gp_msbfs_run has not been called");
    for (int r = 0; r < x->world; ++r)
        GP_REQUIRE(x->peer[r] != nullptr, GP_ERR_INVALID, "exchange: rank %d's buffer has not been set", r);
    const int64_t kr = h->num_anchors;
    GP_REQUIRE(kr > 0 && kr % 8 == 0, GP_ERR_INVALID, "exchange: anchors per rank must be a positive multiple of 8");
    GP_REQUIRE(d_out != nullptr && ldo >= coff + kr * x->world && ldo % 4 == 0 && coff % 4 == 0 &&
                   (reinterpret_cast<uintptr_t>(d_out) & 15u) == 0,
               GP_ERR_INVALID, "exchange: output must be 16-byte aligned with ld_out, col_offset multiples of 4");
    XchgParams p;
    memset(&p, 0, sizeof(p));
    p.result = h->seen;
    p.status = h->status;
    p.plane_stride = (long long)h->wb * h->batches * h->num_nodes;
    GP_REQUIRE((size_t)p.plane_stride <= x->cap_words, GP_ERR_INVALID, "exchange: shard larger than the slots");
    p.n = h->num_nodes;
    p.wb = h->wb;
    p.batches = h->batches;
    p.kr = (int)kr;
    p.world = x->world;
    p.rank = x->rank;
    p.parity = parity;
    p.pk_stride = x->pk_stride;
    for (int r = 0; r < x->world; ++r) p.peer[r] = x->peer[r];
    p.local = x->local;
    p.x = d_x;
    p.num_features = d_x ? f : 0;
    p.ld_x = ldx;
    p.out = d_out;
    p.ld_out = ldo;
    p.col_offset = coff;
    // rows per streamed block: as many as fit XCHG_STAGE_CAP bytes of peer segments, a multiple of 8 in [8, 64]
    const int row_bytes = h->wb * 8;
    const int per_row = (x->world > 1 ? x->world - 1 : 1) * GP_PACKED_ARRAYS * h->batches * row_bytes;
    int rb = XCHG_STAGE_CAP / per_row / 8 * 8;
    rb = rb < 8 ? 8 : (rb > 64 ? 64 : rb);
    p.block_rows = rb;
    p.seg_stride = rb * row_bytes;
    p.stage_bytes = x->world > 1 ? (per_row * rb + 127) / 128 * 128 : 0;
    const int smem = XCHG_STAGES * p.stage_bytes;
    if (x->grid_blocks == 0 || x->smem_bytes != smem) {
        int occ = 0;
        GP_CUDA_CHECK(cudaFuncSetAttribute(exchange_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           smem > 48 * 1024 ? smem : 48 * 1024));
        GP_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, exchange_decode_kernel, XCHG_THREADS, smem));
        GP_REQUIRE(occ >= 1, GP_ERR_CUDA, "exchange kernel does not fit on an SM");
        if (occ > 4) occ = 4;
        x->grid_blocks = occ * gp_sm_count();
        x->smem_bytes = smem;
        const int cap = x->grid_cap > 0 ? x->grid_cap : gp_env().xchg_grid;
        if (cap > 0 && cap < x->grid_blocks) x->grid_blocks = cap;
    }
    p.debug = gp_env().xchg_debug;
    p.vec_x = d_x != nullptr && (reinterpret_cast<uintptr_t>(d_x) & 15u) == 0 && ldx % 4 == 0;
    if (p.n == 0) return GP_OK;
    void *args[] = {&p};
    gp_count_launch();
    GP_CUDA_CHECK(cudaLaunchCooperativeKernel((const void *)exchange_decode_kernel, dim3(x->grid_blocks),
                                              dim3(XCHG_THREADS), args, (size_t)smem, stream));
    return GP_OK;
}

// async, COLLECTIVE.  The fused kernel alone, for callers that ran gp_csr_build / gp_msbfs_run themselves.
extern "C" int gp_exchange_run(gp_exchange_t *x, const float *d_x, int64_t num_features, int64_t ld_x, float *d_out,
                               int64_t ld_out, int64_t col_offset, gp_stream_t stream)
{
    GP_REQUIRE(x != nullptr, GP_ERR_INVALID, "gp_exchange_run: NULL argument");
    return gp_exchange_launch(x, gp_exchange_next_parity(x), d_x, num_features, ld_x, d_out, ld_out, col_offset,
                              (cudaStream_t)stream);
}
