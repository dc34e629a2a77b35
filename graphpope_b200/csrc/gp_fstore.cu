// gp_fstore.cu — compact anchor-distance feature store: packs the MS-BFS result into it, and gathers mini-batch rows
// of concat_into_features(x, features) (utils.py:129-135) from it, as main.py:120,177 index them (x[n_id]).
//
// Format, one contiguous record per node: uint64 [N][P][W], W = ceil(K/64).  Plane 0 is the reached mask, plane
// 1 + q holds bit q of the hop count; column j is word j >> 6, bit j & 63 of a plane (on the little-endian device
// also byte j >> 3, bit j & 7).  P = 1 + bit_length(max hop) (1..17), so a column costs P bits instead of the 32 of
// the dense [N, F+K] float32 matrix.  Padding bits past K and hop bits of unreached lanes are zero.  The value of
// column j is inv_hops(d) = 1/(d+1) in IEEE fp32 if reached, else 0.0f — the dense epilogue's convention, so a
// gathered row is bit-equal to the same row of gp_msbfs_features.
#include "gp_epilogue.cuh"
#include "gp_msbfs.cuh"

namespace {

constexpr int FS_MAX_PLANES = 1 + GP_BFS_PLANES;  // 17: hops up to 65534

// One thread per (node, lane word).  Hop bits 0..3 are ORs of the level arrays R[1..levels], as in
// the exchange's pack (gp_exchange.cu); lanes first reached at hop >= 16 carry their whole hop count in the deep planes R[16 + q] and
// have zeros in R[1..15], so the two sources are disjoint.
__global__ void __launch_bounds__(256) fstore_pack_kernel(const u64 *__restrict__ result, long long plane_stride,
                                                          long long n, int wb, int words, int levels, int deep,
                                                          int num_planes, u64 *__restrict__ store)
{
    const long long total = n * words;
    const long long step = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += step) {
        const long long u = i / words;
        const int j = (int)(i - u * words);
        const int b = j / wb, w = j - b * wb;
        const size_t src = ((size_t)b * n + (size_t)u) * wb + w;
        u64 m0 = 0, m1 = 0, m2 = 0, m3 = 0;
        for (int l = 1; l <= levels; ++l) {
            const u64 v = result[(size_t)l * plane_stride + src];
            if (l & 1) m0 |= v;
            if (l & 2) m1 |= v;
            if (l & 4) m2 |= v;
            if (l & 8) m3 |= v;
        }
        u64 *dst = store + (size_t)u * num_planes * words + j;
        dst[0] = result[src];
        const u64 *pl = result + (size_t)(1 + GP_BFS_LEVEL_ARRAYS) * plane_stride + src;
#pragma unroll
        for (int q = 0; q < FS_MAX_PLANES - 1; ++q) {
            if (q + 1 < num_planes) {
                u64 v = q == 0 ? m0 : q == 1 ? m1 : q == 2 ? m2 : q == 3 ? m3 : 0ull;
                if (deep) v |= pl[(size_t)q * plane_stride];
                dst[(size_t)(1 + q) * words] = v;
            }
        }
    }
}

// One thread per destination word (record row r = node * P + plane, word w): the shards of `per` columns each that
// overlap columns [64w, 64w + 64) are ORed in, each through at most two of its own words funnel-shifted into place
// and masked to its column range.  Shard and store rows share the [N][P] row order, so the row index carries over.
// When per % 64 == 0 every shift is zero and exactly one shard covers a word: the merge is a word permutation.
__global__ void __launch_bounds__(256) fstore_merge_kernel(const u64 *__restrict__ shards, long long per,
                                                           long long shard_words, long long rows, long long words,
                                                           long long k, u64 *__restrict__ store)
{
    const long long step = (long long)gridDim.x * blockDim.x;
    const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long step_r = step / words, step_w = step - step_r * words;
    long long r = i0 / words, w = i0 - r * words;
    const size_t shard_stride = (size_t)rows * shard_words;
    while (r < rows) {
        const long long c0 = w << 6;
        const long long c1 = c0 + 64 < k ? c0 + 64 : k;
        u64 v = 0;
        for (long long s = c0 / per, s_last = (c1 - 1) / per; s <= s_last; ++s) {
            const long long base = s * per;
            const long long cnt = k - base < per ? k - base : per;  // columns shard s holds
            const long long off = c0 - base;  // shard column of destination bit 0; in (-64, 0) if s starts mid-word
            const long long a = off >> 6;     // floor: -1 when off < 0
            const int sh = (int)(off & 63);
            const int t0 = off < 0 ? (int)-off : 0;
            const int t1 = cnt - off < 64 ? (int)(cnt - off) : 64;
            const long long last = (cnt - 1) >> 6;  // last shard word holding columns of s
            const u64 *src = shards + (size_t)s * shard_stride + (size_t)r * shard_words;
            u64 x = a >= 0 ? __ldg(src + a) >> sh : 0ull;
            if (sh != 0 && a + 1 <= last) x |= __ldg(src + a + 1) << (64 - sh);
            const u64 mask = (t1 == 64 ? ~0ull : (1ull << t1) - 1) & (~0ull << t0);
            v |= x & mask;
        }
        store[(size_t)r * words + w] = v;
        w += step_w;
        r += step_r;
        if (w >= words) {
            w -= words;
            ++r;
        }
    }
}

struct FsGather {
    const u64 *store;
    long long n, k, words;  // nodes, anchors, uint64 words per plane
    int planes;
    const long long *rows;
    long long num_rows;
    const float *x;         // nullptr: F = 0
    long long f, ld_x;
    float *out;
    long long ld_out, col_offset;
    int *bad_rows;          // optional device counter of ids outside [-N, N)
};

// Node of batch row i, with torch's single wrap of negative ids; -1 for an id outside [-N, N).
__device__ __forceinline__ long long fs_node(const FsGather &p, long long i)
{
    long long r = __ldg(p.rows + i);
    if (r < 0) r += p.n;
    return (r >= 0 && r < p.n) ? r : -1;
}

// A bad id gets an all-zero row and is counted; nothing is loaded for it.
__device__ void fs_bad_row(const FsGather &p, float *orow, int lane)
{
    if (lane == 0 && p.bad_rows != nullptr) atomicAdd(p.bad_rows, 1);
    for (long long c = lane; c < p.f; c += 32) orow[c] = 0.0f;
    for (long long c = lane; c < p.k; c += 32) orow[p.col_offset + c] = 0.0f;
}

// Bit c of a byte to bit 4c of a word.
__device__ __forceinline__ u32 spread_nibbles(u32 b)
{
    b = (b | (b << 12)) & 0x000F000Fu;
    b = (b | (b << 6)) & 0x03030303u;
    return (b | (b << 3)) & 0x11111111u;
}

// Fast path (K % 8 == 0, 16-byte aligned output rows and anchor block): one warp per output row, the mapping of
// decode_features_bytes_kernel.  A lane owns 8 consecutive columns = ONE BYTE of every plane, so the 32 lanes read
// 32 contiguous bytes of each plane per 256 columns and store 1 KB contiguously.  The reach and hop-bit 0..3 bytes
// of the first 256 columns and the x row are requested before any store.  The hop count of the lane's 8 columns is
// assembled four bits at a time: each plane byte is spread to one bit per nibble, four planes make one nibble per
// column.  (Holding all 17 plane bytes at once spilled at the 64 registers that 4 CTAs per SM allow.)
__global__ void __launch_bounds__(256, 4) fstore_gather_kernel(FsGather p, int vec_x)
{
    __shared__ float s_inv[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_inv[i] = inv_hops((u32)i);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const size_t plane_bytes = (size_t)p.words * 8;
    const int chunks = (int)((p.k + 255) >> 8);  // 256 columns = 32 bytes of a plane
    const int groups = (p.planes + 2) >> 2;      // nibbles of the hop count: ceil((planes - 1) / 4)
    for (long long i = warp; i < p.num_rows; i += nwarps) {
        float *orow = p.out + (size_t)i * p.ld_out;
        const long long u = fs_node(p, i);
        if (u < 0) {
            fs_bad_row(p, orow, lane);
            continue;
        }
        const unsigned char *rec =
            reinterpret_cast<const unsigned char *>(p.store + (size_t)u * p.planes * p.words) + lane;
        for (int c = 0; c < chunks; ++c) {
            const bool act = (long long)c * 256 + lane * 8 < p.k;
            const unsigned char *src = rec + (size_t)c * 32;
            // plane byte q of this chunk (0 past the planes of the record)
            auto plane = [&](int q) -> u32 {
                return (act && q < p.planes) ? (u32)__ldg(src + (size_t)q * plane_bytes) : 0u;
            };
            // reach mask and hop bits 0..3: all a store with hops <= 15 has, requested together
            const u32 reach = plane(0);
            u32 e1 = plane(1), e2 = plane(2), e3 = plane(3), e4 = plane(4);
            if (c == 0 && p.x != nullptr) copy_x_row(p.x + (size_t)u * p.ld_x, orow, (int)p.f, lane, vec_x);
            if (!act) continue;
            u32 nib[4];
            nib[0] = spread_nibbles(e1) | (spread_nibbles(e2) << 1) | (spread_nibbles(e3) << 2) |
                     (spread_nibbles(e4) << 3);
#pragma unroll
            for (int g = 1; g < 4; ++g) {
                nib[g] = 0;
                if (g < groups) {  // hops >= 16: the next four bit planes
                    e1 = plane(1 + 4 * g);
                    e2 = plane(2 + 4 * g);
                    e3 = plane(3 + 4 * g);
                    e4 = plane(4 + 4 * g);
                    nib[g] = spread_nibbles(e1) | (spread_nibbles(e2) << 1) | (spread_nibbles(e3) << 2) |
                             (spread_nibbles(e4) << 3);
                }
            }
            float v[8];
#pragma unroll
            for (int cc = 0; cc < 8; ++cc) {
                u32 d = (nib[0] >> (4 * cc)) & 15u;
                if (groups > 1)
                    d |= (((nib[1] >> (4 * cc)) & 15u) << 4) | (((nib[2] >> (4 * cc)) & 15u) << 8) |
                         (((nib[3] >> (4 * cc)) & 15u) << 12);
                v[cc] = ((reach >> cc) & 1u) ? (d < 256 ? s_inv[d] : inv_hops(d)) : 0.0f;
            }
            float4 *dst = reinterpret_cast<float4 *>(orow + p.col_offset + (size_t)c * 256 + lane * 8);
            __stcs(dst, make_float4(v[0], v[1], v[2], v[3]));
            __stcs(dst + 1, make_float4(v[4], v[5], v[6], v[7]));
        }
    }
}

// Any K, any output alignment: one warp per output row, a lane per column.
__global__ void __launch_bounds__(256) fstore_gather_scalar_kernel(FsGather p, int vec_x)
{
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long i = warp; i < p.num_rows; i += nwarps) {
        float *orow = p.out + (size_t)i * p.ld_out;
        const long long u = fs_node(p, i);
        if (u < 0) {
            fs_bad_row(p, orow, lane);
            continue;
        }
        if (p.x != nullptr) copy_x_row(p.x + (size_t)u * p.ld_x, orow, (int)p.f, lane, vec_x);
        const u64 *rec = p.store + (size_t)u * p.planes * p.words;
        for (long long j = lane; j < p.k; j += 32) {
            const long long w = j >> 6;
            const int bit = (int)(j & 63);
            float v = 0.0f;
            if ((__ldg(rec + w) >> bit) & 1ull) {
                u32 d = 0;
                for (int q = 1; q < p.planes; ++q)
                    d |= (u32)((__ldg(rec + (size_t)q * p.words + w) >> bit) & 1ull) << (q - 1);
                v = inv_hops(d);
            }
            __stcs(orow + p.col_offset + j, v);
        }
    }
}

int fs_grid(long long work_items, int per_block)
{
    const long long b = gp_ceil_div(work_items > 0 ? work_items : 1, per_block);
    const long long cap = (long long)gp_sm_count() * 8;
    return (int)(b < cap ? b : cap);
}

bool fs_aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int fs_planes(int max_level)
{
    int bits = 0;
    while (bits < 31 && (max_level >> bits) != 0) ++bits;
    return 1 + bits;
}

}  // namespace

extern "C" int gp_fstore_layout(gp_msbfs_t *h, int32_t *num_planes, int64_t *words_per_plane, gp_stream_t stream)
{
    GP_REQUIRE(h != nullptr && num_planes != nullptr && words_per_plane != nullptr, GP_ERR_INVALID,
               "gp_fstore_layout: NULL argument");
    gp_msbfs_stats_t st;
    GP_TRY(gp_msbfs_stats(h, &st, stream));  // syncs; reports a run that failed
    *num_planes = fs_planes(st.max_level);
    *words_per_plane = (h->num_anchors + 63) / 64;
    return GP_OK;
}

extern "C" int gp_fstore_pack(gp_msbfs_t *h, uint64_t *d_store, int32_t num_planes, gp_stream_t stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    GP_REQUIRE(h != nullptr, GP_ERR_INVALID, "gp_fstore_pack: handle is NULL");
    gp_msbfs_stats_t st;
    GP_TRY(gp_msbfs_stats(h, &st, stream_));
    const int need = fs_planes(st.max_level);
    GP_REQUIRE(num_planes >= need && num_planes <= FS_MAX_PLANES, GP_ERR_INVALID,
               "gp_fstore_pack: num_planes %d outside [%d, %d] (max hop %d)", (int)num_planes, need, FS_MAX_PLANES,
               (int)st.max_level);
    const int64_t words = (h->num_anchors + 63) / 64;
    if (h->num_nodes == 0 || words == 0) return GP_OK;
    GP_REQUIRE(d_store != nullptr, GP_ERR_INVALID, "gp_fstore_pack: store is NULL");
    const long long plane_stride = (long long)h->wb * h->batches * h->num_nodes;
    const int levels = st.max_level < GP_BFS_LEVEL_ARRAYS ? st.max_level : GP_BFS_LEVEL_ARRAYS;
    const int deep = st.max_level > GP_BFS_LEVEL_ARRAYS;
    GP_LAUNCH(fstore_pack_kernel, fs_grid(h->num_nodes * words, 256), 256, 0, stream, h->seen, plane_stride,
              (long long)h->num_nodes, h->wb, (int)words, levels, deep, (int)num_planes, (u64 *)d_store);
    GP_CUDA_CHECK(cudaGetLastError());
    GP_CUDA_CHECK(cudaStreamSynchronize(stream));  // the store must not depend on bfs once this returns
    return GP_OK;
}

extern "C" int gp_fstore_merge(const uint64_t *d_shards, int32_t num_shards, int64_t cols_per_shard,
                               int64_t words_per_shard, int64_t num_nodes, int32_t num_planes, int64_t num_anchors,
                               uint64_t *d_store, gp_stream_t stream_)
{
    GP_REQUIRE(num_shards >= 1 && cols_per_shard >= 0 && num_nodes >= 0 && num_anchors >= 0, GP_ERR_INVALID,
               "gp_fstore_merge: bad shape arguments");
    GP_REQUIRE(num_planes >= 1 && num_planes <= FS_MAX_PLANES, GP_ERR_INVALID,
               "gp_fstore_merge: num_planes %d outside [1, %d]", (int)num_planes, FS_MAX_PLANES);
    GP_REQUIRE(words_per_shard >= (cols_per_shard + 63) / 64, GP_ERR_INVALID,
               "gp_fstore_merge: %lld words per shard plane cannot hold %lld columns", (long long)words_per_shard,
               (long long)cols_per_shard);
    GP_REQUIRE((int64_t)num_shards * cols_per_shard >= num_anchors, GP_ERR_INVALID,
               "gp_fstore_merge: %d shards of %lld columns cannot hold %lld anchors", (int)num_shards,
               (long long)cols_per_shard, (long long)num_anchors);
    const int64_t words = (num_anchors + 63) / 64;
    if (num_nodes == 0 || words == 0) return GP_OK;
    GP_REQUIRE(d_shards != nullptr && d_store != nullptr, GP_ERR_INVALID, "gp_fstore_merge: NULL argument");
    const long long rows = num_nodes * num_planes;
    GP_LAUNCH(fstore_merge_kernel, fs_grid(rows * words, 256), 256, 0, (cudaStream_t)stream_, (const u64 *)d_shards,
              (long long)cols_per_shard, (long long)words_per_shard, rows, (long long)words, (long long)num_anchors,
              (u64 *)d_store);
    GP_CUDA_CHECK(cudaGetLastError());
    return GP_OK;
}

extern "C" int gp_fstore_gather(const uint64_t *d_store, int64_t num_nodes, int64_t num_anchors, int32_t num_planes,
                                const int64_t *d_rows, int64_t num_rows, const float *d_x, int64_t num_features,
                                int64_t ld_x, float *d_out, int64_t ld_out, int64_t col_offset, int32_t *d_bad_rows,
                                gp_stream_t stream_)
{
    GP_REQUIRE(num_nodes >= 0 && num_anchors >= 0 && num_rows >= 0 && num_features >= 0 && col_offset >= 0 &&
                   num_planes >= 1 && num_planes <= FS_MAX_PLANES,
               GP_ERR_INVALID, "gp_fstore_gather: bad shape arguments");
    if (num_rows == 0) return GP_OK;
    GP_REQUIRE(d_rows != nullptr && d_out != nullptr, GP_ERR_INVALID, "gp_fstore_gather: NULL argument");
    GP_REQUIRE(d_store != nullptr || num_nodes == 0 || num_anchors == 0, GP_ERR_INVALID,
               "gp_fstore_gather: store is NULL");
    const int64_t f = d_x != nullptr ? num_features : 0;
    GP_REQUIRE(ld_out >= col_offset + num_anchors && ld_out >= f && (d_x == nullptr || ld_x >= f), GP_ERR_INVALID,
               "gp_fstore_gather: inconsistent leading dimensions");
    FsGather p;
    p.store = (const u64 *)d_store;
    p.n = num_nodes;
    p.k = num_anchors;
    p.words = (num_anchors + 63) / 64;
    p.planes = num_planes;
    p.rows = (const long long *)d_rows;
    p.num_rows = num_rows;
    p.x = f > 0 ? d_x : nullptr;
    p.f = f;
    p.ld_x = ld_x;
    p.out = d_out;
    p.ld_out = ld_out;
    p.col_offset = col_offset;
    p.bad_rows = d_bad_rows;
    const int vec_x = p.x != nullptr && fs_aligned16(p.x) && fs_aligned16(d_out) && ld_x % 4 == 0 && ld_out % 4 == 0;
    const bool fast = num_anchors > 0 && num_anchors % 8 == 0 && fs_aligned16(d_out) && ld_out % 4 == 0 &&
                      col_offset % 4 == 0;
    cudaStream_t stream = (cudaStream_t)stream_;
    if (fast)
        GP_LAUNCH(fstore_gather_kernel, fs_grid(num_rows, 8), 256, 0, stream, p, vec_x);
    else
        GP_LAUNCH(fstore_gather_scalar_kernel, fs_grid(num_rows, 8), 256, 0, stream, p, vec_x);
    GP_CUDA_CHECK(cudaGetLastError());
    return GP_OK;
}
