// gp_epilogue.cu — fused normalise / unreachable-fill / concat epilogue and the uint16 decode.
//
// Reproduces the reference value convention (utils.py:72-76): value = 1/len(path) = 1/(d+1),
// anchor itself = 1.0, no path = 0; float32 output (utils.py:125) — computed here as IEEE
// fp32 1.0f/(float)(d+1), which is bit-identical to the reference's float64 divide followed
// by the float32 rounding of torch.as_tensor for every d+1 in [1, 65536].  Also performs
// concat_into_features (utils.py:129-135) by streaming x into columns [0, F) of the same
// output rows, so each [N, F+K] row is written once, contiguously.
//
// Input is the result block R of gp_msbfs.cu (R[0] = reached mask, R[l] = lanes first reached at
// hop l for l <= 15, R[16+q] = bit q of deeper hop counts); HBM-bound: reads (1+L)*N*K/8 bytes of
// masks (+4NF of x), writes 4*N*(F+K) bytes.
#include "gp_epilogue.cuh"
#include "gp_msbfs.cuh"

namespace {

// How much of R is valid: hop arrays R[1..levels] and, for deep graphs, `deep` bit planes.
struct Valid {
    int levels, deep;
};

__device__ __forceinline__ Valid valid_arrays(const GpDecodeParams &p)
{
    int na = p.num_arrays;
    if (p.packed) na = GP_PACKED_ARRAYS;
    if (na < 0) {
        const int ml = p.status[GP_BFS_ST_MAX_LEVEL];
        na = ml <= GP_BFS_LEVEL_ARRAYS ? 1 + ml : GP_BFS_RESULT_ARRAYS;
    }
    Valid v;
    v.levels = min(na - 1, GP_BFS_LEVEL_ARRAYS);
    v.deep = na > 1 + GP_BFS_LEVEL_ARRAYS ? GP_BFS_PLANES : 0;
    return v;
}

// Word that holds column j (global anchor index) of node u, and the bit inside it.
__device__ __forceinline__ const u64 *lane_word(const GpDecodeParams &p, long long u, long long j, int &bit)
{
    const u32 kr = (u32)p.anchors_per_rank, jj = (u32)j;  // anchor counts fit 32 bits
    const u32 r = jj / kr, jl = jj - r * kr;
    const u32 wsh = p.wb == 4 ? 2 : (p.wb == 2 ? 1 : 0);
    const u32 b = jl >> (6 + wsh);
    const u32 w = (jl >> 6) & ((1u << wsh) - 1u);
    bit = (int)(jl & 63u);
    return p.planes0 + (size_t)r * p.rank_stride + ((size_t)b * p.n + (size_t)u) * p.wb + w;
}

// Hop count of one reached lane.
__device__ __forceinline__ u32 hops_one(const GpDecodeParams &p, Valid va, const u64 *w, int bit)
{
    u32 d = 0;
    for (int l = 1; l <= va.levels; ++l)
        if ((w[(size_t)l * p.plane_stride] >> bit) & 1ull) d = (u32)l;
    if (va.deep) {
        u32 dd = 0;
        const u64 *pl = w + (size_t)(1 + GP_BFS_LEVEL_ARRAYS) * p.plane_stride;
        for (int q = 0; q < va.deep; ++q) dd |= (u32)((pl[(size_t)q * p.plane_stride] >> bit) & 1ull) << q;
        if (dd) d = dd;  // lanes first reached at hop >= 16 carry their whole hop count in the planes
    }
    return d;
}

__device__ __forceinline__ float decode_one(const GpDecodeParams &p, Valid va, long long u, long long j)
{
    int bit;
    const u64 *w = lane_word(p, u, j, bit);
    if (!((w[0] >> bit) & 1ull)) return 0.0f;
    return inv_hops(hops_one(p, va, w, bit));
}

// One warp per output row.
__global__ void __launch_bounds__(256) decode_features_kernel(GpDecodeParams p, long long k_total, int vec_x,
                                                              int vec_f)
{
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const Valid va = valid_arrays(p);
    for (long long u = warp; u < p.n; u += nwarps) {
        float *orow = p.out + (size_t)u * p.ld_out;
        if (p.x != nullptr) copy_x_row(p.x + (size_t)u * p.ld_x, orow, (int)p.num_features, lane, vec_x);
        float *frow = orow + p.col_offset;
        if (vec_f) {
            // groups of 4 columns never straddle a lane word or a rank (anchors_per_rank % 4 == 0)
            const long long groups = k_total >> 2;
            for (long long g = lane; g < groups; g += 32) {
                const long long j0 = g << 2;
                int bit;
                const u64 *w = lane_word(p, u, j0, bit);
                const u32 reach = (u32)(w[0] >> bit) & 0xFu;
                u32 d0 = 0, d1 = 0, d2 = 0, d3 = 0;
                if (reach) {
                    for (int l = 1; l <= va.levels; ++l) {
                        const u32 nib = (u32)(w[(size_t)l * p.plane_stride] >> bit) & 0xFu;
                        if (nib) {
                            if (nib & 1u) d0 = l;
                            if (nib & 2u) d1 = l;
                            if (nib & 4u) d2 = l;
                            if (nib & 8u) d3 = l;
                        }
                    }
                    if (va.deep) {
                        const u64 *pl = w + (size_t)(1 + GP_BFS_LEVEL_ARRAYS) * p.plane_stride;
                        u32 e0 = 0, e1 = 0, e2 = 0, e3 = 0;
                        for (int q = 0; q < va.deep; ++q) {
                            const u32 nib = (u32)(pl[(size_t)q * p.plane_stride] >> bit) & 0xFu;
                            e0 |= (nib & 1u) << q;
                            e1 |= ((nib >> 1) & 1u) << q;
                            e2 |= ((nib >> 2) & 1u) << q;
                            e3 |= ((nib >> 3) & 1u) << q;
                        }
                        if (e0) d0 = e0;
                        if (e1) d1 = e1;
                        if (e2) d2 = e2;
                        if (e3) d3 = e3;
                    }
                }
                float4 v;
                v.x = (reach & 1u) ? inv_hops(d0) : 0.0f;
                v.y = (reach & 2u) ? inv_hops(d1) : 0.0f;
                v.z = (reach & 4u) ? inv_hops(d2) : 0.0f;
                v.w = (reach & 8u) ? inv_hops(d3) : 0.0f;
                reinterpret_cast<float4 *>(frow)[g] = v;
            }
            for (long long j = (groups << 2) + lane; j < k_total; j += 32) frow[j] = decode_one(p, va, u, j);
        } else {
            for (long long j = lane; j < k_total; j += 32) frow[j] = decode_one(p, va, u, j);
        }
    }
}

// Fast path (anchors_per_rank % 8 == 0, 16-byte aligned rows): one warp per output row; a lane owns
// 8 consecutive anchor columns = ONE BYTE of every mask array, so the 32 lanes read one 32-byte row
// sector per array with a single coalesced byte load, bit-slice the hop index of their 8 columns and
// store two float4.  x is streamed into columns [0, F) by the same warp.
__global__ void __launch_bounds__(256, 4) decode_features_bytes_kernel(GpDecodeParams p, int vec_x)
{
    __shared__ float s_inv[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_inv[i] = inv_hops((u32)i);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const Valid va = valid_arrays(p);
    const int row_bytes = p.wb * 8;                       // bytes of one node row in one batch
    const int kr = (int)p.anchors_per_rank;
    const int batches = (kr + 64 * p.wb - 1) / (64 * p.wb);
    const size_t plane_bytes = (size_t)p.plane_stride * 8;
    for (long long u = warp; u < p.n; u += nwarps) {
        float *orow = p.out + (size_t)u * p.ld_out;
        if (p.x != nullptr) copy_x_row(p.x + (size_t)u * p.ld_x, orow, (int)p.num_features, lane, vec_x);
        for (int r = 0; r < p.num_ranks; ++r) {
            const unsigned char *blk = reinterpret_cast<const unsigned char *>(p.planes0 + (size_t)r * p.rank_stride);
            for (int b = 0; b < batches; ++b) {
                const int col0 = b * 64 * p.wb + lane * 8;  // first of this lane's 8 columns inside the rank
                if (lane >= row_bytes || col0 >= kr) continue;
                const unsigned char *rowp = blk + ((size_t)b * p.n + (size_t)u) * row_bytes + lane;
                const u32 reach = rowp[0];
                u32 m0 = 0, m1 = 0, m2 = 0, m3 = 0;
                if (reach) {
#pragma unroll
                    for (int l = 1; l <= GP_BFS_LEVEL_ARRAYS; ++l) {
                        if (l <= va.levels) {
                            const u32 bl = rowp[(size_t)l * plane_bytes];
                            if (l & 1) m0 |= bl;
                            if (l & 2) m1 |= bl;
                            if (l & 4) m2 |= bl;
                            if (l & 8) m3 |= bl;
                        }
                    }
                }
                float v[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const u32 d = ((m0 >> c) & 1u) | (((m1 >> c) & 1u) << 1) | (((m2 >> c) & 1u) << 2) |
                                  (((m3 >> c) & 1u) << 3);
                    v[c] = ((reach >> c) & 1u) ? s_inv[d] : 0.0f;
                }
                if (va.deep && reach) {
                    const unsigned char *pl = rowp + (size_t)(1 + GP_BFS_LEVEL_ARRAYS) * plane_bytes;
                    u32 e[GP_BFS_PLANES];
#pragma unroll
                    for (int q = 0; q < GP_BFS_PLANES; ++q) e[q] = pl[(size_t)q * plane_bytes];
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        u32 dd = 0;
#pragma unroll
                        for (int q = 0; q < GP_BFS_PLANES; ++q) dd |= ((e[q] >> c) & 1u) << q;
                        if (dd) v[c] = dd < 256 ? s_inv[dd] : inv_hops(dd);
                    }
                }
                float4 *dst = reinterpret_cast<float4 *>(orow + p.col_offset + (size_t)r * kr + col0);
                __stcs(dst, make_float4(v[0], v[1], v[2], v[3]));
                __stcs(dst + 1, make_float4(v[4], v[5], v[6], v[7]));
            }
        }
    }
}

// Peer assembly (packed exchange format, gp_decode_peers): same row / lane mapping as the kernel above,
// but the five bytes of EVERY rank's shard are requested up front, so the NVLink round trips of all
// peers overlap (one dependent round trip per row instead of two per peer).  Per row a warp is bound by
// that round trip (~3 us over NVLink), so what matters is rows in flight: the kernel is instantiated for
// 2, 4 and 8 ranks (the mask registers of absent ranks cost occupancy: 114 registers and 2 CTAs per SM
// for everyone made the 2-GPU epilogue run at half the HBM rate), and the first 2 KB of the x row are
// requested together with the masks instead of after the columns have been stored.
template <int R>
__global__ void __launch_bounds__(256, R <= 2 ? 3 : 2)
decode_features_peers_kernel(GpDecodeParams p, int vec_x)
{
    __shared__ float s_inv[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_inv[i] = inv_hops((u32)i);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const int row_bytes = p.wb * 8;
    const int kr = (int)p.anchors_per_rank;
    const int batches = (kr + 64 * p.wb - 1) / (64 * p.wb);
    const size_t plane_bytes = (size_t)p.plane_stride * 8;
    const int f = (int)p.num_features, q = f >> 2;
    const bool fast_x = p.x != nullptr && vec_x;
    for (long long u = warp; u < p.n; u += nwarps) {
        float *orow = p.out + (size_t)u * p.ld_out;
        const float *xrow = p.x != nullptr ? p.x + (size_t)u * p.ld_x : nullptr;
        float4 xv[4];
        if (fast_x) {
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int i = lane + 32 * t;
                if (i < q) xv[t] = __ldcs(reinterpret_cast<const float4 *>(xrow) + i);
            }
        }
        for (int b = 0; b < batches; ++b) {
            const int col0 = b * 64 * p.wb + lane * 8;  // first of this lane's 8 columns inside the rank
            const bool act = lane < row_bytes && col0 < kr;
            const size_t roff = ((size_t)b * p.n + (size_t)u) * row_bytes + lane;
            u32 m[R][GP_PACKED_ARRAYS];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                if (act && r < p.num_ranks) {
                    const unsigned char *rowp = reinterpret_cast<const unsigned char *>(p.rank_ptr[r]) + roff;
#pragma unroll
                    for (int a = 0; a < GP_PACKED_ARRAYS; ++a) m[r][a] = rowp[(size_t)a * plane_bytes];
                }
            }
            if (b == 0 && fast_x) {  // the x row goes out while the peer bytes are still in flight
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const int i = lane + 32 * t;
                    if (i < q) __stcs(reinterpret_cast<float4 *>(orow) + i, xv[t]);
                }
            }
            if (!act) continue;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                if (r < p.num_ranks) {
                    const u32 reach = m[r][0];
                    float v[8];
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const u32 d = ((m[r][1] >> c) & 1u) | (((m[r][2] >> c) & 1u) << 1) | (((m[r][3] >> c) & 1u) << 2) |
                                      (((m[r][4] >> c) & 1u) << 3);
                        v[c] = ((reach >> c) & 1u) ? s_inv[d] : 0.0f;
                    }
                    float4 *dst = reinterpret_cast<float4 *>(orow + p.col_offset + (size_t)r * kr + col0);
                    __stcs(dst, make_float4(v[0], v[1], v[2], v[3]));
                    __stcs(dst + 1, make_float4(v[4], v[5], v[6], v[7]));
                }
            }
        }
        // the rest of x: rows longer than 128 float4, the scalar tail, or unaligned rows
        if (fast_x) {
            if (q > 128) copy_x_row(xrow + 512, orow + 512, f - 512, lane, 1);
            else
                for (int i = (q << 2) + lane; i < f; i += 32) orow[i] = __ldcs(xrow + i);
        } else if (xrow != nullptr) {
            copy_x_row(xrow, orow, f, lane, 0);
        }
    }
}

__global__ void __launch_bounds__(256) decode_u16_kernel(GpDecodeParams p, long long k_total, uint16_t *dist,
                                                         long long ld, long long col_offset)
{
    const Valid va = valid_arrays(p);
    const long long total = p.n * k_total;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const long long u = i / k_total, j = i - u * k_total;
        int bit;
        const u64 *w = lane_word(p, u, j, bit);
        u32 d = GP_UNREACHABLE_U16;
        if ((w[0] >> bit) & 1ull) d = hops_one(p, va, w, bit);
        dist[(size_t)u * ld + col_offset + j] = (uint16_t)d;
    }
}

__global__ void __launch_bounds__(256) normalize_u16_kernel(const uint16_t *__restrict__ dist, long long n,
                                                            long long k, long long ld_dist,
                                                            float *__restrict__ out, long long ld_out,
                                                            long long col_offset)
{
    const long long total = n * k;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const long long u = i / k, j = i - u * k;
        const u32 d = dist[(size_t)u * ld_dist + j];
        out[(size_t)u * ld_out + col_offset + j] = d == GP_UNREACHABLE_U16 ? 0.0f : inv_hops(d);
    }
}

// Exchange format for the multi-GPU assembly: P[0] = reached mask, P[1 + q] = bit q of the hop count
// (hops <= 15).  Five arrays whatever the depth, so ranks need not agree on a size before exchanging.
__global__ void __launch_bounds__(256) pack_result_kernel(const u64 *__restrict__ result, long long stride,
                                                          const int *__restrict__ status, u64 *__restrict__ packed,
                                                          int *deep_flag)
{
    const int ml = status[GP_BFS_ST_MAX_LEVEL];
    if (blockIdx.x == 0 && threadIdx.x == 0) *deep_flag = ml > GP_BFS_LEVEL_ARRAYS ? 1 : 0;
    const int levels = min(ml, GP_BFS_LEVEL_ARRAYS);
    const long long step = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < stride; i += step) {
        u64 m0 = 0, m1 = 0, m2 = 0, m3 = 0;
        for (int l = 1; l <= levels; ++l) {
            const u64 w = result[(size_t)l * stride + i];
            if (l & 1) m0 |= w;
            if (l & 2) m1 |= w;
            if (l & 4) m2 |= w;
            if (l & 8) m3 |= w;
        }
        packed[i] = result[i];
        packed[(size_t)1 * stride + i] = m0;
        packed[(size_t)2 * stride + i] = m1;
        packed[(size_t)3 * stride + i] = m2;
        packed[(size_t)4 * stride + i] = m3;
    }
}

int grid_for(long long work_items, int per_block)
{
    long long b = gp_ceil_div(work_items > 0 ? work_items : 1, per_block);
    const long long cap = (long long)gp_sm_count() * 8;
    return (int)(b < cap ? b : cap);
}

bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

int gp_launch_decode_features(const GpDecodeParams &p, cudaStream_t stream)
{
    const long long k_total = p.anchors_per_rank * p.num_ranks;
    if (p.n == 0 || (k_total == 0 && (p.x == nullptr || p.num_features == 0))) return GP_OK;
    const int vec_x = p.x != nullptr && aligned16(p.x) && aligned16(p.out) && (p.ld_x % 4 == 0) &&
                      (p.ld_out % 4 == 0);
    const int vec_f = aligned16(p.out) && (p.ld_out % 4 == 0) && (p.col_offset % 4 == 0) &&
                      (p.anchors_per_rank % 4 == 0 || p.num_ranks == 1);
    if (vec_f && p.anchors_per_rank % 8 == 0 && p.anchors_per_rank > 0 && p.packed)
    {
        if (p.num_ranks <= 2) GP_LAUNCH(decode_features_peers_kernel<2>, grid_for(p.n, 8), 256, 0, stream, p, vec_x);
        else if (p.num_ranks <= 4) GP_LAUNCH(decode_features_peers_kernel<4>, grid_for(p.n, 8), 256, 0, stream, p, vec_x);
        else GP_LAUNCH(decode_features_peers_kernel<8>, grid_for(p.n, 8), 256, 0, stream, p, vec_x);
    }
    else if (vec_f && p.anchors_per_rank % 8 == 0 && p.anchors_per_rank > 0) {
        // one resident wave: 4 CTAs per SM (launch bound), rows dealt round-robin to the warps
        const int wave = gp_sm_count() * 4, want = grid_for(p.n, 8);
        GP_LAUNCH(decode_features_bytes_kernel, want < wave ? want : wave, 256, 0, stream, p, vec_x);
    }
    else
        GP_LAUNCH(decode_features_kernel, grid_for(p.n, 8), 256, 0, stream, p, k_total, vec_x, vec_f);
    GP_CUDA_CHECK(cudaGetLastError());
    return GP_OK;
}

static GpDecodeParams local_params(gp_msbfs *h)
{
    GpDecodeParams p;
    memset(&p, 0, sizeof(p));
    p.planes0 = h->seen;
    p.rank_stride = 0;
    p.plane_stride = (long long)h->wb * h->batches * h->num_nodes;
    p.num_ranks = 1;
    p.num_arrays = -1;
    p.status = h->status;
    p.n = h->num_nodes;
    p.anchors_per_rank = h->num_anchors;
    p.wb = h->wb;
    return p;
}

extern "C" int gp_msbfs_features(gp_msbfs_t *h, const float *d_x, int64_t num_features, int64_t ld_x,
                                 float *d_out, int64_t ld_out, int64_t col_offset, gp_stream_t stream_)
{
    GP_REQUIRE(h != nullptr && d_out != nullptr, GP_ERR_INVALID, "gp_msbfs_features: NULL argument");
    GP_REQUIRE(h->ran, GP_ERR_INVALID, "gp_msbfs_features: gp_msbfs_run has not been called");
    GP_REQUIRE(num_features >= 0 && col_offset >= 0 && ld_out >= col_offset + h->num_anchors &&
                   (d_x == nullptr || (ld_x >= num_features && ld_out >= num_features)),
               GP_ERR_INVALID, "gp_msbfs_features: inconsistent leading dimensions");
    GpDecodeParams p = local_params(h);
    p.x = d_x;
    p.num_features = d_x ? num_features : 0;
    p.ld_x = ld_x;
    p.out = d_out;
    p.ld_out = ld_out;
    p.col_offset = col_offset;
    return gp_launch_decode_features(p, (cudaStream_t)stream_);
}

extern "C" int gp_msbfs_hops_u16(gp_msbfs_t *h, uint16_t *d_dist, int64_t ld, int64_t col_offset,
                                 gp_stream_t stream_)
{
    GP_REQUIRE(h != nullptr && d_dist != nullptr, GP_ERR_INVALID, "gp_msbfs_hops_u16: NULL argument");
    GP_REQUIRE(h->ran, GP_ERR_INVALID, "gp_msbfs_hops_u16: gp_msbfs_run has not been called");
    GP_REQUIRE(col_offset >= 0 && ld >= col_offset + h->num_anchors, GP_ERR_INVALID,
               "gp_msbfs_hops_u16: leading dimension too small");
    if (h->num_nodes == 0 || h->num_anchors == 0) return GP_OK;
    GpDecodeParams p = local_params(h);
    GP_LAUNCH(decode_u16_kernel, grid_for(p.n * h->num_anchors, 256), 256, 0, (cudaStream_t)stream_, p, h->num_anchors, d_dist, ld, col_offset);
    GP_CUDA_CHECK(cudaGetLastError());
    return GP_OK;
}

extern "C" int gp_decode_gathered(const uint64_t *d_gathered, int64_t rank_stride_words, int32_t num_ranks,
                                  int64_t num_nodes, int64_t anchors_per_rank, int32_t num_planes,
                                  int32_t batches, int32_t words_per_batch, int64_t plane_stride_words,
                                  const float *d_x, int64_t num_features, int64_t ld_x, float *d_out,
                                  int64_t ld_out, int64_t col_offset, gp_stream_t stream_)
{
    GP_REQUIRE(d_gathered != nullptr && d_out != nullptr, GP_ERR_INVALID, "gp_decode_gathered: NULL argument");
    GP_REQUIRE(num_ranks >= 1 && num_nodes >= 0 && anchors_per_rank >= 0 && batches >= 1 &&
                   (words_per_batch == 1 || words_per_batch == 2 || words_per_batch == 4),
               GP_ERR_INVALID, "gp_decode_gathered: bad shape arguments");
    // what gp_msbfs_planes reports: 1 + max_level <= 16 planes, or all 32 once a hop exceeds 15 (the decoder then
    // reads the 16 deep-hop planes whole, so 17..31 would read past the shard)
    GP_REQUIRE((num_planes >= 1 && num_planes <= 1 + GP_BFS_LEVEL_ARRAYS) || num_planes == GP_BFS_RESULT_ARRAYS,
               GP_ERR_INVALID, "gp_decode_gathered: num_planes %d is not 1..%d or %d", num_planes,
               1 + GP_BFS_LEVEL_ARRAYS, GP_BFS_RESULT_ARRAYS);
    GP_REQUIRE(anchors_per_rank <= (int64_t)batches * words_per_batch * 64, GP_ERR_INVALID,
               "gp_decode_gathered: anchors_per_rank exceeds the lane capacity of a shard");
    GP_REQUIRE(plane_stride_words >= (int64_t)batches * words_per_batch * num_nodes &&
                   (num_ranks == 1 || rank_stride_words >= (int64_t)num_planes * plane_stride_words),
               GP_ERR_INVALID, "gp_decode_gathered: plane or rank stride smaller than a plane or a shard");
    GP_REQUIRE(num_features >= 0 && col_offset >= 0 && ld_out >= col_offset + anchors_per_rank * num_ranks &&
                   (d_x == nullptr || (ld_x >= num_features && ld_out >= num_features)),
               GP_ERR_INVALID, "gp_decode_gathered: inconsistent leading dimensions");
    GpDecodeParams p;
    memset(&p, 0, sizeof(p));
    p.planes0 = (const u64 *)d_gathered;
    p.rank_stride = rank_stride_words;
    p.plane_stride = plane_stride_words;
    p.num_ranks = num_ranks;
    p.num_arrays = num_planes;
    p.status = nullptr;
    p.n = num_nodes;
    p.anchors_per_rank = anchors_per_rank;
    p.wb = words_per_batch;
    p.x = d_x;
    p.num_features = d_x ? num_features : 0;
    p.ld_x = ld_x;
    p.out = d_out;
    p.ld_out = ld_out;
    p.col_offset = col_offset;
    return gp_launch_decode_features(p, (cudaStream_t)stream_);
}

extern "C" int gp_normalize_into(const uint16_t *d_dist, int64_t num_nodes, int64_t num_anchors,
                                 int64_t ld_dist, float *d_out, int64_t ld_out, int64_t col_offset,
                                 gp_stream_t stream_)
{
    GP_REQUIRE(d_dist != nullptr && d_out != nullptr, GP_ERR_INVALID, "gp_normalize_into: NULL argument");
    GP_REQUIRE(num_nodes >= 0 && num_anchors >= 0 && ld_dist >= num_anchors && col_offset >= 0 &&
                   ld_out >= col_offset + num_anchors,
               GP_ERR_INVALID, "gp_normalize_into: inconsistent sizes");
    if (num_nodes == 0 || num_anchors == 0) return GP_OK;
    GP_LAUNCH(normalize_u16_kernel, grid_for(num_nodes * num_anchors, 256), 256, 0, (cudaStream_t)stream_, d_dist, num_nodes, num_anchors, ld_dist, d_out, ld_out, col_offset);
    GP_CUDA_CHECK(cudaGetLastError());
    return GP_OK;
}

// ------------------------------------------------------------------ peer-to-peer assembly
extern "C" int gp_msbfs_pack(gp_msbfs_t *h, int32_t slot, const uint64_t **d_packed, int64_t *plane_stride_words,
                             int32_t *batches, int32_t *words_per_batch, const int32_t **d_deep_flag,
                             gp_stream_t stream_)
{
    GP_REQUIRE(h != nullptr && (slot == 0 || slot == 1), GP_ERR_INVALID, "gp_msbfs_pack: bad argument");
    GP_REQUIRE(h->ran, GP_ERR_INVALID, "gp_msbfs_pack: gp_msbfs_run has not been called");
    const size_t cap_words = (size_t)h->cap_words_per_node * (size_t)(h->num_nodes > 0 ? h->num_nodes : 1);
    if (h->packed == nullptr) {
        GP_CUDA_CHECK(cudaMalloc((void **)&h->packed, 2 * GP_PACKED_ARRAYS * cap_words * sizeof(u64)));
        GP_CUDA_CHECK(cudaMalloc((void **)&h->deep_flag, sizeof(int)));
    }
    const long long stride = (long long)h->wb * h->batches * h->num_nodes;
    u64 *dst = h->packed + (size_t)slot * GP_PACKED_ARRAYS * cap_words;
    if (stride > 0 && h->num_anchors > 0)
        GP_LAUNCH(pack_result_kernel, grid_for(stride, 256), 256, 0, (cudaStream_t)stream_, h->seen, stride, h->status,
                  dst, h->deep_flag);
    GP_CUDA_CHECK(cudaGetLastError());
    if (d_packed) *d_packed = (const uint64_t *)dst;
    if (plane_stride_words) *plane_stride_words = stride;
    if (batches) *batches = h->batches;
    if (words_per_batch) *words_per_batch = h->wb;
    if (d_deep_flag) *d_deep_flag = h->deep_flag;
    return GP_OK;
}

extern "C" int gp_msbfs_packed_info(gp_msbfs_t *h, int32_t slot, const uint64_t **d_packed, int64_t *plane_stride_words,
                                    int32_t *batches, int32_t *words_per_batch, const int32_t **d_deep_flag)
{
    GP_REQUIRE(h != nullptr && (slot == 0 || slot == 1), GP_ERR_INVALID, "gp_msbfs_packed_info: bad argument");
    GP_REQUIRE(h->packed != nullptr, GP_ERR_INVALID, "gp_msbfs_packed_info: nothing has been packed yet");
    const size_t cap_words = (size_t)h->cap_words_per_node * (size_t)(h->num_nodes > 0 ? h->num_nodes : 1);
    if (d_packed) *d_packed = (const uint64_t *)(h->packed + (size_t)slot * GP_PACKED_ARRAYS * cap_words);
    if (plane_stride_words) *plane_stride_words = (int64_t)h->wb * h->batches * h->num_nodes;
    if (batches) *batches = h->batches;
    if (words_per_batch) *words_per_batch = h->wb;
    if (d_deep_flag) *d_deep_flag = h->deep_flag;
    return GP_OK;
}

extern "C" int gp_msbfs_ipc_export(gp_msbfs_t *h, uint8_t *handle64, int64_t *slot_stride_words)
{
    GP_REQUIRE(h != nullptr && handle64 != nullptr && slot_stride_words != nullptr, GP_ERR_INVALID,
               "gp_msbfs_ipc_export: NULL argument");
    const size_t cap_words = (size_t)h->cap_words_per_node * (size_t)(h->num_nodes > 0 ? h->num_nodes : 1);
    if (h->packed == nullptr) {
        GP_CUDA_CHECK(cudaMalloc((void **)&h->packed, 2 * GP_PACKED_ARRAYS * cap_words * sizeof(u64)));
        GP_CUDA_CHECK(cudaMalloc((void **)&h->deep_flag, sizeof(int)));
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t hd;
    GP_CUDA_CHECK(cudaIpcGetMemHandle(&hd, h->packed));
    memcpy(handle64, &hd, 64);
    *slot_stride_words = (int64_t)(GP_PACKED_ARRAYS * cap_words);
    return GP_OK;
}

extern "C" int gp_ipc_open(const uint8_t *handle64, void **d_ptr)
{
    GP_REQUIRE(handle64 != nullptr && d_ptr != nullptr, GP_ERR_INVALID, "gp_ipc_open: NULL argument");
    cudaIpcMemHandle_t hd;
    memcpy(&hd, handle64, 64);
    GP_CUDA_CHECK(cudaIpcOpenMemHandle(d_ptr, hd, cudaIpcMemLazyEnablePeerAccess));
    return GP_OK;
}

extern "C" int gp_ipc_close(void *d_ptr)
{
    if (d_ptr) GP_CUDA_CHECK(cudaIpcCloseMemHandle(d_ptr));
    return GP_OK;
}

extern "C" int gp_decode_peers(const uint64_t *const *h_rank_ptrs, int32_t num_ranks, int64_t num_nodes,
                               int64_t anchors_per_rank, int32_t batches, int32_t words_per_batch,
                               int64_t plane_stride_words, const float *d_x, int64_t num_features, int64_t ld_x,
                               float *d_out, int64_t ld_out, int64_t col_offset, gp_stream_t stream_)
{
    GP_REQUIRE(h_rank_ptrs != nullptr && d_out != nullptr, GP_ERR_INVALID, "gp_decode_peers: NULL argument");
    GP_REQUIRE(num_ranks >= 1 && num_ranks <= GP_MAX_RANKS, GP_ERR_UNSUPPORTED, "gp_decode_peers: 1..%d ranks",
               GP_MAX_RANKS);
    GP_REQUIRE(num_nodes >= 0 && anchors_per_rank > 0 && anchors_per_rank % 8 == 0 && batches >= 1 &&
                   (words_per_batch == 1 || words_per_batch == 2 || words_per_batch == 4),
               GP_ERR_INVALID, "gp_decode_peers: bad shape (anchors per rank must be a multiple of 8)");
    GP_REQUIRE(ld_out >= col_offset + anchors_per_rank * num_ranks && ld_out % 4 == 0 && col_offset % 4 == 0 &&
                   (reinterpret_cast<uintptr_t>(d_out) & 15u) == 0,
               GP_ERR_INVALID, "gp_decode_peers: output must be 16-byte aligned with ld_out, col_offset multiples of 4");
    GpDecodeParams p;
    memset(&p, 0, sizeof(p));
    p.packed = 1;
    for (int r = 0; r < num_ranks; ++r) {
        GP_REQUIRE(h_rank_ptrs[r] != nullptr, GP_ERR_INVALID, "gp_decode_peers: NULL rank pointer");
        p.rank_ptr[r] = (const u64 *)h_rank_ptrs[r];
    }
    p.plane_stride = plane_stride_words;
    p.num_ranks = num_ranks;
    p.num_arrays = GP_PACKED_ARRAYS;
    p.n = num_nodes;
    p.anchors_per_rank = anchors_per_rank;
    p.wb = words_per_batch;
    p.x = d_x;
    p.num_features = d_x ? num_features : 0;
    p.ld_x = ld_x;
    p.out = d_out;
    p.ld_out = ld_out;
    p.col_offset = col_offset;
    (void)batches;
    return gp_launch_decode_features(p, (cudaStream_t)stream_);
}
