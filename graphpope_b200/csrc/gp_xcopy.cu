// gp_xcopy.cu — concat_into_features' copy of x (reference utils.py:133-134: torch.cat((data.x, emb), 1)) as a
// TMA bulk-copy pipeline: the stand-alone form of the copy (gp_concat_x).
//
// ONE thread per SM keeps XC_STAGES x 16 KB in flight through shared memory (cp.async.bulk global -> shared,
// completion on an mbarrier; cp.async.bulk shared -> global, completion by bulk group): 32 threads, a handful of
// uniform registers and 64 KB of shared memory per SM, so the kernel can stay resident next to two MS-BFS CTAs.
// Both directions carry an L2 evict-first policy.  Alone it moves the Flickr-size rows (357 MB) in 72 us = 4.9 TB/s
// (a strided cudaMemcpy2DAsync: 0.6 TB/s; torch's strided copy_: 2.9 TB/s).  Run BESIDE the csr build / the MS-BFS
// it does not shorten the step: those stages are bound by L2 / HBM latency and slow down by about the copy's
// duration while the rows stream through the memory system (profiles/r02_notes.md), so gp_geodesic_run keeps the
// copy fused in its epilogue kernel.
#include "gp_msbfs.cuh"
#include "gp_tma.cuh"

namespace {

constexpr int XC_STAGE_BYTES = 16384;
constexpr int XC_STAGES = 4;  // alone: 4.98 TB/s; 3 stages 4.35, 6 or 8 stages 4.84 (profiles/r02_notes.md)

// One CTA per SM, one thread drives the pipeline.  Row blocks of R rows are dealt round-robin to the CTAs; block
// i of a CTA lives in stage i % S (S = XC_STAGES).  Loads run S - 2 blocks ahead of the stores: before stage s is
// refilled the store group that read it two iterations ago must have finished READING shared memory
// (cp.async.bulk.wait_group.read 1), which it has long done by then, so the driver thread never waits on a
// store it has only just issued.
__global__ void __launch_bounds__(32, 1)
xcopy_tma_kernel(const unsigned char *__restrict__ x, long long n, u32 row_bytes, long long ldx_bytes,
                 unsigned char *__restrict__ out, long long ldo_bytes, int rows_per_stage)
{
    extern __shared__ __align__(128) unsigned char s_stage[];
    __shared__ __align__(8) u64 s_full[XC_STAGES];
    if (threadIdx.x != 0) return;
    for (int s = 0; s < XC_STAGES; ++s) gp_mbar_init(gp_smem_addr(&s_full[s]), 1);
    gp_mbar_init_fence();
    u64 policy;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));

    const int R = rows_per_stage;
    const long long nblk = (n + R - 1) / R;
    const long long first = blockIdx.x, step = gridDim.x;
    const long long cnt = nblk > first ? (nblk - first + step - 1) / step : 0;
    const bool contiguous = ldx_bytes == (long long)row_bytes;
    const u32 stage0 = gp_smem_addr(s_stage);

    auto load = [&](long long i) {
        const int s = (int)(i % XC_STAGES);
        const long long r0 = (first + i * step) * R;
        const int rows = (int)(n - r0 < R ? n - r0 : R);
        const u32 bar = gp_smem_addr(&s_full[s]);
        const u32 dst = stage0 + (u32)s * XC_STAGE_BYTES;
        gp_mbar_expect_tx(bar, (u32)rows * row_bytes);
        if (contiguous) {
            gp_bulk_load_hint(dst, x + r0 * ldx_bytes, (u32)rows * row_bytes, bar, policy);
        } else {
            for (int r = 0; r < rows; ++r)
                gp_bulk_load_hint(dst + (u32)r * row_bytes, x + (r0 + r) * ldx_bytes, row_bytes, bar, policy);
        }
    };

    const int ahead = XC_STAGES - 2;
    for (long long i = 0; i < ahead && i < cnt; ++i) load(i);
    for (long long i = 0; i < cnt; ++i) {
        if (i + ahead < cnt) {
            // stage (i + ahead) % S == (i - 2) % S was read by store group i - 2
            asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            load(i + ahead);
        }
        const int s = (int)(i % XC_STAGES);
        gp_mbar_wait(gp_smem_addr(&s_full[s]), (u32)((i / XC_STAGES) & 1));
        const long long r0 = (first + i * step) * R;
        const int rows = (int)(n - r0 < R ? n - r0 : R);
        const u32 src = stage0 + (u32)s * XC_STAGE_BYTES;
        for (int r = 0; r < rows; ++r) gp_bulk_store_hint(out + (r0 + r) * ldo_bytes, src + (u32)r * row_bytes, row_bytes, policy);
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // every row has reached global memory
}

}  // namespace

// True when the bulk-copy engine can take this copy: 16-byte aligned rows on both sides, a row fits a stage.
bool gp_xcopy_tma_ok(const float *d_x, int64_t num_features, int64_t ld_x, const float *d_out, int64_t ld_out)
{
    const int64_t row_bytes = num_features * 4;
    return d_x != nullptr && d_out != nullptr && row_bytes > 0 && row_bytes % 16 == 0 && row_bytes <= XC_STAGE_BYTES &&
           (ld_x * 4) % 16 == 0 && (ld_out * 4) % 16 == 0 && (reinterpret_cast<uintptr_t>(d_x) & 15u) == 0 &&
           (reinterpret_cast<uintptr_t>(d_out) & 15u) == 0;
}

int gp_launch_xcopy_tma(const float *d_x, int64_t num_nodes, int64_t num_features, int64_t ld_x, float *d_out,
                        int64_t ld_out, cudaStream_t stream)
{
    if (num_nodes == 0 || num_features == 0) return GP_OK;
    GP_REQUIRE(gp_xcopy_tma_ok(d_x, num_features, ld_x, d_out, ld_out), GP_ERR_INVALID,
               "gp_launch_xcopy_tma: rows must be 16-byte aligned and at most %d bytes long", XC_STAGE_BYTES);
    GP_CUDA_CHECK(cudaFuncSetAttribute(xcopy_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       XC_STAGES * XC_STAGE_BYTES));
    const u32 row_bytes = (u32)(num_features * 4);
    const int rows_per_stage = XC_STAGE_BYTES / (int)row_bytes;
    const long long nblk = (num_nodes + rows_per_stage - 1) / rows_per_stage;
    const int grid = (int)(nblk < gp_sm_count() ? nblk : gp_sm_count());  // one block per SM
    GP_LAUNCH(xcopy_tma_kernel, grid, 32, (size_t)XC_STAGES * XC_STAGE_BYTES, stream,
              reinterpret_cast<const unsigned char *>(d_x), (long long)num_nodes, row_bytes, (long long)ld_x * 4,
              reinterpret_cast<unsigned char *>(d_out), (long long)ld_out * 4, rows_per_stage);
    GP_CUDA_CHECK(cudaGetLastError());
    return GP_OK;
}
