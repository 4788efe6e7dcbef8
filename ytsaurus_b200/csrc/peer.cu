// peer.cu — in-box shuffle over NVLink peer memory: the slab scatter of the partition step writes every
// destination's rows straight into that GPU's receive buffer (peer-mapped through CUDA IPC), so the
// reference's "Partition job writes tagged blocks -> Sort job fetches them" hand-off
// (yt/yt/ytlib/table_client/schemaless_chunk_writer.cpp:1604-1667, partition_chunk_reader.cpp:82-86) is ONE
// kernel: random 64-byte row reads from local HBM, coalesced row writes over NVLink.  No NCCL call moves rows.
#include <cstring>
#include <vector>

#include "context.cuh"
#include "radix_sort.cuh"
#include "rows.cuh"
#include "peer_kernels.cuh"

using namespace ytgpu;

namespace {

constexpr int kMaxScatterPartitions = 4096;

// out position j (rows grouped by partition, stable) -> partition p with start[p] <= j < start[p+1].
template <int UNROLL>
__global__ void __launch_bounds__(256) scatter_rows_to_peers_kernel(const uint4* __restrict__ in, const SortPlan* plan,
                                                                    const u32* __restrict__ pa, const u32* __restrict__ pb,
                                                                    u64 n, u32 gr, u32 parts, const u64* __restrict__ start,
                                                                    uint4* const* __restrict__ dest) {
    extern __shared__ u64 s_start[];  // [parts + 1]
    uint4** s_dest = reinterpret_cast<uint4**>(s_start + parts + 1);
    for (u32 i = threadIdx.x; i <= parts; i += blockDim.x) s_start[i] = start[i];
    for (u32 i = threadIdx.x; i < parts; i += blockDim.x) s_dest[i] = dest[i];
    __syncthreads();
    const u32 f = plan_final_idx(plan);
    const u32* perm = f == 1 ? pb : pa;
    const u64 total = n * gr;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (u64 q0 = (u64)blockIdx.x * blockDim.x + threadIdx.x; q0 < total; q0 += stride * UNROLL) {
        uint4 v[UNROLL];
        uint4* dst[UNROLL];
#pragma unroll
        for (int k = 0; k < UNROLL; ++k) {
            const u64 q = q0 + (u64)k * stride;
            dst[k] = nullptr;
            if (q < total) {
                const u64 j = q / gr;
                const u32 g = (u32)(q - j * gr);
                const u64 src = f == 2 ? j : (u64)perm[j];
                v[k] = ld_stream_u128(in + src * gr + g);
                u32 lo = 0, cnt = parts;  // last p with start[p] <= j
                while (cnt > 1) {
                    u32 half = cnt >> 1;
                    if (s_start[lo + half] <= j) { lo += half; cnt -= half; } else cnt = half;
                }
                dst[k] = s_dest[lo] + (j - s_start[lo]) * gr + g;
            }
        }
#pragma unroll
        for (int k = 0; k < UNROLL; ++k)
            if (dst[k]) *dst[k] = v[k];
    }
}

Status scatter_stream(Context* ctx, const ytgpu_fixed_rows_view* in, const i32* index, u32 parts, const std::vector<u64>& start,
                      void* const* dest_base) {
    const u64 n = in->row_count;
    const u32 gr = in->row_bytes / 16;
    const u64 tiles = (n + kStreamTile - 1) / kStreamTile;
    const u64 cells = (u64)parts * tiles;
    const u64 nblocks = (cells + 1023) / 1024;
    DevBuf<u64> counts, sums;
    YTGPU_TRY(counts.allocate(ctx, cells));
    YTGPU_TRY(sums.allocate(ctx, nblocks));
    DestTable D{};
    for (u32 p = 0; p < parts; ++p) {
        D.base[p] = reinterpret_cast<uint4*>(dest_base[p]);
        D.start[p] = start[p];
    }
    u32 bits = 0;
    while ((1u << bits) < parts) ++bits;
    DevBuf<u64> dstart;
    YTGPU_TRY(dstart.allocate(ctx, parts + 1));
    YTGPU_CUDA_TRY(cudaMemcpyAsync(dstart.p, start.data(), (parts + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    {
        KernelTimer t(ctx, KC_PARTITION, 5);
        tile_count_kernel<<<(u32)tiles, kStreamThreads, 0, ctx->stream>>>(index, n, parts, tiles, counts.p, ctx->dev_err);
        pscan_blocks_kernel<false><<<(u32)nblocks, 256, 0, ctx->stream>>>(counts.p, cells, sums.p);
        pscan_sums_kernel<<<1, 256, 0, ctx->stream>>>(sums.p, nblocks);
        pscan_blocks_kernel<true><<<(u32)nblocks, 256, 0, ctx->stream>>>(counts.p, cells, sums.p);
        check_partition_totals_kernel<<<1, 32, 0, ctx->stream>>>(counts.p, tiles, n, parts, dstart.p, ctx->dev_err);
    }
    // caller-supplied indices / counts are validated BEFORE anything is written into another GPU's memory
    YTGPU_TRY(check_device_errors(ctx));
    {
        KernelTimer t(ctx, KC_SCATTER);
        scatter_stream_kernel<<<(u32)tiles, kStreamThreads, 0, ctx->stream>>>(reinterpret_cast<const uint4*>(in->rows), index, n, gr, parts,
                                                                             bits, tiles, counts.p, D);
    }
    YTGPU_CUDA_TRY(cudaGetLastError());
    YTGPU_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return Status{};
}

Status scatter_impl(Context* ctx, const ytgpu_fixed_rows_view* in, const i32* index, i32 parts, const u64* part_rows,
                    void* const* dest_base) {
    if (!in || !index || !part_rows || !dest_base) return make_status(YTGPU_ERR_INVALID_ARGUMENT, "null argument");
    if (in->mem != YTGPU_MEM_DEVICE) return make_status(YTGPU_ERR_INVALID_ARGUMENT, "peer scatter needs device-resident rows");
    if (parts <= 0 || parts > kMaxScatterPartitions) return make_status(YTGPU_ERR_INVALID_ARGUMENT, "partition_count must be in [1, %d]", kMaxScatterPartitions);
    const u64 n = in->row_count;
    const u32 rb = in->row_bytes;
    if (rb == 0 || rb % 16) return make_status(YTGPU_ERR_INVALID_ARGUMENT, "row_bytes must be a positive multiple of 16");
    YTGPU_CUDA_TRY(cudaSetDevice(ctx->device));
    std::vector<u64> start(parts + 1, 0);
    for (i32 p = 0; p < parts; ++p) start[p + 1] = start[p] + part_rows[p];
    if (start[parts] != n) return make_status(YTGPU_ERR_INVALID_ARGUMENT, "partition row counts sum to %llu, table has %llu rows",
                                              (unsigned long long)start[parts], (unsigned long long)n);
    if (n == 0) return Status{};
    if (parts <= kStreamMaxParts) return scatter_stream(ctx, in, index, (u32)parts, start, dest_base);
    // many partitions: partition index -> sort key chunk -> stable permutation (one radix pass per 256 partitions)
    DevBuf<u64> chunk, dstart;
    DevBuf<void*> ddest;
    YTGPU_TRY(chunk.allocate(ctx, n));
    YTGPU_TRY(dstart.allocate(ctx, parts + 1));
    YTGPU_TRY(ddest.allocate(ctx, parts));
    YTGPU_CUDA_TRY(cudaMemcpyAsync(dstart.p, start.data(), (parts + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    YTGPU_CUDA_TRY(cudaMemcpyAsync(ddest.p, dest_base, parts * sizeof(void*), cudaMemcpyHostToDevice, ctx->stream));
    YTGPU_TRY(widen_index(ctx, index, n, chunk.p));
    SortScratch scratch;
    PermRef perm;
    const u64* cptr[1] = {chunk.p};
    YTGPU_TRY(radix_sort_chunks(ctx, cptr, 1, n, &scratch, &perm));
    {
        KernelTimer t(ctx, KC_GATHER);
        constexpr int UNROLL = 4;
        const u32 gr = rb / 16;
        const u64 items = (n * gr + UNROLL - 1) / UNROLL;
        const u32 grid = (u32)std::max<u64>(1, std::min<u64>((items + 255) / 256, (u64)kNumSms * 8));
        const size_t smem = (size_t)(parts + 1) * 8 + (size_t)parts * sizeof(void*);
        scatter_rows_to_peers_kernel<UNROLL><<<grid, 256, smem, ctx->stream>>>(
            reinterpret_cast<const uint4*>(in->rows), perm.plan, perm.idx[0], perm.idx[1], n, gr, (u32)parts, dstart.p,
            reinterpret_cast<uint4* const*>(ddest.p));
        YTGPU_CUDA_TRY(cudaGetLastError());
    }
    // start/dest host vectors are consumed by the async copies: wait before they go out of scope
    YTGPU_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return Status{};
}

}  // namespace

extern "C" {

int ytgpu_peer_buffer_create(ytgpu_context* h, uint64_t bytes, void** out_dev_ptr, uint8_t* out_handle, ytgpu_error* err) {
    if (!h || !out_dev_ptr || !out_handle) return fill_error(err, make_status(YTGPU_ERR_INVALID_ARGUMENT, "null argument"));
    CtxLock lock(h);
    Context* ctx = as_context(h);
    auto run = [&]() -> Status {
        YTGPU_CUDA_TRY(cudaSetDevice(ctx->device));
        void* p = nullptr;
        cudaError_t e = cudaMalloc(&p, bytes ? bytes : 256);
        if (e == cudaErrorMemoryAllocation) {
            cudaGetLastError();
            return make_status(YTGPU_ERR_OUT_OF_MEMORY, "cudaMalloc(%llu bytes) failed", (unsigned long long)bytes);
        }
        if (e != cudaSuccess) return cuda_status(e, "cudaMalloc");
        static_assert(sizeof(cudaIpcMemHandle_t) == YTGPU_IPC_HANDLE_BYTES, "IPC handle size");
        cudaIpcMemHandle_t ih;
        e = cudaIpcGetMemHandle(&ih, p);
        if (e != cudaSuccess) {
            cudaFree(p);
            return cuda_status(e, "cudaIpcGetMemHandle");
        }
        memcpy(out_handle, &ih, sizeof(ih));
        *out_dev_ptr = p;
        return Status{};
    };
    return fill_error(err, run());
}

int ytgpu_peer_buffer_destroy(ytgpu_context* h, void* dev_ptr, ytgpu_error* err) {
    if (!h) return fill_error(err, make_status(YTGPU_ERR_INVALID_ARGUMENT, "null context"));
    CtxLock lock(h);
    Context* ctx = as_context(h);
    auto run = [&]() -> Status {
        YTGPU_CUDA_TRY(cudaSetDevice(ctx->device));
        YTGPU_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        if (dev_ptr) YTGPU_CUDA_TRY(cudaFree(dev_ptr));
        return Status{};
    };
    return fill_error(err, run());
}

int ytgpu_peer_buffer_open(ytgpu_context* h, const uint8_t* handle, void** out_dev_ptr, ytgpu_error* err) {
    if (!h || !handle || !out_dev_ptr) return fill_error(err, make_status(YTGPU_ERR_INVALID_ARGUMENT, "null argument"));
    CtxLock lock(h);
    Context* ctx = as_context(h);
    auto run = [&]() -> Status {
        YTGPU_CUDA_TRY(cudaSetDevice(ctx->device));
        cudaIpcMemHandle_t ih;
        memcpy(&ih, handle, sizeof(ih));
        YTGPU_CUDA_TRY(cudaIpcOpenMemHandle(out_dev_ptr, ih, cudaIpcMemLazyEnablePeerAccess));
        return Status{};
    };
    return fill_error(err, run());
}

int ytgpu_peer_buffer_close(ytgpu_context* h, void* dev_ptr, ytgpu_error* err) {
    if (!h) return fill_error(err, make_status(YTGPU_ERR_INVALID_ARGUMENT, "null context"));
    CtxLock lock(h);
    Context* ctx = as_context(h);
    auto run = [&]() -> Status {
        YTGPU_CUDA_TRY(cudaSetDevice(ctx->device));
        YTGPU_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        if (dev_ptr) YTGPU_CUDA_TRY(cudaIpcCloseMemHandle(dev_ptr));
        return Status{};
    };
    return fill_error(err, run());
}

int ytgpu_scatter_rows_to_peers(ytgpu_context* h, const ytgpu_fixed_rows_view* in, const int32_t* partition_index,
                                int32_t partition_count, const uint64_t* partition_rows, void* const* dest_base,
                                ytgpu_error* err) {
    if (!h) return fill_error(err, make_status(YTGPU_ERR_INVALID_ARGUMENT, "null context"));
    CtxLock lock(h);
    return fill_error(err, scatter_impl(as_context(h), in, partition_index, partition_count, partition_rows, dest_base));
}

}  // extern "C"
