// rows.cu — key extraction / normalisation and row gather kernels (HBM-bound byte movers).
//
// The gather replaces TSortingReader::Read serving rows in sorted order
// (yt/yt/ytlib/table_client/sorting_reader.cpp:58-81) and TPartitionSortReader::Read's
// JumpToRowIndex + GetRow random-access decode (partition_sort_reader.cpp:136-146).
#include "rows.cuh"

namespace ytgpu {
namespace {

// ---- single 8-byte scalar key of a fixed-width row: 8 B written per row, one 32 B sector read ----
template <bool HIST>
__global__ void __launch_bounds__(256) extract_scalar_key_kernel(const u8* __restrict__ rows, u64 n, u32 row_bytes,
                                                                 u32 offset, u8 type, u8 desc, u64* __restrict__ out,
                                                                 u32* __restrict__ hist) {
    __shared__ u32 sh[HIST ? kPassesPerChunk * kRadix : 1];
    if (HIST) {
        for (int i = threadIdx.x; i < kPassesPerChunk * kRadix; i += 256) sh[i] = 0;
        __syncthreads();
    }
    const u64 stride = (u64)gridDim.x * blockDim.x;
    // warp-uniform trip count so that hist_accumulate sees whole warps
    for (u64 base = (u64)blockIdx.x * blockDim.x; base < n; base += stride) {
        const u64 i = base + threadIdx.x;
        const bool valid = i < n;
        u64 v = 0;
        if (valid) {
            v = ld_stream_u64(reinterpret_cast<const u64*>(rows + i * row_bytes + offset));
            if (type == YTGPU_TYPE_INT64) v ^= 0x8000000000000000ull;
            else if (type == YTGPU_TYPE_DOUBLE) v = normalize_double_bits(v);
            if (desc) v = ~v;
            out[i] = v;
        }
        if (HIST) hist_accumulate(sh, v, valid);
    }
    if (HIST) {
        __syncthreads();
        for (int i = threadIdx.x; i < kPassesPerChunk * kRadix; i += 256) {
            u32 c = sh[i];
            if (c) atomicAdd(&hist[i], c);
        }
    }
}

__global__ void __launch_bounds__(256) normalize_fixed_rows_kernel(const KeyLayout L, const u8* __restrict__ rows, u64 n,
                                                                   u32 row_bytes, const ChunkPtrs chunks) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        u64 words[kMaxKeyChunks];
        ChunkWriter w(words);
        const u8* row = rows + i * row_bytes;
        for (u32 c = 0; c < L.ncols; ++c) normalize_fixed(L.col[c], row, w);
        w.finish();
        for (u32 c = 0; c < L.nchunks; ++c) chunks.p[c][i] = words[c];
    }
}

// ---- fixed rows whose key columns are all whole 64-bit words (8-byte scalars and strings of 8k bytes at 8-aligned
// offsets, no type bytes): every chunk of the normalised key is ONE transformed word of the row.  Up to
// kWordHistChunks chunks get their digit histograms in the same pass. ----
constexpr int kWordHistChunks = 4;
struct WordProgram {
    u16 src_off[kMaxKeyChunks];
    u8 kind[kMaxKeyChunks];  // 0 uint64, 1 int64, 2 double, 3 string word (bytes are big-endian already: swap)
    u8 desc[kMaxKeyChunks];
    u32 nchunks;
};

__device__ __forceinline__ u64 bswap64(u64 v) {
    const u32 lo = (u32)v, hi = (u32)(v >> 32);
    return ((u64)__byte_perm(lo, 0, 0x0123) << 32) | __byte_perm(hi, 0, 0x0123);
}

template <bool HIST>
__global__ void __launch_bounds__(256) normalize_fixed_words_kernel(const WordProgram W, const u8* __restrict__ rows, u64 n, u32 row_bytes,
                                                                    const ChunkPtrs chunks, u32* __restrict__ hist) {
    __shared__ u32 sh[HIST ? kWordHistChunks * kPassesPerChunk * kRadix : 1];
    if (HIST) {
        for (int i = threadIdx.x; i < (int)W.nchunks * kPassesPerChunk * kRadix; i += 256) sh[i] = 0;
        __syncthreads();
    }
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (u64 base = (u64)blockIdx.x * blockDim.x; base < n; base += stride) {  // warp-uniform trips (hist_accumulate)
        const u64 i = base + threadIdx.x;
        const bool valid = i < n;
        for (u32 c = 0; c < W.nchunks; ++c) {
            u64 v = 0;
            if (valid) {
                v = *reinterpret_cast<const u64*>(rows + i * row_bytes + W.src_off[c]);
                const u32 kind = W.kind[c];
                if (kind == 3) v = bswap64(v);
                else if (kind == 1) v ^= 0x8000000000000000ull;
                else if (kind == 2) v = normalize_double_bits(v);
                if (W.desc[c]) v = ~v;
                chunks.p[c][i] = v;
            }
            if (HIST) hist_accumulate(sh + c * kPassesPerChunk * kRadix, v, valid);
        }
    }
    if (HIST) {
        __syncthreads();
        for (int i = threadIdx.x; i < (int)W.nchunks * kPassesPerChunk * kRadix; i += 256) {
            const u32 c = sh[i];
            if (c) atomicAdd(&hist[i], c);
        }
    }
}

// Builds the word program when the layout qualifies.
static bool make_word_program(const KeyLayout& L, u32 row_bytes, WordProgram* W) {
    if (row_bytes % 8) return false;
    u32 nc = 0;
    for (u32 c = 0; c < L.ncols; ++c) {
        const KeyColLayout& k = L.col[c];
        if (k.has_type_byte || k.index % 8) return false;
        if (k.type == YTGPU_TYPE_STRING) {
            if (k.width == 0 || k.width % 8) return false;
            for (u32 w = 0; w < k.width / 8; ++w) {
                if (nc >= (u32)kMaxKeyChunks) return false;
                W->src_off[nc] = (u16)(k.index + 8 * w);
                W->kind[nc] = 3;
                W->desc[nc] = k.descending;
                ++nc;
            }
        } else if (k.type == YTGPU_TYPE_UINT64 || k.type == YTGPU_TYPE_INT64 || k.type == YTGPU_TYPE_DOUBLE) {
            if (nc >= (u32)kMaxKeyChunks) return false;
            W->src_off[nc] = (u16)k.index;
            W->kind[nc] = k.type == YTGPU_TYPE_UINT64 ? 0 : (k.type == YTGPU_TYPE_INT64 ? 1 : 2);
            W->desc[nc] = k.descending;
            ++nc;
        } else {
            return false;
        }
    }
    W->nchunks = nc;
    return nc == L.nchunks && row_bytes < 65536;
}

__global__ void __launch_bounds__(256) normalize_rowset_kernel(const KeyLayout L, const ytgpu_value* __restrict__ values,
                                                               u32 value_count, const u8* __restrict__ heap, u64 n,
                                                               const ChunkPtrs chunks, u32* __restrict__ err_word) {
    u32 err = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        u64 words[kMaxKeyChunks];
        ChunkWriter w(words);
        const ytgpu_value* row = values + i * value_count;
        for (u32 c = 0; c < L.ncols; ++c) {
            uint4 raw = *reinterpret_cast<const uint4*>(row + L.col[c].index);
            ytgpu_value v;
            v.id = (u16)(raw.x & 0xffff);
            v.type = (u8)((raw.x >> 16) & 0xff);
            v.flags = (u8)(raw.x >> 24);
            v.length = raw.y;
            v.data = ((u64)raw.w << 32) | raw.z;
            err |= normalize_value(L.col[c], v, heap, w);
        }
        w.finish();
        for (u32 c = 0; c < L.nchunks; ++c) chunks.p[c][i] = words[c];
    }
    if (err) atomicOr(err_word, err);
}

struct WidthCols {
    u32 index[kMaxKeyColumns];
    u32 ncols;
};

__global__ void __launch_bounds__(256) max_string_length_kernel(const WidthCols W, const ytgpu_value* __restrict__ values,
                                                                u32 value_count, u64 n, u32* __restrict__ out) {
    u32 mx[kMaxKeyColumns];
    for (u32 c = 0; c < W.ncols; ++c) mx[c] = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        for (u32 c = 0; c < W.ncols; ++c) {
            const ytgpu_value* v = values + i * value_count + W.index[c];
            uint2 head = *reinterpret_cast<const uint2*>(v);
            u8 type = (u8)((head.x >> 16) & 0xff);
            if (type == YTGPU_TYPE_STRING) mx[c] = max(mx[c], head.y);
        }
    }
    for (u32 c = 0; c < W.ncols; ++c) {
        u32 m = __reduce_max_sync(0xffffffffu, mx[c]);
        if (lane_id() == 0 && m) atomicMax(&out[c], m);
    }
}

// ---- gather: 16-byte granules; GR granules per row; each thread moves UNROLL granules ----
// Loads and stores bypass L1 (L1::no_allocate): every granule is touched once.
template <int UNROLL, bool PLAIN>
__global__ void __launch_bounds__(256) gather_rows_kernel(const uint4* __restrict__ in, const SortPlan* plan,
                                                          const u32* __restrict__ pa, const u32* __restrict__ pb,
                                                          uint4* __restrict__ out, u64 n, u32 gr, u32 gr_shift) {
    const u64 total = n * gr;
    const u32 f = PLAIN ? 0u : plan_final_idx(plan);
    const u32* perm = f == 1 ? pb : pa;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    u64 q0 = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    for (; q0 < total; q0 += stride * UNROLL) {
        uint4 v[UNROLL];
        bool ok[UNROLL];
#pragma unroll
        for (int k = 0; k < UNROLL; ++k) {
            u64 q = q0 + (u64)k * stride;
            ok[k] = q < total;
            if (ok[k]) {
                u64 j;
                u32 g;
                if (gr_shift != 0xffffffffu) {
                    j = q >> gr_shift;
                    g = (u32)(q & (gr - 1));
                } else {
                    j = q / gr;
                    g = (u32)(q - j * gr);
                }
                u64 src = (f == 2 ? j : (u64)perm[j]);
                v[k] = ld_stream_u128(in + src * gr + g);
            }
        }
#pragma unroll
        for (int k = 0; k < UNROLL; ++k) {
            u64 q = q0 + (u64)k * stride;
            if (ok[k]) st_stream_u128(out + q, v[k]);
        }
    }
}

__global__ void __launch_bounds__(256) widen_index_kernel(const i32* __restrict__ in, u64 n, u64* __restrict__ out) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) out[i] = (u64)(u32)in[i];
}

inline u32 grid_for(u64 work_items, int threads, int blocks_per_sm) {
    u64 b = (work_items + threads - 1) / threads;
    u64 cap = (u64)kNumSms * blocks_per_sm;
    return (u32)std::max<u64>(1, std::min(b, cap));
}

}  // namespace

Status normalize_fixed_rows(Context* ctx, const KeyLayout& L, const u8* rows_dev, u64 n, u32 row_bytes,
                            const ChunkPtrs& chunks, u32* hist, bool* hist_done) {
    if (hist_done) *hist_done = false;
    if (n == 0) return Status{};
    KernelTimer t(ctx, KC_EXTRACT);
    const KeyColLayout& c0 = L.col[0];
    bool scalar8 = L.ncols == 1 && !c0.has_type_byte && c0.payload_bytes == 8 && c0.type != YTGPU_TYPE_STRING &&
                   (c0.index % 8 == 0) && (row_bytes % 8 == 0);
    if (scalar8) {
        if (hist) {
            extract_scalar_key_kernel<true><<<grid_for(n, 256, 8), 256, 0, ctx->stream>>>(rows_dev, n, row_bytes, c0.index, c0.type,
                                                                                         c0.descending, chunks.p[0], hist);
            if (hist_done) *hist_done = true;
        } else {
            extract_scalar_key_kernel<false><<<grid_for(n, 256, 8), 256, 0, ctx->stream>>>(rows_dev, n, row_bytes, c0.index, c0.type,
                                                                                          c0.descending, chunks.p[0], nullptr);
        }
    } else {
        WordProgram W{};
        if (make_word_program(L, row_bytes, &W)) {
            if (hist && W.nchunks <= (u32)kWordHistChunks) {
                normalize_fixed_words_kernel<true><<<grid_for(n, 256, 4), 256, 0, ctx->stream>>>(W, rows_dev, n, row_bytes, chunks, hist);
                if (hist_done) *hist_done = true;
            } else {
                normalize_fixed_words_kernel<false><<<grid_for(n, 256, 8), 256, 0, ctx->stream>>>(W, rows_dev, n, row_bytes, chunks, nullptr);
            }
        } else {
            normalize_fixed_rows_kernel<<<grid_for(n, 256, 8), 256, 0, ctx->stream>>>(L, rows_dev, n, row_bytes, chunks);
        }
    }
    YTGPU_CUDA_TRY(cudaGetLastError());
    return Status{};
}

Status normalize_rowset(Context* ctx, const KeyLayout& L, const ytgpu_value* values_dev, u32 value_count,
                        const u8* heap_dev, u64 n, const ChunkPtrs& chunks) {
    if (n == 0) return Status{};
    KernelTimer t(ctx, KC_EXTRACT);
    normalize_rowset_kernel<<<grid_for(n, 256, 8), 256, 0, ctx->stream>>>(L, values_dev, value_count, heap_dev, n, chunks,
                                                                          ctx->dev_err);
    YTGPU_CUDA_TRY(cudaGetLastError());
    return Status{};
}

Status measure_string_widths(Context* ctx, const ytgpu_sort_spec* spec, const ytgpu_value* values_dev,
                             u32 value_count, u64 n, u32* max_len_host) {
    WidthCols W{};
    W.ncols = spec->column_count;
    for (u32 c = 0; c < W.ncols; ++c) {
        W.index[c] = spec->columns[c].index;
        max_len_host[c] = 0;
    }
    if (n == 0) return Status{};
    DevBuf<u32> out;
    YTGPU_TRY(out.allocate(ctx, kMaxKeyColumns));
    YTGPU_CUDA_TRY(cudaMemsetAsync(out.p, 0, kMaxKeyColumns * 4, ctx->stream));
    max_string_length_kernel<<<grid_for(n, 256, 8), 256, 0, ctx->stream>>>(W, values_dev, value_count, n, out.p);
    ctx->count_launch();
    YTGPU_CUDA_TRY(cudaMemcpyAsync(max_len_host, out.p, W.ncols * 4, cudaMemcpyDeviceToHost, ctx->stream));
    YTGPU_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return Status{};
}

static Status gather_launch(Context* ctx, const u8* in_dev, const SortPlan* plan, const u32* pa, const u32* pb,
                            u8* out_dev, u64 n, u32 row_bytes, bool plain) {
    if (n == 0) return Status{};
    if (row_bytes == 0 || row_bytes % 16 != 0)
        return make_status(YTGPU_ERR_INVALID_ARGUMENT, "row_bytes (%u) must be a positive multiple of 16", row_bytes);
    u32 gr = row_bytes / 16;
    u32 shift = (gr & (gr - 1)) == 0 ? (u32)__builtin_ctz(gr) : 0xffffffffu;
    KernelTimer t(ctx, KC_GATHER);
    constexpr int UNROLL = 4;
    u32 grid = grid_for((n * gr + UNROLL - 1) / UNROLL, 256, 8);
    const uint4* in4 = reinterpret_cast<const uint4*>(in_dev);
    uint4* out4 = reinterpret_cast<uint4*>(out_dev);
    if (plain) gather_rows_kernel<UNROLL, true><<<grid, 256, 0, ctx->stream>>>(in4, nullptr, pa, pb, out4, n, gr, shift);
    else gather_rows_kernel<UNROLL, false><<<grid, 256, 0, ctx->stream>>>(in4, plan, pa, pb, out4, n, gr, shift);
    YTGPU_CUDA_TRY(cudaGetLastError());
    return Status{};
}

Status widen_index(Context* ctx, const i32* index_dev, u64 n, u64* chunk_dev) {
    if (n == 0) return Status{};
    widen_index_kernel<<<grid_for(n, 256, 8), 256, 0, ctx->stream>>>(index_dev, n, chunk_dev);
    ctx->count_launch();
    YTGPU_CUDA_TRY(cudaGetLastError());
    return Status{};
}

Status gather_rows(Context* ctx, const u8* in_dev, const PermRef& perm, u8* out_dev, u64 n, u32 row_bytes) {
    return gather_launch(ctx, in_dev, perm.plan, perm.idx[0], perm.idx[1], out_dev, n, row_bytes, false);
}

Status gather_rows_plain(Context* ctx, const u8* in_dev, const u32* perm_dev, u8* out_dev, u64 n, u32 row_bytes) {
    return gather_launch(ctx, in_dev, nullptr, perm_dev, perm_dev, out_dev, n, row_bytes, true);
}

}  // namespace ytgpu
