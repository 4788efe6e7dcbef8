// shuffle.cu — the in-box distributed sort behind the C ABI (ytgpu_shuffle_*), one process (or thread) per GPU.
//
// Reference shape: the sort controller samples keys, builds partition keys from the samples
// (yt/yt/server/controller_agent/helpers.cpp:263-425), partition jobs route every row with the ordered partitioner
// (yt/yt/ytlib/table_client/partitioner.cpp:41-57) into per-partition blocks
// (schemaless_chunk_writer.cpp:1604-1667), sort jobs fetch their partition (partition_chunk_reader.cpp:82-86) and
// sort it (sort_controller.cpp:3444-3456, partition_sort_reader.cpp:384-529).  Inside one NVSwitch box all of that is
// a fixed sequence of kernels on every rank's stream; ranks talk ONLY through peer-mapped device memory:
//   sample keys  -> normalised sample keys stored straight into every peer's sample area
//   barrier      -> one warp: st.release.sys of an epoch into every peer's control block, ld.acquire.sys spin
//   pivots       -> every rank sorts the same samples with the same kernels and picks the same P-1 lower bounds
//                   (weights = rows represented by a sample; equal keys collapse into maniac partitions)
//   partition    -> ONE pass over the rows: normalise key, binary search over the pivots, partition index + per-tile
//                   partition counts (for the stable scatter)
//   counts       -> every rank stores its row of the g x g count matrix into every peer, barrier
//   scatter      -> rows are read sequentially and written to their stable slot of the destination's receive
//                   buffer over NVLink (peer_kernels.cuh), barrier
//   local sort   -> the rank's key range (capi_sort.cu)
// The host takes part once per sort (it reads the count matrix to size the local sort); no NCCL, no host barrier.
#include <cstring>
#include <new>
#include <vector>

#include "context.cuh"
#include "keys.cuh"
#include "partition_keys.cuh"
#include "peer_kernels.cuh"
#include "radix_sort.cuh"
#include "rows.cuh"

using namespace ytgpu;

namespace {

constexpr int kMaxRanks = kStreamMaxParts;  // 32
constexpr u32 kSamplesPerRank = 2048;       // >= TSortOperationSpecBase::SamplesPerPartition (1000) per partition
constexpr u64 kBarrierTimeoutNs = 20ull * 1000 * 1000 * 1000;

// Head of every rank's peer-visible allocation.  Rows [src] are written by rank src (remotely), read locally.
struct ShuffleCtrl {
    u32 arrive[kMaxRanks];             // barrier epochs
    u64 counts[kMaxRanks][kMaxRanks];  // counts[src][dst]: rows src sends to dst
    u64 rows[kMaxRanks];               // rows held by src
    u32 take[kMaxRanks];               // real samples contributed by src (the rest of its kSamplesPerRank are padding)
};

constexpr size_t kCtrlBytes = (sizeof(ShuffleCtrl) + 4095) / 4096 * 4096;

inline size_t sample_area_bytes(int world) { return (size_t)kMaxKeyChunks * world * kSamplesPerRank * 8; }
inline size_t rows_offset(int world) { return kCtrlBytes + (sample_area_bytes(world) + 4095) / 4096 * 4096; }

struct PeerBases {
    u8* base[kMaxRanks];
};

struct Pivots {  // device-resident result of the pivot selection, identical on every rank
    u64 words[kMaxRanks][kMaxKeyChunks];  // lower bound of partition p+1 (normalised key)
    u8 inclusive[kMaxRanks];
    u8 maniac[kMaxRanks];  // partition p holds a single key
    u32 count;             // == world - 1
};

__device__ __forceinline__ u64 global_timer_ns() {
    u64 t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void st_release_sys(u32* p, u32 v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ u32 ld_acquire_sys(const u32* p) {
    u32 v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// One warp.  Lane q signals peer q and waits for peer q.  Epochs only grow, so no flag is ever reset.
__global__ void peer_barrier_kernel(const PeerBases peers, int world, int rank, u32 epoch, u32* err_word) {
    const int lane = threadIdx.x;
    __threadfence_system();  // everything this GPU wrote before (earlier kernels included) precedes the flag
    if (lane < world) st_release_sys(&reinterpret_cast<ShuffleCtrl*>(peers.base[lane])->arrive[rank], epoch);
    if (lane < world) {
        const u32* mine = &reinterpret_cast<const ShuffleCtrl*>(peers.base[rank])->arrive[lane];
        const u64 t0 = global_timer_ns();
        while ((i32)(ld_acquire_sys(mine) - epoch) < 0) {
            if (global_timer_ns() - t0 > kBarrierTimeoutNs) {
                atomicOr(err_word, (u32)DE_PEER_TIMEOUT);
                break;
            }
            __nanosleep(200);
        }
    }
    __threadfence_system();
}

// Normalised key words of one fixed-width row.
template <bool SCALAR8>
__device__ __forceinline__ void row_key(const KeyLayout& L, const u8* row, u64* words) {
    if (SCALAR8) {
        const KeyColLayout& c = L.col[0];
        u64 v = *reinterpret_cast<const u64*>(row + c.index);
        if (c.type == YTGPU_TYPE_INT64) v ^= 0x8000000000000000ull;
        else if (c.type == YTGPU_TYPE_DOUBLE) v = normalize_double_bits(v);
        if (c.descending) v = ~v;
        words[0] = v;
    } else {
        ChunkWriter w(words);
        for (u32 c = 0; c < L.ncols; ++c) normalize_fixed(L.col[c], row, w);
        w.finish();
    }
}

// Every rank contributes exactly kSamplesPerRank samples so that the sample count is known to every host:
// t < take are evenly spaced rows (each stands for n / take rows), the rest repeat the last one with weight 0.
// Sample area layout (per rank): [chunk][src rank][t] -> chunk c of all samples is one contiguous array.
template <bool SCALAR8>
__global__ void __launch_bounds__(256) sample_keys_kernel(const KeyLayout L, const u8* __restrict__ rows, u64 n, u32 row_bytes, u32 take,
                                                          const PeerBases peers, int world, int rank) {
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= kSamplesPerRank) return;
    u64 words[SCALAR8 ? 1 : kMaxKeyChunks];
    for (u32 c = 0; c < L.nchunks; ++c) words[c] = 0;
    if (n > 0) {
        const u32 tt = t < take ? t : take - 1;
        const u64 i = take > 1 ? (u64)(((unsigned __int128)tt * (n - 1)) / (take - 1)) : 0;
        row_key<SCALAR8>(L, rows + i * row_bytes, words);
    }
    const size_t per_chunk = (size_t)world * kSamplesPerRank;
    for (int q = 0; q < world; ++q) {
        u64* area = reinterpret_cast<u64*>(peers.base[q] + kCtrlBytes);
        for (u32 c = 0; c < L.nchunks; ++c) area[c * per_chunk + (size_t)rank * kSamplesPerRank + t] = words[c];
        if (t == 0) {
            ShuffleCtrl* ctrl = reinterpret_cast<ShuffleCtrl*>(peers.base[q]);
            ctrl->rows[rank] = n;
            ctrl->take[rank] = take;
        }
    }
    __threadfence_system();
}

// Pivot selection over the sorted samples: one block.  Weighted prefix sums in sorted order, then thread 0 runs
// BuildPartitionKeysFromSamples (partition_keys.cuh) with one binary search per partition.
constexpr int kPivotThreads = 1024;
__global__ void __launch_bounds__(kPivotThreads) select_pivots_kernel(const u8* local_base, int world, u32 nchunks, const SortPlan* plan,
                                                                      const u32* pa, const u32* pb, double* cum /*[m]*/, Pivots* out) {
    __shared__ double s_part[kPivotThreads];
    __shared__ double s_weight[kMaxRanks];
    const ShuffleCtrl* ctrl = reinterpret_cast<const ShuffleCtrl*>(local_base);
    const u64* area = reinterpret_cast<const u64*>(local_base + kCtrlBytes);
    const u32 m = (u32)world * kSamplesPerRank;
    if (threadIdx.x < (u32)world) {
        const u32 take = ctrl->take[threadIdx.x];
        s_weight[threadIdx.x] = take ? (double)ctrl->rows[threadIdx.x] / (double)take : 0.0;
    }
    __syncthreads();
    auto weight_of = [&](u32 sorted_pos) -> double {
        const u32 j = perm_at(plan, pa, pb, sorted_pos);
        const u32 src = j / kSamplesPerRank, t = j % kSamplesPerRank;
        return t < ctrl->take[src] ? s_weight[src] : 0.0;
    };
    // inclusive prefix sums, the same association order on every rank
    const u32 per = (m + kPivotThreads - 1) / kPivotThreads;
    const u32 lo = min(m, threadIdx.x * per), hi = min(m, lo + per);
    double sum = 0;
    for (u32 i = lo; i < hi; ++i) sum += weight_of(i);
    s_part[threadIdx.x] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        double run = 0;
        for (int i = 0; i < kPivotThreads; ++i) {
            const double v = s_part[i];
            s_part[i] = run;
            run += v;
        }
    }
    __syncthreads();
    double run = s_part[threadIdx.x];
    for (u32 i = lo; i < hi; ++i) {
        run += weight_of(i);
        cum[i] = run;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    const size_t per_chunk = (size_t)world * kSamplesPerRank;
    auto same_key = [&](u32 a, u32 b) -> bool {
        const u32 ja = perm_at(plan, pa, pb, a), jb = perm_at(plan, pa, pb, b);
        for (u32 c = 0; c < nchunks; ++c)
            if (area[c * per_chunk + ja] != area[c * per_chunk + jb]) return false;
        return true;
    };
    PartitionKeyPick picks[kMaxRanks];
    const int npicks = build_partition_keys_from_sorted_samples(m, cum, same_key, world, picks);
    for (int p = 0; p < kMaxRanks; ++p) out->maniac[p] = 0;
    int have = 0;
    for (int k = 0; k < world - 1; ++k) {
        const int src = k < npicks ? k : npicks - 1;  // fewer distinct pivots than ranks: duplicate bounds are legal
        if (src < 0) {  // no samples at all: every bound is the zero key, everything lands in the last partition
            for (u32 c = 0; c < nchunks; ++c) out->words[k][c] = 0;
            out->inclusive[k] = 1;
        } else {
            const u32 j = perm_at(plan, pa, pb, picks[src].sample);
            for (u32 c = 0; c < nchunks; ++c) out->words[k][c] = area[c * per_chunk + j];
            out->inclusive[k] = picks[src].inclusive;
            if (k < npicks && picks[k].maniac) out->maniac[k + 1] = 1;
        }
        ++have;
    }
    out->count = (u32)have;
}

// One pass over the rows: partition index of every row + per-tile partition counts [parts][tiles].
template <bool SCALAR8>
__global__ void __launch_bounds__(kStreamThreads) partition_count_kernel(const KeyLayout L, const u8* __restrict__ rows, u64 n, u32 row_bytes,
                                                                         const Pivots* __restrict__ piv, u32 parts, u64 tiles,
                                                                         i32* __restrict__ index, u64* __restrict__ counts) {
    __shared__ u32 s_cnt[kMaxRanks];
    __shared__ u64 s_piv[SCALAR8 ? kMaxRanks : kMaxRanks * kMaxKeyChunks];
    __shared__ u8 s_inc[kMaxRanks];
    const u32 C = SCALAR8 ? 1 : L.nchunks;
    const u32 nb = parts - 1;
    if (threadIdx.x < kMaxRanks) s_cnt[threadIdx.x] = 0;
    for (u32 i = threadIdx.x; i < nb * C; i += kStreamThreads) s_piv[i] = piv->words[i / C][i % C];
    if (threadIdx.x < nb) s_inc[threadIdx.x] = piv->inclusive[threadIdx.x];
    __syncthreads();
    const u64 base = (u64)blockIdx.x * kStreamTile;
#pragma unroll
    for (int it = 0; it < kStreamItems; ++it) {
        const u64 r = base + (u64)it * kStreamThreads + threadIdx.x;
        if (r >= n) continue;
        u64 words[SCALAR8 ? 1 : kMaxKeyChunks];
        row_key<SCALAR8>(L, rows + r * row_bytes, words);
        // partition = number of lower bounds the key passes (bounds are sorted: binary search)
        u32 lo = 0, cnt = nb;
        while (cnt > 0) {
            const u32 step = cnt >> 1, mid = lo + step;
            int cmp = 0;
            for (u32 c = 0; c < C; ++c) {
                const u64 b = s_piv[mid * C + c];
                if (words[c] != b) {
                    cmp = words[c] > b ? 1 : -1;
                    break;
                }
            }
            if (cmp > 0 || (cmp == 0 && s_inc[mid])) {
                lo = mid + 1;
                cnt -= step + 1;
            } else {
                cnt = step;
            }
        }
        index[r] = (i32)lo;
        atomicAdd(&s_cnt[lo], 1u);
    }
    __syncthreads();
    if (threadIdx.x < parts) counts[(u64)threadIdx.x * tiles + blockIdx.x] = s_cnt[threadIdx.x];
}

// After the scan of the [parts][tiles] count matrix: rows this rank sends to every destination -> all peers.
__global__ void publish_counts_kernel(const u64* __restrict__ scanned, u64 tiles, u64 n, u32 parts, const PeerBases peers, int world,
                                      int rank) {
    const u32 p = threadIdx.x;
    if (p >= parts) return;
    const u64 start = scanned[(u64)p * tiles];
    const u64 end = p + 1 < parts ? scanned[(u64)(p + 1) * tiles] : n;
    for (int q = 0; q < world; ++q) reinterpret_cast<ShuffleCtrl*>(peers.base[q])->counts[rank][p] = end - start;
    __threadfence_system();
}

struct Shuffle {
    Context* ctx = nullptr;
    int world = 0, rank = 0;
    u64 capacity_rows = 0;
    u32 row_bytes = 0;
    u8* base = nullptr;  // this rank's peer-visible allocation
    size_t bytes = 0;
    PeerBases peers{};
    bool opened[kMaxRanks] = {false};
    bool connected = false;
    u32 epoch = 0;
    Pivots* pivots = nullptr;      // device
    double* cum = nullptr;         // device, [world * kSamplesPerRank]
    u8* host_stage = nullptr;      // pinned: ShuffleCtrl counts matrix + Pivots tail
};

Status barrier(Shuffle* s) {
    ++s->epoch;
    peer_barrier_kernel<<<1, 32, 0, s->ctx->stream>>>(s->peers, s->world, s->rank, s->epoch, s->ctx->dev_err);
    s->ctx->count_launch();
    YTGPU_CUDA_TRY(cudaGetLastError());
    return Status{};
}

bool is_scalar8(const KeyLayout& L, u32 row_bytes) {
    const KeyColLayout& c0 = L.col[0];
    return L.ncols == 1 && !c0.has_type_byte && c0.payload_bytes == 8 && c0.type != YTGPU_TYPE_STRING && (c0.index % 8 == 0) &&
           (row_bytes % 8 == 0);
}

Status shuffle_sort_impl(Shuffle* s, const ytgpu_fixed_rows_view* in, const ytgpu_sort_spec* spec, u8* out_rows, u64 out_capacity_rows,
                         u64* out_row_count, ytgpu_shuffle_stats* stats) {
    if (!in || !spec || !spec->columns || !out_row_count) return make_status(YTGPU_ERR_INVALID_ARGUMENT, "null argument");
    if (!s->connected) return make_status(YTGPU_ERR_INVALID_ARGUMENT, "ytgpu_shuffle_connect has not been called");
    if (in->mem != YTGPU_MEM_DEVICE) return make_status(YTGPU_ERR_INVALID_ARGUMENT, "the in-box shuffle sorts device-resident rows");
    if (in->row_bytes != s->row_bytes) return make_status(YTGPU_ERR_INVALID_ARGUMENT, "row_bytes %u differs from the shuffle's %u", in->row_bytes, s->row_bytes);
    Context* ctx = s->ctx;
    cudaStream_t st = ctx->stream;
    const int world = s->world, rank = s->rank;
    const u64 n = in->row_count;
    const u32 rb = in->row_bytes;
    KeyLayout L;
    YTGPU_TRY(build_key_layout(spec, /*fixed_rows*/ true, false, &L));
    for (u32 c = 0; c < L.ncols; ++c)
        if ((u64)L.col[c].index + L.col[c].payload_bytes > rb) return make_status(YTGPU_ERR_INVALID_ARGUMENT, "key column %u exceeds the row", c);
    YTGPU_CUDA_TRY(cudaSetDevice(ctx->device));
    const bool scalar8 = is_scalar8(L, rb);
    const u32 m = (u32)world * kSamplesPerRank;
    const u32 parts = (u32)world;

    // ---- 1. samples into every peer, barrier ----
    {
        KernelTimer t(ctx, KC_SHUFFLE_SYNC, 2);
        const u32 take = (u32)std::min<u64>(n, kSamplesPerRank);
        if (scalar8) sample_keys_kernel<true><<<kSamplesPerRank / 256, 256, 0, st>>>(L, in->rows, n, rb, take, s->peers, world, rank);
        else sample_keys_kernel<false><<<kSamplesPerRank / 256, 256, 0, st>>>(L, in->rows, n, rb, take, s->peers, world, rank);
        YTGPU_TRY(barrier(s));
    }
    // ---- 2. identical pivots on every rank ----
    SortScratch sample_scratch;
    {
        const bool timers = ctx->timers_enabled;
        KernelTimer t(ctx, KC_SHUFFLE_SYNC, 1);
        ctx->timers_enabled = false;  // the sample sort's tiny passes are not radix-pass measurements
        const u64* cptrs[kMaxKeyChunks];
        for (u32 c = 0; c < L.nchunks; ++c) cptrs[c] = reinterpret_cast<const u64*>(s->base + kCtrlBytes) + (size_t)c * m;
        PermRef perm;
        Status ss = radix_sort_chunks(ctx, cptrs, (int)L.nchunks, m, &sample_scratch, &perm);
        ctx->timers_enabled = timers;
        YTGPU_TRY(ss);
        select_pivots_kernel<<<1, kPivotThreads, 0, st>>>(s->base, world, L.nchunks, perm.plan, perm.idx[0], perm.idx[1], s->cum, s->pivots);
        YTGPU_CUDA_TRY(cudaGetLastError());
    }
    // ---- 3. partition index + per-tile counts, scan, publish the counts, barrier ----
    const u64 tiles = std::max<u64>(1, (n + kStreamTile - 1) / kStreamTile);
    const u64 cells = (u64)parts * tiles;
    const u64 nblocks = (cells + 1023) / 1024;
    DevBuf<i32> index;
    DevBuf<u64> counts, sums;
    YTGPU_TRY(index.allocate(ctx, std::max<u64>(n, 1)));
    YTGPU_TRY(counts.allocate(ctx, cells));
    YTGPU_TRY(sums.allocate(ctx, nblocks));
    {
        KernelTimer t(ctx, KC_PARTITION);  // one timed unit: the partition/count pass + the three tiny scan launches
        ctx->count_launch(3);
        if (scalar8) partition_count_kernel<true><<<(u32)tiles, kStreamThreads, 0, st>>>(L, in->rows, n, rb, s->pivots, parts, tiles, index.p, counts.p);
        else partition_count_kernel<false><<<(u32)tiles, kStreamThreads, 0, st>>>(L, in->rows, n, rb, s->pivots, parts, tiles, index.p, counts.p);
        pscan_blocks_kernel<false><<<(u32)nblocks, 256, 0, st>>>(counts.p, cells, sums.p);
        pscan_sums_kernel<<<1, 256, 0, st>>>(sums.p, nblocks);
        pscan_blocks_kernel<true><<<(u32)nblocks, 256, 0, st>>>(counts.p, cells, sums.p);
        YTGPU_CUDA_TRY(cudaGetLastError());
    }
    {
        KernelTimer t(ctx, KC_SHUFFLE_SYNC, 2);
        publish_counts_kernel<<<1, 32, 0, st>>>(counts.p, tiles, n, parts, s->peers, world, rank);
        YTGPU_TRY(barrier(s));
    }
    // ---- 4. the host's one look at the data: the g x g count matrix ----
    ShuffleCtrl* hc = reinterpret_cast<ShuffleCtrl*>(s->host_stage);
    Pivots* hp = reinterpret_cast<Pivots*>(s->host_stage + kCtrlBytes);
    YTGPU_CUDA_TRY(cudaMemcpyAsync(hc, s->base, sizeof(ShuffleCtrl), cudaMemcpyDeviceToHost, st));
    YTGPU_CUDA_TRY(cudaMemcpyAsync(hp, s->pivots, sizeof(Pivots), cudaMemcpyDeviceToHost, st));
    YTGPU_TRY(check_device_errors(ctx));  // synchronises the stream
    u64 total_in = 0, before_me[kMaxRanks] = {0};
    for (int d = 0; d < world; ++d) {
        u64 into_d = 0;
        for (int src = 0; src < world; ++src) {
            if (src == rank) before_me[d] = into_d;
            into_d += hc->counts[src][d];
        }
        if (into_d > s->capacity_rows)  // the same matrix on every rank: all ranks fail together
            return make_status(YTGPU_ERR_INVALID_ARGUMENT, "rank %d would receive %llu rows, its receive buffer holds %llu: raise capacity_rows", d,
                               (unsigned long long)into_d, (unsigned long long)s->capacity_rows);
        if (d == rank) total_in = into_d;
    }
    if (stats) {
        memset(stats, 0, sizeof(*stats));
        stats->rows_in = n;
        stats->rows_out = total_in;
        stats->world = (uint32_t)world;
        stats->maniac = hp->maniac[rank];
        for (int q = 0; q < world; ++q) {
            stats->sent[q] = hc->counts[rank][q];
            stats->received[q] = hc->counts[q][rank];
        }
    }
    *out_row_count = total_in;
    if (out_rows && total_in > out_capacity_rows)
        return make_status(YTGPU_ERR_INVALID_ARGUMENT, "output holds %llu rows, the rank's key range has %llu", (unsigned long long)out_capacity_rows,
                           (unsigned long long)total_in);
    // ---- 5. scatter straight into the destinations' receive buffers, barrier ----
    if (n > 0) {
        DestTable D{};
        u64 startp = 0;
        for (u32 p = 0; p < parts; ++p) {
            D.base[p] = reinterpret_cast<uint4*>(s->peers.base[p] + rows_offset(world) + before_me[p] * rb);
            D.start[p] = startp;
            startp += hc->counts[rank][p];
        }
        u32 bits = 0;
        while ((1u << bits) < parts) ++bits;
        KernelTimer t(ctx, KC_SCATTER);
        // Rows go from the streaming kernel straight to their slabs.  Regrouping a whole tile by destination in shared
        // memory first measured SLOWER at 2 ranks (6.64 vs 4.97 ms for 5*10^7 rows out): the 64-byte row stores already
        // fill whole NVLink packets, staging only adds a shared-memory round trip and a barrier.
        scatter_stream_kernel<<<(u32)tiles, kStreamThreads, 0, st>>>(reinterpret_cast<const uint4*>(in->rows), index.p, n, rb / 16, parts, bits,
                                                                    tiles, counts.p, D);
        YTGPU_CUDA_TRY(cudaGetLastError());
    }
    {
        KernelTimer t(ctx, KC_SHUFFLE_SYNC, 1);
        YTGPU_TRY(barrier(s));
    }
    // ---- 6. local sort of this rank's key range ----
    if (out_rows && total_in > 0) {
        const u8* received = s->base + rows_offset(world);
        if (hp->maniac[rank]) {  // a single key: rows are already in (source rank, position) order
            YTGPU_CUDA_TRY(cudaMemcpyAsync(out_rows, received, total_in * rb, cudaMemcpyDeviceToDevice, st));
        } else {
            ytgpu_fixed_rows_view v{received, total_in, rb, YTGPU_MEM_DEVICE};
            YTGPU_TRY(sort_fixed_rows_impl(ctx, &v, spec, out_rows, nullptr, YTGPU_MEM_DEVICE));
        }
    }
    return Status{};
}

}  // namespace

extern "C" {

int ytgpu_shuffle_create(ytgpu_context* h, int world, int rank, uint64_t capacity_rows, uint32_t row_bytes, ytgpu_shuffle** out,
                         uint8_t* out_handle, ytgpu_error* err) {
    if (!h || !out || !out_handle) return fill_error(err, make_status(YTGPU_ERR_INVALID_ARGUMENT, "null argument"));
    CtxLock lock(h);
    Context* ctx = as_context(h);
    *out = nullptr;
    auto run = [&]() -> Status {
        if (world < 1 || world > kMaxRanks || rank < 0 || rank >= world)
            return make_status(YTGPU_ERR_INVALID_ARGUMENT, "world must be in [1, %d] and rank in [0, world)", kMaxRanks);
        if (row_bytes == 0 || row_bytes % 16) return make_status(YTGPU_ERR_INVALID_ARGUMENT, "row_bytes must be a positive multiple of 16");
        YTGPU_CUDA_TRY(cudaSetDevice(ctx->device));
        Shuffle* s = new (std::nothrow) Shuffle();
        if (!s) return make_status(YTGPU_ERR_OUT_OF_MEMORY, "host allocation failed");
        s->ctx = ctx;
        s->world = world;
        s->rank = rank;
        s->capacity_rows = capacity_rows;
        s->row_bytes = row_bytes;
        s->bytes = rows_offset(world) + capacity_rows * row_bytes + 256;
        cudaError_t e = cudaMalloc(&s->base, s->bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            delete s;
            return e == cudaErrorMemoryAllocation ? make_status(YTGPU_ERR_OUT_OF_MEMORY, "cudaMalloc(%zu bytes) for the receive buffer failed", s->bytes)
                                                  : cuda_status(e, "cudaMalloc");
        }
        auto fail = [&](Status stt) {
            cudaFree(s->base);
            if (s->pivots) cudaFree(s->pivots);
            if (s->cum) cudaFree(s->cum);
            if (s->host_stage) cudaFreeHost(s->host_stage);
            delete s;
            return stt;
        };
        if ((e = cudaMemset(s->base, 0, rows_offset(world))) != cudaSuccess) return fail(cuda_status(e, "cudaMemset"));
        if ((e = cudaMalloc(&s->pivots, sizeof(Pivots))) != cudaSuccess) return fail(cuda_status(e, "cudaMalloc"));
        if ((e = cudaMalloc(&s->cum, (size_t)world * kSamplesPerRank * 8)) != cudaSuccess) return fail(cuda_status(e, "cudaMalloc"));
        if ((e = cudaHostAlloc(&s->host_stage, kCtrlBytes + sizeof(Pivots), cudaHostAllocDefault)) != cudaSuccess)
            return fail(cuda_status(e, "cudaHostAlloc"));
        static_assert(sizeof(cudaIpcMemHandle_t) == YTGPU_IPC_HANDLE_BYTES, "IPC handle size");
        cudaIpcMemHandle_t ih;
        memset(&ih, 0, sizeof(ih));
        if (world > 1 && (e = cudaIpcGetMemHandle(&ih, s->base)) != cudaSuccess) return fail(cuda_status(e, "cudaIpcGetMemHandle"));
        memcpy(out_handle, &ih, sizeof(ih));
        s->peers.base[rank] = s->base;
        if (world == 1) s->connected = true;
        *out = reinterpret_cast<ytgpu_shuffle*>(s);
        return Status{};
    };
    return fill_error(err, run());
}

int ytgpu_shuffle_connect(ytgpu_shuffle* hs, const uint8_t* handles, ytgpu_error* err) {
    if (!hs || !handles) return fill_error(err, make_status(YTGPU_ERR_INVALID_ARGUMENT, "null argument"));
    Shuffle* s = reinterpret_cast<Shuffle*>(hs);
    std::unique_lock<std::mutex> lock(s->ctx->mu);
    auto run = [&]() -> Status {
        YTGPU_CUDA_TRY(cudaSetDevice(s->ctx->device));
        for (int q = 0; q < s->world; ++q) {
            if (q == s->rank || s->opened[q]) continue;
            cudaIpcMemHandle_t ih;
            memcpy(&ih, handles + (size_t)q * YTGPU_IPC_HANDLE_BYTES, sizeof(ih));
            void* p = nullptr;
            YTGPU_CUDA_TRY(cudaIpcOpenMemHandle(&p, ih, cudaIpcMemLazyEnablePeerAccess));
            s->peers.base[q] = static_cast<u8*>(p);
            s->opened[q] = true;
        }
        s->connected = true;
        return Status{};
    };
    return fill_error(err, run());
}

int ytgpu_shuffle_sort(ytgpu_shuffle* hs, const ytgpu_fixed_rows_view* in, const ytgpu_sort_spec* spec, uint8_t* out_rows,
                       uint64_t out_capacity_rows, uint64_t* out_row_count, ytgpu_shuffle_stats* stats, ytgpu_error* err) {
    if (!hs) return fill_error(err, make_status(YTGPU_ERR_INVALID_ARGUMENT, "null shuffle"));
    Shuffle* s = reinterpret_cast<Shuffle*>(hs);
    std::unique_lock<std::mutex> lock(s->ctx->mu);
    return fill_error(err, shuffle_sort_impl(s, in, spec, out_rows, out_capacity_rows, out_row_count, stats));
}

// CPU-test hook (tests/test_partition_keys.py): the SAME pivot-selection code the shuffle runs on the device, compiled
// for the host; keys are single 64-bit words here.
int ytgpu_hostcheck_partition_keys(const uint64_t* sorted_keys, const double* weights, uint32_t sample_count, int partition_count,
                                   uint32_t* out_sample, uint8_t* out_inclusive, uint8_t* out_maniac) {
    if (partition_count > kMaxRanks) return -1;
    std::vector<double> cum(sample_count);
    double run = 0;
    for (uint32_t i = 0; i < sample_count; ++i) cum[i] = (run += weights[i]);
    PartitionKeyPick picks[kMaxRanks];
    const int n = build_partition_keys_from_sorted_samples(sample_count, cum.data(),
                                                           [&](u32 a, u32 b) { return sorted_keys[a] == sorted_keys[b]; }, partition_count, picks);
    for (int i = 0; i < n; ++i) {
        out_sample[i] = picks[i].sample;
        out_inclusive[i] = picks[i].inclusive;
        out_maniac[i] = picks[i].maniac;
    }
    return n;
}

int ytgpu_shuffle_destroy(ytgpu_shuffle* hs, ytgpu_error* err) {
    if (!hs) return fill_error(err, Status{});
    Shuffle* s = reinterpret_cast<Shuffle*>(hs);
    std::unique_lock<std::mutex> lock(s->ctx->mu);
    auto run = [&]() -> Status {
        YTGPU_CUDA_TRY(cudaSetDevice(s->ctx->device));
        YTGPU_CUDA_TRY(cudaStreamSynchronize(s->ctx->stream));
        for (int q = 0; q < s->world; ++q)
            if (s->opened[q]) cudaIpcCloseMemHandle(s->peers.base[q]);
        cudaFree(s->base);
        cudaFree(s->pivots);
        cudaFree(s->cum);
        cudaFreeHost(s->host_stage);
        cudaGetLastError();
        return Status{};
    };
    Status r = run();
    lock.unlock();
    delete s;
    return fill_error(err, r);
}

}  // extern "C"
