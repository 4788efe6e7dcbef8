// radix_sort.cu — onesweep LSD radix sort core (see radix_sort.cuh).
//
// Replaces the comparison sorts of the reference's sort jobs:
//   std::sort over row pointers      yt/yt/ytlib/table_client/sorting_reader.cpp:179-187
//   10k-bucket std::sort + heap merge yt/yt/ytlib/table_client/partition_sort_reader.cpp:461-529
// with a stable radix sort over order-preserving normalised keys (keys.cuh).
#include <algorithm>
#include <vector>

#include "radix_sort.cuh"

namespace ytgpu {
namespace {

constexpr int kSortThreads = 256;  // one thread per digit bin in the tile's digit phase

constexpr u32 kFlagPartial = 1u << 30;
constexpr u32 kFlagInclusive = 2u << 30;
constexpr u32 kValueMask = (1u << 30) - 1;

// ---------------------------------------------------------------------------------------------
// Upfront histogram of all 8 digits of one key chunk.  Algorithmic traffic: 8 B per row (read).
// Warp-uniform digits (constant high bytes, duplicated keys) are detected with one REDUX per half
// word and counted with a single shared-memory add per warp instead of 32 same-address atomics.
// ---------------------------------------------------------------------------------------------
constexpr int kHistThreads = 512;
constexpr int kHistItems = 4;

__global__ void __launch_bounds__(kHistThreads) histogram_kernel(const u64* __restrict__ keys, u64 n,
                                                                 u32* __restrict__ hist) {
    __shared__ u32 sh[kPassesPerChunk * kRadix];
    for (int i = threadIdx.x; i < kPassesPerChunk * kRadix; i += kHistThreads) sh[i] = 0;
    __syncthreads();

    const u64 stride = (u64)gridDim.x * kHistThreads * kHistItems;
    for (u64 base = (u64)blockIdx.x * kHistThreads * kHistItems; base < n; base += stride) {
        u64 key[kHistItems];
        bool valid[kHistItems];
#pragma unroll
        for (int k = 0; k < kHistItems; ++k) {
            u64 i = base + (u64)k * kHistThreads + threadIdx.x;
            valid[k] = i < n;
            key[k] = valid[k] ? ld_stream_u64(keys + i) : 0;
        }
#pragma unroll
        for (int k = 0; k < kHistItems; ++k) hist_accumulate(sh, key[k], valid[k]);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kPassesPerChunk * kRadix; i += kHistThreads) {
        u32 c = sh[i];
        if (c) atomicAdd(&hist[i], c);
    }
}

// ---------------------------------------------------------------------------------------------
// Plan: turns counts into exclusive digit offsets, finds skippable digits, and fixes the buffer
// ping-pong schedule for every (chunk, digit) pass.  One block of 256 threads.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 block_exclusive_scan_256(u32 v, u32* s_warp_tot) {
    const u32 lane = lane_id(), warp = threadIdx.x >> 5;
    u32 inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u32 t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (u32)o) inc += t;
    }
    if (lane == 31) s_warp_tot[warp] = inc;
    __syncthreads();
    u32 wp = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) wp += (w < (int)warp) ? s_warp_tot[w] : 0;
    __syncthreads();
    return inc - v + wp;
}

// Builds the ping-pong schedule over the passes listed in `sel` (execution order).  Returns the final
// permutation buffer (2 = identity) and reports the final key buffer and the last scheduled pass.
__device__ void build_schedule(PassDesc* descs, const int* sel, int nsel, bool mark_last, u32* final_idx, u32* final_key) {
    u32 cur_idx = 2, cur_key = 2;
    int last = -1;
    for (int k = 0; k < nsel; ++k) {
        PassDesc d{};
        d.active = 1;
        d.src_kind = cur_key == 2 ? (cur_idx == 2 ? 0 : 1) : 2;
        d.key_src = (u8)(cur_key & 1);
        d.idx_src = (u8)(cur_idx & 1);
        d.key_dst = cur_key == 2 ? 0 : (u8)(cur_key ^ 1);
        d.idx_dst = cur_idx == 2 ? 0 : (u8)(cur_idx ^ 1);
        cur_key = d.key_dst;
        cur_idx = d.idx_dst;
        descs[sel[k]] = d;
        last = sel[k];
    }
    if (mark_last && last >= 0) descs[last].last = 1;  // only the permutation is consumed: skip the key write
    *final_idx = cur_idx;
    *final_key = cur_key;
}

__global__ void __launch_bounds__(256) plan_kernel(u32* hist, int nchunks, u32 n, SortPlan* plan, int allow_hybrid, int keep_keys) {
    __shared__ u32 s_warp_tot[8];
    __shared__ u8 s_active[kMaxKeyChunks * kPassesPerChunk];
    const int total = nchunks * kPassesPerChunk;
    for (int rp = 0; rp < total; ++rp) {
        u32 c = hist[rp * kRadix + threadIdx.x];
        int full = __syncthreads_or(c == n);
        u32 ex = block_exclusive_scan_256(c, s_warp_tot);
        hist[rp * kRadix + threadIdx.x] = ex;
        if (threadIdx.x == 0) s_active[rp] = !full;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    for (int rp = 0; rp < total; ++rp) plan->pass[rp] = PassDesc{};
    for (int p = 0; p < kPassesPerChunk; ++p) plan->pass_b[p] = PassDesc{};
    plan->hybrid = plan->fallback = plan->hybrid_shift = plan->final_key_a = 0;
    plan->final_idx_b = 2;
    plan->active_passes_b = 0;
    plan->final_key = plan->final_key_b = 2;
    u32 final_key = 2;
    if (nchunks == 1) {
        int act[kPassesPerChunk], m = 0;
        for (int p = 0; p < kPassesPerChunk; ++p)
            if (s_active[p]) act[m++] = p;
        // Hybrid: sort by the `need` most significant active digits only, where 256^need >= 16 n keeps the
        // expected share of rows in runs of equal prefixes small; worth it when it saves >= 2 passes.
        int need = 1;
        unsigned long long span = 256;
        while (span < 16ull * n && need < kPassesPerChunk) { span <<= 8; ++need; }
        if (allow_hybrid && m >= need + 2) {
            build_schedule(plan->pass, act + (m - need), need, false, &plan->final_idx, &final_key);
            build_schedule(plan->pass_b, act, m, !keep_keys, &plan->final_idx_b, &plan->final_key_b);
            plan->hybrid = 1;
            plan->hybrid_shift = 8u * (u32)act[m - need];
            plan->final_key_a = plan->pass[act[m - 1]].key_dst;
            plan->active_passes = (u32)need;
            plan->active_passes_b = (u32)m;
        } else {
            build_schedule(plan->pass, act, m, !keep_keys, &plan->final_idx, &plan->final_key);
            plan->active_passes = (u32)m;
        }
        return;
    }
    // multi-chunk keys: chunks from least to most significant, eight digits each, one continuous ping-pong
    u32 cur_idx = 2, active = 0;
    int last_rp = -1;
    for (int r = nchunks - 1; r >= 0; --r) {
        u32 cur_key = 2;  // the chunk itself
        for (int p = 0; p < kPassesPerChunk; ++p) {
            int rp = r * kPassesPerChunk + p;
            if (!s_active[rp]) continue;
            PassDesc d{};
            d.active = 1;
            d.src_kind = cur_key == 2 ? (cur_idx == 2 ? 0 : 1) : 2;
            d.key_src = (u8)(cur_key & 1);
            d.idx_src = (u8)(cur_idx & 1);
            d.key_dst = cur_key == 2 ? 0 : (u8)(cur_key ^ 1);
            d.idx_dst = cur_idx == 2 ? 0 : (u8)(cur_idx ^ 1);
            cur_key = d.key_dst;
            cur_idx = d.idx_dst;
            ++active;
            last_rp = rp;
            plan->pass[rp] = d;
        }
    }
    if (last_rp >= 0) plan->pass[last_rp].last = 1;
    plan->final_idx = cur_idx;
    plan->active_passes = active;
}

// After the hybrid passes the (key, index) pairs are ordered by the top digits and, inside a run of equal
// top digits, still in input order.  tie_fix_kernel:
//   * runs of <= kMaxTieRun equal prefixes: the run-start thread orders them by the full key (stable insertion sort;
//     runs are 2-3 rows long when the keys spread over the prefix space);
//   * longer runs are only REGISTERED (the element 32 places into the run appends the run's start to a list), and
//     every warp stores which of its 32 positions hold "same prefix as the left neighbour, different key" — a long run of
//     EQUAL keys (duplicates, "maniac" keys) has no such position and is already in its final stable order.
// classify_long_runs_kernel then finds each long run's end and looks for a marked position inside it: runs that mix
// different keys go to the mixed list.  The host reads the summary once and either is done, re-sorts the few mixed runs
// in a side buffer (sort_mixed_runs), or — clustered keys: many / very long mixed runs — runs the complete LSD schedule.
constexpr int kMaxTieRun = 32;
constexpr u32 kMixedCap = 16384;       // mixed long runs handled individually; more = clustered keys = complete schedule
constexpr u64 kHybridMinRows = 1u << 18;  // smaller sorts are launch bound: plain schedule, no host round trip

struct MixedRun {
    u32 s, e;
};
struct HybridSummary {
    u32 hybrid, final_idx, final_key;
    u32 long_count, mixed_count;
    unsigned long long mixed_elems;
};

__global__ void __launch_bounds__(256) tie_fix_kernel(SortPlan* plan, u64* keys0, u64* keys1, u32* idx0, u32* idx1, u32 n,
                                                      u32* __restrict__ mixedmask, u32* __restrict__ longlist, HybridSummary* sum) {
    if (!plan->hybrid) return;
    u64* keys = plan->final_key_a ? keys1 : keys0;
    u32* idx = plan->final_idx ? idx1 : idx0;
    const u32 shift = plan->hybrid_shift;
    const u32 lane = threadIdx.x & 31;
    for (u64 base = (u64)blockIdx.x * blockDim.x; base < n; base += (u64)gridDim.x * blockDim.x) {  // warp-uniform trips
        const u64 i64 = base + threadIdx.x;
        const bool in = i64 < n;
        const u32 i = (u32)i64;
        const u64 key = in ? keys[i] : 0;
        const u64 pref = key >> shift;
        // neighbours through shuffles; only the edge lanes touch memory again
        u64 pkey = __shfl_up_sync(0xffffffffu, key, 1);
        u64 next = __shfl_down_sync(0xffffffffu, pref, 1);
        if (in && lane == 0) pkey = i > 0 ? keys[i - 1] : ~key;
        if (in && (lane == 31 || i + 1 >= n)) next = i + 1 < n ? (keys[i + 1] >> shift) : ~pref;
        const bool same_prev = in && i > 0 && (pkey >> shift) == pref;
        // (a short run may be permuted concurrently by its start thread: harmless, only long runs consult the mask)
        const u32 mixed = __ballot_sync(0xffffffffu, same_prev && pkey != key);
        if (lane == 0 && in) mixedmask[i >> 5] = mixed;  // base is a multiple of 32: one word per warp trip
        if (!in) continue;
        if (same_prev) {
            // the element kMaxTieRun places into a run registers it as long
            if (i >= (u32)kMaxTieRun && (keys[i - kMaxTieRun] >> shift) == pref &&
                (i == (u32)kMaxTieRun || (keys[i - kMaxTieRun - 1] >> shift) != pref))
                longlist[atomicAdd(&sum->long_count, 1u)] = i - kMaxTieRun;  // at most n / 33 entries
            continue;
        }
        if (next != pref) continue;  // run of one
        u32 len = 2;
        while (i + len < n && len <= (u32)kMaxTieRun && (keys[i + len] >> shift) == pref) ++len;
        if (len > (u32)kMaxTieRun) continue;  // long run: registered by its 33rd element
        for (u32 a = 1; a < len; ++a) {  // stable insertion sort by the full key
            const u64 k = keys[i + a];
            const u32 v = idx[i + a];
            u32 b = a;
            while (b > 0 && keys[i + b - 1] > k) {
                keys[i + b] = keys[i + b - 1];
                idx[i + b] = idx[i + b - 1];
                --b;
            }
            keys[i + b] = k;
            idx[i + b] = v;
        }
    }
}

// One warp per registered long run: find its end (gallop + binary search over the prefix-sorted keys), then look for
// a "different key than the left neighbour" mark inside it.
__global__ void __launch_bounds__(256) classify_long_runs_kernel(const SortPlan* plan, const u64* keys0, const u64* keys1, u32 n,
                                                                 const u32* __restrict__ mixedmask, const u32* __restrict__ longlist,
                                                                 HybridSummary* sum, MixedRun* __restrict__ mixedlist) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        sum->hybrid = plan->hybrid;
        sum->final_idx = plan->final_idx;
        sum->final_key = plan->final_key_a;
    }
    if (!plan->hybrid) return;
    const u64* keys = plan->final_key_a ? keys1 : keys0;
    const u32 shift = plan->hybrid_shift;
    const u32 lane = threadIdx.x & 31;
    const u32 count = sum->long_count;
    const u32 warps = gridDim.x * (blockDim.x >> 5);
    for (u32 r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < count; r += warps) {
        const u32 s = longlist[r];
        // end of the run, searched by the whole warp: lane l probes s + (32 << l) (exponential), then the bracket is cut
        // 32 ways per round — 2-4 rounds of parallel loads instead of ~2 log2(length) dependent ones
        const u64 pref = keys[s] >> shift;
        u64 lo, hi;
        {
            const u64 pos = (u64)s + ((u64)kMaxTieRun << lane);
            const bool diff = pos >= n || (keys[pos] >> shift) != pref;  // lane 0 probes s + 32: same prefix by construction
            const int first = __ffs(__ballot_sync(0xffffffffu, diff)) - 1;  // >= 1; lane 31 is always past the end (n < 2^30)
            lo = (u64)s + ((u64)kMaxTieRun << (first - 1));
            hi = min((u64)n, (u64)s + ((u64)kMaxTieRun << first));
        }
        while (hi - lo > 1) {  // prefix(lo) == pref; hi == n or prefix(hi) != pref
            const u64 len = hi - lo;
            const u64 pos = lo + ((len * (lane + 1)) >> 5);
            const bool diff = pos >= hi || (keys[pos] >> shift) != pref;
            const int first = __ffs(__ballot_sync(0xffffffffu, diff)) - 1;  // lane 31 probes hi: always set
            const u64 new_hi = __shfl_sync(0xffffffffu, pos, first);
            const u64 new_lo = first > 0 ? __shfl_sync(0xffffffffu, pos, first - 1) : lo;
            hi = new_hi;
            lo = new_lo;
        }
        const u32 e = (u32)hi;
        // marks at positions s+1 .. e-1
        const u32 fw = (s + 1) >> 5, lw = (e - 1) >> 5;
        bool any = false;
        for (u32 w = fw + lane; w <= lw; w += 32) {
            u32 m = mixedmask[w];
            if (w == fw) m &= 0xffffffffu << ((s + 1) & 31);
            if (w == lw && ((e & 31) != 0)) m &= (1u << (e & 31)) - 1;
            any |= m != 0;
        }
        if (__any_sync(0xffffffffu, any) && lane == 0) {
            const u32 slot = atomicAdd(&sum->mixed_count, 1u);
            if (slot < kMixedCap) mixedlist[slot] = MixedRun{s, e};
            atomicAdd(&sum->mixed_elems, (unsigned long long)(e - s));
        }
    }
}

// Side buffer of the mixed long runs (in run order == key order == position order), and the way back.
__global__ void __launch_bounds__(256) expand_mixed_runs_kernel(const u64* __restrict__ keys, const u32* __restrict__ idx, const u32* __restrict__ rs,
                                                                const u32* __restrict__ re, const u32* __restrict__ roff, u32 nruns,
                                                                u64* __restrict__ side_key, u32* __restrict__ side_idx, u32* __restrict__ side_pos) {
    for (u32 r = blockIdx.x; r < nruns; r += gridDim.x) {
        const u32 s = rs[r], len = re[r] - s, off = roff[r];
        for (u32 j = threadIdx.x; j < len; j += blockDim.x) {
            side_key[off + j] = keys[s + j];
            side_idx[off + j] = idx[s + j];
            side_pos[off + j] = s + j;
        }
    }
}
__global__ void __launch_bounds__(256) writeback_mixed_runs_kernel(const SortPlan* splan, const u32* sa, const u32* sb, u32 m,
                                                                   const u64* __restrict__ side_key, const u32* __restrict__ side_idx,
                                                                   const u32* __restrict__ side_pos, u64* __restrict__ keys, u32* __restrict__ idx) {
    for (u32 k = blockIdx.x * blockDim.x + threadIdx.x; k < m; k += gridDim.x * blockDim.x) {
        const u32 src = perm_at(splan, sa, sb, k);  // k-th smallest side element goes to the k-th marked position
        const u32 pos = side_pos[k];
        keys[pos] = side_key[src];
        idx[pos] = side_idx[src];
    }
}

// ---------------------------------------------------------------------------------------------
// One digit pass.  Per row: read 8 B key + 4 B index, write 8 B key + 4 B index.
// ---------------------------------------------------------------------------------------------
struct PassParams {
    const u64* chunk;
    u64* keys[2];
    u32* idx[2];
    const u32* digit_base;  // exclusive offsets of this pass's 256 digits
    u32* status;            // [tiles][256] look-back words, zeroed
    u32* counter;           // dynamic tile id, zeroed
    const SortPlan* plan;
    int plan_index;
    int schedule;  // 0: plan->pass[plan_index]; 1: plan->pass_b[plan_index], launched only after plan->fallback is set
    int shift;
    u32 n;
};

template <int THREADS, int ITEMS, bool FULL>
__device__ __forceinline__ void onesweep_tile(const PassParams& P, const PassDesc pd, const u32 tile, unsigned char* smem_raw) {
    constexpr int WARPS = THREADS / 32;
    constexpr int TILE = THREADS * ITEMS;
    u64* s_keys = reinterpret_cast<u64*>(smem_raw);                      // TILE keys
    u32* s_vals = reinterpret_cast<u32*>(smem_raw + (size_t)TILE * 8);   // TILE row indices
    u32* s_hist = reinterpret_cast<u32*>(smem_raw + (size_t)TILE * 12);  // [WARPS][256]
    u32* s_excl = s_hist + WARPS * kRadix;                      // [256]
    u32* s_gbase = s_excl + kRadix;                             // [256]
    u32* s_misc = s_gbase + kRadix;                             // [0..7] warp totals, [8] tile id

    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u32 base = tile * (u32)TILE;
    const u32 tile_count = FULL ? (u32)TILE : P.n - base;

    const u64* kin = pd.src_kind == 2 ? (pd.key_src ? P.keys[1] : P.keys[0]) : P.chunk;
    const u32* iin = pd.idx_src ? P.idx[1] : P.idx[0];
    u64* kout = pd.key_dst ? P.keys[1] : P.keys[0];
    u32* iout = pd.idx_dst ? P.idx[1] : P.idx[0];
    const int shift = P.shift;

    // The row indices of this tile are needed only after ranking: pull their lines into L2 now so the
    // later loads do not expose DRAM latency (one 128-byte line per thread).
    if (pd.src_kind == 2) {
        const char* ibase = reinterpret_cast<const char*>(iin + base);
        const u32 ibytes = tile_count * 4;
        for (u32 off = tid * 128; off < ibytes; off += THREADS * 128)
            asm volatile("prefetch.global.L2 [%0];" :: "l"(ibase + off));
    }

    // ---- load keys, warp-striped: item i of lane l sits at warp_base + i*32 + l ----
    const u32 wbase = base + warp * (32 * ITEMS) + lane;
    u64 key[ITEMS];
    if (pd.src_kind == 1) {
        u32 src[ITEMS];
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) {
            u32 pos = wbase + i * 32;
            src[i] = (FULL || pos < P.n) ? ld_stream_u32(iin + pos) : 0u;
        }
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) {
            u32 pos = wbase + i * 32;
            key[i] = (FULL || pos < P.n) ? kin[src[i]] : ~0ull;
        }
    } else {
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) {
            u32 pos = wbase + i * 32;
            key[i] = (FULL || pos < P.n) ? ld_stream_u64(kin + pos) : ~0ull;
        }
    }

    // ---- rank inside the warp: stable (item-major, then lane) ----
    // Peers with the same digit are found with 8 ballots (one per digit bit).  MATCH.ANY is NOT used:
    // on B200 it costs ~2 SM-cycles per distinct value in the warp (~59 cycles for random 8-bit
    // digits, scratch/match_bench.cu), the 8 ballots cost ~25.  The running per-digit counts of the
    // warp live in its private shared histogram: every lane reads its bin (same-digit lanes broadcast),
    // the lowest lane of each digit group writes the bumped count back.
    u32 rank[ITEMS];
    u32* wh = s_hist + warp * kRadix;
    const u32 lt = lanemask_lt();
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
        const u32 d = (u32)(key[i] >> shift) & 0xff;
        u32 m = 0xffffffffu;
#pragma unroll
        for (int b = 0; b < kRadixBits; ++b) {
            const bool bit = (d >> b) & 1;
            const u32 v = __ballot_sync(0xffffffffu, bit);
            m &= bit ? v : ~v;
        }
        bool valid = true;
        if (!FULL) {
            valid = wbase + i * 32 < P.n;
            m &= __ballot_sync(0xffffffffu, valid);
        }
        const u32 prev = wh[d];
        __syncwarp();
        if (valid && (m & lt) == 0) wh[d] = prev + __popc(m);
        rank[i] = prev + __popc(m & lt);
        __syncwarp();
    }
    __syncthreads();

    // ---- per digit (thread d): offsets of each warp inside the digit, tile count, publish ----
    u32 cnt = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) cnt += s_hist[w * kRadix + tid];
    u32* my_status = P.status + (size_t)tile * kRadix + tid;
    st_volatile_u32(my_status, (tile == 0 ? kFlagInclusive : kFlagPartial) | cnt);
    const u32 local_excl = block_exclusive_scan_256(cnt, s_misc);
    {
        // s_hist[w][d] := position in the tile-sorted order of the first key of warp w with digit d
        u32 run = local_excl;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) {
            u32 c = s_hist[w * kRadix + tid];
            s_hist[w * kRadix + tid] = run;
            run += c;
        }
    }
    __syncthreads();

    // ---- decoupled look-back, software-pipelined with the shared-memory scatter below ----
    // Thread `tid` owns the chain of digit `tid`.  Tiles reach this point every few dozen cycles but a
    // status word costs an L2 round trip, so a tile typically has to add the partial counts of ~10
    // predecessors.  Instead of spinning, one status load is kept in flight while the keys and row
    // indices are scattered into shared memory; whatever is left is finished by the loop after them.
    u32 lb_excl = 0;
    i32 lb_tile = (i32)tile - 1;
    bool lb_done = tile == 0;
    u32 lb_word = 0;
    auto lb_issue = [&]() {
        if (!lb_done) lb_word = ld_volatile_u32(P.status + (size_t)lb_tile * kRadix + tid);
    };
    auto lb_consume = [&]() {
        if (!lb_done) {
            const u32 f = lb_word >> 30;
            if (f != 0) {
                lb_excl += lb_word & kValueMask;
                if (f == 2) lb_done = true;
                else --lb_tile;
            }
        }
    };

    // ---- keys and row indices -> shared memory in tile-sorted order ----
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
        if ((i & 3) == 0) lb_issue();
        const u32 d = (u32)(key[i] >> shift) & 0xff;
        const u32 lp = wh[d] + rank[i];
        rank[i] = lp;
        if (FULL || (wbase + i * 32 < P.n)) s_keys[lp] = key[i];
        if ((i & 3) == 3) lb_consume();
    }
    if (pd.src_kind == 0) {
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) {
            if ((i & 3) == 0) lb_issue();
            const u32 pos = wbase + i * 32;
            if (FULL || pos < P.n) s_vals[rank[i]] = pos;
            if ((i & 3) == 3) lb_consume();
        }
    } else {
        constexpr int VB = 4;
#pragma unroll
        for (int b0 = 0; b0 < ITEMS; b0 += VB) {
            lb_issue();
            u32 v[VB];
#pragma unroll
            for (int i = 0; i < VB; ++i) {
                const u32 pos = wbase + (b0 + i) * 32;
                v[i] = (FULL || pos < P.n) ? ld_stream_u32(iin + pos) : 0u;
            }
#pragma unroll
            for (int i = 0; i < VB; ++i) {
                const u32 pos = wbase + (b0 + i) * 32;
                if (FULL || pos < P.n) s_vals[rank[b0 + i]] = v[i];
            }
            lb_consume();
        }
    }
    while (!lb_done) {
        lb_issue();
        lb_consume();
    }
    if (tile > 0) st_volatile_u32(my_status, kFlagInclusive | ((lb_excl + cnt) & kValueMask));
    s_gbase[tid] = P.digit_base[tid] + lb_excl - local_excl;
    __syncthreads();

    // ---- write out: consecutive threads -> consecutive shared slots -> runs of one digit ----
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        const u32 j = tid + k * THREADS;
        if (FULL || j < tile_count) {
            const u64 kk = s_keys[j];
            const u32 g = s_gbase[(u32)(kk >> shift) & 0xff] + j;
            if (!pd.last) kout[g] = kk;
            iout[g] = s_vals[j];
        }
    }
}

template <int THREADS, int ITEMS, int MINB>
__global__ void __launch_bounds__(THREADS, MINB) onesweep_pass_kernel(const PassParams P) {
    constexpr int WARPS = THREADS / 32;
    constexpr int TILE = THREADS * ITEMS;
    static_assert(THREADS == 256, "digit phase assumes one thread per bin");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    u32* s_hist = reinterpret_cast<u32*>(smem_raw + (size_t)TILE * 12);
    u32* s_misc = s_hist + WARPS * kRadix + 2 * kRadix;

    const PassDesc pd = P.schedule == 1 ? P.plan->pass_b[P.plan_index] : P.plan->pass[P.plan_index];
    if (!pd.active) return;
    // One tile per CTA.  (A persistent variant — 3 CTAs per SM looping over an atomic tile counter — measured 8 %
    // slower on the active passes: 6.51 vs 5.96 ms for 8 passes over 10^8 rows; hardware CTA launch is cheaper
    // than the extra barrier per tile.)  Tile ids still come from the atomic counter so that they are handed
    // out in start order, which the decoupled look-back relies on.
    const u32 tiles = (u32)(((u64)P.n + TILE - 1) / TILE);
    if (threadIdx.x == 0) s_misc[8] = atomicAdd(P.counter, 1u);
#pragma unroll
    for (int i = threadIdx.x; i < WARPS * kRadix; i += THREADS) s_hist[i] = 0;
    __syncthreads();
    const u32 tile = s_misc[8];
    if (tile >= tiles) return;
    if ((u64)(tile + 1) * TILE <= (u64)P.n) onesweep_tile<THREADS, ITEMS, true>(P, pd, tile, smem_raw);
    else onesweep_tile<THREADS, ITEMS, false>(P, pd, tile, smem_raw);
}

__global__ void materialize_perm_kernel(const SortPlan* plan, const u32* a, const u32* b, u64 n, u32* dst) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        dst[i] = perm_at(plan, a, b, i);
}

constexpr size_t pass_smem_bytes(int items) {
    return (size_t)kSortThreads * items * 12 + (size_t)(kSortThreads / 32) * kRadix * 4 + 2 * kRadix * 4 + 16 * 4;
}

// 16 items per thread at 3 resident CTAs per SM measured best on B200 (DESIGN.md §4).
constexpr int kSortItems = 16;
constexpr int kSortCtasPerSm = 3;

void prepare_pass_kernel(Context* ctx) {
    if (!(ctx->func_attrs_done & FA_SORT_PASS)) {  // per device (the attribute belongs to the current device's function)
        cudaFuncSetAttribute(onesweep_pass_kernel<kSortThreads, kSortItems, kSortCtasPerSm>,
                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pass_smem_bytes(kSortItems));
        ctx->func_attrs_done |= FA_SORT_PASS;
    }
}

// Allocates and fills s->hist with the raw digit counts of every chunk.
Status histogram_chunks(Context* ctx, const u64* const* chunks, int nchunks, u64 n, SortScratch* s) {
    YTGPU_TRY(prepare_histogram(ctx, nchunks, s));
    KernelTimer t(ctx, KC_HISTOGRAM, nchunks);
    const u64 per_block = (u64)kHistThreads * kHistItems;
    const u32 blocks = (u32)std::min<u64>((n + per_block - 1) / per_block, (u64)kNumSms * 4);
    for (int c = 0; c < nchunks; ++c)
        histogram_kernel<<<blocks, kHistThreads, 0, ctx->stream>>>(chunks[c], n, s->hist.p + (size_t)c * kPassesPerChunk * kRadix);
    return Status{};
}

}  // namespace

// Stable re-sort of the few long runs of equal prefixes that mix different keys: their (key, index) pairs are copied
// to a side buffer in run order, sorted by the full key with the plain schedule, and written back — the k-th smallest
// side element belongs at the k-th marked position because runs are ordered by prefix, i.e. by key.
static Status sort_mixed_runs(Context* ctx, SortScratch* s, const HybridSummary& hs, const MixedRun* mixedlist_dev) {
    cudaStream_t st = ctx->stream;
    const u32 w = hs.mixed_count;
    std::vector<MixedRun> runs(w);
    YTGPU_CUDA_TRY(cudaMemcpyAsync(runs.data(), mixedlist_dev, (size_t)w * sizeof(MixedRun), cudaMemcpyDeviceToHost, st));
    YTGPU_CUDA_TRY(cudaStreamSynchronize(st));
    std::sort(runs.begin(), runs.end(), [](const MixedRun& a, const MixedRun& b) { return a.s < b.s; });
    std::vector<u32> host(3 * (size_t)w);
    u32 total = 0;
    for (u32 r = 0; r < w; ++r) {
        host[r] = runs[r].s;
        host[w + r] = runs[r].e;
        host[2 * (size_t)w + r] = total;
        total += runs[r].e - runs[r].s;
    }
    DevBuf<u32> meta, side_idx, side_pos;
    DevBuf<u64> side_key;
    YTGPU_TRY(meta.allocate(ctx, 3 * (size_t)w));
    YTGPU_TRY(side_key.allocate(ctx, total));
    YTGPU_TRY(side_idx.allocate(ctx, total));
    YTGPU_TRY(side_pos.allocate(ctx, total));
    YTGPU_CUDA_TRY(cudaMemcpyAsync(meta.p, host.data(), host.size() * 4, cudaMemcpyHostToDevice, st));
    u64* keys = hs.final_key ? s->keys[1].p : s->keys[0].p;
    u32* idx = hs.final_idx ? s->idx[1].p : s->idx[0].p;
    expand_mixed_runs_kernel<<<std::min<u32>(w, (u32)kNumSms * 8), 256, 0, st>>>(keys, idx, meta.p, meta.p + w, meta.p + 2 * (size_t)w, w, side_key.p,
                                                                              side_idx.p, side_pos.p);
    ctx->count_launch();
    SortScratch side;
    side.no_hybrid = true;
    PermRef sperm;
    const u64* sptr[1] = {side_key.p};
    YTGPU_TRY(radix_sort_chunks(ctx, sptr, 1, total, &side, &sperm));
    writeback_mixed_runs_kernel<<<(u32)std::min<u64>(((u64)total + 255) / 256, (u64)kNumSms * 8), 256, 0, st>>>(sperm.plan, sperm.idx[0], sperm.idx[1],
                                                                                                              total, side_key.p, side_idx.p,
                                                                                                              side_pos.p, keys, idx);
    ctx->count_launch();
    YTGPU_CUDA_TRY(cudaGetLastError());
    YTGPU_CUDA_TRY(cudaStreamSynchronize(st));  // `host` / `runs` back the asynchronous upload
    return Status{};
}

Status radix_sort_chunks(Context* ctx, const u64* const* chunks, int nchunks, u64 n, SortScratch* s,
                         PermRef* out) {
    if (nchunks < 1 || nchunks > kMaxKeyChunks)
        return make_status(YTGPU_ERR_UNSUPPORTED, "normalised key of %d bytes exceeds the %d-byte limit",
                           nchunks * 8, kMaxKeyChunks * 8);
    if (n >= (1ull << 30))
        return make_status(YTGPU_ERR_UNSUPPORTED, "row count %llu exceeds 2^30-1 rows per sort call",
                           (unsigned long long)n);
    cudaStream_t st = ctx->stream;
    YTGPU_CUDA_TRY(cudaSetDevice(ctx->device));
    prepare_pass_kernel(ctx);
    const u32 tile_rows = (u32)kSortThreads * kSortItems;
    const u32 tiles = (u32)((n + tile_rows - 1) / tile_rows);
    const int total_passes = nchunks * kPassesPerChunk;

    YTGPU_TRY(s->keys[0].allocate(ctx, n));
    YTGPU_TRY(s->keys[1].allocate(ctx, n));
    YTGPU_TRY(s->idx[0].allocate(ctx, n));
    YTGPU_TRY(s->idx[1].allocate(ctx, n));
    if (!s->hist_precomputed) YTGPU_TRY(histogram_chunks(ctx, chunks, nchunks, n, s));
    YTGPU_TRY(s->status.allocate(ctx, (size_t)kPassesPerChunk * tiles * kRadix));
    YTGPU_TRY(s->counters.allocate(ctx, (size_t)total_passes + kPassesPerChunk));
    YTGPU_TRY(s->plan.allocate(ctx, 1));

    YTGPU_CUDA_TRY(cudaMemsetAsync(s->counters.p, 0, ((size_t)total_passes + kPassesPerChunk) * 4, st));
    const int allow_hybrid = ctx->opt_sort_hybrid && !s->no_hybrid && n >= kHybridMinRows;
    plan_kernel<<<1, 256, 0, st>>>(s->hist.p, nchunks, (u32)n, s->plan.p, allow_hybrid, s->keep_keys ? 1 : 0);
    ctx->count_launch();

    // Digit p of chunk r, from the plan's main schedule (0) or its complete fallback schedule (1, single chunk only).
    auto launch_pass = [&](int r, int p, int schedule) {
        KernelTimer t(ctx, KC_RADIX_PASS);
        PassParams P;
        P.chunk = chunks[r];
        P.keys[0] = s->keys[0].p;
        P.keys[1] = s->keys[1].p;
        P.idx[0] = s->idx[0].p;
        P.idx[1] = s->idx[1].p;
        P.digit_base = s->hist.p + (size_t)(r * kPassesPerChunk + p) * kRadix;
        P.status = s->status.p + (size_t)p * tiles * kRadix;
        P.counter = s->counters.p + (schedule * total_passes + r * kPassesPerChunk + p);
        P.plan = s->plan.p;
        P.plan_index = r * kPassesPerChunk + p;
        P.schedule = schedule;
        P.shift = p * kRadixBits;
        P.n = (u32)n;
        onesweep_pass_kernel<kSortThreads, kSortItems, kSortCtasPerSm><<<tiles, kSortThreads, pass_smem_bytes(kSortItems), st>>>(P);
    };
    for (int r = nchunks - 1; r >= 0; --r) {
        YTGPU_CUDA_TRY(cudaMemsetAsync(s->status.p, 0, (size_t)kPassesPerChunk * tiles * kRadix * 4, st));
        for (int p = 0; p < kPassesPerChunk; ++p) launch_pass(r, p, 0);
    }
    if (nchunks == 1 && allow_hybrid) {
        // hybrid tail: order the short runs of equal prefixes, classify the long ones
        DevBuf<u32> mixedmask, longlist;
        DevBuf<HybridSummary> summary;
        DevBuf<MixedRun> mixedlist;
        YTGPU_TRY(mixedmask.allocate(ctx, n / 32 + 2));
        YTGPU_TRY(longlist.allocate(ctx, n / 32 + 2));
        YTGPU_TRY(summary.allocate(ctx, 1));
        YTGPU_TRY(mixedlist.allocate(ctx, kMixedCap));
        YTGPU_CUDA_TRY(cudaMemsetAsync(summary.p, 0, sizeof(HybridSummary), st));
        {
            KernelTimer t(ctx, KC_HISTOGRAM, 2);
            const u32 blocks = (u32)std::min<u64>((n + 255) / 256, (u64)kNumSms * 8);
            tie_fix_kernel<<<blocks, 256, 0, st>>>(s->plan.p, s->keys[0].p, s->keys[1].p, s->idx[0].p, s->idx[1].p, (u32)n, mixedmask.p,
                                                   longlist.p, summary.p);
            classify_long_runs_kernel<<<kNumSms * 4, 256, 0, st>>>(s->plan.p, s->keys[0].p, s->keys[1].p, (u32)n, mixedmask.p, longlist.p,
                                                                   summary.p, mixedlist.p);
        }
        YTGPU_CUDA_TRY(cudaGetLastError());
        // the sort's one host round trip (sorts below kHybridMinRows rows never take the hybrid schedule)
        HybridSummary hs{};
        YTGPU_CUDA_TRY(cudaMemcpyAsync(&hs, summary.p, sizeof(hs), cudaMemcpyDeviceToHost, st));
        YTGPU_CUDA_TRY(cudaStreamSynchronize(st));
        if (hs.hybrid && hs.mixed_count > 0) {
            if (hs.mixed_count > kMixedCap || hs.mixed_elems > n / 8) {
                // clustered keys: the complete LSD schedule (pass_b) from the chunk
                const u32 one = 1;
                YTGPU_CUDA_TRY(cudaMemcpyAsync(&s->plan.p->fallback, &one, 4, cudaMemcpyHostToDevice, st));
                YTGPU_CUDA_TRY(cudaMemsetAsync(s->status.p, 0, (size_t)kPassesPerChunk * tiles * kRadix * 4, st));
                for (int p = 0; p < kPassesPerChunk; ++p) launch_pass(0, p, 1);
                YTGPU_CUDA_TRY(cudaStreamSynchronize(st));  // `one` lives on this stack frame
            } else {
                YTGPU_TRY(sort_mixed_runs(ctx, s, hs, mixedlist.p));
            }
        }
    }
    YTGPU_CUDA_TRY(cudaGetLastError());
    YTGPU_CUDA_TRY(cudaMemcpyAsync(ctx->host_err + 1, &s->plan.p->active_passes, 4, cudaMemcpyDeviceToHost, st));
    YTGPU_CUDA_TRY(cudaMemcpyAsync(ctx->host_err + 2, &s->plan.p->active_passes_b, 4, cudaMemcpyDeviceToHost, st));
    YTGPU_CUDA_TRY(cudaMemcpyAsync(ctx->host_err + 3, &s->plan.p->fallback, 4, cudaMemcpyDeviceToHost, st));
    out->plan = s->plan.p;
    out->idx[0] = s->idx[0].p;
    out->idx[1] = s->idx[1].p;
    return Status{};
}

// ---------------------------------------------------------------------------------------------
// Multi-chunk keys: sort by a synthetic prefix chunk made of the 8 most significant ACTIVE bytes.
// ---------------------------------------------------------------------------------------------
namespace {

struct PrefixSel {
    u8 chunk[8];   // source chunk of prefix byte j (j = 0 most significant)
    u8 digit[8];   // digit (byte index, 0 = least significant) inside that chunk
    u32 count;     // bytes selected (< 8 when the key has fewer active bytes)
    u32 complete;  // every active byte of the key is part of the prefix: equal prefixes == equal keys
    u32 mixed_long_run;  // set by deep_tie_fix_kernel: the complete schedule has to run
};

// One block: a digit is active when no single bin holds all n keys.  hist holds RAW counts here.
__global__ void __launch_bounds__(256) select_prefix_kernel(const u32* __restrict__ hist, int nchunks, u32 n, PrefixSel* sel) {
    __shared__ u8 s_active[kMaxKeyChunks * kPassesPerChunk];
    const int total = nchunks * kPassesPerChunk;
    for (int rp = 0; rp < total; ++rp) {
        const int full = __syncthreads_or(hist[rp * kRadix + threadIdx.x] == n);
        if (threadIdx.x == 0) s_active[rp] = !full;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    u32 cnt = 0, active = 0;
    for (int c = 0; c < nchunks; ++c)
        for (int p = kPassesPerChunk - 1; p >= 0; --p) {  // most significant byte of the key first
            if (!s_active[c * kPassesPerChunk + p]) continue;
            ++active;
            if (cnt < 8) {
                sel->chunk[cnt] = (u8)c;
                sel->digit[cnt] = (u8)p;
                ++cnt;
            }
        }
    sel->count = cnt;
    sel->complete = active <= 8;
    sel->mixed_long_run = 0;
}

struct ChunkList {
    const u64* p[kMaxKeyChunks];
};

// H[i] = the selected bytes of row i, most significant first; + the digit histogram of H (input of its sort).
__global__ void __launch_bounds__(256) build_prefix_chunk_kernel(const ChunkList chunks, const PrefixSel* __restrict__ sel, u64 n,
                                                                 u64* __restrict__ out, u32* __restrict__ hist) {
    __shared__ u32 sh[kPassesPerChunk * kRadix];
    __shared__ PrefixSel s_sel;
    for (int i = threadIdx.x; i < kPassesPerChunk * kRadix; i += 256) sh[i] = 0;
    if (threadIdx.x == 0) s_sel = *sel;
    __syncthreads();
    const u32 cnt = s_sel.count;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (u64 base = (u64)blockIdx.x * blockDim.x; base < n; base += stride) {  // warp-uniform trips (hist_accumulate)
        const u64 i = base + threadIdx.x;
        const bool valid = i < n;
        u64 h = 0;
        if (valid) {
            u32 last_chunk = 0xffffffffu;
            u64 w = 0;
            for (u32 j = 0; j < cnt; ++j) {
                const u32 c = s_sel.chunk[j];
                if (c != last_chunk) {
                    w = ld_stream_u64(chunks.p[c] + i);
                    last_chunk = c;
                }
                h |= ((w >> (8 * s_sel.digit[j])) & 0xff) << (8 * (7 - j));
            }
            out[i] = h;
        }
        hist_accumulate(sh, h, valid);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kPassesPerChunk * kRadix; i += 256) {
        const u32 c = sh[i];
        if (c) atomicAdd(&hist[i], c);
    }
}

__device__ __forceinline__ int compare_full_keys(const ChunkList& chunks, int nchunks, u32 a, u32 b) {
    for (int c = 0; c < nchunks; ++c) {
        const u64 x = chunks.p[c][a], y = chunks.p[c][b];
        if (x != y) return x < y ? -1 : 1;
    }
    return 0;
}

// After the prefix chunk is sorted: rows whose prefixes tie are ordered by their full keys.  Same structure as
// tie_fix_kernel — the run-start thread insertion-sorts a short run (only the permutation moves: the prefixes are equal);
// a run longer than kMaxTieRun is fine when all of its full keys are equal, adjacent different keys inside a long run
// request the complete schedule.  Full keys are read through the permutation (random 8-byte loads), so a table made of
// few distinct composite keys pays ~2 extra passes' worth of traffic here; keys that differ inside the prefix pay nothing.
__global__ void __launch_bounds__(256) deep_tie_fix_kernel(const SortPlan* plan, const u64* chunk_h, const u64* keys0, const u64* keys1,
                                                           u32* idx0, u32* idx1, const ChunkList chunks, int nchunks, PrefixSel* sel, u32 n) {
    if (sel->complete) return;
    const u32 fk = plan_final_key(plan);
    const u64* keys = fk == 2 ? chunk_h : (fk ? keys1 : keys0);
    const u32 fi = plan_final_idx(plan);
    u32* idx = fi ? idx1 : idx0;  // fi == 2 (identity, no pass ran) means every prefix is equal: handled as one long run
    const u32 lane = threadIdx.x & 31;
    for (u64 base = (u64)blockIdx.x * blockDim.x; base < n; base += (u64)gridDim.x * blockDim.x) {
        const u64 i64 = base + threadIdx.x;
        const bool in = i64 < n;
        const u32 i = (u32)i64;
        const u64 h = in ? keys[i] : 0;
        u64 prev = __shfl_up_sync(0xffffffffu, h, 1);
        u64 next = __shfl_down_sync(0xffffffffu, h, 1);
        if (!in) continue;
        if (lane == 0) prev = i > 0 ? keys[i - 1] : ~h;
        if (lane == 31 || i + 1 >= n) next = i + 1 < n ? keys[i + 1] : ~h;
        if (i > 0 && prev == h) {
            const u32 a = fi == 2 ? i - 1 : idx[i - 1], b = fi == 2 ? i : idx[i];
            if (compare_full_keys(chunks, nchunks, a, b) != 0) {
                u32 s = i;
                while (s > 0 && i - s < (u32)kMaxTieRun && keys[s - 1] == h) --s;
                bool long_run = i - s >= (u32)kMaxTieRun;
                if (!long_run) {
                    u32 e = i + 1;
                    while (e < n && e - s <= (u32)kMaxTieRun && keys[e] == h) ++e;
                    long_run = e - s > (u32)kMaxTieRun;
                }
                if (long_run || fi == 2) sel->mixed_long_run = 1;
            }
            continue;
        }
        if (next != h || fi == 2) continue;
        u32 len = 2;
        while (i + len < n && len <= (u32)kMaxTieRun && keys[i + len] == h) ++len;
        if (len > (u32)kMaxTieRun) continue;
        for (u32 a = 1; a < len; ++a) {  // stable insertion sort of the permutation by the full key
            const u32 v = idx[i + a];
            u32 b = a;
            while (b > 0 && compare_full_keys(chunks, nchunks, idx[i + b - 1], v) > 0) {
                idx[i + b] = idx[i + b - 1];
                --b;
            }
            idx[i + b] = v;
        }
    }
}

}  // namespace

Status radix_sort_keys(Context* ctx, const u64* const* chunks, int nchunks, u64 n, SortScratch* s, PermRef* out) {
    if (nchunks == 1 || n < 2) return radix_sort_chunks(ctx, chunks, nchunks, n, s, out);
    if (nchunks < 1 || nchunks > kMaxKeyChunks)
        return make_status(YTGPU_ERR_UNSUPPORTED, "normalised key of %d bytes exceeds the %d-byte limit", nchunks * 8, kMaxKeyChunks * 8);
    if (n >= (1ull << 30))
        return make_status(YTGPU_ERR_UNSUPPORTED, "row count %llu exceeds 2^30-1 rows per sort call", (unsigned long long)n);
    cudaStream_t st = ctx->stream;
    YTGPU_CUDA_TRY(cudaSetDevice(ctx->device));
    // 1. raw digit counts of every chunk (the complete schedule needs them as well)
    if (!s->hist_precomputed) {
        YTGPU_TRY(histogram_chunks(ctx, chunks, nchunks, n, s));
        s->hist_precomputed = true;
    }
    // 2. prefix chunk of the 8 most significant active bytes + its histogram
    DevBuf<PrefixSel> sel;
    DevBuf<u64> hchunk;
    SortScratch hs;
    YTGPU_TRY(sel.allocate(ctx, 1));
    YTGPU_TRY(hchunk.allocate(ctx, n));
    YTGPU_TRY(prepare_histogram(ctx, 1, &hs));
    ChunkList cl{};
    for (int c = 0; c < nchunks; ++c) cl.p[c] = chunks[c];
    {
        KernelTimer t(ctx, KC_EXTRACT, 2);
        select_prefix_kernel<<<1, 256, 0, st>>>(s->hist.p, nchunks, (u32)n, sel.p);
        const u32 blocks = (u32)std::min<u64>((n + 255) / 256, (u64)kNumSms * 8);
        build_prefix_chunk_kernel<<<blocks, 256, 0, st>>>(cl, sel.p, n, hchunk.p, hs.hist.p);
        YTGPU_CUDA_TRY(cudaGetLastError());
    }
    hs.hist_precomputed = true;
    hs.keep_keys = true;
    // 3. sort it (hybrid schedule and all), then order the rows whose prefixes tie
    PermRef hperm;
    const u64* hptr[1] = {hchunk.p};
    YTGPU_TRY(radix_sort_chunks(ctx, hptr, 1, n, &hs, &hperm));
    {
        KernelTimer t(ctx, KC_HISTOGRAM);
        const u32 blocks = (u32)std::min<u64>((n + 255) / 256, (u64)kNumSms * 8);
        deep_tie_fix_kernel<<<blocks, 256, 0, st>>>(hs.plan.p, hchunk.p, hs.keys[0].p, hs.keys[1].p, hs.idx[0].p, hs.idx[1].p, cl, nchunks, sel.p,
                                                    (u32)n);
        YTGPU_CUDA_TRY(cudaGetLastError());
    }
    // 4. the one host round trip of the multi-chunk path: did a long run of equal prefixes mix different keys?
    PrefixSel hsel;
    YTGPU_CUDA_TRY(cudaMemcpyAsync(&hsel, sel.p, sizeof(PrefixSel), cudaMemcpyDeviceToHost, st));
    YTGPU_CUDA_TRY(cudaStreamSynchronize(st));
    if (hsel.mixed_long_run) return radix_sort_chunks(ctx, chunks, nchunks, n, s, out);  // complete LSD over every active byte
    // hand the prefix sort's buffers over to the caller's scratch (they hold the permutation)
    s->plan = std::move(hs.plan);
    s->idx[0] = std::move(hs.idx[0]);
    s->idx[1] = std::move(hs.idx[1]);
    out->plan = s->plan.p;
    out->idx[0] = s->idx[0].p;
    out->idx[1] = s->idx[1].p;
    return Status{};
}

Status prepare_histogram(Context* ctx, int nchunks, SortScratch* s) {
    const size_t words = (size_t)nchunks * kPassesPerChunk * kRadix;
    YTGPU_TRY(s->hist.allocate(ctx, words));
    YTGPU_CUDA_TRY(cudaMemsetAsync(s->hist.p, 0, words * 4, ctx->stream));
    return Status{};
}

Status materialize_perm(Context* ctx, const PermRef& perm, u64 n, u32* dst_dev) {
    if (n == 0) return Status{};
    u32 blocks = (u32)std::min<u64>((n + 255) / 256, (u64)kNumSms * 8);
    materialize_perm_kernel<<<blocks, 256, 0, ctx->stream>>>(perm.plan, perm.idx[0], perm.idx[1], n, dst_dev);
    ctx->count_launch();
    YTGPU_CUDA_TRY(cudaGetLastError());
    return Status{};
}

}  // namespace ytgpu
