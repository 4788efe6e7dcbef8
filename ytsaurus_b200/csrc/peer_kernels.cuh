// peer_kernels.cuh — the streaming slab scatter (rows read sequentially, written to stable per-destination slots in
// local or peer-mapped memory) shared by peer.cu (ytgpu_scatter_rows_to_peers) and shuffle.cu (ytgpu_shuffle_sort).
// Kernels are `static` (TU-local) so both translation units may include it.
#pragma once

#include "context.cuh"

namespace ytgpu {

// ---------------------------------------------------------------------------------------------
// Streaming scatter for few partitions (the in-box shuffle: one partition per GPU).  Rows are read
// SEQUENTIALLY (no 128-byte read amplification of random 64-byte accesses, DESIGN.md §4) and each row is
// written to its stable destination slot:  slot = (rows of its partition in earlier tiles) + (rank inside
// the tile).  Per-tile partition counts come from a counting pass over the 4-byte partition index; one
// exclusive scan over the partition-major count matrix [partition][tile] yields every tile's base slot.
// ---------------------------------------------------------------------------------------------
constexpr int kStreamThreads = 256;
constexpr int kStreamItems = 4;
constexpr int kStreamTile = kStreamThreads * kStreamItems;  // rows per tile
constexpr int kStreamMaxParts = 32;

static __global__ void __launch_bounds__(kStreamThreads) tile_count_kernel(const i32* __restrict__ index, u64 n, u32 parts,
                                                                    u64 tiles, u64* __restrict__ counts /*[parts][tiles]*/,
                                                                    u32* __restrict__ err_word) {
    __shared__ u32 s_cnt[kStreamMaxParts];
    if (threadIdx.x < kStreamMaxParts) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const u64 base = (u64)blockIdx.x * kStreamTile;
#pragma unroll
    for (int i = 0; i < kStreamItems; ++i) {
        const u64 r = base + (u64)i * kStreamThreads + threadIdx.x;
        if (r < n) {
            u32 p = (u32)index[r];
            if (p >= parts) {  // caller-supplied index outside [0, parts): flag it, never index shared memory with it
                atomicOr(err_word, (u32)DE_BAD_PARTITION_INDEX);
                p = 0;
            }
            atomicAdd(&s_cnt[p], 1u);
        }
    }
    __syncthreads();
    if (threadIdx.x < parts) counts[(u64)threadIdx.x * tiles + blockIdx.x] = s_cnt[threadIdx.x];
}

// three-phase exclusive scan of u64 (1024 elements per block), in place
static __device__ __forceinline__ u64 scan_block_excl(u64 v, u64* s_warp, u64* total) {
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u64 inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u64 t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (u32)o) inc += t;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    u64 wp = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        u64 x = s_warp[w];
        if (w < (int)warp) wp += x;
        tot += x;
    }
    __syncthreads();
    *total = tot;
    return inc - v + wp;
}
template <bool WRITE>
static __global__ void __launch_bounds__(256) pscan_blocks_kernel(u64* data, u64 n, u64* block_sums) {
    __shared__ u64 s_warp[8];
    const u64 base = (u64)blockIdx.x * 1024 + (u64)threadIdx.x * 4;
    u64 v[4], sum = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        v[i] = base + i < n ? data[base + i] : 0;
        sum += v[i];
    }
    u64 total;
    const u64 ex = scan_block_excl(sum, s_warp, &total);
    if (!WRITE) {
        if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
    } else {
        u64 run = ex + block_sums[blockIdx.x];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (base + i < n) data[base + i] = run;
            run += v[i];
        }
    }
}
static __global__ void __launch_bounds__(256) pscan_sums_kernel(u64* sums, u64 nblocks) {
    __shared__ u64 s_warp[8];
    __shared__ u64 s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (u64 base = 0; base < nblocks; base += 256) {
        const u64 i = base + threadIdx.x;
        const u64 v = i < nblocks ? sums[i] : 0;
        u64 total;
        const u64 ex = scan_block_excl(v, s_warp, &total);
        if (i < nblocks) sums[i] = ex + s_carry;
        __syncthreads();
        if (threadIdx.x == 0) s_carry += total;
        __syncthreads();
    }
}

// The per-partition totals of the counting pass must equal what the caller said it would send: otherwise rows would land
// outside the slabs reserved in the destination buffers.
static __global__ void check_partition_totals_kernel(const u64* __restrict__ scanned /*[parts][tiles]*/, u64 tiles, u64 n, u32 parts,
                                                     const u64* __restrict__ expected_start /*[parts + 1]*/, u32* __restrict__ err_word) {
    const u32 p = threadIdx.x;
    if (p < parts && scanned[(u64)p * tiles] != expected_start[p]) atomicOr(err_word, (u32)DE_BAD_PARTITION_INDEX);
}

struct DestTable {
    uint4* base[kStreamMaxParts];  // destination of partition p's slab
    u64 start[kStreamMaxParts];    // global slot of its first row (scan value of tile 0)
};

// 5 resident CTAs per SM (48 registers): left to itself the compiler takes 54 registers, 4 CTAs per SM, and the 64-byte
// row scatter measured 12 % slower (1.48 vs 1.32 ms for 5*10^7 rows into 4 partitions; B200 at a 1000 W power limit).
static __global__ void __launch_bounds__(kStreamThreads, 5) scatter_stream_kernel(const uint4* __restrict__ in, const i32* __restrict__ index,
                                                                        u64 n, u32 gr, u32 parts, u32 part_bits, u64 tiles,
                                                                        const u64* __restrict__ tile_base /*[parts][tiles]*/,
                                                                        const DestTable D) {
    constexpr int WARPS = kStreamThreads / 32;
    __shared__ u32 s_wcnt[WARPS][kStreamMaxParts];  // running per-warp counts -> warp offsets inside the tile
    __shared__ u64 s_slot[kStreamMaxParts];         // first slot of this tile per partition
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < WARPS * kStreamMaxParts) (&s_wcnt[0][0])[tid] = 0;
    __syncthreads();
    const u64 tile = blockIdx.x;
    const u64 wbase = tile * kStreamTile + (u64)warp * (32 * kStreamItems) + lane;  // warp-striped: stable (item, lane) order
    u32 part[kStreamItems], rank[kStreamItems], pos[kStreamItems];
    u32 lt;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(lt));
#pragma unroll
    for (int i = 0; i < kStreamItems; ++i) {
        const u64 r = wbase + (u64)i * 32;
        const bool valid = r < n;
        part[i] = valid ? min((u32)index[r], parts - 1) : 0u;  // out-of-range values were flagged by the counting pass
        // One sweep of ballots, most significant bit first, yields both the lanes holding the same partition (eq) and
        // the lanes holding a smaller one (less); rows past the end sort after every partition.
        const u32 kk = valid ? part[i] : (1u << part_bits);
        u32 m = 0xffffffffu, less = 0;
        for (int b = (int)part_bits; b >= 0; --b) {
            const bool bit = (kk >> b) & 1;
            const u32 v = __ballot_sync(0xffffffffu, bit);
            if (bit) less |= m & ~v;
            m &= bit ? v : ~v;
        }
        const u32 prev = s_wcnt[warp][part[i]];
        __syncwarp();
        if (valid && (m & lt) == 0) s_wcnt[warp][part[i]] = prev + __popc(m);
        rank[i] = prev + __popc(m & lt);
        pos[i] = __popc(less) + __popc(m & lt);  // position of this row when the round is ordered by destination
        __syncwarp();
    }
    __syncthreads();
    if (tid < parts) {
        u32 run = 0;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) {
            const u32 c = s_wcnt[w][tid];
            s_wcnt[w][tid] = run;
            run += c;
        }
        s_slot[tid] = tile_base[(u64)tid * tiles + tile];
    }
    __syncthreads();
    if (gr == 4) {
        // 64-byte rows: a thread loads its whole row, the warp transposes through shared memory so that four
        // consecutive lanes store the four 16-byte granules of ONE row: every store instruction writes whole
        // 64-byte rows (16-byte stores to scattered rows cost a read-modify-write in L2 and 16-byte NVLink
        // packets — measured 3x slower).  XOR swizzle keeps both the stores and the loads conflict free.
        __shared__ uint4 s_rows[WARPS][32 * 4];
        __shared__ u8 s_order[WARPS][32];  // s_order[q] = lane whose row is the q-th of the round in destination order
        uint4* wr = s_rows[warp];
#pragma unroll
        for (int i = 0; i < kStreamItems; ++i) {
            const u64 r = wbase + (u64)i * 32;
            const bool valid = r < n;
            const u32 p = part[i];
            u64 dst_addr = 0;
            if (valid) {
                const u64 slot = s_slot[p] + s_wcnt[warp][p] + rank[i] - D.start[p];
                dst_addr = reinterpret_cast<u64>(D.base[p] + slot * 4);
            }
            // the 32 rows of this round are contiguous in the input: one coalesced 2 KB copy into shared memory
            const u64 round_row0 = r - lane;
#pragma unroll
            for (u32 s = 0; s < 4; ++s) {
                const u32 q = s * 32 + lane, row = q >> 2, g = q & 3;
                if (round_row0 + row < n) wr[row * 4 + (g ^ ((row >> 1) & 3))] = ld_stream_u128(in + round_row0 * 4 + q);
            }
            // Rows leave in destination order: rows of one partition sit next to each other in its slab, so a store
            // instruction writes runs of whole rows (128 B and more) instead of isolated 64-byte rows — fewer, larger
            // NVLink write packets.
            s_order[warp][pos[i]] = (u8)lane;
            __syncwarp();
#pragma unroll
            for (u32 s = 0; s < 4; ++s) {
                const u32 src_lane = s_order[warp][(lane >> 2) + 8 * s], g = lane & 3;
                const u64 d = __shfl_sync(0xffffffffu, dst_addr, src_lane);
                if (d) reinterpret_cast<uint4*>(d)[g] = wr[src_lane * 4 + (g ^ ((src_lane >> 1) & 3))];
            }
            __syncwarp();
        }
        __threadfence_system();  // peer stores are ordered before whatever signals completion to the other GPU
        return;
    }
#pragma unroll
    for (int i = 0; i < kStreamItems; ++i) {
        const u64 r = wbase + (u64)i * 32;
        if (r >= n) continue;
        const u32 p = part[i];
        const u64 slot = s_slot[p] + s_wcnt[warp][p] + rank[i] - D.start[p];
        const uint4* src = in + r * gr;
        uint4* dst = D.base[p] + slot * gr;
        for (u32 g = 0; g < gr; ++g) dst[g] = ld_stream_u128(src + g);
    }
    __threadfence_system();
}

}  // namespace ytgpu
