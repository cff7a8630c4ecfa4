// smx_k_pack.cu -- device packer of smx_match_device: ASCII reads already in device memory -> the smx_batch encoding,
// written straight into the lanes' batch buffers.  The per-thread work items are the routines of smx_pack.cuh that
// the host packer uses too; what is here is their launch geometry and the scan of the side-stream offsets.
#include "smx_launch.hpp"
#include "smx_pack.cuh"

namespace smx {

namespace {

constexpr int kPackThreads = 256;
constexpr int kPackPerThread = kPackTile / kPackThreads;
static_assert(kPackTile % kPackThreads == 0, "scan tile");

// grid of a grid-stride loop over `items`: at most 2^20 blocks
unsigned pack_blocks(u64 items, int threads) {
    const u64 b = (items + threads - 1) / threads;
    return (unsigned)(b < 1 ? 1 : b > (1u << 20) ? (1u << 20) : b);
}

// exclusive scan of one value per thread over a block of kPackThreads threads; *total receives the block's sum
__device__ u64 block_exclusive_scan(u64 v, u64 *total) {
    __shared__ u64 warp_sum[kPackThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u64 x = v;
    for (int o = 1; o < 32; o <<= 1) {
        const u64 y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_sum[warp] = x;
    __syncthreads();
    if (warp == 0) {
        u64 s = lane < kPackThreads / 32 ? warp_sum[lane] : 0;
        for (int o = 1; o < 32; o <<= 1) {
            const u64 y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        if (lane < kPackThreads / 32) warp_sum[lane] = s;         // inclusive over warps
    }
    __syncthreads();
    const u64 before = warp ? warp_sum[warp - 1] : 0;
    *total = warp_sum[kPackThreads / 32 - 1];
    __syncthreads();                                             // warp_sum is reused by the next call
    return before + x - v;
}

}  // namespace

// One thread per read; the smallest (read << 2 | reason) of a refused read wins.
__global__ void __launch_bounds__(kPackThreads) k_pack_validate(const u64 *seq_off, u32 n, u64 n_bases, unsigned long long *bad) {
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (u64)gridDim.x * blockDim.x) {
        const int why = pack_check_read(seq_off, n_bases, (u32)r);
        if (why) atomicMin(bad, (unsigned long long)(r << 2 | (u64)why));
    }
}

// One thread per (read, packed2 word).  The first word of a read found to hold a non-ACGT byte flags the read and
// appends it to `list` (unordered; off4 gives the order).
__global__ void __launch_bounds__(kPackThreads) k_pack_fixed(const unsigned char *bases, const u64 *seq_off, u32 n, PackLanes d,
                                                             u32 *flag, u32 *list, unsigned long long *n_flagged) {
    const u64 items = (u64)n * d.stride;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < items; i += (u64)gridDim.x * blockDim.x) {
        if (pack_fixed_item(bases, seq_off, n, d, i)) {
            const u32 r = (u32)(i / d.stride);
            if (atomicCAS(&flag[r], 0u, 1u) == 0u) list[atomicAdd(n_flagged, 1ull)] = r;
        }
    }
}

// Side-stream words of the reads of tile b (kPackTile reads, kPackPerThread consecutive reads per thread)
__global__ void __launch_bounds__(kPackThreads) k_pack_tile_sums(const u64 *seq_off, u32 n, u32 clip, const u32 *flag, u64 *tile_sum) {
    const u64 r0 = (u64)blockIdx.x * kPackTile + (u64)threadIdx.x * kPackPerThread;
    u64 s = 0;
    for (int k = 0; k < kPackPerThread; ++k)
        if (r0 + k < n) s += pack_count4(seq_off, clip, flag[r0 + k] != 0, (u32)(r0 + k));
    u64 total;
    block_exclusive_scan(s, &total);
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = total;
}

// Exclusive scan of the tile sums in place, one block.
__global__ void __launch_bounds__(kPackThreads) k_pack_scan_tiles(u64 *tile_sum, u32 n_tiles) {
    u64 carry = 0;
    for (u32 base = 0; base < n_tiles; base += kPackThreads) {
        const u32 t = base + threadIdx.x;
        const u64 v = t < n_tiles ? tile_sum[t] : 0;
        u64 total;
        const u64 ex = block_exclusive_scan(v, &total);
        if (t < n_tiles) tile_sum[t] = carry + ex;
        carry += total;
    }
}

// off4 of every read: tile prefix + the scan within the tile
__global__ void __launch_bounds__(kPackThreads) k_pack_off4(const u64 *seq_off, u32 n, const u32 *flag, const u64 *tile_sum, PackLanes d) {
    const u64 r0 = (u64)blockIdx.x * kPackTile + (u64)threadIdx.x * kPackPerThread;
    u64 cnt[kPackPerThread], s = 0;
    for (int k = 0; k < kPackPerThread; ++k) {
        cnt[k] = r0 + k < n ? pack_count4(seq_off, d.clip, flag[r0 + k] != 0, (u32)(r0 + k)) : 0;
        s += cnt[k];
    }
    u64 total;
    u64 off = tile_sum[blockIdx.x] + block_exclusive_scan(s, &total);
    for (int k = 0; k < kPackPerThread; ++k) {
        if (r0 + k < n) pack_set_off4(d, (u32)(r0 + k), cnt[k] != 0, off);
        off += cnt[k];
    }
}

// One warp per flagged read: its 2 * n4 side-stream words.
__global__ void __launch_bounds__(kPackThreads) k_pack_side(const unsigned char *bases, const u64 *seq_off, const u32 *list, u32 n_list,
                                                            PackLanes d, u32 *packed4) {
    const u64 warps = ((u64)gridDim.x * blockDim.x) >> 5;
    for (u64 k = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5; k < n_list; k += warps) {
        const u32 r = list[k];
        const u64 n4 = pack_words4(pack_stored_len(seq_off[r + 1] - seq_off[r], d.clip));
        for (u64 w = threadIdx.x & 31; w < 2 * n4; w += 32) pack_side_word(bases, seq_off, d, packed4, r, w);
    }
}

cudaError_t launch_pack_validate(const u64 *seq_off, u32 n, u64 n_bases, unsigned long long *bad, cudaStream_t st) {
    k_pack_validate<<<pack_blocks(n, kPackThreads), kPackThreads, 0, st>>>(seq_off, n, n_bases, bad);
    return cudaGetLastError();
}

cudaError_t launch_pack_fixed(const unsigned char *bases, const u64 *seq_off, u32 n, const PackLanes &d, u32 *flag, u32 *list,
                              unsigned long long *n_flagged, cudaStream_t st) {
    k_pack_fixed<<<pack_blocks((u64)n * d.stride, kPackThreads), kPackThreads, 0, st>>>(bases, seq_off, n, d, flag, list, n_flagged);
    return cudaGetLastError();
}

cudaError_t launch_pack_off4(const u64 *seq_off, u32 n, const u32 *flag, u64 *tile_sum, const PackLanes &d, cudaStream_t st) {
    const u32 tiles = (u32)(((u64)n + kPackTile - 1) / kPackTile);
    k_pack_tile_sums<<<tiles, kPackThreads, 0, st>>>(seq_off, n, d.clip, flag, tile_sum);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    k_pack_scan_tiles<<<1, kPackThreads, 0, st>>>(tile_sum, tiles);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    k_pack_off4<<<tiles, kPackThreads, 0, st>>>(seq_off, n, flag, tile_sum, d);
    return cudaGetLastError();
}

cudaError_t launch_pack_side(const unsigned char *bases, const u64 *seq_off, const u32 *list, u32 n_list, const PackLanes &d,
                             u32 *packed4, cudaStream_t st) {
    k_pack_side<<<pack_blocks((u64)n_list * 32, kPackThreads), kPackThreads, 0, st>>>(bases, seq_off, list, n_list, d, packed4);
    return cudaGetLastError();
}

}  // namespace smx
