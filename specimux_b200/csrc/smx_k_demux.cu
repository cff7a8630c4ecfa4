// smx_k_demux.cu -- device demultiplexer of smx_demux_device: records + reads in device memory -> the trimmed, oriented
// sequences and qualities grouped by destination file.  The per-record and per-tile work items are the routines of
// smx_out.cuh that the host writer and tests/demuxsim use too; what is here is their launch geometry, the stable
// radix sort of (destination, record), the scan of the output lengths and the group boundaries (CUB).
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "smx_launch.hpp"

namespace smx {

using namespace smx_out;

namespace {

constexpr int kDemuxThreads = 256;
constexpr u32 kDemuxTileChunks = kDemuxThreads;     // one 16-byte chunk per thread and buffer per tile

unsigned demux_blocks(u64 items) {
    const u64 b = (items + kDemuxThreads - 1) / kDemuxThreads;
    return (unsigned)(b < 1 ? 1 : b > (1u << 20) ? (1u << 20) : b);
}

}  // namespace

// One thread per record; the smallest (record << 3 | OutFault) of a refused record wins.
__global__ void __launch_bounds__(kDemuxThreads) k_demux_plan(const smx_record *records, u64 n, const u64 *seq_off, u32 n_reads,
                                                              OutCounts cnt, OutShape shape, u64 *sort_key, u32 *rec, u32 *len,
                                                              u64 *src, unsigned long long *bad) {
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (u64)gridDim.x * blockDim.x) {
        const u64 key = demux_plan_item(records, seq_off, n_reads, cnt, shape, r, sort_key, len, src);
        rec[r] = (u32)r;
        if (key != ~0ull) atomicMin(bad, (unsigned long long)key);
    }
}

__global__ void __launch_bounds__(kDemuxThreads) k_demux_gather(const u32 *sorted_rec, const u32 *len, const u64 *src, u64 n,
                                                                u64 *order, u64 *out_off, u64 *out_src) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        demux_gather_item(sorted_rec, len, src, n, i, order, out_off, out_src);
}

// Group keys: the compact keys UniqueByKey left in group_key, widened in place; group_off[G] = n; ctl[3] = total bytes.
__global__ void __launch_bounds__(kDemuxThreads) k_demux_groups(u64 n, OutShape shape, const u64 *out_off, u64 *group_key,
                                                                u64 *group_off, unsigned long long *ctl) {
    const u64 g = ctl[2];
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < g; i += (u64)gridDim.x * blockDim.x)
        group_key[i] = out_key_of_sort(group_key[i], shape);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        group_off[g] = n;
        ctl[3] = out_off[n];
    }
}

__global__ void __launch_bounds__(kDemuxThreads) k_demux_tiles(const u64 *out_off, u64 n_out, u64 n_marks, u64 *tile_first) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_out; i += (u64)gridDim.x * blockDim.x)
        demux_tile_item(out_off, n_out, (u64)kDemuxTileChunks * kDemuxChunk, n_marks, i, tile_first);
}

// One block per tile of output bytes: thread k copies chunk k of the tile in each buffer.
__global__ void __launch_bounds__(kDemuxThreads) k_demux_copy(DemuxCopy seq, DemuxCopy qual, u64 seq_chunks, u64 qual_chunks,
                                                              const u64 *tile_first) {
    const u64 t = blockIdx.x, c = t * kDemuxTileChunks + threadIdx.x;
    const u64 lo = tile_first[t], hi = tile_first[t + 2];
    if (c < seq_chunks) demux_copy_chunk(seq, c, lo, hi);
    if (c < qual_chunks) demux_copy_chunk(qual, c, lo, hi);
}

cudaError_t demux_temp_bytes(u64 n, size_t *bytes) {
    size_t a = 0, b = 0, c = 0;
    cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, a, (const u64 *)nullptr, (u64 *)nullptr, (const u32 *)nullptr,
                                                    (u32 *)nullptr, (int)n, 0, 64);
    if (e != cudaSuccess) return e;
    if ((e = cub::DeviceScan::ExclusiveSum(nullptr, b, (u64 *)nullptr, (u64 *)nullptr, (int)(n + 1))) != cudaSuccess) return e;
    e = cub::DeviceSelect::UniqueByKey(nullptr, c, (const u64 *)nullptr, thrust::counting_iterator<u64>(0), (u64 *)nullptr,
                                       (u64 *)nullptr, (unsigned long long *)nullptr, (int)n);
    *bytes = std::max(a, std::max(b, c));
    return e;
}

cudaError_t launch_demux_index(const DemuxIndex &a, cudaStream_t st) {
    const u64 n = a.n_records;
    const DemuxScratch &s = a.scratch;
    k_demux_plan<<<demux_blocks(n), kDemuxThreads, 0, st>>>(a.records, n, a.seq_off, a.n_reads, a.counts, a.shape, s.key_in,
                                                            s.rec_in, s.len, s.src, s.ctl + 1);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    size_t bytes = s.temp_bytes;
    if ((e = cub::DeviceRadixSort::SortPairs(s.temp, bytes, s.key_in, s.key_out, s.rec_in, s.rec_out, (int)n, 0,
                                             (int)a.shape.total_bits, st)) != cudaSuccess) return e;
    k_demux_gather<<<demux_blocks(n), kDemuxThreads, 0, st>>>(s.rec_out, s.len, s.src, n, a.order, a.out_off, s.out_src);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    bytes = s.temp_bytes;
    if ((e = cub::DeviceScan::ExclusiveSum(s.temp, bytes, a.out_off, a.out_off, (int)(n + 1), st)) != cudaSuccess) return e;
    bytes = s.temp_bytes;
    if ((e = cub::DeviceSelect::UniqueByKey(s.temp, bytes, s.key_out, thrust::counting_iterator<u64>(0), a.group_key, a.group_off,
                                            s.ctl + 2, (int)n, st)) != cudaSuccess) return e;
    k_demux_groups<<<demux_blocks(n), kDemuxThreads, 0, st>>>(n, a.shape, a.out_off, a.group_key, a.group_off, s.ctl);
    return cudaGetLastError();
}

u64 demux_tile_marks(u64 total, const void *out_seq, const void *out_qual) {
    u64 chunks = demux_chunks(total, out_seq);
    if (out_qual) chunks = std::max(chunks, demux_chunks(total, out_qual));
    return (chunks + kDemuxTileChunks - 1) / kDemuxTileChunks + 2;
}

cudaError_t launch_demux_copy(const unsigned char *bases, const unsigned char *quals, const u64 *out_off, const u64 *out_src,
                              u64 n_out, u64 total, unsigned char *out_seq, unsigned char *out_qual, u64 *tile_first,
                              cudaStream_t st) {
    if (!total) return cudaSuccess;
    const u64 n_marks = demux_tile_marks(total, out_seq, out_qual);
    k_demux_tiles<<<demux_blocks(n_out), kDemuxThreads, 0, st>>>(out_off, n_out, n_marks, tile_first);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const DemuxCopy seq = {bases, out_seq, true, out_off, out_src, n_out, total};
    const DemuxCopy qual = {quals, out_qual, false, out_off, out_src, n_out, total};
    k_demux_copy<<<(unsigned)(n_marks - 2), kDemuxThreads, 0, st>>>(seq, qual, demux_chunks(total, out_seq),
                                                                     quals ? demux_chunks(total, out_qual) : 0, tile_first);
    return cudaGetLastError();
}

}  // namespace smx
