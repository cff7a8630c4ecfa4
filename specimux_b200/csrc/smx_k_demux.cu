// smx_k_demux.cu -- device demultiplexer of smx_demux_device (records + reads in device memory -> the trimmed, oriented
// sequences and qualities grouped by destination file) and of smx_demux_files_device (-> every output file's complete
// contents, headers and pool-level copies included).  The per-record and per-tile work items are the routines of
// smx_out.cuh that the host writer and tests/demuxsim / tests/filesim use too; what is here is their launch geometry,
// the stable radix sort of (destination, slot), the scan of the output lengths and the group boundaries (CUB).
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

__global__ void __launch_bounds__(kDemuxThreads) k_files_plan(const smx_record *records, u64 n, const u64 *seq_off, u32 n_reads,
                                                              FilesPlan plan, OutShape shape, u64 *sort_key, u32 *slot, u64 *len,
                                                              u64 *src, u64 *hdr, u64 *id_pos, unsigned long long *bad) {
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (u64)gridDim.x * blockDim.x) {
        const u64 key = files_plan_item(records, seq_off, n_reads, plan, shape, r, sort_key, len, src, hdr, id_pos);
        slot[2 * r] = (u32)(2 * r);
        slot[2 * r + 1] = (u32)(2 * r + 1);
        if (key != ~0ull) atomicMin(bad, (unsigned long long)key);
    }
}

template <class Len>
__global__ void __launch_bounds__(kDemuxThreads) k_demux_gather(const u32 *sorted_rec, const Len *len, const u64 *src, u64 n,
                                                                u64 *order, u64 *out_off, u64 *out_src, u32 shift) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        demux_gather_item(sorted_rec, len, src, n, i, order, out_off, out_src, shift);
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

// Files: the slots before the first empty one (sorted keys) are the outputs; the empty slots form the last group, if
// any, which is dropped.  File keys widened in place, file_off in bytes; ctl[3] total bytes, ctl[4] files, ctl[5] outputs.
__global__ void __launch_bounds__(kDemuxThreads) k_files_groups(u64 n_slots, OutShape shape, const u64 *sorted_key,
                                                                const u64 *out_off, u64 *group_key, const u64 *group_idx,
                                                                u64 *file_off, unsigned long long *ctl) {
    const u64 empty = out_empty_slot(shape);
    u64 lo = 0, hi = n_slots;                      // first slot whose key is the empty one
    while (lo < hi) {
        const u64 mid = (lo + hi) >> 1;
        if (sorted_key[mid] < empty) lo = mid + 1; else hi = mid;
    }
    const u64 n_out = lo, g = ctl[2] - (n_out < n_slots ? 1 : 0);
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < g; i += (u64)gridDim.x * blockDim.x) {
        group_key[i] = out_key_of_sort(group_key[i], shape);
        file_off[i] = out_off[group_idx[i]];
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        file_off[g] = out_off[n_out];
        ctl[3] = out_off[n_out];
        ctl[4] = g;
        ctl[5] = n_out;
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

// One block per tile of output bytes: thread k copies chunk k of the tile.  The byte-wise path (headers, section
// boundaries) needs more registers than the launch bounds' default of 64 leaves without spills; 96 gives it room.
__global__ void __maxnreg__(96) k_files_copy(FilesCopy f, u64 chunks, const u64 *tile_first) {
    const u64 t = blockIdx.x, c = t * kDemuxTileChunks + threadIdx.x;
    if (c < chunks) demux_copy_chunk(f, c, tile_first[t], tile_first[t + 2]);
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
    const FilesIndex *f = a.files;
    const u64 slots = f ? 2 * n : n;
    if (f)
        k_files_plan<<<demux_blocks(n), kDemuxThreads, 0, st>>>(a.records, n, a.seq_off, a.n_reads, f->plan, a.shape, s.key_in,
                                                                s.rec_in, f->len, s.src, f->hdr, f->id_pos, s.ctl + 1);
    else
        k_demux_plan<<<demux_blocks(n), kDemuxThreads, 0, st>>>(a.records, n, a.seq_off, a.n_reads, a.counts, a.shape, s.key_in,
                                                                s.rec_in, s.len, s.src, s.ctl + 1);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    size_t bytes = s.temp_bytes;
    if ((e = cub::DeviceRadixSort::SortPairs(s.temp, bytes, s.key_in, s.key_out, s.rec_in, s.rec_out, (int)slots, 0,
                                             (int)a.shape.total_bits + (f ? 1 : 0), st)) != cudaSuccess) return e;
    if (f)
        k_demux_gather<<<demux_blocks(slots), kDemuxThreads, 0, st>>>(s.rec_out, (const u64 *)f->len, s.src, slots, a.order,
                                                                      a.out_off, s.out_src, 1u);
    else
        k_demux_gather<<<demux_blocks(n), kDemuxThreads, 0, st>>>(s.rec_out, (const u32 *)s.len, s.src, n, a.order, a.out_off,
                                                                  s.out_src, 0u);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    bytes = s.temp_bytes;
    if ((e = cub::DeviceScan::ExclusiveSum(s.temp, bytes, a.out_off, a.out_off, (int)(slots + 1), st)) != cudaSuccess) return e;
    bytes = s.temp_bytes;
    if ((e = cub::DeviceSelect::UniqueByKey(s.temp, bytes, s.key_out, thrust::counting_iterator<u64>(0), a.group_key,
                                            f ? f->group_idx : a.group_off, s.ctl + 2, (int)slots, st)) != cudaSuccess) return e;
    if (f)
        k_files_groups<<<demux_blocks(slots), kDemuxThreads, 0, st>>>(slots, a.shape, s.key_out, a.out_off, a.group_key,
                                                                      f->group_idx, f->file_off, s.ctl);
    else
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

cudaError_t launch_files_copy(const FilesCopy &f, u64 *tile_first, cudaStream_t st) {
    if (!f.total) return cudaSuccess;
    const u64 n_marks = demux_tile_marks(f.total, f.dst, nullptr);
    k_demux_tiles<<<demux_blocks(f.n_out), kDemuxThreads, 0, st>>>(f.out_off, f.n_out, n_marks, tile_first);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    k_files_copy<<<(unsigned)(n_marks - 2), kDemuxThreads, 0, st>>>(f, demux_chunks(f.total, f.dst), tile_first);
    return cudaGetLastError();
}

}  // namespace smx
