// demuxsim.cpp -- the device demultiplexer of smx_demux_device (specimux_b200/csrc/smx_k_demux.cu) run as host loops over
// the same work items (smx_out.cuh): validation of the offsets per read, the plan per record, a stable sort of
// (compact key, record), the gather per output, the scan, the group boundaries, the tile marks per output and the copy
// per (tile, chunk) -- with tiles of any number of chunks.  TEST ONLY.
#include <algorithm>
#include <cstdint>
#include <numeric>
#include <vector>

#include "../../specimux_b200/csrc/smx_out.cuh"
#include "../../specimux_b200/csrc/smx_pack.cuh"

using namespace smx_out;

extern "C" {

int demuxsim_complement(int ch) { return dna_complement((unsigned char)ch); }

// Returns 0, 1 (bad offsets: *bad = read << 2 | PackFault), 2 (bad records: *bad = record << 3 | OutFault) or 4 (out_cap
// below *n_out_bytes).  counts: n_specimens, n_b1, n_b2, n_pools, n_primers.
int demuxsim_run(const unsigned char *bases, const unsigned char *quals, uint64_t n_bases, const uint64_t *seq_off,
                 uint32_t n_reads, const smx_record *records, uint64_t n, const uint32_t *counts, uint32_t tile_chunks,
                 uint64_t *order, uint64_t *out_off, unsigned char *out_seq, unsigned char *out_qual, uint64_t out_cap,
                 uint64_t *group_key, uint64_t *group_off, uint64_t *n_groups, uint64_t *n_out_bytes, uint64_t *bad) {
    *n_groups = 0; *n_out_bytes = 0; *bad = ~0ull;
    for (uint32_t r = 0; r < n_reads; ++r) {
        const int why = smx::pack_check_read(seq_off, n_bases, r);
        if (why) { *bad = (uint64_t)r << 2 | (uint64_t)why; return 1; }
    }
    const OutCounts cnt = {counts[0], counts[1], counts[2], counts[3], counts[4]};
    const OutShape shape = out_shape(cnt);
    std::vector<uint64_t> key(n), src(n), out_src(n);
    std::vector<uint32_t> len(n), rec(n);
    for (uint64_t r = 0; r < n; ++r) *bad = std::min(*bad, demux_plan_item(records, seq_off, n_reads, cnt, shape, r, key.data(), len.data(), src.data()));
    if (*bad != ~0ull) return 2;
    std::iota(rec.begin(), rec.end(), 0u);
    const uint64_t mask = shape.total_bits >= 64 ? ~0ull : (1ull << shape.total_bits) - 1;
    std::stable_sort(rec.begin(), rec.end(), [&](uint32_t a, uint32_t b) { return (key[a] & mask) < (key[b] & mask); });
    for (uint64_t i = 0; i < n; ++i) demux_gather_item(rec.data(), len.data(), src.data(), n, i, order, out_off, out_src.data());
    if (!n) out_off[0] = 0;
    uint64_t run = 0;
    for (uint64_t i = 0; i <= n; ++i) { const uint64_t v = out_off[i]; out_off[i] = run; run += v; }
    uint64_t g = 0;
    for (uint64_t i = 0; i < n; ++i)
        if (i == 0 || key[rec[i]] != key[rec[i - 1]]) { group_key[g] = out_key_of_sort(key[rec[i]], shape); group_off[g++] = i; }
    group_off[g] = n;
    *n_groups = g;
    const uint64_t total = out_off[n];
    *n_out_bytes = total;
    if (total > out_cap) return 4;
    if (!total) return 0;
    const uint64_t tile_bytes = (uint64_t)tile_chunks * kDemuxChunk;
    uint64_t chunks = demux_chunks(total, out_seq);
    if (quals) chunks = std::max(chunks, demux_chunks(total, out_qual));
    const uint64_t n_marks = (chunks + tile_chunks - 1) / tile_chunks + 2;
    std::vector<uint64_t> tile_first(n_marks, ~0ull);
    for (uint64_t i = 0; i < n; ++i) demux_tile_item(out_off, n, tile_bytes, n_marks, i, tile_first.data());
    const DemuxCopy seq = {bases, out_seq, true, out_off, out_src.data(), n, total};
    const DemuxCopy qual = {quals, out_qual, false, out_off, out_src.data(), n, total};
    const uint64_t seq_chunks = demux_chunks(total, out_seq), qual_chunks = quals ? demux_chunks(total, out_qual) : 0;
    for (uint64_t t = 0; t + 2 < n_marks; ++t)
        for (uint64_t k = 0; k < tile_chunks; ++k) {
            const uint64_t c = t * tile_chunks + k;
            if (c < seq_chunks) demux_copy_chunk(seq, c, tile_first[t], tile_first[t + 2]);
            if (c < qual_chunks) demux_copy_chunk(qual, c, tile_first[t], tile_first[t + 2]);
        }
    return 0;
}

}  // extern "C"
