// filesim.cpp -- the device file formatter of smx_demux_files_device (specimux_b200/csrc/smx_k_demux.cu) run as host
// loops over the same work items (smx_out.cuh): the name-count check, validation of the read, title and name offsets,
// the plan per record (two slots), a stable sort of (compact key, slot), the gather per slot, the scan, the file
// boundaries without the empty slots, the tile marks per output and the copy per (tile, chunk) -- with tiles of any
// number of chunks.  TEST ONLY.
#include <algorithm>
#include <cstdint>
#include <numeric>
#include <vector>

#include "../../specimux_b200/csrc/smx_out.cuh"
#include "../../specimux_b200/csrc/smx_pack.cuh"

using namespace smx_out;

extern "C" {

// Returns 0; 6 (a name table's count differs from `counts`: *bad = table); 1, 3, 5 (bad read / title / name offsets:
// *bad = item << 2 | PackFault); 2 (bad records: *bad = record << 3 | OutFault); or 4 (out_cap below *n_out_bytes).
// counts: n_specimens, n_b1, n_b2, n_pools, n_primers of the tables; name_counts: those the names claim.
int filesim_run(const unsigned char *bases, const unsigned char *quals, uint64_t n_bases, const uint64_t *seq_off,
                uint32_t n_reads, const unsigned char *titles, uint64_t n_title_bytes, const uint64_t *title_off,
                const smx_record *records, uint64_t n, const char *names, uint64_t n_name_bytes, const uint64_t *name_off,
                const uint32_t *counts, const uint32_t *name_counts, int is_fastq, uint32_t tile_chunks,
                uint64_t *out_record, uint64_t *out_off, unsigned char *out, uint64_t out_cap, uint64_t *file_key,
                uint64_t *file_off, uint64_t *n_files, uint64_t *n_outputs, uint64_t *n_out_bytes, uint64_t *bad) {
    *n_files = 0; *n_outputs = 0; *n_out_bytes = 0; *bad = ~0ull;
    const OutCounts cnt = {counts[0], counts[1], counts[2], counts[3], counts[4]};
    const int table = out_names_mismatch(cnt, name_counts);
    if (table >= 0) { *bad = (uint64_t)table; return 6; }
    for (uint32_t r = 0; r < n_reads; ++r) {
        const int why = smx::pack_check_read(seq_off, n_bases, r);
        if (why) { *bad = (uint64_t)r << 2 | (uint64_t)why; return 1; }
    }
    for (uint32_t r = 0; r < n_reads; ++r) {
        const int why = smx::pack_check_read(title_off, n_title_bytes, r);
        if (why) { *bad = (uint64_t)r << 2 | (uint64_t)why; return 3; }
    }
    const uint64_t n_names = (uint64_t)cnt.n_specimens + cnt.n_b1 + cnt.n_b2 + cnt.n_pools + cnt.n_primers;
    for (uint32_t k = 0; k < n_names; ++k) {
        const int why = smx::pack_check_read(name_off, n_name_bytes, k);
        if (why) { *bad = (uint64_t)k << 2 | (uint64_t)why; return 5; }
    }
    const OutShape shape = out_shape(cnt);
    const FilesPlan plan = {titles, title_off, n_title_bytes, {names, name_off, cnt}, is_fastq != 0};
    const uint64_t slots = 2 * n;
    std::vector<uint64_t> key(slots), len(slots), src(n), hdr(n), id_pos(n), out_src(slots);
    std::vector<uint32_t> slot(slots);
    for (uint64_t r = 0; r < n; ++r)
        *bad = std::min(*bad, files_plan_item(records, seq_off, n_reads, plan, shape, r, key.data(), len.data(), src.data(),
                                              hdr.data(), id_pos.data()));
    if (*bad != ~0ull) return 2;
    if (!n) { out_off[0] = 0; file_off[0] = 0; return 0; }
    std::iota(slot.begin(), slot.end(), 0u);
    std::stable_sort(slot.begin(), slot.end(), [&](uint32_t a, uint32_t b) { return key[a] < key[b]; });
    for (uint64_t i = 0; i < slots; ++i)
        demux_gather_item(slot.data(), len.data(), src.data(), slots, i, out_record, out_off, out_src.data(), 1u);
    uint64_t run = 0;
    for (uint64_t i = 0; i <= slots; ++i) { const uint64_t v = out_off[i]; out_off[i] = run; run += v; }
    uint64_t n_out = 0;
    while (n_out < slots && key[slot[n_out]] != out_empty_slot(shape)) ++n_out;
    uint64_t g = 0;
    for (uint64_t i = 0; i < n_out; ++i)
        if (i == 0 || key[slot[i]] != key[slot[i - 1]]) { file_key[g] = out_key_of_sort(key[slot[i]], shape); file_off[g++] = out_off[i]; }
    file_off[g] = out_off[n_out];
    *n_files = g;
    *n_outputs = n_out;
    const uint64_t total = out_off[n_out];
    *n_out_bytes = total;
    if (total > out_cap) return 4;
    if (!total) return 0;
    const uint64_t tile_bytes = (uint64_t)tile_chunks * kDemuxChunk, chunks = demux_chunks(total, out);
    const uint64_t n_marks = (chunks + tile_chunks - 1) / tile_chunks + 2;
    std::vector<uint64_t> tile_first(n_marks, ~0ull);
    for (uint64_t i = 0; i < n_out; ++i) demux_tile_item(out_off, n_out, tile_bytes, n_marks, i, tile_first.data());
    const FilesCopy fc = {bases, is_fastq ? quals : nullptr, out, is_fastq != 0, out_off, out_src.data(), out_record,
                          hdr.data(), id_pos.data(), records, titles, {names, name_off, cnt}, n_out, total};
    for (uint64_t t = 0; t + 2 < n_marks; ++t)
        for (uint64_t k = 0; k < tile_chunks; ++k) {
            const uint64_t c = t * tile_chunks + k;
            if (c < chunks) demux_copy_chunk(fc, c, tile_first[t], tile_first[t + 2]);
        }
    return 0;
}

}  // extern "C"
