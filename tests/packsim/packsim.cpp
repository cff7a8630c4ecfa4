// packsim.cpp -- the device packer of smx_match_device (specimux_b200/csrc/smx_k_pack.cu) run as host loops over the
// same per-thread work items (smx_pack.cuh): validation per read, the fixed-stride pass per (read, word), the off4 scan
// in kPackTile-read tiles of kPackThreads threads, and the side stream per (flagged read, word).  TEST ONLY.
#include <algorithm>
#include <cstdint>
#include <vector>

#include "../../specimux_b200/csrc/smx_pack.cuh"

using namespace smx;

namespace {
constexpr int kPackThreads = 256;       // as smx_k_pack.cu
constexpr int kPackPerThread = kPackTile / kPackThreads;
}

extern "C" {

int packsim_read_code(int ch) { return read_code((unsigned char)ch); }
int packsim_read_code_rc(int ch) { return read_code_rc((unsigned char)ch); }

// Validation key of the batch: min over refused reads of (read << 2 | PackFault), ~0 when every read passes.
uint64_t packsim_validate(const uint64_t *seq_off, uint32_t n, uint64_t n_bases) {
    uint64_t key = ~0ull;
    for (uint32_t r = 0; r < n; ++r) {
        const int why = pack_check_read(seq_off, n_bases, r);
        if (why && ((uint64_t)r << 2 | (uint64_t)why) < key) key = (uint64_t)r << 2 | (uint64_t)why;
    }
    return key;
}

// Packs reads [0, n) cut into n_lanes lanes at cuts[0..n_lanes] (cuts[0] = 0, cuts[n_lanes] = n).  packed2 receives the
// lanes' packed2 buffers back to back ((cuts[l + 1] - cuts[l]) * stride + 1 words each), lengths / off4 n entries,
// packed4 the side stream (cap4 words).  Returns the validation key; nothing is packed unless it is ~0.
uint64_t packsim_pack(const unsigned char *bases, uint64_t n_bases, const uint64_t *seq_off, uint32_t n, uint32_t clip,
                      int n_lanes, const uint32_t *cuts, uint32_t *packed2, uint32_t *lengths, uint64_t *off4,
                      uint32_t *packed4, uint64_t cap4, uint64_t *words4, uint32_t *n_flagged) {
    const uint64_t key = packsim_validate(seq_off, n, n_bases);
    *words4 = 0; *n_flagged = 0;
    if (key != ~0ull) return key;
    PackLanes d = {};
    d.n_lanes = n_lanes; d.clip = clip; d.stride = (2 * clip + 15) / 16;
    uint64_t at = 0;
    for (int l = 0; l < n_lanes; ++l) {
        d.r0[l] = cuts[l]; d.r0[l + 1] = cuts[l + 1];
        d.packed2[l] = packed2 + at;
        d.lengths[l] = lengths + cuts[l];
        d.off4[l] = off4 + cuts[l];
        at += (uint64_t)(cuts[l + 1] - cuts[l]) * d.stride + 1;
    }
    // fixed-stride pass: one item per (read, word); the first item to see a non-ACGT byte lists the read
    std::vector<uint32_t> flag(n, 0), list;
    for (uint64_t i = 0; i < (uint64_t)n * d.stride; ++i)
        if (pack_fixed_item(bases, seq_off, n, d, i)) {
            const uint32_t r = (uint32_t)(i / d.stride);
            if (!flag[r]) { flag[r] = 1; list.push_back(r); }
        }
    *n_flagged = (uint32_t)list.size();
    if (list.empty()) return key;
    // tile sums, their exclusive scan, then the scan within each tile (per thread: kPackPerThread consecutive reads)
    const uint64_t tiles = ((uint64_t)n + kPackTile - 1) / kPackTile;
    std::vector<uint64_t> tile_sum(tiles, 0);
    for (uint64_t b = 0; b < tiles; ++b)
        for (uint64_t r = b * kPackTile; r < std::min<uint64_t>((b + 1) * kPackTile, n); ++r)
            tile_sum[b] += pack_count4(seq_off, clip, flag[r] != 0, (uint32_t)r);
    uint64_t carry = 0;
    for (uint64_t b = 0; b < tiles; ++b) { const uint64_t v = tile_sum[b]; tile_sum[b] = carry; carry += v; }
    for (uint64_t b = 0; b < tiles; ++b) {
        uint64_t thread_off = tile_sum[b];
        for (int t = 0; t < kPackThreads; ++t) {
            const uint64_t r0 = b * kPackTile + (uint64_t)t * kPackPerThread;
            uint64_t off = thread_off;
            for (int k = 0; k < kPackPerThread; ++k) {
                if (r0 + k >= n) break;
                const uint64_t c = pack_count4(seq_off, clip, flag[r0 + k] != 0, (uint32_t)(r0 + k));
                pack_set_off4(d, (uint32_t)(r0 + k), c != 0, off);
                off += c;
            }
            thread_off = off;
        }
    }
    *words4 = carry;
    if (carry > cap4) return key;
    // side stream: one warp per listed read, 32 words at a time
    for (uint32_t r : list) {
        const uint64_t n4 = pack_words4(pack_stored_len(seq_off[r + 1] - seq_off[r], clip));
        for (uint64_t w = 0; w < 2 * n4; ++w) pack_side_word(bases, seq_off, d, packed4, r, w);
    }
    return key;
}

}  // extern "C"
