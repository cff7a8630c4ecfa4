// minesim.cpp -- specimine on device files (smx_mine_device, specimux_b200/csrc/smx_k_mine_device.cu) run as host loops
// over the same work items (smx_mine.cuh): the host checks of the group table, locate per involved file and output, the
// group scan, the plan per pattern (limits, work items per class), the items at their class cursors, the entries' texts,
// a stand-in for k_hw_best (the caller's `search`, over the items), the decision per entry, the scans, the compaction,
// the .mined file offsets and the record text.  TEST ONLY.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../specimux_b200/csrc/smx_mine.cuh"

using namespace smx_mine;

extern "C" {

// keys[e] = min over the items' (pattern, entry) pairs of (floor(d * 2^40 / m) << 23) | rank, as k_hw_best leaves it
typedef void (*minesim_search)(const HwItem *items, uint64_t n_items, const uint64_t *beg, const uint32_t *len,
                               const int32_t *k, const uint32_t *ent_txt, uint64_t n_ent, unsigned long long *keys);

// Returns 0; 1 (a bad group table); 2 (a fault on the device side: *bad = file << 35 | output << 3 | MineFault); or 4
// (out_cap or rec_cap below *n_out_bytes / *n_records).
int minesim_run(const unsigned char *data, uint64_t n_data, const uint64_t *out_off, uint64_t n_outputs,
                const uint64_t *file_off, uint64_t n_files, uint32_t n_groups, const uint32_t *grp_file,
                const uint8_t *grp_kind, const uint32_t *grp_part_off, const uint32_t *grp_part, uint32_t n_mined,
                const uint32_t *mined_grp, double min_identity, minesim_search search, unsigned char *out,
                uint64_t out_cap, uint64_t rec_cap, uint64_t *mined_off, int64_t *rec_partial, int64_t *rec_winner,
                int32_t *rec_dist, uint64_t *n_records, uint64_t *n_out_bytes, uint64_t *bad) {
    *n_records = 0; *n_out_bytes = 0; *bad = ~0ull;
    const uint32_t G = n_groups;
    if (n_files >= kMineMaxFiles || mined_grp[0] != 0 || mined_grp[n_mined] != G || (G && grp_part_off[0] != 0)) return 1;
    for (uint64_t f = 0; f < n_files; ++f)
        if (file_off[f + 1] < file_off[f] || file_off[f + 1] > n_data) return 1;
    std::vector<char> seen(n_files, 0);
    std::vector<uint32_t> involved;
    auto take = [&](uint32_t f) { if (!seen[f]) { seen[f] = 1; involved.push_back(f); } };
    for (uint32_t g = 0; g < G; ++g) {
        if (grp_file[g] >= n_files || grp_kind[g] > 1 || grp_part_off[g + 1] < grp_part_off[g]) return 1;
        take(grp_file[g]);
        for (uint32_t k = grp_part_off[g]; k < grp_part_off[g + 1]; ++k) {
            if (grp_part[k] >= n_files) return 1;
            take(grp_part[k]);
        }
    }
    // locate
    std::vector<uint64_t> rng(2 * n_files), beg(n_outputs + 1);
    std::vector<uint32_t> len(n_outputs + 1);
    std::vector<int32_t> kk(n_outputs + 1);
    for (uint32_t f : involved) {
        uint64_t o0, o1;
        *bad = std::min(*bad, mine_locate_file(out_off, n_outputs, file_off, f, o0, o1));
        rng[2 * f] = o0; rng[2 * f + 1] = o1;
        for (uint64_t o = o0; o < o1; ++o) {
            const int fault = mine_locate_output(data, n_data, out_off, o, beg[o], len[o]);
            if (fault) *bad = std::min(*bad, mine_fault_key(f, o - o0, fault));
            kk[o] = mine_k(len[o], min_identity);
        }
    }
    if (*bad != ~0ull) return 2;
    // group scan
    std::vector<uint64_t> pat_base(G + 1, 0), ent_base(G + 1, 0);
    for (uint32_t g = 0; g < G; ++g) {
        uint64_t ne = 0;
        for (uint32_t k = grp_part_off[g]; k < grp_part_off[g + 1]; ++k) ne += rng[2 * grp_part[k] + 1] - rng[2 * grp_part[k]];
        pat_base[g + 1] = pat_base[g] + rng[2 * grp_file[g] + 1] - rng[2 * grp_file[g]];
        ent_base[g + 1] = ent_base[g] + ne;
    }
    const uint64_t P = pat_base[G], E = ent_base[G];
    // plan
    uint64_t count[kHwClasses] = {};
    for (uint32_t g = 0; g < G; ++g)
        for (uint64_t r = 0; r < pat_base[g + 1] - pat_base[g]; ++r) {
            const uint64_t o = rng[2 * grp_file[g]] + r, m = len[o];
            if (r >= kMineMaxRank) { *bad = std::min(*bad, mine_fault_key(grp_file[g], r, kMineRank)); continue; }
            if (m > kMineMaxPattern) { *bad = std::min(*bad, mine_fault_key(grp_file[g], r, kMineLong)); continue; }
            uint32_t mask[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            mine_byte_set(data + beg[o], 0, m, 1, mask);
            if (mine_popc8(mask) > kMineMaxCodes) { *bad = std::min(*bad, mine_fault_key(grp_file[g], r, kMineCodes)); continue; }
            int cls;
            const uint64_t n = mine_items(m, ent_base[g + 1] - ent_base[g], cls);
            if (n) count[cls] += n;
        }
    if (*bad != ~0ull) return 2;
    (void)P;
    // items at their class cursors, entries, search
    uint64_t cursor[kHwClasses], n_items = 0;
    for (int c = 0; c < kHwClasses; ++c) { cursor[c] = n_items; n_items += count[c]; }
    std::vector<HwItem> items(n_items + 1);
    for (uint32_t g = 0; g < G; ++g)
        for (uint64_t r = 0; r < pat_base[g + 1] - pat_base[g]; ++r) {
            const uint64_t o = rng[2 * grp_file[g]] + r, m = len[o], e0 = ent_base[g], ne = ent_base[g + 1] - e0;
            int cls;
            const uint64_t n = mine_items(m, ne, cls);
            int sw, w;
            if (n) hw_best_class((int)((m + 31) / 32), &sw, &w);
            for (uint64_t i = 0; i < n; ++i) {
                const uint64_t lo = i * hw_best_chunk(sw);
                items[cursor[cls]++] = HwItem{(uint32_t)o, (uint32_t)r, e0 + lo, (uint32_t)std::min<uint64_t>(ne - lo, hw_best_chunk(sw)), 0u};
            }
        }
    std::vector<uint32_t> ent_txt(E + 1);
    for (uint32_t g = 0; g < G; ++g) {
        uint64_t at = ent_base[g];
        for (uint32_t k = grp_part_off[g]; k < grp_part_off[g + 1]; ++k)
            for (uint64_t o = rng[2 * grp_part[k]]; o < rng[2 * grp_part[k] + 1]; ++o) ent_txt[at++] = (uint32_t)o;
    }
    std::vector<unsigned long long> keys(E + 1, ~0ull);
    if (n_items) search(items.data(), n_items, beg.data(), len.data(), kk.data(), ent_txt.data(), E, keys.data());
    // decide, scans
    std::vector<uint64_t> size(E + 1, 0), flag(E + 1, 0), win(E + 1), dist(E + 1), size_off(E + 1), flag_off(E + 1);
    std::vector<uint32_t> grp_of(E + 1);
    for (uint32_t g = 0; g < G; ++g)
        for (uint64_t e = ent_base[g]; e < ent_base[g + 1]; ++e) {
            grp_of[e] = g;
            size[e] = mine_decide_item(data, out_off, beg.data(), len.data(), ent_txt[e], rng[2 * grp_file[g]], keys[e],
                                       min_identity, grp_kind[g] != 0, win[e], dist[e]);
            flag[e] = size[e] ? 1 : 0;
        }
    uint64_t s = 0, q = 0;
    for (uint64_t e = 0; e <= E; ++e) { size_off[e] = s; flag_off[e] = q; s += size[e]; q += flag[e]; }
    const uint64_t total = size_off[E], R = flag_off[E];
    *n_records = R; *n_out_bytes = total;
    if (total > out_cap || R > rec_cap) return 4;
    // compact, .mined offsets, format
    std::vector<uint64_t> rec_off(R + 1);
    std::vector<unsigned char> kind(R + 1);
    for (uint64_t e = 0; e < E; ++e) {
        if (!flag[e]) continue;
        const uint64_t j = flag_off[e];
        rec_partial[j] = ent_txt[e]; rec_winner[j] = (int64_t)win[e]; rec_dist[j] = (int32_t)dist[e];
        rec_off[j] = size_off[e]; kind[j] = grp_kind[grp_of[e]] != 0;
    }
    for (uint32_t j = 0; j <= n_mined; ++j) mined_off[j] = E ? size_off[ent_base[mined_grp[j]]] : 0;
    for (uint64_t j = 0; j < R; ++j) {
        const uint64_t o = (uint64_t)rec_partial[j], w = (uint64_t)rec_winner[j];
        double ident;
        mine_pass((uint64_t)rec_dist[j], len[w], min_identity, ident);
        char b[16];
        const uint32_t bl = smx_out::out_fmt2(ident, b);
        const smx_out::OutMined h = mine_title(data, out_off, o, beg[o], kind[j] != 0, b, bl);
        smx_out::OutWrite wr = {(char *)out + rec_off[j]};
        smx_out::out_mined_emit(h, wr);
        memcpy(wr.p, data + beg[o], out_off[o + 1] - beg[o]);
    }
    return 0;
}

// The routines the CPU tier checks against Python one by one.
uint32_t minesim_fmt2(double x, char *dst) { return smx_out::out_fmt2(x, dst); }
int32_t minesim_k(uint64_t m, double min_identity) { return mine_k(m, min_identity); }
int minesim_pass(uint64_t d, uint64_t m, double min_identity) { double i; return mine_pass(d, m, min_identity, i) ? 1 : 0; }
// the rewritten title line of `title` (without '@' / '\n'), as out_mined_emit writes it; returns its length
uint64_t minesim_title(const unsigned char *title, uint64_t n, int reverse, const char *b, uint32_t b_len, char *dst) {
    const smx_out::OutMined h = smx_out::out_mined_title(title, n, reverse != 0, b, b_len);
    smx_out::OutWrite wr = {dst};
    smx_out::out_mined_emit(h, wr);
    return (uint64_t)(wr.p - dst);
}
// every (m, d) for 1 <= m <= max_m, 0 <= d <= m: the identity text at dst[(m * (m + 1) / 2 + d) * 8] (NUL-padded)
void minesim_fmt2_table(uint32_t max_m, char *dst) {
    for (uint64_t m = 1; m <= max_m; ++m)
        for (uint64_t d = 0; d <= m; ++d) {
            double ident;
            mine_pass(d, m, 0.0, ident);
            char *p = dst + (m * (m + 1) / 2 + d) * 8;
            memset(p, 0, 8);
            smx_out::out_fmt2(ident, p);
        }
}

}  // extern "C"
