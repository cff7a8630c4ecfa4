// smx_mine.cuh -- the work items of specimine on device files (smx_mine_device, smx_k_mine_device.cu), defined once for
// the kernels and the host loops of tests/minesim: where an output's sequence lies in its file, a full read's search
// limit and (lanes, words per lane) class, the decision on a best match and the size of a mined record.  The grouped
// search's work item (HwItem) and class rule live here too, so smx_hw_best_grouped plans with the same routines.
// Every routine is __host__ __device__; nothing here needs smx_core.cuh.
#pragma once
#include <stdint.h>

#include "smx_out.cuh"

namespace smx_mine {

typedef uint32_t u32;
typedef uint64_t u64;
typedef int32_t i32;

// ---------------------------------------------------------------------------------------------------------------------
// Grouped best match (k_hw_best): one work item = a pattern and a run of n consecutive entries [e_lo, e_lo + n) of its
// group's text list; rank = the pattern's index within its group.  Items of one launch are all of one (SW, W) class.
struct HwItem { u32 pat, rank; u64 e_lo; u32 n, pad; };

constexpr int kHwClasses = 17;
// the (lanes per segment, words per lane) classes k_hw_best is instantiated for, as sw * 8 + w
SMX_HD int hw_class_code(int k) {
    const unsigned short codes[kHwClasses] = {3 * 8 + 1, 3 * 8 + 2, 3 * 8 + 3, 4 * 8 + 1, 4 * 8 + 2, 4 * 8 + 3, 4 * 8 + 4,
                                              5 * 8 + 2, 5 * 8 + 4, 6 * 8 + 3, 8 * 8 + 3, 8 * 8 + 4, 10 * 8 + 4,
                                              16 * 8 + 3, 16 * 8 + 4, 32 * 8 + 3, 32 * 8 + 4};
    return codes[k];
}

// (lanes per segment, words per lane) of the grouped kernel for a pattern of `words` 32-bit words: the fewest lane-steps
// per text, (W + 1) / (32 / SW) -- W words of Myers arithmetic plus about one word's worth of cross-lane work (two
// ballots, two shuffles) per column, shared by the 32 / SW texts of a warp -- ties to fewer words per lane, then fewer
// lanes.  Segment widths are those long_carry_in<> is checked for.  A 700-nt pattern (22 words) runs as SW = 8, W = 3:
// four texts per warp, 8 % of the lane-words padding, where k_hw_distance's power-of-two SW = 32 pads 31 %.
SMX_HD void hw_best_class(int words, int *sw, int *w) {
    const int kSW[8] = {3, 4, 5, 6, 8, 10, 16, 32};
    int bs = 32, bw = 4;
    for (int cw = 1; cw <= 4; ++cw)
        for (int i = 0; i < 8; ++i) {
            const int cs = kSW[i];
            if (cs * cw < words) continue;
            // (cw + 1) / (32 / cs) < (bw + 1) / (32 / bs), exactly
            if ((cw + 1) * (32 / bs) < (bw + 1) * (32 / cs)) { bs = cs; bw = cw; }
        }
    *sw = bs; *w = bw;
}

// entries one work item covers
SMX_HD u32 hw_best_chunk(int sw) { return 16u * (u32)(32 / sw); }

// index into the class list of a pattern of m >= 1 bytes (m <= 4096)
SMX_HD int hw_class_of(u64 m) {
    int sw, w;
    hw_best_class((int)((m + 31) / 32), &sw, &w);
    for (int k = 0; k < kHwClasses; ++k)
        if (hw_class_code(k) == sw * 8 + w) return k;
    return -1;
}

// ---------------------------------------------------------------------------------------------------------------------
// Float64 as Python computes it: no contraction into fused multiply-adds.
SMX_HD double py_mul(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    volatile double r = a * b;
    return r;
#endif
}
SMX_HD double py_sub(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dsub_rn(a, b);
#else
    volatile double r = a - b;
    return r;
#endif
}
SMX_HD double py_div(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __ddiv_rn(a, b);
#else
    volatile double r = a / b;
    return r;
#endif
}

// specimine's search limit of a full read of m bytes: int(m * (1 - min_identity)) (clamped to the int32 range)
SMX_HD i32 mine_k(u64 m, double min_identity) {
    const double x = py_mul((double)m, py_sub(1.0, min_identity));
    if (!(x > -2147483648.0)) return INT32_MIN;
    if (x >= 2147483647.0) return INT32_MAX;
    return (i32)x;                                              // truncation, as int() does
}

// identity = 1 - d / m; mined when identity >= min_identity and identity > 0 (mine_files)
SMX_HD bool mine_pass(u64 d, u64 m, double min_identity, double &identity) {
    identity = py_sub(1.0, py_div((double)d, (double)m));
    return identity >= min_identity && identity > 0;
}

// The best pattern of an entry from its key, (floor(d * 2^40 / m) << 23) | rank: false when no pattern qualified.
constexpr u32 kRankBits = 23;
SMX_HD bool mine_key_rank(unsigned long long key, u32 &rank) {
    if (key == ~0ull) return false;
    rank = (u32)(key & ((1u << kRankBits) - 1));
    return true;
}
// d = ceil(q * m / 2^40), since q * m lies in (d * 2^40 - m, d * 2^40]
SMX_HD u64 mine_key_dist(unsigned long long key, u64 m) { return ((key >> kRankBits) * m + (1ull << 40) - 1) >> 40; }

// ---------------------------------------------------------------------------------------------------------------------
// Locate.  Faults name (file, output within the file) as file << 35 | output << 3 | fault; the least key is reported.
enum MineFault {
    kMineOk = 0,
    kMineFileRange = 1,     // the file's byte range does not start and end on output boundaries
    kMineOffsets = 2,       // output offsets descend or pass the data
    kMineRecord = 3,        // not a FASTQ record: '@' title '\n' sequence '\n' '+' '\n' qualities '\n'
    kMineLong = 4,          // a full read longer than 4,096 bytes
    kMineCodes = 5,         // a full read holding more than 64 distinct byte values
    kMineRank = 6,          // a full read beyond the first 2^23 of its file: the key's rank field holds 23 bits
};
constexpr u64 kMineMaxFiles = 1ull << 29;
constexpr u64 kMineMaxPattern = 4096;
constexpr int kMineMaxCodes = 64;
constexpr u64 kMineMaxRank = 1ull << 23;           // full reads per group, as smx_hw_best_grouped allows (kRankBits)

SMX_HD u64 mine_fault_key(u64 file, u64 output, int fault) { return file << 35 | output << 3 | (u64)fault; }

// the first index i in [0, n] with off[i] >= v
SMX_HD u64 mine_lower_bound(const u64 *off, u64 n, u64 v) {
    u64 lo = 0, hi = n;
    while (lo < hi) {
        const u64 mid = (lo + hi) >> 1;
        if (off[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Outputs [o0, o1) of file f: the outputs whose offsets are file_off[f] and file_off[f + 1].  Returns a fault key or ~0.
SMX_HD u64 mine_locate_file(const u64 *out_off, u64 n_outputs, const u64 *file_off, u64 f, u64 &o0, u64 &o1) {
    o0 = mine_lower_bound(out_off, n_outputs, file_off[f]);
    o1 = mine_lower_bound(out_off, n_outputs, file_off[f + 1]);
    if (out_off[o0] != file_off[f] || out_off[o1] != file_off[f + 1] || o1 < o0 || o1 - o0 >= (1ull << 32)) {
        o0 = o1 = 0;
        return mine_fault_key(f, 0, kMineFileRange);
    }
    return ~0ull;
}

// Output o's sequence: bytes [beg, beg + len) of data, its qualities the same length after "\n+\n".  The title is
// [out_off[o] + 1, beg - 1).  Returns a MineFault.
SMX_HD int mine_locate_output(const unsigned char *data, u64 n_data, const u64 *out_off, u64 o, u64 &beg, u32 &len) {
    beg = 0; len = 0;
    const u64 a = out_off[o], b = out_off[o + 1];
    if (b < a || b > n_data) return kMineOffsets;
    if (b - a < 6 || data[a] != '@') return kMineRecord;
    u64 nl = a + 1;
    while (nl < b && data[nl] != '\n') ++nl;
    const u64 rest = nl < b ? b - nl - 1 : 0;              // seq '\n' '+' '\n' qual '\n'
    if (nl >= b || rest < 4 || (rest & 1) || (rest - 4) / 2 >= (1ull << 31)) return kMineRecord;
    const u64 n = (rest - 4) / 2, s = nl + 1;
    if (data[s + n] != '\n' || data[s + n + 1] != '+' || data[s + n + 2] != '\n' || data[b - 1] != '\n') return kMineRecord;
    beg = s; len = (u32)n;
    return kMineOk;
}

// The 256-bit set of byte values of p[0 .. m), accumulated into mask (8 words).
SMX_HD void mine_byte_set(const unsigned char *p, u64 lo, u64 hi, u64 step, u32 mask[8]) {
    for (u64 i = lo; i < hi; i += step) mask[p[i] >> 5] |= 1u << (p[i] & 31);
}
SMX_HD int mine_popc8(const u32 mask[8]) {
    int n = 0;
    for (int k = 0; k < 8; ++k) {
        u32 v = mask[k];
        while (v) { v &= v - 1; ++n; }
    }
    return n;
}

// Work items of one pattern (a full read of m bytes) over its group's `entries` entries; 0 for an empty pattern.
SMX_HD u64 mine_items(u64 m, u64 entries, int &cls) {
    cls = -1;
    if (!m || !entries) return 0;
    cls = hw_class_of(m);
    int sw, w;
    hw_best_class((int)((m + 31) / 32), &sw, &w);
    const u64 chunk = hw_best_chunk(sw);
    return (entries + chunk - 1) / chunk;
}

// ---------------------------------------------------------------------------------------------------------------------
// Decide + format.  A mined record is the rewritten title line (smx_out::out_mined_emit) followed by the partial
// record's bytes after its title line: sequence, "\n+\n", qualities, '\n'.

// The title line of partial output o (title at data[out_off[o] + 1 .. beg - 1)), with b the identity text.
SMX_HD smx_out::OutMined mine_title(const unsigned char *data, const u64 *out_off, u64 o, u64 beg, bool reverse,
                                    const char *b, u32 b_len) {
    const u64 t0 = out_off[o] + 1;
    return smx_out::out_mined_title(data + t0, beg - 1 - t0, reverse, b, b_len);
}

// Decision on entry e: its text is output `txt`, the winner's length is known from its output.  Returns the mined
// record's size (0 when not mined), with the winner's rank and the distance.
SMX_HD u64 mine_decide_item(const unsigned char *data, const u64 *out_off, const u64 *beg, const u32 *len, u64 txt,
                            u64 pat0, unsigned long long key, double min_identity, bool reverse, u64 &winner, u64 &dist) {
    u32 rank;
    winner = ~0ull; dist = 0;
    if (!mine_key_rank(key, rank)) return 0;
    const u64 w = pat0 + rank, m = len[w], d = mine_key_dist(key, m);
    double ident;
    if (!mine_pass(d, m, min_identity, ident)) return 0;
    winner = w; dist = d;
    char b[16];
    const u32 bl = smx_out::out_fmt2(ident, b);
    return smx_out::out_mined_len(mine_title(data, out_off, txt, beg[txt], reverse, b, bl)) + (out_off[txt + 1] - beg[txt]);
}

}  // namespace smx_mine
