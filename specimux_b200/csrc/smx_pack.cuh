// smx_pack.cuh -- the read encoding of smx_batch (include/specimux_b200.h), defined once for the host packer
// (smx_pack_reads / smx_pack_reads_fixed in smx_api.cu) and the device packer (smx_k_pack.cu).  Every routine is
// __host__ __device__, and the device packer's per-thread work items live here too, so a host loop over them
// (tests/packsim) reproduces the kernels' decomposition exactly.
#pragma once
#include "smx_core.cuh"

namespace smx {

// 4-bit code of an input byte: A0 C1 G2 T3 R4 Y5 S6 W7 K8 M9 B10 D11 H12 V13 N14, anything else (lower case, U,
// bytes >= 0x80) kSymOther.  Nibble i of the two words is the code of the letter 'A' + i ('Q' + i).
SMX_HD int read_code(unsigned char ch) {
    const u64 a_to_p = 0xffe9f8ffc2ffb1a0ull, q_to_z = 0xfffffff5f7df364full;
    const u32 i = (u32)ch - 'A';
    if (i >= 26) return kSymOther;
    return (int)(((i < 16 ? a_to_p : q_to_z) >> (4 * (i & 15))) & 15);
}

// symbol of the reverse-complement strand for an input byte (Bio.Seq: complement, case kept, U->A)
SMX_HD int read_code_rc(unsigned char ch) {
    if (ch == 'U') return 0;
    const int c = read_code(ch);
    return c == kSymOther ? kSymOther : sym_complement(c);
}

// Middle clip: a read longer than 2 * clip keeps its first and last `clip` bases (clip 0 = whole reads).
SMX_HD u64 pack_stored_len(u64 len, u32 clip) { return (clip && len > 2ull * clip) ? 2ull * clip : len; }
// stored index i -> source index
SMX_HD u64 pack_src(u64 i, u64 len, u32 clip) {
    return (clip && len > 2ull * clip && i >= clip) ? i + (len - 2ull * clip) : i;
}
// packed4 words per strand of a flagged read
SMX_HD u64 pack_words4(u64 slen) { return (slen + 7) / 8; }

// packed2 word w of a read (symbols 16w .. 16w + 15 of the stored read, 2 bits each; 0 past its end).  A symbol other
// than ACGT is stored as 0 and sets `exotic`.
SMX_HD u32 pack_word2(const unsigned char *s, u64 len, u32 clip, u64 w, bool &exotic) {
    const u64 slen = pack_stored_len(len, clip);
    if (w * 16 >= slen) return 0;
    const u64 lim = slen - w * 16 < 16 ? slen - w * 16 : 16;
    u32 v = 0;
    for (u64 i = 0; i < lim; ++i) {
        int c = read_code(s[pack_src(w * 16 + i, len, clip)]);
        if (c > 3) { exotic = true; c = 0; }
        v |= (u32)c << (2 * i);
    }
    return v;
}

// packed4 word w of strand `strand` (0 = forward, 1 = reverse complement) of a flagged read.  The reverse strand is
// clipped the same way: its stored index x holds the base at stored index slen - 1 - x of the forward strand.
SMX_HD u32 pack_word4(const unsigned char *s, u64 len, u32 clip, int strand, u64 w) {
    const u64 slen = pack_stored_len(len, clip);
    u32 v = 0;
    for (u32 q = 0; q < 8 && w * 8 + q < slen; ++q) {
        const u64 x = w * 8 + q;
        const int c = strand ? read_code_rc(s[pack_src(slen - 1 - x, len, clip)]) : read_code(s[pack_src(x, len, clip)]);
        v |= (u32)c << (4 * q);
    }
    return v;
}

// ------------------------------------------------------------------------------------------------------------------
// Device packer (smx_match_device): reads [0, n) given as bases + seq_off (n + 1 offsets), clip = stride's clip.

// Why a read is refused, in the low two bits of the validation key (read << 2 | reason).
enum PackFault { kPackOk = 0, kPackDescending = 1, kPackPastEnd = 2, kPackTooLong = 3 };

// Validation of read r: its offsets ascend, its end lies within the n_bases bytes of `bases`, it is below 2^31 long.
// The kernels read no base of a batch in which any read fails this.
SMX_HD int pack_check_read(const u64 *seq_off, u64 n_bases, u32 r) {
    const u64 a = seq_off[r], b = seq_off[r + 1];
    if (b < a) return kPackDescending;
    if (b > n_bases) return kPackPastEnd;
    if (b - a > 0x7FFFFFFFull) return kPackTooLong;
    return kPackOk;
}

// Where the packed reads go: reads [r0[l], r0[l + 1]) into lane l's buffers, laid out as lane_upload lays out the
// host-packed batch (read r at word (r - r0[l]) * stride of packed2[l]; packed2[l] ends with one slack word, the next
// lane's first word or 0 after the last read).
constexpr int kPackMaxLanes = 8;
constexpr int kPackTile = 1024;       // reads per tile of the off4 scan
struct PackLanes {
    int n_lanes;
    u32 stride, clip;
    u32 r0[kPackMaxLanes + 1];
    u32 *packed2[kPackMaxLanes];
    u32 *lengths[kPackMaxLanes];
    u64 *off4[kPackMaxLanes];
};

SMX_HD int pack_lane(const PackLanes &d, u32 r) {
    int l = 0;
    while (l + 1 < d.n_lanes && r >= d.r0[l + 1]) ++l;
    return l;
}

// Fixed-stride pass, work item i = (read i / stride, word i % stride): writes that packed2 word (and the lane's slack
// word where it doubles as one), the read's length with word 0, and returns whether the word holds a non-ACGT byte.
SMX_HD bool pack_fixed_item(const unsigned char *bases, const u64 *seq_off, u32 n, const PackLanes &d, u64 i) {
    const u32 r = (u32)(i / d.stride), w = (u32)(i % d.stride);
    const u64 a = seq_off[r], len = seq_off[r + 1] - a;
    bool exotic = false;
    const u32 v = pack_word2(bases + a, len, d.clip, w, exotic);
    const int l = pack_lane(d, r);
    d.packed2[l][(u64)(r - d.r0[l]) * d.stride + w] = v;
    if (w == 0) {
        d.lengths[l][r - d.r0[l]] = (u32)len;
        if (l > 0 && r == d.r0[l]) d.packed2[l - 1][(u64)(r - d.r0[l - 1]) * d.stride] = v;
    }
    if (i + 1 == (u64)n * d.stride) d.packed2[d.n_lanes - 1][(u64)(n - d.r0[d.n_lanes - 1]) * d.stride] = 0;
    return exotic;
}

// packed4 words (both strands) a read takes: 0 unless it is flagged
SMX_HD u64 pack_count4(const u64 *seq_off, u32 clip, bool flagged, u32 r) {
    return flagged ? 2 * pack_words4(pack_stored_len(seq_off[r + 1] - seq_off[r], clip)) : 0;
}

// off4 of read r: its first packed4 word (the exclusive scan of pack_count4 in read order), ~0 when it is not flagged
SMX_HD void pack_set_off4(const PackLanes &d, u32 r, bool flagged, u64 off) {
    const int l = pack_lane(d, r);
    d.off4[l][r - d.r0[l]] = flagged ? off : ~0ull;
}

// Side stream, word w in [0, 2 * n4) of flagged read r: forward strand words, then the reverse-complement strand's.
SMX_HD void pack_side_word(const unsigned char *bases, const u64 *seq_off, const PackLanes &d, u32 *packed4, u32 r, u64 w) {
    const u64 a = seq_off[r], len = seq_off[r + 1] - a;
    const u64 n4 = pack_words4(pack_stored_len(len, d.clip));
    const int l = pack_lane(d, r);
    const u64 off = d.off4[l][r - d.r0[l]];
    packed4[off + w] = w < n4 ? pack_word4(bases + a, len, d.clip, 0, w) : pack_word4(bases + a, len, d.clip, 1, w - n4);
}

}  // namespace smx
