// smx_out.cuh -- the output rules of the per-specimen tree, defined once for the host reader and writer (smx_io.cpp,
// compiled by g++) and the device demultiplexer and file formatter (smx_demux_device, smx_demux_files_device,
// smx_k_demux.cu): the id of a title, the header line and length of a formatted record, the Python slice of a trim
// extent, Biopython's ambiguous-DNA complement, the destination key of a record with its range checks, and the
// per-record and per-tile work items of the device kernels, so that a host loop over them (tests/demuxsim,
// tests/filesim) runs the kernels' decomposition exactly.  Every routine is __host__ __device__; nothing here needs
// smx_core.cuh.
#pragma once
#include <stdint.h>
#include <string.h>

#include "../../include/specimux_b200.h"

#ifndef SMX_HD
#if defined(__CUDACC__)
#define SMX_HD __host__ __device__ __forceinline__
#else
#define SMX_HD inline
#endif
#endif

namespace smx_out {

typedef uint32_t u32;
typedef uint64_t u64;

// ---------------------------------------------------------------------------------------------------------------------
// Record text: the reader's id rule, the header line and the length of a formatted record (smx_writer::format).

// Python str whitespace (str.strip / str.split(None) on text decoded as UTF-8): the byte length of the whitespace
// character starting at p, 0 if none.
SMX_HD int out_ws_at(const unsigned char *p, const unsigned char *end) {
    const unsigned char c = *p;
    if (c < 0x80) return ((c >= 9 && c <= 13) || (c >= 28 && c <= 32)) ? 1 : 0;
    if (c == 0xC2 && p + 1 < end && (p[1] == 0x85 || p[1] == 0xA0)) return 2;
    if (p + 2 < end) {
        if (c == 0xE1 && p[1] == 0x9A && p[2] == 0x80) return 3;                       // U+1680
        if (c == 0xE2 && p[1] == 0x80 && (p[2] <= 0x8A || p[2] == 0xA8 || p[2] == 0xA9 || p[2] == 0xAF) && p[2] >= 0x80) return 3;
        if (c == 0xE2 && p[1] == 0x81 && p[2] == 0x9F) return 3;                       // U+205F
        if (c == 0xE3 && p[1] == 0x80 && p[2] == 0x80) return 3;                       // U+3000
    }
    return 0;
}

// record.id of a title: its first whitespace-delimited token, bytes [a, b) of the title.
SMX_HD void out_title_id(const unsigned char *t, u64 len, u64 &a, u64 &b) {
    const unsigned char *e = t + len, *p = t;
    for (int k; p < e && (k = out_ws_at(p, e)) != 0;) p += k;
    const unsigned char *q = p;
    while (q < e && !out_ws_at(q, e)) ++q;
    a = (u64)(p - t); b = (u64)(q - t);
}

// distance_code (models.py:206-218) of one int8 distance: its decimal digits, 'X' when negative, as up to three characters
// packed little-endian into *t.  Returns the length.
SMX_HD u32 out_dist_text(int v, u32 *t) {
    if (v < 0) { *t = 'X'; return 1; }
    u32 w = 0, n = 0;
    do { w = (w << 8) | (u32)('0' + v % 10); v /= 10; ++n; } while (v && n < 3);
    *t = w;
    return n;
}

// The header line of a record (OutputManager.write_sequence, io_utils.py:245-256):
//   <lead><id> <d0>,<d1>,<d2>,<d3> pool=<pool> primers=<p1>+<p2> <sample>\n
// without the pool / primers part in the console form (files == false).
struct OutHeader {
    char lead;                      // '@' FASTQ, '>' FASTA
    bool files;
    const int8_t *dist;             // the record's four distances
    const char *id, *pool, *p1, *p2, *sample;
    u64 id_len, pool_len, p1_len, p2_len, sample_len;
};

// Hands the header to put piece by piece: put(const char *, u64) for strings, put.chars(w, n) for n <= 4 characters
// packed little-endian into w.
template <class Put> SMX_HD void out_header_emit(const OutHeader &h, Put &put) {
    put.chars((u32)(unsigned char)h.lead, 1);
    put(h.id, h.id_len);
    for (int d = 0; d < 4; ++d) {
        u32 t;
        const u32 k = out_dist_text(h.dist[d], &t);
        put.chars((d ? ',' : ' ') | t << 8, k + 1);
    }
    if (h.files) {
        put(" pool=", 6); put(h.pool, h.pool_len);
        put(" primers=", 9); put(h.p1, h.p1_len); put.chars('+', 1); put(h.p2, h.p2_len);
    }
    put.chars(' ', 1); put(h.sample, h.sample_len); put.chars('\n', 1);
}

struct OutCount {
    u64 n;
    SMX_HD void operator()(const char *, u64 k) { n += k; }
    SMX_HD void chars(u32, u32 k) { n += k; }
};
struct OutWrite {
    char *p;
    SMX_HD void operator()(const char *s, u64 k) { memcpy(p, s, k); p += k; }
    SMX_HD void chars(u32 w, u32 k) { for (u32 j = 0; j < k; ++j) p[j] = (char)(w >> (8 * j)); p += k; }
};
// Keeps the bytes [lo, hi) of what is put, at dst[0 .. hi - lo).
struct OutWindow {
    u64 pos, lo, hi;
    unsigned char *dst;
    SMX_HD void operator()(const char *s, u64 k) {
        const u64 a = pos > lo ? pos : lo, b = pos + k < hi ? pos + k : hi;
        for (u64 j = a; j < b; ++j) dst[j - lo] = (unsigned char)s[j - pos];
        pos += k;
    }
    SMX_HD void chars(u32 w, u32 k) {
        for (u32 j = 0; j < k; ++j)
            if (pos + j >= lo && pos + j < hi) dst[pos + j - lo] = (unsigned char)(w >> (8 * j));
        pos += k;
    }
};

SMX_HD u64 out_header_len(const OutHeader &h) { OutCount c = {0}; out_header_emit(h, c); return c.n; }
// Writes the header at dst; returns its length.
SMX_HD u64 out_header_write(const OutHeader &h, char *dst) { OutWrite w = {dst}; out_header_emit(h, w); return (u64)(w.p - dst); }

// Bytes of a formatted record with an n-byte sequence: header, sequence, '\n' and, for FASTQ, "+\n", qualities, '\n'.
SMX_HD u64 out_record_len(u64 header, u64 n, bool fastq) { return header + n + 1 + (fastq ? n + 3 : 0); }
// Its sequence length, from the record and header lengths.
SMX_HD u64 out_record_body(u64 len, u64 header, bool fastq) { return fastq ? (len - header - 4) / 2 : len - header - 1; }

// Python slice bounds seq[s:e] for non-None ints.
SMX_HD void py_slice(long long s, long long e, long long len, u64 &a, u64 &b) {
    if (s < 0) { s += len; if (s < 0) s = 0; } else if (s > len) s = len;
    if (e < 0) { e += len; if (e < 0) e = 0; } else if (e > len) e = len;
    if (e < s) e = s;
    a = (u64)s; b = (u64)e;
}

// ---------------------------------------------------------------------------------------------------------------------
// Bio.Seq's ambiguous-DNA complement (ACGTMRWSYKVHDBXN -> TGCAKYWSRMBDHVXN, U -> A, case kept, anything else unchanged),
// four bytes at a time.  A byte in 0x40..0x7F keeps its top three bits and maps its low five through a 32-entry table;
// the table is four 8-byte rows picked by bits 3 and 4, each read with one byte permute.  Bytes outside 0x40..0x7F pass.

SMX_HD u32 byte_perm(u32 x, u32 y, u32 s) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(x, y, s);
#else
    const u64 v = (u64)y << 32 | x;
    u32 r = 0;
    for (int k = 0; k < 4; ++k) r |= (u32)((v >> (8 * ((s >> (4 * k)) & 7))) & 0xFF) << (8 * k);
    return r;
#endif
}

// a where m is 0, b where m is 1
SMX_HD u32 bit_select(u32 a, u32 b, u32 m) { return (a & ~m) | (b & m); }

SMX_HD u32 dna_complement4(u32 x) {
    //                    low 5 bits:  0 '@'  1 A>T  2 B>V  3 C>G  4 D>H  5 E  6 F  7 G>C
    const u32 t0_lo = 0x07161400u, t0_hi = 0x03060508u;
    //                                 8 H>D  9 I  10 J  11 K>M  12 L  13 M>K  14 N  15 O
    const u32 t1_lo = 0x0D0A0904u, t1_hi = 0x0F0E0B0Cu;
    //                                16 P  17 Q  18 R>Y  19 S  20 T>A  21 U>A  22 V>B  23 W
    const u32 t2_lo = 0x13191110u, t2_hi = 0x17020101u;
    //                                24 X  25 Y>R  26 Z  27..31
    const u32 t3_lo = 0x1B1A1218u, t3_hi = 0x1F1E1D1Cu;
    const u32 t = x & 0x07070707u, u = t | (t >> 4);
    const u32 sel = (u & 0xFFu) | ((u >> 8) & 0xFF00u);              // nibble k = bits 0..2 of byte k
    const u32 m3 = ((x >> 3) & 0x01010101u) * 0xFFu, m4 = ((x >> 4) & 0x01010101u) * 0xFFu;
    const u32 lo = bit_select(byte_perm(t0_lo, t0_hi, sel), byte_perm(t1_lo, t1_hi, sel), m3);
    const u32 hi = bit_select(byte_perm(t2_lo, t2_hi, sel), byte_perm(t3_lo, t3_hi, sel), m3);
    const u32 mapped = bit_select(lo, hi, m4) | (x & 0xE0E0E0E0u);
    const u32 letter = (((x & (~x >> 1)) >> 6) & 0x01010101u) * 0xFFu;  // bit 6 set, bit 7 clear
    return bit_select(x, mapped, letter);
}

SMX_HD unsigned char dna_complement(unsigned char ch) { return (unsigned char)(dna_complement4(ch) & 0xFF); }

// ---------------------------------------------------------------------------------------------------------------------
// Destination of a record: OutputManager._make_filename (io_utils.py:206-220) as the writer's planning pass resolves it.

// Table sizes the record indices are checked against (the name lists of smx_names / the context's tables).
struct OutCounts { u32 n_specimens, n_b1, n_b2, n_pools, n_primers; };

// Which name table's count differs from the context's (0 specimens, 1 b1, 2 b2, 3 pools, 4 primers), -1 when none.
SMX_HD int out_names_mismatch(const OutCounts &n, const u32 counts[5]) {
    const u32 want[5] = {n.n_specimens, n.n_b1, n.n_b2, n.n_pools, n.n_primers};
    for (int k = 0; k < 5; ++k)
        if (counts[k] != want[k]) return k;
    return -1;
}

// Why a record is refused (low three bits of a validation key: record << 3 | fault).
enum OutFault { kOutOk = 0, kOutRead = 1, kOutSpecimen = 2, kOutB1 = 3, kOutB2 = 4, kOutPool = 5, kOutP1 = 6, kOutP2 = 7 };

// top: 0 full, 1 partial, 2 unknown.  kind: 0 specimen, 1 b1, 2 b2, 3 unknown (sample index 0).  pool / p1 / p2:
// index + 1, 0 = "unknown".  Trim-empty records go to unknown/unknown/unknown-unknown/unknown.
struct OutDest { u32 top, kind, sample, pool, p1, p2; };

// Resolves and range-checks a record's destination; returns an OutFault (the first failing check, in the writer's order).
SMX_HD int out_dest(const smx_record &rec, const OutCounts &n, OutDest &d) {
    d.top = 2; d.kind = 3; d.sample = 0; d.pool = d.p1 = d.p2 = 0;
    if (rec.trim_empty) return kOutOk;
    const uint8_t res = rec.resolution;
    if (res == SMX_RES_FULL_MATCH || res == SMX_RES_DEREPLICATED_FULL || res == SMX_RES_MULTIPLE_SPECIMENS) {
        if (rec.sample < 0 || (u32)rec.sample >= n.n_specimens) return kOutSpecimen;
        d.kind = 0;
    } else if (res == SMX_RES_PARTIAL_FORWARD) {
        if (rec.sample < 0 || (u32)rec.sample >= n.n_b1) return kOutB1;
        d.kind = 1;
    } else if (res == SMX_RES_PARTIAL_REVERSE) {
        if (rec.sample < 0 || (u32)rec.sample >= n.n_b2) return kOutB2;
        d.kind = 2;
    }
    if (d.kind < 3) d.sample = (u32)rec.sample;
    if (rec.pool >= 0) { if ((u32)rec.pool >= n.n_pools) return kOutPool; d.pool = (u32)rec.pool + 1; }
    if (rec.p1 >= 0) { if ((u32)rec.p1 >= n.n_primers) return kOutP1; d.p1 = (u32)rec.p1 + 1; }
    if (rec.p2 >= 0) { if ((u32)rec.p2 >= n.n_primers) return kOutP2; d.p2 = (u32)rec.p2 + 1; }
    d.top = res == SMX_RES_UNKNOWN ? 2 : (res == SMX_RES_PARTIAL_FORWARD || res == SMX_RES_PARTIAL_REVERSE) ? 1 : 0;
    return kOutOk;
}

// The 64-bit key of a primary file: top (2 bits) | pool (10) | p1 (8) | p2 (8) | 4 zero bits | kind (2) | sample (30).
constexpr u32 kOutMaxPools = 1023;
constexpr u32 kOutMaxSamples = 1u << 30;
SMX_HD u64 out_key(const OutDest &d) {
    return ((u64)d.top << 62) | ((u64)d.pool << 52) | ((u64)d.p1 << 44) | ((u64)d.p2 << 36) | ((u64)d.kind << 30) | d.sample;
}
// Key of the pool-level copy (full/<pool>/<sample>) that full matches also go to: top 3, no primers.
SMX_HD u64 out_pool_key(const OutDest &d) { return (3ull << 62) | ((u64)d.pool << 52) | ((u64)d.kind << 30) | d.sample; }
SMX_HD bool out_has_pool_copy(const smx_record &rec) {
    return !rec.trim_empty && (rec.resolution == SMX_RES_FULL_MATCH || rec.resolution == SMX_RES_DEREPLICATED_FULL);
}
// Slice [a, b) of the oriented read that is written: the trim extent, the whole read for trim-empty records.
SMX_HD void out_slice(const smx_record &rec, long long len, u64 &a, u64 &b) {
    if (rec.trim_empty) { a = 0; b = (u64)len; } else py_slice(rec.trim_start, rec.trim_end, len, a, b);
}

// ---------------------------------------------------------------------------------------------------------------------
// Device demultiplexer (smx_demux_device).  The sort runs on a compact form of the key: the same fields in the same
// order, each only as wide as the context's tables need, so that the radix sort passes over only the bits in use.

SMX_HD u32 bits_for(u64 v) { u32 b = 0; while (v >> b) ++b; return b; }     // bits that hold 0..v

struct OutShape { u32 pool_bits, primer_bits, sample_bits, total_bits; };
SMX_HD OutShape out_shape(const OutCounts &n) {
    OutShape s;
    u32 m = n.n_specimens > n.n_b1 ? n.n_specimens : n.n_b1;
    m = m > n.n_b2 ? m : n.n_b2;
    s.pool_bits = bits_for(n.n_pools); s.primer_bits = bits_for(n.n_primers); s.sample_bits = bits_for(m ? m - 1 : 0);
    s.total_bits = 2 + s.pool_bits + 2 * s.primer_bits + 2 + s.sample_bits;
    return s;
}
SMX_HD u64 out_sort_key(const OutDest &d, const OutShape &s) {
    u64 k = d.top;
    k = (k << s.pool_bits) | d.pool;
    k = (k << s.primer_bits) | d.p1;
    k = (k << s.primer_bits) | d.p2;
    k = (k << 2) | d.kind;
    return (k << s.sample_bits) | d.sample;
}
SMX_HD u64 out_key_of_sort(u64 k, const OutShape &s) {
    OutDest d;
    d.sample = (u32)(k & ((1ull << s.sample_bits) - 1)); k >>= s.sample_bits;
    d.kind = (u32)(k & 3); k >>= 2;
    d.p2 = (u32)(k & ((1ull << s.primer_bits) - 1)); k >>= s.primer_bits;
    d.p1 = (u32)(k & ((1ull << s.primer_bits) - 1)); k >>= s.primer_bits;
    d.pool = (u32)(k & ((1ull << s.pool_bits) - 1)); k >>= s.pool_bits;
    d.top = (u32)k;
    return out_key(d);
}

constexpr u64 kOutReverse = 1ull << 63;

// Plan, work item r = record r: validation (returns record << 3 | fault, or ~0 when the record passes), its sort key,
// output length, and the position of its first output byte in `bases` (the LAST byte of the reversed source run, with
// kOutReverse, for reverse records).  Reads no base.
SMX_HD int demux_plan_record(const smx_record &rec, const u64 *seq_off, u32 n_reads, const OutCounts &n, OutDest &d, u64 &a,
                             u64 &b, u64 &src) {
    d = OutDest{};
    const int fault = rec.read >= n_reads ? (int)kOutRead : out_dest(rec, n, d);
    a = b = src = 0;
    if (!fault) {
        const u64 s0 = seq_off[rec.read];
        const long long len = (long long)(seq_off[rec.read + 1] - s0);
        out_slice(rec, len, a, b);
        src = rec.reverse ? ((s0 + (u64)len - 1 - a) | kOutReverse) : s0 + a;
    }
    return fault;
}

SMX_HD u64 demux_plan_item(const smx_record *records, const u64 *seq_off, u32 n_reads, const OutCounts &n, const OutShape &s,
                           u64 r, u64 *sort_key, u32 *len_out, u64 *src) {
    OutDest d;
    u64 a, b;
    const int fault = demux_plan_record(records[r], seq_off, n_reads, n, d, a, b, src[r]);
    sort_key[r] = fault ? 0 : out_sort_key(d, s);
    len_out[r] = (u32)(b - a);
    return fault ? (r << 3 | (u64)fault) : ~0ull;
}

// Gather, work item i = output i (after the sort of slots; slot >> shift is the record): record index, output length
// (scanned in place into out_off next; out_off[n] = 0 so that the scan leaves the total there), source position.
template <class Len>
SMX_HD void demux_gather_item(const u32 *sorted_rec, const Len *len, const u64 *src, u64 n, u64 i, u64 *order, u64 *out_off,
                              u64 *out_src, u32 shift = 0) {
    const u32 slot = sorted_rec[i], r = slot >> shift;
    order[i] = r;
    out_off[i] = len[slot];
    out_src[i] = src[r];
    if (i + 1 == n) out_off[n] = 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// Device file formatter (smx_demux_files_device): every record gives slot 2r, its primary file's record, and slot
// 2r + 1, its pool-level copy or -- when it has none -- an empty slot whose compact key (out_empty_slot) sorts after
// every file.  Each output is the complete formatted record, header included.

// The name tables in one blob: specimen ids, b1 ids, b2 ids, pools, primer names, in that order; name k is
// bytes[off[k] .. off[k + 1]).
struct OutNames {
    const char *bytes;
    const u64 *off;
    OutCounts n;
};

SMX_HD u64 out_empty_slot(const OutShape &s) { return 1ull << s.total_bits; }

// The header of a (validated) record whose destination is d, with the id at title[0 .. id_len).
SMX_HD OutHeader out_header_of(const smx_record &rec, const OutDest &d, const OutNames &nm, const char *id, u64 id_len, bool fastq) {
    OutHeader h;
    h.lead = fastq ? '@' : '>';
    h.files = true;
    h.dist = rec.dist;
    h.id = id; h.id_len = id_len;
    auto name = [&](bool known, u64 k, const char *&p, u64 &len) {
        if (known) { p = nm.bytes + nm.off[k]; len = nm.off[k + 1] - nm.off[k]; } else { p = "unknown"; len = 7; }
    };
    const u64 b1 = nm.n.n_specimens, b2 = b1 + nm.n.n_b1, pools = b2 + nm.n.n_b2, primers = pools + nm.n.n_pools;
    name(d.kind < 3, (d.kind == 0 ? 0 : d.kind == 1 ? b1 : b2) + d.sample, h.sample, h.sample_len);
    name(d.pool != 0, pools + d.pool - 1, h.pool, h.pool_len);
    name(d.p1 != 0, primers + d.p1 - 1, h.p1, h.p1_len);
    name(d.p2 != 0, primers + d.p2 - 1, h.p2, h.p2_len);
    return h;
}

// Files plan, work item r = record r: validation (as demux_plan_item; records are checked in the same order), the
// compact keys and output lengths of slots 2r and 2r + 1, and per record the source position, header length and id
// position in `titles`.  Reads the title (id bounds), not the bases; a title whose offsets descend or end past the
// titles is not read (the offsets check refuses the call for it).
struct FilesPlan {
    const unsigned char *titles;
    const u64 *title_off;
    u64 n_title_bytes;
    OutNames names;
    bool fastq;
};

SMX_HD u64 files_plan_item(const smx_record *records, const u64 *seq_off, u32 n_reads, const FilesPlan &f, const OutShape &s,
                           u64 r, u64 *sort_key, u64 *len, u64 *src, u64 *hdr, u64 *id_pos) {
    const smx_record &rec = records[r];
    OutDest d;
    u64 a, b;
    const int fault = demux_plan_record(rec, seq_off, n_reads, f.names.n, d, a, b, src[r]);
    u64 ia = 0, ib = 0, t0 = 0;
    if (!fault) {
        const u64 t1 = f.title_off[rec.read + 1];
        t0 = f.title_off[rec.read];
        if (t0 <= t1 && t1 <= f.n_title_bytes) out_title_id(f.titles + t0, t1 - t0, ia, ib);
    }
    const u64 h = fault ? 0 : out_header_len(out_header_of(rec, d, f.names, nullptr, ib - ia, f.fastq));
    const u64 n = out_record_len(h, b - a, f.fastq);
    hdr[r] = h;
    id_pos[r] = t0 + ia;
    sort_key[2 * r] = fault ? 0 : out_sort_key(d, s);
    len[2 * r] = n;
    const bool copy = !fault && out_has_pool_copy(rec);
    OutDest pd = d;
    pd.top = 3; pd.p1 = pd.p2 = 0;
    sort_key[2 * r + 1] = copy ? out_sort_key(pd, s) : out_empty_slot(s);
    len[2 * r + 1] = copy ? n : 0;
    return fault ? (r << 3 | (u64)fault) : ~0ull;
}

// Copy: output bytes go in chunks of kDemuxChunk, chunk c of a buffer covering output bytes [16c - m, 16c - m + 16)
// with m = the buffer's address mod 16, so every full chunk is one aligned 16-byte store.  tile_chunks chunks make a
// tile; tile_first[t] is the output that holds byte max(0, t * tile_bytes - 16), and every byte of tile t lies in an
// output of [tile_first[t], tile_first[t + 2]].  tile_first has n_tiles + 2 entries.
constexpr u32 kDemuxChunk = 16;

SMX_HD u32 demux_misalign(const void *p) { return (u32)((uintptr_t)p & (kDemuxChunk - 1)); }
SMX_HD u64 demux_chunks(u64 total, const void *p) { return (total + demux_misalign(p) + kDemuxChunk - 1) / kDemuxChunk; }

// Tile marks, work item i = output i: tile_first[t] = i for every tile boundary inside output i (and, for the last
// output, every boundary at or past the end).
SMX_HD void demux_tile_item(const u64 *out_off, u64 n_out, u64 tile_bytes, u64 n_marks, u64 i, u64 *tile_first) {
    const u64 a = out_off[i], b = out_off[i + 1];
    // boundary t sits at max(0, t * tile_bytes - 16): the first t at or past position p
    auto first_at = [&](u64 p) { return p == 0 ? 0 : (p + 16 + tile_bytes - 1) / tile_bytes; };
    u64 t0 = first_at(a), t1 = i + 1 == n_out ? n_marks : first_at(b);
    if (a == b && i + 1 < n_out) return;
    if (t1 > n_marks) t1 = n_marks;
    for (u64 t = t0; t < t1; ++t) tile_first[t] = i;
}

// The output holding byte p: the largest i in [lo, hi] with out_off[i] <= p.
SMX_HD u64 demux_find(const u64 *out_off, u64 lo, u64 hi, u64 p) {
    while (lo < hi) {
        const u64 mid = (lo + hi + 1) >> 1;
        if (out_off[mid] <= p) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// 16 source bytes from p (any alignment) as four little-endian words
SMX_HD void demux_load16(const unsigned char *p, u32 w[4]) {
#if defined(__CUDA_ARCH__)
    const u32 *q = (const u32 *)((uintptr_t)p & ~(uintptr_t)3);
    const u32 sh = (u32)((uintptr_t)p & 3);
    const u32 x0 = q[0], x1 = q[1], x2 = q[2], x3 = q[3], x4 = sh ? q[4] : 0;
    w[0] = __funnelshift_r(x0, x1, 8 * sh); w[1] = __funnelshift_r(x1, x2, 8 * sh);
    w[2] = __funnelshift_r(x2, x3, 8 * sh); w[3] = __funnelshift_r(x3, x4, 8 * sh);
#else
    memcpy(w, p, 16);
#endif
}

SMX_HD void demux_store16(unsigned char *p, const u32 w[4]) {
#if defined(__CUDA_ARCH__)
    *(uint4 *)p = make_uint4(w[0], w[1], w[2], w[3]);
#else
    memcpy(p, w, 16);
#endif
}

// Byte j of the run of source bytes that starts at position s (demux_plan_item; kOutReverse: running backwards).
SMX_HD unsigned char demux_src_byte(const unsigned char *src, u64 s, u64 j, bool complement) {
    if (!(s & kOutReverse)) return src[s + j];
    const unsigned char ch = src[(s & ~kOutReverse) - j];
    return complement ? dna_complement(ch) : ch;
}

// What a full chunk inside one output copies: 16 bytes from p (forward), the 16 bytes ending at p reversed (and
// complemented), or 16 fill bytes when p is null.
struct DemuxRun {
    const unsigned char *p;
    bool reverse, complement;
    unsigned char fill;
};

SMX_HD DemuxRun demux_run(const unsigned char *src, u64 s, u64 j, bool complement) {
    DemuxRun r;
    r.reverse = (s & kOutReverse) != 0;
    r.p = r.reverse ? src + (s & ~kOutReverse) - j : src + s + j;
    r.complement = complement;
    r.fill = 0;
    return r;
}

// The dense layout of smx_demux_device: output i is the sequence (or quality) slice of its record and nothing else.
struct DemuxCopy {
    const unsigned char *src;       // bases or qualities
    unsigned char *dst;             // out_seq or out_qual
    bool complement;                // sequences: reverse records are complemented; qualities only reversed
    const u64 *out_off, *out_src;   // n_out + 1 offsets, n_out source positions (demux_plan_item)
    u64 n_out, total;

    // the run of a full chunk at byte j of output i, false when the chunk needs the byte-wise path
    SMX_HD bool run16(u64 i, u64 j, DemuxRun &r) const { r = demux_run(src, out_src[i], j, complement); return true; }
    // bytes [j0, j1) of output i into out
    SMX_HD void bytes(u64 i, u64 j0, u64 j1, unsigned char *out) const {
        for (u64 j = j0; j < j1; ++j) out[j - j0] = demux_src_byte(src, out_src[i], j, complement);
    }
};

// The file layout of smx_demux_files_device: output i is the complete formatted record of record order[i] (header,
// sequence, and for FASTQ the separator, qualities -- 'I' without qualities -- and newlines).
struct FilesCopy {
    const unsigned char *bases, *quals;   // quals null: 'I' fill
    unsigned char *dst;
    bool fastq;
    const u64 *out_off, *out_src, *order; // per output (n_out + 1, n_out, n_out)
    const u64 *hdr, *id_pos;              // per record (files_plan_item)
    const smx_record *records;
    const unsigned char *titles;
    OutNames names;
    u64 n_out, total;

    SMX_HD bool run16(u64 i, u64 j, DemuxRun &r) const {
        const u64 h = hdr[order[i]], n = out_record_body(out_off[i + 1] - out_off[i], h, fastq);
        if (j >= h && j + kDemuxChunk <= h + n) { r = demux_run(bases, out_src[i], j - h, true); return true; }
        const u64 q = h + n + 3;
        if (!fastq || j < q || j + kDemuxChunk > q + n) return false;
        if (quals) r = demux_run(quals, out_src[i], j - q, false);
        else { r.p = nullptr; r.reverse = r.complement = false; r.fill = 'I'; }
        return true;
    }
    SMX_HD void bytes(u64 i, u64 j0, u64 j1, unsigned char *out) const {
        const u64 rec = order[i], h = hdr[rec], s = out_src[i], n = out_record_body(out_off[i + 1] - out_off[i], h, fastq);
        if (j0 < h) {
            const smx_record &rc = records[rec];
            OutDest d;
            out_dest(rc, names.n, d);
            // the id length is what the header holds beyond its other parts
            OutHeader hd = out_header_of(rc, d, names, (const char *)titles + id_pos[rec], 0, fastq);
            hd.id_len = h - out_header_len(hd);
            OutWindow w = {0, j0, j1 < h ? j1 : h, out};
            out_header_emit(hd, w);
        }
        for (u64 j = j0 > h ? j0 : h; j < j1; ++j) {
            const u64 k = j - h;
            unsigned char ch = '\n';
            if (k < n) ch = demux_src_byte(bases, s, k, true);
            else if (k == n + 1) ch = '+';
            else if (k >= n + 3 && k < 2 * n + 3) ch = quals ? demux_src_byte(quals, s, k - n - 3, false) : 'I';
            out[j - j0] = ch;
        }
    }
};

// Copy, work item c = chunk c of tile t (whose outputs lie in [lo, hi]).  A full chunk inside one run of an output is
// one 16-byte load (a reversed one: byte-reversed words in reverse order, complemented four bytes at a time) and one
// aligned store; any other chunk goes byte by byte.  L: DemuxCopy or FilesCopy.
template <class L>
SMX_HD void demux_copy_chunk(const L &d, u64 c, u64 lo, u64 hi) {
    const long long p0 = (long long)(c * kDemuxChunk) - (long long)demux_misalign(d.dst);
    const u64 p = p0 < 0 ? 0 : (u64)p0, e = (u64)p0 + kDemuxChunk < d.total ? (u64)p0 + kDemuxChunk : d.total;
    if (p >= e) return;
    u64 i = demux_find(d.out_off, lo, hi, p);
    DemuxRun run;
    if (p0 >= 0 && e - p == kDemuxChunk && d.out_off[i + 1] >= e && d.run16(i, p - d.out_off[i], run)) {
        u32 w[4];
        if (!run.p) {
            w[0] = w[1] = w[2] = w[3] = run.fill * 0x01010101u;
        } else if (!run.reverse) {
            demux_load16(run.p, w);
        } else {
            u32 v[4];
            demux_load16(run.p - (kDemuxChunk - 1), v);
            for (int k = 0; k < 4; ++k) {
                const u32 x = byte_perm(v[3 - k], 0, 0x0123);
                w[k] = run.complement ? dna_complement4(x) : x;
            }
        }
        demux_store16(d.dst + p, w);
        return;
    }
    for (u64 q = p; q < e;) {
        while (d.out_off[i + 1] <= q) ++i;
        const u64 a = d.out_off[i], stop = d.out_off[i + 1] < e ? d.out_off[i + 1] : e;
        d.bytes(i, q - a, stop - a, d.dst + q);
        q = stop;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// specimine's record text (smx_mine_device): the identity as '%.2f' formats it and the rewritten title of a mined read.

// Python's '%.2f' % x for 0 <= x < 2^32: x * 100 rounded to the nearest integer, ties to even, decided exactly on the
// binary double -- x = mant * 2^-s, so x * 100 = mant * 100 / 2^s with mant * 100 < 2^60 -- then printed as
// <integer part>.<two digits>.  Writes the text at dst (at most 13 bytes) and returns its length.
SMX_HD u32 out_fmt2(double x, char *dst) {
    u64 bits;
    memcpy(&bits, &x, 8);
    const int e = (int)((bits >> 52) & 0x7FF);
    const u64 mant = e ? ((bits & ((1ull << 52) - 1)) | (1ull << 52)) : (bits & ((1ull << 52) - 1));
    const int s = 1075 - (e ? e : 1);                          // x = mant * 2^-s
    u64 q = 0;
    if (s < 64) {
        const u64 v = mant * 100, half = 1ull << (s - 1), rem = v & ((half << 1) - 1);
        q = v >> s;
        if (rem > half || (rem == half && (q & 1))) ++q;
    }
    char tmp[16];
    int n = 0;
    u64 ip = q / 100;
    do { tmp[n++] = (char)('0' + ip % 10); ip /= 10; } while (ip);
    u32 len = 0;
    while (n) dst[len++] = tmp[--n];
    dst[len++] = '.';
    dst[len++] = (char)('0' + (q / 10) % 10);
    dst[len++] = (char)('0' + q % 10);
    return len;
}

// The title line of a mined partial read as specimine writes it (write_fastq(_rewrite_mined(...))):
//   @<id>_mined_<kind>_<b> <description> mined_<kind> identity=<b>\n
// with <id> the title's first token (out_title_id), <description> the title without trailing whitespace (the reader's
// rstrip), <kind> "forward" or "reverse" and <b> the identity as out_fmt2 prints it.
struct OutMined {
    const char *title;
    u64 id_a, id_b, desc_len;
    bool reverse;
    const char *b;
    u32 b_len;
};

// The description's length: the title up to the end of its last non-whitespace character.
SMX_HD u64 out_rstrip_len(const unsigned char *t, u64 len) {
    const unsigned char *e = t + len;
    u64 keep = 0;
    for (const unsigned char *p = t; p < e;) {
        const int k = out_ws_at(p, e);
        if (k) { p += k; continue; }
        ++p;
        keep = (u64)(p - t);
    }
    return keep;
}

SMX_HD OutMined out_mined_title(const unsigned char *title, u64 len, bool reverse, const char *b, u32 b_len) {
    OutMined h;
    h.title = (const char *)title;
    h.desc_len = out_rstrip_len(title, len);
    out_title_id(title, h.desc_len, h.id_a, h.id_b);
    h.reverse = reverse;
    h.b = b; h.b_len = b_len;
    return h;
}

template <class Put> SMX_HD void out_mined_emit(const OutMined &h, Put &put) {
    const char *kind = h.reverse ? "reverse" : "forward";
    put.chars('@', 1);
    put(h.title + h.id_a, h.id_b - h.id_a);
    put("_mined_", 7); put(kind, 7); put.chars('_', 1); put(h.b, h.b_len);
    put.chars(' ', 1); put(h.title, h.desc_len);
    put(" mined_", 7); put(kind, 7); put(" identity=", 10); put(h.b, h.b_len); put.chars('\n', 1);
}

SMX_HD u64 out_mined_len(const OutMined &h) { OutCount c = {0}; out_mined_emit(h, c); return c.n; }

}  // namespace smx_out
