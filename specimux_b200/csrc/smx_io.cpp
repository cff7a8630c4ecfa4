// smx_io.cpp -- native FASTQ/FASTA(.gz) reader and per-specimen output-tree writer
// (include/specimux_io.h; SURVEY.md 8f rank 1).  Host code only: no CUDA, no matching.
//
// Behavioural model (cited per function): the reference's use of Bio.SeqIO.parse
// (io_utils.py:429-450), create_write_operation (demultiplex.py:30-103), OutputManager
// (io_utils.py:179-268) and output_write_operation (io_utils.py:452-471).
#include <cerrno>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <condition_variable>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include "../../include/specimux_io.h"
#include "smx_out.cuh"

namespace {

thread_local char g_err[1024] = "";

int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

// ---------------------------------------------------------------------------------------------
// Python str whitespace (str.strip / str.split(None) on text decoded as UTF-8): smx_out.cuh defines it for the device
// formatter too.  Returns the byte length of the whitespace character starting at p, 0 if none.
inline int ws_at(const unsigned char *p, const unsigned char *end) { return smx_out::out_ws_at(p, end); }

// Length of the whitespace character ENDING at end (exclusive), 0 if none.
inline int ws_before(const unsigned char *begin, const unsigned char *end) {
    if (end <= begin) return 0;
    const unsigned char c = end[-1];
    if (c < 0x80) return ((c >= 9 && c <= 13) || (c >= 28 && c <= 32)) ? 1 : 0;
    if (end - begin >= 2 && ws_at(end - 2, end) == 2) return 2;
    if (end - begin >= 3 && ws_at(end - 3, end) == 3) return 3;
    return 0;
}

inline void lstrip(const char *&b, const char *e) {
    for (int n; b < e && (n = ws_at((const unsigned char *)b, (const unsigned char *)e)) != 0;) b += n;
}
inline void rstrip(const char *b, const char *&e) {
    for (int n; e > b && (n = ws_before((const unsigned char *)b, (const unsigned char *)e)) != 0;) e -= n;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// Blocks

struct smx_block {
    std::vector<char> bases, quals, titles;
    std::vector<uint64_t> seq_off, title_off;
    std::vector<uint32_t> id_start, id_len;
    bool has_qual = false;
    void clear(bool fastq) {
        bases.clear(); quals.clear(); titles.clear();
        seq_off.assign(1, 0); title_off.assign(1, 0);
        id_start.clear(); id_len.clear();
        has_qual = fastq;
    }
    uint32_t n() const { return (uint32_t)id_len.size(); }
};

// ---------------------------------------------------------------------------------------------
// Reader

struct smx_reader {
    int fd = -1;
    gzFile gz = nullptr;
    bool fastq = true, eof = false;
    std::vector<char> buf;
    size_t pos = 0, end = 0;
    std::string path;
    // FASTA: the title of the record whose sequence lines are being collected
    bool fasta_open = false;
    std::string fasta_title;
    // byte-range readers (smx_reader_open_range): the file position the next read() starts at and the position the
    // range ends at (the reader sees end-of-file there); stop_off == UINT64_MAX for whole-file readers
    uint64_t read_off = 0, stop_off = UINT64_MAX;

    // Fills the buffer; returns false on a read error.
    bool refill() {
        if (pos > 0) { memmove(buf.data(), buf.data() + pos, end - pos); end -= pos; pos = 0; }
        if (end == buf.size()) buf.resize(buf.size() * 2);
        long got;
        if (gz) got = gzread(gz, buf.data() + end, (unsigned)std::min<size_t>(buf.size() - end, 1u << 30));
        else {
            size_t want = buf.size() - end;
            if (stop_off != UINT64_MAX) want = (size_t)std::min<uint64_t>(want, stop_off > read_off ? stop_off - read_off : 0);
            got = want ? (long)read(fd, buf.data() + end, want) : 0;
            if (got > 0) read_off += (uint64_t)got;
        }
        if (got < 0) return false;
        if (got == 0) eof = true;
        end += (size_t)got;
        return true;
    }

    // Next line without its terminator ('\n'; a preceding '\r' is whitespace and stripped by every
    // consumer).  Returns 0 at end of file, 1 with [b, e) set, -1 on a read error.  The pointers
    // stay valid until the next call.
    int line(const char *&b, const char *&e) {
        for (;;) {
            const char *nl = (const char *)memchr(buf.data() + pos, '\n', end - pos);
            if (nl) { b = buf.data() + pos; e = nl; pos = (size_t)(nl - buf.data()) + 1; return 1; }
            if (eof) {
                if (pos == end) return 0;
                b = buf.data() + pos; e = buf.data() + end; pos = end; return 1;
            }
            if (!refill()) return -1;
        }
    }
};

namespace {

void add_title(smx_block &blk, const char *b, const char *e) {
    // record.description = whole title; record.id = first whitespace-delimited token
    blk.titles.insert(blk.titles.end(), b, e);
    blk.title_off.push_back(blk.titles.size());
    uint64_t ia, ib;
    smx_out::out_title_id((const unsigned char *)b, (uint64_t)(e - b), ia, ib);
    blk.id_start.push_back((uint32_t)ia);
    blk.id_len.push_back((uint32_t)(ib - ia));
}

// One FASTQ record (FastqGeneralIterator semantics as restated in specimux_b200/seqio.py:
// blank lines between records skipped, multi-line sequence / quality accepted).
// Returns 1 record parsed, 0 end of file, <0 error.  `blk` may be null (skip).
int next_fastq(smx_reader &r, smx_block *blk) {
    const char *b, *e;
    int rc;
    for (;;) {
        if ((rc = r.line(b, e)) <= 0) return rc < 0 ? -SMX_IO_ERR_IO : 0;
        const char *sb = b, *se = e;
        lstrip(sb, se);
        if (sb < se) break;
    }
    if (*b != '@') return -fail(SMX_IO_ERR_FORMAT, "Records in Fastq files should start with '@' character");
    const char *tb = b + 1, *te = e;
    rstrip(tb, te);
    std::string skipped_title;           // skip mode only: the title is needed for an error message
    if (blk) add_title(*blk, tb, te); else skipped_title.assign(tb, te);
    // Fast path: the common four-line record lying completely in the buffer (one memchr per line,
    // one memcpy each for bases and qualities).  Anything else -- wrapped sequence or quality lines,
    // a record cut by the end of the buffer or of the file -- takes the general path below, which
    // starts again right after the title line (nothing is consumed here unless the record fits).
    {
        const char *p = r.buf.data() + r.pos, *end = r.buf.data() + r.end;
        const char *nl1 = (const char *)memchr(p, '\n', (size_t)(end - p));
        if (nl1 && nl1 + 1 < end && nl1[1] == '+') {
            const char *nl2 = (const char *)memchr(nl1 + 1, '\n', (size_t)(end - nl1 - 1));
            const char *nl3 = nl2 ? (const char *)memchr(nl2 + 1, '\n', (size_t)(end - nl2 - 1)) : nullptr;
            if (nl3) {
                const char *sb = p, *se = nl1, *qb = nl2 + 1, *qe = nl3;
                lstrip(sb, se); rstrip(sb, se);
                lstrip(qb, qe); rstrip(qb, qe);
                if (se - sb == qe - qb && se > sb) {
                    if (blk) {
                        blk->bases.insert(blk->bases.end(), sb, se);
                        blk->quals.insert(blk->quals.end(), qb, qe);
                        blk->seq_off.push_back(blk->bases.size());
                    }
                    r.pos = (size_t)(nl3 - r.buf.data()) + 1;
                    return 1;
                }
            }
        }
    }
    size_t seq_len = 0, qual_len = 0;
    // sequence lines up to the '+' line
    bool first = true;
    for (;;) {
        if ((rc = r.line(b, e)) < 0) return -SMX_IO_ERR_IO;
        if (rc == 0) break;
        if (!first && b < e && *b == '+') break;
        const char *sb = b, *se = e;
        lstrip(sb, se); rstrip(sb, se);
        if (blk) blk->bases.insert(blk->bases.end(), sb, se);
        seq_len += (size_t)(se - sb);
        first = false;
    }
    // quality lines until as long as the sequence
    bool got_one = false;
    while (!got_one || qual_len < seq_len) {
        if ((rc = r.line(b, e)) < 0) return -SMX_IO_ERR_IO;
        if (rc == 0) break;
        const char *sb = b, *se = e;
        lstrip(sb, se); rstrip(sb, se);
        if (blk) blk->quals.insert(blk->quals.end(), sb, se);
        qual_len += (size_t)(se - sb);
        got_one = true;
    }
    if (qual_len != seq_len) {
        std::string title = blk ? std::string(blk->titles.data() + blk->title_off[blk->title_off.size() - 2],
                                              blk->titles.data() + blk->title_off.back())
                                : skipped_title;
        return -fail(SMX_IO_ERR_FORMAT, "Lengths of sequence and quality values differs for %s", title.c_str());
    }
    if (blk) blk->seq_off.push_back(blk->bases.size());
    return 1;
}

// One FASTA record (SimpleFastaParser semantics: lines before the first '>' ignored, sequence
// lines stripped and concatenated).
int next_fasta(smx_reader &r, smx_block *blk) {
    const char *b, *e;
    int rc;
    while (!r.fasta_open) {
        if ((rc = r.line(b, e)) <= 0) return rc < 0 ? -SMX_IO_ERR_IO : 0;
        if (b < e && *b == '>') {
            const char *tb = b + 1, *te = e;
            rstrip(tb, te);
            r.fasta_title.assign(tb, te);
            r.fasta_open = true;
        }
    }
    if (blk) add_title(*blk, r.fasta_title.data(), r.fasta_title.data() + r.fasta_title.size());
    r.fasta_open = false;
    for (;;) {
        if ((rc = r.line(b, e)) < 0) return -SMX_IO_ERR_IO;
        if (rc == 0) break;
        if (b < e && *b == '>') {
            const char *tb = b + 1, *te = e;
            rstrip(tb, te);
            r.fasta_title.assign(tb, te);
            r.fasta_open = true;
            break;
        }
        const char *sb = b, *se = e;
        lstrip(sb, se); rstrip(sb, se);
        if (blk) blk->bases.insert(blk->bases.end(), sb, se);
    }
    if (blk) blk->seq_off.push_back(blk->bases.size());
    return 1;
}

bool ends_with(const std::string &s, const char *suffix) {
    size_t n = strlen(suffix);
    return s.size() >= n && s.compare(s.size() - n, n, suffix) == 0;
}

}  // namespace

extern "C" {

int smx_io_abi_version(void) { return SMX_IO_ABI_VERSION; }
const char *smx_io_last_error(void) { return g_err; }

int smx_reader_open(const char *path, int is_fastq, smx_reader **out) {
    if (!path || !out) return fail(SMX_IO_ERR_ARG, "smx_reader_open: null argument");
    smx_reader *r = new smx_reader();
    r->path = path;
    r->fastq = is_fastq != 0;
    r->buf.resize(8u << 20);
    if (ends_with(r->path, ".gz") || ends_with(r->path, ".gzip")) {
        r->gz = gzopen(path, "rb");
        if (!r->gz) { delete r; return fail(SMX_IO_ERR_OPEN, "cannot open %s: %s", path, strerror(errno)); }
        gzbuffer(r->gz, 1u << 20);
    } else {
        r->fd = open(path, O_RDONLY);
        if (r->fd < 0) { delete r; return fail(SMX_IO_ERR_OPEN, "cannot open %s: %s", path, strerror(errno)); }
#ifdef POSIX_FADV_SEQUENTIAL
        posix_fadvise(r->fd, 0, 0, POSIX_FADV_SEQUENTIAL);
#endif
    }
    *out = r;
    return SMX_IO_OK;
}

// First FASTQ record boundary at or after byte `off` of a plain four-line FASTQ file: the first line start p with
// line(p) beginning '@' and line(p + 2) beginning '+'.  Exact for four-line records: a quality line that happens to
// begin with '@' is followed two lines later by a sequence line, which never begins with '+'.  Returns the file
// size when no record starts after `off`, -1 on a read error.
static int64_t fastq_sync(int fd, uint64_t off, uint64_t file_size) {
    if (off == 0) return 0;
    if (off >= file_size) return (int64_t)file_size;
    size_t window = 1u << 20;
    std::vector<char> w;
    for (;;) {
        const uint64_t from = off - 1;                      // the byte before `off` tells whether `off` starts a line
        const size_t len = (size_t)std::min<uint64_t>(window, file_size - from);
        w.resize(len);
        size_t got = 0;
        while (got < len) {
            ssize_t k = pread(fd, w.data() + got, len - got, (off_t)(from + got));
            if (k < 0) return -1;
            if (k == 0) break;
            got += (size_t)k;
        }
        const bool whole = from + got >= file_size;
        // line starts inside the window
        std::vector<size_t> starts;
        for (size_t i = 0; i + 1 <= got; ++i)
            if (w[i] == '\n' && i + 1 < got) starts.push_back(i + 1);
        for (size_t k = 0; k + 2 < starts.size(); ++k)
            if (w[starts[k]] == '@' && w[starts[k + 2]] == '+') return (int64_t)(from + starts[k]);
        if (whole) return (int64_t)file_size;
        window *= 4;
    }
}

int smx_reader_open_range(const char *path, int is_fastq, uint64_t byte_start, uint64_t byte_end, smx_reader **out) {
    if (!path || !out) return fail(SMX_IO_ERR_ARG, "smx_reader_open_range: null argument");
    if (!is_fastq) return fail(SMX_IO_ERR_ARG, "smx_reader_open_range: byte ranges need a FASTQ file");
    std::string p(path);
    if (ends_with(p, ".gz") || ends_with(p, ".gzip")) return fail(SMX_IO_ERR_ARG, "smx_reader_open_range: compressed files are read serially");
    int rc = smx_reader_open(path, is_fastq, out);
    if (rc) return rc;
    smx_reader *r = *out;
    struct stat st;
    if (fstat(r->fd, &st) != 0) { smx_reader_close(r); *out = nullptr; return fail(SMX_IO_ERR_IO, "cannot stat %s", path); }
    const uint64_t size = (uint64_t)st.st_size;
    const int64_t a = fastq_sync(r->fd, std::min(byte_start, size), size);
    const int64_t b = byte_end >= size ? (int64_t)size : fastq_sync(r->fd, byte_end, size);
    if (a < 0 || b < 0) { smx_reader_close(r); *out = nullptr; return fail(SMX_IO_ERR_IO, "read error on %s", path); }
    if (lseek(r->fd, (off_t)a, SEEK_SET) < 0) { smx_reader_close(r); *out = nullptr; return fail(SMX_IO_ERR_IO, "cannot seek %s", path); }
    r->read_off = (uint64_t)a;
    r->stop_off = (uint64_t)std::max(a, b);
    return SMX_IO_OK;
}

void smx_reader_close(smx_reader *r) {
    if (!r) return;
    if (r->gz) gzclose(r->gz);
    if (r->fd >= 0) close(r->fd);
    delete r;
}

smx_block *smx_block_create(void) {
    smx_block *b = new smx_block();
    b->clear(false);
    return b;
}

void smx_block_destroy(smx_block *b) { delete b; }

void smx_block_get(const smx_block *b, smx_block_view *out) {
    if (!b || !out) return;
    out->n_reads = b->n();
    out->bases = b->bases.data();
    out->seq_off = b->seq_off.data();
    static const char kEmpty[1] = {0};
    out->quals = b->has_qual ? (b->quals.empty() ? kEmpty : b->quals.data()) : nullptr;     // FASTQ with no bases at all: still "has qualities"
    out->titles = b->titles.data();
    out->title_off = b->title_off.data();
    out->id_start = b->id_start.data();
    out->id_len = b->id_len.data();
}

int smx_reader_next(smx_reader *r, uint32_t max_reads, smx_block *blk) {
    if (!r || !blk) return fail(SMX_IO_ERR_ARG, "smx_reader_next: null argument");
    blk->clear(r->fastq);
    if (r->stop_off != UINT64_MAX && r->stop_off > r->read_off) {
        // byte-range reader: the whole range lands in this block -- size the buffers once (bases and qualities are
        // each a little under half of a four-line FASTQ file) instead of growing them by doubling
        const size_t span = (size_t)(r->stop_off - r->read_off);
        if (blk->bases.capacity() < span / 2) blk->bases.reserve(span / 2 + 4096);
        if (r->fastq && blk->quals.capacity() < span / 2) blk->quals.reserve(span / 2 + 4096);
    }
    for (uint32_t i = 0; i < max_reads; ++i) {
        int rc = r->fastq ? next_fastq(*r, blk) : next_fasta(*r, blk);
        if (rc < 0) {
            if (-rc == SMX_IO_ERR_IO) return fail(SMX_IO_ERR_IO, "read error on %s", r->path.c_str());
            return -rc;
        }
        if (rc == 0) break;
    }
    return SMX_IO_OK;
}

int smx_reader_skip(smx_reader *r, uint64_t n, uint64_t *skipped) {
    if (!r) return fail(SMX_IO_ERR_ARG, "smx_reader_skip: null argument");
    uint64_t done = 0;
    for (; done < n; ++done) {
        int rc = r->fastq ? next_fastq(*r, nullptr) : next_fasta(*r, nullptr);
        if (rc < 0) {
            if (-rc == SMX_IO_ERR_IO) return fail(SMX_IO_ERR_IO, "read error on %s", r->path.c_str());
            return -rc;
        }
        if (rc == 0) break;
    }
    if (skipped) *skipped = done;
    return SMX_IO_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// Writer

namespace {

struct Complement {
    unsigned char t[256];
    Complement() {
        // Bio.Seq's ambiguous-DNA complement as the reference applies it through SeqRecord.reverse_complement
        // (demultiplex.py:142); smx_out.cuh defines it for the device demultiplexer too
        for (int i = 0; i < 256; ++i) t[i] = smx_out::dna_complement((unsigned char)i);
    }
};
const Complement kComplement;

// dst[j] = tab[src_last[-j]] (reverse complement) / dst[j] = src_last[-j] (reverse copy), n bytes; src_last points at
// the LAST byte of the source run.  Half the reads of a mixed-orientation run are written reversed, byte by byte in
// the first form of the writer; on x86-64 with SSSE3 sixteen bytes go at a time: the reversal is one byte shuffle, the
// complement two 16-entry table look-ups on the low five bits of a letter (A..Z / a..z keep their case bits; bytes
// outside 0x40..0x7F pass through), the same mapping as kComplement.
void reverse_complement_scalar(char *dst, const unsigned char *src_last, size_t n) {
    const unsigned char *tab = kComplement.t;
    for (size_t j = 0; j < n; ++j) dst[j] = (char)tab[src_last[-(long long)j]];
}
void reverse_copy_scalar(char *dst, const char *src_last, size_t n) {
    for (size_t j = 0; j < n; ++j) dst[j] = src_last[-(long long)j];
}

#if defined(__x86_64__) && defined(__GNUC__)
#include <immintrin.h>
__attribute__((target("ssse3"))) void reverse_complement_ssse3(char *dst, const unsigned char *src_last, size_t n) {
    // index = byte & 0x1F: 0 '@', 1..26 'A'..'Z', 27..31 '[' .. '_'
    //                          @   A   B   C   D   E   F   G   H   I   J   K   L   M   N   O
    const __m128i lo = _mm_setr_epi8(0, 20, 22, 7, 8, 5, 6, 3, 4, 9, 10, 13, 12, 11, 14, 15);
    //                          P   Q   R   S   T   U   V   W   X   Y   Z   [   \   ]   ^   _
    const __m128i hi = _mm_setr_epi8(16, 17, 25, 19, 1, 1, 2, 23, 24, 18, 26, 27, 28, 29, 30, 31);
    const __m128i rev = _mm_setr_epi8(15, 14, 13, 12, 11, 10, 9, 8, 7, 6, 5, 4, 3, 2, 1, 0);
    const __m128i m1f = _mm_set1_epi8(0x1F), m0f = _mm_set1_epi8(0x0F), me0 = _mm_set1_epi8((char)0xE0),
                  mc0 = _mm_set1_epi8((char)0xC0), v40 = _mm_set1_epi8(0x40), v10 = _mm_set1_epi8(0x10);
    size_t j = 0;
    for (; j + 16 <= n; j += 16) {
        __m128i v = _mm_loadu_si128((const __m128i *)(src_last - j - 15));
        v = _mm_shuffle_epi8(v, rev);
        const __m128i idx = _mm_and_si128(v, m1f);
        const __m128i from_lo = _mm_shuffle_epi8(lo, _mm_and_si128(idx, m0f));
        const __m128i from_hi = _mm_shuffle_epi8(hi, _mm_and_si128(idx, m0f));
        const __m128i is_hi = _mm_cmpeq_epi8(_mm_and_si128(idx, v10), v10);
        const __m128i mapped = _mm_or_si128(_mm_and_si128(is_hi, from_hi), _mm_andnot_si128(is_hi, from_lo));
        const __m128i letter = _mm_cmpeq_epi8(_mm_and_si128(v, mc0), v40);          // 0x40..0x7F
        const __m128i out = _mm_or_si128(_mm_and_si128(letter, _mm_or_si128(mapped, _mm_and_si128(v, me0))),
                                         _mm_andnot_si128(letter, v));
        _mm_storeu_si128((__m128i *)(dst + j), out);
    }
    reverse_complement_scalar(dst + j, src_last - j, n - j);
}
__attribute__((target("ssse3"))) void reverse_copy_ssse3(char *dst, const char *src_last, size_t n) {
    const __m128i rev = _mm_setr_epi8(15, 14, 13, 12, 11, 10, 9, 8, 7, 6, 5, 4, 3, 2, 1, 0);
    size_t j = 0;
    for (; j + 16 <= n; j += 16)
        _mm_storeu_si128((__m128i *)(dst + j), _mm_shuffle_epi8(_mm_loadu_si128((const __m128i *)(src_last - j - 15)), rev));
    reverse_copy_scalar(dst + j, src_last - j, n - j);
}
const bool kHaveSsse3 = __builtin_cpu_supports("ssse3") && !getenv("SMX_IO_NO_SIMD");     // (switch for A/B runs)
#else
const bool kHaveSsse3 = false;
void reverse_complement_ssse3(char *dst, const unsigned char *src_last, size_t n) { reverse_complement_scalar(dst, src_last, n); }
void reverse_copy_ssse3(char *dst, const char *src_last, size_t n) { reverse_copy_scalar(dst, src_last, n); }
#endif

inline void reverse_complement_into(char *dst, const unsigned char *src_last, size_t n) {
    if (kHaveSsse3) reverse_complement_ssse3(dst, src_last, n); else reverse_complement_scalar(dst, src_last, n);
}
inline void reverse_copy_into(char *dst, const char *src_last, size_t n) {
    if (kHaveSsse3) reverse_copy_ssse3(dst, src_last, n); else reverse_copy_scalar(dst, src_last, n);
}

// Growable byte buffer without value-initialisation (std::vector<char>::resize zero-fills what the
// formatter overwrites straight away; realloc can also remap large blocks instead of copying them).
struct Bytes {
    char *p = nullptr;
    size_t n = 0, cap = 0;
    Bytes() = default;
    Bytes(const Bytes &) = delete;
    Bytes &operator=(const Bytes &) = delete;
    Bytes(Bytes &&o) noexcept : p(o.p), n(o.n), cap(o.cap) { o.p = nullptr; o.n = o.cap = 0; }
    ~Bytes() { free(p); }
    char *grow(size_t extra) {           // room for `extra` more bytes; returns the write position
        if (n + extra > cap) {
            size_t want = cap ? cap * 2 : 4096;
            while (want < n + extra) want *= 2;
            char *q = (char *)realloc(p, want);
            if (!q) throw std::bad_alloc();
            p = q; cap = want;
        }
        return p + n;
    }
    bool empty() const { return n == 0; }
    size_t size() const { return n; }
    const char *data() const { return p; }
    void clear() { n = 0; }
};

struct OutFile {
    std::string path;
    Bytes buf;
    bool dir_made = false;
};

// Per-file buffer before an append.  Small on purpose: with ~1,500 open specimen files the buffers
// are the writer's working set, and first-touch page faults of large buffers cost more than the
// extra open/append/close calls (measured: tools/io_bench.py).  SMX_IO_FLUSH_KB overrides.
size_t flush_bytes() {
    static const size_t v = [] {
        const char *e = getenv("SMX_IO_FLUSH_KB");
        long kb = e ? atol(e) : 0;
        return (size_t)(kb > 0 ? kb : 64) << 10;
    }();
    return v;
}

inline void put(Bytes &v, const char *s, size_t n) { memcpy(v.grow(n), s, n); v.n += n; }
inline void put(Bytes &v, const std::string &s) { put(v, s.data(), s.size()); }
inline void put(Bytes &v, char c) { *v.grow(1) = c; ++v.n; }

bool make_dirs(const std::string &dir) {          // os.makedirs(exist_ok=True)
    struct stat st;
    if (stat(dir.c_str(), &st) == 0) return S_ISDIR(st.st_mode);
    size_t slash = dir.find_last_of('/');
    if (slash != std::string::npos && slash > 0 && !make_dirs(dir.substr(0, slash))) return false;
    return mkdir(dir.c_str(), 0777) == 0 || errno == EEXIST;
}

}  // namespace

// One formatted-record destination.  A file is owned by exactly one worker thread (fixed at
// creation), so its buffer and its appends need no lock and keep arrival order.
struct Target {
    OutFile file;
    int owner = 0;
};

// What the planning pass resolves for a record: names, slice bounds, destinations.
struct Plan {
    const std::string *sample, *pool, *p1, *p2;
    uint64_t a, b;               // slice [a, b) of the oriented read
    Target *primary, *pool_level;
};

// One record for one worker: formatted once into `dst`; `copy` (the pool-level duplicate of a full match, owned by
// the same worker) receives the same bytes.
struct Task { uint32_t rec; Target *dst; Target *copy; };

struct smx_writer {
    bool to_files = true, fastq = true;
    std::string dir, prefix, ext;
    std::vector<std::string> specimen_id, specimen_file, b1_id, b1_file, b2_id, b2_file, pool, primer;
    std::unordered_map<uint64_t, Target *> files;     // keyed by packed (level, top, pool, p1, p2, sample kind, sample)
    std::vector<Target *> all_files;
    Bytes console;
    uint64_t n_records = 0, n_bytes = 0;
    std::mutex err_mu;
    int first_error = SMX_IO_OK;
    std::string first_error_msg;

    // worker pool (file output only): thread t formats the tasks of the files it owns
    int n_threads = 1;
    std::vector<std::thread> threads;
    // Two sets of planning storage: while the workers format call i from one set, the calling thread plans call i + 1
    // into the other (smx_writer_write*_deferred).
    std::vector<std::vector<Task>> task_sets[2];      // per thread, in record order
    std::vector<Plan> plan_sets[2];
    std::vector<smx_record> full_sets[2];             // widened records of the 16 / 32-byte forms
    int next_set = 0;
    bool in_flight = false;                           // a dispatched call the workers may still be formatting
    const std::vector<std::vector<Task>> *cur_tasks = nullptr;
    std::vector<uint64_t> thread_bytes;
    std::mutex mu;
    std::condition_variable cv_go, cv_done;
    uint64_t generation = 0;
    int pending = 0;
    bool stop = false;
    const smx_block *cur_blk = nullptr;
    const smx_record *cur_recs = nullptr;
    const std::vector<Plan> *cur_plans = nullptr;

    void note_error(int code, const std::string &msg) {
        std::lock_guard<std::mutex> g(err_mu);
        if (first_error == SMX_IO_OK) { first_error = code; first_error_msg = msg; }
    }
    // first error seen so far (workers of a deferred call may still be reporting: read under the lock)
    int error_status() {
        std::lock_guard<std::mutex> g(err_mu);
        return first_error == SMX_IO_OK ? SMX_IO_OK : fail(first_error, "%s", first_error_msg.c_str());
    }

    void flush(OutFile &f) {
        if (f.buf.empty()) return;
        if (!f.dir_made) {
            size_t slash = f.path.find_last_of('/');
            if (slash != std::string::npos && !make_dirs(f.path.substr(0, slash)))
                note_error(SMX_IO_ERR_OPEN, "cannot create directory for " + f.path + ": " + strerror(errno));
            f.dir_made = true;
        }
        int fd = open(f.path.c_str(), O_WRONLY | O_CREAT | O_APPEND, 0666);
        if (fd < 0) {
            note_error(SMX_IO_ERR_OPEN, "cannot open " + f.path + ": " + strerror(errno));
        } else {
            size_t off = 0;
            while (off < f.buf.size()) {
                ssize_t w = ::write(fd, f.buf.data() + off, f.buf.size() - off);
                if (w < 0) {
                    if (errno == EINTR) continue;
                    note_error(SMX_IO_ERR_IO, "write to " + f.path + ": " + strerror(errno));
                    break;
                }
                off += (size_t)w;
            }
            close(fd);
        }
        f.buf.clear();
    }

    // owner_key: files with the same key belong to the same worker (a specimen's primer-pair file and its
    // pool-level duplicate: the record is formatted once and copied)
    Target *target(uint64_t key, const std::string &path, uint64_t owner_key) {
        auto it = files.find(key);
        if (it != files.end()) return it->second;
        Target *t = new Target();
        t->file.path = path;
        t->owner = (int)((owner_key * 0x9E3779B97F4A7C15ull >> 33) % (uint64_t)n_threads);
        all_files.push_back(t);
        files.emplace(key, t);
        return t;
    }

    void format(Bytes &c, const smx_block &blk, const smx_record &rec, const Plan &pl);
    int write_planned(const smx_block *blk, const smx_record *recs, uint64_t n_records, int set, bool deferred);
    void wait_in_flight();
    void run_tasks(int t);
    void worker(int t);
    ~smx_writer() { for (Target *t : all_files) delete t; }
};

namespace {

void copy_names(std::vector<std::string> &dst, const char *const *src, uint32_t n) {
    dst.clear();
    for (uint32_t i = 0; i < n; ++i) dst.emplace_back(src && src[i] ? src[i] : "");
}

const std::string kUnknown = "unknown";

}  // namespace

// One record, formatted in place at the end of `c` (create_write_operation's string work,
// demultiplex.py:30-103, and the header of OutputManager.write_sequence, io_utils.py:245-256).
void smx_writer::format(Bytes &c, const smx_block &blk, const smx_record &rec, const Plan &pl) {
    const uint32_t r = rec.read;
    const char *seq = blk.bases.data() + blk.seq_off[r];
    const long long len = (long long)(blk.seq_off[r + 1] - blk.seq_off[r]);
    const char *qual = blk.has_qual ? blk.quals.data() + blk.seq_off[r] : nullptr;
    const size_t a = pl.a, n_out = pl.b - pl.a;
    smx_out::OutHeader h;
    h.lead = fastq ? '@' : '>';
    h.files = to_files;
    h.dist = rec.dist;
    h.id = blk.titles.data() + blk.title_off[r] + blk.id_start[r]; h.id_len = blk.id_len[r];
    h.pool = pl.pool->data(); h.pool_len = pl.pool->size();
    h.p1 = pl.p1->data(); h.p1_len = pl.p1->size();
    h.p2 = pl.p2->data(); h.p2_len = pl.p2->size();
    h.sample = pl.sample->data(); h.sample_len = pl.sample->size();
    const uint64_t hl = smx_out::out_header_len(h);
    char *dst = c.grow(hl + 2 * n_out + 4);
    dst += smx_out::out_header_write(h, dst);
    if (rec.reverse) {
        // oriented read = reverse complement; its slice [a, b) = original (len-b .. len-a] reversed
        reverse_complement_into(dst, (const unsigned char *)seq + (len - (long long)a) - 1, n_out);
    } else if (n_out) {
        memcpy(dst, seq + a, n_out);
    }
    dst += n_out;
    *dst++ = '\n';
    if (fastq) {
        *dst++ = '+'; *dst++ = '\n';
        if (!qual) memset(dst, 'I', n_out);          // get_quality_seq: [40] * len (alignment.py:52-56)
        else if (rec.reverse) {
            reverse_copy_into(dst, qual + (len - (long long)a) - 1, n_out);
        } else if (n_out) memcpy(dst, qual + a, n_out);
        dst += n_out;
        *dst++ = '\n';
    }
    c.n = (size_t)(dst - c.p);
}

void smx_writer::run_tasks(int t) {
    uint64_t bytes = 0;
    for (const Task &k : (*cur_tasks)[(size_t)t]) {
        Bytes &buf = k.dst->file.buf;
        const size_t before = buf.size();
        const Plan &pl = (*cur_plans)[k.rec];
        format(buf, *cur_blk, cur_recs[k.rec], pl);
        const size_t len = buf.size() - before;
        bytes += len;                                               // payload counted once per record
        if (k.copy) {
            Bytes &dup = k.copy->file.buf;
            memcpy(dup.grow(len), buf.data() + before, len);
            dup.n += len;
            if (dup.size() >= flush_bytes()) flush(k.copy->file);
        }
        if (buf.size() >= flush_bytes()) flush(k.dst->file);
    }
    thread_bytes[t] = bytes;
}

void smx_writer::worker(int t) {
    uint64_t seen = 0;
    for (;;) {
        {
            std::unique_lock<std::mutex> lk(mu);
            cv_go.wait(lk, [&] { return stop || generation != seen; });
            if (stop) return;
            seen = generation;
        }
        try {
            run_tasks(t);
        } catch (const std::exception &e) {
            note_error(SMX_IO_ERR_IO, std::string("writer thread: ") + e.what());
        }
        std::lock_guard<std::mutex> lk(mu);
        if (--pending == 0) cv_done.notify_one();
    }
}

extern "C" {

int smx_writer_open(const char *output_dir, const char *prefix, int is_fastq, const smx_names *nm, smx_writer **out) {
    if (!nm || !out) return fail(SMX_IO_ERR_ARG, "smx_writer_open: null argument");
    smx_writer *w = new smx_writer();
    w->to_files = output_dir != nullptr;
    w->fastq = is_fastq != 0;
    w->dir = output_dir ? output_dir : "";
    w->prefix = prefix ? prefix : "";
    w->ext = is_fastq ? ".fastq" : ".fasta";
    copy_names(w->specimen_id, nm->specimen_id, nm->n_specimens);
    copy_names(w->specimen_file, nm->specimen_file, nm->n_specimens);
    copy_names(w->b1_id, nm->b1_id, nm->n_b1);
    copy_names(w->b1_file, nm->b1_file, nm->n_b1);
    copy_names(w->b2_id, nm->b2_id, nm->n_b2);
    copy_names(w->b2_file, nm->b2_file, nm->n_b2);
    copy_names(w->pool, nm->pool, nm->n_pools);
    copy_names(w->primer, nm->primer_name, nm->n_primers);
    if (w->to_files && !make_dirs(w->dir)) {
        int rc = fail(SMX_IO_ERR_OPEN, "cannot create %s: %s", w->dir.c_str(), strerror(errno));
        delete w;
        return rc;
    }
    if (w->to_files) {
        // formatting + appending is spread over worker threads by destination file
        const char *e = getenv("SMX_IO_THREADS");
        int n = e ? atoi(e) : 0;
        if (n <= 0) {
            unsigned hw = std::thread::hardware_concurrency();
            n = (int)std::min<unsigned>(8u, std::max<unsigned>(1u, hw / 2));
        }
        w->n_threads = std::min(n, 64);
    }
    for (auto &ts : w->task_sets) ts.resize((size_t)w->n_threads);
    w->thread_bytes.assign((size_t)w->n_threads, 0);
    if (w->n_threads > 1)
        for (int t = 0; t < w->n_threads; ++t) w->threads.emplace_back(&smx_writer::worker, w, t);
    *out = w;
    return SMX_IO_OK;
}

}  // extern "C"

// Waits for the workers of the last dispatched call (deferred form) and books their byte counts.
void smx_writer::wait_in_flight() {
    if (!in_flight) return;
    {
        std::unique_lock<std::mutex> lk(mu);
        cv_done.wait(lk, [&] { return pending == 0; });
    }
    for (uint64_t v : thread_bytes) n_bytes += v;
    cur_blk = nullptr; cur_recs = nullptr; cur_plans = nullptr; cur_tasks = nullptr;
    in_flight = false;
}

// Plans `recs` into planning set `set` (this thread; the workers may still be formatting the previous call from the
// other set), waits for that previous call, hands the new one to the workers and -- unless `deferred` -- waits for it.
int smx_writer::write_planned(const smx_block *blk, const smx_record *recs, uint64_t n_records, int set, bool deferred) {
    smx_writer *w = this;
    const uint32_t n_reads = blk->n();
    std::vector<Plan> &plans = plan_sets[set];
    plans.assign((size_t)n_records, Plan());
    std::vector<std::vector<Task>> &tasks = task_sets[set];
    for (auto &t : tasks) t.clear();
    const smx_out::OutCounts counts = {(uint32_t)w->specimen_id.size(), (uint32_t)w->b1_id.size(), (uint32_t)w->b2_id.size(),
                                       (uint32_t)w->pool.size(), (uint32_t)w->primer.size()};
    // ---- planning pass (this thread): names, slice bounds, destination files
    for (uint64_t i = 0; i < n_records; ++i) {
        const smx_record &rec = recs[i];
        if (rec.read >= n_reads) return fail(SMX_IO_ERR_ARG, "record %llu names read %u of a %u-read block", (unsigned long long)i, rec.read, n_reads);
        const long long len = (long long)(blk->seq_off[rec.read + 1] - blk->seq_off[rec.read]);
        Plan &pl = plans[i];
        // names (demultiplex.py:47-73 empty-trim fallback; :541-598 sample ids) and the destination
        // (OutputManager._make_filename, io_utils.py:206-220): the rules of smx_out.cuh
        smx_out::OutDest d;
        switch (smx_out::out_dest(rec, counts, d)) {
        case smx_out::kOutSpecimen: return fail(SMX_IO_ERR_ARG, "record %llu: specimen %d out of range", (unsigned long long)i, rec.sample);
        case smx_out::kOutB1: return fail(SMX_IO_ERR_ARG, "record %llu: b1 %d out of range", (unsigned long long)i, rec.sample);
        case smx_out::kOutB2: return fail(SMX_IO_ERR_ARG, "record %llu: b2 %d out of range", (unsigned long long)i, rec.sample);
        case smx_out::kOutPool: return fail(SMX_IO_ERR_ARG, "record %llu: pool out of range", (unsigned long long)i);
        case smx_out::kOutP1: return fail(SMX_IO_ERR_ARG, "record %llu: p1 out of range", (unsigned long long)i);
        case smx_out::kOutP2: return fail(SMX_IO_ERR_ARG, "record %llu: p2 out of range", (unsigned long long)i);
        default: break;
        }
        smx_out::out_slice(rec, len, pl.a, pl.b);
        const std::string *sample_file = &kUnknown;
        pl.sample = &kUnknown;
        if (d.kind == 0) { pl.sample = &w->specimen_id[d.sample]; sample_file = &w->specimen_file[d.sample]; }
        else if (d.kind == 1) { pl.sample = &w->b1_id[d.sample]; sample_file = &w->b1_file[d.sample]; }
        else if (d.kind == 2) { pl.sample = &w->b2_id[d.sample]; sample_file = &w->b2_file[d.sample]; }
        pl.pool = d.pool ? &w->pool[d.pool - 1] : &kUnknown;
        pl.p1 = d.p1 ? &w->primer[d.p1 - 1] : &kUnknown;
        pl.p2 = d.p2 ? &w->primer[d.p2 - 1] : &kUnknown;
        pl.primary = pl.pool_level = nullptr;
        if (!w->to_files) continue;
        const uint64_t skey = ((uint64_t)d.kind << 30) | d.sample;
        const uint64_t key = smx_out::out_key(d);
        static const char *kTop[3] = {"full", "partial", "unknown"};
        auto it = w->files.find(key);
        pl.primary = it != w->files.end() ? it->second
                   : w->target(key, w->dir + "/" + kTop[d.top] + "/" + *pl.pool + "/" + *pl.p1 + "-" + *pl.p2 + "/" + w->prefix + *sample_file + w->ext, skey);
        if (smx_out::out_has_pool_copy(rec)) {
            // pool-level duplicate of full matches (io_utils.py:259-268): same worker, the formatted bytes are copied
            const uint64_t pkey = smx_out::out_pool_key(d);
            auto pit = w->files.find(pkey);
            pl.pool_level = pit != w->files.end() ? pit->second
                          : w->target(pkey, w->dir + "/full/" + *pl.pool + "/" + w->prefix + *sample_file + w->ext, skey);
        }
        tasks[(size_t)pl.primary->owner].push_back(Task{(uint32_t)i, pl.primary, pl.pool_level});
    }
    wait_in_flight();                                   // the previous call's block and records are free from here on
    w->n_records += n_records;
    // ---- formatting
    if (!w->to_files) {
        for (uint64_t i = 0; i < n_records; ++i) {
            const size_t before = w->console.size();
            w->format(w->console, *blk, recs[i], plans[i]);
            w->n_bytes += w->console.size() - before;
            if (w->console.size() >= flush_bytes()) { fwrite(w->console.data(), 1, w->console.size(), stdout); w->console.clear(); }
        }
    } else {
        w->cur_blk = blk; w->cur_recs = recs; w->cur_plans = &plans; w->cur_tasks = &tasks;
        if (w->n_threads > 1) {
            {
                std::lock_guard<std::mutex> lk(w->mu);
                w->pending = w->n_threads;
                ++w->generation;
            }
            w->cv_go.notify_all();
            w->in_flight = true;
            if (!deferred) wait_in_flight();
        } else {
            try { w->run_tasks(0); } catch (const std::exception &e) { w->note_error(SMX_IO_ERR_IO, e.what()); }
            for (uint64_t v : w->thread_bytes) w->n_bytes += v;
            w->cur_blk = nullptr; w->cur_recs = nullptr; w->cur_plans = nullptr; w->cur_tasks = nullptr;
        }
    }
    return w->error_status();
}

extern "C" {

int smx_writer_write(smx_writer *w, const smx_block *blk, const smx_record *recs, uint64_t n_records) {
    if (!w || !blk || (!recs && n_records)) return fail(SMX_IO_ERR_ARG, "smx_writer_write: null argument");
    if (n_records > 0xFFFFFFFFull) return fail(SMX_IO_ERR_ARG, "smx_writer_write: too many records in one call");
    const int set = w->next_set;
    w->next_set ^= 1;
    return w->write_planned(blk, recs, n_records, set, false);
}

int smx_writer_wait(smx_writer *w) {
    if (!w) return SMX_IO_OK;
    w->wait_in_flight();
    return w->error_status();
}


int smx_writer_write32(smx_writer *w, const smx_block *blk, const smx_record32 *recs, uint64_t n_records) {
    if (!w || !blk || (!recs && n_records)) return fail(SMX_IO_ERR_ARG, "smx_writer_write32: null argument");
    if (n_records > 0xFFFFFFFFull) return fail(SMX_IO_ERR_ARG, "smx_writer_write32: too many records in one call");
    // widen into the full layout (locations unused by the writer) and take the common path
    const int set = w->next_set;
    w->next_set ^= 1;
    std::vector<smx_record> &full = w->full_sets[set];
    full.resize((size_t)n_records);
    for (uint64_t i = 0; i < n_records; ++i) {
        const smx_record32 &c = recs[i];
        smx_record &r = full[i];
        memset(&r, 0, sizeof(r));
        r.read = c.read; r.sample = c.sample; r.trim_start = c.trim_start; r.trim_end = c.trim_end;
        r.pool = c.pool; r.p1 = c.p1; r.p2 = c.p2;
        for (int k = 0; k < 4; ++k) r.dist[k] = c.dist[k];
        r.resolution = c.resolution;
        r.reverse = c.flags & 1; r.trim_empty = (c.flags >> 1) & 1;
        r.candidate = c.candidate;
    }
    return w->write_planned(blk, full.data(), n_records, set, false);
}

static int write16_common(smx_writer *w, const smx_block *blk, const smx_record16 *recs, uint64_t n_records, bool deferred) {
    if (!w || !blk || (!recs && n_records)) return fail(SMX_IO_ERR_ARG, "smx_writer_write16: null argument");
    if (n_records > 0xFFFFFFFFull) return fail(SMX_IO_ERR_ARG, "smx_writer_write16: too many records in one call");
    // widen into the full layout: the read index comes from the last-of-read flags (records are in read order),
    // trim_end from the read's length
    const int set = w->next_set;
    w->next_set ^= 1;
    std::vector<smx_record> &full = w->full_sets[set];
    full.resize((size_t)n_records);
    uint32_t read = 0;
    const uint32_t n_reads = blk->n();
    for (uint64_t i = 0; i < n_records; ++i) {
        const smx_record16 &c = recs[i];
        if (read >= n_reads) return fail(SMX_IO_ERR_ARG, "smx_writer_write16: records run past the block's %u reads", n_reads);
        smx_record &r = full[i];
        memset(&r, 0, sizeof(r));
        const int64_t len = (int64_t)(blk->seq_off[read + 1] - blk->seq_off[read]);
        r.read = read; r.sample = c.sample; r.trim_start = c.trim_start; r.trim_end = (int32_t)(len - c.trim_tail);
        r.pool = c.pool; r.p1 = c.p1 == 0xFF ? -1 : c.p1; r.p2 = c.p2 == 0xFF ? -1 : c.p2;
        r.dist[0] = c.dist_p1 == 0xFF ? -1 : (int8_t)c.dist_p1;
        r.dist[1] = (c.dist_b & 0xF) == 0xF ? -1 : (int8_t)(c.dist_b & 0xF);
        r.dist[2] = (c.dist_b >> 4) == 0xF ? -1 : (int8_t)(c.dist_b >> 4);
        r.dist[3] = c.dist_p2 == 0xFF ? -1 : (int8_t)c.dist_p2;
        r.resolution = c.flags & 7;
        r.reverse = (c.flags >> 3) & 1; r.trim_empty = (c.flags >> 4) & 1;
        if (c.flags & 32) ++read;
    }
    return w->write_planned(blk, full.data(), n_records, set, deferred);
}

int smx_writer_write16(smx_writer *w, const smx_block *blk, const smx_record16 *recs, uint64_t n_records) {
    return write16_common(w, blk, recs, n_records, false);
}

int smx_writer_write16_deferred(smx_writer *w, const smx_block *blk, const smx_record16 *recs, uint64_t n_records) {
    return write16_common(w, blk, recs, n_records, true);
}

int smx_writer_close(smx_writer *w) {
    if (!w) return SMX_IO_OK;
    w->wait_in_flight();
    if (!w->threads.empty()) {
        { std::lock_guard<std::mutex> lk(w->mu); w->stop = true; }
        w->cv_go.notify_all();
        for (auto &t : w->threads) t.join();
    }
    for (Target *t : w->all_files) w->flush(t->file);
    if (!w->console.empty()) fwrite(w->console.data(), 1, w->console.size(), stdout);
    if (!w->to_files) fflush(stdout);
    int rc = w->first_error;
    if (rc != SMX_IO_OK) fail(rc, "%s", w->first_error_msg.c_str());
    delete w;
    return rc;
}

void smx_writer_stats(const smx_writer *w, uint64_t *records, uint64_t *bytes) {
    if (!w) return;
    if (records) *records = w->n_records;
    if (bytes) *bytes = w->n_bytes;
}

}  // extern "C"
