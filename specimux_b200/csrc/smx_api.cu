// smx_api.cu -- C ABI of libspecimux_b200.so (see include/specimux_b200.h).
// Context / table construction, batch buffers, kernel launches.  No CPU matching path exists:
// without a usable GPU every compute entry point fails with SMX_ERR_NO_DEVICE.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <memory>
#include <string>
#include <vector>

#include "smx_host_tables.hpp"
#include "smx_kernels.cuh"
#include "smx_launch.hpp"

using namespace smx;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail(e_ == cudaErrorNoDevice || e_ == cudaErrorInsufficientDriver          \
                            ? SMX_ERR_NO_DEVICE : SMX_ERR_CUDA,                               \
                        "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// Every CUDA resource the library keeps for itself is held by one of the owner types below and freed by its destructor.
template <typename T> struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { if (p) cudaFree(p); }
    // The first allocation is exact; a buffer that has to GROW takes a quarter more than asked: cudaFree / cudaMalloc
    // synchronise the device, and a stream of batches of slightly different sizes (the file pipeline's byte-range
    // chunks) would otherwise reallocate every buffer of a lane each time a new largest batch comes by.
    cudaError_t ensure(size_t n) {
        if (n <= cap) return cudaSuccess;
        size_t want = n;
        if (p) { cudaFree(p); want = n + n / 4; }
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc((void **)&p, want * sizeof(T));
        if (e != cudaSuccess && want != n) { (void)cudaGetLastError(); want = n; e = cudaMalloc((void **)&p, want * sizeof(T)); }
        if (e == cudaSuccess) cap = want;
        return e;
    }
};

// An event, stream or pinned host block: converts to the raw handle; the subclasses' ensure() creates it only while it
// is still null, so a call after a failed one creates what is missing and nothing twice.
template <typename H, cudaError_t (*Destroy)(H)> struct Handle {
    H h = nullptr;
    Handle() = default;
    Handle(const Handle &) = delete;
    Handle &operator=(const Handle &) = delete;
    ~Handle() { if (h) Destroy(h); }
    operator H() const { return h; }
};

struct Event : Handle<cudaEvent_t, cudaEventDestroy> {
    cudaError_t ensure(unsigned flags = cudaEventDefault) { return h ? cudaSuccess : cudaEventCreateWithFlags(&h, flags); }
};

struct Stream : Handle<cudaStream_t, cudaStreamDestroy> {
    cudaError_t ensure(int prio = 0) { return h ? cudaSuccess : cudaStreamCreateWithPriority(&h, cudaStreamNonBlocking, prio); }
};

template <typename T> cudaError_t free_host(T *p) { return cudaFreeHost(p); }

template <typename T> struct Pinned : Handle<T *, free_host<T>> {
    cudaError_t ensure(size_t n) {
        return this->h ? cudaSuccess : cudaHostAlloc((void **)&this->h, n * sizeof(T), cudaHostAllocDefault);
    }
};

template <typename T> cudaError_t upload(DevBuf<T> &d, const std::vector<T> &h) {
    cudaError_t e = d.ensure(h.size() ? h.size() : 1);
    if (e != cudaSuccess) return e;
    if (h.empty()) return cudaSuccess;
    return cudaMemcpy(d.p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice);
}

}  // namespace

// One pipeline lane: a stream plus every per-batch device buffer.  Lane 0 serves the resident API
// (upload / run / download on a whole batch); smx_match_batch splits large batches into chunks that
// rotate over all lanes so one chunk's H2D, another's kernels and a third's D2H overlap.
constexpr int kMaxLanes = 8;          // upper bound; the number in use is smx_ctx::n_lanes (SMX_PIPELINE_LANES)
constexpr int kAuxStreams = 2;
constexpr int kKernelMarks = 10;
constexpr int kKernelTimes = 9;
constexpr size_t kCtlWords = kCtrWords + SMX_MAX_PRIMERS;     // unsigned long long words of a lane's control block

// Members are destroyed in reverse order, so the streams, declared first, go last.
struct Lane {
    Stream stream;                          // H2D + kernels
    Stream out_stream;                      // D2H of finished results (pipelined form)
    Event ev_ready, ev_drained;             // records compacted / records copied out
    Stream aux[kAuxStreams];                // the per-primer sliced searches run side by side
    Event ev_fork, ev_join[kAuxStreams];
    Event ev_dp_done;                       // stage 1 + 2 (the ALU-bound kernels) of the lane's current chunk are through
    bool drain_pending = false;
    bool built = false;                     // lane_init has run to its end
    Event ev[5];
    Event kev[kKernelMarks];                // per-kernel boundaries of a timed (resident) run
    Batch b;
    DevBuf<u32> packed2, lengths, packed4, win, win2, tmix, endmask, impmask, rec_count, rec_offset, rec_offset_out, ticket;
    DevBuf<u64> word_off, off4;
    DevBuf<smx_primer_hit> phit;
    DevBuf<unsigned char> orient_hit, read_flags, bh_count;
    DevBuf<smx_barcode_hit> bh_list;
    DevBuf<BarcodeDigest> bdig;
    DevBuf<u32> ent_base, ent_read, rec_extra, big_list;
    DevBuf<unsigned short> ent_pos;
    DevBuf<u32> defer_list;
    DevBuf<smx_record> rec_stage, rec_pool, records;
    DevBuf<smx_record32> records32;             // compact copy of `records` (only when the caller asks for it)
    DevBuf<smx_record16> records16;             // 16-byte wire form of `records` (only when the caller asks for it)
    DevBuf<unsigned short> lengths16;           // 16-bit lengths as uploaded (expanded into `lengths` on the device)
    DevBuf<u32> bad16;                          // records whose extents did not fit smx_record16 (cumulative, must stay 0)
    DevBuf<unsigned char> big_scratch;
    // control block: 8 counters (4 work, matched, (u32,u32) overflow, (u32,u32) total/pool, hit overflow)
    // followed by the 2 * SMX_MAX_PRIMERS per-slot entry counts -- one memset, one read-back
    DevBuf<unsigned long long> counters;
    DevBuf<unsigned long long> tile_status;     // k_scan_compact: look-back status words (epoch-tagged, never cleared)
    u32 tickets_issued = 0, epoch = 0;          // cumulative tile tickets / launch epoch of k_scan_compact
    const u32 *offsets_src = nullptr;           // record offsets to copy out: rec_offset, or its rebased copy
    Event ev_counters;                          // control block has reached the pinned mirror
    u32 e_cap = 0, pool_cap = 0;
    int hit_cap = 0;                        // hit sub-list capacity the lane's buffers are laid out for
    Pinned<unsigned long long> h_counters;      // pinned mirror of the control block
    u32 *h_slot_counts = nullptr;               // = (u32 *)(h_counters + 8)
    bool have_batch = false, have_results = false;
    u64 n_records = 0, n_matched = 0;
    unsigned long long work[4] = {0, 0, 0, 0}, useful[2] = {0, 0};
    int launches = 0;
    u32 n_deferred = 0;
};

struct smx_ctx {
    int device = 0;
    Tables t;
    // table storage
    DevBuf<u64> peq_rc, peq_rcrev, peq_fw, spec_key, spec_p1, spec_p2;
    DevBuf<unsigned char> b_len, bw_len, bw_primer, b_codes;
    DevBuf<u32> b_code_off, bw_iupac;
    DevBuf<u32> pb_barcode, pair_fwd, pair_rev, spec_key_off, spec_row, bw_row, bw_valid, beq, peq_long;
    DevBuf<unsigned short> bw_list, bt_g0, bt_class_tasks;
    DevBuf<unsigned char> bt_nw;
    DevBuf<u32> bt_row, bt_eq, bt_quad;
    DevBuf<i32> bt_quad_row;
    std::vector<BtClass> bt_classes;
    DevBuf<i32> pair_pool, spec_pool, spec_dense;
    int max_nb = 0;
    std::vector<unsigned char> prow_code;   // [primer][32] pattern row codes (sliced primer search)
    Lane lane[kMaxLanes];
    int n_lanes = 3;
    // resident (upload / run / download) form: a large batch is cut into `resident_split` sub-batches
    // that run concurrently on separate lanes, so one sub-batch's latency-bound tail (general
    // selection, scan, compaction) overlaps another's ALU-bound search kernels
    int resident_split = 2, resident_lanes = 1;
    int resident_skew = 50;                 // two sub-batches: percent of the reads in the first (SMX_RESIDENT_SKEW)
    u32 resident_n = 0;
    Event ev_t0, ev_t1, ev_lane_done[kMaxLanes];
    DevBuf<u32> shared_packed4;            // pipelined mode: the (small) exact side stream, uploaded once
    DevBuf<unsigned char> l2_scratch;
    u32 chunk_reads = 256 * 1024;          // pipelined smx_match_batch: reads per chunk (SMX_PIPELINE_CHUNK); measured best
                                           // for the 16-byte wire records: 1.21 ms at 256k vs 1.29 ms at 128k (config 2)
    float total_ms = 0, stage_ms[4] = {0, 0, 0, 0}, kernel_ms[kKernelTimes] = {};
    int last_chunks = 0;
    bool trace = false;
    bool tiny_caps = false;                 // SMX_TEST_TINY_CAPS=1: see lane_upload
    bool start_sliced = false;              // bit-sliced start recovery kernel (SMX_START_SLICED=1): 4x fewer instructions than the
                                            // single-word form fused into the finish kernel, but latency-bound on its gather and
                                            // slower on the box (215 vs 58 us, profiles/r2_k_ab.md), so it is off by default
    bool lane_priorities = false;           // SMX_PIPELINE_PRIORITIES=1: earlier lanes get higher stream priority
    // pipelined smx_match_batch chunking (SMX_PIPELINE_RAMP): 0 = even split (default); 1 = two extra small
    // chunks first (measured 1.83 vs 1.76 ms on config 2: the extra chunks cost more kernel-chain latency than
    // the earlier first copy-out saves); 2 = same chunk count, first two chunks smaller (1.70 vs 1.70 ms)
    int ramp = 0;
    // pipelined smx_match_batch, SMX_PIPELINE_CHAIN=1: a chunk's kernels start only when the previous chunk's
    // ALU-bound stages (1 + 2) are through, so that chunks take the SMs one after the other and finish staggered.
    // Measured (profiles/r2_g_e2e_probe.txt): no gain -- one 128k..256k-read chunk does not fill the GPU (its ten
    // dependent launches take ~0.3 ms alone against 0.11 ms of pure throughput), so sharing the SMs among the
    // in-flight chunks is what keeps them busy: 1.21 ms unchained vs 1.23..1.37 ms chained on config 2.  Off.
    bool chain = false;
    // the device routes (DeviceCall): control words with their pinned mirror, the event that joins the caller's stream
    // and the timing marks
    DevBuf<unsigned long long> call_ctl;
    Pinned<unsigned long long> call_host;
    Event call_ev_in, call_ev_t[4];
    // smx_match_device: device packer scratch (per-read flags, the flagged-read list, scan tiles) and the event that
    // starts lanes 1.. after the packer
    DevBuf<u32> pk_flag, pk_list;
    DevBuf<u64> pk_tiles;
    Event pk_ev_packed;
    // smx_demux_device: the table sizes records are checked against, scratch of the index pass, tile marks of the copy
    smx_out::OutCounts out_counts = {};
    DevBuf<u64> dm_key_in, dm_key_out, dm_src, dm_out_src, dm_tiles;
    DevBuf<u32> dm_rec_in, dm_rec_out, dm_len;
    DevBuf<unsigned char> dm_temp;
    // smx_demux_files_device (besides the dm_ scratch): 64-bit slot lengths, header lengths and id positions per record,
    // first slot of each file
    DevBuf<u64> fl_len, fl_hdr, fl_id, fl_group;
    // smx_mine_device: the file offsets and group table as uploaded, per file its output range, per output its sequence,
    // length and search limit, per group its first pattern and entry, the work items, per entry its text, key, record
    // size, flag, winner and distance with the scans, per mined record its offset and kind
    DevBuf<u64> mn_file_off, mn_rng, mn_beg, mn_pat_base, mn_ent_base, mn_size, mn_size_off, mn_flag, mn_flag_off, mn_win, mn_rec_off;
    DevBuf<u32> mn_tab, mn_len, mn_ent_txt, mn_dist;
    DevBuf<i32> mn_k;
    DevBuf<HwItem> mn_items;
    DevBuf<unsigned long long> mn_keys;
    DevBuf<unsigned char> mn_kind, mn_temp;
    DevBuf<u32> mn_bad;
};
static_assert(kMaxLanes <= kPackMaxLanes, "PackLanes holds every lane");

// `prio`: CUDA stream priority of the lane (lower number = served first).  Lanes are filled in index
// order, so with SMX_PIPELINE_PRIORITIES=1 pending blocks of an earlier chunk are scheduled before a
// later one's instead of all in-flight chunks sharing the SMs evenly and finishing together.
static cudaError_t lane_init(Lane &ln, int prio = 0) {
    cudaError_t e;
    if (ln.built) return cudaSuccess;
    if ((e = ln.stream.ensure(prio)) != cudaSuccess) return e;
    if ((e = ln.out_stream.ensure()) != cudaSuccess) return e;
    if ((e = ln.ev_ready.ensure(cudaEventDisableTiming)) != cudaSuccess) return e;
    if ((e = ln.ev_fork.ensure(cudaEventDisableTiming)) != cudaSuccess) return e;
    if ((e = ln.ev_dp_done.ensure(cudaEventDisableTiming)) != cudaSuccess) return e;
    for (auto &a : ln.aux) if ((e = a.ensure(prio)) != cudaSuccess) return e;
    for (auto &j : ln.ev_join) if ((e = j.ensure(cudaEventDisableTiming)) != cudaSuccess) return e;
    if ((e = ln.ev_drained.ensure(cudaEventDisableTiming)) != cudaSuccess) return e;
    if ((e = ln.ev_counters.ensure(cudaEventDisableTiming)) != cudaSuccess) return e;
    for (auto &ev : ln.ev) if ((e = ev.ensure()) != cudaSuccess) return e;
    for (auto &ev : ln.kev) if ((e = ev.ensure()) != cudaSuccess) return e;
    if ((e = ln.h_counters.ensure(kCtlWords)) != cudaSuccess) return e;
    ln.h_slot_counts = (u32 *)(ln.h_counters + kCtrWords);
    if ((e = ln.counters.ensure(kCtlWords)) != cudaSuccess) return e;
    if ((e = ln.bad16.ensure(1)) != cudaSuccess) return e;
    if ((e = cudaMemset(ln.bad16.p, 0, sizeof(u32))) != cudaSuccess) return e;
    memset(&ln.b, 0, sizeof(ln.b));
    ln.built = true;
    return cudaSuccess;
}

static cudaError_t ensure_entry_buffers(smx_ctx *c, Lane &ln) {
    const Tables &t = c->t;
    cudaError_t e;
    if ((e = ln.ent_read.ensure((size_t)2 * t.n_primers * ln.e_cap)) != cudaSuccess) return e;
    if ((e = ln.ent_pos.ensure((size_t)2 * t.n_primers * ln.e_cap)) != cudaSuccess) return e;
    if ((e = ln.bh_count.ensure((size_t)2 * t.n_bwords * ln.e_cap + 1)) != cudaSuccess) return e;
    if ((e = ln.bh_list.ensure((size_t)2 * t.n_bwords * ln.hit_cap * ln.e_cap + 1)) != cudaSuccess) return e;
    if ((e = ln.bdig.ensure((size_t)2 * t.n_btasks * ln.e_cap + 1)) != cudaSuccess) return e;
    if ((e = ln.rec_pool.ensure(ln.pool_cap)) != cudaSuccess) return e;
    Batch &b = ln.b;
    b.e_cap = ln.e_cap; b.pool_cap = ln.pool_cap;
    b.ent_read = ln.ent_read.p; b.ent_pos = ln.ent_pos.p; b.bh_count = ln.bh_count.p; b.bh_list = ln.bh_list.p; b.bdig = ln.bdig.p;
    b.rec_pool = ln.rec_pool.p;
    return cudaSuccess;
}

// Tables as launched from this lane (the hit sub-list capacity is a per-lane layout parameter).
static Tables lane_tables(const smx_ctx *c, const Lane &ln) {
    Tables t = c->t;
    t.hit_cap = ln.hit_cap;
    return t;
}

// Sizes every per-batch buffer of a lane for n reads in `words` packed2 words (word_off: per-read offsets,
// lengths16: 16-bit lengths on the wire; the side stream is sized by the caller).  Issues nothing that reads the batch.
static int lane_size(smx_ctx *c, Lane &ln, u32 n, u64 words, bool word_off, bool lengths16) {
    const Tables &t = c->t;
    const u32 n_pad = (n + 127u) & ~127u;
    const int nP = t.n_primers;
    {
        int prio = 0;
        if (c->lane_priorities) {
            int lo = 0, hi = 0;                                 // hi = greatest priority (numerically lowest)
            CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));
            const int idx = (int)(&ln - c->lane);
            prio = std::min(lo, hi + idx);
        }
        CU(lane_init(ln, prio));
    }
    ln.launches = 0;
    CU(ln.packed2.ensure(words + 2)); if (word_off) CU(ln.word_off.ensure(n)); CU(ln.lengths.ensure(n));
    if (lengths16) CU(ln.lengths16.ensure(n));
    CU(ln.win.ensure((size_t)2 * t.wpw * n_pad));
    CU(ln.win2.ensure((size_t)2 * t.nw2 * n_pad));
    if (t.sliced) CU(ln.tmix.ensure((size_t)2 * nP * t.nw2 * n_pad));
    CU(ln.phit.ensure((size_t)2 * nP * n_pad));
    CU(ln.endmask.ensure((size_t)2 * nP * t.mw * n_pad));
    CU(ln.impmask.ensure((size_t)2 * nP * t.mw * n_pad));
    CU(ln.orient_hit.ensure((size_t)2 * nP * n_pad));
    CU(ln.ent_base.ensure((size_t)2 * nP * n_pad));
    CU(ln.defer_list.ensure(n_pad)); CU(ln.big_list.ensure(n_pad));
    if (c->tiny_caps) {
        // test hook (SMX_TEST_TINY_CAPS=1): start every growable buffer far too small so that each
        // capacity re-run of lane_resolve() is exercised on the device
        if (ln.e_cap < 128) ln.e_cap = 128;
        if (ln.pool_cap < 4) ln.pool_cap = 4;
    } else {
        if (ln.e_cap < n_pad + n_pad / 4) ln.e_cap = n_pad + n_pad / 4;     // ~1.2 equal-best ends per matched slot is typical
        if (ln.pool_cap < n_pad / 8 + 1024) ln.pool_cap = n_pad / 8 + 1024;
    }
    if (ln.hit_cap < c->t.hit_cap) ln.hit_cap = c->t.hit_cap;
    CU(ensure_entry_buffers(c, ln));
    CU(ln.rec_stage.ensure(n_pad)); CU(ln.rec_extra.ensure(n_pad));
    CU(ln.rec_count.ensure(n)); CU(ln.rec_offset.ensure((size_t)n + 1)); CU(ln.rec_offset_out.ensure((size_t)n + 1));
    CU(ln.read_flags.ensure(n));
    cudaStream_t st = ln.stream;
    {
        const size_t tiles = ((size_t)n + kScanTile - 1) / kScanTile + 1;
        if (ln.tile_status.cap < tiles) {       // fresh status words must not carry a plausible epoch tag
            CU(ln.tile_status.ensure(tiles));
            CU(cudaMemsetAsync(ln.tile_status.p, 0, ln.tile_status.cap * sizeof(unsigned long long), st));
        }
        if (!ln.ticket.p) {
            CU(ln.ticket.ensure(1));
            CU(cudaMemsetAsync(ln.ticket.p, 0, sizeof(u32), st));
            ln.tickets_issued = 0;
        }
    }
    // compacted records: one per read plus whatever the pool can hold (grown by lane_resolve if a
    // second selection pass produces more)
    if (ln.records.cap < (size_t)n_pad + ln.pool_cap + 1) {
        if (ln.drain_pending) CU(cudaEventSynchronize(ln.ev_drained));      // the old buffer is still being copied out
        CU(ln.records.ensure((size_t)n_pad + ln.pool_cap + 1));
    }
    return SMX_OK;
}

// Binds the lane's buffers to its Batch: n reads, the caller's reads [r0, r0 + n), packed2[0] = stream word w0;
// packed4 / off4 nullptr when no read of the batch is flagged.
static void lane_bind(Lane &ln, u32 n, u32 clip, u32 stride, u64 w0, u32 r0, const u32 *packed4, const u64 *off4) {
    Batch &b = ln.b;
    b.n_reads = n; b.n_pad = (n + 127u) & ~127u; b.clip = clip; b.stride = stride; b.word_base = w0; b.read_base = r0;
    b.packed2 = ln.packed2.p; b.word_off = stride ? nullptr : ln.word_off.p; b.lengths = ln.lengths.p;
    b.packed4 = packed4; b.off4 = off4;
    b.win = ln.win.p; b.win2 = ln.win2.p; b.tmix = ln.tmix.p; b.phit = ln.phit.p; b.endmask = ln.endmask.p; b.impmask = ln.impmask.p; b.orient_hit = ln.orient_hit.p;
    b.slot_count = (u32 *)(ln.counters.p + kCtrWords); b.ent_base = ln.ent_base.p; b.defer_list = ln.defer_list.p; b.big_list = ln.big_list.p;
    b.rec_stage = ln.rec_stage.p; b.rec_extra = ln.rec_extra.p;
    b.rec_count = ln.rec_count.p; b.rec_offset = ln.rec_offset.p;
    b.records = ln.records.p; b.read_flags = ln.read_flags.p; b.counters = ln.counters.p;
    ln.have_batch = true; ln.have_results = false;
}

// H2D of reads [r0, r1) of `in` onto the lane (asynchronous on the lane's stream) and binding of
// every per-batch buffer.  `shared4`: device copy of the whole packed4 stream (pipelined mode) or
// nullptr (the lane uploads it itself; only valid for r0 == 0, r1 == n_reads).
static int lane_upload(smx_ctx *c, Lane &ln, const smx_batch *in, u32 r0, u32 r1, const u32 *shared4) {
    const u32 n = r1 - r0;
    const u64 stride = in->stride_words;
    const u64 w0 = stride ? (u64)r0 * stride : in->word_off[r0];
    const u64 w1 = stride ? std::min<u64>((u64)r1 * stride + 1, in->packed2_words)
                          : ((r1 < in->n_reads) ? std::min<u64>(in->word_off[r1] + 1, in->packed2_words) : in->packed2_words);
    if (w1 < w0) return fail(SMX_ERR_ARG, "smx_batch: word_off is not ascending");
    int rc = lane_size(c, ln, n, w1 - w0, !stride, in->lengths16 != nullptr);
    if (rc) return rc;
    const bool flagged = in->packed4 && in->off4 && in->packed4_words;
    if (flagged) { CU(ln.off4.ensure(n)); if (!shared4) CU(ln.packed4.ensure(in->packed4_words)); }
    cudaStream_t st = ln.stream;
    CU(cudaMemcpyAsync(ln.packed2.p, in->packed2 + w0, (w1 - w0) * sizeof(u32), cudaMemcpyHostToDevice, st));
    if (!stride) CU(cudaMemcpyAsync(ln.word_off.p, in->word_off + r0, (size_t)n * sizeof(u64), cudaMemcpyHostToDevice, st));
    if (in->lengths16) {
        CU(cudaMemcpyAsync(ln.lengths16.p, in->lengths16 + r0, (size_t)n * sizeof(unsigned short), cudaMemcpyHostToDevice, st));
        CU(launch_expand_lengths(ln.lengths16.p, n, ln.lengths.p, st));
        ++ln.launches;
    } else {
        CU(cudaMemcpyAsync(ln.lengths.p, in->lengths + r0, (size_t)n * sizeof(u32), cudaMemcpyHostToDevice, st));
    }
    if (flagged) {
        if (!shared4)
            CU(cudaMemcpyAsync(ln.packed4.p, in->packed4, in->packed4_words * sizeof(u32), cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(ln.off4.p, in->off4 + r0, (size_t)n * sizeof(u64), cudaMemcpyHostToDevice, st));
    }
    lane_bind(ln, n, in->clip_len, (u32)stride, w0, r0, flagged ? (shared4 ? shared4 : ln.packed4.p) : nullptr,
              flagged ? ln.off4.p : nullptr);
    return SMX_OK;
}

// rec_count -> rec_offset, flag counters and the read-ordered compaction of the records in one
// launch (k_scan_compact), then the asynchronous read-back of the whole control block (counters +
// per-slot entry counts).  Nothing waits for the host here: the records buffer is sized up front and
// lane_resolve() re-runs this step if a second selection pass outgrows it.
static cudaError_t enqueue_scan_compact(smx_ctx *c, Lane &ln) {
    Batch &b = ln.b;
    const u32 n = b.n_reads;
    cudaStream_t st = ln.stream;
    cudaError_t e;
    if (ln.drain_pending) {                 // the previous chunk's records are still being copied out of ln.records
        if ((e = cudaStreamWaitEvent(st, ln.ev_drained, 0)) != cudaSuccess) return e;
        ln.drain_pending = false;
    }
    const unsigned tiles = (n + kScanTile - 1) / kScanTile;
    ln.epoch = ln.epoch % ((1u << 30) - 1u) + 1u;
    const u32 cap = (u32)std::min<size_t>(ln.records.cap, 0xFFFFFFFFu);
    if ((e = launch_scan_compact(lane_tables(c, ln), b, cap, ln.tile_status.p, ln.ticket.p, ln.tickets_issued, ln.epoch, st)) != cudaSuccess) return e;
    ln.tickets_issued += tiles;
    ++ln.launches;
    if ((e = cudaMemcpyAsync(ln.h_counters, ln.counters.p, kCtlWords * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
    return cudaEventRecord(ln.ev_counters, st);
}

// Zeroes what k_scan_compact accumulates into (matched reads, overflow flags, record total) but
// keeps the pool usage in the upper half of counter 6.
static cudaError_t reset_scan_counters(Lane &ln) {
    cudaError_t e = cudaMemsetAsync(ln.counters.p + 4, 0, 2 * sizeof(unsigned long long), ln.stream);
    if (e != cudaSuccess) return e;
    return cudaMemsetAsync(ln.counters.p + 6, 0, sizeof(u32), ln.stream);
}

// Enqueues stages `from`..3 (0 = from window staging) through the scan and the counter read-back.
// Nothing here synchronises; lane_resolve() looks at the counters.
static int lane_enqueue(smx_ctx *c, Lane &ln, int from, bool timed) {
    const Tables t = lane_tables(c, ln);
    Batch &b = ln.b;
    const u32 n = b.n_reads;
    const int nP = t.n_primers;
    cudaStream_t st = ln.stream;
#define KMARK(i) do { if (timed) CU(cudaEventRecord(ln.kev[i], st)); } while (0)
    bool start_forked = false;
    (void)n;
    if (from <= 0) {
        CU(cudaMemsetAsync(ln.counters.p, 0, kCtlWords * sizeof(unsigned long long), st));     // the only memset of a fresh run
        if (timed) CU(cudaEventRecord(ln.ev[0], st));
        KMARK(0);
        CU(launch_stage_windows(t, b, st));
        ++ln.launches;
    }
    if (from <= 1) {   // stage 1
        if (from == 1) CU(cudaMemsetAsync(ln.counters.p, 0, kCtlWords * sizeof(unsigned long long), st));   // re-run
        if (timed) CU(cudaEventRecord(ln.ev[1], st));
        KMARK(1);
        if (t.sliced) {
            // forward pass bit-sliced across reads, one launch per primer (pattern length = template)
            // The primers' kernels are independent and each fills only ~2.5 warps per scheduler at
            // 765k reads, so they run concurrently on auxiliary streams (fork / join on events).
            const bool fork = nP > 1;
            if (fork) CU(cudaEventRecord(ln.ev_fork, st));
            for (int p = 0; p < nP; ++p) {
                cudaStream_t ps = fork ? ln.aux[p % kAuxStreams] : st;
                if (fork && p < kAuxStreams) CU(cudaStreamWaitEvent(ps, ln.ev_fork, 0));
                CU(launch_primer_sliced(t, b, p, c->prow_code.data() + (size_t)p * 32, ps));
                ++ln.launches;
            }
            if (fork)
                for (int a = 0; a < kAuxStreams && a < nP; ++a) {
                    CU(cudaEventRecord(ln.ev_join[a], ln.aux[a]));
                    CU(cudaStreamWaitEvent(st, ln.ev_join[a], 0));
                }
        }
        KMARK(2);
        CU(launch_primer_finish(t, b, c->start_sliced ? 1 : 2, st));
        for (int p = 0; p < nP; ++p) {
            if (!t.p_sw[p]) continue;
            // long primer: warp-cooperative multi-word search, p_sw lanes per read
            CU(launch_primer_long(t, b, p, st));
            ++ln.launches;
        }
        KMARK(3);
        ++ln.launches;
        // start of the first location, bit-sliced across work entries: independent of the barcode search (selection
        // needs both), so outside timed one-lane runs it goes to an auxiliary stream beside stage 2
        if (c->start_sliced) {
            cudaStream_t ss = st;
            bool any = false;
            for (int p = 0; p < nP; ++p) any |= start_sliced_ok(t, p);
            if (any && !timed) {
                ss = ln.aux[0];
                CU(cudaEventRecord(ln.ev_fork, st));
                CU(cudaStreamWaitEvent(ss, ln.ev_fork, 0));
                start_forked = true;
            }
            for (int p = 0; p < nP; ++p) {
                if (!start_sliced_ok(t, p)) continue;
                CU(launch_primer_start_sliced(t, b, p, c->prow_code.data() + (size_t)p * 32, ss));
                ++ln.launches;
            }
            if (start_forked) CU(cudaEventRecord(ln.ev_join[0], ss));
        }
    }
    if (from <= 2) {   // stage 2
        if (from == 2) {                                                                                     // re-run
            CU(cudaMemsetAsync(ln.counters.p + 1, 0, sizeof(unsigned long long), st));
            CU(cudaMemsetAsync(ln.counters.p + 3, 0, sizeof(unsigned long long), st));
            CU(cudaMemsetAsync(ln.counters.p + 7, 0, sizeof(unsigned long long), st));
            CU(cudaMemsetAsync(ln.counters.p + kCtrUseful2, 0, sizeof(unsigned long long), st));
        }
        if (timed) CU(cudaEventRecord(ln.ev[2], st));
        KMARK(4);
        if (t.n_btasks) CU(launch_barcode_tasks(t, b, c->bt_class_tasks.p, c->bt_classes.data(), (int)c->bt_classes.size(), st, &ln.launches));
    }
    CU(cudaEventRecord(ln.ev_dp_done, st));
    if (start_forked) CU(cudaStreamWaitEvent(st, ln.ev_join[0], 0));
    // stage 3: slot digests, single-pass selection, scan
    if (from >= 2) {                                                                                           // re-run
        CU(cudaMemsetAsync(ln.counters.p + 4, 0, 3 * sizeof(unsigned long long), st));
        CU(cudaMemsetAsync(ln.counters.p + kCtrDeferred, 0, 2 * sizeof(unsigned long long), st));      // + kCtrBig
    }
    if (timed) CU(cudaEventRecord(ln.ev[3], st));
    KMARK(5);
    // fast path for (nearly) every read, then the general routine over the reads it deferred
    CU(launch_select_fast(t, b, st));
    KMARK(6);
    CU(launch_select(t, b, st));
    ln.launches += 2;
    KMARK(7);
    CU(enqueue_scan_compact(c, ln));
    KMARK(8);
#undef KMARK
    return SMX_OK;
}

// Waits for the lane's counters and resolves every capacity overflow by re-running the affected
// stages with larger buffers (never "unsupported"); runs the second selection pass for reads that
// overflowed the thread-local group storage.  On return n_records / n_matched / work are final.
static int lane_resolve(smx_ctx *c, Lane &ln, bool timed) {
    Batch &b = ln.b;
    const int nP = c->t.n_primers;
    cudaStream_t st = ln.stream;
    bool big_done = false;
    for (;;) {
        CU(cudaEventSynchronize(ln.ev_counters));
        unsigned long long *hc = ln.h_counters;
        u32 max_entries = 0;
        for (int i = 0; i < 2 * nP; ++i) max_entries = std::max(max_entries, ln.h_slot_counts[i]);
        int from = -1;
        if (max_entries > ln.e_cap) {
            ln.e_cap = (max_entries + 127u) & ~127u;
            from = 1;
        } else if (hc[7]) {
            if (ln.hit_cap >= kMaxWordHits) return fail(SMX_ERR_INTERNAL, "hit list overflow at maximum capacity");
            ln.hit_cap = std::min(kMaxWordHits, ln.hit_cap * 4);
            if (c->t.hit_cap < ln.hit_cap) c->t.hit_cap = ln.hit_cap;     // later uploads start there
            from = 2;
        } else if ((u32)(hc[6] >> 32) > ln.pool_cap) {
            ln.pool_cap = (u32)(hc[6] >> 32) + 1024;
            from = 3;
        }
        if (from >= 0) {
            CU(cudaStreamSynchronize(st));              // buffers are about to be replaced
            CU(ensure_entry_buffers(c, ln));
            int rc = lane_enqueue(c, ln, from, timed);
            if (rc) return rc;
            big_done = false;
            continue;
        }
        const u32 n_big = (u32)hc[kCtrBig];
        if (n_big && !big_done) {
            // some reads overflowed the thread-local group storage or emit many records: second GPU
            // pass for those reads only, on kBigGroups-entry global scratch, list already on the device
            if (c->trace) fprintf(stderr, "[smx resolve] %u of %u reads take the second selection pass\n", n_big, b.n_reads);
            const Tables t = lane_tables(c, ln);
            const size_t chunk = 512;
            CU(ln.big_scratch.ensure(std::min<size_t>(chunk, n_big) * kBigScratchBytes));
            for (size_t off = 0; off < n_big; off += chunk) {
                u32 cnt = (u32)std::min<size_t>(chunk, n_big - off);
                CU(launch_select_big(t, b, ln.big_list.p + off, cnt, ln.big_scratch.p, st));
                ++ln.launches;
            }
            CU(reset_scan_counters(ln));
            CU(enqueue_scan_compact(c, ln));            // offsets and compaction again, now with the big reads' records
            big_done = true;
            continue;
        }
        if ((u32)(hc[5] >> 32))
            return fail(SMX_ERR_INTERNAL, "selection: %u read(s) exceed %d dereplication groups",
                        (unsigned)(hc[5] >> 32), kBigGroups);
        if ((u32)hc[6] > ln.records.cap) {
            // more records than the compaction buffer holds (k_scan_compact skipped what did not fit)
            CU(cudaStreamSynchronize(st));
            if (ln.drain_pending) { CU(cudaEventSynchronize(ln.ev_drained)); ln.drain_pending = false; }
            CU(ln.records.ensure((size_t)(u32)hc[6] + 1024));
            b.records = ln.records.p;
            CU(reset_scan_counters(ln));
            CU(enqueue_scan_compact(c, ln));
            continue;
        }
        break;
    }
    ln.n_records = (u32)ln.h_counters[6];
    ln.n_matched = ln.h_counters[4];
    ln.n_deferred = (u32)ln.h_counters[kCtrDeferred];
    for (int i = 0; i < 4; ++i) ln.work[i] = ln.h_counters[i];
    ln.useful[0] = ln.h_counters[kCtrUseful1]; ln.useful[1] = ln.h_counters[kCtrUseful2];
    return SMX_OK;
}

// Compact forms of the lane's compacted records (smx_record32 / smx_record16), produced on the lane's OWN stream: the
// kernels read the lane's batch buffers (lengths), which the lane's next upload overwrites.
static int lane_pack_records(Lane &ln, const smx_results *out) {
    if (!ln.n_records || out->records) return SMX_OK;
    cudaStream_t st = ln.stream;
    if (out->records32) {
        CU(ln.records32.ensure((size_t)ln.n_records));
        CU(launch_pack_records32(ln.records.p, (u32)ln.n_records, ln.records32.p, st));
        ++ln.launches;
    } else if (out->records16) {
        CU(ln.records16.ensure((size_t)ln.n_records));
        CU(launch_pack_records16(ln.records.p, (u32)ln.n_records, ln.b.lengths, ln.b.read_base, ln.records16.p, ln.bad16.p, st));
        ++ln.launches;
    }
    return SMX_OK;
}

// Copy-out of a lane's records into the caller's array, full or compact form (asynchronous on `st`, which must
// already be ordered after the lane's kernels and lane_pack_records).
static int lane_copy_records(Lane &ln, smx_results *out, u64 rec_base, cudaStream_t st) {
    if (!ln.n_records) return SMX_OK;
    if (out->records)
        CU(cudaMemcpyAsync(out->records + rec_base, ln.records.p, (size_t)ln.n_records * sizeof(smx_record), cudaMemcpyDeviceToHost, st));
    else if (out->records32)
        CU(cudaMemcpyAsync(out->records32 + rec_base, ln.records32.p, (size_t)ln.n_records * sizeof(smx_record32), cudaMemcpyDeviceToHost, st));
    else if (out->records16)
        CU(cudaMemcpyAsync(out->records16 + rec_base, ln.records16.p, (size_t)ln.n_records * sizeof(smx_record16), cudaMemcpyDeviceToHost, st));
    return SMX_OK;
}

// The records are already compacted (k_scan_compact); what is left is the sub-batch's record offsets
// in the caller's whole batch (asynchronous).
static int lane_compact(smx_ctx *c, Lane &ln, u32 rec_base, bool timed) {
    (void)c;
    Batch &b = ln.b;
    cudaStream_t st = ln.stream;
    if (timed) CU(cudaEventRecord(ln.kev[9], st));
    ln.offsets_src = b.rec_offset;
    if (rec_base) {
        CU(launch_rebase_offsets(b.rec_offset, b.n_reads, rec_base, ln.rec_offset_out.p, st));
        ++ln.launches;
        ln.offsets_src = ln.rec_offset_out.p;
    }
    if (timed) CU(cudaEventRecord(ln.ev[4], st));
    CU(cudaGetLastError());
    ln.have_results = true;
    return SMX_OK;
}

// smx_record16 carries 16-bit extents: fail loudly if a record of the last call did not fit (never observed:
// both extents lie within search_len + barcode length of a read end).
static int check_record16_fit(smx_ctx *c) {
    u32 bad = 0;
    for (auto &ln : c->lane) {
        if (!ln.stream || !ln.bad16.p) continue;
        u32 v = 0;
        CU(cudaMemcpy(&v, ln.bad16.p, sizeof(u32), cudaMemcpyDeviceToHost));
        if (v) CU(cudaMemset(ln.bad16.p, 0, sizeof(u32)));
        bad += v;
    }
    if (bad) return fail(SMX_ERR_INTERNAL, "%u record(s) do not fit smx_record16 (trim extent or id beyond its field); "
                                           "ask for smx_record32 records", bad);
    return SMX_OK;
}

extern "C" {

int smx_abi_version(void) { return SMX_ABI_VERSION; }

const char *smx_last_error(void) { return g_err; }

int smx_device_pci_bus_id(int device, char *out, int len) {
    if (!out || len < 16) return fail(SMX_ERR_ARG, "smx_device_pci_bus_id: buffer too small");
    CU(cudaDeviceGetPCIBusId(out, len, device));
    return SMX_OK;
}

int smx_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

void smx_destroy(smx_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    for (auto &ln : c->lane) if (ln.stream) { cudaStreamSynchronize(ln.stream); cudaStreamSynchronize(ln.out_stream); }
    delete c;
}

int smx_create(int device, const smx_tables *tb, const smx_params *pr, smx_ctx **out) {
    if (!tb || !pr || !out) return fail(SMX_ERR_ARG, "smx_create: null argument");
    *out = nullptr;
    HostTables ht;
    if (!ht.build(tb, pr)) return fail(SMX_ERR_ARG, "smx_create: %s", ht.error.c_str());
    if (ht.t.k_idx > kMaxBarcodeK)
        return fail(SMX_ERR_ARG, "smx_create: barcode distance threshold %d exceeds the supported %d", ht.t.k_idx, kMaxBarcodeK);
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(SMX_ERR_NO_DEVICE, "smx_create: no CUDA device (%s); this library has no CPU path",
                    ce != cudaSuccess ? cudaGetErrorString(ce) : "device count 0");
    }
    if (device < 0 || device >= ndev) return fail(SMX_ERR_ARG, "smx_create: device %d of %d", device, ndev);

    std::unique_ptr<smx_ctx> c(new smx_ctx());     // freed with everything it holds unless it reaches *out
    c->device = device;
    c->max_nb = ht.max_nb;
    c->prow_code = ht.prow_code;
    {
        // pool ids are dense over the pairs' and specimens' pools (smx_names.pool lists them in id order)
        int32_t top = -1;
        for (u32 i = 0; i < tb->n_pairs; ++i) top = std::max(top, tb->pair_pool[i]);
        for (u32 i = 0; i < tb->n_specimens; ++i) top = std::max(top, tb->spec_pool[i]);
        c->out_counts = {tb->n_specimens, tb->n_b1, tb->n_b2, (u32)(top + 1), tb->n_primers};
    }
    CU(cudaSetDevice(device));
    {
        int prio = 0;
        if (const char *env = getenv("SMX_PIPELINE_PRIORITIES")) c->lane_priorities = atoi(env) != 0;
        if (c->lane_priorities) { int lo = 0; CU(cudaDeviceGetStreamPriorityRange(&lo, &prio)); }
        CU(lane_init(c->lane[0], prio));
    }
    CU(upload(c->peq_rc, ht.peq_rc)); CU(upload(c->peq_rcrev, ht.peq_rcrev)); CU(upload(c->peq_fw, ht.peq_fw));
    CU(upload(c->b_len, ht.b_len)); CU(upload(c->pb_barcode, ht.pb_barcode));
    CU(upload(c->bw_len, ht.bw_len)); CU(upload(c->bw_primer, ht.bw_primer)); CU(upload(c->bw_row, ht.bw_row));
    CU(upload(c->bw_valid, ht.bw_valid)); CU(upload(c->bw_list, ht.bw_list)); CU(upload(c->beq, ht.beq));
    CU(upload(c->pair_fwd, ht.pair_fwd)); CU(upload(c->pair_rev, ht.pair_rev)); CU(upload(c->pair_pool, ht.pair_pool));
    CU(upload(c->spec_key, ht.spec_key)); CU(upload(c->spec_key_off, ht.spec_key_off));
    CU(upload(c->spec_row, ht.spec_row)); CU(upload(c->spec_p1, ht.spec_p1)); CU(upload(c->spec_p2, ht.spec_p2));
    CU(upload(c->spec_pool, ht.spec_pool));
    CU(upload(c->spec_dense, ht.spec_dense));
    CU(upload(c->peq_long, ht.peq_long));
    CU(upload(c->bt_g0, ht.bt_g0)); CU(upload(c->bt_nw, ht.bt_nw)); CU(upload(c->bt_row, ht.bt_row));
    CU(upload(c->bt_eq, ht.bt_eq)); CU(upload(c->bt_class_tasks, ht.bt_class_tasks));
    c->bt_classes = ht.bt_classes;
    ht.set_task_pointers(c->bt_g0.p, c->bt_nw.p, c->bt_row.p, c->bt_eq.p);
    CU(upload(c->bt_quad, ht.bt_quad)); CU(upload(c->bt_quad_row, ht.bt_quad_row));
    ht.set_quad_pointers(c->bt_quad_row.p, c->bt_quad.p);
    CU(upload(c->b_codes, ht.b_codes)); CU(upload(c->b_code_off, ht.b_code_off)); CU(upload(c->bw_iupac, ht.bw_iupac));
    ht.set_code_pointers(c->b_codes.p, c->b_code_off.p, c->bw_iupac.p);
    ht.set_bword_pointers(c->bw_len.p, c->bw_primer.p, c->bw_row.p, c->bw_valid.p, c->bw_list.p, c->beq.p);
    ht.set_pointers(c->peq_rc.p, c->peq_rcrev.p, c->peq_fw.p, c->b_len.p, c->pb_barcode.p,
                    c->pair_fwd.p, c->pair_rev.p, c->pair_pool.p, c->spec_key.p, c->spec_key_off.p,
                    c->spec_row.p, c->spec_p1.p, c->spec_p2.p, c->spec_pool.p);
    c->t = ht.t;
    c->t.spec_dense = ht.spec_dense.empty() ? nullptr : c->spec_dense.p;
    c->t.peq_long = c->peq_long.p;
    if (const char *env = getenv("SMX_PIPELINE_CHUNK")) {
        long v = atol(env);
        if (v >= 128) c->chunk_reads = (u32)std::min<long>(v, 1L << 30);
        else if (v == 0) c->chunk_reads = 0;                   // 0 disables the pipelined form
    }
    if (const char *env = getenv("SMX_PIPELINE_LANES")) c->n_lanes = std::max(2, std::min(kMaxLanes, atoi(env)));
    if (const char *env = getenv("SMX_RESIDENT_SKEW")) c->resident_skew = std::max(10, std::min(90, atoi(env)));
    if (const char *env = getenv("SMX_RESIDENT_SPLIT")) c->resident_split = std::max(1, std::min(kMaxLanes, atoi(env)));
    if (const char *env = getenv("SMX_PRIMER_SLICED")) if (atoi(env) == 0) c->t.sliced = 0;     // A/B switch: classic stage 1
    if (const char *env = getenv("SMX_PIPELINE_PRIORITIES")) c->lane_priorities = atoi(env) != 0;
    if (const char *env = getenv("SMX_TEST_TINY_CAPS")) c->tiny_caps = atoi(env) != 0;
    if (const char *env = getenv("SMX_START_SLICED")) c->start_sliced = atoi(env) != 0;
    if (const char *env = getenv("SMX_PIPELINE_RAMP")) c->ramp = atoi(env);
    if (const char *env = getenv("SMX_PIPELINE_CHAIN")) c->chain = atoi(env) != 0;
    if (const char *env = getenv("SMX_PIPELINE_TRACE")) c->trace = atoi(env) != 0;
    *out = c.release();
    return SMX_OK;
}

uint64_t smx_result_bound(const smx_ctx *c, uint32_t n_reads) {
    // Every read yields >= 1 record; multi-record reads (tied specimens / partial barcodes) are rare.
    // smx_download_results reports SMX_ERR_CAPACITY with the exact need if this is ever exceeded.
    (void)c;
    return (uint64_t)n_reads * 2 + 1024;
}

static int check_batch(const smx_ctx *c, const smx_batch *in, const char *who) {
    if (!c || !in) return fail(SMX_ERR_ARG, "%s: null argument", who);
    if (in->n_reads == 0) return fail(SMX_ERR_ARG, "%s: empty batch", who);
    if (!in->packed2 || (!in->word_off && !in->stride_words) || (!in->lengths && !in->lengths16))
        return fail(SMX_ERR_ARG, "%s: null batch array", who);
    if (in->stride_words && (u64)in->n_reads * in->stride_words > in->packed2_words)
        return fail(SMX_ERR_ARG, "%s: packed2 holds fewer than n_reads * stride_words words", who);
    if (in->clip_len && (int)in->clip_len < c->t.L)
        return fail(SMX_ERR_ARG, "%s: clip_len %u is below search_len %d", who, in->clip_len, c->t.L);
    if ((in->packed4 == nullptr) != (in->off4 == nullptr) && in->packed4_words)
        return fail(SMX_ERR_ARG, "%s: packed4 and off4 must be given together", who);
    return SMX_OK;
}

constexpr u32 kResidentSplitMin = 1u << 17;     // batches below this many reads stay on one lane

static void resident_bounds(const smx_ctx *c, int i, u32 &r0, u32 &r1) {
    const u32 n = c->resident_n;
    if (c->resident_lanes == 2 && c->resident_skew != 50) {
        // uneven halves: the lanes then reach their latency-bound selection tails at different times
        const u32 mid = (u32)(((u64)n * (u32)c->resident_skew / 100u) + 127u) & ~127u;
        r0 = i == 0 ? 0 : std::min(mid, n);
        r1 = i == 0 ? std::min(mid, n) : n;
        return;
    }
    const u32 per = (((n + (u32)c->resident_lanes - 1) / (u32)c->resident_lanes) + 127u) & ~127u;
    r0 = (u32)std::min<u64>((u64)i * per, n);
    r1 = (u32)std::min<u64>((u64)(i + 1) * per, n);
}

// A new resident batch of n reads: how many lanes it takes (resident_bounds cuts it); no lane holds a batch or results.
static void resident_begin(smx_ctx *c, u32 n) {
    c->resident_n = n;
    c->resident_lanes = (c->resident_split > 1 && n >= kResidentSplitMin) ? c->resident_split : 1;
    for (auto &ln : c->lane) { ln.have_batch = false; ln.have_results = false; }
}

// The bound sub-batches of lanes 0..S-1, untimed and side by side: every lane's kernels are enqueued before any lane
// is resolved; lane i's records follow those of lanes 0..i-1.  Lane::launches accumulates (the callers reset it).
static int resident_lanes_run(smx_ctx *c, int S, const char *fn, u64 *n_records, u64 *n_matched) {
    int rc;
    for (int i = 0; i < S; ++i)
        if ((rc = lane_enqueue(c, c->lane[i], 0, false))) return rc;
    u64 rec_base = 0, matched = 0;
    for (int i = 0; i < S; ++i) {
        Lane &ln = c->lane[i];
        if ((rc = lane_resolve(c, ln, false))) return rc;
        if (rec_base + ln.n_records > 0xFFFFFFFFull) return fail(SMX_ERR_CAPACITY, "%s: more than 2^32 records", fn);
        if ((rc = lane_compact(c, ln, (u32)rec_base, false))) return rc;
        rec_base += ln.n_records;
        matched += ln.n_matched;
    }
    *n_records = rec_base;
    *n_matched = matched;
    return SMX_OK;
}

// Lane 0 waits for everything enqueued so far on lanes 1..S-1.
static int resident_lanes_join(smx_ctx *c, int S) {
    for (int i = 1; i < S; ++i) {
        CU(c->ev_lane_done[i].ensure(cudaEventDisableTiming));
        CU(cudaEventRecord(c->ev_lane_done[i], c->lane[i].stream));
        CU(cudaStreamWaitEvent(c->lane[0].stream, c->ev_lane_done[i], 0));
    }
    return SMX_OK;
}

int smx_upload_batch(smx_ctx *c, const smx_batch *in) {
    int rc = check_batch(c, in, "smx_upload_batch");
    if (rc) return rc;
    CU(cudaSetDevice(c->device));
    resident_begin(c, in->n_reads);
    if (c->resident_lanes == 1) {
        Lane &ln = c->lane[0];
        rc = lane_upload(c, ln, in, 0, in->n_reads, nullptr);
        if (rc) return rc;
        CU(cudaStreamSynchronize(ln.stream));
        return SMX_OK;
    }
    const u32 *shared4 = nullptr;
    if (in->packed4 && in->off4 && in->packed4_words) {
        CU(c->shared_packed4.ensure(in->packed4_words));
        CU(cudaMemcpy(c->shared_packed4.p, in->packed4, in->packed4_words * sizeof(u32), cudaMemcpyHostToDevice));
        shared4 = c->shared_packed4.p;
    }
    for (int i = 0; i < c->resident_lanes; ++i) {
        u32 r0, r1;
        resident_bounds(c, i, r0, r1);
        if (r0 >= r1) { c->resident_lanes = i; break; }
        if ((rc = lane_upload(c, c->lane[i], in, r0, r1, shared4))) return rc;
    }
    for (int i = 0; i < c->resident_lanes; ++i) CU(cudaStreamSynchronize(c->lane[i].stream));
    return SMX_OK;
}

int smx_set_resident_split(smx_ctx *c, uint32_t n_sub_batches) {
    if (!c) return fail(SMX_ERR_ARG, "smx_set_resident_split: null context");
    if (n_sub_batches < 1 || n_sub_batches > (uint32_t)kMaxLanes)
        return fail(SMX_ERR_ARG, "smx_set_resident_split: 1..%d sub-batches", kMaxLanes);
    c->resident_split = (int)n_sub_batches;
    return SMX_OK;
}

int smx_run_resident(smx_ctx *c) {
    if (!c) return fail(SMX_ERR_ARG, "smx_run_resident: null context");
    if (!c->lane[0].have_batch) return fail(SMX_ERR_ARG, "smx_run_resident: no batch uploaded");
    CU(cudaSetDevice(c->device));
    int rc;
    if (c->resident_lanes == 1) {
        Lane &ln = c->lane[0];
        ln.launches = 0;
        if ((rc = lane_enqueue(c, ln, 0, true))) return rc;
        if ((rc = lane_resolve(c, ln, true))) return rc;
        if ((rc = lane_compact(c, ln, 0, true))) return rc;
        CU(cudaStreamSynchronize(ln.stream));
        CU(cudaGetLastError());
        for (int i = 0; i < 4; ++i) CU(cudaEventElapsedTime(&c->stage_ms[i], ln.ev[i], ln.ev[i + 1]));
        CU(cudaEventElapsedTime(&c->total_ms, ln.ev[0], ln.ev[4]));
        for (int i = 0; i < 8; ++i) CU(cudaEventElapsedTime(&c->kernel_ms[i], ln.kev[i], ln.kev[i + 1]));
        CU(cudaEventElapsedTime(&c->kernel_ms[8], ln.kev[9], ln.ev[4]));
        return SMX_OK;
    }
    // concurrent sub-batches: every lane starts after t0 (recorded on lane 0) and lane 0 joins them
    // all before t1, so t1 - t0 is the device time of the whole batch.  Per-kernel marks are not
    // taken here (kernels of different lanes overlap); a split of 1 measures them.
    const int S = c->resident_lanes;
    CU(c->ev_t0.ensure()); CU(c->ev_t1.ensure());
    CU(cudaEventRecord(c->ev_t0, c->lane[0].stream));
    for (int i = 1; i < S; ++i) CU(cudaStreamWaitEvent(c->lane[i].stream, c->ev_t0, 0));
    for (int i = 0; i < S; ++i) c->lane[i].launches = 0;
    u64 n_records, n_matched;
    if ((rc = resident_lanes_run(c, S, "smx_run_resident", &n_records, &n_matched))) return rc;
    if ((rc = resident_lanes_join(c, S))) return rc;
    CU(cudaEventRecord(c->ev_t1, c->lane[0].stream));
    CU(cudaStreamSynchronize(c->lane[0].stream));
    CU(cudaGetLastError());
    CU(cudaEventElapsedTime(&c->total_ms, c->ev_t0, c->ev_t1));
    for (auto &v : c->stage_ms) v = 0.f;
    for (auto &v : c->kernel_ms) v = 0.f;
    return SMX_OK;
}

int smx_download_results(smx_ctx *c, smx_results *out) {
    if (!c || !out) return fail(SMX_ERR_ARG, "smx_download_results: null argument");
    Lane &ln = c->lane[0];
    if (!ln.have_results) return fail(SMX_ERR_ARG, "smx_download_results: nothing to download");
    CU(cudaSetDevice(c->device));
    if (c->resident_lanes > 1) {
        if (out->primer_hits || out->endmask_bits || out->barcode_hits || out->orient_hits)
            return fail(SMX_ERR_ARG, "smx_download_results: per-search detail needs an unsplit batch (smx_set_resident_split(ctx, 1))");
        u64 total = 0, matched = 0;
        for (int i = 0; i < c->resident_lanes; ++i) { total += c->lane[i].n_records; matched += c->lane[i].n_matched; }
        out->n_records = total;
        out->n_matched = matched;
        if (total > out->records_cap)
            return fail(SMX_ERR_CAPACITY, "smx_download_results: %llu records, capacity %llu",
                        (unsigned long long)total, (unsigned long long)out->records_cap);
        u64 rec_base = 0;
        for (int i = 0; i < c->resident_lanes; ++i) {
            Lane &l = c->lane[i];
            u32 r0, r1;
            resident_bounds(c, i, r0, r1);
            if (out->rec_offset)
                CU(cudaMemcpyAsync(out->rec_offset + r0, l.offsets_src, (size_t)(r1 - r0) * sizeof(u32), cudaMemcpyDeviceToHost, l.stream));
            { int rc2 = lane_pack_records(l, out); if (!rc2) rc2 = lane_copy_records(l, out, rec_base, l.stream); if (rc2) return rc2; }
            rec_base += l.n_records;
        }
        for (int i = 0; i < c->resident_lanes; ++i) CU(cudaStreamSynchronize(c->lane[i].stream));
        if (out->rec_offset) out->rec_offset[c->resident_n] = (u32)total;
        if (out->records16 && !out->records && !out->records32) return check_record16_fit(c);
        return SMX_OK;
    }
    const Batch &b = ln.b;
    const Tables t = lane_tables(c, ln);
    const u32 n = b.n_reads;
    out->n_records = ln.n_records;
    out->n_matched = ln.n_matched;
    if (ln.n_records > out->records_cap)
        return fail(SMX_ERR_CAPACITY, "smx_download_results: %llu records, capacity %llu",
                    (unsigned long long)ln.n_records, (unsigned long long)out->records_cap);
    cudaStream_t st = ln.stream;
    if (out->rec_offset)
        CU(cudaMemcpyAsync(out->rec_offset, b.rec_offset, ((size_t)n + 1) * sizeof(u32), cudaMemcpyDeviceToHost, st));
    { int rc2 = lane_pack_records(ln, out); if (!rc2) rc2 = lane_copy_records(ln, out, 0, st); if (rc2) return rc2; }
    // level-1 detail is stored padded ([slot][n_pad]) on the device and returned dense ([slot][n])
    if (out->primer_hits)
        CU(cudaMemcpy2DAsync(out->primer_hits, (size_t)n * sizeof(smx_primer_hit), b.phit,
                             (size_t)b.n_pad * sizeof(smx_primer_hit), (size_t)n * sizeof(smx_primer_hit),
                             (size_t)2 * t.n_primers, cudaMemcpyDeviceToHost, st));
    if (out->orient_hits)
        CU(cudaMemcpy2DAsync(out->orient_hits, (size_t)n, b.orient_hit, (size_t)b.n_pad, (size_t)n,
                             (size_t)2 * t.n_primers, cudaMemcpyDeviceToHost, st));
    if (out->endmask_bits)
        CU(cudaMemcpy2DAsync(out->endmask_bits, (size_t)n * sizeof(u32), b.endmask, (size_t)b.n_pad * sizeof(u32),
                             (size_t)n * sizeof(u32), (size_t)2 * t.n_primers * t.mw, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (out->barcode_hits && t.total_bslots) {
        // expand the compact per-(entry, bword) hit lists into the dense [barcode slot][read] detail
        // layout, merging a barcode's hits over the primer end locations (strictly smaller wins)
        std::vector<smx_primer_hit> ph((size_t)2 * t.n_primers * b.n_pad);
        std::vector<u32> ebase((size_t)2 * t.n_primers * b.n_pad);
        std::vector<unsigned char> cnt((size_t)2 * t.n_bwords * b.e_cap);
        std::vector<smx_barcode_hit> lst((size_t)2 * t.n_bwords * t.hit_cap * b.e_cap);
        std::vector<unsigned char> bwp(t.n_bwords);
        CU(cudaMemcpy(ph.data(), b.phit, ph.size() * sizeof(smx_primer_hit), cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(ebase.data(), b.ent_base, ebase.size() * sizeof(u32), cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(cnt.data(), b.bh_count, cnt.size(), cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(lst.data(), b.bh_list, lst.size() * sizeof(smx_barcode_hit), cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(bwp.data(), t.bw_primer, bwp.size(), cudaMemcpyDeviceToHost));
        smx_barcode_hit none;
        none.end_mask = 0; none.search_start = 0; none.distance = -1; none.barcode = 0;
        for (size_t i = 0; i < (size_t)t.total_bslots * n; ++i) out->barcode_hits[i] = none;
        uint64_t n_loc_hits = 0;
        for (int sd = 0; sd < 2; ++sd)
            for (int g = 0; g < t.n_bwords; ++g) {
                int p = bwp[g];
                u32 slot = (u32)(sd * t.n_primers + p);
                u64 gslot = (u64)sd * t.n_bwords + g;
                for (u32 r = 0; r < n; ++r) {
                    const smx_primer_hit &h0 = ph[(size_t)slot * b.n_pad + r];
                    if (h0.distance < 0) continue;
                    for (u32 l = 0; l < h0.n_locations; ++l) {
                        u64 e = (u64)ebase[(size_t)slot * b.n_pad + r] + l;
                        int k = std::min<int>(cnt[gslot * b.e_cap + e], t.hit_cap);
                        for (int x = 0; x < k; ++x) {
                            const smx_barcode_hit &h = lst[(gslot * t.hit_cap + x) * b.e_cap + e];
                            smx_barcode_hit &dst = out->barcode_hits[((size_t)t.bslot_base[slot] + h.barcode) * n + r];
                            if (dst.distance < 0 || h.distance < dst.distance) dst = h;
                            if (out->barcode_loc_hits) {
                                if (n_loc_hits < out->barcode_loc_cap) {
                                    smx_barcode_loc_hit &lh = out->barcode_loc_hits[n_loc_hits];
                                    lh.read = r; lh.slot = (uint16_t)slot; lh.location = (uint16_t)l; lh.hit = h;
                                }
                                ++n_loc_hits;
                            }
                        }
                    }
                }
            }
        out->n_barcode_loc_hits = n_loc_hits;
    }
    if (out->records16 && !out->records && !out->records32) return check_record16_fit(c);
    return SMX_OK;
}

// Pipelined form of the whole path for large batches: the reads are cut into chunks that rotate
// over n_lanes lanes (stream + buffers each), so chunk i+1's H2D, chunk i's kernels and chunk i-1's
// D2H run concurrently (two copy engines + the SMs).  Results land in the caller's arrays exactly
// as the one-shot form writes them.
static int match_batch_pipelined(smx_ctx *c, const smx_batch *in, smx_results *out) {
    const u32 n = in->n_reads, chunk = c->chunk_reads;
    // Chunk boundaries (128-read aligned), an even split.  Optionally (SMX_PIPELINE_RAMP=1) the first
    // two chunks are a quarter and a half of the nominal size so that the copy-out engine starts
    // earlier.
    std::vector<u32> cuts{0};
    u32 k_total = (n + chunk - 1) / chunk;                     // chunks of the even split
    if (c->ramp == 1 && (u64)n > 2ull * chunk) {
        const u32 c0 = ((chunk / 4) + 127u) & ~127u, c1 = ((chunk / 2) + 127u) & ~127u;
        cuts.push_back(c0);
        cuts.push_back(c0 + c1);
        k_total = 0;
    } else if (c->ramp == 2 && k_total >= 4) {
        // same NUMBER of chunks as the even split, but the first two are a third and two thirds of the
        // average and the others make up for it
        const u32 avg = n / k_total;
        const u32 c0 = ((avg / 3) + 127u) & ~127u, c1 = ((2 * avg / 3) + 127u) & ~127u;
        cuts.push_back(c0);
        cuts.push_back(c0 + c1);
        k_total -= 2;
    }
    {
        const u32 rest = n - cuts.back();
        const u32 k = k_total ? k_total : (rest + chunk - 1) / chunk;
        const u32 per = (((rest + k - 1) / k) + 127u) & ~127u;
        while (cuts.back() < n) cuts.push_back((u32)std::min<u64>((u64)cuts.back() + per, n));
    }
    const u32 n_chunks = (u32)cuts.size() - 1;
    const u32 *shared4 = nullptr;
    if (in->packed4 && in->off4 && in->packed4_words) {
        CU(c->shared_packed4.ensure(in->packed4_words));
        CU(cudaMemcpy(c->shared_packed4.p, in->packed4, in->packed4_words * sizeof(u32), cudaMemcpyHostToDevice));
        shared4 = c->shared_packed4.p;
    }
    u64 rec_base = 0, matched = 0;
    bool overflow = false;
    int rc = SMX_OK;
    // SMX_PIPELINE_TRACE=1: per-chunk device timeline (events) + host enqueue times on stderr
    const bool trace = c->trace;
    std::vector<Event> tev(trace ? (size_t)n_chunks * 4 : 0);
    std::vector<double> thost(tev.size(), 0.0);
    auto now_ms = [] { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; };
    const double t_begin = now_ms();
    for (auto &e : tev) e.ensure();
    auto mark = [&](u32 i, int k, cudaStream_t st) { if (trace) { cudaEventRecord(tev[(size_t)i * 4 + k], st); thost[(size_t)i * 4 + k] = now_ms() - t_begin; } };
    auto bounds = [&](u32 i, u32 &r0, u32 &r1) { r0 = cuts[i]; r1 = cuts[i + 1]; };
    auto finish = [&](u32 i) -> int {
        Lane &ln = c->lane[i % c->n_lanes];
        u32 r0, r1;
        bounds(i, r0, r1);
        int r = lane_resolve(c, ln, false);
        if (r) return r;
        if (rec_base + ln.n_records > out->records_cap || rec_base + ln.n_records > 0xFFFFFFFFull) overflow = true;
        if (!overflow) {
            if ((r = lane_compact(c, ln, (u32)rec_base, false))) return r;
            if ((r = lane_pack_records(ln, out))) return r;
            // the copy-out runs on its own stream so the lane's next H2D + kernels need not wait for it
            CU(cudaEventRecord(ln.ev_ready, ln.stream));
            CU(cudaStreamWaitEvent(ln.out_stream, ln.ev_ready, 0));
            if (out->rec_offset)
                CU(cudaMemcpyAsync(out->rec_offset + r0, ln.offsets_src, (size_t)(r1 - r0) * sizeof(u32),
                                   cudaMemcpyDeviceToHost, ln.out_stream));
            if ((r = lane_copy_records(ln, out, rec_base, ln.out_stream))) return r;
            CU(cudaEventRecord(ln.ev_drained, ln.out_stream));
            ln.drain_pending = true;
            mark(i, 3, ln.out_stream);
        }
        rec_base += ln.n_records;
        matched += ln.n_matched;
        return SMX_OK;
    };
    u32 issued = 0, finished = 0;
    for (; issued < n_chunks && rc == SMX_OK; ++issued) {
        // a lane is reused only after its previous chunk has been finished (stream order covers the rest)
        while (rc == SMX_OK && issued - finished >= (u32)c->n_lanes) rc = finish(finished++);
        if (rc) break;
        Lane &ln = c->lane[issued % c->n_lanes];
        u32 r0, r1;
        bounds(issued, r0, r1);
        if (r0 >= r1) { ln.have_batch = false; continue; }
        mark(issued, 0, ln.stream);
        if ((rc = lane_upload(c, ln, in, r0, r1, shared4))) break;
        if (c->chain && issued > 0) {
            Lane &prev = c->lane[(issued - 1) % c->n_lanes];
            if (prev.ev_dp_done && prev.stream) CU(cudaStreamWaitEvent(ln.stream, prev.ev_dp_done, 0));
        }
        mark(issued, 1, ln.stream);
        if ((rc = lane_enqueue(c, ln, 0, false))) break;
        mark(issued, 2, ln.stream);
        // keep at most n_lanes - 1 chunks ahead so the finished chunk's D2H starts while the next computes
        while (rc == SMX_OK && issued + 1 - finished >= (u32)c->n_lanes) rc = finish(finished++);
    }
    while (rc == SMX_OK && finished < issued) rc = finish(finished++);
    for (auto &ln : c->lane) if (ln.stream) { cudaStreamSynchronize(ln.stream); cudaStreamSynchronize(ln.out_stream); ln.drain_pending = false; }
    if (trace) {
        fprintf(stderr, "[smx pipeline] %u chunks (first %u, last %u reads), host total %.3f ms\n", n_chunks, cuts[1] - cuts[0], cuts[n_chunks] - cuts[n_chunks - 1], now_ms() - t_begin);
        for (u32 i = 0; i < n_chunks && rc == SMX_OK && !overflow; ++i) {
            float t[4];
            for (int k = 0; k < 4; ++k) cudaEventElapsedTime(&t[k], tev[0], tev[(size_t)i * 4 + k]);
            fprintf(stderr, "[smx pipeline] chunk %u dev: h2d %.3f-%.3f kernels-end %.3f d2h-end %.3f | host enq: %.3f %.3f %.3f %.3f\n",
                    i, t[0], t[1], t[2], t[3], thost[i * 4], thost[i * 4 + 1], thost[i * 4 + 2], thost[i * 4 + 3]);
        }
    }
    c->lane[0].have_batch = false; c->lane[0].have_results = false;     // the resident API needs a fresh upload
    if (rc) return rc;
    CU(cudaGetLastError());
    out->n_records = rec_base;
    out->n_matched = matched;
    c->last_chunks = (int)n_chunks;
    if (overflow)
        return fail(SMX_ERR_CAPACITY, "smx_match_batch: %llu records, capacity %llu",
                    (unsigned long long)rec_base, (unsigned long long)out->records_cap);
    if (out->rec_offset) out->rec_offset[n] = (u32)rec_base;
    if (out->records16 && !out->records && !out->records32) return check_record16_fit(c);
    return SMX_OK;
}

int smx_match_batch(smx_ctx *c, const smx_batch *in, smx_results *out) {
    if (!out) return fail(SMX_ERR_ARG, "smx_match_batch: null argument");
    int rc = check_batch(c, in, "smx_match_batch");
    if (rc) return rc;
    const bool detail = out->primer_hits || out->endmask_bits || out->barcode_hits || out->orient_hits;
    out->n_barcode_loc_hits = 0;
    if (!detail && c->chunk_reads && in->n_reads > (u64)c->chunk_reads + c->chunk_reads / 2) {
        CU(cudaSetDevice(c->device));
        return match_batch_pipelined(c, in, out);
    }
    c->last_chunks = 1;
    const int split = c->resident_split;
    if (detail) c->resident_split = 1;          // the per-search detail arrays are laid out for one lane
    rc = smx_upload_batch(c, in);
    c->resident_split = split;
    if (rc) return rc;
    rc = smx_run_resident(c);
    if (rc) return rc;
    return smx_download_results(c, out);
}

// Without a GPU every device route fails with SMX_ERR_NO_DEVICE, before it looks at its arguments.
static int require_device(const char *fn) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(SMX_ERR_NO_DEVICE, "%s: no CUDA device; this library has no CPU path", fn);
    }
    return SMX_OK;
}

constexpr size_t kCallCtlWords = kMineCtlWords > 8 ? kMineCtlWords : 8;     // the most control words a route uses

// The frame of one device-route call (smx_match_device, smx_demux_device, smx_demux_files_device, smx_mine_device):
// open -> the route's pointer checks and scratch sizing -> begin (join the caller's stream, mark 0) -> the route's
// kernels and read-backs on lane 0's stream -> finish.  The routes share one set of control words, pinned mirror and
// events: each one synchronises lane 0's stream before it returns and touches the control words only on that stream,
// and writes the mirror only after a read-back, so even a call that failed midway is ordered before the next one's.
struct DeviceCall {
    smx_ctx *c;
    const char *fn;
    cudaStream_t s0 = nullptr;
    unsigned long long *ctl = nullptr, *h = nullptr;       // kCallCtlWords control words on the device / pinned mirror

    int open() {
        CU(cudaSetDevice(c->device));
        CU(c->call_ctl.ensure(kCallCtlWords));
        CU(c->call_host.ensure(kCallCtlWords));
        CU(c->call_ev_in.ensure(cudaEventDisableTiming));
        for (auto &e : c->call_ev_t) CU(e.ensure());
        s0 = c->lane[0].stream;
        ctl = c->call_ctl.p;
        h = c->call_host;
        return SMX_OK;
    }
    // The caller's pointer must be device (or managed) memory of the context's device.
    int device_ptr(const void *p, const char *what) const {
        cudaPointerAttributes a;
        const cudaError_t e = cudaPointerGetAttributes(&a, p);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            return fail(SMX_ERR_ARG, "%s: %s is not device memory (%s)", fn, what, cudaGetErrorString(e));
        }
        if ((a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != c->device)
            return fail(SMX_ERR_ARG, "%s: %s is not memory of device %d", fn, what, c->device);
        return SMX_OK;
    }
    // Lane 0 starts after everything already enqueued on the caller's stream; mark 0.
    int begin(void *stream) {
        CU(cudaEventRecord(c->call_ev_in, (cudaStream_t)stream));
        CU(cudaStreamWaitEvent(s0, c->call_ev_in, 0));
        return mark(0);
    }
    int mark(int i) {
        CU(cudaEventRecord(c->call_ev_t[i], s0));
        return SMX_OK;
    }
    // Control words [0, n) into the mirror h.
    int read_back(size_t n) {
        CU(cudaMemcpyAsync(h, ctl, n * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s0));
        CU(cudaStreamSynchronize(s0));
        return SMX_OK;
    }
    // Mark d ends the call; device_ms (optional) = {mark a -> b, mark e -> d}.
    int finish(float *device_ms, int a, int b, int e, int d) {
        CU(cudaEventRecord(c->call_ev_t[d], s0));
        CU(cudaStreamSynchronize(s0));
        CU(cudaGetLastError());
        if (device_ms) {
            CU(cudaEventElapsedTime(&device_ms[0], c->call_ev_t[a], c->call_ev_t[b]));
            CU(cudaEventElapsedTime(&device_ms[1], c->call_ev_t[e], c->call_ev_t[d]));
        }
        return SMX_OK;
    }
    // A refusal key of launch_pack_validate: item << 2 | 1 offsets descend, 2 ends past `bound`, 3 is 2^31 `unit` or longer.
    int offsets_refused(const char *item, unsigned long long key, const char *unit, const char *bound) const {
        static const char *why[4] = {"", "offsets descend", "ends past %s", "is 2^31 %s or longer"};
        char reason[64];
        snprintf(reason, sizeof(reason), why[key & 3], (key & 3) == 2 ? bound : unit);
        return fail(SMX_ERR_ARG, "%s: %s %llu %s", fn, item, key >> 2, reason);
    }
    // A refusal key of the record check (launch_demux_index): record << 3 | the field out of range.
    int record_refused(unsigned long long key, u32 n_reads) const {
        static const char *why[8] = {"", "names a read past the batch's reads", "specimen out of range", "b1 out of range",
                                     "b2 out of range", "pool out of range", "p1 out of range", "p2 out of range"};
        const smx_out::OutCounts &cnt = c->out_counts;
        return fail(SMX_ERR_ARG, "%s: record %llu %s (%u reads, %u specimens, %u b1, %u b2, %u pools, %u primers)", fn,
                    key >> 3, why[key & 7], n_reads, cnt.n_specimens, cnt.n_b1, cnt.n_b2, cnt.n_pools, cnt.n_primers);
    }
};

// Whole path for reads already in device memory: the device packer (smx_k_pack.cu) fills the lanes' batch buffers
// where lane_upload would copy them, then the lanes run exactly as smx_run_resident runs them.
int smx_match_device(smx_ctx *c, const char *bases, uint64_t n_bases, const uint64_t *seq_off, uint32_t n_reads,
                     void *stream, uint32_t *rec_offset, smx_record *records, uint64_t records_cap,
                     uint64_t *n_records, uint64_t *n_matched, float *device_ms) {
    DeviceCall call = {c, "smx_match_device"};
    if (device_ms) device_ms[0] = device_ms[1] = 0.f;
    int rc;
    if ((rc = require_device(call.fn))) return rc;
    if (!c || !seq_off || !rec_offset || !n_records || !n_matched || (n_bases && !bases) || (records_cap && !records))
        return fail(SMX_ERR_ARG, "smx_match_device: null argument");
    *n_records = 0; *n_matched = 0;
    if (!n_reads) return fail(SMX_ERR_ARG, "smx_match_device: empty batch");
    if ((rc = call.open())) return rc;
    if (n_bases && (rc = call.device_ptr(bases, "bases"))) return rc;
    if ((rc = call.device_ptr(seq_off, "seq_off"))) return rc;
    if ((rc = call.device_ptr(rec_offset, "rec_offset"))) return rc;
    if (records_cap && (rc = call.device_ptr(records, "records"))) return rc;

    const u32 n = n_reads, clip = (u32)c->t.L, stride = smx_pack_stride(clip);
    resident_begin(c, n);
    PackLanes d;
    memset(&d, 0, sizeof(d));
    d.stride = stride; d.clip = clip;
    for (int i = 0; i < c->resident_lanes; ++i) {
        u32 r0, r1;
        resident_bounds(c, i, r0, r1);
        if (r0 >= r1) { c->resident_lanes = i; break; }
        Lane &ln = c->lane[i];
        if ((rc = lane_size(c, ln, r1 - r0, (u64)(r1 - r0) * stride + 1, false, false))) return rc;
        CU(ln.off4.ensure(r1 - r0));
        d.r0[i] = r0; d.r0[i + 1] = r1;
        d.packed2[i] = ln.packed2.p; d.lengths[i] = ln.lengths.p; d.off4[i] = ln.off4.p;
    }
    const int S = c->resident_lanes;
    d.n_lanes = S;
    CU(c->pk_ev_packed.ensure(cudaEventDisableTiming));
    CU(c->pk_flag.ensure(n)); CU(c->pk_list.ensure(n));
    CU(c->pk_tiles.ensure(((size_t)n + kPackTile - 1) / kPackTile));

    // lanes 1.. start after pk_ev_packed, which lane 0 records after the join
    if ((rc = call.begin(stream))) return rc;
    Lane &l0 = c->lane[0];
    cudaStream_t s0 = call.s0;
    const unsigned char *src = (const unsigned char *)bases;
    // control words: [0] validation key, [1] flagged reads.  The offsets are read back before any kernel reads a base.
    CU(cudaMemsetAsync(call.ctl, 0xFF, sizeof(unsigned long long), s0));
    CU(cudaMemsetAsync(call.ctl + 1, 0, sizeof(unsigned long long), s0));
    CU(launch_pack_validate(seq_off, n, n_bases, call.ctl, s0));
    if ((rc = call.read_back(1))) return rc;
    if (call.h[0] != ~0ull) return call.offsets_refused("read", call.h[0], "bases", "n_bases");
    // fixed-stride pass, then (only when some read holds a non-ACGT byte) off4 and the side stream
    CU(cudaMemsetAsync(c->pk_flag.p, 0, (size_t)n * sizeof(u32), s0));
    CU(launch_pack_fixed(src, seq_off, n, d, c->pk_flag.p, c->pk_list.p, call.ctl + 1, s0));
    if ((rc = call.read_back(2))) return rc;
    int launches = 2;
    const u32 n_flagged = (u32)call.h[1];
    u32 *packed4 = nullptr;
    if (n_flagged) {
        const u64 words4 = (u64)n_flagged * 2 * pack_words4(2ull * clip);     // every flagged read takes at most this
        DevBuf<u32> &buf4 = S > 1 ? c->shared_packed4 : l0.packed4;
        CU(buf4.ensure(words4));
        packed4 = buf4.p;
        CU(launch_pack_off4(seq_off, n, c->pk_flag.p, c->pk_tiles.p, d, s0));
        CU(launch_pack_side(src, seq_off, c->pk_list.p, n_flagged, d, packed4, s0));
        launches += 4;
    }
    if ((rc = call.mark(1))) return rc;
    CU(cudaEventRecord(c->pk_ev_packed, s0));
    for (int i = 0; i < S; ++i) {
        Lane &ln = c->lane[i];
        lane_bind(ln, d.r0[i + 1] - d.r0[i], clip, stride, (u64)d.r0[i] * stride, d.r0[i], packed4, packed4 ? ln.off4.p : nullptr);
        if (i) CU(cudaStreamWaitEvent(ln.stream, c->pk_ev_packed, 0));
    }
    l0.launches += launches;

    // the unchanged kernel path, lane by lane as smx_run_resident runs it
    u64 rec_base, matched;
    if ((rc = resident_lanes_run(c, S, call.fn, &rec_base, &matched))) return rc;
    *n_records = rec_base;
    *n_matched = matched;
    if (rec_base <= records_cap) {
        u64 base = 0;
        for (int i = 0; i < S; ++i) {
            Lane &ln = c->lane[i];
            CU(cudaMemcpyAsync(rec_offset + d.r0[i], ln.offsets_src, (size_t)(d.r0[i + 1] - d.r0[i]) * sizeof(u32),
                               cudaMemcpyDeviceToDevice, ln.stream));
            if (ln.n_records)
                CU(cudaMemcpyAsync(records + base, ln.records.p, (size_t)ln.n_records * sizeof(smx_record), cudaMemcpyDeviceToDevice, ln.stream));
            base += ln.n_records;
        }
        call.h[0] = rec_base;                  // rec_offset[n]: the record total
        CU(cudaMemcpyAsync(rec_offset + n, call.h, sizeof(u32), cudaMemcpyHostToDevice, s0));
    }
    if ((rc = resident_lanes_join(c, S))) return rc;
    // a capacity refusal leaves device_ms at 0, as in the other routes
    if ((rc = call.finish(rec_base <= records_cap ? device_ms : nullptr, 0, 1, 0, 2))) return rc;
    for (auto &ln : c->lane) { ln.have_batch = false; ln.have_results = false; }     // the resident API needs a fresh upload
    if (rec_base > records_cap)
        return fail(SMX_ERR_CAPACITY, "smx_match_device: %llu records, capacity %llu", (unsigned long long)rec_base,
                    (unsigned long long)records_cap);
    return SMX_OK;
}

// Device demultiplexer: the index pass (smx_k_demux.cu) validates, sorts and scans without reading a base; one read-back
// of the control words decides refusal and capacity; then the copy kernels write every output byte.
int smx_demux_device(smx_ctx *c, const char *bases, const char *quals, uint64_t n_bases, const uint64_t *seq_off,
                     uint32_t n_reads, const smx_record *records, uint64_t n_records, void *stream, uint64_t *order,
                     uint64_t *out_off, char *out_seq, char *out_qual, uint64_t out_cap, uint64_t *group_key,
                     uint64_t *group_off, uint64_t *n_groups, uint64_t *n_out_bytes, float *device_ms) {
    DeviceCall call = {c, "smx_demux_device"};
    if (device_ms) device_ms[0] = device_ms[1] = 0.f;
    int rc;
    if ((rc = require_device(call.fn))) return rc;
    if (!c || !seq_off || !out_off || !group_off || !n_groups || !n_out_bytes || (n_bases && !bases) ||
        (n_records && (!records || !order || !group_key)) || (out_cap && (!out_seq || (quals && !out_qual))))
        return fail(SMX_ERR_ARG, "smx_demux_device: null argument");
    *n_groups = 0; *n_out_bytes = 0;
    const smx_out::OutCounts &cnt = c->out_counts;
    if (cnt.n_pools > smx_out::kOutMaxPools)
        return fail(SMX_ERR_ARG, "smx_demux_device: %u pools, the destination key holds %u", cnt.n_pools, smx_out::kOutMaxPools);
    if (std::max(cnt.n_specimens, std::max(cnt.n_b1, cnt.n_b2)) > smx_out::kOutMaxSamples)
        return fail(SMX_ERR_ARG, "smx_demux_device: more than 2^30 specimens or barcodes, the destination key holds 2^30");
    if (n_records > 0x7FFFFFFFull) return fail(SMX_ERR_ARG, "smx_demux_device: more than 2^31 - 1 records");
    if ((rc = call.open())) return rc;
    if (n_bases && (rc = call.device_ptr(bases, "bases"))) return rc;
    if (n_bases && quals && (rc = call.device_ptr(quals, "quals"))) return rc;
    if ((rc = call.device_ptr(seq_off, "seq_off"))) return rc;
    if (n_records && (rc = call.device_ptr(records, "records"))) return rc;
    if (n_records && (rc = call.device_ptr(order, "order"))) return rc;
    if ((rc = call.device_ptr(out_off, "out_off"))) return rc;
    if (out_cap && (rc = call.device_ptr(out_seq, "out_seq"))) return rc;
    if (out_cap && quals && (rc = call.device_ptr(out_qual, "out_qual"))) return rc;
    if (n_records && (rc = call.device_ptr(group_key, "group_key"))) return rc;
    if ((rc = call.device_ptr(group_off, "group_off"))) return rc;

    // control words: [0] offsets key, [1] records key, [2] groups, [3] output bytes
    const u64 n = n_records;
    DemuxIndex ix = {};
    if (n) {
        CU(c->dm_key_in.ensure(n)); CU(c->dm_key_out.ensure(n)); CU(c->dm_src.ensure(n)); CU(c->dm_out_src.ensure(n));
        CU(c->dm_rec_in.ensure(n)); CU(c->dm_rec_out.ensure(n)); CU(c->dm_len.ensure(n));
        size_t temp = 0;
        CU(demux_temp_bytes(n, &temp));
        CU(c->dm_temp.ensure(temp));
        ix.records = records; ix.n_records = n; ix.seq_off = seq_off; ix.n_reads = n_reads;
        ix.counts = cnt; ix.shape = smx_out::out_shape(cnt);
        ix.order = order; ix.out_off = out_off; ix.group_key = group_key; ix.group_off = group_off;
        ix.scratch = {c->dm_key_in.p, c->dm_key_out.p, c->dm_src.p, c->dm_out_src.p, c->dm_rec_in.p, c->dm_rec_out.p,
                      c->dm_len.p, c->dm_temp.p, c->dm_temp.cap, call.ctl};
    }

    if ((rc = call.begin(stream))) return rc;
    cudaStream_t s0 = call.s0;
    CU(cudaMemsetAsync(call.ctl, 0xFF, 2 * sizeof(unsigned long long), s0));
    CU(cudaMemsetAsync(call.ctl + 2, 0, 2 * sizeof(unsigned long long), s0));
    if (n_reads) CU(launch_pack_validate(seq_off, n_reads, n_bases, call.ctl, s0));
    if (n) {
        CU(launch_demux_index(ix, s0));
    } else {
        CU(cudaMemsetAsync(out_off, 0, sizeof(u64), s0));
        CU(cudaMemsetAsync(group_off, 0, sizeof(u64), s0));
    }
    // one read-back: refusals, group count, output bytes; no base has been read yet
    if ((rc = call.read_back(4))) return rc;
    const unsigned long long *h = call.h;
    if (h[0] != ~0ull) return call.offsets_refused("read", h[0], "bases", "n_bases");
    if (h[1] != ~0ull) return call.record_refused(h[1], n_reads);
    const u64 total = h[3];
    *n_groups = h[2];
    *n_out_bytes = total;
    if (total > out_cap)
        return fail(SMX_ERR_CAPACITY, "smx_demux_device: %llu output bytes, capacity %llu", (unsigned long long)total,
                    (unsigned long long)out_cap);
    unsigned char *dseq = (unsigned char *)out_seq, *dqual = quals ? (unsigned char *)out_qual : nullptr;
    if (total) CU(c->dm_tiles.ensure(demux_tile_marks(total, dseq, dqual)));
    if ((rc = call.mark(1))) return rc;
    CU(launch_demux_copy((const unsigned char *)bases, (const unsigned char *)quals, out_off, c->dm_out_src.p, n, total, dseq,
                         dqual, c->dm_tiles.p, s0));
    return call.finish(device_ms, 1, 2, 0, 2);
}

// Device file formatter: as smx_demux_device, with two slots per record (primary file, pool-level copy), outputs that
// are whole formatted records and one output buffer; titles and names are checked before the plan reads them.
int smx_demux_files_device(smx_ctx *c, const char *bases, const char *quals, uint64_t n_bases, const uint64_t *seq_off,
                           uint32_t n_reads, const char *titles, uint64_t n_title_bytes, const uint64_t *title_off,
                           const smx_record *records, uint64_t n_records, const char *names, uint64_t n_name_bytes,
                           const uint64_t *name_off, const uint32_t *name_counts, int is_fastq, void *stream,
                           uint64_t *out_record, uint64_t *out_off, char *out, uint64_t out_cap, uint64_t *file_key,
                           uint64_t *file_off, uint64_t *n_files, uint64_t *n_outputs, uint64_t *n_out_bytes,
                           float *device_ms) {
    DeviceCall call = {c, "smx_demux_files_device"};
    if (device_ms) device_ms[0] = device_ms[1] = 0.f;
    int rc;
    if ((rc = require_device(call.fn))) return rc;
    if (!c || !seq_off || !title_off || !name_off || !name_counts || !out_off || !file_off || !n_files || !n_outputs ||
        !n_out_bytes || (n_bases && !bases) || (n_title_bytes && !titles) || (n_name_bytes && !names) ||
        (n_records && (!records || !out_record || !file_key)) || (out_cap && !out))
        return fail(SMX_ERR_ARG, "smx_demux_files_device: null argument");
    *n_files = 0; *n_outputs = 0; *n_out_bytes = 0;
    const smx_out::OutCounts &cnt = c->out_counts;
    const uint32_t want[5] = {cnt.n_specimens, cnt.n_b1, cnt.n_b2, cnt.n_pools, cnt.n_primers};
    static const char *table[5] = {"specimens", "b1 barcodes", "b2 barcodes", "pools", "primers"};
    const int bad_table = smx_out::out_names_mismatch(cnt, name_counts);
    if (bad_table >= 0)
        return fail(SMX_ERR_ARG, "smx_demux_files_device: %u names of %s, the context has %u", name_counts[bad_table],
                    table[bad_table], want[bad_table]);
    if (cnt.n_pools > smx_out::kOutMaxPools)
        return fail(SMX_ERR_ARG, "smx_demux_files_device: %u pools, the destination key holds %u", cnt.n_pools, smx_out::kOutMaxPools);
    if (std::max(cnt.n_specimens, std::max(cnt.n_b1, cnt.n_b2)) > smx_out::kOutMaxSamples)
        return fail(SMX_ERR_ARG, "smx_demux_files_device: more than 2^30 specimens or barcodes, the destination key holds 2^30");
    if (n_records > 0x3FFFFFFFull) return fail(SMX_ERR_ARG, "smx_demux_files_device: more than 2^30 - 1 records");
    const u64 n_names = (u64)cnt.n_specimens + cnt.n_b1 + cnt.n_b2 + cnt.n_pools + cnt.n_primers;
    if ((rc = call.open())) return rc;
    if (n_bases && (rc = call.device_ptr(bases, "bases"))) return rc;
    if (n_bases && quals && (rc = call.device_ptr(quals, "quals"))) return rc;
    if ((rc = call.device_ptr(seq_off, "seq_off"))) return rc;
    if (n_title_bytes && (rc = call.device_ptr(titles, "titles"))) return rc;
    if ((rc = call.device_ptr(title_off, "title_off"))) return rc;
    if (n_name_bytes && (rc = call.device_ptr(names, "names"))) return rc;
    if ((rc = call.device_ptr(name_off, "name_off"))) return rc;
    if (n_records && (rc = call.device_ptr(records, "records"))) return rc;
    if (n_records && (rc = call.device_ptr(out_record, "out_record"))) return rc;
    if ((rc = call.device_ptr(out_off, "out_off"))) return rc;
    if (out_cap && (rc = call.device_ptr(out, "out"))) return rc;
    if (n_records && (rc = call.device_ptr(file_key, "file_key"))) return rc;
    if ((rc = call.device_ptr(file_off, "file_off"))) return rc;

    // control words: [0] read offsets, [1] records, [2] groups with the empty one, [3] bytes, [4] files, [5] outputs,
    // [6] title offsets, [7] name offsets
    const u64 n = n_records, slots = 2 * n;
    const bool fastq = is_fastq != 0;
    DemuxIndex ix = {};
    FilesIndex fx = {};
    if (n) {
        CU(c->dm_key_in.ensure(slots)); CU(c->dm_key_out.ensure(slots)); CU(c->dm_src.ensure(n)); CU(c->dm_out_src.ensure(slots));
        CU(c->dm_rec_in.ensure(slots)); CU(c->dm_rec_out.ensure(slots));
        CU(c->fl_len.ensure(slots)); CU(c->fl_hdr.ensure(n)); CU(c->fl_id.ensure(n)); CU(c->fl_group.ensure(slots + 1));
        size_t temp = 0;
        CU(demux_temp_bytes(slots, &temp));
        CU(c->dm_temp.ensure(temp));
        fx.plan = {(const unsigned char *)titles, title_off, n_title_bytes, {names, name_off, cnt}, fastq};
        fx.len = c->fl_len.p; fx.hdr = c->fl_hdr.p; fx.id_pos = c->fl_id.p; fx.group_idx = c->fl_group.p; fx.file_off = file_off;
        ix.records = records; ix.n_records = n; ix.seq_off = seq_off; ix.n_reads = n_reads;
        ix.counts = cnt; ix.shape = smx_out::out_shape(cnt);
        ix.order = out_record; ix.out_off = out_off; ix.group_key = file_key; ix.group_off = nullptr;
        ix.scratch = {c->dm_key_in.p, c->dm_key_out.p, c->dm_src.p, c->dm_out_src.p, c->dm_rec_in.p, c->dm_rec_out.p,
                      nullptr, c->dm_temp.p, c->dm_temp.cap, call.ctl};
        ix.files = &fx;
    }

    if ((rc = call.begin(stream))) return rc;
    cudaStream_t s0 = call.s0;
    CU(cudaMemsetAsync(call.ctl, 0xFF, 2 * sizeof(unsigned long long), s0));
    CU(cudaMemsetAsync(call.ctl + 2, 0, 4 * sizeof(unsigned long long), s0));
    CU(cudaMemsetAsync(call.ctl + 6, 0xFF, 2 * sizeof(unsigned long long), s0));
    if (n_reads) {
        CU(launch_pack_validate(seq_off, n_reads, n_bases, call.ctl, s0));
        CU(launch_pack_validate(title_off, n_reads, n_title_bytes, call.ctl + 6, s0));
    }
    if (n_names) CU(launch_pack_validate(name_off, (u32)n_names, n_name_bytes, call.ctl + 7, s0));
    if (n) {
        CU(launch_demux_index(ix, s0));
    } else {
        CU(cudaMemsetAsync(out_off, 0, sizeof(u64), s0));
        CU(cudaMemsetAsync(file_off, 0, sizeof(u64), s0));
    }
    // one read-back: refusals, file and output counts, bytes; no byte has been copied yet
    if ((rc = call.read_back(8))) return rc;
    const unsigned long long *h = call.h;
    if (h[0] != ~0ull) return call.offsets_refused("read", h[0], "bytes", "n_bases");
    if (h[6] != ~0ull) return call.offsets_refused("title", h[6], "bytes", "n_title_bytes");
    if (h[7] != ~0ull) return call.offsets_refused("name", h[7], "bytes", "n_name_bytes");
    if (h[1] != ~0ull) return call.record_refused(h[1], n_reads);
    const u64 total = n ? h[3] : 0, n_out = n ? h[5] : 0;
    *n_files = n ? h[4] : 0;
    *n_outputs = n_out;
    *n_out_bytes = total;
    if (total > out_cap)
        return fail(SMX_ERR_CAPACITY, "smx_demux_files_device: %llu output bytes, capacity %llu", (unsigned long long)total,
                    (unsigned long long)out_cap);
    unsigned char *dst = (unsigned char *)out;
    if (total) CU(c->dm_tiles.ensure(demux_tile_marks(total, dst, nullptr)));
    const smx_out::FilesCopy fc = {(const unsigned char *)bases, fastq ? (const unsigned char *)quals : nullptr, dst, fastq,
                                   out_off, c->dm_out_src.p, out_record, c->fl_hdr.p, c->fl_id.p, records,
                                   (const unsigned char *)titles, {names, name_off, cnt}, n_out, total};
    if ((rc = call.mark(1))) return rc;
    CU(launch_files_copy(fc, c->dm_tiles.p, s0));
    return call.finish(device_ms, 1, 2, 0, 2);
}

// specimine on device files: one read-back after the plan (refusals, patterns, entries, work items per class), one after
// the search and the decisions (records, bytes), then the records are written.
int smx_mine_device(smx_ctx *c, const char *data, uint64_t n_data, const uint64_t *out_off, uint64_t n_outputs,
                    const uint64_t *file_off, uint64_t n_files, uint32_t n_groups, const uint32_t *grp_file,
                    const uint8_t *grp_kind, const uint32_t *grp_part_off, const uint32_t *grp_part, uint32_t n_mined,
                    const uint32_t *mined_grp, double min_identity, void *stream, char *out, uint64_t out_cap,
                    uint64_t rec_cap, uint64_t *mined_off, int64_t *rec_partial, int64_t *rec_winner, int32_t *rec_dist,
                    uint64_t *n_records, uint64_t *n_out_bytes, float *device_ms) {
    DeviceCall call = {c, "smx_mine_device"};
    if (device_ms) device_ms[0] = device_ms[1] = 0.f;
    int rc;
    if ((rc = require_device(call.fn))) return rc;
    if (!c || !out_off || !file_off || !mined_grp || !mined_off || !n_records || !n_out_bytes || (n_data && !data) ||
        (n_groups && (!grp_file || !grp_kind || !grp_part_off)) || (out_cap && !out) ||
        (rec_cap && (!rec_partial || !rec_winner || !rec_dist)))
        return fail(SMX_ERR_ARG, "smx_mine_device: null argument");
    *n_records = 0; *n_out_bytes = 0;
    if (!(min_identity == min_identity)) return fail(SMX_ERR_ARG, "smx_mine_device: min_identity is not a number");
    if (n_files >= smx_mine::kMineMaxFiles) return fail(SMX_ERR_ARG, "smx_mine_device: %llu files (limit 2^29 - 1)", (unsigned long long)n_files);
    if (n_outputs >= 0xFFFFFFFFull) return fail(SMX_ERR_ARG, "smx_mine_device: %llu outputs (limit 2^32 - 2)", (unsigned long long)n_outputs);
    for (u64 f = 0; f < n_files; ++f)
        if (file_off[f + 1] < file_off[f] || file_off[f + 1] > n_data)
            return fail(SMX_ERR_ARG, "smx_mine_device: file %llu: offsets descend or end past n_data", (unsigned long long)f);
    if (mined_grp[0] != 0 || mined_grp[n_mined] != n_groups)
        return fail(SMX_ERR_ARG, "smx_mine_device: the .mined files' groups must start at 0 and end at n_groups");
    for (u32 j = 0; j < n_mined; ++j)
        if (mined_grp[j + 1] < mined_grp[j]) return fail(SMX_ERR_ARG, "smx_mine_device: .mined file %u: group offsets descend", j);
    if (n_groups && grp_part_off[0] != 0) return fail(SMX_ERR_ARG, "smx_mine_device: group 0's partial files must start at 0");
    std::vector<char> seen(n_files, 0);
    std::vector<u32> involved;
    auto take = [&](u32 f) { if (!seen[f]) { seen[f] = 1; involved.push_back(f); } };
    for (u32 g = 0; g < n_groups; ++g) {
        if (grp_file[g] >= n_files) return fail(SMX_ERR_ARG, "smx_mine_device: group %u names file %u of %llu", g, grp_file[g], (unsigned long long)n_files);
        if (grp_kind[g] > 1) return fail(SMX_ERR_ARG, "smx_mine_device: group %u has kind %u (0 forward, 1 reverse)", g, grp_kind[g]);
        if (grp_part_off[g + 1] < grp_part_off[g]) return fail(SMX_ERR_ARG, "smx_mine_device: group %u: partial file offsets descend", g);
        take(grp_file[g]);
        for (u32 k = grp_part_off[g]; k < grp_part_off[g + 1]; ++k) {
            if (!grp_part) return fail(SMX_ERR_ARG, "smx_mine_device: null argument");
            if (grp_part[k] >= n_files)
                return fail(SMX_ERR_ARG, "smx_mine_device: group %u names partial file %u of %llu", g, grp_part[k], (unsigned long long)n_files);
            take(grp_part[k]);
        }
    }
    if ((rc = call.open())) return rc;
    if (n_data && (rc = call.device_ptr(data, "data"))) return rc;
    if ((rc = call.device_ptr(out_off, "out_off"))) return rc;
    if (out_cap && (rc = call.device_ptr(out, "out"))) return rc;
    if ((rc = call.device_ptr(mined_off, "mined_off"))) return rc;
    if (rec_cap && (rc = call.device_ptr(rec_partial, "rec_partial"))) return rc;
    if (rec_cap && (rc = call.device_ptr(rec_winner, "rec_winner"))) return rc;
    if (rec_cap && (rc = call.device_ptr(rec_dist, "rec_dist"))) return rc;

    // the group table in one upload: grp_file, grp_kind, grp_part_off, grp_part, mined_grp, involved files
    const u32 G = n_groups, K = G ? grp_part_off[G] : 0, I = (u32)involved.size();
    std::vector<u32> tab;
    tab.reserve(3 * (size_t)G + 2 + K + n_mined + I);
    tab.insert(tab.end(), grp_file, grp_file + G);
    for (u32 g = 0; g < G; ++g) tab.push_back(grp_kind[g]);
    if (G) tab.insert(tab.end(), grp_part_off, grp_part_off + G + 1); else tab.push_back(0);
    if (K) tab.insert(tab.end(), grp_part, grp_part + K);
    tab.insert(tab.end(), mined_grp, mined_grp + n_mined + 1);
    tab.insert(tab.end(), involved.begin(), involved.end());
    CU(c->mn_file_off.ensure(n_files + 1)); CU(c->mn_tab.ensure(tab.size())); CU(c->mn_rng.ensure(2 * n_files + 2));
    CU(c->mn_beg.ensure(n_outputs + 1)); CU(c->mn_len.ensure(n_outputs + 1)); CU(c->mn_k.ensure(n_outputs + 1));
    CU(c->mn_pat_base.ensure(G + 1)); CU(c->mn_ent_base.ensure(G + 1)); CU(c->mn_bad.ensure(1));
    MineArgs a = {};
    a.data = (const unsigned char *)data; a.n_data = n_data; a.out_off = out_off; a.file_off = c->mn_file_off.p;
    a.n_outputs = n_outputs; a.n_files = n_files; a.n_groups = G; a.n_mined = n_mined; a.n_involved = I;
    const u32 *t = c->mn_tab.p;
    a.grp_file = t; a.grp_kind = t + G; a.grp_part_off = t + 2 * G; a.grp_part = t + 3 * G + 1;
    a.mined_grp = t + 3 * G + 1 + K; a.involved = t + 3 * G + 2 + K + n_mined;
    a.min_identity = min_identity;
    a.file_rng = c->mn_rng.p; a.seq_beg = c->mn_beg.p; a.seq_len = c->mn_len.p; a.k = c->mn_k.p;
    a.pat_base = c->mn_pat_base.p; a.ent_base = c->mn_ent_base.p; a.ctl = call.ctl;

    if ((rc = call.begin(stream))) return rc;
    cudaStream_t s0 = call.s0;
    CU(cudaMemcpyAsync(c->mn_file_off.p, file_off, (n_files + 1) * sizeof(u64), cudaMemcpyHostToDevice, s0));
    CU(cudaMemcpyAsync(c->mn_tab.p, tab.data(), tab.size() * sizeof(u32), cudaMemcpyHostToDevice, s0));
    CU(cudaMemsetAsync(call.ctl, 0xFF, sizeof(unsigned long long), s0));
    CU(cudaMemsetAsync(call.ctl + 1, 0, (kMineCtlWords - 1) * sizeof(unsigned long long), s0));
    CU(launch_mine_locate(a, s0));
    // read-back 1: refusals, patterns, entries, work items per class; no search has run
    if ((rc = call.read_back(3 + smx_mine::kHwClasses))) return rc;
    unsigned long long *h = call.h;
    if (h[0] != ~0ull) {
        static const char *why[7] = {"", "does not start and end on output boundaries", "output offsets descend or pass n_data",
                                     "is not a FASTQ record", "is a full read longer than 4096 bytes",
                                     "is a full read holding more than 64 distinct byte values",
                                     "is a full read beyond the 2^23 a file may hold for the search"};
        const unsigned long long f = h[0] >> 35, o = (h[0] >> 3) & 0xFFFFFFFFull;
        const int k = (int)(h[0] & 7);
        if (k == smx_mine::kMineFileRange) return fail(SMX_ERR_ARG, "smx_mine_device: file %llu %s", f, why[k]);
        return fail(SMX_ERR_ARG, "smx_mine_device: file %llu output %llu %s", f, o, why[k]);
    }
    const u64 P = h[1], E = h[2];
    u64 base[smx_mine::kHwClasses], n_items = 0;
    for (int k = 0; k < smx_mine::kHwClasses; ++k) { base[k] = n_items; n_items += h[3 + k]; }
    if (n_items > 0x7fffffffu) return fail(SMX_ERR_ARG, "smx_mine_device: %llu work items in one call (limit 2^31 - 1)", (unsigned long long)n_items);
    CU(c->mn_items.ensure(n_items + 1)); CU(c->mn_ent_txt.ensure(E + 1)); CU(c->mn_keys.ensure(E + 1));
    CU(c->mn_size.ensure(E + 1)); CU(c->mn_size_off.ensure(E + 1)); CU(c->mn_flag.ensure(E + 1)); CU(c->mn_flag_off.ensure(E + 1));
    CU(c->mn_win.ensure(E + 1)); CU(c->mn_dist.ensure(E + 1));
    size_t temp = 0;
    CU(mine_scan_temp_bytes(E + 1, &temp));
    CU(c->mn_temp.ensure(temp + 1));
    a.items = c->mn_items.p; a.ent_txt = c->mn_ent_txt.p; a.keys = c->mn_keys.p; a.size = c->mn_size.p;
    a.size_off = c->mn_size_off.p; a.flag = c->mn_flag.p; a.flag_off = c->mn_flag_off.p; a.winner = c->mn_win.p;
    a.dist = c->mn_dist.p; a.temp = c->mn_temp.p; a.temp_bytes = c->mn_temp.cap;
    for (int k = 0; k < smx_mine::kHwClasses; ++k) h[3 + smx_mine::kHwClasses + k] = base[k];
    CU(cudaMemcpyAsync(call.ctl + 3 + smx_mine::kHwClasses, h + 3 + smx_mine::kHwClasses,
                       smx_mine::kHwClasses * sizeof(unsigned long long), cudaMemcpyHostToDevice, s0));
    CU(launch_mine_items(a, P, E, s0));
    if (E) CU(cudaMemsetAsync(c->mn_keys.p, 0xFF, E * sizeof(unsigned long long), s0));
    CU(cudaMemsetAsync(c->mn_bad.p, 0, sizeof(u32), s0));
    if ((rc = call.mark(1))) return rc;
    const HwSpans spans = {a.data, a.seq_beg, a.seq_len};
    for (int k = 0; k < smx_mine::kHwClasses; ++k) {
        const int code = smx_mine::hw_class_code(k);
        CU(launch_hw_best(code >> 3, code & 7, spans, a.k, a.items + base[k], (u32)h[3 + k], spans, a.ent_txt, a.keys,
                          c->mn_bad.p, s0));
    }
    if ((rc = call.mark(2))) return rc;
    CU(launch_mine_decide(a, E, s0));
    // read-back 2: records, bytes, the search's refusal word
    if (E) {
        CU(cudaMemcpyAsync(h, c->mn_size_off.p + E, sizeof(u64), cudaMemcpyDeviceToHost, s0));
        CU(cudaMemcpyAsync(h + 1, c->mn_flag_off.p + E, sizeof(u64), cudaMemcpyDeviceToHost, s0));
    }
    CU(cudaMemcpyAsync(h + 2, c->mn_bad.p, sizeof(u32), cudaMemcpyDeviceToHost, s0));
    CU(cudaStreamSynchronize(s0));
    if ((u32)h[2]) return fail(SMX_ERR_ARG, "smx_mine_device: a full read holds more than 64 distinct byte values");
    const u64 total = E ? h[0] : 0, R = E ? h[1] : 0;
    *n_records = R;
    *n_out_bytes = total;
    if (total > out_cap || R > rec_cap)
        return fail(SMX_ERR_CAPACITY, "smx_mine_device: %llu records of %llu bytes, capacity %llu records, %llu bytes",
                    (unsigned long long)R, (unsigned long long)total, (unsigned long long)rec_cap, (unsigned long long)out_cap);
    if (E) {
        CU(c->mn_rec_off.ensure(R + 1)); CU(c->mn_kind.ensure(R + 1));
        a.rec_off = c->mn_rec_off.p; a.rec_kind = c->mn_kind.p;
        const MineOut mo = {(unsigned char *)out, mined_off, rec_partial, rec_winner, rec_dist};
        CU(launch_mine_format(a, E, R, mo, s0));
    } else {
        CU(cudaMemsetAsync(mined_off, 0, ((size_t)n_mined + 1) * sizeof(u64), s0));
    }
    return call.finish(device_ms, 1, 2, 0, 3);
}

int smx_set_pipeline_chunk(smx_ctx *c, uint32_t reads_per_chunk) {
    if (!c) return fail(SMX_ERR_ARG, "smx_set_pipeline_chunk: null context");
    if (reads_per_chunk && reads_per_chunk < 128) return fail(SMX_ERR_ARG, "smx_set_pipeline_chunk: chunk below 128 reads");
    c->chunk_reads = reads_per_chunk;
    return SMX_OK;
}

int smx_last_chunk_count(const smx_ctx *c) { return c ? c->last_chunks : 0; }

uint64_t smx_last_deferred(const smx_ctx *c) {
    if (!c) return 0;
    uint64_t v = 0;
    for (int i = 0; i < std::max(1, c->resident_lanes); ++i) v += c->lane[i].n_deferred;
    return v;
}

int smx_last_timing(const smx_ctx *c, float *total_ms, float stage_ms[4]) {
    if (!c) return fail(SMX_ERR_ARG, "smx_last_timing: null context");
    if (total_ms) *total_ms = c->total_ms;
    if (stage_ms) for (int i = 0; i < 4; ++i) stage_ms[i] = c->stage_ms[i];
    return SMX_OK;
}

int smx_last_kernel_times(const smx_ctx *c, float *ms, int n) {
    if (!c || !ms) return 0;
    for (int i = 0; i < n && i < kKernelTimes; ++i) ms[i] = c->kernel_ms[i];
    return kKernelTimes;
}

int smx_last_launch_count(const smx_ctx *c) {
    if (!c) return 0;
    int total = 0;
    for (const auto &ln : c->lane) total += ln.launches;
    return total;
}

int smx_last_work(const smx_ctx *c, uint64_t cells[2], uint64_t wordcols[2]) {
    if (!c || !c->lane[0].have_results) return fail(SMX_ERR_ARG, "smx_last_work: no results");
    cells[0] = cells[1] = wordcols[0] = wordcols[1] = 0;
    for (int i = 0; i < std::max(1, c->resident_lanes); ++i) {
        const Lane &ln = c->lane[i];
        cells[0] += ln.work[0]; cells[1] += ln.work[1];
        wordcols[0] += ln.work[2]; wordcols[1] += ln.work[3];
    }
    return SMX_OK;
}

int smx_last_useful_cells(const smx_ctx *c, uint64_t cells[2]) {
    if (!c || !c->lane[0].have_results) return fail(SMX_ERR_ARG, "smx_last_useful_cells: no results");
    cells[0] = cells[1] = 0;
    for (int i = 0; i < std::max(1, c->resident_lanes); ++i) { cells[0] += c->lane[i].useful[0]; cells[1] += c->lane[i].useful[1]; }
    return SMX_OK;
}

int smx_pairwise_nw(int device, const char *seqs, const uint32_t *seq_off, uint32_t n, int32_t *out) {
    if (!seqs || !seq_off || !out) return fail(SMX_ERR_ARG, "smx_pairwise_nw: null argument");
    if (n == 0) return SMX_OK;
    for (u32 i = 0; i < n; ++i)
        if (seq_off[i + 1] - seq_off[i] > 64) return fail(SMX_ERR_ARG, "smx_pairwise_nw: sequence %u longer than 64", i);
    int rc;
    if ((rc = require_device("smx_pairwise_nw"))) return rc;
    CU(cudaSetDevice(device));
    DevBuf<char> d_seq;
    DevBuf<u32> d_off;
    DevBuf<i32> d_out;
    const size_t bytes = seq_off[n];
    const u64 total = (u64)n * n;
    CU(d_seq.ensure(bytes ? bytes : 1));
    CU(d_off.ensure((size_t)(n + 1)));
    CU(d_out.ensure(total));
    CU(cudaMemcpy(d_seq.p, seqs, bytes, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_off.p, seq_off, (size_t)(n + 1) * sizeof(u32), cudaMemcpyHostToDevice));
    CU(launch_pairwise_nw(d_seq.p, d_off.p, n, d_out.p, 0));
    CU(cudaMemcpy(out, d_out.p, total * sizeof(i32), cudaMemcpyDeviceToHost));
    return SMX_OK;
}

int smx_hw_distances(int device, const char *patterns, const uint64_t *pat_off, const int32_t *pat_k, uint32_t n_patterns,
                     const char *texts, const uint64_t *txt_off, uint32_t n_texts, int32_t *out) {
    if (!patterns || !pat_off || !pat_k || !texts || !txt_off || !out) return fail(SMX_ERR_ARG, "smx_hw_distances: null argument");
    if (!n_patterns || !n_texts) return SMX_OK;
    int rc;
    if ((rc = require_device("smx_hw_distances"))) return rc;
    // classes by pattern length: lanes per problem and words per lane of the multi-word column vector
    struct Cls { int sw, w; std::vector<u32> list; };
    std::vector<Cls> classes;
    std::vector<u32> empty_pat;
    for (u32 i = 0; i < n_patterns; ++i) {
        const u64 m = pat_off[i + 1] - pat_off[i];
        if (m == 0) { empty_pat.push_back(i); continue; }
        if (m > 4096) return fail(SMX_ERR_ARG, "smx_hw_distances: pattern %u is %llu long (limit 4096)", i, (unsigned long long)m);
        const int words = (int)((m + 31) / 32);
        int sw = 4, w = 1;
        if (words <= 32) { while (sw < words) sw *= 2; }
        else { sw = 32; w = words <= 64 ? 2 : 4; }
        size_t c = 0;
        for (; c < classes.size(); ++c) if (classes[c].sw == sw && classes[c].w == w) break;
        if (c == classes.size()) { Cls n; n.sw = sw; n.w = w; classes.push_back(n); }
        classes[c].list.push_back(i);
    }
    CU(cudaSetDevice(device));
    DevBuf<unsigned char> d_pat, d_txt;
    DevBuf<u64> d_po, d_to;
    DevBuf<i32> d_k, d_out;
    DevBuf<u32> d_list, d_bad;
    const size_t pb = pat_off[n_patterns], tb = txt_off[n_texts];
    const size_t total = (size_t)n_patterns * n_texts;
    CU(d_pat.ensure(pb ? pb : 1)); CU(d_txt.ensure(tb ? tb : 1));
    CU(d_po.ensure((size_t)(n_patterns + 1))); CU(d_to.ensure((size_t)(n_texts + 1)));
    CU(d_k.ensure(n_patterns)); CU(d_out.ensure(total));
    CU(d_list.ensure(n_patterns)); CU(d_bad.ensure(1));
    CU(cudaMemcpy(d_pat.p, patterns, pb, cudaMemcpyHostToDevice)); CU(cudaMemcpy(d_txt.p, texts, tb, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_po.p, pat_off, (size_t)(n_patterns + 1) * sizeof(u64), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_to.p, txt_off, (size_t)(n_texts + 1) * sizeof(u64), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_k.p, pat_k, (size_t)n_patterns * sizeof(i32), cudaMemcpyHostToDevice));
    CU(cudaMemset(d_bad.p, 0, sizeof(u32)));
    size_t off = 0;
    for (const Cls &c : classes) {
        CU(cudaMemcpy(d_list.p + off, c.list.data(), c.list.size() * sizeof(u32), cudaMemcpyHostToDevice));
        CU(launch_hw_distance(c.sw, c.w, d_pat.p, d_po.p, d_k.p, d_list.p + off, (u32)c.list.size(), d_txt.p, d_to.p, n_texts, d_out.p,
                              d_bad.p, 0));
        off += c.list.size();
    }
    CU(cudaDeviceSynchronize());
    u32 bad = 0;
    CU(cudaMemcpy(&bad, d_bad.p, sizeof(u32), cudaMemcpyDeviceToHost));
    if (bad) return fail(SMX_ERR_ARG, "smx_hw_distances: %u pattern(s) hold more than 64 distinct byte values", bad);
    CU(cudaMemcpy(out, d_out.p, total * sizeof(i32), cudaMemcpyDeviceToHost));
    // an empty pattern has distance 0 everywhere; an empty text leaves the whole pattern unmatched (edlib: editDistance =
    // pattern length whatever k is -- SURVEY.md Q4)
    for (u32 i : empty_pat) for (u32 j = 0; j < n_texts; ++j) out[(size_t)i * n_texts + j] = 0;
    for (u32 j = 0; j < n_texts; ++j)
        if (txt_off[j + 1] == txt_off[j])
            for (u32 i = 0; i < n_patterns; ++i) out[(size_t)i * n_texts + j] = (int32_t)(pat_off[i + 1] - pat_off[i]);
    return SMX_OK;
}

int smx_hw_best_grouped(int device, const char *patterns, const uint64_t *pat_off, const int32_t *pat_k, uint32_t n_patterns,
                        const char *texts, const uint64_t *txt_off, uint32_t n_texts, uint32_t n_groups,
                        const uint32_t *grp_pat_off, const uint64_t *grp_txt_off, const uint32_t *grp_txt_idx,
                        int32_t *best_pat, int32_t *best_dist, float *device_ms) {
    constexpr u32 kMaxGroup = 1u << 23;                         // pattern rank field of the key
    if (device_ms) *device_ms = 0.f;
    if (!pat_off || !pat_k || !txt_off || !grp_pat_off || !grp_txt_off) return fail(SMX_ERR_ARG, "smx_hw_best_grouped: null argument");
    if (grp_pat_off[0] != 0 || grp_txt_off[0] != 0 || grp_pat_off[n_groups] > n_patterns)
        return fail(SMX_ERR_ARG, "smx_hw_best_grouped: group offsets must start at 0 and stay within the patterns");
    const u64 n_ent = grp_txt_off[n_groups];
    if (n_ent && (!grp_txt_idx || !best_pat || !best_dist)) return fail(SMX_ERR_ARG, "smx_hw_best_grouped: null argument");
    if ((pat_off[n_patterns] && !patterns) || (txt_off[n_texts] && !texts)) return fail(SMX_ERR_ARG, "smx_hw_best_grouped: null argument");
    for (u32 g = 0; g < n_groups; ++g) {
        if (grp_pat_off[g + 1] < grp_pat_off[g] || grp_txt_off[g + 1] < grp_txt_off[g])
            return fail(SMX_ERR_ARG, "smx_hw_best_grouped: group %u has decreasing offsets", g);
        if (grp_pat_off[g + 1] - grp_pat_off[g] > kMaxGroup)
            return fail(SMX_ERR_ARG, "smx_hw_best_grouped: group %u has %u patterns (limit %u)", g, grp_pat_off[g + 1] - grp_pat_off[g], kMaxGroup);
    }
    for (u32 i = 0; i < n_patterns; ++i)
        if (pat_off[i + 1] - pat_off[i] > 4096)
            return fail(SMX_ERR_ARG, "smx_hw_best_grouped: pattern %u is %llu long (limit 4096)", i, (unsigned long long)(pat_off[i + 1] - pat_off[i]));
    for (u64 e = 0; e < n_ent; ++e) {
        if (grp_txt_idx[e] >= n_texts) return fail(SMX_ERR_ARG, "smx_hw_best_grouped: entry %llu names text %u of %u", (unsigned long long)e, grp_txt_idx[e], n_texts);
        best_pat[e] = -1; best_dist[e] = -1;
    }
    // work items by (lanes, words per lane) class: every non-empty pattern of a group x runs of its group's entries
    // (empty patterns never win: their identity 1 - 0/0 is no number)
    struct Cls { int sw, w; std::vector<HwItem> items; };
    std::vector<Cls> classes;
    for (u32 g = 0; g < n_groups; ++g) {
        const u64 e0 = grp_txt_off[g], ne = grp_txt_off[g + 1] - e0;
        if (!ne) continue;
        for (u32 i = grp_pat_off[g]; i < grp_pat_off[g + 1]; ++i) {
            const u64 m = pat_off[i + 1] - pat_off[i];
            if (!m) continue;
            int sw, w;
            hw_best_class((int)((m + 31) / 32), &sw, &w);
            size_t c = 0;
            for (; c < classes.size(); ++c) if (classes[c].sw == sw && classes[c].w == w) break;
            if (c == classes.size()) { Cls n; n.sw = sw; n.w = w; classes.push_back(n); }
            const u32 chunk = hw_best_chunk(sw);
            for (u64 lo = 0; lo < ne; lo += chunk)
                classes[c].items.push_back(HwItem{i, i - grp_pat_off[g], e0 + lo, (u32)std::min<u64>(chunk, ne - lo), 0u});
        }
    }
    size_t n_items = 0;
    for (const Cls &c : classes) n_items += c.items.size();
    if (!n_items) return SMX_OK;
    if (n_items > 0x7fffffffu) return fail(SMX_ERR_ARG, "smx_hw_best_grouped: %zu work items in one call (limit 2^31 - 1)", n_items);
    int rc;
    if ((rc = require_device("smx_hw_best_grouped"))) return rc;
    CU(cudaSetDevice(device));
    DevBuf<unsigned char> d_pat, d_txt;
    DevBuf<u64> d_po, d_to;
    DevBuf<i32> d_k;
    DevBuf<u32> d_ent, d_bad;
    DevBuf<unsigned long long> d_keys;
    DevBuf<HwItem> d_items;
    Event ev[2];
    std::vector<unsigned long long> keys(n_ent);
    const size_t pb = pat_off[n_patterns], tb = txt_off[n_texts];
    CU(d_pat.ensure(pb ? pb : 1)); CU(d_txt.ensure(tb ? tb : 1));
    CU(d_po.ensure((size_t)(n_patterns + 1))); CU(d_to.ensure((size_t)(n_texts + 1)));
    CU(d_k.ensure(std::max(1u, n_patterns)));
    CU(d_ent.ensure(n_ent)); CU(d_keys.ensure(n_ent));
    CU(d_items.ensure(n_items)); CU(d_bad.ensure(1));
    CU(cudaMemcpy(d_pat.p, patterns, pb, cudaMemcpyHostToDevice)); CU(cudaMemcpy(d_txt.p, texts, tb, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_po.p, pat_off, (size_t)(n_patterns + 1) * sizeof(u64), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_to.p, txt_off, (size_t)(n_texts + 1) * sizeof(u64), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_k.p, pat_k, (size_t)n_patterns * sizeof(i32), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_ent.p, grp_txt_idx, n_ent * sizeof(u32), cudaMemcpyHostToDevice));
    CU(cudaMemset(d_keys.p, 0xFF, n_ent * sizeof(unsigned long long)));         // ~0: no candidate
    CU(cudaMemset(d_bad.p, 0, sizeof(u32)));
    size_t off = 0;
    for (const Cls &c : classes) {
        CU(cudaMemcpy(d_items.p + off, c.items.data(), c.items.size() * sizeof(HwItem), cudaMemcpyHostToDevice));
        off += c.items.size();
    }
    CU(ev[0].ensure()); CU(ev[1].ensure());
    CU(cudaEventRecord(ev[0], 0));
    off = 0;
    for (const Cls &c : classes) {
        CU(launch_hw_best(c.sw, c.w, HwContig{d_pat.p, d_po.p}, d_k.p, d_items.p + off, (u32)c.items.size(), HwContig{d_txt.p, d_to.p},
                          d_ent.p, d_keys.p, d_bad.p, 0));
        off += c.items.size();
    }
    CU(cudaEventRecord(ev[1], 0));
    CU(cudaEventSynchronize(ev[1]));
    if (device_ms) CU(cudaEventElapsedTime(device_ms, ev[0], ev[1]));
    u32 bad = 0;
    CU(cudaMemcpy(&bad, d_bad.p, sizeof(u32), cudaMemcpyDeviceToHost));
    if (bad) return fail(SMX_ERR_ARG, "smx_hw_best_grouped: a pattern holds more than 64 distinct byte values");
    CU(cudaMemcpy(keys.data(), d_keys.p, n_ent * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    // key = (floor(d * 2^40 / m) << 23) | rank; d = ceil(q * m / 2^40) since q * m lies in (d * 2^40 - m, d * 2^40]
    for (u32 g = 0; g < n_groups; ++g)
        for (u64 e = grp_txt_off[g]; e < grp_txt_off[g + 1]; ++e) {
            const unsigned long long key = keys[e];
            if (key == ~0ull) continue;
            const u32 rank = (u32)(key & (kMaxGroup - 1));
            const u64 m = pat_off[grp_pat_off[g] + rank + 1] - pat_off[grp_pat_off[g] + rank];
            best_pat[e] = (int32_t)rank;
            best_dist[e] = (int32_t)(((key >> 23) * m + (1ull << 40) - 1) >> 40);
        }
    return SMX_OK;
}

int smx_int_alu_peak(int device, double out_tops[3]) {
    if (!out_tops) return fail(SMX_ERR_ARG, "smx_int_alu_peak: null argument");
    int rc;
    if ((rc = require_device("smx_int_alu_peak"))) return rc;
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    DevBuf<u32> d_out;
    CU(d_out.ensure(1));
    Event e0, e1;
    CU(e0.ensure()); CU(e1.ensure());
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    const double ops = (double)blocks * threads * iters * 64.0;
    for (int mode = 0; mode < 3; ++mode) {
        float best = 1e30f;
        for (int rep = 0; rep < 5; ++rep) {
            CU(cudaEventRecord(e0));
            CU(launch_int_peak(mode, blocks, threads, d_out.p, iters, 17u + rep, 0));
            CU(cudaEventRecord(e1));
            CU(cudaEventSynchronize(e1));
            float ms = 0;
            CU(cudaEventElapsedTime(&ms, e0, e1));
            if (rep > 0 && ms < best) best = ms;
        }
        out_tops[mode] = ops / (best * 1e-3) / 1e12;
    }
    return SMX_OK;
}

int smx_flush_l2(smx_ctx *c) {
    if (!c) return fail(SMX_ERR_ARG, "smx_flush_l2: null context");
    CU(cudaSetDevice(c->device));
    const size_t bytes = 512ull << 20;
    CU(c->l2_scratch.ensure(bytes));
    CU(cudaMemsetAsync(c->l2_scratch.p, 0x5a, bytes, c->lane[0].stream));
    CU(cudaStreamSynchronize(c->lane[0].stream));
    return SMX_OK;
}

void *smx_host_alloc(uint64_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        fail(SMX_ERR_CUDA, "smx_host_alloc: cudaHostAlloc(%llu) failed", (unsigned long long)bytes);
        return nullptr;
    }
    return p;
}

void smx_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

// ------------------------------------------------------------------------------------------------
// Host-side packer (batching layer; no matching happens here).

void smx_pack_bound(const uint64_t *seq_off, uint32_t n_reads, uint32_t clip_len,
                    uint64_t *packed2_words, uint64_t *packed4_words_max) {
    uint64_t w2 = 0, w4 = 0;
    for (uint32_t r = 0; r < n_reads; ++r) {
        uint64_t len = seq_off[r + 1] - seq_off[r];
        if (clip_len && len > 2ull * clip_len) len = 2ull * clip_len;
        w2 += (len + 15) / 16;
        w4 += 2 * ((len + 7) / 8);
    }
    if (packed2_words) *packed2_words = w2 + 1;
    if (packed4_words_max) *packed4_words_max = w4 + 1;
}

int smx_pack_reads(const char *bases, const uint64_t *seq_off, uint32_t n_reads, uint32_t clip_len,
                   uint32_t *packed2, uint64_t *word_off, uint32_t *lengths,
                   uint32_t *packed4, uint64_t *off4, uint64_t *packed4_words, uint32_t *n_flagged) {
    if (!bases || !seq_off || !packed2 || !word_off || !lengths)
        return fail(SMX_ERR_ARG, "smx_pack_reads: null argument");
    uint64_t w2 = 0, w4 = 0;
    uint32_t flagged = 0;
    for (uint32_t r = 0; r < n_reads; ++r) {
        const unsigned char *s = (const unsigned char *)bases + seq_off[r];
        const uint64_t len = seq_off[r + 1] - seq_off[r];
        if (len > 0x7FFFFFFFull) return fail(SMX_ERR_ARG, "smx_pack_reads: read %u too long", r);
        const uint64_t slen = pack_stored_len(len, clip_len);      // stored bases
        word_off[r] = w2;
        lengths[r] = (uint32_t)len;
        bool exotic = false;
        const uint64_t nw = (slen + 15) / 16;
        for (uint64_t w = 0; w < nw; ++w) packed2[w2 + w] = pack_word2(s, len, clip_len, w, exotic);
        w2 += nw;
        if (off4) off4[r] = ~0ull;
        if (exotic) {
            if (!packed4 || !off4) return fail(SMX_ERR_ARG, "smx_pack_reads: read %u needs the packed4 stream", r);
            off4[r] = w4;
            const uint64_t n4 = pack_words4(slen);
            for (uint64_t w = 0; w < n4; ++w) {
                packed4[w4 + w] = pack_word4(s, len, clip_len, 0, w);
                packed4[w4 + n4 + w] = pack_word4(s, len, clip_len, 1, w);
            }
            w4 += 2 * n4;
            ++flagged;
        }
    }
    if (packed4_words) *packed4_words = w4;
    if (n_flagged) *n_flagged = flagged;
    return SMX_OK;
}

uint32_t smx_pack_stride(uint32_t clip_len) { return (2 * clip_len + 15) / 16; }

int smx_pack_reads_fixed(const char *bases, const uint64_t *seq_off, uint32_t n_reads, uint32_t clip_len,
                         uint32_t *packed2, uint32_t *lengths, uint16_t *lengths16, int *lengths_fit16,
                         uint32_t *packed4, uint64_t *off4, uint64_t *packed4_words, uint32_t *n_flagged) {
    if (!bases || !seq_off || !packed2 || (!lengths && !lengths16)) return fail(SMX_ERR_ARG, "smx_pack_reads_fixed: null argument");
    if (!clip_len) return fail(SMX_ERR_ARG, "smx_pack_reads_fixed: needs clip_len > 0 (unclipped reads have no common stride)");
    const uint32_t stride = smx_pack_stride(clip_len);
    uint64_t w4 = 0;
    uint32_t flagged = 0;
    bool fit16 = true;
    for (uint32_t r = 0; r < n_reads; ++r) {
        const unsigned char *s = (const unsigned char *)bases + seq_off[r];
        const uint64_t len = seq_off[r + 1] - seq_off[r];
        if (len > 0x7FFFFFFFull) return fail(SMX_ERR_ARG, "smx_pack_reads_fixed: read %u too long", r);
        const uint64_t slen = pack_stored_len(len, clip_len);
        if (lengths) lengths[r] = (uint32_t)len;
        if (len > 0xFFFFull) fit16 = false;
        else if (lengths16) lengths16[r] = (uint16_t)len;
        bool exotic = false;
        uint32_t *dst = packed2 + (uint64_t)r * stride;
        for (uint64_t w = 0; w < stride; ++w) dst[w] = pack_word2(s, len, clip_len, w, exotic);
        if (off4) off4[r] = ~0ull;
        if (exotic) {
            if (!packed4 || !off4) return fail(SMX_ERR_ARG, "smx_pack_reads_fixed: read %u needs the packed4 stream", r);
            off4[r] = w4;
            const uint64_t n4 = pack_words4(slen);
            for (uint64_t w = 0; w < n4; ++w) {
                packed4[w4 + w] = pack_word4(s, len, clip_len, 0, w);
                packed4[w4 + n4 + w] = pack_word4(s, len, clip_len, 1, w);
            }
            w4 += 2 * n4;
            ++flagged;
        }
    }
    packed2[(uint64_t)n_reads * stride] = 0;             // the slack word window extraction may read
    if (packed4_words) *packed4_words = w4;
    if (n_flagged) *n_flagged = flagged;
    if (lengths_fit16) *lengths_fit16 = fit16 ? 1 : 0;
    return SMX_OK;
}

int smx_copy_peak(int device, uint64_t bytes, double out_gbs[3]) {
    if (!out_gbs || !bytes) return fail(SMX_ERR_ARG, "smx_copy_peak: null argument");
    int rc;
    if ((rc = require_device("smx_copy_peak"))) return rc;
    CU(cudaSetDevice(device));
    Pinned<unsigned char> h_in, h_out;
    DevBuf<unsigned char> d_in, d_out;
    Stream s0, s1;
    Event e0, e1, e2;
    CU(h_in.ensure(bytes)); CU(h_out.ensure(bytes));
    memset(h_in, 0x5a, bytes); memset(h_out, 0, bytes);
    CU(d_in.ensure(bytes)); CU(d_out.ensure(bytes));
    CU(s0.ensure()); CU(s1.ensure());
    CU(e0.ensure()); CU(e1.ensure()); CU(e2.ensure());
    for (int mode = 0; mode < 3; ++mode) {
        float best = 1e30f;
        for (int rep = 0; rep < 6; ++rep) {
            CU(cudaEventRecord(e0, s0));
            CU(cudaStreamWaitEvent(s1, e0, 0));
            if (mode != 1) CU(cudaMemcpyAsync(d_in.p, h_in, bytes, cudaMemcpyHostToDevice, s0));
            if (mode != 0) CU(cudaMemcpyAsync(h_out, d_out.p, bytes, cudaMemcpyDeviceToHost, s1));
            CU(cudaEventRecord(e2, s1));
            CU(cudaStreamWaitEvent(s0, e2, 0));
            CU(cudaEventRecord(e1, s0));
            CU(cudaEventSynchronize(e1));
            float ms = 0;
            CU(cudaEventElapsedTime(&ms, e0, e1));
            if (rep > 0 && ms < best) best = ms;
        }
        out_gbs[mode] = (mode == 2 ? 2.0 : 1.0) * (double)bytes / (best * 1e-3) / 1e9;
    }
    return SMX_OK;
}

}  // extern "C"
