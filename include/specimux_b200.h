/*
 * specimux_b200.h -- C ABI of the B200 read-matching library (libspecimux_b200.so).
 *
 * Drop-in boundary for specimux's per-read matching path.  The reference has no FFI: its seam is
 * the Python callable
 *     process_sequences(seq_records, parameters, specimens, args, prefilter, trace_logger, record_offset)
 *         (reference: src/specimux/demultiplex.py:108-212)
 * whose arithmetic is edlib.align behind align_seq (src/specimux/alignment.py:21-50).  This header is
 * what a ctypes/cffi stub inside that function binds (see INTEGRATION.md); every entry point cites the
 * reference code it replaces.  Plain pointers and sizes only; no C++/torch types; errors are non-zero
 * int codes plus a thread-local message (smx_last_error) -- nothing throws across the boundary.
 *
 * Threading: one context per GPU; a context is not re-entrant.  Do not fork after smx_create.
 */
#ifndef SPECIMUX_B200_H
#define SPECIMUX_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMX_ABI_VERSION 3

#define SMX_MAX_PRIMERS 254     /* canonical primers (distinct sequences); 0xFF = "unknown" in smx_record16 */
#define SMX_MAX_PAIRS 4096      /* primer pairs (candidate enumeration order)                     */
#define SMX_MAX_PATTERN 64      /* primer / barcode length handled by the single-thread kernels   */
#define SMX_MAX_LONG_PATTERN 1024 /* primer length handled by the warp-cooperative multi-word kernel */
#define SMX_MAX_SEARCH_LEN 1024 /* --search-len                                                   */

/* error codes */
#define SMX_OK 0
#define SMX_ERR_ARG 1        /* invalid argument / table                                        */
#define SMX_ERR_CUDA 2       /* CUDA runtime failure (message has the CUDA error string)        */
#define SMX_ERR_NO_DEVICE 3  /* no usable GPU: the library has no CPU path by design            */
#define SMX_ERR_CAPACITY 4   /* caller-provided result buffer too small (see smx_result_bound)  */
#define SMX_ERR_INTERNAL 5

/* trim modes (reference: constants.py:40-45 TrimMode) */
#define SMX_TRIM_NONE 0
#define SMX_TRIM_PRIMERS 1
#define SMX_TRIM_BARCODES 2
#define SMX_TRIM_TAILS 3

/* resolution types (reference: constants.py:54-61 ResolutionType) */
#define SMX_RES_FULL_MATCH 1
#define SMX_RES_PARTIAL_FORWARD 2
#define SMX_RES_PARTIAL_REVERSE 3
#define SMX_RES_MULTIPLE_SPECIMENS 4
#define SMX_RES_UNKNOWN 5
#define SMX_RES_DEREPLICATED_FULL 6

/*
 * Pattern / match tables.  Replaces the in-memory registries the reference builds in
 * databases.py:123-308 (Specimens), models.py:20-31 (PrimerInfo) and the thresholds of
 * orchestration.py:548-641 (setup_match_parameters).  All arrays are caller-owned and copied.
 *
 * Primers are the reference's *canonical* primers (Specimens._primers, keyed by sequence,
 * databases.py:152-165) in first-appearance order.  Barcodes are listed per primer in the pinned
 * order the host iterates them (reference iterates a Python set, demultiplex.py:781; SURVEY.md Q2).
 */
typedef struct smx_tables {
    uint32_t n_primers;
    const char *primer_seq;        /* concatenated forward-sense primer strings (upper-case IUPAC)   */
    const char *primer_rc;         /* concatenated reverse complements (what match_one_end searches) */
    const uint32_t *primer_off;    /* n_primers+1 offsets into both strings                          */
    const uint8_t *primer_dir;     /* 0 = forward, 1 = reverse (constants.py:100-103)                */
    const int32_t *primer_k;       /* max edit distance per primer (orchestration.py:603-614)        */
    const int32_t *primer_file_index; /* order in primers.fasta (io_utils.py:279)                    */

    /* per-primer barcode lists: primer p owns entries [pb_off[p], pb_off[p+1]) of pb_barcode, each a
     * global barcode id; forward primers index the b1 namespace, reverse primers the b2 namespace.  */
    const uint32_t *pb_off;        /* n_primers+1 */
    const uint32_t *pb_barcode;

    uint32_t n_b1, n_b2;           /* distinct forward / reverse barcodes                            */
    const char *b1_rc;             /* concatenated reverse complements of forward barcodes           */
    const uint32_t *b1_off;        /* n_b1+1 */
    const char *b2_rc;
    const uint32_t *b2_off;        /* n_b2+1 */

    /* primer pairs in the reference's candidate enumeration order (demultiplex.py:699-700):
     * for fwd in get_primers(FWD): for rev in get_paired_primers(fwd).                              */
    uint32_t n_pairs;
    const uint32_t *pair_fwd;
    const uint32_t *pair_rev;
    const int32_t *pair_pool;      /* get_pool_from_primers(fwd, rev), demultiplex.py:640-665; -1 = none */

    /* specimen rows in file order (databases.py:167).  p1_mask / p2_mask: bit c set iff canonical
     * primer c is (by identity) one of the row's resolved primers (databases.py:224-225,241; Q7);
     * ceil(n_primers / 64) words per row, row r at [r * words, (r + 1) * words), bit c in word c / 64. */
    uint32_t n_specimens;
    const uint32_t *spec_b1;
    const uint32_t *spec_b2;
    const uint64_t *spec_p1_mask;
    const uint64_t *spec_p2_mask;
    const int32_t *spec_pool;
} smx_tables;

/* Flags that change results (reference: cli.py:23-41, models.py:331-338 MatchParameters). */
typedef struct smx_params {
    int32_t search_len;        /* -l / --search-len                                                */
    int32_t max_dist_index;    /* barcode threshold k_idx                                          */
    int32_t barcode_length;    /* Specimens.b_length(), databases.py:273                           */
    int32_t preorient;         /* !--disable-preorient                                             */
    int32_t prefilter;         /* !--disable-prefilter: emulate the Bloom prefilter exactly (Q5)   */
    int32_t trim;              /* SMX_TRIM_*                                                       */
    int32_t dereplicate_best;  /* --dereplicate best (1) | none (0)                                */
    int32_t min_length;        /* -1 = off                                                         */
    int32_t max_length;        /* -1 = off                                                         */
} smx_params;

/*
 * One batch of reads, packed by the host batching layer.
 *  packed2  : 2 bits per base, A=0 C=1 G=2 T=3, base i of read r at bit 2*(i%16) of word
 *             word_off[r] + i/16 (little-endian within the word); non-ACGT bases hold 0 there.
 *  clip_len : 0 = whole reads are packed.  Otherwise every read longer than 2*clip_len is stored as
 *             its first clip_len bases followed by its last clip_len bases (the only bases the
 *             path ever looks at when clip_len >= search_len); `lengths` keeps the TRUE length.
 *  stride_words : 0 = reads are packed back to back and word_off gives every read's first word.  Otherwise
 *             every read owns exactly stride_words words (read r starts at word r * stride_words) and word_off
 *             is not read (may be NULL): the form the packer produces for clipped batches, where all but the
 *             rare short reads store 2 * clip_len bases anyway.  Saves the 8-byte offset per read on the wire.
 *  lengths16: optional 16-bit form of `lengths` (all reads shorter than 65,536 bases); when non-NULL
 *             `lengths` is not read.
 *  packed4  : optional exact side stream for reads containing any non-ACGT symbol (NULL if none).
 *             For such a read r, off4[r] != UINT64_MAX and packed4 holds the forward strand then the
 *             reverse-complement strand (Biopython ambiguous-DNA complement, U->A), each
 *             ceil(len/8) words of 4-bit codes:
 *               A0 C1 G2 T3 R4 Y5 S6 W7 K8 M9 B10 D11 H12 V13 N14, 15 = any other byte (matches nothing)
 */
typedef struct smx_batch {
    uint32_t n_reads;
    const uint32_t *packed2;
    uint64_t packed2_words;
    const uint64_t *word_off;   /* n_reads */
    const uint32_t *lengths;    /* n_reads */
    const uint32_t *packed4;    /* may be NULL */
    uint64_t packed4_words;
    const uint64_t *off4;       /* may be NULL when packed4 is NULL */
    uint32_t clip_len;          /* see above; must be 0 or >= search_len */
    uint32_t stride_words;      /* see above; 0 = use word_off */
    const uint16_t *lengths16;  /* may be NULL (then `lengths` is used) */
} smx_batch;

/*
 * One output record == one WriteOperation of the reference (models.py:341-357), before string
 * formatting.  Coordinates are in the orientation-normalised sequence (candidate.sequence) and
 * already include the reference's mutating-trim behaviour (SURVEY.md Q3).  INT32_MIN = None.
 */
typedef struct smx_record {
    uint32_t read;             /* index of the read in the batch                                  */
    int32_t sample;            /* specimen row | global b1 id | global b2 id | -1, by `resolution` */
    int32_t trim_start;        /* slice [trim_start, trim_end) of the oriented read               */
    int32_t trim_end;
    int32_t p1_loc[2];         /* WriteOperation.p1_location (start, end)                         */
    int32_t p2_loc[2];
    int32_t b1_loc[2];
    int32_t b2_loc[2];
    int16_t pool;              /* pool id, -1 = "unknown"                                         */
    int16_t p1;                /* canonical primer index or -1 = "unknown"                        */
    int16_t p2;
    int8_t dist[4];            /* p1, b1, b2, p2 edit distances, -1 = 'X' (models.py:206-218)      */
    uint8_t resolution;        /* SMX_RES_*                                                       */
    uint8_t reverse;           /* 1: the record carries the reverse-complemented read             */
    uint8_t trim_empty;        /* 1: empty-trim fallback record (demultiplex.py:47-73)            */
    uint8_t candidate;         /* index of the candidate match within the read (trace ids)        */
    uint8_t pad[2];
} smx_record;               /* 64 bytes */

/*
 * Compact form of smx_record for output paths that never look at the four location pairs: in the
 * reference those feed only --color highlighting (alignment.py:59-95) and the trace, while the
 * per-specimen files need sample / names / trim extents / distance code / orientation
 * (io_utils.py:233-268).  Half the bytes on the wire: the copy-out of the records is what bounds
 * smx_match_batch with host buffers.
 */
typedef struct smx_record32 {
    uint32_t read;
    int32_t sample;
    int32_t trim_start;
    int32_t trim_end;
    int16_t pool;
    int16_t p1;
    int16_t p2;
    int8_t dist[4];
    uint8_t resolution;
    uint8_t flags;             /* bit 0: reverse, bit 1: trim_empty                               */
    uint8_t candidate;
    uint8_t pad[3];
} smx_record32;             /* 32 bytes */

/*
 * Wire form of a record for output paths that write the per-specimen files (io_utils.py:233-268): 16 bytes.
 * Records come in read order, a read's records consecutive; `flags` bit 5 marks the LAST record of its read,
 * so neither the read index nor rec_offset travels.  trim_end is sent as its distance from the read end:
 * both extents lie within search_len + barcode length of an end of the read (models.py:278-319), so 16 bits
 * hold them (SMX_MAX_SEARCH_LEN = 1024); should one ever not fit, the call fails with SMX_ERR_INTERNAL
 * (never a silently wrong extent) and the caller asks for smx_record32 records instead.
 */
typedef struct smx_record16 {
    int32_t sample;            /* as smx_record.sample                                            */
    uint16_t trim_start;       /* slice [trim_start, length - trim_tail) of the oriented read     */
    uint16_t trim_tail;
    int16_t pool;              /* -1 = "unknown"                                                  */
    uint8_t p1, p2;            /* canonical primer index, 0xFF = "unknown"                        */
    uint8_t dist_p1, dist_p2;  /* primer edit distances, 0xFF = 'X'                               */
    uint8_t dist_b;            /* barcode distances: b1 in the low nibble, b2 in the high one, 0xF = 'X' */
    uint8_t flags;             /* bits 0-2 resolution (SMX_RES_*), bit 3 reverse, bit 4 trim_empty, bit 5 last of read */
} smx_record16;             /* 16 bytes */

/* Optional per-search detail (level-1 results), used by parity tests and trace emission.
 * Slot index: ((strand * n_primers + primer) * n_reads + read); strand 0 = read as given,
 * 1 = its reverse complement.  Coordinates are the values align_seq reports (alignment.py:49). */
typedef struct smx_primer_hit {
    int32_t first_start;       /* start of locations()[0]                                         */
    int32_t first_end;         /* end of locations()[0] (smallest end)                            */
    int16_t distance;          /* -1 = no match within k                                          */
    uint16_t n_locations;      /* number of equal-best end positions                              */
} smx_primer_hit;

/* Barcode slot index: (bslot_base[strand * n_primers + primer] + j) * n_reads + read for the j-th
 * barcode of the primer; bslot_base is the running sum of barcode-list lengths over
 * (strand, primer) pairs in index order.  Valid only where the primer slot matched.             */
typedef struct smx_barcode_hit {
    uint64_t end_mask;         /* bit j: flank column j is an equal-best SHW end (end = start + j) */
    int32_t search_start;      /* barcode_search_start of the winning primer location             */
    int16_t distance;          /* -1 = none within k_idx at any primer location                   */
    uint16_t barcode;          /* position j of the barcode in its primer's list                  */
} smx_barcode_hit;

/* One barcode hit at ONE primer end location (the unmerged form of smx_barcode_hit, for -d3 traces). */
typedef struct smx_barcode_loc_hit {
    uint32_t read;
    uint16_t slot;             /* strand * n_primers + primer                                      */
    uint16_t location;         /* index of the primer end location in ascending end order          */
    smx_barcode_hit hit;       /* hit.barcode = position in the primer's list; hit.search_start = that location's */
} smx_barcode_loc_hit;      /* 24 bytes */

typedef struct smx_results {
    /* per read: records [rec_offset[r], rec_offset[r+1]) ; rec_offset has n_reads+1 entries */
    uint32_t *rec_offset;
    smx_record *records;
    uint64_t records_cap;      /* capacity of `records` (see smx_result_bound)                    */
    uint64_t n_records;        /* out                                                             */
    uint64_t n_matched;        /* out: reads with >= 1 full match (demultiplex.py:199-201)        */
    uint8_t *endmask_bits;     /* optional, may be NULL: per primer slot, search_len bits
                                  (ceil(search_len/32) words) of equal-best end positions          */
    smx_primer_hit *primer_hits;   /* optional, may be NULL: 2 * n_primers * n_reads entries      */
    smx_barcode_hit *barcode_hits; /* optional, may be NULL: 2 * sum(barcodes) * n_reads entries  */
    uint8_t *orient_hits;      /* optional, may be NULL: 2 * n_primers * n_reads flags of the explicit
                                  determine_orientation test (demultiplex.py:602-638): entry
                                  (strand * n_primers + primer) * n_reads + read = forward-sense primer found in the
                                  first search_len bases of that strand.  Only computed for reads where it can differ
                                  from the tail-window match of the other strand (shorter than search_len - 1, or
                                  with non-ACGT symbols); 0 elsewhere.  Used by the trace replay.                 */
    smx_barcode_loc_hit *barcode_loc_hits; /* optional (needs barcode_hits too): every barcode hit at every primer
                                  end location, in no particular order; at most barcode_loc_cap entries are written */
    uint64_t barcode_loc_cap;
    uint64_t n_barcode_loc_hits; /* out: entries that exist (may exceed the capacity: call again with more)       */
    smx_record32 *records32;   /* optional: when non-NULL (and `records` NULL) the records are returned in the
                                  compact form; records_cap then counts smx_record32 entries                     */
    smx_record16 *records16;   /* optional: when non-NULL (and the two above NULL) the records are returned in the
                                  16-byte wire form; records_cap counts smx_record16 entries; rec_offset may be
                                  NULL (the last-of-read flag carries the grouping)                              */
} smx_results;

typedef struct smx_ctx smx_ctx;

/* ABI version of the loaded library. */
int smx_abi_version(void);

/* Thread-local message of the last failing call on this thread. */
const char *smx_last_error(void);

/* Number of visible CUDA devices (0 when none; never an error). */
int smx_device_count(void);

/* PCI bus id of a device ("0000:1b:00.0"), so that the host layer can pin its feeder thread and its
 * pinned buffers to the NUMA node the GPU hangs off (SURVEY.md 8e: the host is the scaling limiter). */
int smx_device_pci_bus_id(int device, char *out, int len);

/* Build a context on `device`: copies the tables, builds IUPAC-aware Peq masks (edlib
 * additionalEqualities semantics, constants.py:13-20) and the specimen lookup table.
 * Replaces read_primers_file/read_specimen_file products + setup_match_parameters thresholds. */
int smx_create(int device, const smx_tables *tables, const smx_params *params, smx_ctx **out);

void smx_destroy(smx_ctx *ctx);

/* Upper bound on records for a batch of n reads (sizing of smx_results.records). */
uint64_t smx_result_bound(const smx_ctx *ctx, uint32_t n_reads);

/* Whole path for one batch with HOST buffers: H2D copy, window staging, primer HW search,
 * barcode SHW search, selection/dereplication, D2H of the records.
 * Replaces process_sequences' matching and selection (demultiplex.py:108-212,216-598,602-820). */
int smx_match_batch(smx_ctx *ctx, const smx_batch *batch, smx_results *out);

/* smx_match_batch cuts batches of more than 1.5 * reads_per_chunk reads into chunks that rotate over
 * three streams, overlapping one chunk's H2D, another's kernels and a third's D2H; the results are
 * identical to the one-shot form.  Default 262144 (env SMX_PIPELINE_CHUNK); 0 disables.  The
 * reference's unit of work is a 1000-read batch per worker process (orchestration.py:165,199). */
int smx_set_pipeline_chunk(smx_ctx *ctx, uint32_t reads_per_chunk);
int smx_last_chunk_count(const smx_ctx *ctx);   /* chunks used by the last smx_match_batch */

/* Reads of the last smx_run_resident that left the fast selection kernel for the general one
 * (several equal-best candidates, tied barcodes, TAILS trimming): a tuning statistic. */
uint64_t smx_last_deferred(const smx_ctx *ctx);

/* Split form of smx_match_batch for pipelining and device-resident timing. */
int smx_upload_batch(smx_ctx *ctx, const smx_batch *batch);   /* H2D only                         */
int smx_run_resident(smx_ctx *ctx);                           /* kernels only, on the last upload  */
int smx_download_results(smx_ctx *ctx, smx_results *out);     /* D2H only                         */

/* The resident form cuts batches of >= 131072 reads into `n_sub_batches` (default 2, env
 * SMX_RESIDENT_SPLIT, 1..8) pieces that run concurrently on separate streams: one piece's
 * latency-bound tail (general selection, scan, compaction) overlaps another's ALU-bound search
 * kernels.  Results are identical.  With more than one piece the per-stage / per-kernel times below
 * read 0 (the kernels overlap); set 1 to measure them.  Takes effect at the next smx_upload_batch. */
int smx_set_resident_split(smx_ctx *ctx, uint32_t n_sub_batches);

/* Whole path for reads that are already in device memory of the context's device: `bases` (n_bases bytes) and
 * seq_off (n_reads + 1 offsets into bases) are device pointers, packed on the device with clip = search_len.
 * rec_offset (n_reads + 1) and records (records_cap) are device pointers; n_records / n_matched / device_ms are host.
 * Work is ordered after everything already enqueued on `stream` (a cudaStream_t, 0 = legacy default stream); the call
 * returns when records and offsets are written.  Records, offsets and n_matched equal smx_match_batch on the same
 * reads packed by smx_pack_reads_fixed(clip_len = search_len).  device_ms (optional, 2 floats): [0] pack kernels,
 * [1] the whole call on the device.  SMX_ERR_CAPACITY sets *n_records to the need.
 * Offsets that descend, end past n_bases or give a read of 2^31 bases or more fail the call with SMX_ERR_ARG naming the
 * first such read (checked on the device before any base is read), as do pointers that are not memory of the context's
 * device.  Batches of >= 131072 reads run as smx_set_resident_split sub-batches.  Afterwards the resident form needs a
 * fresh smx_upload_batch; smx_last_timing / smx_last_kernel_times still describe the last smx_run_resident. */
int smx_match_device(smx_ctx *ctx, const char *bases, uint64_t n_bases, const uint64_t *seq_off, uint32_t n_reads,
                     void *stream, uint32_t *rec_offset, smx_record *records, uint64_t records_cap,
                     uint64_t *n_records, uint64_t *n_matched, float *device_ms);

/* The demultiplexed output of records, in device memory: for each destination file of the output tree, the trimmed,
 * oriented sequences and qualities that the output-tree writer of include/specimux_io.h writes to it, byte for byte.  bases / quals
 * (n_bases bytes; quals NULL: none) and seq_off (n_reads + 1 offsets) are the reads the records index, records
 * (n_records) e.g. what smx_match_device returned for them.  Every array is a device pointer of the context's device;
 * n_groups, n_out_bytes and device_ms are host pointers.
 *  - Output i is record order[i] (n_records entries).  Outputs are sorted stably by destination: within a file they
 *    keep record order, the order in which the writer appends them.
 *  - out_seq[out_off[i] .. out_off[i + 1]) (out_off: n_records + 1 entries) is the slice [trim_start, trim_end) of the
 *    oriented read as Python slices it (the whole read for trim_empty records), reverse-complemented (Biopython's
 *    ambiguous-DNA complement: IUPAC, lower case, U -> A) when `reverse` is set.  out_qual holds the same slice of the
 *    qualities, reversed when `reverse` is set (not written when quals is NULL).
 *  - Destination g (of *n_groups) owns outputs [group_off[g], group_off[g + 1]); group_key[g] is its 64-bit key:
 *    top (0 full, 1 partial, 2 unknown) << 62 | pool + 1 << 52 | p1 + 1 << 44 | p2 + 1 << 36 | kind << 30 | sample,
 *    where a 0 field is "unknown" and kind is 0 specimen, 1 b1, 2 b2, 3 unknown; the path of the file is
 *    <top>/<pool>/<p1>-<p2>/<prefix><sample file id><ext>.  Capacities: n_records keys, n_records + 1 offsets.
 *  - The pool-level copies of full matches (full/<pool>/<prefix><sample file id><ext>) are not separate groups: such a
 *    file holds the outputs of that pool and specimen whose record is a full match (SMX_RES_FULL_MATCH or
 *    SMX_RES_DEREPLICATED_FULL, not trim_empty), taken in the order of `order` (record order).
 * Work is ordered after everything already enqueued on `stream` (a cudaStream_t, 0 = legacy default stream); the call
 * returns when everything is written.  device_ms (optional, 2 floats): [0] the copy kernels, [1] the whole call.
 * Offsets that descend, end past n_bases or give a read of 2^31 bases or more, records that name a read >= n_reads or a
 * specimen / barcode / pool / primer outside the context's tables, tables with more than 1,023 pools or 2^30
 * specimens or barcodes, and pointers that are not memory of the context's device fail the call with SMX_ERR_ARG naming
 * the first such item; offsets and records are checked on the device before any base is read, and the context stays
 * usable.  An out_cap (bytes of out_seq, and of out_qual) below the need fails with SMX_ERR_CAPACITY and sets
 * *n_out_bytes to the need. */
int smx_demux_device(smx_ctx *ctx, const char *bases, const char *quals, uint64_t n_bases, const uint64_t *seq_off,
                     uint32_t n_reads, const smx_record *records, uint64_t n_records, void *stream, uint64_t *order,
                     uint64_t *out_off, char *out_seq, char *out_qual, uint64_t out_cap, uint64_t *group_key,
                     uint64_t *group_off, uint64_t *n_groups, uint64_t *n_out_bytes, float *device_ms);

/* Every output file's complete contents, in device memory: what the output-tree writer of include/specimux_io.h
 * (output_dir given) appends to each file for these records, byte for byte, headers included.  The reads, qualities and
 * records are as for smx_demux_device; besides them:
 *  - titles (n_title_bytes) with title_off (n_reads + 1 offsets): each read's whole title line without its '@' / '>',
 *    as the native reader's block holds them.  The header's id is the title's first token split at Python whitespace
 *    (UTF-8 whitespace included).
 *  - names (n_name_bytes) with name_off: the name tables in one blob -- specimen ids, b1 ids ("barcode_fwd_<b1>"),
 *    b2 ids ("barcode_rev_<b2>"), pools, primer names, in that order; name k is names[name_off[k] .. name_off[k + 1]).
 *    name_counts (host, 5 entries) gives the size of each table and must equal the context's tables.
 *  - is_fastq: FASTQ records (qualities; 'I' for every base when quals is NULL) or FASTA records.
 * Every array is a device pointer of the context's device; name_counts, n_files, n_outputs, n_out_bytes and
 * device_ms are host pointers.
 *  - Output i (of *n_outputs) is the formatted record of record out_record[i]; its bytes are
 *    out[out_off[i] .. out_off[i + 1]).  A record goes to its primary file and, when it is a full match (SMX_RES_FULL_MATCH
 *    or SMX_RES_DEREPLICATED_FULL, not trim_empty), to the pool-level copy full/<pool>/<prefix><sample file id><ext> too.
 *  - Outputs are sorted stably by file key; file f (of *n_files) is out[file_off[f] .. file_off[f + 1]) and has the key
 *    file_key[f]: the primary files' 64-bit key of smx_demux_device, and for the pool-level copies
 *    3 << 62 | pool + 1 << 52 | kind << 30 | sample.  Within a file the records keep their order.
 *  - Capacities: out_record and file_key 2 * n_records entries, out_off and file_off 2 * n_records + 1.
 * Work is ordered after everything already enqueued on `stream`; the call returns when everything is written.
 * device_ms (optional, 2 floats): [0] the copy kernels, [1] the whole call.  All lengths and offsets are 64-bit.
 * Read or title offsets that descend, end past their buffer or give an item of 2^31 bytes or more, bad name offsets,
 * name counts unlike the context's tables, records as smx_demux_device refuses them, more than 2^30 - 1 records and
 * pointers that are not memory of the context's device fail the call with SMX_ERR_ARG naming the first such item; the
 * offsets and records are checked on the device before any byte is copied, and the context stays usable.  An out_cap
 * below the need fails with SMX_ERR_CAPACITY and sets *n_out_bytes to the need. */
int smx_demux_files_device(smx_ctx *ctx, const char *bases, const char *quals, uint64_t n_bases, const uint64_t *seq_off,
                           uint32_t n_reads, const char *titles, uint64_t n_title_bytes, const uint64_t *title_off,
                           const smx_record *records, uint64_t n_records, const char *names, uint64_t n_name_bytes,
                           const uint64_t *name_off, const uint32_t *name_counts, int is_fastq, void *stream,
                           uint64_t *out_record, uint64_t *out_off, char *out, uint64_t out_cap, uint64_t *file_key,
                           uint64_t *file_off, uint64_t *n_files, uint64_t *n_outputs, uint64_t *n_out_bytes,
                           float *device_ms);

/* specimine over the files of smx_demux_files_device (FASTQ), in device memory: for each group, the best full read of
 * every partial read, the identity rule and the rewritten records, byte for byte what specimine writes into
 * <full file>.mined on the tree those files make.  The file buffer is the one smx_demux_files_device wrote:
 *  - data (n_data bytes) with out_off (n_outputs + 1 offsets, device): output i is data[out_off[i] .. out_off[i + 1]),
 *    one formatted FASTQ record, '@' title '\n' sequence '\n' '+' '\n' qualities '\n'.
 *  - file_off (host, n_files + 1): file f is data[file_off[f] .. file_off[f + 1]) and starts and ends on output
 *    boundaries.
 * The groups (host, CSR): group g searches the outputs of file grp_file[g] (the full reads, in file order) in the outputs
 * of files grp_part[grp_part_off[g] .. grp_part_off[g + 1]) (the partial reads, in that order); grp_kind[g] is 0 forward,
 * 1 reverse.  .mined file j holds the mined records of groups [mined_grp[j], mined_grp[j + 1]) in group order
 * (mined_grp: n_mined + 1 entries, from 0 to n_groups).  min_identity as specimine's --min-identity: a full read of m
 * bytes searches with limit int(m * (1 - min_identity)), and a partial read is mined when its best full read (the
 * smallest d / m, ties to the first) has identity 1 - d / m >= min_identity and > 0.
 * Outputs (device): out holds every mined record, .mined file j is out[mined_off[j] .. mined_off[j + 1]) (n_mined + 1
 * entries); mined record r rewrites partial output rec_partial[r], whose best full read is output rec_winner[r] at
 * distance rec_dist[r].
 * Work is ordered after everything already enqueued on `stream`; the call returns when everything is written.
 * device_ms (optional, 2 floats): [0] the search kernels, [1] the whole call.  All lengths and offsets are 64-bit.
 * A group table that names a file outside [0, n_files) or whose offsets descend, file offsets that descend or end past
 * n_data, min_identity NaN, more than 2^29 - 1 files or 2^32 - 2 outputs, a file whose range does not start and end on
 * output boundaries, an output that is not a FASTQ record, a full read longer than 4,096 bytes or holding more than 64
 * distinct byte values, a full file of more than 2^23 outputs (the search key holds the winner's rank in 23 bits, as
 * smx_hw_best_grouped limits its groups; the first output past the limit is named), and pointers that are not memory
 * of the context's device fail the call with SMX_ERR_ARG naming the first such item (file and output within it); the outputs are checked on the device before any search runs, and
 * the context stays usable.  An out_cap (bytes) or rec_cap (records) below the need fails with SMX_ERR_CAPACITY and
 * sets *n_out_bytes and *n_records to the need. */
int smx_mine_device(smx_ctx *ctx, const char *data, uint64_t n_data, const uint64_t *out_off, uint64_t n_outputs,
                    const uint64_t *file_off, uint64_t n_files, uint32_t n_groups, const uint32_t *grp_file,
                    const uint8_t *grp_kind, const uint32_t *grp_part_off, const uint32_t *grp_part, uint32_t n_mined,
                    const uint32_t *mined_grp, double min_identity, void *stream, char *out, uint64_t out_cap,
                    uint64_t rec_cap, uint64_t *mined_off, int64_t *rec_partial, int64_t *rec_winner, int32_t *rec_dist,
                    uint64_t *n_records, uint64_t *n_out_bytes, float *device_ms);

/* CUDA-event time (ms) of the last smx_run_resident, and of its stages:
 * stage 0 staging, 1 primer search, 2 barcode search, 3 selection. */
int smx_last_timing(const smx_ctx *ctx, float *total_ms, float stage_ms[4]);

/* CUDA-event time (ms) of the individual kernels of the last smx_run_resident (first pass; a
 * capacity re-run overwrites the marks it passes again).  Fills up to n entries and returns the
 * number available, in this order: 0 window staging, 1 sliced primer search (all primers, they run
 * concurrently), 2 primer finish / classic search, 3 primer start recovery, 4 barcode search,
 * 5 fast selection, 6 general selection, 7 record scan + compaction (one kernel), 8 offset rebase. */
int smx_last_kernel_times(const smx_ctx *ctx, float *ms, int n);

/* Number of kernel launches issued by the last smx_run_resident. */
int smx_last_launch_count(const smx_ctx *ctx);

/* Work done by the last smx_run_resident, counted on the device with the SURVEY.md 8d formulas:
 * cells[0] = HW cells, cells[1] = SHW cells, wordcols[0..1] the same in 32-bit word-columns. */
int smx_last_work(const smx_ctx *ctx, uint64_t cells[2], uint64_t wordcols[2]);

/* Bit-sliced DP cells the last smx_run_resident actually evaluated, counted on the device: cells[0] = stage 1
 * (pattern rows x window columns per group of 32 reads, strand and primer), cells[1] = stage 2 (band cells x
 * 32-barcode words per work entry).  One cell of either automaton costs 5 three-input logic ops for its 32
 * problems, so 5 x cells / kernel time is the useful-op rate set against the measured integer peak. */
int smx_last_useful_cells(const smx_ctx *ctx, uint64_t cells[2]);

/* Batched global (NW) edit distances between all pairs of `n` strings, on the GPU.
 * Replaces the O(B^2) edlib.align(task="distance") loop of orchestration.py:549-555.
 * out[i*n + j] = distance(seq_i, seq_j). */
int smx_pairwise_nw(int device, const char *seqs, const uint32_t *seq_off, uint32_t n, int32_t *out);

/* All-pairs infix (HW) edit distances of `n_patterns` byte strings in `n_texts` byte strings on the GPU, plain byte
 * equality: out[i * n_texts + j] = min over substrings s of text j of the edit distance (pattern i, s), or -1 when
 * that exceeds pat_k[i] (pat_k[i] < 0: unbounded).  Patterns up to 4096 bytes.  Replaces the
 * edlib.align(full_seq, partial_seq, mode="HW", task="path", k=max_distance) loop of specimine
 * (specimine.py:226-248), which reads only editDistance from the result.  Empty pattern: 0; empty text: the
 * pattern's length whatever k (edlib's empty-sequence rule). */
int smx_hw_distances(int device, const char *patterns, const uint64_t *pat_off, const int32_t *pat_k, uint32_t n_patterns,
                     const char *texts, const uint64_t *txt_off, uint32_t n_texts, int32_t *out);

/* Grouped best match, the arithmetic of specimine over many specimens in one call.  Group g owns patterns
 * [grp_pat_off[g], grp_pat_off[g + 1]) and the text-list entries [grp_txt_off[g], grp_txt_off[g + 1]) (CSR), entry e
 * naming text grp_txt_idx[e]; texts may be named by several groups.  With d(i, t) the value smx_hw_distances reports
 * (-1 above pat_k[i], the pattern's length for an empty text), the winner of an entry is the pattern of its group with
 * the smallest d / m (exact rational) among those with d != -1 and m > 0, ties to the smallest index: best_pat[e] is
 * its index within the group, best_dist[e] its distance, both -1 when there is none.  1 - d / m in float64 orders the
 * patterns the same way (m <= 4096), so the winner is specimine's first full read with the highest identity.
 * Patterns up to 4096 bytes, groups up to 2^23 patterns (SMX_ERR_ARG beyond), a pattern with more than 64 distinct
 * bytes fails the call (SMX_ERR_ARG).  device_ms (optional) receives the CUDA-event time of the kernels.  No
 * distance matrix is stored: device memory is the inputs plus 8 bytes per entry. */
int smx_hw_best_grouped(int device, const char *patterns, const uint64_t *pat_off, const int32_t *pat_k, uint32_t n_patterns,
                        const char *texts, const uint64_t *txt_off, uint32_t n_texts, uint32_t n_groups,
                        const uint32_t *grp_pat_off, const uint64_t *grp_txt_off, const uint32_t *grp_txt_idx,
                        int32_t *best_pat, int32_t *best_dist, float *device_ms);

/* Integer-ALU roofline denominator: measured throughput (10^12 ops/s) of independent 32-bit
 * LOP3 (logic) and IADD3 (add) chains over the whole chip, the two instruction classes of the
 * Myers column step.  out[0] = LOP3-only, out[1] = IADD3-only, out[2] = 1:1 mix. */
int smx_int_alu_peak(int device, double out_tops[3]);

/* Evict the L2 cache (writes a buffer larger than L2) -- timing hygiene between benchmark steps. */
int smx_flush_l2(smx_ctx *ctx);

/* Pinned host memory for batch / result buffers (cudaHostAlloc / cudaFreeHost). */
void *smx_host_alloc(uint64_t bytes);
void smx_host_free(void *p);

/* Host-side packer (no matching): ASCII reads -> the smx_batch encoding above.
 * Replaces nothing in the reference (it works on Python strings); part of the batching layer.
 * Call with out arrays sized by smx_pack_bound. Returns the number of flagged (packed4) reads in
 * *n_flagged. */
void smx_pack_bound(const uint64_t *seq_off, uint32_t n_reads, uint32_t clip_len,
                    uint64_t *packed2_words, uint64_t *packed4_words_max);
int smx_pack_reads(const char *bases, const uint64_t *seq_off, uint32_t n_reads, uint32_t clip_len,
                   uint32_t *packed2, uint64_t *word_off, uint32_t *lengths,
                   uint32_t *packed4, uint64_t *off4, uint64_t *packed4_words, uint32_t *n_flagged);

/* Fixed-stride form of the packer for clipped batches (clip_len > 0): every read owns
 * smx_pack_stride(clip_len) words of `packed2` (n_reads * stride + 1 words in all), no word_off.  lengths16
 * (optional) receives the 16-bit lengths when every read is shorter than 65,536 bases; *lengths_fit16 says so. */
uint32_t smx_pack_stride(uint32_t clip_len);
int smx_pack_reads_fixed(const char *bases, const uint64_t *seq_off, uint32_t n_reads, uint32_t clip_len,
                         uint32_t *packed2, uint32_t *lengths, uint16_t *lengths16, int *lengths_fit16,
                         uint32_t *packed4, uint64_t *off4, uint64_t *packed4_words, uint32_t *n_flagged);

/* Measured pinned-memory copy bandwidth of `device` (GB/s) for `bytes`-sized transfers: out[0] host-to-device,
 * out[1] device-to-host, out[2] both directions at once (sum of the two).  The roofline of the host-buffer path. */
int smx_copy_peak(int device, uint64_t bytes, double out_gbs[3]);

#ifdef __cplusplus
}
#endif
#endif /* SPECIMUX_B200_H */
