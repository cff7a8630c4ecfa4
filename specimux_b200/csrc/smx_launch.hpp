// smx_launch.hpp -- host-callable launchers of the kernels (one translation unit per stage, see Makefile).
// Every launcher enqueues on `st` and returns the launch error (cudaGetLastError), nothing synchronises.
#pragma once
#include <cuda_runtime.h>

#include "smx_core.cuh"
#include "smx_mine.cuh"
#include "smx_out.cuh"
#include "smx_pack.cuh"

namespace smx {

constexpr int kScanTile = 1024;         // reads per tile of k_scan_compact (sizes the tile status array)

// stage 0 / 1
cudaError_t launch_stage_windows(const Tables &t, const Batch &b, cudaStream_t st);
// prow_code: the primer's 32 pattern-row IUPAC codes (HostTables::prow_code + 32 * primer)
cudaError_t launch_primer_sliced(const Tables &t, const Batch &b, int primer, const unsigned char *prow_code, cudaStream_t st);
// finish of both strands per (read, primer) + work entries + start of the first location in the single-word form:
// with_start 0 = none, 1 = only what launch_primer_start_sliced leaves out, 2 = every matched slot
cudaError_t launch_primer_finish(const Tables &t, const Batch &b, int with_start, cudaStream_t st);
// start of the first location, bit-sliced across 32 work entries (primers with start_sliced_ok); prow_code as above
cudaError_t launch_primer_start_sliced(const Tables &t, const Batch &b, int primer, const unsigned char *prow_code, cudaStream_t st);
cudaError_t launch_primer_long(const Tables &t, const Batch &b, int primer, cudaStream_t st);
// stage 2: one launch per (task width, barcode length) class; class_tasks is the DEVICE copy of
// HostTables::bt_class_tasks.  *launches receives the number of kernels enqueued.
cudaError_t launch_barcode_tasks(const Tables &t, const Batch &b, const unsigned short *class_tasks,
                                 const BtClass *classes, int n_classes, cudaStream_t st, int *launches);
// one translation unit per barcode threshold (smx_k_stage2.cu, -DSMX_STAGE2_K=k)
#define SMX_DECL_K2(KK) cudaError_t launch_barcode_class_k##KK(const Tables &t, const Batch &b, const unsigned short *list, \
                                                                int n_list, int nw, int m, int quad, cudaStream_t st);
SMX_DECL_K2(0) SMX_DECL_K2(1) SMX_DECL_K2(2) SMX_DECL_K2(3) SMX_DECL_K2(4) SMX_DECL_K2(5) SMX_DECL_K2(6) SMX_DECL_K2(7) SMX_DECL_K2(8)
SMX_DECL_K2(9) SMX_DECL_K2(10) SMX_DECL_K2(11) SMX_DECL_K2(12)
#undef SMX_DECL_K2
// stage 3
cudaError_t launch_select_fast(const Tables &t, const Batch &b, cudaStream_t st);
cudaError_t launch_select(const Tables &t, const Batch &b, cudaStream_t st);
cudaError_t launch_select_big(const Tables &t, const Batch &b, const u32 *list, u32 n_list, unsigned char *scratch, cudaStream_t st);
cudaError_t launch_scan_compact(const Tables &t, const Batch &b, u32 rec_cap, unsigned long long *tile_status, u32 *ticket,
                                u32 ticket_base, u32 epoch, cudaStream_t st);
cudaError_t launch_pack_records32(const smx_record *in, u32 n, smx_record32 *out, cudaStream_t st);
cudaError_t launch_pack_records16(const smx_record *in, u32 n, const u32 *lengths, u32 read_base, smx_record16 *out, u32 *bad,
                                  cudaStream_t st);
cudaError_t launch_expand_lengths(const unsigned short *in, u32 n, u32 *out, cudaStream_t st);
cudaError_t launch_rebase_offsets(const u32 *in, u32 n, u32 rec_base, u32 *out, cudaStream_t st);
// specimine: HW distances of the patterns listed in pat_list (all of one (lanes, words per lane) class) in every text
cudaError_t launch_hw_distance(int sw, int w, const unsigned char *pat, const u64 *pat_off, const i32 *pat_k, const u32 *pat_list,
                               u32 n_list, const unsigned char *txt, const u64 *txt_off, u32 n_txt, i32 *out, u32 *bad,
                               cudaStream_t st);
// specimine, grouped (HwItem, hw_best_class, hw_best_chunk: smx_mine.cuh).  Items of one launch are all of one (SW, W)
// class, each covers at most hw_best_chunk(SW) entries.  Pattern / text i is the bytes [start(i), start(i) + len(i)).
using smx_mine::HwItem;
using smx_mine::hw_best_class;
using smx_mine::hw_best_chunk;
struct HwContig {                       // contiguous: item i is bytes[off[i] .. off[i + 1])
    const unsigned char *bytes;
    const u64 *off;
    __device__ __forceinline__ u64 start(u32 i) const { return off[i]; }
    __device__ __forceinline__ int len(u32 i) const { return (int)(off[i + 1] - off[i]); }
};
struct HwSpans {                        // outputs of a device file buffer: item i is bytes[beg[i] .. beg[i] + n[i])
    const unsigned char *bytes;
    const u64 *beg;
    const u32 *n;
    __device__ __forceinline__ u64 start(u32 i) const { return beg[i]; }
    __device__ __forceinline__ int len(u32 i) const { return (int)n[i]; }
};
template <class Seqs>
cudaError_t launch_hw_best(int sw, int w, Seqs pats, const i32 *pat_k, const HwItem *items, u32 n_items, Seqs txts,
                           const u32 *ent_txt, unsigned long long *keys, u32 *bad, cudaStream_t st);
// specimine on device files (smx_k_mine_device.cu, smx_mine_device).  locate: the output range of every involved file,
// every output's sequence (seq_beg, seq_len) and search limit (k), the group scan (pat_base, ent_base; ctl[1] patterns,
// ctl[2] entries) and the plan (limits into ctl[0] as the least fault key, work items per class into ctl[3 + c]).
// items: the work items at the class cursors ctl[3 + kHwClasses + c] and every entry's text.  decide: per entry the
// size of its mined record, flag, winner and distance, and the exclusive scans size_off / flag_off over E + 1 entries.
// format: the record arrays, the .mined file offsets and every byte of the records.
struct MineArgs {
    const unsigned char *data;
    u64 n_data;
    const u64 *out_off, *file_off;
    u64 n_outputs, n_files;
    u32 n_groups, n_mined, n_involved;
    const u32 *grp_file, *grp_kind, *grp_part_off, *grp_part, *mined_grp, *involved;
    double min_identity;
    u64 *file_rng, *seq_beg;
    u32 *seq_len;
    i32 *k;
    u64 *pat_base, *ent_base;
    unsigned long long *ctl;
    HwItem *items;
    u32 *ent_txt;
    unsigned long long *keys;
    u64 *size, *size_off, *flag, *flag_off, *winner, *rec_off;
    u32 *dist;
    unsigned char *rec_kind;
    void *temp;
    size_t temp_bytes;
};
struct MineOut {
    unsigned char *bytes;
    u64 *mined_off;
    int64_t *partial, *winner;
    int32_t *dist;
};
constexpr int kMineCtlWords = 3 + 2 * smx_mine::kHwClasses;
cudaError_t launch_mine_locate(const MineArgs &a, cudaStream_t st);
cudaError_t launch_mine_items(const MineArgs &a, u64 P, u64 E, cudaStream_t st);
cudaError_t mine_scan_temp_bytes(u64 n, size_t *bytes);
cudaError_t launch_mine_decide(const MineArgs &a, u64 E, cudaStream_t st);
cudaError_t launch_mine_format(const MineArgs &a, u64 E, u64 R, const MineOut &out, cudaStream_t st);
// device packer (smx_k_pack.cu), clip and stride in `d`.  validate: *bad = min over refused reads of
// (read << 2 | PackFault), left untouched when every read passes.  fixed: packed2 + lengths of every lane, flag[r] (zeroed
// by the caller) and the unordered list of flagged reads, counted in *n_flagged (zeroed by the caller).  off4: every
// read's off4 (tile_sum holds ceil(n / kPackTile) words of scratch, kPackTile in smx_pack.cuh).  side: the packed4 words of the listed reads.
cudaError_t launch_pack_validate(const u64 *seq_off, u32 n, u64 n_bases, unsigned long long *bad, cudaStream_t st);
cudaError_t launch_pack_fixed(const unsigned char *bases, const u64 *seq_off, u32 n, const PackLanes &d, u32 *flag, u32 *list,
                              unsigned long long *n_flagged, cudaStream_t st);
cudaError_t launch_pack_off4(const u64 *seq_off, u32 n, const u32 *flag, u64 *tile_sum, const PackLanes &d, cudaStream_t st);
cudaError_t launch_pack_side(const unsigned char *bases, const u64 *seq_off, const u32 *list, u32 n_list, const PackLanes &d,
                             u32 *packed4, cudaStream_t st);
// device demultiplexer (smx_k_demux.cu).  index: plan (validation into ctl[1], min over refused records of
// record << 3 | OutFault, left untouched when all pass), stable radix sort of (compact key, record), order / out_off (the
// exclusive scan of the output lengths, total in out_off[n]) / the sorted source positions, the groups (count into
// ctl[2], group_off[G] = n) and ctl[3] = total bytes.  Reads no base; n_records >= 1.  temp: demux_temp_bytes(n) bytes.
// copy: every output byte (tile_first: demux_tile_marks entries).
struct DemuxScratch {
    u64 *key_in, *key_out, *src, *out_src;
    u32 *rec_in, *rec_out, *len;
    void *temp;
    size_t temp_bytes;
    unsigned long long *ctl;
};
struct DemuxIndex {
    const smx_record *records;
    u64 n_records;
    const u64 *seq_off;
    u32 n_reads;
    smx_out::OutCounts counts;
    smx_out::OutShape shape;
    u64 *order, *out_off, *group_key, *group_off;
    DemuxScratch scratch;
    const struct FilesIndex *files;     // null: smx_demux_device; else smx_demux_files_device
};
// smx_demux_files_device's index pass: files_plan_item over two slots per record (lengths in `len`, 2n; hdr, id_pos
// per record), the sort over shape.total_bits + 1 bits, order / out_off / out_src over the 2n slots, file keys into
// group_key and their first slots into group_idx (2n + 1), file_off[f] = out_off[group_idx[f]] (bytes), ctl[4] = files,
// ctl[5] = outputs (the slots before the first empty one).  Scratch arrays of DemuxScratch hold 2n entries.
struct FilesIndex {
    smx_out::FilesPlan plan;
    u64 *len, *hdr, *id_pos, *group_idx, *file_off;
};
cudaError_t demux_temp_bytes(u64 n, size_t *bytes);
cudaError_t launch_demux_index(const DemuxIndex &a, cudaStream_t st);
u64 demux_tile_marks(u64 total, const void *out_seq, const void *out_qual);
cudaError_t launch_demux_copy(const unsigned char *bases, const unsigned char *quals, const u64 *out_off, const u64 *out_src,
                              u64 n_out, u64 total, unsigned char *out_seq, unsigned char *out_qual, u64 *tile_first,
                              cudaStream_t st);
cudaError_t launch_files_copy(const smx_out::FilesCopy &f, u64 *tile_first, cudaStream_t st);
// utilities
cudaError_t launch_pairwise_nw(const char *seqs, const u32 *off, u32 n, i32 *out, cudaStream_t st);
cudaError_t launch_int_peak(int mode, int blocks, int threads, u32 *out, int iters, u32 seed, cudaStream_t st);

}  // namespace smx
