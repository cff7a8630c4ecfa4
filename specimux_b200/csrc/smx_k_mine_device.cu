// smx_k_mine_device.cu -- specimine on the files of smx_demux_files_device, in device memory (smx_mine_device).  The
// per-file, per-output, per-pattern and per-entry work items are the routines of smx_mine.cuh that tests/minesim runs
// as host loops; what is here is their launch geometry, the group scan, the scans of the decisions (CUB) and the
// warp-per-record copy of the mined records.  The search itself is k_hw_best (smx_k_mine.cu) over HwSpans.
#include <cub/cub.cuh>

#include "smx_launch.hpp"

namespace smx {

using namespace smx_mine;

namespace {

constexpr int kMineThreads = 256;
constexpr int kMineScanThreads = 256;

unsigned mine_blocks(u64 items) {
    const u64 b = (items + kMineThreads - 1) / kMineThreads;
    return (unsigned)(b < 1 ? 1 : b > (1u << 16) ? (1u << 16) : b);
}

__device__ __forceinline__ bool mine_refused(const unsigned long long *ctl) { return *(volatile const unsigned long long *)ctl != ~0ull; }

// the group owning flat index i of a CSR whose offsets are base[0 .. G]
__device__ __forceinline__ u32 mine_group_of(const u64 *base, u32 G, u64 i) {
    u32 lo = 0, hi = G - 1;
    while (lo < hi) {
        const u32 mid = (lo + hi + 1) >> 1;
        if (base[mid] <= i) lo = mid; else hi = mid - 1;
    }
    return lo;
}

}  // namespace

// One block per involved file: its output range (thread 0), then every output's sequence, length and search limit.
__global__ void __launch_bounds__(kMineThreads) k_mine_locate(MineArgs a) {
    __shared__ u64 s_rng[2];
    const u32 f = a.involved[blockIdx.x];
    if (threadIdx.x == 0) {
        u64 o0, o1;
        const u64 key = mine_locate_file(a.out_off, a.n_outputs, a.file_off, f, o0, o1);
        if (key != ~0ull) atomicMin(a.ctl, (unsigned long long)key);
        s_rng[0] = o0; s_rng[1] = o1;
        a.file_rng[2 * f] = o0; a.file_rng[2 * f + 1] = o1;
    }
    __syncthreads();
    const u64 o0 = s_rng[0], o1 = s_rng[1];
    for (u64 o = o0 + threadIdx.x; o < o1; o += blockDim.x) {
        u64 beg;
        u32 len;
        const int fault = mine_locate_output(a.data, a.n_data, a.out_off, o, beg, len);
        if (fault) atomicMin(a.ctl, (unsigned long long)mine_fault_key(f, o - o0, fault));
        a.seq_beg[o] = beg; a.seq_len[o] = len;
        a.k[o] = mine_k(len, a.min_identity);
    }
}

// One block: per group its patterns (the full file's outputs) and entries (its partial files' outputs), scanned into
// pat_base / ent_base (G + 1 each); ctl[1] = patterns, ctl[2] = entries.
__global__ void __launch_bounds__(kMineScanThreads) k_mine_groups(MineArgs a) {
    typedef cub::BlockScan<unsigned long long, kMineScanThreads> Scan;
    __shared__ typename Scan::TempStorage s_scan;
    __shared__ unsigned long long s_carry[2];
    if (mine_refused(a.ctl)) return;
    if (threadIdx.x == 0) s_carry[0] = s_carry[1] = 0;
    __syncthreads();
    for (u32 g0 = 0; g0 < a.n_groups; g0 += kMineScanThreads) {
        const u32 g = g0 + threadIdx.x;
        unsigned long long np = 0, ne = 0;
        if (g < a.n_groups) {
            const u32 f = a.grp_file[g];
            np = a.file_rng[2 * f + 1] - a.file_rng[2 * f];
            for (u32 k = a.grp_part_off[g]; k < a.grp_part_off[g + 1]; ++k) {
                const u32 p = a.grp_part[k];
                ne += a.file_rng[2 * p + 1] - a.file_rng[2 * p];
            }
        }
        unsigned long long xp, xe, tp, te;
        Scan(s_scan).ExclusiveSum(np, xp, tp);
        __syncthreads();
        Scan(s_scan).ExclusiveSum(ne, xe, te);
        if (g < a.n_groups) { a.pat_base[g] = s_carry[0] + xp; a.ent_base[g] = s_carry[1] + xe; }
        __syncthreads();
        if (threadIdx.x == 0) { s_carry[0] += tp; s_carry[1] += te; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        a.pat_base[a.n_groups] = s_carry[0]; a.ent_base[a.n_groups] = s_carry[1];
        a.ctl[1] = s_carry[0]; a.ctl[2] = s_carry[1];
    }
}

// A pattern of flat index p: its group, rank and output.
__device__ __forceinline__ void mine_pattern(const MineArgs &a, u64 p, u32 &g, u32 &rank, u64 &o) {
    g = mine_group_of(a.pat_base, a.n_groups, p);
    rank = (u32)(p - a.pat_base[g]);
    o = a.file_rng[2 * a.grp_file[g]] + rank;
}

// One warp per pattern: the limits of the search (length, distinct bytes), then its work items per class into ctl[3 + c].
__global__ void __launch_bounds__(kMineThreads) k_mine_plan(MineArgs a) {
    if (mine_refused(a.ctl)) return;
    const u64 P = a.ctl[1];
    const int lane = threadIdx.x & 31;
    const u64 warps = (u64)gridDim.x * (blockDim.x >> 5);
    for (u64 p = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5; p < P; p += warps) {
        u32 g, rank;
        u64 o;
        mine_pattern(a, p, g, rank, o);
        const u64 m = a.seq_len[o];
        if (rank >= kMineMaxRank) {
            if (lane == 0) atomicMin(a.ctl, (unsigned long long)mine_fault_key(a.grp_file[g], rank, kMineRank));
            continue;
        }
        if (m > kMineMaxPattern) {
            if (lane == 0) atomicMin(a.ctl, (unsigned long long)mine_fault_key(a.grp_file[g], rank, kMineLong));
            continue;
        }
        u32 mask[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        mine_byte_set(a.data + a.seq_beg[o], lane, m, 32, mask);
        for (int k = 0; k < 8; ++k) mask[k] = __reduce_or_sync(0xffffffffu, mask[k]);
        if (lane) continue;
        if (mine_popc8(mask) > kMineMaxCodes) {
            atomicMin(a.ctl, (unsigned long long)mine_fault_key(a.grp_file[g], rank, kMineCodes));
            continue;
        }
        int cls;
        const u64 n = mine_items(m, a.ent_base[g + 1] - a.ent_base[g], cls);
        if (n) atomicAdd(&a.ctl[3 + cls], (unsigned long long)n);
    }
}

// One thread per pattern: its work items at the class cursor (ctl[3 + kHwClasses + c], set to the class's first item).
__global__ void __launch_bounds__(kMineThreads) k_mine_scatter(MineArgs a, u64 P) {
    for (u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += (u64)gridDim.x * blockDim.x) {
        u32 g, rank;
        u64 o;
        mine_pattern(a, p, g, rank, o);
        const u64 m = a.seq_len[o], e0 = a.ent_base[g], ne = a.ent_base[g + 1] - e0;
        int cls;
        const u64 n = mine_items(m, ne, cls);
        if (!n) continue;
        int sw, w;
        hw_best_class((int)((m + 31) / 32), &sw, &w);
        const u64 chunk = hw_best_chunk(sw);
        const u64 at = atomicAdd(&a.ctl[3 + kHwClasses + cls], (unsigned long long)n);
        for (u64 i = 0; i < n; ++i) {
            const u64 lo = i * chunk;
            a.items[at + i] = HwItem{(u32)o, rank, e0 + lo, (u32)(ne - lo < chunk ? ne - lo : chunk), 0u};
        }
    }
}

// One block per group: the text (output) of each of its entries, its partial files' outputs in order.
__global__ void __launch_bounds__(kMineThreads) k_mine_entries(MineArgs a) {
    const u32 g = blockIdx.x;
    u64 at = a.ent_base[g];
    for (u32 k = a.grp_part_off[g]; k < a.grp_part_off[g + 1]; ++k) {
        const u32 p = a.grp_part[k];
        const u64 o0 = a.file_rng[2 * p], n = a.file_rng[2 * p + 1] - o0;
        for (u64 i = threadIdx.x; i < n; i += blockDim.x) a.ent_txt[at + i] = (u32)(o0 + i);
        at += n;
    }
}

// One thread per entry: the decision on its best full read and the size of its mined record (0: not mined).
__global__ void __launch_bounds__(kMineThreads) k_mine_decide(MineArgs a, u64 E) {
    for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (u64)gridDim.x * blockDim.x) {
        const u32 g = mine_group_of(a.ent_base, a.n_groups, e);
        u64 w, d;
        const u64 n = mine_decide_item(a.data, a.out_off, a.seq_beg, a.seq_len, a.ent_txt[e], a.file_rng[2 * a.grp_file[g]],
                                       a.keys[e], a.min_identity, a.grp_kind[g] != 0, w, d);
        a.size[e] = n;
        a.flag[e] = n ? 1 : 0;
        a.winner[e] = w;
        a.dist[e] = (u32)d;
        if (e == 0) { a.size[E] = 0; a.flag[E] = 0; }
    }
}

// One thread per entry: mined entries into the record arrays (stable: group, then entry order); one per .mined file:
// its first byte.
__global__ void __launch_bounds__(kMineThreads) k_mine_compact(MineArgs a, u64 E, MineOut out) {
    for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (u64)gridDim.x * blockDim.x) {
        if (!a.flag[e]) continue;
        const u64 j = a.flag_off[e];
        const u32 g = mine_group_of(a.ent_base, a.n_groups, e);
        out.partial[j] = a.ent_txt[e];
        out.winner[j] = a.winner[e];
        out.dist[j] = (i32)a.dist[e];
        a.rec_off[j] = a.size_off[e];
        a.rec_kind[j] = (unsigned char)(a.grp_kind[g] != 0);
    }
    for (u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x; j <= a.n_mined; j += (u64)gridDim.x * blockDim.x)
        out.mined_off[j] = a.size_off[a.ent_base[a.mined_grp[j]]];
}

// One warp per mined record: the rewritten title line (each lane a 16-byte window of it), then the partial record's
// sequence, separator, qualities and newline, as aligned 16-byte stores.
__global__ void __launch_bounds__(kMineThreads) k_mine_format(MineArgs a, u64 R, MineOut out) {
    const int lane = threadIdx.x & 31;
    const u64 warps = (u64)gridDim.x * (blockDim.x >> 5);
    for (u64 j = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < R; j += warps) {
        const u64 o = (u64)out.partial[j], w = (u64)out.winner[j];
        double ident;
        mine_pass((u64)out.dist[j], a.seq_len[w], a.min_identity, ident);
        char b[16];
        const u32 bl = smx_out::out_fmt2(ident, b);
        const smx_out::OutMined h = mine_title(a.data, a.out_off, o, a.seq_beg[o], a.rec_kind[j] != 0, b, bl);
        const u64 H = smx_out::out_mined_len(h);
        unsigned char *dst = out.bytes + a.rec_off[j];
        for (u64 lo = (u64)lane * 16; lo < H; lo += 32 * 16) {
            smx_out::OutWindow win = {0, lo, lo + 16 < H ? lo + 16 : H, dst + lo};
            smx_out::out_mined_emit(h, win);
        }
        const unsigned char *src = a.data + a.seq_beg[o];
        unsigned char *body = dst + H;
        const u64 L = a.out_off[o + 1] - a.seq_beg[o];
        u64 head = (16 - ((uintptr_t)body & 15)) & 15;
        if (head > L) head = L;
        const u64 chunks = (L - head) / 16;
        for (u64 i = lane; i < head; i += 32) body[i] = src[i];
        for (u64 c = lane; c < chunks; c += 32) {
            u32 v[4];
            smx_out::demux_load16(src + head + 16 * c, v);
            smx_out::demux_store16(body + head + 16 * c, v);
        }
        for (u64 i = head + 16 * chunks + lane; i < L; i += 32) body[i] = src[i];
    }
}

cudaError_t launch_mine_locate(const MineArgs &a, cudaStream_t st) {
    if (a.n_involved) k_mine_locate<<<a.n_involved, kMineThreads, 0, st>>>(a);
    if (a.n_groups) k_mine_groups<<<1, kMineScanThreads, 0, st>>>(a);
    if (a.n_groups) k_mine_plan<<<1024, kMineThreads, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_mine_items(const MineArgs &a, u64 P, u64 E, cudaStream_t st) {
    if (P) k_mine_scatter<<<mine_blocks(P), kMineThreads, 0, st>>>(a, P);
    if (E) k_mine_entries<<<a.n_groups, kMineThreads, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t mine_scan_temp_bytes(u64 n, size_t *bytes) {
    return cub::DeviceScan::ExclusiveSum(nullptr, *bytes, (const u64 *)nullptr, (u64 *)nullptr, (int64_t)n);
}

cudaError_t launch_mine_decide(const MineArgs &a, u64 E, cudaStream_t st) {
    if (!E) return cudaSuccess;
    k_mine_decide<<<mine_blocks(E), kMineThreads, 0, st>>>(a, E);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    size_t temp = a.temp_bytes;
    if ((e = cub::DeviceScan::ExclusiveSum(a.temp, temp, a.size, a.size_off, (int64_t)E + 1, st)) != cudaSuccess) return e;
    temp = a.temp_bytes;
    return cub::DeviceScan::ExclusiveSum(a.temp, temp, a.flag, a.flag_off, (int64_t)E + 1, st);
}

cudaError_t launch_mine_format(const MineArgs &a, u64 E, u64 R, const MineOut &out, cudaStream_t st) {
    k_mine_compact<<<mine_blocks(E > a.n_mined + 1 ? E : a.n_mined + 1), kMineThreads, 0, st>>>(a, E, out);
    if (R) k_mine_format<<<mine_blocks(32 * R), kMineThreads, 0, st>>>(a, R, out);
    return cudaGetLastError();
}

}  // namespace smx
