// smx_k_mine.cu -- all-pairs HW (infix) edit distances of long patterns in long texts: the arithmetic of specimine
// (reference specimine.py:226-241: edlib.align(full_seq, partial_seq, mode="HW", task="path", k=max_distance), of
// whose result only editDistance is read, :243-248).  Plain byte equality (edlib's default alphabet, no
// additionalEqualities, case-sensitive).
//
// Warp-cooperative multi-word Myers/Hyyro, the same scheme as k_primer_long: the pattern occupies the top m bits of a
// 32*SW*W-bit column vector spread over SW consecutive lanes with W words each; per column the carry of
// (Eq & Pv) + Pv ripples inside a lane and crosses lanes through two ballots and one integer addition
// (long_carry_in<SW>), the one-bit shifts of Ph / Mh cross lanes by __shfl_up.  One block per pattern: its Peq
// table (one row per distinct byte of the pattern) is built once in shared memory, the block's warps then walk the
// texts, 32 / SW texts per warp at a time.
//
// k_hw_best is the grouped form for many specimens in one launch (smx_hw_best_grouped): a block is one pattern and a
// run of its group's text list, and only the best pattern of every text is kept (a 64-bit key per text entry, reduced
// by atomicMin), so no distance matrix is stored.  Its segments need not be a power of two wide (hw_best_class).  Both
// kernels share the Peq build (build_peq) and the column step (hw_column).  k_hw_best finds the bytes of its patterns
// and texts through an accessor (HwContig: contiguous offsets, smx_hw_best_grouped; HwSpans: begin / length per output
// of a device file buffer, smx_mine_device), so both callers run the same kernel.
#include <cuda_runtime.h>

#include "smx_device.cuh"
#include "smx_launch.hpp"

namespace smx {

constexpr int kMineCodes = 64;          // distinct byte values a pattern may hold (reads: a handful)

// Peq of the block's pattern in shared memory: row c has the bits of the pattern rows holding the byte of code c, the
// pattern in the top m bits of the 32*NW-bit column vector; row kMineCodes stays zero (bytes the pattern does not
// hold).  Returns false (uniformly over the block) when the pattern holds more than kMineCodes distinct bytes.
template <int NW>
__device__ __forceinline__ bool build_peq(const unsigned char *P, int m, u32 *s_peq, unsigned char *s_code, int &s_ncodes) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_code[i] = 0xFF;
    for (int i = threadIdx.x; i < (kMineCodes + 1) * NW; i += blockDim.x) s_peq[i] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < m; i += blockDim.x) s_code[P[i]] = 0xFE;          // present
    __syncthreads();
    if (threadIdx.x == 0) {
        int n = 0;
        for (int c = 0; c < 256; ++c)
            if (s_code[c] == 0xFE) s_code[c] = (unsigned char)(n < kMineCodes ? n : kMineCodes), ++n;
            else s_code[c] = (unsigned char)kMineCodes;
        s_ncodes = n;
    }
    __syncthreads();
    if (s_ncodes > kMineCodes) return false;                    // never for nucleotide reads; reported, not computed
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
        const int pos = 32 * NW - m + i;                        // row i at bit pos: row m is the top bit
        atomicOr(&s_peq[s_code[P[i]] * NW + (pos >> 5)], 1u << (pos & 31));
    }
    __syncthreads();
    return true;
}

// One DP column for every segment of the warp (must be called by all 32 lanes): lane `sub` of a segment holds words
// [sub * W, sub * W + W) of the column vector, eqrow points at the column's Peq row plus sub * W.  Pv / Mv advance
// where `active`; returns the score delta of the last row (meaningful in a segment's top lane).
template <int SW, int W>
__device__ __forceinline__ int hw_column(const u32 *eqrow, u32 (&Pv)[W], u32 (&Mv)[W], bool active, int sub, int lane) {
    u32 eq[W], sum[W];
    u32 carry = 0, allones = 1;
#pragma unroll
    for (int w = 0; w < W; ++w) {
        eq[w] = eqrow[w];
        const u32 a = eq[w] & Pv[w];
        const u32 s = a + Pv[w];
        const u32 s2 = s + carry;
        carry = (u32)(s < a) | (u32)(s2 < s);
        sum[w] = s2;
        allones &= (u32)(s2 == 0xFFFFFFFFu);
    }
    const u32 G = __ballot_sync(0xffffffffu, carry != 0);
    const u32 Pm = __ballot_sync(0xffffffffu, allones != 0);
    u32 cin = (long_carry_in<SW>(G, Pm) >> lane) & 1u;
    u32 Ph[W], Mh[W], Xv[W];
#pragma unroll
    for (int w = 0; w < W; ++w) {
        const u32 s = sum[w] + cin;
        cin = (u32)(s < sum[w]);
        const u32 Xh = (s ^ Pv[w]) | eq[w];
        Xv[w] = eq[w] | Mv[w];
        Ph[w] = Mv[w] | ~(Xh | Pv[w]);
        Mh[w] = Pv[w] & Xh;
    }
    const int d = (int)(Ph[W - 1] >> 31) - (int)(Mh[W - 1] >> 31);
    u32 Ph_in = __shfl_up_sync(0xffffffffu, Ph[W - 1], 1), Mh_in = __shfl_up_sync(0xffffffffu, Mh[W - 1], 1);
    if (sub == 0) { Ph_in = 0u; Mh_in = 0u; }                                  // HW: D[0][j] = 0
    u32 nPv[W], nMv[W];
#pragma unroll
    for (int w = 0; w < W; ++w) {
        const u32 plo = w ? Ph[w - 1] : Ph_in, mlo = w ? Mh[w - 1] : Mh_in;
        const u32 ph = __funnelshift_l(plo, Ph[w], 1), mh = __funnelshift_l(mlo, Mh[w], 1);
        nPv[w] = mh | ~(Xv[w] | ph);
        nMv[w] = ph & Xv[w];
    }
    if (active) {
#pragma unroll
        for (int w = 0; w < W; ++w) { Pv[w] = nPv[w]; Mv[w] = nMv[w]; }
    }
    return d;
}

template <int SW, int W>
__global__ void __launch_bounds__(128) k_hw_distance(const unsigned char *pat, const u64 *pat_off, const i32 *pat_k,
                                                     const u32 *pat_list, const unsigned char *txt, const u64 *txt_off,
                                                     u32 n_txt, i32 *out, u32 *bad) {
    constexpr int NW = SW * W;                                  // words of the column vector
    __shared__ u32 s_peq[(kMineCodes + 1) * NW];
    __shared__ unsigned char s_code[256];
    __shared__ int s_ncodes;
    const u32 pi = pat_list[blockIdx.y];
    const unsigned char *P = pat + pat_off[pi];
    const int m = (int)(pat_off[pi + 1] - pat_off[pi]);
    if (!build_peq<NW>(P, m, s_peq, s_code, s_ncodes)) {
        if (threadIdx.x == 0 && blockIdx.x == 0) atomicAdd(bad, 1u);
        return;
    }
    const int lane = threadIdx.x & 31, sub = lane % SW, warp = threadIdx.x >> 5;
    const bool top = sub == SW - 1;
    const int k = pat_k[pi];
    constexpr int per_warp = 32 / SW;
    const u32 warps = gridDim.x * (blockDim.x >> 5);
    for (u32 t0 = (blockIdx.x * (blockDim.x >> 5) + warp) * per_warp; t0 < n_txt; t0 += warps * per_warp) {
        const u32 ti = t0 + lane / SW;
        const bool valid = ti < n_txt;
        const unsigned char *T = txt + (valid ? txt_off[ti] : 0);
        const int n = valid ? (int)(txt_off[ti + 1] - txt_off[ti]) : 0;
        const int maxn = __reduce_max_sync(0xffffffffu, n);
        u32 Pv[W], Mv[W];
#pragma unroll
        for (int w = 0; w < W; ++w) { Pv[w] = ~0u; Mv[w] = 0u; }
        int score = m, best = m;
        for (int j = 0; j < maxn; ++j) {
            const bool active = j < n;
            const int d = hw_column<SW, W>(s_peq + (active ? s_code[T[j]] : kMineCodes) * NW + sub * W, Pv, Mv, active, sub, lane);
            if (active) {
                score += d;
                best = score < best ? score : best;
            }
        }
        if (valid && top) out[(u64)pi * n_txt + ti] = (k >= 0 && best > k) ? -1 : best;
    }
}

// Grouped best match (smx_hw_best_grouped): one block per work item = (pattern, run of consecutive entries of its
// group's text list); 32 / SW whole segments per warp (lanes beyond them idle, LongSeg<SW>), the four warps take turns
// along the run.  Every (pattern, text) result goes straight into the entry's key,
// (floor(d * 2^40 / m) << 23) | rank of the pattern in its group, by atomicMin: the least key is the least d / m, ties
// to the first pattern, whatever order the blocks run in.  Distances above k leave the key alone; an empty text counts
// d = m whatever k (edlib's empty-sequence rule, as smx_hw_distances).
template <int SW, int W, class Seqs>
__global__ void __launch_bounds__(128) k_hw_best(Seqs pats, const i32 *pat_k, const HwItem *items, Seqs txts,
                                                 const u32 *ent_txt, unsigned long long *keys, u32 *bad) {
    constexpr int NW = SW * W;
    constexpr int kTexts = LongSeg<SW>::kReads;                 // texts (whole segments) per warp
    __shared__ u32 s_peq[(kMineCodes + 1) * NW];
    __shared__ unsigned char s_code[256];
    __shared__ int s_ncodes;
    const HwItem it = items[blockIdx.x];
    const unsigned char *P = pats.bytes + pats.start(it.pat);
    const int m = pats.len(it.pat);
    if (!build_peq<NW>(P, m, s_peq, s_code, s_ncodes)) {
        if (threadIdx.x == 0) atomicAdd(bad, 1u);
        return;
    }
    const int lane = threadIdx.x & 31, sub = lane % SW, warp = threadIdx.x >> 5;
    const bool top = sub == SW - 1, in_seg = lane < kTexts * SW;
    const int k = pat_k[it.pat];
    for (u32 e0 = (u32)warp * kTexts; e0 < it.n; e0 += (blockDim.x >> 5) * kTexts) {
        const u32 e = e0 + (u32)(lane / SW);
        const bool valid = in_seg && e < it.n;
        const u64 ent = it.e_lo + (valid ? e : 0);
        const u32 ti = valid ? ent_txt[ent] : 0;
        const unsigned char *T = txts.bytes + (valid ? txts.start(ti) : 0);
        const int n = valid ? txts.len(ti) : 0;
        const int maxn = __reduce_max_sync(0xffffffffu, n);
        u32 Pv[W], Mv[W];
#pragma unroll
        for (int w = 0; w < W; ++w) { Pv[w] = ~0u; Mv[w] = 0u; }
        int score = m, best = m;
        for (int j = 0; j < maxn; ++j) {
            const bool active = j < n;
            const int d = hw_column<SW, W>(s_peq + (active ? s_code[T[j]] : kMineCodes) * NW + sub * W, Pv, Mv, active, sub, lane);
            if (active) {
                score += d;
                best = score < best ? score : best;
            }
        }
        if (valid && top && (n == 0 || k < 0 || best <= k)) {
            const unsigned long long q = ((unsigned long long)best << 40) / (unsigned long long)m;
            atomicMin(&keys[ent], (q << 23) | it.rank);
        }
    }
}

cudaError_t launch_hw_distance(int sw, int w, const unsigned char *pat, const u64 *pat_off, const i32 *pat_k, const u32 *pat_list,
                               u32 n_list, const unsigned char *txt, const u64 *txt_off, u32 n_txt, i32 *out, u32 *bad,
                               cudaStream_t st) {
    if (!n_list || !n_txt) return cudaSuccess;
    const int per_block = 4 * (32 / sw);                        // texts one block covers per pass
    unsigned gx = (n_txt + per_block - 1) / per_block;
    if (gx > 64) gx = 64;                                       // the Peq build is per block: a block walks several texts
    dim3 grid(gx, n_list);
#define SMX_HW(SS, WW) k_hw_distance<SS, WW><<<grid, 128, 0, st>>>(pat, pat_off, pat_k, pat_list, txt, txt_off, n_txt, out, bad)
    if (w == 1) {
        switch (sw) {
            case 4: SMX_HW(4, 1); break;
            case 8: SMX_HW(8, 1); break;
            case 16: SMX_HW(16, 1); break;
            default: SMX_HW(32, 1); break;
        }
    } else if (w == 2) SMX_HW(32, 2);
    else SMX_HW(32, 4);
#undef SMX_HW
    return cudaGetLastError();
}


template <class Seqs>
cudaError_t launch_hw_best(int sw, int w, Seqs pats, const i32 *pat_k, const HwItem *items, u32 n_items, Seqs txts,
                           const u32 *ent_txt, unsigned long long *keys, u32 *bad, cudaStream_t st) {
    if (!n_items) return cudaSuccess;
#define SMX_HB(SS, WW) case SS * 8 + WW: k_hw_best<SS, WW, Seqs><<<n_items, 128, 0, st>>>(pats, pat_k, items, txts, ent_txt, keys, bad); break;
    switch (sw * 8 + w) {
        SMX_HB(3, 1) SMX_HB(3, 2) SMX_HB(3, 3) SMX_HB(4, 1) SMX_HB(4, 2) SMX_HB(4, 3) SMX_HB(4, 4) SMX_HB(5, 2) SMX_HB(5, 4)
        SMX_HB(6, 3) SMX_HB(8, 3) SMX_HB(8, 4) SMX_HB(10, 4) SMX_HB(16, 3) SMX_HB(16, 4) SMX_HB(32, 3) SMX_HB(32, 4)
        default: return cudaErrorInvalidValue;
    }
#undef SMX_HB
    return cudaGetLastError();
}

template cudaError_t launch_hw_best<HwContig>(int, int, HwContig, const i32 *, const HwItem *, u32, HwContig, const u32 *,
                                              unsigned long long *, u32 *, cudaStream_t);
template cudaError_t launch_hw_best<HwSpans>(int, int, HwSpans, const i32 *, const HwItem *, u32, HwSpans, const u32 *,
                                             unsigned long long *, u32 *, cudaStream_t);

}  // namespace smx
