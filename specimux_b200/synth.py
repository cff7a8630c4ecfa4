"""Seeded synthetic datasets of the BASELINE.json shapes (SURVEY.md 8d).

Reads are laid out ``[tail 0-30][b1][fwd primer][insert][RC(rev primer)][RC(b2)][tail 0-30]``,
reverse-complemented with probability 0.5, then hit by per-base errors
(substitution : insertion : deletion = 4 : 3 : 3 of the stated total rate).  IUPAC primer
positions are instantiated uniformly from their base sets, qualities are uniform Q5-Q40,
2 % of reads are primer-less junk.  Everything is vectorised over the whole read set so the
full-size configs (765 k - 20 M reads) generate in seconds to minutes.

Bases are produced as uint8 codes A=0 C=1 G=2 T=3 in one flat array plus offsets; use
``SynthDataset.read_str`` / ``write_fastq`` for text.
"""
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import numpy as np

IUPAC_SETS = {"A": "A", "C": "C", "G": "G", "T": "T", "Y": "CT", "R": "AG", "N": "ACGT", "W": "AT",
              "M": "AC", "S": "CG", "K": "GT", "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG"}
_CODE = {"A": 0, "C": 1, "G": 2, "T": 3}
_BASES = np.frombuffer(b"ACGT", dtype=np.uint8)
_COMP = str.maketrans("ACGTMRWSYKVHDBN", "TGCAKYWSRMBDHVN")

ITS1F = "CTTGGTCATTTAGAGGAAGTAA"
ITS4 = "TCCTCCGCTTATTGATATGC"
GITS7 = "GTGARTCATCGARTCTTTG"
RPB2_5F = "GAYGAYMGWGATCAYTTYGG"
RPB2_7R = "CCCATRGCYTGYTTMCCCATDGC"
LR_REV = "TCCTGAGGGAAACTTCGGCA"


def revcomp(s: str) -> str:
    return s.translate(_COMP)[::-1]


def pairwise_levenshtein(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """Edit distance between every row of `a` (n, m) and every row of `b` (k, m'), vectorised DP."""
    n, m = a.shape
    k, mb = b.shape
    prev = np.broadcast_to(np.arange(mb + 1, dtype=np.int16), (n, k, mb + 1)).copy()
    for i in range(1, m + 1):
        cur = np.empty_like(prev)
        cur[:, :, 0] = i
        neq = (a[:, None, i - 1, None] != b[None, :, :]).astype(np.int16)     # (n, k, mb)
        best = np.minimum(prev[:, :, :-1] + neq, prev[:, :, 1:] + 1)
        for j in range(1, mb + 1):
            cur[:, :, j] = np.minimum(best[:, :, j - 1], cur[:, :, j - 1] + 1)
        prev = cur
    return prev[:, :, mb]


def make_barcodes(n_fwd: int, n_rev: int, length: int, min_dist: int, seed: int) -> Tuple[List[str], List[str]]:
    """Greedy seeded set with pairwise Levenshtein >= min_dist over {b1} U {RC(b2)} (orchestration.py:581)."""
    rng = np.random.default_rng(seed)
    total = n_fwd + n_rev
    acc = np.empty((0, length), dtype=np.uint8)
    while acc.shape[0] < total:
        cand = rng.integers(0, 4, size=(512, length), dtype=np.uint8)
        # no homopolymer runs >= 4, keeps barcodes realistic
        runs = (cand[:, 3:] == cand[:, 2:-1]) & (cand[:, 2:-1] == cand[:, 1:-2]) & (cand[:, 1:-2] == cand[:, :-3])
        cand = cand[~runs.any(axis=1)]
        if acc.shape[0]:
            cand = cand[(pairwise_levenshtein(cand, acc) >= min_dist).all(axis=1)]
        if not cand.shape[0]:
            continue
        dd = pairwise_levenshtein(cand, cand)
        keep: List[int] = []
        for i in range(cand.shape[0]):
            if all(dd[i, j] >= min_dist for j in keep):
                keep.append(i)
                if acc.shape[0] + len(keep) >= total:
                    break
        acc = np.concatenate([acc, cand[keep]], axis=0)
    strs = ["".join("ACGT"[c] for c in row) for row in acc[:total]]
    fwd = strs[:n_fwd]
    rev = [revcomp(s) for s in strs[n_fwd:]]        # the set was built over RC(b2)
    return fwd, rev


@dataclass
class SynthDataset:
    name: str
    primers: List[Tuple[str, str, str, List[str]]]                  # (name, seq, position, pools)
    specimens: List[Tuple[str, str, str, str, str, str]]            # (id, pool, b1, p1, b2, p2)
    codes: np.ndarray                                               # uint8 flat base codes 0..3
    offsets: np.ndarray                                             # int64, n+1
    quals: Optional[np.ndarray] = None                              # uint8 flat phred (same layout) or None
    truth: Dict[str, np.ndarray] = field(default_factory=dict)      # specimen index (-1 junk), orientation
    search_len: int = 80
    error_rate: float = 0.07

    @property
    def n_reads(self) -> int:
        return len(self.offsets) - 1

    @property
    def lengths(self) -> np.ndarray:
        return np.diff(self.offsets)

    def read_id(self, i: int) -> str:
        return "%s_%08d" % (self.name, i)

    def read_str(self, i: int) -> str:
        return _BASES[self.codes[self.offsets[i]:self.offsets[i + 1]]].tobytes().decode()

    def qual_str(self, i: int) -> str:
        if self.quals is None:
            return "I" * int(self.offsets[i + 1] - self.offsets[i])
        return (self.quals[self.offsets[i]:self.offsets[i + 1]] + 33).astype(np.uint8).tobytes().decode()

    def reads(self, lo: int = 0, hi: Optional[int] = None):
        hi = self.n_reads if hi is None else min(hi, self.n_reads)
        return [(self.read_id(i), self.read_str(i), self.qual_str(i)) for i in range(lo, hi)]

    def write_fastq(self, path: str, lo: int = 0, hi: Optional[int] = None) -> None:
        with open(path, "w") as fh:
            for rid, s, q in self.reads(lo, hi):
                fh.write("@%s\n%s\n+\n%s\n" % (rid, s, q))

    def write_tables(self, primers_path: str, specimens_path: str) -> None:
        with open(primers_path, "w") as fh:
            for name, seq, pos, pools in self.primers:
                fh.write(">%s pool=%s position=%s\n%s\n" % (name, ",".join(pools), pos, seq))
        with open(specimens_path, "w") as fh:
            fh.write("SampleID\tPrimerPool\tFwIndex\tFwPrimer\tRvIndex\tRvPrimer\n")
            for row in self.specimens:
                fh.write("\t".join(row) + "\n")


def _segments_to_flat(seg_codes: List[np.ndarray], seg_lens: List[np.ndarray]) -> Tuple[np.ndarray, np.ndarray]:
    """Interleave per-read segments (each given as its own flat array + per-read lengths) read by read."""
    n = len(seg_lens[0])
    lens = np.stack(seg_lens, axis=1).astype(np.int64)                # (n, S)
    total = lens.sum(axis=1)
    offs = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(total, out=offs[1:])
    out = np.empty(int(offs[-1]), dtype=np.uint8)
    seg_start = offs[:-1, None] + np.concatenate([np.zeros((n, 1), np.int64), np.cumsum(lens, axis=1)[:, :-1]], axis=1)
    for s, (codes, ln) in enumerate(zip(seg_codes, seg_lens)):
        ln = ln.astype(np.int64)
        src_off = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(ln, out=src_off[1:])
        # destination index of every element of this segment
        rep_start = np.repeat(seg_start[:, s] - src_off[:-1], ln)
        out[rep_start + np.arange(int(src_off[-1]), dtype=np.int64)] = codes
    return out, offs


def _instantiate(rng, seq: str, count: int) -> np.ndarray:
    """(count, len) concrete base codes for an IUPAC pattern."""
    out = np.empty((count, len(seq)), dtype=np.uint8)
    for j, ch in enumerate(seq):
        opts = np.array([_CODE[c] for c in IUPAC_SETS[ch]], dtype=np.uint8)
        out[:, j] = opts[0] if len(opts) == 1 else opts[rng.integers(0, len(opts), size=count)]
    return out


def _gather_rows(table: np.ndarray, idx: np.ndarray) -> np.ndarray:
    return table[idx].reshape(-1)


def _codes_of(strs: List[str]) -> np.ndarray:
    return np.array([[_CODE[c] for c in s] for s in strs], dtype=np.uint8)


def _apply_errors(rng, codes: np.ndarray, offs: np.ndarray, rate: float) -> Tuple[np.ndarray, np.ndarray]:
    n_bases = codes.shape[0]
    u = rng.random(n_bases, dtype=np.float32)
    sub = u < 0.4 * rate
    ins = (u >= 0.4 * rate) & (u < 0.7 * rate)
    dele = (u >= 0.7 * rate) & (u < rate)
    cnt = np.ones(n_bases, dtype=np.int8)
    cnt[ins] = 2
    cnt[dele] = 0
    new = codes.copy()
    nsub = int(sub.sum())
    new[sub] = (codes[sub] + rng.integers(1, 4, size=nsub, dtype=np.uint8)) & 3
    out = np.repeat(new, cnt)
    # the first copy of an `ins` position becomes a random inserted base
    first_pos = np.cumsum(cnt, dtype=np.int64) - cnt
    ins_pos = first_pos[ins]
    out[ins_pos] = rng.integers(0, 4, size=ins_pos.shape[0], dtype=np.uint8)
    csum = np.zeros(n_bases + 1, dtype=np.int64)
    np.cumsum(cnt, out=csum[1:])
    return out, csum[offs]


def _reverse_complement_reads(codes: np.ndarray, offs: np.ndarray, flip: np.ndarray) -> np.ndarray:
    lens = np.diff(offs)
    start = np.repeat(offs[:-1], lens)
    pos = np.arange(codes.shape[0], dtype=np.int64) - start
    ln = np.repeat(lens, lens)
    fl = np.repeat(flip, lens)
    src = np.where(fl, start + ln - 1 - pos, start + pos)
    out = codes[src]
    out[fl] ^= 3
    return out


_CHUNK = 8192


def _build(name, primers, specimens, spec_struct, n_reads, seed, insert_sampler, error_rate, search_len,
           with_quals=True, junk_frac=0.02) -> SynthDataset:
    """Generate in fixed-size chunks (each with its own spawned seed) so any prefix of a dataset is
    identical regardless of the total size requested, and the working set stays cache-sized."""
    n_chunks = max(1, -(-n_reads // _CHUNK))
    seeds = np.random.SeedSequence(seed).spawn(n_chunks)
    parts = []
    for ci in range(n_chunks):
        parts.append(_build_chunk(spec_struct, _CHUNK, np.random.default_rng(seeds[ci]), insert_sampler,
                                  error_rate, with_quals, junk_frac))
    lens = np.concatenate([np.diff(p[1]) for p in parts])[:n_reads]
    n_bases = int(lens.sum())
    codes = np.concatenate([p[0] for p in parts])[:n_bases]
    offs = np.zeros(n_reads + 1, dtype=np.int64)
    np.cumsum(lens, out=offs[1:])
    quals = np.concatenate([p[2] for p in parts])[:n_bases] if with_quals else None
    truth = {"specimen": np.concatenate([p[3] for p in parts])[:n_reads],
             "flipped": np.concatenate([p[4] for p in parts])[:n_reads]}
    return SynthDataset(name, primers, specimens, codes, offs, quals, truth, search_len, error_rate)


def _build_chunk(spec_struct, n_reads, rng, insert_sampler, error_rate, with_quals, junk_frac):
    """spec_struct: per specimen (b1 str, fwd primer seq, rev primer seq, b2 str, weight)."""
    w = np.array([s[4] for s in spec_struct], dtype=np.float64)
    spec_idx = rng.choice(len(spec_struct), size=n_reads, p=w / w.sum())
    junk = rng.random(n_reads) < junk_frac
    flip = rng.random(n_reads) < 0.5
    tail1 = rng.integers(0, 31, size=n_reads)
    tail2 = rng.integers(0, 31, size=n_reads)
    insert = insert_sampler(rng, n_reads)

    b1_tab = _codes_of([s[0] for s in spec_struct])
    b2rc_tab = _codes_of([revcomp(s[3]) for s in spec_struct])
    blen = b1_tab.shape[1]
    fwd_seqs = sorted({s[1] for s in spec_struct})
    rev_seqs = sorted({s[2] for s in spec_struct})
    fwd_of = np.array([fwd_seqs.index(s[1]) for s in spec_struct])[spec_idx]
    rev_of = np.array([rev_seqs.index(s[2]) for s in spec_struct])[spec_idx]

    def primer_segment(seqs, which, rc):
        lens = np.array([len(x) for x in seqs])[which]
        flat = np.empty(int(lens.sum()), dtype=np.uint8)
        o = np.zeros(n_reads + 1, dtype=np.int64)
        np.cumsum(lens, out=o[1:])
        for pi, seq in enumerate(seqs):
            sel = np.nonzero(which == pi)[0]
            if not sel.size:
                continue
            inst = _instantiate(rng, revcomp(seq) if rc else seq, sel.size)
            dst = (o[sel][:, None] + np.arange(len(seq))[None, :]).reshape(-1)
            flat[dst] = inst.reshape(-1)
        return flat, lens

    fp_codes, fp_len = primer_segment(fwd_seqs, fwd_of, False)
    rp_codes, rp_len = primer_segment(rev_seqs, rev_of, True)
    zero = np.zeros(n_reads, dtype=np.int64)
    blen_arr = np.where(junk, 0, blen)
    # junk reads: only random sequence (tails + insert), no barcodes or primers
    keep = ~junk
    fp_codes = fp_codes[np.repeat(keep, fp_len)]
    rp_codes = rp_codes[np.repeat(keep, rp_len)]
    fp_len = np.where(junk, zero, fp_len)
    rp_len = np.where(junk, zero, rp_len)
    segs = [
        (rng.integers(0, 4, size=int(tail1.sum()), dtype=np.uint8), tail1),
        (_gather_rows(b1_tab, spec_idx[keep]), blen_arr),
        (fp_codes, fp_len),
        (rng.integers(0, 4, size=int(insert.sum()), dtype=np.uint8), insert),
        (rp_codes, rp_len),
        (_gather_rows(b2rc_tab, spec_idx[keep]), blen_arr),
        (rng.integers(0, 4, size=int(tail2.sum()), dtype=np.uint8), tail2),
    ]
    codes, offs = _segments_to_flat([s[0] for s in segs], [s[1] for s in segs])
    codes = _reverse_complement_reads(codes, offs, flip)
    codes, offs = _apply_errors(rng, codes, offs, error_rate)
    quals = rng.integers(5, 41, size=codes.shape[0], dtype=np.uint8) if with_quals else None
    return codes, offs, quals, np.where(junk, -1, spec_idx).astype(np.int32), flip


def _normal_insert(mean, sd, lo):
    return lambda rng, n: np.maximum(lo, rng.normal(mean, sd, size=n)).astype(np.int64)


def _uniform_insert(lo, hi):
    return lambda rng, n: rng.integers(lo, hi + 1, size=n).astype(np.int64)


def _grid_specimens(prefix, pool, fwd_bcs, rev_bcs, p1name, p2name, p1seq, p2seq, weight=1.0):
    rows, struct = [], []
    for i, b1 in enumerate(fwd_bcs):
        for j, b2 in enumerate(rev_bcs):
            rows.append(("%s_P%02d_W%02d" % (prefix, i + 1, j + 1), pool, b1, p1name, b2, p2name))
            struct.append((b1, p1seq, p2seq, b2, weight))
    return rows, struct


def ont037(n_reads=765_000, seed=37, with_quals=True) -> SynthDataset:
    """BASELINE config 2: 768 specimens (8 x 96), single ITS pool, ~700 bp, 7 % errors."""
    fb, rb = make_barcodes(8, 96, 13, 6, seed)
    primers = [("ITS1F", ITS1F, "forward", ["ITS"]), ("ITS4", ITS4, "reverse", ["ITS"])]
    rows, struct = _grid_specimens("ONT037", "ITS", fb, rb, "ITS1F", "ITS4", ITS1F, ITS4)
    return _build("ont037", primers, rows, struct, n_reads, seed, _normal_insert(640, 60, 50), 0.07, 80, with_quals)


def multipool(n_reads=5_000_000, seed=3, with_quals=True) -> SynthDataset:
    """BASELINE config 3: ITS + RPB2 (IUPAC-degenerate) + a Mixed pool sharing ITS primers, wildcards."""
    fb, rb = make_barcodes(16, 96, 13, 6, seed)
    primers = [("ITS1F", ITS1F, "forward", ["ITS", "Mixed"]), ("ITS4", ITS4, "reverse", ["ITS", "Mixed"]),
               ("gITS7", GITS7, "forward", ["Mixed"]),
               ("fRPB2-5F", RPB2_5F, "forward", ["RPB2"]), ("RPB2-7.1R", RPB2_7R, "reverse", ["RPB2"])]
    r1, s1 = _grid_specimens("ITS", "ITS", fb[:8], rb, "ITS1F", "ITS4", ITS1F, ITS4, 0.5)
    r2, s2 = _grid_specimens("RPB2", "RPB2", fb[:8], rb, "fRPB2-5F", "RPB2-7.1R", RPB2_5F, RPB2_7R, 0.4)
    # Mixed pool: wildcard forward primer (ITS1F or gITS7), distinct forward barcodes
    r3, s3 = _grid_specimens("MIX", "Mixed", fb[8:], rb, "*", "ITS4", ITS1F, ITS4, 0.05)
    s3b = [(b1, GITS7, p2, b2, 0.05) for (b1, _p1, p2, b2, _w) in s3]
    rows = r1 + r2 + r3
    struct = s1 + s2 + s3
    # reads drawn from the gITS7 flavour of the Mixed specimens reuse the same specimen rows
    ds_struct = struct + s3b
    ds = _build("multipool", primers, rows, ds_struct, n_reads, seed,
                lambda rng, n: np.maximum(50, rng.normal(800, 250, size=n)).astype(np.int64), 0.07, 80, with_quals)
    sp = ds.truth["specimen"]
    ds.truth["specimen"] = np.where(sp >= len(struct), sp - len(s3), sp).astype(np.int32)
    return ds


def long_amplicon(n_reads=20_000_000, seed=4, search_len=200, with_quals=True) -> SynthDataset:
    """BASELINE config 4: 2-4 kb amplicons, widened search windows (-l 200 / -l 500)."""
    fb, rb = make_barcodes(8, 96, 13, 6, seed)
    primers = [("ITS1F", ITS1F, "forward", ["LSU"]), ("LRx", LR_REV, "reverse", ["LSU"])]
    rows, struct = _grid_specimens("LONG", "LSU", fb, rb, "ITS1F", "LRx", ITS1F, LR_REV)
    return _build("long", primers, rows, struct, n_reads, seed, _uniform_insert(2000, 4000), 0.07, search_len,
                  with_quals)


def dense_grid(n_reads=2_000_000, seed=5, with_quals=True) -> SynthDataset:
    """BASELINE config 5: 96 x 96 dual-index grid (9,216 specimens), 12 % errors, min barcode distance 5."""
    fb, rb = make_barcodes(96, 96, 13, 5, seed)
    primers = [("ITS1F", ITS1F, "forward", ["ITS"]), ("ITS4", ITS4, "reverse", ["ITS"])]
    rows, struct = _grid_specimens("GRID", "ITS", fb, rb, "ITS1F", "ITS4", ITS1F, ITS4)
    return _build("dense", primers, rows, struct, n_reads, seed, _normal_insert(640, 60, 50), 0.12, 80, with_quals)


def tie_storm(n_reads=40_000, seed=11, with_quals=True) -> SynthDataset:
    """Stress case of the parity tests (not a BASELINE config): a 96 x 96 grid whose barcodes are 1-2
    substitutions away from six seed 13-mers, to be searched with a forced k_idx = 3.  Every flank is then
    within k of a dozen or more barcodes: hit sub-lists overflow, equal-best ties map to many specimens
    (dereplication groups beyond the thread-local storage, many records per read)."""
    rng = np.random.default_rng(seed)

    def family(count):
        out, seen = [], set()
        seeds = rng.integers(0, 4, size=(6, 13), dtype=np.uint8)
        while len(out) < count:
            v = seeds[len(out) % 6].copy()
            for pos in rng.choice(13, size=int(rng.integers(1, 3)), replace=False):
                v[pos] = (v[pos] + rng.integers(1, 4)) & 3
            sv = "".join("ACGT"[c] for c in v)
            if sv not in seen:
                seen.add(sv)
                out.append(sv)
        return out
    fb, rb = family(96), family(96)
    primers = [("ITS1F", ITS1F, "forward", ["ITS"]), ("ITS4", ITS4, "reverse", ["ITS"])]
    rows, struct = _grid_specimens("TIE", "ITS", fb, rb, "ITS1F", "ITS4", ITS1F, ITS4)
    return _build("tiestorm", primers, rows, struct, n_reads, seed, _normal_insert(640, 60, 50), 0.05, 80, with_quals)


CONFIGS = {"tiestorm": tie_storm, "ont037": ont037, "multipool": multipool, "long": long_amplicon, "dense": dense_grid}


def mining_reads(n_fwd: int = 8, n_rev: int = 96, n_full: int = 16, n_partial: int = 4, n_other: int = 32,
                 amplicon: int = 640, error_rate: float = 0.03, seed: int = 41, pool: str = "ITS") -> SynthDataset:
    """Reads for specimine after demultiplexing, in the shape of specimine_tree: n_fwd x n_rev specimens (ITS1F / ITS4,
    the config-2 plate at 8 x 96), each with one amplicon of about `amplicon` nt of its own.  Every specimen gives n_full
    reads with both barcodes (full matches) and n_partial reads of each partial kind, whose forward or reverse barcode is
    replaced by random bases, so they go to barcode_rev_<b2> / barcode_fwd_<b1>; every barcode also gets n_other
    unrelated reads (a random insert) with only that barcode.  Only the inserts carry `error_rate` substitutions /
    insertions / deletions, so full and partial reads of a specimen are about 2 * error_rate apart and mining finds them;
    half the reads are reverse-complemented.  truth["specimen"] is the specimen (-1 for unrelated reads) and
    truth["kind"] 0 full, 1 partial reverse (b1 destroyed), 2 partial forward (b2 destroyed)."""
    rng = np.random.default_rng(seed)
    fb, rb = make_barcodes(n_fwd, n_rev, 13, 6, seed)
    primers = [("ITS1F", ITS1F, "forward", [pool]), ("ITS4", ITS4, "reverse", [pool])]
    rows, struct = _grid_specimens("MINE", pool, fb, rb, "ITS1F", "ITS4", ITS1F, ITS4)

    def rnd(n):
        return _BASES[rng.integers(0, 4, size=n)].tobytes().decode()

    def mutate(s):
        u = rng.random(len(s))
        out = []
        for ch, x in zip(s, u):
            if x < error_rate / 3:
                out.append("ACGT"[rng.integers(0, 4)])
            elif x < 2 * error_rate / 3:
                out.append(ch + "ACGT"[rng.integers(0, 4)])
            elif x >= error_rate:
                out.append(ch)
        return "".join(out)

    def primer(seq):
        return "".join(IUPAC_SETS[c][rng.integers(0, len(IUPAC_SETS[c]))] for c in seq)

    def read(b1, insert, b2):
        s = rnd(int(rng.integers(0, 31))) + b1 + primer(ITS1F) + insert + primer(revcomp(ITS4)) + revcomp(b2) + rnd(int(rng.integers(0, 31)))
        return revcomp(s) if rng.random() < 0.5 else s

    amp = [rnd(int(amplicon + rng.integers(-amplicon // 20, amplicon // 20 + 1))) for _ in struct]
    reads, spec, kind = [], [], []
    for i, (b1, _p1, _p2, b2, _w) in enumerate(struct):
        for k, n in ((0, n_full), (1, n_partial), (2, n_partial)):
            for _ in range(n):
                reads.append(read(rnd(len(b1)) if k == 1 else b1, mutate(amp[i]), rnd(len(b2)) if k == 2 else b2))
                spec.append(i)
                kind.append(k)
    for k, bcs in ((1, rb), (2, fb)):
        for bc in bcs:
            for _ in range(n_other):
                insert = rnd(int(amplicon + rng.integers(-amplicon // 20, amplicon // 20 + 1)))
                reads.append(read(rnd(13), insert, bc) if k == 1 else read(bc, insert, rnd(13)))
                spec.append(-1)
                kind.append(k)
    order = rng.permutation(len(reads))
    reads = [reads[o] for o in order]
    offs = np.zeros(len(reads) + 1, dtype=np.int64)
    np.cumsum([len(r) for r in reads], out=offs[1:])
    codes = np.frombuffer("".join(reads).translate(str.maketrans("ACGT", "\x00\x01\x02\x03")).encode("latin-1"),
                          dtype=np.uint8).copy()
    quals = rng.integers(5, 41, size=codes.shape[0], dtype=np.uint8)
    truth = {"specimen": np.array(spec, dtype=np.int32)[order], "kind": np.array(kind, dtype=np.int8)[order]}
    return SynthDataset("mining", primers, rows, codes, offs, quals, truth, 80, error_rate)


def specimine_tree(root: str, n_fwd: int = 8, n_rev: int = 96, n_full: int = 8, n_partial: int = 4, n_other: int = 16,
                   amplicon: int = 700, error_rate: float = 0.07, seed: int = 8, pool: str = "ITS",
                   pair: str = "ITS1F-ITS4") -> List[str]:
    """A demultiplexed output tree for specimine, written under `root`: n_fwd x n_rev specimens (the config-2 plate is
    8 x 96), each with its own random amplicon of about `amplicon` nt.  full/<pool>/<specimen>.fastq holds n_full reads
    of the specimen's amplicon; partial/<pool>/<pair>/barcode_rev_<b2>.fastq and barcode_fwd_<b1>.fastq hold n_partial
    reads of every specimen with that barcode, mixed with n_other unrelated reads.  Every read carries `error_rate`
    substitutions / insertions / deletions, so full and partial reads of one specimen are about 2 * error_rate apart
    and mining finds hits at the default identity.  Also writes index.txt.  Returns the full-match paths in plate
    order."""
    import os
    rng = np.random.default_rng(seed)
    b1s, b2s = make_barcodes(n_fwd, n_rev, 13, 3, seed)

    def rnd(n):
        return _BASES[rng.integers(0, 4, size=n)].tobytes().decode()

    def mutate(s):
        out = []
        for ch, u in zip(s, rng.random(len(s))):
            if u < error_rate / 3:
                out.append("ACGT"[rng.integers(0, 4)])
            elif u < 2 * error_rate / 3:
                out.append(ch + "ACGT"[rng.integers(0, 4)])
            elif u >= error_rate:
                out.append(ch)
        return "".join(out)

    def write(path, reads):
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "w") as fh:
            for rid, seq in reads:
                fh.write("@%s %s\n%s\n+\n%s\n" % (rid, "sp=" + rid.rsplit("_", 1)[0], seq, "I" * len(seq)))

    names = [[f"SP{i:02d}-{j:03d}" for j in range(n_rev)] for i in range(n_fwd)]
    amp = [[rnd(int(amplicon + rng.integers(-amplicon // 20, amplicon // 20 + 1))) for _ in range(n_rev)] for _ in range(n_fwd)]
    with open(os.path.join(root, "index.txt"), "w") as fh:
        fh.write("SampleID\tPrimerPool\tFwIndex\tFwPrimer\tRvIndex\tRvPrimer\n")
        for i in range(n_fwd):
            for j in range(n_rev):
                fh.write(f"{names[i][j]}\t{pool}\t{b1s[i]}\tITS1F\t{b2s[j]}\tITS4\n")
    paths = []
    for i in range(n_fwd):
        for j in range(n_rev):
            p = os.path.join(root, "full", pool, names[i][j] + ".fastq")
            write(p, [(f"{names[i][j]}_f{r}", mutate(amp[i][j])) for r in range(n_full)])
            paths.append(p)
    pdir = os.path.join(root, "partial", pool, pair)
    for tag, barcodes, members in (("rev", b2s, lambda j: [(i, j) for i in range(n_fwd)]),
                                   ("fwd", b1s, lambda i: [(i, j) for j in range(n_rev)])):
        for x, bc in enumerate(barcodes):
            reads = [(f"{names[i][j]}_{tag}{r}", mutate(amp[i][j])) for i, j in members(x) for r in range(n_partial)]
            reads += [(f"other-{tag}{x}_{r}", rnd(int(amplicon + rng.integers(-amplicon // 20, amplicon // 20 + 1))))
                      for r in range(n_other)]
            order = rng.permutation(len(reads))
            write(os.path.join(pdir, f"barcode_{tag}_{bc}.fastq"), [reads[o] for o in order])
    return paths
