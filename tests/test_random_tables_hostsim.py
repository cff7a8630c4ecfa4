"""Randomised tables and reads (mixed barcode lengths, IUPAC-degenerate primers, shared primers,
wildcards, every k from 0 to 5, N / IUPAC / lower-case symbols, reads shorter than the search
window): CUDA per-thread routines (via the CPU kernel simulator) against the live oracle."""
import random

import pytest

import helpers as H
from oracle import pipeline as orc
from specimux_b200.demultiplex import process_sequences
from specimux_b200.models import MatchParameters
from specimux_b200.seqio import reverse_complement

IUPAC = {"R": "AG", "Y": "CT", "S": "CG", "W": "AT", "K": "GT", "M": "AC", "B": "CGT", "D": "AGT", "H": "ACT",
         "V": "ACG", "N": "ACGT"}


def rand_seq(rng, n, alphabet="ACGT"):
    return "".join(rng.choice(alphabet) for _ in range(n))


def mutate(rng, s, rate):
    out = []
    for c in s:
        u = rng.random()
        if u < rate * 0.4:
            out.append(rng.choice("ACGT"))
        elif u < rate * 0.7:
            out.append(rng.choice("ACGT") + c)
        elif u < rate:
            continue
        else:
            out.append(c)
    return "".join(out)


def instantiate(rng, s):
    return "".join(rng.choice(IUPAC[c]) if c in IUPAC else c for c in s)


def make_case(seed, long_primers=False, primer_lens=None, barcode_lens=None, search_lens=None, primer_k=None):
    """long_primers: some primers of 65..300 nt (the warp-cooperative multi-word search) and search
    windows wide enough to hold them.

    The keyword lists replace the default draws (left at None, a seed gives the same case as ever):
    primer_lens the primer lengths (with long_primers, the lengths of the long primers), barcode_lens the
    barcode lengths (k is then kept to length + k <= 64), search_lens the windows (inserts then reach
    past 2 x search_len, so reads are clipped).  primer_k, as flags["primer_k"]: {primer name: k}, or
    one k that caps every primer's default threshold."""
    rng = random.Random(seed)
    n_fwd, n_rev = rng.randint(1, 3), rng.randint(1, 3)
    pools = ["P%d" % i for i in range(rng.randint(1, 2))]
    primers = []
    for i in range(n_fwd + n_rev):
        seq = rand_seq(rng, rng.choice(primer_lens) if primer_lens and not long_primers else rng.randint(16, 26))
        if long_primers and (i == 0 or rng.random() < 0.5):
            seq = rand_seq(rng, rng.choice(primer_lens or [65, 66, 96, 97, 127, 128, 129, 150, 200, 256, 257, 300]))
        if rng.random() < 0.5:
            seq = "".join(rng.choice("RYNWM") if rng.random() < 0.12 else c for c in seq)
        ppools = sorted(rng.sample(pools, rng.randint(1, len(pools))))
        primers.append(("F%d" % i if i < n_fwd else "R%d" % i, seq, "forward" if i < n_fwd else "reverse", ppools))
    for pool in pools:      # every pool needs both directions
        for direction in ("forward", "reverse"):
            if not any(pool in p[3] and p[2] == direction for p in primers):
                idx = next(i for i, p in enumerate(primers) if p[2] == direction)
                primers[idx] = (primers[idx][0], primers[idx][1], direction, sorted(set(primers[idx][3]) | {pool}))
    lens = [rng.choice(barcode_lens or [9, 11, 13, 13, 13, 16]) for _ in range(2)]
    mixed = rng.random() < 0.4
    nb1, nb2 = rng.randint(2, 40), rng.randint(2, 70)

    def barcodes(n, ln):
        out = set()
        while len(out) < n:
            out.add(rand_seq(rng, min(rng.choice([ln, ln - 2, ln + 1]), 64) if mixed else ln))
        return sorted(out, key=lambda _: rng.random())
    b1s, b2s = barcodes(nb1, lens[0]), barcodes(nb2, lens[1])
    specimens = []
    seen = set()
    for i in range(rng.randint(3, 120)):
        pool = rng.choice(pools)
        fw = [p for p in primers if p[2] == "forward" and pool in p[3]]
        rv = [p for p in primers if p[2] == "reverse" and pool in p[3]]
        p1 = "*" if rng.random() < 0.15 else rng.choice(fw)[0]
        p2 = "-" if rng.random() < 0.1 else rng.choice(rv)[0]
        b1, b2 = rng.choice(b1s), rng.choice(b2s)
        if (pool, b1, b2, p1, p2) in seen:
            continue
        seen.add((pool, b1, b2, p1, p2))
        specimens.append(("S%03d" % i, pool, b1, p1, b2, p2))
    k_idx = rng.choice([0, 1, 2, 3, 3, 4, 5])
    k_idx = min(k_idx, min(len(b) for b in b1s + b2s) - 1, 64 - max(len(b) for b in b1s + b2s))
    L = rng.choice([40, 80, 80, 120, 200])
    if long_primers:
        L = rng.choice([120, 200, 333, 512])
    if search_lens:
        L = rng.choice(search_lens)
    reads = []
    by_name = {p[0]: p for p in primers}
    for r in range(rng.randint(40, 90)):
        sp = rng.choice(specimens)
        fw = [p for p in primers if p[2] == "forward" and sp[1] in p[3]]
        rv = [p for p in primers if p[2] == "reverse" and sp[1] in p[3]]
        p1 = by_name[sp[3]] if sp[3] in by_name else rng.choice(fw)
        p2 = by_name[sp[5]] if sp[5] in by_name else rng.choice(rv)
        kind = rng.random()
        insert = rand_seq(rng, rng.randint(0, 300 if not search_lens else 2 * L + 100))
        left = rand_seq(rng, rng.randint(0, 25)) + sp[2] + instantiate(rng, p1[1])
        right = reverse_complement(instantiate(rng, p2[1])) + reverse_complement(sp[4]) + rand_seq(rng, rng.randint(0, 25))
        if kind < 0.1:
            s = insert
        elif kind < 0.2:
            s = left + insert
        elif kind < 0.3:
            s = insert + right
        else:
            s = left + insert + right
        s = mutate(rng, s, rng.choice([0.0, 0.05, 0.12]))
        if rng.random() < 0.5:
            s = reverse_complement(s)
        u = rng.random()
        if u < 0.1:
            s = "".join("N" if rng.random() < 0.05 else c for c in s)
        elif u < 0.15:
            s = "".join(rng.choice("RYKMSWBDHV") if rng.random() < 0.05 else c for c in s)
        elif u < 0.2:
            s = s[:30].lower() + s[30:]
        elif u < 0.3:
            s = s[:rng.randint(0, L + 3)]
        elif u < 0.35:
            s = s[len(s) - min(len(s), rng.randint(0, L + 3)):]
        reads.append(("r%04d" % r, s, "".join(chr(33 + rng.randint(2, 40)) for _ in s)))
    flags = dict(search_len=L, trim=rng.choice(["barcodes", "primers", "tails", "none"]),
                 dereplicate=rng.choice(["best", "none"]), disable_preorient=rng.random() < 0.3,
                 disable_prefilter=rng.random() < 0.5)
    if primer_k is not None:
        flags["primer_k"] = primer_k
    return primers, specimens, reads, k_idx, flags


def make_iupac_barcode_case(seed):
    """Barcodes that hold IUPAC codes, searched with the Bloom prefilter ON (the default flags): the reference builds
    the filter's variants from the barcode STRING (bloom_filter.py:70-101), so an N in a barcode only passes the
    filter where the read has a literal N or an edit is spent on it, while edlib itself matches it for free.
    Uniform barcode length (the reference takes the filter's key length from one barcode)."""
    rng = random.Random(7000 + seed)
    primers = [("F0", rand_seq(rng, 20), "forward", ["P0"]), ("R0", rand_seq(rng, 22), "reverse", ["P0"])]
    if rng.random() < 0.5:
        primers.append(("F1", rand_seq(rng, 18), "forward", ["P0"]))
    blen = rng.choice([11, 13, 13])

    def barcode():
        s = list(rand_seq(rng, blen))
        if rng.random() < 0.6:
            for _ in range(rng.randint(1, 2)):
                i = rng.randrange(blen)
                s[i] = rng.choice([c for c, v in IUPAC.items() if s[i] in v or s[i] == c])
        return "".join(s)
    b1s = sorted({barcode() for _ in range(rng.randint(3, 20))})
    b2s = sorted({barcode() for _ in range(rng.randint(3, 40))})
    specimens, seen = [], set()
    for i in range(rng.randint(5, 60)):
        p1 = rng.choice([p[0] for p in primers if p[2] == "forward"])
        b1, b2 = rng.choice(b1s), rng.choice(b2s)
        if (b1, b2, p1) in seen:
            continue
        seen.add((b1, b2, p1))
        specimens.append(("S%03d" % i, "P0", b1, p1, b2, "R0"))
    by_name = {p[0]: p for p in primers}
    reads = []
    for r in range(70):
        sp = rng.choice(specimens)

        def concrete(bc):           # what a read carries where the barcode has a code: a base of the set, or a literal N
            return "".join((("N" if rng.random() < 0.3 else rng.choice(IUPAC[c])) if c in IUPAC else c) for c in bc)
        s = (rand_seq(rng, rng.randint(0, 20)) + concrete(sp[2]) + by_name[sp[3]][1] + rand_seq(rng, rng.randint(30, 200)) +
             reverse_complement(by_name[sp[5]][1]) + reverse_complement(concrete(sp[4])) + rand_seq(rng, rng.randint(0, 20)))
        s = mutate(rng, s, rng.choice([0.0, 0.03, 0.08]))
        if rng.random() < 0.5:
            s = reverse_complement(s)
        reads.append(("q%04d" % r, s, "I" * len(s)))
    flags = dict(search_len=80, trim=rng.choice(["barcodes", "tails"]), dereplicate=rng.choice(["best", "none"]),
                 disable_preorient=False, disable_prefilter=False)
    return primers, specimens, reads, rng.choice([1, 2, 3]), flags


@pytest.mark.parametrize("seed", range(12))
def test_iupac_barcodes_with_prefilter(seed):
    run_case(*make_iupac_barcode_case(seed), tag="iupac barcode seed %d" % seed)


def make_large_k_case(seed, barcode_lens=None):
    """Long barcodes searched with thresholds beyond 8 (the reference derives k = ceil(min pairwise distance / 2),
    orchestration.py:583-600): the general band walk of stage 2 with up to 25 diagonals.  barcode_lens replaces
    the barcode lengths drawn from; k is then lowered to keep length + k <= 64 and the windows hold the barcode."""
    rng = random.Random(9000 + seed)
    primers = [("F0", rand_seq(rng, 21), "forward", ["P0"]), ("R0", rand_seq(rng, 19), "reverse", ["P0"])]
    blen = rng.choice(barcode_lens or [24, 28, 30])
    b1s = sorted({rand_seq(rng, blen) for _ in range(rng.randint(2, 12))})
    b2s = sorted({rand_seq(rng, blen) for _ in range(rng.randint(2, 40))})
    specimens = [("S%03d" % i, "P0", rng.choice(b1s), "F0", rng.choice(b2s), "R0") for i in range(25)]
    specimens = list({(s[2], s[4]): s for s in specimens}.values())
    reads = []
    for r in range(50):
        sp = rng.choice(specimens)
        s = (rand_seq(rng, rng.randint(0, 20)) + sp[2] + primers[0][1] + rand_seq(rng, rng.randint(30, 200)) +
             reverse_complement(primers[1][1]) + reverse_complement(sp[4]) + rand_seq(rng, rng.randint(0, 20)))
        s = mutate(rng, s, rng.choice([0.05, 0.15, 0.3]))
        if rng.random() < 0.5:
            s = reverse_complement(s)
        if rng.random() < 0.1:
            s = s[:40] + "N" + s[41:]
        reads.append(("k%04d" % r, s, "I" * len(s)))
    flags = dict(search_len=rng.choice([128, 200] if barcode_lens else [80, 120]), trim=rng.choice(["barcodes", "tails"]),
                 dereplicate=rng.choice(["best", "none"]), disable_preorient=False, disable_prefilter=rng.random() < 0.5)
    return primers, specimens, reads, min(rng.choice([9, 10, 11, 12]), 64 - blen), flags


@pytest.mark.parametrize("seed", range(8))
def test_barcode_threshold_beyond_eight(seed):
    run_case(*make_large_k_case(seed), tag="large k seed %d" % seed)


def make_many_primers_case(seed, n_fwd=100, n_rev=100, n_pairs=300):
    """200 canonical primers in 300 primer pairs (the reference is unbounded, databases.py:247-264): multi-word
    primer-identity masks, the 254-primer selection instantiation, one sliced launch per primer; one barcode holds N."""
    rng = random.Random(11000 + seed)
    pools = ["PA", "PB", "PC"]
    seqs = set()
    while len(seqs) < n_fwd + n_rev:
        seqs.add(rand_seq(rng, rng.randint(18, 24)))
    seqs = sorted(seqs, key=lambda _: rng.random())
    primers = []
    for i, sq in enumerate(seqs):
        pool = pools[i % 3]
        primers.append(("F%03d" % i if i < n_fwd else "R%03d" % i, sq, "forward" if i < n_fwd else "reverse", [pool]))
    b1s = [rand_seq(rng, 13) for _ in range(12)]
    b2s = [rand_seq(rng, 13) for _ in range(24)]
    b1s[3] = b1s[3][:5] + "N" + b1s[3][6:]
    specimens, seen = [], set()
    while len(seen) < n_pairs:
        pool = rng.choice(pools)
        f = rng.choice([p for p in primers if p[2] == "forward" and p[3] == [pool]])
        r = rng.choice([p for p in primers if p[2] == "reverse" and p[3] == [pool]])
        if (f[0], r[0]) in seen:
            continue
        seen.add((f[0], r[0]))
        specimens.append(("S%04d" % len(specimens), pool, rng.choice(b1s), f[0], rng.choice(b2s), r[0]))
    by_name = {p[0]: p for p in primers}
    reads = []
    for r in range(60):
        sp = rng.choice(specimens)
        b1 = sp[2].replace("N", rng.choice("ACGTN"))
        s = (rand_seq(rng, rng.randint(0, 20)) + b1 + by_name[sp[3]][1] + rand_seq(rng, rng.randint(30, 150)) +
             reverse_complement(by_name[sp[5]][1]) + reverse_complement(sp[4]) + rand_seq(rng, rng.randint(0, 20)))
        s = mutate(rng, s, rng.choice([0.0, 0.04, 0.08]))
        if rng.random() < 0.5:
            s = reverse_complement(s)
        reads.append(("m%04d" % r, s, "I" * len(s)))
    flags = dict(search_len=80, trim="barcodes", dereplicate=rng.choice(["best", "none"]), disable_preorient=rng.random() < 0.5,
                 disable_prefilter=False)
    return primers, specimens, reads, 3, flags


@pytest.mark.parametrize("seed", range(3))
def test_two_hundred_primers_three_hundred_pairs(seed):
    run_case(*make_many_primers_case(seed), tag="many primers seed %d" % seed)


def test_long_primer_carry_lookahead():
    """The kernel's one-addition carry-lookahead over the words of every segment of a warp
    (long_carry_in<SW>) against a rippled carry chain, 2M random generate/propagate masks per width."""
    lib = H.hostsim_binding()
    assert lib.hostsim_check_long_carry(2_000_000) == 0


@pytest.mark.parametrize("seed", range(1000, 1016))
def test_random_case_long_primers(seed):
    run_case(*make_case(seed, long_primers=True), tag="long seed %d" % seed)


@pytest.mark.parametrize("seed", range(60))
def test_random_case(seed):
    run_case(*make_case(seed), tag="seed %d" % seed)


# Cases across the ranges the C ABI accepts (primers of 1..1024 nt with k <= 127, barcode length + k <= 64,
# search_len 1..1024), where the launchers pick other kernels or instantiations than the cases above reach.
SLICED_LENS = list(range(9, 16)) + list(range(27, 33))          # k_primer_sliced<M>; m + k crosses 32 at 27..32
U64_LENS = [33, 40, 48, 63, 64]                                  # t.use64: every primer through k_primer_finish<u64>
# (long primer length, primer_k, search_len): every segment width, L below the primer length, k = 127 and k = 0
LONG_WIDTH_CASES = [(161, None, 512), (192, None, 761), (321, None, 1024), (383, None, 640), (384, 127, 1000),
                    (512, 100, 512), (513, 127, 1024), (700, 90, 640), (1024, 127, 1000), (1024, 127, 1024),
                    (200, {"F0": 0}, 761)]
LONG_WIDTH_SEEDS = [3001, 3002, 3003, 3004, 3005, 3008, 3009, 3010, 3011, 3012, 3013]       # each table also holds a short primer
LONG_BARCODE_LENS = [31, 40, 47, 52, 55, 58, 61, 64]


def make_range_case(cls, i):
    """Case i of class cls (see RANGE_CLASSES)."""
    if cls == "sliced":
        return make_case(2000 + i, primer_lens=SLICED_LENS, search_lens=[80, 120, 200])
    if cls == "u64":
        return make_case(2100 + i, primer_lens=[20, 20, U64_LENS[i % 5], U64_LENS[(i + 2) % 5]], search_lens=[120, 200])
    if cls == "long_width":
        length, k, L = LONG_WIDTH_CASES[i]
        return make_case(LONG_WIDTH_SEEDS[i], long_primers=True, primer_lens=[length], search_lens=[L], primer_k=k)
    if cls == "wide_window":
        return make_case(2300 + i, search_lens=[761, 1024])
    if cls == "long_barcode":
        return make_large_k_case(100 + i, barcode_lens=LONG_BARCODE_LENS)
    if cls == "long_barcode_mixed":
        return make_case(2500 + i, barcode_lens=[31, 40, 52, 63, 64], search_lens=[128, 200])
    raise KeyError(cls)


RANGE_CLASSES = {"sliced": 8, "u64": 8, "long_width": len(LONG_WIDTH_CASES), "wide_window": 6, "long_barcode": 8,
                 "long_barcode_mixed": 6}
RANGE_CASES = [(c, i) for c, n in RANGE_CLASSES.items() for i in range(n)]


def range_case_id(case):
    return "%s-%d" % case


@pytest.mark.parametrize("cls,i", RANGE_CASES, ids=[range_case_id(c) for c in RANGE_CASES])
def test_accepted_range_case(cls, i):
    run_case(*make_range_case(cls, i), tag="%s case %d" % (cls, i))


def segment_width(m):
    """smx_host_tables.hpp's kWidths rule: lanes per read of k_primer_long for a primer of m > 64 nt."""
    return next((w for w in (3, 4, 5, 6, 8, 10, 16, 32) if w >= (m + 31) // 32), 32)


def test_range_cases_reach_every_kernel():
    """The classes above reach what they are named for: every segment width (with the long seeds), the sliced
    lengths on both sides of m + k = 32, 33..64-nt primers beside 20-nt ones, windows past the shared tile with
    clipped reads, barcode length + k = 64, k = 0 and k = 127 on long primers, L below a long primer's length."""
    widths = set()
    for seed in range(1000, 1016):
        widths |= {segment_width(len(p[1])) for p in make_case(seed, long_primers=True)[0] if len(p[1]) > 64}
    for i in range(RANGE_CLASSES["long_width"]):
        primers, _sp, _r, _k, flags = make_range_case("long_width", i)
        longs = [len(p[1]) for p in primers if len(p[1]) > 64]
        assert any(len(p[1]) <= 64 for p in primers), "long-width case %d has no short primer beside the long one" % i
        widths |= {segment_width(m) for m in longs}
    assert widths == {3, 4, 5, 6, 8, 10, 16, 32}, widths
    short_k = set()
    for i in range(RANGE_CLASSES["sliced"]):
        primers, _sp, _r, _k, _f = make_range_case("sliced", i)
        assert all(len(p[1]) in SLICED_LENS for p in primers)
        short_k |= {len(p[1]) + int(orc_default_k(p[1])) > 32 for p in primers}
    assert short_k == {False, True}
    u64 = set()
    for i in range(RANGE_CLASSES["u64"]):
        lens = {len(p[1]) for p in make_range_case("u64", i)[0]}
        u64 |= lens
    assert set(U64_LENS) | {20} <= u64
    for i in range(RANGE_CLASSES["wide_window"]):
        _p, _sp, reads, _k, flags = make_range_case("wide_window", i)
        assert flags["search_len"] > 760 and max(len(r[1]) for r in reads) > 2 * flags["search_len"]
    mk = []
    for i in range(RANGE_CLASSES["long_barcode"]):
        _p, specimens, _r, k, _f = make_range_case("long_barcode", i)
        mk.append(max(len(s[2]) for s in specimens) + k)
    for i in range(RANGE_CLASSES["long_barcode_mixed"]):
        _p, specimens, _r, k, _f = make_range_case("long_barcode_mixed", i)
        mk.append(max(len(b) for s in specimens for b in (s[2], s[4])) + k)
    assert max(mk) == 64 and mk.count(64) >= 2, mk
    ks = [make_range_case("long_width", i)[4].get("primer_k") for i in range(RANGE_CLASSES["long_width"])]
    assert 127 in ks and {"F0": 0} in ks
    assert any(length > L for length, _k, L in LONG_WIDTH_CASES)


def orc_default_k(seq):
    """The reference's default primer threshold (orchestration.py:564-570, 603-614)."""
    score = sum(3 if c in "ACGT" else 2 if c in "KMRSWY" else 1 if c in "BDHV" else 0 for c in seq)
    return int(score / 3.0 / 3)


def primer_thresholds(oparams, primers, flags):
    """Applies flags["primer_k"] (see make_case) to the oracle's per-sequence primer thresholds."""
    pk = flags.get("primer_k")
    if isinstance(pk, int):
        for seq in oparams.max_dist_primers:
            oparams.max_dist_primers[seq] = min(oparams.max_dist_primers[seq], pk)
    elif pk:
        seq_of = {p[0]: p[1] for p in primers}
        for name, k in pk.items():
            oparams.max_dist_primers[seq_of[name]] = k
    return oparams


def run_case(primers, specimens, reads, k_idx, flags, tag, binding=None):
    """binding="cuda": through the CUDA library (GPU tests); default: the CPU kernel simulator."""
    try:
        tables = orc.Tables(primers, specimens)
    except ValueError:
        pytest.skip("generator produced an invalid table")
    oparams = orc.setup_params(tables, index_edit_distance=k_idx, search_len=flags["search_len"],
                               preorient=not flags["disable_preorient"], prefilter=not flags["disable_prefilter"],
                               trim=flags["trim"], dereplicate=flags["dereplicate"])
    primer_thresholds(oparams, primers, flags)
    expected, total, matched = orc.process_reads(tables, oparams, reads)
    sp = H.build_specimens(primers, specimens)
    params = MatchParameters(dict(oparams.max_dist_primers), k_idx, flags["search_len"], not flags["disable_preorient"])
    args = H.make_args(flags)
    ops, n, m = process_sequences(H.records(reads), params, sp, args, H.prefilter_for(args), None, 0,
                                  _binding=None if binding == "cuda" else H.hostsim_binding())
    assert (n, m) == (total, matched)
    H.assert_ops_equal([H.op_to_dict(o) for o in ops], [H.op_to_dict(o) for o in expected], tag)


# One step past each limit of the C ABI, and the value one step inside it: (name, refused, accepted) as keyword
# arguments of limit_tables.
LIMITS = [("primer_length", dict(primer_len=1025, primer_k=30, search_len=1024), dict(primer_len=1024, primer_k=30, search_len=1024)),
          ("primer_k", dict(primer_len=1024, primer_k=128, search_len=1024), dict(primer_len=1024, primer_k=127, search_len=1024)),
          ("search_len", dict(search_len=1025), dict(search_len=1024)),
          ("barcode_length_plus_k", dict(barcode_len=60, k_idx=5), dict(barcode_len=60, k_idx=4))]


def limit_case(primer_len=20, primer_k=None, search_len=80, barcode_len=13, k_idx=2):
    """make_case's form: one pool, F0 of primer_len nt (threshold primer_k, default the reference's), a 22-nt R0,
    three barcodes of barcode_len nt per end, and reads built from them."""
    rng = random.Random(primer_len * 7 + barcode_len)
    primers = [("F0", rand_seq(rng, primer_len), "forward", ["P0"]), ("R0", rand_seq(rng, 22), "reverse", ["P0"])]
    b1s = [rand_seq(rng, barcode_len) for _ in range(3)]
    b2s = [rand_seq(rng, barcode_len) for _ in range(3)]
    specimens = [("S%d" % i, "P0", b1s[i], "F0", b2s[i], "R0") for i in range(3)]
    reads = []
    for i in range(8):
        s = (rand_seq(rng, 5) + b1s[i % 3] + primers[0][1] + rand_seq(rng, search_len + 40) + reverse_complement(primers[1][1]) +
             reverse_complement(b2s[i % 3]) + rand_seq(rng, 5))
        s = mutate(rng, s, 0.02 * (i % 3))
        reads.append(("l%d" % i, reverse_complement(s) if i % 2 else s, "I" * len(s)))
    flags = dict(search_len=search_len, trim="barcodes", dereplicate="best", disable_preorient=False,
                 disable_prefilter=True)
    if primer_k is not None:
        flags["primer_k"] = {"F0": primer_k}
    return primers, specimens, reads + [("empty", "", "")], k_idx, flags


def limit_tables(primers, specimens, reads, k_idx, flags):
    """The MatchTables of a limit_case."""
    from specimux_b200.tables import MatchTables
    thr = {p[1]: orc_default_k(p[1]) for p in primers}
    for name, k in flags.get("primer_k", {}).items():
        thr[next(p[1] for p in primers if p[0] == name)] = k
    sp = H.build_specimens(primers, specimens)
    return MatchTables(sp, MatchParameters(thr, k_idx, flags["search_len"], True), prefilter=False)


@pytest.mark.parametrize("name,refused,accepted", LIMITS, ids=[x[0] for x in LIMITS])
def test_limits_refused_and_accepted(name, refused, accepted):
    """The table build shared with the CUDA library refuses one step past each limit with SMX_ERR_ARG; one step
    inside it the simulator matches the reads as the oracle does."""
    from specimux_b200 import _lib
    from specimux_b200.engine import Matcher, PackedBatch
    case = limit_case(**refused)
    with pytest.raises(_lib.SmxError) as e:
        Matcher(limit_tables(*case), binding=H.hostsim_binding()).match(PackedBatch([r[1] for r in case[2]]))
    assert e.value.code == _lib.SMX_ERR_ARG, e.value
    run_case(*limit_case(**accepted), tag="limit %s" % name)
