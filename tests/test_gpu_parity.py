"""Parity of the CUDA path (through the C ABI) against the oracle, the golden vectors and -- at
full BASELINE sizes -- size-independent properties.  Needs a GPU: `pytest -m gpu`."""
import argparse

import numpy as np
import pytest

import helpers as H
from specimux_b200 import synth
from specimux_b200.demultiplex import process_sequences, records_to_write_ops
from specimux_b200.engine import Matcher, PackedBatch
from specimux_b200.models import MatchParameters
from specimux_b200.orchestration import thresholds_for
from specimux_b200.tables import MatchTables

pytestmark = pytest.mark.gpu


def _golden_cases():
    for name in H.golden_names():
        for run in H.load_golden(name)["runs"]:
            yield name, run


@pytest.mark.parametrize("name,run_name", list(_golden_cases()))
def test_cuda_matches_golden(name, run_name):
    g = H.load_golden(name)
    run = g["runs"][run_name]
    specimens = H.build_specimens(g["primers"], g["specimens"])
    args = H.make_args(run["flags"])
    params = H.params_from_run(run, specimens)
    ops, total, matched = process_sequences(H.records(g["reads"]), params, specimens, args, H.prefilter_for(args))
    assert (total, matched) == (run["total"], run["matched"])
    H.assert_ops_equal([H.op_to_dict(o) for o in ops], run["ops"], "%s/%s" % (name, run_name))


def test_thresholds_on_gpu_match_golden():
    """setup_match_parameters' NW distances (orchestration.py:549-600) computed by the GPU kernel."""
    for name in ("fixture", "synth_ont037", "synth_dense", "synth_multipool"):
        g = H.load_golden(name)
        run = g["runs"]["default"]
        specimens = H.build_specimens(g["primers"], g["specimens"])
        k_idx, k_primers = thresholds_for(specimens)
        assert k_idx == run["k_index"], name
        assert k_primers == run["k_primers"], name


def _setup(ds, **flags):
    specimens = H.build_specimens(ds.primers, ds.specimens)
    k_idx, k_primers = thresholds_for(specimens)
    params = MatchParameters(k_primers, k_idx, ds.search_len, not flags.get("disable_preorient", False))
    args = H.make_args(dict(flags, search_len=ds.search_len))
    return specimens, params, args


@pytest.mark.parametrize("cfg,n,flags", [
    ("ont037", 1500, {}), ("ont037", 800, {"dereplicate": "none", "trim": "tails"}),
    ("dense", 1200, {}), ("dense", 600, {"dereplicate": "none", "trim": "primers"}),
    ("multipool", 1200, {}), ("multipool", 600, {"disable_preorient": True, "trim": "tails"}),
    ("long", 300, {}),
])
def test_cuda_matches_live_oracle(cfg, n, flags):
    """Seeded synthetic slices (different seeds from the goldens), oracle run live as the checker."""
    from oracle import pipeline as orc
    ds = synth.CONFIGS[cfg](n_reads=n, seed=1234 + n)
    reads = ds.reads()
    tables = orc.Tables(ds.primers, ds.specimens)
    oparams = orc.setup_params(tables, search_len=ds.search_len, preorient=not flags.get("disable_preorient", False),
                               trim=flags.get("trim", "barcodes"), dereplicate=flags.get("dereplicate", "best"))
    expected, total, matched = orc.process_reads(tables, oparams, reads)
    specimens, params, args = _setup(ds, **flags)
    assert params.max_dist_index == oparams.max_dist_index
    ops, n_total, n_matched = process_sequences(H.records(reads), params, specimens, args, H.prefilter_for(args))
    assert (n_total, n_matched) == (total, matched)
    H.assert_ops_equal([H.op_to_dict(o) for o in ops], [H.op_to_dict(o) for o in expected], cfg)


def _end_columns_to_x(n, L):
    """(woff, delta) of smx_core.cuh's make_geo: end-mask column c of a read of n symbols is X index woff + c + delta."""
    raw = n - L
    woff = max(raw, 0)
    if raw >= 0:
        off = shift = raw
    elif raw == -1:
        off = shift = 0
    else:
        off, shift = max(n + raw, 0), raw
    return woff, shift - off


def _level1_detail(primers, specimen_rows, reads, k_primers, k_idx, search_len, min_checked):
    """Every primer distance / first location / location count / end mask and every barcode distance / end set of
    the CUDA library against orc.match_one_end (prefilter off); then primer_hits, endmask, orient_hits,
    barcode_hits and the records bit for bit against the kernel simulator, with clip = search_len and clip = 0."""
    from oracle import pipeline as orc
    specimens = H.build_specimens(primers, specimen_rows)
    params = MatchParameters(dict(k_primers), k_idx, search_len, True)
    mt = MatchTables(specimens, params, prefilter=False)
    bases = [r[1] for r in reads]
    with Matcher(mt) as m:
        res = m.match(PackedBatch(bases), detail=True)
        for clip in (search_len, 0):
            batch = PackedBatch(bases, clip=clip)
            gpu = m.match(batch, detail=True)
            sim = Matcher(mt, binding=H.hostsim_binding()).match(batch, detail=True)
            assert gpu.n_matched == sim.n_matched, clip
            assert np.array_equal(gpu.rec_offset, sim.rec_offset), clip
            assert gpu.records.tobytes() == sim.records.tobytes(), clip
            assert np.array_equal(gpu.primer_hits, sim.primer_hits), clip
            assert np.array_equal(gpu.endmask, sim.endmask), clip
            assert np.array_equal(gpu.orient_hits, sim.orient_hits), clip
            assert np.array_equal(gpu.barcode_hits, sim.barcode_hits), clip
    tables = orc.Tables([tuple(p) for p in primers], [tuple(s) for s in specimen_rows])
    oparams = orc.Params(dict(k_primers), k_idx, search_len=search_len, prefilter=False)
    oprimers = list(tables.by_seq.values())
    nP = len(oprimers)
    mw = res.endmask.shape[1]
    checked = 0
    for r, bases_r in enumerate(bases):
        strands = (bases_r, orc.revcomp(bases_r))
        woff, delta = _end_columns_to_x(len(bases_r), search_len)
        for s in range(2):
            for p, prim in enumerate(oprimers):
                pd, plocs, hits = orc.match_one_end(tables, oparams, strands[s], prim)
                ph = res.primer_hits[s * nP + p, r]
                assert int(ph["distance"]) == pd, (r, s, p)
                if pd < 0:
                    continue
                assert (int(ph["first_start"]), int(ph["first_end"])) == tuple(plocs[0]), (r, s, p, plocs)
                assert int(ph["n_locations"]) == len(plocs)
                em = res.endmask[s * nP + p, :, r]
                ends = [woff + 32 * w + c + delta for w in range(mw) for c in range(32) if (int(em[w]) >> c) & 1]
                assert ends == [e for _s, e in plocs], (r, s, p, ends, plocs)
                hitmap = {b: (d, locs) for b, d, locs in hits}
                base = sum(len(q.barcodes) for q in oprimers) * s + sum(len(q.barcodes) for q in oprimers[:p])
                for j, bc in enumerate(prim.barcodes):
                    bh = res.barcode_hits[base + j, r]
                    if bc in hitmap:
                        d, locs = hitmap[bc]
                        assert int(bh["distance"]) == d, (r, s, p, bc)
                        shift = 0 if int(bh["search_start"]) == -1 else int(bh["search_start"])
                        ends = [shift + c for c in range(64) if (int(bh["end_mask"]) >> c) & 1]
                        assert ends == [e for _s, e in locs], (r, s, p, bc, ends, locs)
                        checked += 1
                    else:
                        assert int(bh["distance"]) == -1, (r, s, p, bc)
    assert checked >= min_checked, checked


def test_level1_detail_matches_oracle():
    """Every primer distance / first location / end count and every barcode distance / end set."""
    g = H.load_golden("fixture_crafted")
    run = g["runs"]["no_prefilter"]
    _level1_detail(g["primers"], g["specimens"], [tuple(r) for r in g["reads"]], run["k_primers"], run["k_index"],
                   run["flags"].get("search_len", 80), 21)


def _range_case(cls, i):
    from test_random_tables_hostsim import make_range_case
    return make_range_case(cls, i)


def _range_cases():
    from test_random_tables_hostsim import RANGE_CASES, range_case_id
    return RANGE_CASES, [range_case_id(c) for c in RANGE_CASES]


@pytest.mark.parametrize("cls,i", _range_cases()[0], ids=_range_cases()[1])
def test_cuda_accepted_range_case(cls, i):
    """Primers of 9..15, 27..32 and 33..64 nt, long primers of every segment width up to 1024 nt with k up to 127
    (and 0), windows of 761 and 1024 with clipped reads, barcodes of 31..64 nt with length + k up to 64: the
    CUDA library against the live oracle."""
    from test_random_tables_hostsim import run_case
    run_case(*_range_case(cls, i), tag="%s case %d" % (cls, i), binding="cuda")


# one case of each class (long widths: segment widths 6, 16 and 32, the last with k = 127 on 1024 nt, and k = 0)
LEVEL1_RANGE_CASES = [("sliced", 0), ("u64", 0), ("long_width", 0), ("long_width", 4), ("long_width", 9),
                      ("long_width", 10), ("wide_window", 0), ("long_barcode", 0), ("long_barcode_mixed", 0)]


@pytest.mark.parametrize("cls,i", LEVEL1_RANGE_CASES, ids=["%s-%d" % c for c in LEVEL1_RANGE_CASES])
def test_cuda_range_case_level1_detail(cls, i):
    """_level1_detail on one case of each accepted-range class."""
    from oracle import pipeline as orc
    from test_random_tables_hostsim import primer_thresholds
    primers, specimen_rows, reads, k_idx, flags = _range_case(cls, i)
    oparams = orc.setup_params(orc.Tables(primers, specimen_rows), index_edit_distance=k_idx)
    primer_thresholds(oparams, primers, flags)
    _level1_detail(primers, specimen_rows, reads, oparams.max_dist_primers, k_idx, flags["search_len"], 1)


def _limits():
    from test_random_tables_hostsim import LIMITS
    return LIMITS


@pytest.mark.parametrize("name,refused,accepted", _limits(), ids=[x[0] for x in _limits()])
def test_cuda_limits_refused_and_accepted(name, refused, accepted):
    """smx_create refuses one step past each limit with SMX_ERR_ARG, an open context keeps its results, and one
    step inside the limit the CUDA library matches as the oracle does."""
    from specimux_b200 import _lib
    from test_random_tables_hostsim import limit_case, limit_tables, run_case
    ok = limit_case()
    ok_batch = PackedBatch([r[1] for r in ok[2]])
    with Matcher(limit_tables(*ok)) as m:
        want = m.match(ok_batch, detail=True)
        with pytest.raises(_lib.SmxError) as e:
            Matcher(limit_tables(*limit_case(**refused)))
        assert e.value.code == _lib.SMX_ERR_ARG, e.value
        got = m.match(ok_batch, detail=True)
        assert got.records.tobytes() == want.records.tobytes()
        assert np.array_equal(got.primer_hits, want.primer_hits) and np.array_equal(got.barcode_hits, want.barcode_hits)
    run_case(*limit_case(**accepted), tag="limit %s" % name, binding="cuda")


def _nw_sequences(rng, n):
    alphabet = list("ACGTACGTRYKMNacgtn")
    lens = [0, 64, 1, 63] + list(rng.integers(0, 65, size=max(n - 4, 0)))
    return ["".join(rng.choice(alphabet, size=int(k))) for k in lens[:n]]


@pytest.mark.parametrize("n", [1, 2, 129, 601])
def test_pairwise_nw_full_matrix_matches_oracle(n):
    """smx_pairwise_nw's whole n x n matrix (sequences of 0..64 symbols, IUPAC codes and lower case compared as
    plain characters) equals the oracle's NW distance pair by pair; it is symmetric with a zero diagonal."""
    from oracle import pipeline as orc
    from specimux_b200.orchestration import pairwise_nw
    rng = np.random.default_rng(n)
    seqs = _nw_sequences(rng, n)
    if n > 4:
        seqs[5] = seqs[4]                         # a duplicate: distance 0 off the diagonal
    got = pairwise_nw(seqs)
    assert got.shape == (n, n)
    want = np.array([[orc.nw_distance(a, b) for b in seqs] for a in seqs], dtype=np.int32)
    assert np.array_equal(got, want), np.argwhere(got != want)[:10]
    assert np.array_equal(got, got.T)
    assert not np.diagonal(got).any()


def test_pairwise_nw_refuses_65_symbols():
    """A 65-symbol sequence fails with SMX_ERR_ARG; the next call works."""
    from oracle import pipeline as orc
    from specimux_b200 import _lib
    from specimux_b200.orchestration import pairwise_nw
    with pytest.raises(_lib.SmxError) as e:
        pairwise_nw(["ACGT", "A" * 65, "C"])
    assert e.value.code == _lib.SMX_ERR_ARG, e.value
    seqs = ["A" * 64, "C" * 64, "ACGT"]
    assert pairwise_nw(seqs).tolist() == [[orc.nw_distance(a, b) for b in seqs] for a in seqs]


@pytest.mark.parametrize("cfg,n", [("ont037", 30000), ("dense", 20000), ("multipool", 20000), ("long", 8000)])
def test_cuda_equals_kernel_simulator_at_scale(cfg, n):
    """Bit-identical records between the CUDA launch and the CPU loop over the same thread routines:
    catches indexing / race / launch-geometry faults the small oracle cases cannot."""
    ds = synth.CONFIGS[cfg](n_reads=n, seed=77)
    specimens, params, args = _setup(ds)
    mt = MatchTables(specimens, params)
    blob = np.frombuffer(b"ACGT", dtype=np.uint8)[ds.codes].tobytes()
    batch = PackedBatch.from_blob(blob, ds.offsets.astype(np.uint64))
    with Matcher(mt) as m:
        gpu = m.match(batch, detail=True)
    sim = Matcher(mt, binding=H.hostsim_binding()).match(batch, detail=True)
    assert gpu.n_matched == sim.n_matched
    assert np.array_equal(gpu.rec_offset, sim.rec_offset)
    assert gpu.records.tobytes() == sim.records.tobytes()
    assert np.array_equal(gpu.primer_hits, sim.primer_hits)


@pytest.mark.parametrize("cfg,n,chunk", [("ont037", 20000, 1024), ("dense", 12000, 1152), ("multipool", 9000, 128)])
def test_pipelined_match_equals_one_shot(cfg, n, chunk):
    """smx_match_batch's chunked, three-stream form returns exactly the one-shot result (records,
    offsets, matched count), including reads on the exact 4-bit side stream and multi-record reads."""
    ds = synth.CONFIGS[cfg](n_reads=n, seed=4242)
    specimens, params, args = _setup(ds)
    mt = MatchTables(specimens, params, dereplicate="none" if cfg == "dense" else "best")
    codes = np.frombuffer(b"ACGT", dtype=np.uint8)[ds.codes].copy()
    rng = np.random.default_rng(5)
    hits = rng.choice(codes.shape[0], size=codes.shape[0] // 4000, replace=False)
    codes[hits] = np.frombuffer(b"NRYn", dtype=np.uint8)[rng.integers(0, 4, size=hits.shape[0])]
    batch = PackedBatch.from_blob(codes.tobytes(), ds.offsets.astype(np.uint64), clip=ds.search_len)
    assert batch.n_flagged > 0
    with Matcher(mt) as m:
        m.set_pipeline_chunk(0)
        one = m.match(batch)
        assert m.last_chunk_count() == 1
        m.set_pipeline_chunk(chunk)
        for _ in range(2):
            piped = m.match(batch)
            assert -(-n // chunk) <= m.last_chunk_count() <= -(-n // chunk) + 2      # two small ramp-up chunks
            assert piped.n_matched == one.n_matched
            assert np.array_equal(piped.rec_offset, one.rec_offset)
            assert piped.records.tobytes() == one.records.tobytes()
        # the resident API still works after a pipelined call
        m.upload(batch)
        m.run_resident()
        assert m.download().records.tobytes() == one.records.tobytes()


def test_full_size_properties_ont037():
    """BASELINE config 2 at full size (765k reads): determinism, batch-split invariance,
    reverse-complement invariance of the specimen calls, and agreement with the generator's truth."""
    ds = synth.ont037(n_reads=765_000, with_quals=False)
    specimens, params, args = _setup(ds)
    mt = MatchTables(specimens, params)
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    blob = lut[ds.codes].tobytes()
    offs = ds.offsets.astype(np.uint64)
    with Matcher(mt) as m:
        whole = m.match(PackedBatch.from_blob(blob, offs))
        again = m.match(PackedBatch.from_blob(blob, offs))
        assert whole.records.tobytes() == again.records.tobytes()          # deterministic
        # batch-split invariance: three uneven pieces give the same records
        cuts = [0, 100_001, 400_000, 765_000]
        parts = []
        for a, b in zip(cuts[:-1], cuts[1:]):
            sub = PackedBatch.from_blob(blob[int(offs[a]):int(offs[b])], offs[a:b + 1] - offs[a])
            r = m.match(sub)
            rec = r.records.copy()
            rec["read"] += a
            parts.append(rec)
        assert np.concatenate(parts).tobytes() == whole.records.tobytes()
        # reverse-complement invariance: same sample / distances, `reverse` flipped
        n_rc = 200_000
        sub_codes = ds.codes[:int(ds.offsets[n_rc])]
        lens = np.diff(ds.offsets[:n_rc + 1])
        start = np.repeat(ds.offsets[:n_rc], lens)
        pos = np.arange(sub_codes.shape[0]) - start
        rc_codes = 3 - sub_codes[start + np.repeat(lens, lens) - 1 - pos]
        rc = m.match(PackedBatch.from_blob(lut[rc_codes].tobytes(), offs[:n_rc + 1]))
    first = whole.records[whole.rec_offset[:n_rc]]
    first_rc = rc.records[rc.rec_offset[:n_rc]]
    single = (np.diff(whole.rec_offset[:n_rc + 1]) == 1) & (np.diff(rc.rec_offset[:n_rc + 1]) == 1)
    full = single & (first["resolution"] == 6)
    assert np.array_equal(first["sample"][full], first_rc["sample"][full])
    assert np.array_equal(first["dist"][full], first_rc["dist"][full])
    assert np.all(first["reverse"][full] != first_rc["reverse"][full])
    assert np.array_equal(first["trim_end"][full] - first["trim_start"][full],
                          first_rc["trim_end"][full] - first_rc["trim_start"][full])
    # truth: a dereplicated full match must name the specimen the read was generated from
    rec = whole.records
    fullrec = rec[rec["resolution"] == 6]
    truth = ds.truth["specimen"][fullrec["read"]]
    agree = np.mean(fullrec["sample"] == truth)
    assert agree > 0.99, agree      # the rest are genuine mis-calls of the reference algorithm at 7 % error
    assert whole.n_matched / ds.n_reads > 0.90


@pytest.mark.parametrize("seed", range(60))
def test_cuda_random_tables_match_live_oracle(seed):
    """Same randomised tables/reads as tests/test_random_tables_hostsim.py, through the CUDA library
    (exercises mixed barcode lengths, k = 0..5, hit-list and group overflow second passes)."""
    from oracle import pipeline as orc
    from test_random_tables_hostsim import make_case
    primers, specimens_rows, reads, k_idx, flags = make_case(seed)
    try:
        tables = orc.Tables(primers, specimens_rows)
    except ValueError:
        pytest.skip("generator produced an invalid table")
    oparams = orc.setup_params(tables, index_edit_distance=k_idx, search_len=flags["search_len"],
                               preorient=not flags["disable_preorient"], prefilter=not flags["disable_prefilter"],
                               trim=flags["trim"], dereplicate=flags["dereplicate"])
    expected, total, matched = orc.process_reads(tables, oparams, reads)
    sp = H.build_specimens(primers, specimens_rows)
    params = MatchParameters(dict(oparams.max_dist_primers), k_idx, flags["search_len"], not flags["disable_preorient"])
    args = H.make_args(flags)
    ops, n, m = process_sequences(H.records(reads), params, sp, args, H.prefilter_for(args))
    assert (n, m) == (total, matched)
    H.assert_ops_equal([H.op_to_dict(o) for o in ops], [H.op_to_dict(o) for o in expected], "seed %d" % seed)


@pytest.mark.parametrize("seed", range(1000, 1016))
def test_cuda_long_primers_match_live_oracle(seed):
    """Primers of 65..300 nt: the warp-cooperative multi-word search (k_primer_long: ballot carry
    lookahead, shuffled Ph/Mh shifts, in-kernel start recovery) against the live oracle."""
    from test_random_tables_hostsim import make_case, run_case
    run_case(*make_case(seed, long_primers=True), tag="long seed %d" % seed, binding="cuda")


@pytest.mark.parametrize("seed", range(12))
def test_cuda_iupac_barcodes_with_prefilter(seed):
    """Barcodes holding IUPAC codes with the Bloom prefilter on (exact per-barcode emulation), through the CUDA library."""
    from test_random_tables_hostsim import make_iupac_barcode_case, run_case
    run_case(*make_iupac_barcode_case(seed), tag="iupac barcode seed %d" % seed, binding="cuda")


@pytest.mark.parametrize("seed", range(8))
def test_cuda_barcode_threshold_beyond_eight(seed):
    """Barcode thresholds 9..12 on 24-30 nt barcodes (general band walk), through the CUDA library."""
    from test_random_tables_hostsim import make_large_k_case, run_case
    run_case(*make_large_k_case(seed), tag="large k seed %d" % seed, binding="cuda")


@pytest.mark.parametrize("seed", range(3))
def test_cuda_two_hundred_primers_three_hundred_pairs(seed):
    """200 canonical primers, 300 pairs, an N barcode with the prefilter on, through the CUDA library."""
    from test_random_tables_hostsim import make_many_primers_case, run_case
    run_case(*make_many_primers_case(seed), tag="many primers seed %d" % seed, binding="cuda")


@pytest.mark.parametrize("cfg,n", [("ont037", 300_000), ("dense", 150_000), ("multipool", 140_000)])
def test_resident_sub_batches_equal_one_lane(cfg, n):
    """upload / run_resident / download with the batch cut into concurrent sub-batches (2, 3, 5 lanes)
    returns exactly the one-lane records, offsets, matched count and work counters; reads on the exact
    4-bit side stream included."""
    ds = synth.CONFIGS[cfg](n_reads=n, seed=99, with_quals=False)
    specimens, params, args = _setup(ds)
    mt = MatchTables(specimens, params, dereplicate="none" if cfg == "dense" else "best")
    codes = np.frombuffer(b"ACGT", dtype=np.uint8)[ds.codes].copy()
    rng = np.random.default_rng(6)
    hits = rng.choice(codes.shape[0], size=codes.shape[0] // 5000, replace=False)
    codes[hits] = np.frombuffer(b"NRYn", dtype=np.uint8)[rng.integers(0, 4, size=hits.shape[0])]
    batch = PackedBatch.from_blob(codes.tobytes(), ds.offsets.astype(np.uint64), clip=ds.search_len)
    with Matcher(mt) as m:
        m.set_resident_split(1)
        m.upload(batch)
        m.run_resident()
        one = m.download()
        work = m.last_work()
        assert m.last_timing()[0] > 0 and sum(m.last_kernel_times().values()) > 0
        for split in (2, 3, 5):
            m.set_resident_split(split)
            m.upload(batch)
            for _ in range(2):
                m.run_resident()
                got = m.download()
                assert got.n_matched == one.n_matched
                assert np.array_equal(got.rec_offset, one.rec_offset)
                assert got.records.tobytes() == one.records.tobytes()
                assert m.last_work() == work
                assert m.last_timing()[0] > 0
        # a pipelined host-buffer call in between does not disturb the resident state machine
        m.set_resident_split(3)
        piped = m.match(batch)
        assert piped.records.tobytes() == one.records.tobytes()
        m.upload(batch)
        m.run_resident()
        assert m.download().records.tobytes() == one.records.tobytes()


def _edge_batches():
    rng = np.random.default_rng(17)
    g = H.load_golden("fixture")
    good = [r[1] for r in g["reads"]]

    def rnd(n):
        return "".join(rng.choice(list("ACGT"), size=n)) if n else ""
    yield "one_read", [good[0]]
    yield "one_empty_read", [""]
    yield "all_empty", [""] * 130
    yield "n127", (good * 4)[:127]
    yield "n128", (good * 4)[:128]
    yield "n129", (good * 4)[:129]
    yield "every_length_0_to_260", [rnd(n) for n in range(261)]
    yield "tiny_and_huge", [rnd(1), good[1], rnd(120_000) + good[2] + rnd(70_000), rnd(2), good[3][:79], good[3][:80], good[3][:81]]
    yield "all_flagged", [s[:10] + "N" + s[11:] for s in good] + ["N" * 300, "acgt" * 50, "RYKM" * 40]
    yield "good_reads_embedded_in_long_reads", [rnd(5000) + s + rnd(5000) for s in good[:10]] + good


@pytest.mark.parametrize("name,reads", list(_edge_batches()), ids=[n for n, _ in _edge_batches()])
@pytest.mark.parametrize("clip", [0, 80])
def test_edge_case_batches_equal_kernel_simulator(name, reads, clip):
    """Degenerate batch shapes through the C ABI: bit-identical records, offsets and per-search detail between
    the CUDA launch and the CPU loop over the same per-thread routines."""
    g = H.load_golden("fixture")
    run = g["runs"]["default"]
    specimens = H.build_specimens(g["primers"], g["specimens"])
    params = H.params_from_run(run, specimens)
    mt = MatchTables(specimens, params, trim="tails")
    batch = PackedBatch(reads, clip=clip)
    with Matcher(mt) as m:
        for detail in (True, False):
            gpu = m.match(batch, detail=detail)
            sim = Matcher(mt, binding=H.hostsim_binding()).match(batch, detail=detail)
            assert gpu.n_matched == sim.n_matched
            assert np.array_equal(gpu.rec_offset, sim.rec_offset)
            assert gpu.records.tobytes() == sim.records.tobytes()
            if detail:
                assert np.array_equal(gpu.primer_hits, sim.primer_hits)
                assert np.array_equal(gpu.endmask, sim.endmask)
                assert np.array_equal(gpu.barcode_hits, sim.barcode_hits)


def test_contexts_are_independent_and_reusable():
    """Two contexts on one device driven from two threads, created and destroyed repeatedly."""
    import threading
    ds = synth.ont037(n_reads=20_000, seed=5, with_quals=False)
    specimens, params, args = _setup(ds)
    mt = MatchTables(specimens, params)
    blob = np.frombuffer(b"ACGT", dtype=np.uint8)[ds.codes].tobytes()
    batch = PackedBatch.from_blob(blob, ds.offsets.astype(np.uint64), clip=ds.search_len)
    with Matcher(mt) as m:
        want = m.match(batch).records.tobytes()
    errors = []

    def work():
        try:
            for _ in range(3):
                with Matcher(mt) as mm:
                    for _ in range(3):
                        assert mm.match(batch).records.tobytes() == want
        except BaseException as e:      # surfaced below
            errors.append(e)
    threads = [threading.Thread(target=work) for _ in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors


@pytest.mark.parametrize("cfg,n,min_agree,min_rate", [("dense", 400_000, 0.95, 0.80), ("multipool", 400_000, 0.98, 0.88),
                                                      ("long", 120_000, 0.98, 0.88)])
def test_properties_at_scale_other_configs(cfg, n, min_agree, min_rate):
    """BASELINE configs 3-5 at six-figure read counts, through size-independent properties: determinism,
    one-shot == pipelined == resident sub-batches, batch-split invariance, and agreement of every
    dereplicated full match with the specimen the generator drew the read from."""
    ds = synth.CONFIGS[cfg](n_reads=n, with_quals=False)
    specimens, params, args = _setup(ds)
    mt = MatchTables(specimens, params)
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    blob = lut[ds.codes].tobytes()
    offs = ds.offsets.astype(np.uint64)
    batch = PackedBatch.from_blob(blob, offs, clip=ds.search_len)
    with Matcher(mt) as m:
        m.set_pipeline_chunk(0)
        whole = m.match(batch)
        assert m.match(batch).records.tobytes() == whole.records.tobytes()            # deterministic
        m.set_pipeline_chunk(32768)
        piped = m.match(batch)
        assert m.last_chunk_count() > 2
        assert piped.records.tobytes() == whole.records.tobytes() and np.array_equal(piped.rec_offset, whole.rec_offset)
        m.set_resident_split(3)
        m.upload(batch)
        m.run_resident()
        assert m.download().records.tobytes() == whole.records.tobytes()
        cut = n // 3 + 17
        parts = []
        for a, b in ((0, cut), (cut, n)):
            r = m.match(PackedBatch.from_blob(blob[int(offs[a]):int(offs[b])], offs[a:b + 1] - offs[a], clip=ds.search_len))
            rec = r.records.copy()
            rec["read"] += a
            parts.append(rec)
        assert np.concatenate(parts).tobytes() == whole.records.tobytes()            # batch-split invariance
    rec = whole.records
    full = rec[rec["resolution"] == 6]
    agree = float(np.mean(full["sample"] == ds.truth["specimen"][full["read"]]))
    assert agree > min_agree, agree
    assert whole.n_matched / n > min_rate, whole.n_matched / n


def _trace_cases():
    import test_trace_events as TT
    return TT.load_cases(), TT.case_ids()


@pytest.mark.parametrize("idx", range(len(_trace_cases()[0])), ids=_trace_cases()[1])
def test_cuda_trace_events_match_reference_stream(idx, tmp_path):
    """The trace narrated from the CUDA library's detail arrays equals the unmodified reference's event stream."""
    import test_trace_events as TT
    case = TT.load_cases()[idx]
    got, _ops = TT.product_events(case, tmp_path, None)
    TT.compare(case, got)


@pytest.mark.parametrize("cfg,n,derep", [("dense", 6000, "none"), ("dense", 6000, "best"), ("multipool", 5000, "none"),
                                         ("ont037", 4000, "best")])
def test_capacity_reruns_on_the_device(cfg, n, derep, monkeypatch):
    """SMX_TEST_TINY_CAPS starts the work-entry, record-pool and compaction buffers far too small, so every
    capacity re-run of the library (entries -> stage 1 again, pool -> selection again, records -> scan +
    compaction again, plus the second selection pass) happens on the device; the result must equal the
    kernel simulator's, one-shot, as resident sub-batches and pipelined."""
    monkeypatch.setenv("SMX_TEST_TINY_CAPS", "1")
    ds = synth.CONFIGS[cfg](n_reads=n, seed=31, with_quals=False)
    specimens, params, args = _setup(ds)
    mt = MatchTables(specimens, params, dereplicate=derep, trim="tails")
    blob = np.frombuffer(b"ACGT", dtype=np.uint8)[ds.codes].tobytes()
    batch = PackedBatch.from_blob(blob, ds.offsets.astype(np.uint64), clip=ds.search_len)
    sim = Matcher(mt, binding=H.hostsim_binding()).match(batch)
    with Matcher(mt) as m:
        for mode in ("one_shot", "pipelined", "again"):
            m.set_pipeline_chunk(1024 if mode == "pipelined" else 0)
            got = m.match(batch)
            assert got.n_matched == sim.n_matched, mode
            assert np.array_equal(got.rec_offset, sim.rec_offset), mode
            assert got.records.tobytes() == sim.records.tobytes(), mode
