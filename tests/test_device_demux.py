"""Demultiplexed output in device memory: smx_demux_device (smx_k_demux.cu) and Matcher.demux_device.

CPU tier: the kernels' work items (smx_out.cuh) run as host loops (tests/demuxsim) with small tiles; for every golden run,
each primary file of the native writer's tree must hold exactly the sequence and quality lines of the group that
DeviceDemux.groups names with its path, and every pool-level file the merge of its full-match outputs in record order.
GPU tier: Matcher.demux_device against the same trees, a config-2-shaped batch against a numpy gather, sliced inputs,
resident splits, several records per read, empty batches, side streams, refusals and interleaved calls."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import helpers as H
from specimux_b200 import _lib, native_io, synth
from specimux_b200.demultiplex import get_matcher
from specimux_b200.engine import DeviceDemux, Matcher, PackedBatch
from specimux_b200.models import MatchParameters
from specimux_b200.orchestration import thresholds_for
from specimux_b200.tables import MatchTables

U64 = 0xFFFFFFFFFFFFFFFF
FULL_MATCH, PARTIAL_FWD, PARTIAL_REV, MULTIPLE, UNKNOWN, DEREP_FULL = 1, 2, 3, 4, 5, 6
_demuxsim = None


@pytest.fixture(scope="module")
def sim(tmp_path_factory):
    """Builds (g++) and loads tests/demuxsim/demuxsim.cpp into a temporary directory."""
    global _demuxsim
    if _demuxsim is None:
        src = os.path.join(H.HERE, "demuxsim", "demuxsim.cpp")
        so = str(tmp_path_factory.mktemp("demuxsim") / "libdemuxsim.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wextra", "-Wno-unused-function", "-o", so, src])
        lib = C.CDLL(so)
        lib.demuxsim_complement.argtypes = [C.c_int]
        vp = C.c_void_p
        lib.demuxsim_run.argtypes = [vp, vp, C.c_uint64, vp, C.c_uint32, vp, C.c_uint64, vp, C.c_uint32, vp, vp, vp, vp,
                                     C.c_uint64, vp, vp, _lib.u64p, _lib.u64p, _lib.u64p]
        _demuxsim = lib
    return _demuxsim


def _counts(tables):
    return np.array([len(tables.specimen_ids), len(tables.b1), len(tables.b2), len(tables.pools), len(tables.primer_names)],
                    dtype=np.uint32)


def sim_demux(sim, tables, bases, quals, seq_off, records, tile_chunks=3, misalign=(0, 0), out_cap=None):
    """demuxsim on host arrays; returns (rc, DeviceDemux with numpy arrays or None, bad key, bytes needed)."""
    bases = np.frombuffer(bases, dtype=np.uint8) if isinstance(bases, bytes) else bases
    quals = np.frombuffer(quals, dtype=np.uint8) if isinstance(quals, bytes) else quals
    seq_off = np.ascontiguousarray(seq_off, dtype=np.uint64)
    records = np.ascontiguousarray(records)
    n = len(records)
    if out_cap is None:                      # the size the index pass reports, as Matcher.demux_device retries
        rc, _dd, _bad, need = sim_demux(sim, tables, bases, quals, seq_off, records, tile_chunks, misalign, 0)
        out_cap = need if rc == 4 else 0
    cap = out_cap
    seq_buf = np.zeros(cap + 16, dtype=np.uint8)
    qual_buf = np.zeros(cap + 16, dtype=np.uint8)
    out_seq, out_qual = seq_buf[misalign[0]:misalign[0] + cap], qual_buf[misalign[1]:misalign[1] + cap]
    order = np.zeros(max(n, 1), dtype=np.uint64)
    out_off = np.zeros(n + 1, dtype=np.uint64)
    gkey = np.zeros(max(n, 1), dtype=np.uint64)
    goff = np.zeros(n + 1, dtype=np.uint64)
    ng, nb, bad = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    counts = _counts(tables)
    rc = sim.demuxsim_run(bases.ctypes.data, quals.ctypes.data if quals is not None else None, len(bases), seq_off.ctypes.data,
                          len(seq_off) - 1, records.ctypes.data, n, counts.ctypes.data, tile_chunks, order.ctypes.data,
                          out_off.ctypes.data, out_seq.ctypes.data, out_qual.ctypes.data, cap, gkey.ctypes.data,
                          goff.ctypes.data, C.byref(ng), C.byref(nb), C.byref(bad))
    if rc:
        return rc, None, bad.value, nb.value
    g, total = ng.value, nb.value
    dd = DeviceDemux(None, out_seq[:total].tobytes(), out_qual[:total].tobytes() if quals is not None else None,
                     out_off.astype(np.int64), order[:n].astype(np.int64), gkey[:g], goff[:g + 1].astype(np.int64), tables)
    return rc, dd, U64, total


def _bytes(x):
    if isinstance(x, (bytes, bytearray)):
        return bytes(x)
    return x.cpu().numpy().tobytes() if hasattr(x, "cpu") else np.asarray(x).tobytes()


class TreeFromGroups:
    """Accumulates what each file of the output tree holds (sequence and quality lines, in order) from demultiplexed
    batches: primary files from DeviceDemux.groups, pool-level files from the full-match outputs in record order."""

    def __init__(self, prefix, fastq=True):
        self.prefix, self.fastq, self.files = prefix, fastq, {}

    def add(self, dd, records):
        seq, off = _bytes(dd.seq), np.asarray(dd.offsets.cpu() if hasattr(dd.offsets, "cpu") else dd.offsets)
        qual = _bytes(dd.qual) if dd.qual is not None else None
        rec_of = np.asarray(dd.record.cpu() if hasattr(dd.record, "cpu") else dd.record)
        line = lambda i: (seq[off[i]:off[i + 1]], qual[off[i]:off[i + 1]] if qual is not None else None)
        pool_level = {}
        for path, a, b in dd.groups(self.prefix, self.fastq):
            self.files.setdefault(path, []).extend(line(i) for i in range(a, b))
            top, pool, _pair, name = path.split("/")
            for i in range(a, b):
                r = records[rec_of[i]]
                if top == "full" and not r["trim_empty"] and r["resolution"] in (FULL_MATCH, DEREP_FULL):
                    pool_level.setdefault("full/%s/%s" % (pool, name), []).append((int(rec_of[i]), line(i)))
        for path, items in pool_level.items():
            self.files.setdefault(path, []).extend(x for _r, x in sorted(items, key=lambda t: t[0]))


def parse_tree(root, fastq=True):
    out = {}
    for d, _s, fs in os.walk(root):
        for f in fs:
            p = os.path.join(d, f)
            lines = open(p, "rb").read().split(b"\n")
            step = 4 if fastq else 2
            out[os.path.relpath(p, root)] = [(lines[k + 1], lines[k + 3] if fastq else None)
                                             for k in range(0, len(lines) - 1, step)]
    return out


def _block_arrays(blk):
    v = blk._view
    n = blk.n_bases()
    bases = C.string_at(v.bases, n) if n else b""
    quals = (C.string_at(v.quals, n) if n else b"") if v.quals else None
    return bases, quals, np.array(blk.seq_off(), dtype=np.uint64)


def _write_fastq(path, reads, fasta=False):
    with open(path, "wb") as fh:
        for rid, seq, qual in reads:
            seq = seq.encode("latin-1") if isinstance(seq, str) else seq
            qual = qual.encode("latin-1") if isinstance(qual, str) else qual
            fh.write(b">%s x\n%s\n" % (rid.encode(), seq) if fasta else b"@%s x\n%s\n+\n%s\n" % (rid.encode(), seq, qual))


def _golden_runs():
    for name in H.golden_names():
        for run in H.load_golden(name)["runs"]:
            yield name, run


def _golden_matcher(name, run_name, binding):
    g = H.load_golden(name)
    run = g["runs"][run_name]
    specimens = H.build_specimens(g["primers"], g["specimens"])
    args = H.make_args(run["flags"])
    params = H.params_from_run(run, specimens)
    return g, params, get_matcher(params, specimens, args, H.prefilter_for(args), 0, binding)


@pytest.mark.parametrize("name,run_name", list(_golden_runs()))
def test_golden_runs_group_like_the_writer_tree(sim, tmp_path, name, run_name):
    g, params, matcher = _golden_matcher(name, run_name, H.hostsim_binding())
    fq = str(tmp_path / "in.fastq")
    _write_fastq(fq, [tuple(r) for r in g["reads"]][:400])
    got = TreeFromGroups("pre_")
    with native_io.FastxReader(fq, True) as rd, native_io.TreeWriter(str(tmp_path / "tree"), "pre_", True, matcher.tables) as wr:
        blk = native_io.ReadBlock()
        k = 0
        while rd.next_block(97, blk).n_reads:
            res = matcher.match(PackedBatch.from_block(blk, clip=params.search_len))
            wr.write(blk, res.records)
            bases, quals, off = _block_arrays(blk)
            rc, dd, _bad, _need = sim_demux(sim, matcher.tables, bases, quals, off, res.records, tile_chunks=1 + k % 3,
                                           misalign=(k % 16, (5 * k) % 16))
            assert rc == 0
            got.add(dd, res.records)
            k += 1
    assert got.files == parse_tree(str(tmp_path / "tree"))


def _tables():
    g = H.load_golden("fixture")
    specimens = H.build_specimens(g["primers"], g["specimens"])
    return MatchTables(specimens, H.params_from_run(g["runs"]["default"], specimens))


def _records(rng, tables, reads_of, n, lengths):
    """n records over the given reads: every resolution, both orientations, trim-empty ones, trims inside, outside and
    across the read ends (negative, past the end, empty)."""
    rec = np.zeros(n, dtype=_lib.RECORD_DTYPE)
    nt = [len(tables.specimen_ids), len(tables.b1), len(tables.b2)]
    for i in range(n):
        r = reads_of(i)
        L = lengths[r]
        res = (FULL_MATCH, PARTIAL_FWD, PARTIAL_REV, MULTIPLE, UNKNOWN, DEREP_FULL)[int(rng.integers(0, 6))]
        samples = nt[0] if res in (FULL_MATCH, MULTIPLE, DEREP_FULL) else nt[1] if res == PARTIAL_FWD else nt[2] if res == PARTIAL_REV else 1
        rec[i]["read"] = r
        rec[i]["sample"] = int(rng.integers(0, samples)) if res != UNKNOWN else -1
        a = int(rng.integers(-L - 3, L + 4)) if rng.random() < 0.3 else int(rng.integers(0, max(L // 3, 1)))
        b = int(rng.integers(-L - 3, L + 4)) if rng.random() < 0.3 else L - int(rng.integers(0, max(L // 3, 1)))
        rec[i]["trim_start"], rec[i]["trim_end"] = a, b
        rec[i]["pool"] = int(rng.integers(-1, len(tables.pools)))
        rec[i]["p1"] = int(rng.integers(-1, len(tables.primer_names)))
        rec[i]["p2"] = int(rng.integers(-1, len(tables.primer_names)))
        rec[i]["dist"] = rng.integers(-1, 4, size=4)
        rec[i]["resolution"] = res
        rec[i]["reverse"] = int(rng.random() < 0.5)
        rec[i]["trim_empty"] = int(rng.random() < 0.1)
    return rec


def _compare_with_writer(sim, tmp_path, tables, reads, records, fasta=False, tiles=(1, 2, 5, 256), misaligns=((0, 0), (1, 15), (7, 3))):
    os.makedirs(str(tmp_path), exist_ok=True)
    path = str(tmp_path / ("in.fasta" if fasta else "in.fastq"))
    _write_fastq(path, reads, fasta)
    root = str(tmp_path / "tree")
    with native_io.FastxReader(path, not fasta) as rd, native_io.TreeWriter(root, "p_", not fasta, tables) as wr:
        blk = rd.next_block(len(reads) + 1)
        assert blk.n_reads == len(reads)
        wr.write(blk, records)
        bases, quals, off = _block_arrays(blk)
    want = parse_tree(root, not fasta)
    for tile_chunks in tiles:
        for mis in misaligns:
            rc, dd, _bad, _need = sim_demux(sim, tables, bases, quals, off, records, tile_chunks, mis)
            assert rc == 0
            got = TreeFromGroups("p_", not fasta)
            got.add(dd, records)
            assert got.files == want, (tile_chunks, mis)
    return dd


def _qual(rng, n):
    return bytes(rng.integers(33, 127, size=n).astype(np.uint8))


def test_every_length_across_tile_boundaries(sim, tmp_path):
    rng = np.random.default_rng(3)
    tables = _tables()
    iupac = list("ACGTRYSWKMBDHVNacgtrykmbdhvnUuX")
    reads = [("r%d" % i, "".join(rng.choice(iupac, size=n)), None) for i, n in enumerate(range(301))]
    reads = [(rid, s, _qual(rng, len(s))) for rid, s, _q in reads]
    records = np.zeros(2 * 301, dtype=_lib.RECORD_DTYPE)
    for i in range(602):                       # whole reads, forward then reversed: outputs of every length 0..300
        r = i % 301
        records[i]["read"], records[i]["sample"], records[i]["resolution"] = r, r % 3, FULL_MATCH
        records[i]["trim_start"], records[i]["trim_end"], records[i]["reverse"] = 0, r, i >= 301
        records[i]["pool"], records[i]["p1"], records[i]["p2"] = 0, 0, 1
    _compare_with_writer(sim, tmp_path, tables, reads, records)
    lengths = [len(s) for _r, s, _q in reads]
    _compare_with_writer(sim, tmp_path / "mixed", tables, reads, _records(rng, tables, lambda i: i % 301, 900, lengths))


def test_long_empty_and_every_byte_reversed(sim, tmp_path):
    rng = np.random.default_rng(4)
    tables = _tables()
    every = bytes(b for b in range(256) if b not in (10, 13))       # every byte a sequence line can hold
    big = bytes(rng.choice(np.frombuffer(b"ACGTNacgtRY", dtype=np.uint8), size=190_000))
    seqs = [b"", big, b"", b"AC" + every + b"GT", every * 3, b"", b"U" * 40 + b"u" * 40]
    reads = [("r%d" % i, s, _qual(rng, len(s))) for i, s in enumerate(seqs)]
    lengths = [len(s) for s in seqs]
    rec = _records(rng, tables, lambda i: i % len(seqs), 70, lengths)
    for i in (1, 3, 4):                               # whole reads reversed, and the big read cut near both ends
        rec[i]["reverse"], rec[i]["trim_empty"], rec[i]["resolution"], rec[i]["sample"] = 1, 0, FULL_MATCH, 0
        rec[i]["trim_start"], rec[i]["trim_end"] = 0, lengths[i]
    rec[8]["read"], rec[8]["trim_start"], rec[8]["trim_end"], rec[8]["reverse"], rec[8]["trim_empty"] = 1, 3, 189_990, 1, 0
    _compare_with_writer(sim, tmp_path, tables, reads, rec, tiles=(1, 3, 256))
    _compare_with_writer(sim, tmp_path / "fasta", tables, reads, rec, fasta=True, tiles=(2,), misaligns=((3, 0),))


def test_complement_is_biopythons_for_every_byte(sim):
    comp = {a: b for a, b in zip("ACGTMRWSYKVHDBXN", "TGCAKYWSRMBDHVXN")}
    comp.update({a.lower(): b.lower() for a, b in comp.items()})
    comp.update(U="A", u="a")
    for ch in range(256):
        assert sim.demuxsim_complement(ch) == ord(comp.get(chr(ch), chr(ch))), ch


def test_validation_names_the_first_bad_item(sim):
    tables = _tables()
    rng = np.random.default_rng(5)
    seqs = [b"ACGT" * 10, b"GG" * 7, b"T" * 30]
    off = np.array([0, 40, 54, 84], dtype=np.uint64)
    bases = b"".join(seqs)
    rec = _records(rng, tables, lambda i: i % 3, 12, [len(s) for s in seqs])
    rec["trim_empty"] = 0
    rc, dd, bad, _ = sim_demux(sim, tables, bases, None, off, rec)
    assert rc == 0 and dd is not None
    bad_off = off.copy()
    bad_off[2] = 30                                          # read 1 ends before it starts
    assert sim_demux(sim, tables, bases, None, bad_off, rec)[:3:2] == (1, (1 << 2) | 1)
    assert sim_demux(sim, tables, bases[:-1], None, off, rec)[:3:2] == (1, (2 << 2) | 2)
    n = _counts(tables)
    for field, value, fault, res in (("read", 3, 1, FULL_MATCH), ("sample", int(n[0]), 2, FULL_MATCH),
                                     ("sample", int(n[1]), 3, PARTIAL_FWD), ("sample", int(n[2]), 4, PARTIAL_REV),
                                     ("pool", int(n[3]), 5, FULL_MATCH), ("p1", int(n[4]), 6, FULL_MATCH),
                                     ("p2", int(n[4]), 7, FULL_MATCH), ("sample", -2, 2, MULTIPLE)):
        edited = rec.copy()
        for i in (7, 9):
            edited[i]["resolution"], edited[i]["sample"] = res, 0
            edited[i][field] = value
        rc, _dd, bad, _ = sim_demux(sim, tables, bases, None, off, edited)
        assert (rc, bad) == (2, (7 << 3) | fault), (field, value)
    # a trim-empty record is never range-checked (it goes to unknown/), as in the writer
    edited = rec.copy()
    edited[4]["trim_empty"], edited[4]["pool"] = 1, 999
    assert sim_demux(sim, tables, bases, None, off, edited)[0] == 0
    # too small a capacity reports the need
    need = sim_demux(sim, tables, bases, None, off, rec)[3]
    assert sim_demux(sim, tables, bases, None, off, rec, out_cap=need - 1)[::3] == (4, need)
    assert sim_demux(sim, tables, bases, None, off, rec, out_cap=need)[0] == 0


def test_no_records_no_groups(sim):
    rc, dd, _bad, total = sim_demux(sim, _tables(), b"ACGT", None, np.array([0, 4], dtype=np.uint64),
                                    np.zeros(0, dtype=_lib.RECORD_DTYPE))
    assert rc == 0 and total == 0 and dd.groups() == [] and list(dd.group_offset) == [0]


def test_no_gpu_means_no_device_demux():
    lib = _lib.load()
    if lib.smx_device_count() > 0:
        pytest.skip("box has a GPU")
    n = C.c_uint64(0)
    rc = lib.smx_demux_device(None, None, None, 0, None, 0, None, 0, None, None, None, None, None, 0, None, None,
                              C.byref(n), C.byref(n), None)
    assert rc == _lib.SMX_ERR_NO_DEVICE


def test_simulator_matcher_refuses_demux_device():
    g = H.load_golden("fixture")
    specimens = H.build_specimens(g["primers"], g["specimens"])
    m = Matcher(MatchTables(specimens, H.params_from_run(g["runs"]["default"], specimens)), binding=H.hostsim_binding())
    with pytest.raises(RuntimeError, match="no device route"):
        m.demux_device(None, None)


# ---------------------------------------------------------------------------------------------------------------------
# GPU tier

def _device_tree(m, params, blk, quals=True, prefix="pre_", fastq=True):
    import torch
    bases, q, off = _block_arrays(blk)
    tb = torch.tensor(np.frombuffer(bases, dtype=np.uint8).copy(), device="cuda")
    tq = torch.tensor(np.frombuffer(q, dtype=np.uint8).copy(), device="cuda") if quals and q is not None else None
    to = torch.tensor(off.astype(np.int64), device="cuda")
    dd = m.demux_device(tb, to, tq)
    got = TreeFromGroups(prefix, fastq)
    got.add(dd, dd.result.to_host().records)
    return dd, got


@pytest.mark.gpu
@pytest.mark.parametrize("name,run_name", list(_golden_runs()))
def test_golden_runs_on_the_device_equal_the_writer_tree(tmp_path, name, run_name):
    g, params, m = _golden_matcher(name, run_name, None)
    fasta = run_name == "default"
    path = str(tmp_path / "in")
    _write_fastq(path, [tuple(r) for r in g["reads"]], fasta)
    root = str(tmp_path / "tree")
    with native_io.FastxReader(path, not fasta) as rd, native_io.TreeWriter(root, "pre_", not fasta, m.tables) as wr:
        blk = rd.next_block(len(g["reads"]) + 1)
        res = m.match(PackedBatch.from_block(blk, clip=params.search_len))
        wr.write(blk, res.records)
        dd, got = _device_tree(m, params, blk, quals=not fasta, fastq=not fasta)
    assert dd.result.to_host().records.tobytes() == res.records.tobytes()
    assert (dd.qual is None) == fasta
    assert got.files == parse_tree(root, not fasta)


def _numpy_demux(tables, codes, quals, offs, records):
    """The expected outputs by plain numpy: stable argsort of the destination key, slices, complement, reversal."""
    n_pools, n_primers = len(tables.pools), len(tables.primer_names)
    offs = offs.astype(np.int64)
    r = records
    res = np.where(r["trim_empty"] != 0, UNKNOWN, r["resolution"]).astype(np.int64)
    live = r["trim_empty"] == 0
    top = np.where(res == UNKNOWN, 2, np.where((res == PARTIAL_FWD) | (res == PARTIAL_REV), 1, 0))
    kind = np.select([np.isin(res, (FULL_MATCH, DEREP_FULL, MULTIPLE)), res == PARTIAL_FWD, res == PARTIAL_REV], [0, 1, 2], 3)
    sample = np.where(kind < 3, r["sample"], 0).astype(np.uint64)
    field = lambda x: np.where(live & (x >= 0), x.astype(np.int64) + 1, 0).astype(np.uint64)
    assert (r["pool"] < n_pools).all() and (r["p1"] < n_primers).all()
    key = ((top.astype(np.uint64) << np.uint64(62)) | (field(r["pool"]) << np.uint64(52)) | (field(r["p1"]) << np.uint64(44)) |
           (field(r["p2"]) << np.uint64(36)) | (kind.astype(np.uint64) << np.uint64(30)) | sample)
    order = np.argsort(key, kind="stable")
    L = (offs[1:] - offs[:-1]).astype(np.int64)[r["read"]]
    s, e = r["trim_start"].astype(np.int64), r["trim_end"].astype(np.int64)
    s = np.clip(np.where(s < 0, s + L, s), 0, L)
    e = np.clip(np.where(e < 0, e + L, e), 0, L)
    e = np.maximum(e, s)
    s, e = np.where(live, s, 0), np.where(live, e, L)
    comp = np.arange(256, dtype=np.uint8)
    for a, b in zip(b"ACGTMRWSYKVHDBXNacgtmrwsykvhdbxnUu", b"TGCAKYWSRMBDHVXNtgcakywsrmbdhvxnAa"):
        comp[a] = b
    seq, qual = [], []
    for i in order:
        a, b = offs[r["read"][i]] + s[i], offs[r["read"][i]] + e[i]
        if r["reverse"][i]:
            a, b = offs[r["read"][i]] + L[i] - e[i], offs[r["read"][i]] + L[i] - s[i]
            seq.append(comp[codes[a:b][::-1]])
            qual.append(quals[a:b][::-1])
        else:
            seq.append(codes[a:b])
            qual.append(quals[a:b])
    lens = np.array([len(x) for x in seq], dtype=np.int64)
    return order, np.concatenate([[0], np.cumsum(lens)]), np.concatenate(seq), np.concatenate(qual), key


def _ont037_exotic(n, seed):
    ds = synth.ont037(n_reads=n, seed=seed, with_quals=False)
    specimens = H.build_specimens(ds.primers, ds.specimens)
    k_idx, k_primers = thresholds_for(specimens)
    mt = MatchTables(specimens, MatchParameters(k_primers, k_idx, ds.search_len, True))
    codes = np.frombuffer(b"ACGT", dtype=np.uint8)[ds.codes].copy()
    rng = np.random.default_rng(seed)
    hits = rng.choice(codes.shape[0], size=codes.shape[0] // 2000, replace=False)
    codes[hits] = np.frombuffer(b"NRYnacgtUuKM", dtype=np.uint8)[rng.integers(0, 12, size=hits.shape[0])]
    quals = rng.integers(33, 75, size=codes.shape[0]).astype(np.uint8)
    return mt, codes, quals, ds.offsets.astype(np.uint64)


def _assert_numpy_equal(dd, mt, codes, quals, offs):
    recs = dd.result.to_host().records
    order, out_off, seq, qual, key = _numpy_demux(mt, codes, quals, offs, recs)
    assert np.array_equal(dd.record.cpu().numpy(), order)
    assert np.array_equal(dd.offsets.cpu().numpy(), out_off)
    assert dd.seq.cpu().numpy().tobytes() == seq.tobytes()
    assert dd.qual.cpu().numpy().tobytes() == qual.tobytes()
    starts = np.flatnonzero(np.concatenate([[True], key[order][1:] != key[order][:-1]])) if len(order) else np.zeros(0, int)
    assert np.array_equal(dd.group_key, key[order][starts])
    assert np.array_equal(dd.group_offset, np.concatenate([starts, [len(order)]]))


@pytest.mark.gpu
def test_config2_shaped_batch_equals_a_numpy_gather():
    import torch
    mt, codes, quals, offs = _ont037_exotic(200_000, 12)
    with Matcher(mt) as m:
        dd = m.demux_device(torch.tensor(codes, device="cuda"), torch.tensor(offs.astype(np.int64), device="cuda"),
                            torch.tensor(quals, device="cuda"))
        assert dd.device_ms[1] >= dd.device_ms[0] > 0
        _assert_numpy_equal(dd, mt, codes, quals, offs)


@pytest.mark.gpu
def test_odd_storage_offsets_splits_and_side_streams():
    import torch
    mt, codes, quals, offs = _ont037_exotic(150_000, 21)
    full_b = torch.tensor(np.concatenate([np.full(1001, 65, np.uint8), codes, np.full(7, 65, np.uint8)]), device="cuda")
    full_q = torch.tensor(np.concatenate([np.full(333, 40, np.uint8), quals, np.full(9, 40, np.uint8)]), device="cuda")
    bases, q = full_b[1001:1001 + len(codes)], full_q[333:333 + len(quals)]
    assert bases.data_ptr() % 16 == 1001 % 16
    offsets = torch.tensor(offs.astype(np.int64), device="cuda")
    with Matcher(mt) as m:
        for split in (1, 3):                            # above the resident split: 150k reads run as sub-batches
            m.set_resident_split(split)
            _assert_numpy_equal(m.demux_device(bases, offsets, q), mt, codes, quals, offs)
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            b2 = torch.zeros_like(bases)
            torch.cuda._sleep(2_000_000)                  # the side stream is busy before the bases are written
            b2.copy_(bases)
            _assert_numpy_equal(m.demux_device(b2, offsets, q), mt, codes, quals, offs)


def _multi_record_batch():
    """Reads that yield several records each (tied specimens / partial barcodes from concatenated amplicons)."""
    g = H.load_golden("fixture")
    run = g["runs"]["default"]
    specimens = H.build_specimens(g["primers"], g["specimens"])
    mt = MatchTables(specimens, H.params_from_run(run, specimens), dereplicate="none")
    reads = [r[1] for r in g["reads"]]
    reads = [a + b for a, b in zip(reads, reads[1:] + reads[:1])] + reads
    return mt, reads


@pytest.mark.gpu
def test_several_records_per_read_take_the_capacity_retry():
    import torch
    mt, reads = _multi_record_batch()
    blob = "".join(reads).encode()
    offs = np.concatenate([[0], np.cumsum([len(r) for r in reads])]).astype(np.uint64)
    codes = np.frombuffer(blob, dtype=np.uint8).copy()
    quals = np.random.default_rng(1).integers(33, 75, size=len(codes)).astype(np.uint8)
    bases, offsets, q = torch.tensor(codes, device="cuda"), torch.tensor(offs.astype(np.int64), device="cuda"), torch.tensor(quals, device="cuda")
    with Matcher(mt) as m:
        dd = m.demux_device(bases, offsets, q)
        recs = dd.result.to_host().records
        assert len(recs) > len(reads) and int(dd.offsets[-1]) > len(codes)    # the first out_cap was too small
        _assert_numpy_equal(dd, mt, codes, quals, offs)
        # the C call with too small a capacity returns the need
        lib = _lib.load()
        n = len(recs)
        t = lambda k, dt=torch.int64: torch.empty(k, dtype=dt, device="cuda")
        order, off, gk, go, seq, qual = t(n), t(n + 1), t(n), t(n + 1), t(len(codes), torch.uint8), t(len(codes), torch.uint8)
        ng, nb = C.c_uint64(0), C.c_uint64(0)
        rc = lib.smx_demux_device(m._ctx, bases.data_ptr(), q.data_ptr(), len(codes), offsets.data_ptr(), len(reads),
                                  dd.result.records.data_ptr(), n, 0, order.data_ptr(), off.data_ptr(), seq.data_ptr(),
                                  qual.data_ptr(), len(codes), gk.data_ptr(), go.data_ptr(), C.byref(ng), C.byref(nb), None)
        assert rc == _lib.SMX_ERR_CAPACITY and nb.value == int(dd.offsets[-1])


@pytest.mark.gpu
def test_no_records_gives_empty_tensors():
    import torch
    g = H.load_golden("fixture")
    specimens = H.build_specimens(g["primers"], g["specimens"])
    mt = MatchTables(specimens, H.params_from_run(g["runs"]["default"], specimens), min_length=100_000)
    reads = [r[1] for r in g["reads"]]
    codes = np.frombuffer("".join(reads).encode(), dtype=np.uint8).copy()
    offs = np.concatenate([[0], np.cumsum([len(r) for r in reads])]).astype(np.int64)
    with Matcher(mt) as m:
        dd = m.demux_device(torch.tensor(codes, device="cuda"), torch.tensor(offs, device="cuda"),
                            torch.tensor(codes, device="cuda"))
        assert dd.result.records.shape[0] == 0
        assert dd.seq.numel() == 0 and dd.qual.numel() == 0 and dd.record.numel() == 0
        assert dd.offsets.cpu().tolist() == [0] and dd.groups() == [] and list(dd.group_offset) == [0]


@pytest.mark.gpu
def test_refusals_leave_the_matcher_usable_and_routes_interleave():
    import torch
    mt, codes, quals, offs = _ont037_exotic(140_000, 8)
    bases, offsets, q = torch.tensor(codes, device="cuda"), torch.tensor(offs.astype(np.int64), device="cuda"), torch.tensor(quals, device="cuda")
    batch = PackedBatch.from_blob(codes.tobytes(), offs, clip=mt.parameters.search_len)
    with Matcher(mt) as m:
        want = m.match(batch)

        def check_usable():
            _assert_numpy_equal(m.demux_device(bases, offsets, q), mt, codes, quals, offs)

        for bad in (q.to(torch.int8), q[:-1], q.view(1, -1), q[::2], q.cpu(), torch.stack([q, q], 1)[:, 0], "x"):
            with pytest.raises(ValueError):
                m.demux_device(bases, offsets, bad)
        check_usable()
        dd = m.demux_device(bases, offsets, q)
        rec = dd.result.records.clone()
        rec[5, 0:4] = torch.tensor(list(int(len(offs) + 10).to_bytes(4, "little")), dtype=torch.uint8)
        edited = type(dd.result)(rec, dd.result.rec_offset, dd.result.n_matched)
        with pytest.raises(_lib.SmxError, match="record 5 names a read past"):
            m._demux(edited, bases, offsets, q)
        check_usable()
        for _ in range(2):
            got = m.match(batch)
            assert got.records.tobytes() == want.records.tobytes()
            check_usable()
            assert m.match_device(bases, offsets).to_host().records.tobytes() == want.records.tobytes()
            check_usable()
