"""Complete output files in device memory: smx_demux_files_device (smx_k_demux.cu) and Matcher.demux_files_device.

CPU tier: the kernels' work items (smx_out.cuh) run as host loops (tests/filesim) with small tiles and misaligned output
buffers; for every golden run, the tree that DeviceFiles.write builds batch after batch must equal the native writer's
tree byte for byte, headers and pool-level copies included, for FASTQ, FASTA and quality-less FASTQ output.  Header edge
cases (titles with odd whitespace, every distance width, unknown names, every resolution) and validation too.
GPU tier: Matcher.demux_files_device against the same trees and the harness, sliced inputs, resident splits, several
records per read, empty batches, side streams, refusals and calls interleaved with the other device routes."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import helpers as H
from specimux_b200 import _lib, native_io
from specimux_b200.engine import DeviceFiles, Matcher, PackedBatch, _file_paths, name_blob
from test_device_demux import (DEREP_FULL, FULL_MATCH, MULTIPLE, PARTIAL_FWD, PARTIAL_REV, UNKNOWN, _golden_matcher,
                               _golden_runs, _multi_record_batch, _ont037_exotic, _qual, _records, _tables)

U64 = 0xFFFFFFFFFFFFFFFF
_filesim = None


@pytest.fixture(scope="module")
def sim(tmp_path_factory):
    """Builds (g++) and loads tests/filesim/filesim.cpp into a temporary directory."""
    global _filesim
    if _filesim is None:
        src = os.path.join(H.HERE, "filesim", "filesim.cpp")
        so = str(tmp_path_factory.mktemp("filesim") / "libfilesim.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wextra", "-Wno-unused-function", "-o", so, src])
        lib = C.CDLL(so)
        vp = C.c_void_p
        lib.filesim_run.argtypes = [vp, vp, C.c_uint64, vp, C.c_uint32, vp, C.c_uint64, vp, vp, C.c_uint64, vp, C.c_uint64, vp,
                                    vp, vp, C.c_int, C.c_uint32, vp, vp, vp, C.c_uint64, vp, vp, _lib.u64p, _lib.u64p,
                                    _lib.u64p, _lib.u64p]
        _filesim = lib
    return _filesim


def _counts(tables):
    return np.array([len(tables.specimen_ids), len(tables.b1), len(tables.b2), len(tables.pools), len(tables.primer_names)],
                    dtype=np.uint32)


def _u8(x):
    if x is None:
        return None
    return np.frombuffer(x, dtype=np.uint8) if isinstance(x, (bytes, bytearray)) else np.ascontiguousarray(x, dtype=np.uint8)


def sim_files(sim, tables, block, records, fastq=True, tile_chunks=3, misalign=0, out_cap=None, name_counts=None,
              title_off=None, name_off=None, prefix="p_"):
    """filesim on a block's arrays (bases, quals, seq_off, titles, title_off); returns (rc, DeviceFiles or None, bad,
    bytes needed)."""
    bases, quals, off, titles, t_off = block
    bases, quals, titles = _u8(bases), _u8(quals), _u8(titles)
    off = np.ascontiguousarray(off, dtype=np.uint64)
    t_off = np.ascontiguousarray(t_off if title_off is None else title_off, dtype=np.uint64)
    blob, n_off, counts = name_blob(tables)
    n_off = np.ascontiguousarray(n_off if name_off is None else name_off, dtype=np.uint64)
    names = np.frombuffer(blob, dtype=np.uint8) if blob else np.zeros(1, np.uint8)
    name_counts = counts if name_counts is None else np.asarray(name_counts, dtype=np.uint32)
    records = np.ascontiguousarray(records)
    n = len(records)
    if out_cap is None:                      # the size the index pass reports, as Matcher.demux_files_device retries
        rc, _f, _bad, need = sim_files(sim, tables, block, records, fastq, tile_chunks, misalign, 0, name_counts, title_off,
                                       name_off, prefix)
        out_cap = need if rc == 4 else 0
    buf = np.zeros(out_cap + 16, dtype=np.uint8)
    out = buf[misalign:misalign + out_cap]
    rec = np.zeros(max(2 * n, 1), dtype=np.uint64)
    out_off = np.zeros(2 * n + 1, dtype=np.uint64)
    fkey = np.zeros(max(2 * n, 1), dtype=np.uint64)
    foff = np.zeros(2 * n + 1, dtype=np.uint64)
    nf, no, nb, bad = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    table_counts = _counts(tables)
    rc = sim.filesim_run(bases.ctypes.data if len(bases) else None, quals.ctypes.data if quals is not None else None, len(bases),
                         off.ctypes.data, len(off) - 1, titles.ctypes.data if len(titles) else None, len(titles),
                         t_off.ctypes.data, records.ctypes.data, n, names.ctypes.data, len(blob), n_off.ctypes.data,
                         table_counts.ctypes.data, name_counts.ctypes.data, 1 if fastq else 0, tile_chunks,
                         rec.ctypes.data, out_off.ctypes.data, out.ctypes.data, out_cap, fkey.ctypes.data, foff.ctypes.data,
                         C.byref(nf), C.byref(no), C.byref(nb), C.byref(bad))
    if rc:
        return rc, None, bad.value, nb.value
    f, k, total = nf.value, no.value, nb.value
    files = DeviceFiles(None, out[:total].copy(), fkey[:f].copy(), foff[:f + 1].astype(np.int64),
                        _file_paths(tables, fkey[:f], prefix, fastq), rec[:k].astype(np.int64), out_off[:k + 1].astype(np.int64))
    return rc, files, U64, total


def block_arrays(blk):
    """(bases, quals or None, seq_off, titles, title_off) of a native_io.ReadBlock."""
    v = blk._view
    n, nr = blk.n_bases(), blk.n_reads
    bases = C.string_at(v.bases, n) if n else b""
    quals = (C.string_at(v.quals, n) if n else b"") if v.quals else None
    t_off = np.ctypeslib.as_array(v.title_off, shape=(nr + 1,)).copy() if nr else np.zeros(1, np.uint64)
    titles = C.string_at(v.titles, int(t_off[-1])) if int(t_off[-1]) else b""
    return bases, quals, np.array(blk.seq_off(), dtype=np.uint64), titles, t_off


def read_tree(root):
    out = {}
    for d, _s, fs in os.walk(root):
        for f in fs:
            p = os.path.join(d, f)
            out[os.path.relpath(p, root)] = open(p, "rb").read()
    return out


def _write_input(path, reads, fasta=False):
    """reads: (title bytes, sequence, qualities)."""
    with open(path, "wb") as fh:
        for title, seq, qual in reads:
            enc = lambda x: x.encode("latin-1") if isinstance(x, str) else x
            fh.write(b">%s\n%s\n" % (enc(title), enc(seq)) if fasta else b"@%s\n%s\n+\n%s\n" % (enc(title), enc(seq), enc(qual)))


# (input is FASTQ, output is FASTQ): FASTQ, FASTA, and FASTQ output of reads without qualities ('I' fill)
MODES = ((True, True), (False, False), (False, True))


@pytest.mark.parametrize("name,run_name", list(_golden_runs()))
def test_golden_runs_build_the_writer_tree(sim, tmp_path, name, run_name):
    g, params, matcher = _golden_matcher(name, run_name, H.hostsim_binding())
    reads = [(("%s x" % r[0]).encode(), r[1], r[2]) for r in g["reads"]][:400]
    for fq_in, fq_out in MODES:
        tag = "%d%d" % (fq_in, fq_out)
        path = str(tmp_path / ("in%s" % tag))
        _write_input(path, reads, not fq_in)
        want, got = str(tmp_path / ("want" + tag)), str(tmp_path / ("got" + tag))
        with native_io.FastxReader(path, fq_in) as rd, native_io.TreeWriter(want, "pre_", fq_out, matcher.tables) as wr:
            blk = native_io.ReadBlock()
            k = 0
            while rd.next_block(97, blk).n_reads:
                res = matcher.match(PackedBatch.from_block(blk, clip=params.search_len))
                wr.write(blk, res.records)
                rc, files, _bad, _need = sim_files(sim, matcher.tables, block_arrays(blk), res.records, fq_out,
                                                   tile_chunks=1 + k % 3, misalign=(5 * k) % 16, prefix="pre_")
                assert rc == 0
                files.write(got)
                k += 1
        assert read_tree(got) == read_tree(want), (fq_in, fq_out)


def _compare_with_writer(sim, tmp_path, tables, reads, records, fastq_in=True, fastq_out=True, tiles=(1, 2, 5, 256),
                         misaligns=(0, 1, 7, 15)):
    os.makedirs(str(tmp_path), exist_ok=True)
    path = str(tmp_path / "in")
    _write_input(path, reads, not fastq_in)
    want = str(tmp_path / "want")
    with native_io.FastxReader(path, fastq_in) as rd, native_io.TreeWriter(want, "p_", fastq_out, tables) as wr:
        blk = rd.next_block(len(reads) + 1)
        assert blk.n_reads == len(reads)
        wr.write(blk, records)
        arrays = block_arrays(blk)
    want_tree = read_tree(want)
    for tile_chunks in tiles:
        for mis in misaligns:
            rc, files, _bad, _need = sim_files(sim, tables, arrays, records, fastq_out, tile_chunks, mis)
            assert rc == 0
            got = str(tmp_path / ("got_%d_%d" % (tile_chunks, mis)))
            files.write(got)
            assert read_tree(got) == want_tree, (tile_chunks, mis)
    return files, arrays


TITLES = [b"", b"   lead x", b"\ttab\tsep", b"id\x1cfs", b"\xc2\xa0nbsp id", b"id\xc2\x85nel", b"id\xe2\x80\x80en quad",
          b"\xe2\x80\x8aid", b"id\xe2\x80\xa8ls", b"id\xe2\x80\xafnnbsp", b"id\xe2\x81\x9fmmsp", b"\xe3\x80\x80ideo x",
          b"id\xe1\x9a\x80ogham", b"caf\xc3\xa9 \xc3\xa9t\xc3\xa9", b"id\xe2\x80\x8bzwsp-not-space", b"\xc2", b"end\xe2\x80",
          b"plain_id desc text", b" " * 5, b"x" * 300]


def test_header_edge_cases_match_the_writer(sim, tmp_path):
    rng = np.random.default_rng(7)
    tables = _tables()
    iupac = list("ACGTRYSWKMBDHVNacgtUu")
    seqs = ["".join(rng.choice(iupac, size=int(n))) for n in rng.integers(0, 200, size=len(TITLES))]
    reads = [(t, s, _qual(rng, len(s))) for t, s in zip(TITLES, seqs)]
    lengths = [len(s) for s in seqs]
    rec = _records(rng, tables, lambda i: i % len(reads), 240, lengths)
    widths = np.array([-1, 0, 9, 10, 99, 100, 127, -128], dtype=np.int8)
    rec["dist"] = widths[rng.integers(0, len(widths), size=(len(rec), 4))]
    for i, res in enumerate((FULL_MATCH, PARTIAL_FWD, PARTIAL_REV, MULTIPLE, UNKNOWN, DEREP_FULL)):
        rec[i]["resolution"], rec[i]["sample"], rec[i]["trim_empty"] = res, 0 if res != UNKNOWN else -1, 0
        rec[i]["pool"], rec[i]["p1"], rec[i]["p2"] = -1, -1, -1           # unknown pool and primers
        rec[i]["reverse"] = i % 2
    for fq_in, fq_out in MODES:
        _compare_with_writer(sim, tmp_path / ("m%d%d" % (fq_in, fq_out)), tables, reads, rec, fq_in, fq_out,
                             tiles=(1, 3), misaligns=(0, 9))


def test_every_length_across_tile_boundaries(sim, tmp_path):
    rng = np.random.default_rng(3)
    tables = _tables()
    iupac = list("ACGTRYSWKMBDHVNacgtrykmbdhvnUuX")
    reads = [(b"r%d" % i, "".join(rng.choice(iupac, size=n)), None) for i, n in enumerate(range(161))]
    reads = [(t, s, _qual(rng, len(s))) for t, s, _q in reads]
    records = np.zeros(2 * 161, dtype=_lib.RECORD_DTYPE)
    for i in range(322):                       # whole reads, forward then reversed, full matches with pool-level copies
        r = i % 161
        records[i]["read"], records[i]["sample"], records[i]["resolution"] = r, r % 3, FULL_MATCH
        records[i]["trim_start"], records[i]["trim_end"], records[i]["reverse"] = 0, r, i >= 161
        records[i]["pool"], records[i]["p1"], records[i]["p2"] = 0, 0, 1
    files, _ = _compare_with_writer(sim, tmp_path, tables, reads, records)
    assert any(p.startswith("full/") and p.count("/") == 2 for p in files.paths)      # pool-level copies exist
    lengths = [len(s) for _t, s, _q in reads]
    _compare_with_writer(sim, tmp_path / "mixed", tables, reads, _records(rng, tables, lambda i: i % 161, 500, lengths),
                         tiles=(1, 2, 256), misaligns=(0, 13))


def test_long_read_and_every_byte(sim, tmp_path):
    rng = np.random.default_rng(4)
    tables = _tables()
    every = bytes(b for b in range(256) if b not in (10, 13, 43, 62, 64))   # bytes a sequence line can hold
    big = bytes(rng.choice(np.frombuffer(b"ACGTNacgtRY", dtype=np.uint8), size=190_000))
    seqs = [b"", big, b"AC" + every + b"GT", b"U" * 40 + b"u" * 40]
    reads = [(b"r%d desc" % i, s, _qual(rng, len(s))) for i, s in enumerate(seqs)]
    lengths = [len(s) for s in seqs]
    rec = _records(rng, tables, lambda i: i % len(seqs), 40, lengths)
    for i in (1, 2):
        rec[i]["reverse"], rec[i]["trim_empty"], rec[i]["resolution"], rec[i]["sample"] = 1, 0, FULL_MATCH, 0
        rec[i]["trim_start"], rec[i]["trim_end"] = 0, lengths[i]
    for fq_in, fq_out in MODES:
        _compare_with_writer(sim, tmp_path / ("m%d%d" % (fq_in, fq_out)), tables, reads, rec, fq_in, fq_out,
                             tiles=(1, 256), misaligns=(3,))


def _small_block():
    seqs = [b"ACGT" * 10, b"GG" * 7, b"T" * 30]
    titles = [b"a x", b"  b", b"c"]
    off = np.array([0, 40, 54, 84], dtype=np.uint64)
    t_off = np.array([0, 3, 6, 7], dtype=np.uint64)
    return b"".join(seqs), None, off, b"".join(titles), t_off


def test_validation_names_the_first_bad_item(sim):
    tables = _tables()
    rng = np.random.default_rng(5)
    blk = _small_block()
    rec = _records(rng, tables, lambda i: i % 3, 12, [40, 14, 30])
    rec["trim_empty"] = 0
    assert sim_files(sim, tables, blk, rec)[0] == 0
    bases, quals, off, titles, t_off = blk
    bad_off = off.copy()
    bad_off[2] = 30                                          # read 1 ends before it starts
    assert sim_files(sim, tables, (bases, quals, bad_off, titles, t_off), rec)[:3:2] == (1, (1 << 2) | 1)
    bad_t = t_off.copy()
    bad_t[2] = 2                                             # title 1 ends before it starts
    assert sim_files(sim, tables, blk, rec, title_off=bad_t)[:3:2] == (3, (1 << 2) | 1)
    assert sim_files(sim, tables, (bases, quals, off, titles[:-1], t_off), rec)[:3:2] == (3, (2 << 2) | 2)
    _blob, n_off, counts = name_blob(tables)
    bad_n = n_off.copy()
    bad_n[3] = bad_n[2] - 1 if bad_n[2] else U64             # name 2 ends before it starts
    assert sim_files(sim, tables, blk, rec, name_off=bad_n)[:3:2] == (5, (2 << 2) | 1)
    for table in range(5):
        wrong = counts.copy()
        wrong[table] += 1
        assert sim_files(sim, tables, blk, rec, name_counts=wrong)[:3:2] == (6, table)
    n = _counts(tables)
    for field, value, fault, res in (("read", 3, 1, FULL_MATCH), ("sample", int(n[0]), 2, FULL_MATCH),
                                     ("sample", int(n[1]), 3, PARTIAL_FWD), ("sample", int(n[2]), 4, PARTIAL_REV),
                                     ("pool", int(n[3]), 5, FULL_MATCH), ("p1", int(n[4]), 6, FULL_MATCH),
                                     ("p2", int(n[4]), 7, FULL_MATCH)):
        edited = rec.copy()
        for i in (7, 9):
            edited[i]["resolution"], edited[i]["sample"] = res, 0
            edited[i][field] = value
        assert sim_files(sim, tables, blk, edited)[:3:2] == (2, (7 << 3) | fault), (field, value)
    need = sim_files(sim, tables, blk, rec)[3]
    assert sim_files(sim, tables, blk, rec, out_cap=need - 1)[::3] == (4, need)
    assert sim_files(sim, tables, blk, rec, out_cap=need)[0] == 0


def test_no_records_no_files(sim, tmp_path):
    rc, files, _bad, total = sim_files(sim, _tables(), _small_block(), np.zeros(0, dtype=_lib.RECORD_DTYPE))
    assert rc == 0 and total == 0 and files.paths == [] and list(files.file_offset) == [0]
    files.write(str(tmp_path / "t"))
    assert not os.path.exists(str(tmp_path / "t"))


def test_no_gpu_means_no_device_files():
    lib = _lib.load()
    if lib.smx_device_count() > 0:
        pytest.skip("box has a GPU")
    n = C.c_uint64(0)
    counts = np.zeros(5, dtype=np.uint32)
    rc = lib.smx_demux_files_device(None, None, None, 0, None, 0, None, 0, None, None, 0, None, 0, None,
                                    _lib.ptr(counts, _lib.u32p), 1, None, None, None, None, 0, None, None, C.byref(n),
                                    C.byref(n), C.byref(n), None)
    assert rc == _lib.SMX_ERR_NO_DEVICE


def test_simulator_matcher_refuses_demux_files_device():
    m = Matcher(_tables(), binding=H.hostsim_binding())
    with pytest.raises(RuntimeError, match="no device route"):
        m.demux_files_device(None, None, None, None)


# ---------------------------------------------------------------------------------------------------------------------
# GPU tier

def _tensors(arrays, device="cuda"):
    import torch
    bases, quals, off, titles, t_off = arrays
    t = lambda x: torch.tensor(np.frombuffer(x, dtype=np.uint8).copy() if isinstance(x, bytes) else x, device=device)
    return (t(bases), t(quals) if quals is not None else None, torch.tensor(off.astype(np.int64), device=device), t(titles),
            torch.tensor(t_off.astype(np.int64), device=device))


@pytest.mark.gpu
@pytest.mark.parametrize("name,run_name", list(_golden_runs()))
def test_golden_runs_on_the_device_build_the_writer_tree(tmp_path, name, run_name):
    g, params, m = _golden_matcher(name, run_name, None)
    fq = run_name != "default"
    reads = [(("%s x" % r[0]).encode(), r[1], r[2]) for r in g["reads"]]
    path = str(tmp_path / "in")
    _write_input(path, reads, not fq)
    want, got = str(tmp_path / "want"), str(tmp_path / "got")
    with native_io.FastxReader(path, fq) as rd, native_io.TreeWriter(want, "pre_", fq, m.tables) as wr:
        blk = native_io.ReadBlock()
        while rd.next_block(97, blk).n_reads:
            res = m.match(PackedBatch.from_block(blk, clip=params.search_len))
            wr.write(blk, res.records)
            b, q, o, t, to = _tensors(block_arrays(blk))
            files = m.demux_files_device(b, o, t, to, q, prefix="pre_", fastq=fq)
            assert files.result.to_host().records.tobytes() == res.records.tobytes()
            files.write(got)
    assert read_tree(got) == read_tree(want)


def _exotic_block(n, seed):
    mt, codes, quals, offs = _ont037_exotic(n, seed)
    titles = b"".join(b"read_%d runid=abc\tch=%d" % (i, i % 512) for i in range(n))
    lens = np.array([len(b"read_%d runid=abc\tch=%d" % (i, i % 512)) for i in range(n)], dtype=np.uint64)
    t_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    return mt, (codes, quals, offs, titles, t_off)


def _assert_sim_equal(sim, files, mt, arrays, fastq=True):
    recs = files.result.to_host().records
    rc, want, _bad, _need = sim_files(sim, mt, arrays, recs, fastq, tile_chunks=256, prefix="")
    assert rc == 0
    assert files.data.cpu().numpy().tobytes() == want.data.tobytes()
    assert np.array_equal(files.file_key, want.file_key) and np.array_equal(files.file_offset, want.file_offset)
    assert files.paths == want.paths
    assert np.array_equal(files.record.cpu().numpy(), want.record)
    assert np.array_equal(files.offsets.cpu().numpy(), want.offsets)


@pytest.mark.gpu
def test_config2_shaped_batch_equals_the_harness(sim):
    import torch
    mt, arrays = _exotic_block(200_000, 12)
    with Matcher(mt) as m:
        b, q, o, t, to = _tensors(arrays)
        files = m.demux_files_device(b, o, t, to, q)
        assert files.device_ms[1] >= files.device_ms[0] > 0
        assert any(p.startswith("full/") and p.count("/") == 2 for p in files.paths)
        _assert_sim_equal(sim, files, mt, arrays)
        nq = m.demux_files_device(b, o, t, to)                     # FASTQ without qualities: 'I'
        _assert_sim_equal(sim, nq, mt, (arrays[0], None) + arrays[2:])
        fa = m.demux_files_device(b, o, t, to, q, fastq=False)
        _assert_sim_equal(sim, fa, mt, arrays, fastq=False)


@pytest.mark.gpu
def test_odd_storage_offsets_splits_and_side_streams(sim):
    import torch
    mt, arrays = _exotic_block(150_000, 21)
    codes, quals, offs, titles, t_off = arrays
    pad = lambda x, a, b, v: torch.tensor(np.concatenate([np.full(a, v, np.uint8), np.frombuffer(x, np.uint8) if isinstance(x, bytes) else x,
                                                          np.full(b, v, np.uint8)]), device="cuda")[a:a + len(x)]
    bases, q, t = pad(codes, 1001, 7, 65), pad(quals, 333, 9, 40), pad(titles, 77, 3, 32)
    assert bases.data_ptr() % 16 == 1001 % 16 and t.data_ptr() % 16 == 77 % 16
    o, to = torch.tensor(offs.astype(np.int64), device="cuda"), torch.tensor(t_off.astype(np.int64), device="cuda")
    with Matcher(mt) as m:
        for split in (1, 3):
            m.set_resident_split(split)
            _assert_sim_equal(sim, m.demux_files_device(bases, o, t, to, q), mt, arrays)
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            t2 = torch.zeros_like(t)
            torch.cuda._sleep(2_000_000)                  # the side stream is busy before the titles are written
            t2.copy_(t)
            _assert_sim_equal(sim, m.demux_files_device(bases, o, t2, to, q), mt, arrays)


@pytest.mark.gpu
def test_several_records_per_read_take_the_capacity_retry(sim):
    import torch
    mt, reads = _multi_record_batch()
    blob = "".join(reads).encode()
    offs = np.concatenate([[0], np.cumsum([len(r) for r in reads])]).astype(np.uint64)
    titles = b"".join(b"r%d" % i for i in range(len(reads)))
    t_off = np.concatenate([[0], np.cumsum([len(b"r%d" % i) for i in range(len(reads))])]).astype(np.uint64)
    quals = np.random.default_rng(1).integers(33, 75, size=len(blob)).astype(np.uint8)
    arrays = (np.frombuffer(blob, np.uint8).copy(), quals, offs, titles, t_off)
    b, q, o, t, to = _tensors(arrays)
    with Matcher(mt) as m:
        files = m.demux_files_device(b, o, t, to, q)
        recs = files.result.to_host().records
        assert len(recs) > len(reads)
        _assert_sim_equal(sim, files, mt, arrays)
        # the C call with too small a capacity returns the need
        lib = _lib.load()
        n = len(recs)
        blob_n, n_off, counts = name_blob(mt)
        nb_t = torch.tensor(np.frombuffer(blob_n, np.uint8).copy(), device="cuda")
        no_t = torch.tensor(n_off.astype(np.int64), device="cuda")
        e = lambda k, dt=torch.int64: torch.empty(k, dtype=dt, device="cuda")
        rec, off, fk, fo, out = e(2 * n), e(2 * n + 1), e(2 * n), e(2 * n + 1), e(100, torch.uint8)
        nf, no, nb = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        call = lambda cnt, t_off_ptr: lib.smx_demux_files_device(
            m._ctx, b.data_ptr(), q.data_ptr(), b.numel(), o.data_ptr(), len(reads), t.data_ptr(), t.numel(), t_off_ptr,
            files.result.records.data_ptr(), n, nb_t.data_ptr(), nb_t.numel(), no_t.data_ptr(), _lib.ptr(cnt, _lib.u32p), 1, 0,
            rec.data_ptr(), off.data_ptr(), out.data_ptr(), 100, fk.data_ptr(), fo.data_ptr(), C.byref(nf), C.byref(no),
            C.byref(nb), None)
        assert call(counts, to.data_ptr()) == _lib.SMX_ERR_CAPACITY and nb.value == files.data.numel()
        wrong = counts.copy()
        wrong[3] += 1
        assert call(wrong, to.data_ptr()) == _lib.SMX_ERR_ARG and "names of pools" in lib.smx_last_error().decode()
        bad_to = to.clone()
        bad_to[4] = bad_to[3] - 1
        assert call(counts, bad_to.data_ptr()) == _lib.SMX_ERR_ARG and "title 3 offsets descend" in lib.smx_last_error().decode()
        _assert_sim_equal(sim, m.demux_files_device(b, o, t, to, q), mt, arrays)


@pytest.mark.gpu
def test_no_records_gives_no_files(tmp_path):
    import torch
    g = H.load_golden("fixture")
    specimens = H.build_specimens(g["primers"], g["specimens"])
    from specimux_b200.tables import MatchTables
    mt = MatchTables(specimens, H.params_from_run(g["runs"]["default"], specimens), min_length=100_000)
    reads = [r[1] for r in g["reads"]]
    codes = np.frombuffer("".join(reads).encode(), dtype=np.uint8).copy()
    offs = np.concatenate([[0], np.cumsum([len(r) for r in reads])]).astype(np.uint64)
    arrays = (codes, codes, offs, b"t" * len(reads), np.arange(len(reads) + 1, dtype=np.uint64))
    with Matcher(mt) as m:
        files = m.demux_files_device(*[_tensors(arrays)[k] for k in (0, 2, 3, 4, 1)])
        assert files.result.records.shape[0] == 0
        assert files.data.numel() == 0 and files.record.numel() == 0 and files.paths == []
        assert files.offsets.cpu().tolist() == [0] and list(files.file_offset) == [0]
        files.write(str(tmp_path / "t"))
        assert not os.path.exists(str(tmp_path / "t"))


@pytest.mark.gpu
def test_refusals_leave_the_matcher_usable_and_routes_interleave(sim):
    import torch
    mt, arrays = _exotic_block(140_000, 8)
    b, q, o, t, to = _tensors(arrays)
    batch = PackedBatch.from_blob(arrays[0].tobytes(), arrays[2], clip=mt.parameters.search_len)
    with Matcher(mt) as m:
        want = m.match(batch)

        def check_usable():
            _assert_sim_equal(sim, m.demux_files_device(b, o, t, to, q), mt, arrays)

        for bad in (t.to(torch.int8), t.view(1, -1), t[::2], t.cpu(), "x"):
            with pytest.raises(ValueError):
                m.demux_files_device(b, o, bad, to, q)
        for bad in (to.to(torch.int32), to[:-1], to.cpu()):
            with pytest.raises(ValueError):
                m.demux_files_device(b, o, t, bad, q)
        with pytest.raises(ValueError):
            m.demux_files_device(b, o, t, to, q[:-1])
        check_usable()
        files = m.demux_files_device(b, o, t, to, q)
        rec = files.result.records.clone()
        rec[5, 0:4] = torch.tensor(list(int(len(arrays[2]) + 10).to_bytes(4, "little")), dtype=torch.uint8)
        edited = type(files.result)(rec, files.result.rec_offset, files.result.n_matched)
        with pytest.raises(_lib.SmxError, match="record 5 names a read past"):
            m._demux_files(edited, b, o, t, to, q, "", True)
        bad_to = to.clone()
        bad_to[-1] = t.numel() + 1
        with pytest.raises(_lib.SmxError, match="title %d ends past n_title_bytes" % (len(arrays[2]) - 2)):
            m.demux_files_device(b, o, t, bad_to, q)
        check_usable()
        for _ in range(2):
            assert m.match(batch).records.tobytes() == want.records.tobytes()
            check_usable()
            assert m.match_device(b, o).to_host().records.tobytes() == want.records.tobytes()
            dd = m.demux_device(b, o, q)
            assert dd.seq.numel() > 0
            check_usable()
