"""specimine on device files: smx_mine_device (smx_k_mine_device.cu, k_hw_best over HwSpans) and Matcher.mine_device.

CPU tier: the identity text ('%.2f'), the search limit and the pass test against Python; the rewritten title against
specimine's own rewrite; the kernels' work items as host loops (tests/minesim) with a stand-in for k_hw_best (the
exact-ratio argmin over oracle distances) on DeviceFiles built by tests/filesim -- their `.mined` bytes must equal
specimine.mine_files, run with the same stand-in on the tree DeviceFiles.write builds, for golden runs and a synthetic
mining batch under every flag set and -P prefix.  GPU tier: Matcher.mine_device against mine_files with the real grouped
kernel, against the harness, refusals, side streams and batches without pool-level files."""
import ctypes as C
import glob
import os
import subprocess
from fractions import Fraction

import numpy as np
import pytest

import helpers as H
from specimux_b200 import _lib, seqio, specimine, synth
from specimux_b200.engine import DeviceMined, Matcher, PackedBatch, mine_plan
from specimux_b200.models import MatchParameters
from specimux_b200.tables import MatchTables
from test_device_demux import _golden_matcher, _golden_runs
from test_device_files import TITLES, read_tree, sim_files
from test_specimine_grouped import FLAG_SETS, _host_best_grouped, _oracle_distance

_libs = {}


def _build(name):
    if name not in _libs:
        src = os.path.join(H.HERE, name, name + ".cpp")
        so = os.path.join(_tmpdir(), "lib%s.so" % name)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wextra", "-Wno-unused-function",
                               "-o", so, src])
        _libs[name] = C.CDLL(so)
    return _libs[name]


def _tmpdir():
    import tempfile
    d = _libs.get("_dir")
    if d is None:
        d = _libs["_dir"] = tempfile.mkdtemp(prefix="minesim")
    return d


@pytest.fixture(scope="module")
def fsim():
    lib = _build("filesim")
    vp = C.c_void_p
    lib.filesim_run.argtypes = [vp, vp, C.c_uint64, vp, C.c_uint32, vp, C.c_uint64, vp, vp, C.c_uint64, vp, C.c_uint64, vp,
                                vp, vp, C.c_int, C.c_uint32, vp, vp, vp, C.c_uint64, vp, vp, _lib.u64p, _lib.u64p,
                                _lib.u64p, _lib.u64p]
    return lib


class HwItem(C.Structure):
    _fields_ = [("pat", C.c_uint32), ("rank", C.c_uint32), ("e_lo", C.c_uint64), ("n", C.c_uint32), ("pad", C.c_uint32)]


SEARCH = C.CFUNCTYPE(None, C.POINTER(HwItem), C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32),
                     C.POINTER(C.c_int32), C.POINTER(C.c_uint32), C.c_uint64, C.POINTER(C.c_ulonglong))


@pytest.fixture(scope="module")
def msim():
    lib = _build("minesim")
    vp = C.c_void_p
    lib.minesim_run.argtypes = [vp, C.c_uint64, vp, C.c_uint64, vp, C.c_uint64, C.c_uint32, vp, vp, vp, vp, C.c_uint32, vp,
                                C.c_double, SEARCH, vp, C.c_uint64, C.c_uint64, vp, vp, vp, vp, _lib.u64p, _lib.u64p,
                                _lib.u64p]
    lib.minesim_fmt2_table.argtypes = [C.c_uint32, vp]
    lib.minesim_fmt2_table.restype = None
    lib.minesim_k.argtypes = [C.c_uint64, C.c_double]
    lib.minesim_k.restype = C.c_int32
    lib.minesim_pass.argtypes = [C.c_uint64, C.c_uint64, C.c_double]
    lib.minesim_title.argtypes = [C.c_char_p, C.c_uint64, C.c_int, C.c_char_p, C.c_uint32, vp]
    lib.minesim_title.restype = C.c_uint64
    return lib


# ---------------------------------------------------------------------------------------------------------------------
# the record text

def test_identity_text_is_pythons_for_every_ratio(msim):
    M = 4096
    buf = np.zeros(((M + 1) * (M + 2) // 2) * 8, dtype=np.uint8)
    msim.minesim_fmt2_table(M, buf.ctypes.data)
    got = buf.reshape(-1, 8)
    for m in range(1, M + 1):
        base = m * (m + 1) // 2
        want = b"".join(("%.2f" % (1 - d / m)).encode().ljust(8, b"\0") for d in range(m + 1))
        assert got[base:base + m + 1].tobytes() == want, m


MIN_IDENTITIES = (0.5, 0.75, 0.85, 0.9, 1 / 3, 1.0)


@pytest.mark.parametrize("mi", MIN_IDENTITIES)
def test_search_limit_and_pass_test_are_pythons(msim, mi):
    for m in range(0, 4097):
        assert msim.minesim_k(m, mi) == int(m * (1 - mi)), m
    for m in list(range(1, 400)) + list(range(4000, 4097)):
        for d in range(m + 1):
            ident = 1 - (d / m)
            assert msim.minesim_pass(d, m, mi) == int(ident >= mi and ident > 0), (m, d)


def _python_title(title: bytes, ident: float, kind: str) -> bytes:
    text = title.decode("utf-8", "surrogateescape").rstrip()
    rec = seqio.SeqRecord("ACGT", (text.split(None, 1) or [""])[0], text, "IIII")
    mined = specimine._rewrite_mined([rec], np.array([ident]), kind)[0]
    return ("@%s\n" % specimine.fastq_title(mined)).encode("utf-8", "surrogateescape")


def test_title_rewrite_is_specimines(msim):
    headers = [b"read_1 0,1,2,3 pool=ITS primers=ITS1F+ITS4 barcode_rev_ACGT", b"x X,X,X,X pool=unknown primers=unknown+unknown unknown"]
    out = C.create_string_buffer(4096)
    for title in TITLES + headers + [b"trailing \t ", b"id \xe2\x80\x80", b"\t"]:
        for ident, kind in ((0.855, "reverse"), (1.0, "forward"), (0.125, "reverse")):
            b = ("%.2f" % ident).encode()
            n = msim.minesim_title(title, len(title), kind == "reverse", b, len(b), out)
            assert out.raw[:n] == _python_title(title, ident, kind), (title, ident)


# ---------------------------------------------------------------------------------------------------------------------
# the harness against specimine.mine_files

def _search_standin(data):
    """k_hw_best's keys from oracle distances: per entry the exact-ratio argmin (ties to the first rank) over the items'
    patterns, as test_specimine_grouped's stand-in selects."""
    def run(items, n_items, beg, ln, k, ent_txt, n_ent, keys):
        best = {}
        for i in range(n_items):
            it = items[i]
            p = data[beg[it.pat]:beg[it.pat] + ln[it.pat]].tobytes().decode("latin-1")
            m = len(p)
            for e in range(it.e_lo, it.e_lo + it.n):
                t_out = ent_txt[e]
                t = data[beg[t_out]:beg[t_out] + ln[t_out]].tobytes().decode("latin-1")
                d = m if not t else _oracle_distance(p, k[it.pat], t)
                if d == -1:
                    continue
                cand = (Fraction(d, m), it.rank, d, m)
                if e not in best or cand[:2] < best[e][:2]:
                    best[e] = cand
        for e, (_r, rank, d, m) in best.items():
            keys[e] = (((d << 40) // m) << 23) | rank
    return SEARCH(run)


def mine_sim(msim, files, index, partial_forward=False, no_partial_reverse=False, min_identity=0.85, out_cap=None):
    """minesim over a DeviceFiles whose arrays are numpy (sim_files); returns (rc, DeviceMined or None, bad)."""
    jobs, skipped, (gf, gk, gpo, gp, mg), _distinct = mine_plan(files, index, partial_forward, no_partial_reverse)
    data = np.ascontiguousarray(files.data, dtype=np.uint8)
    out_off = np.ascontiguousarray(files.offsets, dtype=np.uint64)
    file_off = np.ascontiguousarray(files.file_offset, dtype=np.uint64)
    search = _search_standin(data)
    nr, nb, bad = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    caps = (0, 0) if out_cap is None else out_cap
    for attempt in range(2):
        out = np.zeros(caps[0] + 1, dtype=np.uint8)
        part, win = np.zeros(caps[1] + 1, dtype=np.int64), np.zeros(caps[1] + 1, dtype=np.int64)
        dist = np.zeros(caps[1] + 1, dtype=np.int32)
        moff = np.zeros(len(jobs) + 1, dtype=np.uint64)
        rc = msim.minesim_run(data.ctypes.data, len(data), out_off.ctypes.data, len(out_off) - 1, file_off.ctypes.data,
                              len(file_off) - 1, len(gf), gf.ctypes.data, gk.ctypes.data, gpo.ctypes.data, gp.ctypes.data,
                              len(jobs), mg.ctypes.data, min_identity, search, out.ctypes.data, caps[0], caps[1],
                              moff.ctypes.data, part.ctypes.data, win.ctypes.data, dist.ctypes.data, C.byref(nr),
                              C.byref(nb), C.byref(bad))
        if rc == 4 and out_cap is None and attempt == 0:
            caps = (nb.value, nr.value)
            continue
        break
    if rc:
        return rc, None, bad.value
    r = nr.value
    return 0, DeviceMined(out[:nb.value], moff.astype(np.int64), [p + ".mined" for p, _ in jobs], part[:r], win[:r],
                          dist[:r], skipped), bad.value


def _write_index(path, specimens):
    with open(path, "w") as fh:
        fh.write("SampleID\tPrimerPool\tFwIndex\tFwPrimer\tRvIndex\tRvPrimer\n")
        for row in specimens:
            fh.write("\t".join(row) + "\n")


def _flags(flags):
    pf = "--partial-forward" in flags
    npr = "--no-partial-reverse" in flags
    mi = float(flags[flags.index("--min-identity") + 1]) if "--min-identity" in flags else 0.85
    return pf, npr, mi


def _sorted_glob(monkeypatch):
    real = glob.glob
    monkeypatch.setattr(specimine.glob, "glob", lambda pattern, **kw: sorted(real(pattern, **kw)))


def host_mined(root, files, index, flags, monkeypatch, caplog=None):
    """specimine.mine_files over the pool-level full files of the tree under root: {path: bytes} of the .mined files."""
    pool_level = [p for p, k in zip(files.paths, files.file_key) if int(k) >> 62 == 3]
    for f in glob.glob(os.path.join(root, "**", "*.mined"), recursive=True):
        os.remove(f)
    _sorted_glob(monkeypatch)
    pf, npr, mi = _flags(flags)
    specimine.mine_files([os.path.join(root, p) for p in pool_level], index, pf, npr, mi)
    return {os.path.relpath(f, root): open(f, "rb").read()
            for f in glob.glob(os.path.join(root, "**", "*.mined"), recursive=True)}


def assert_same_as_host(mined, root, files, index, flags, monkeypatch, caplog):
    caplog.clear()
    want = host_mined(root, files, index, flags, monkeypatch)
    got = {p: bytes(np.asarray(mined.data.cpu() if hasattr(mined.data, "cpu") else mined.data)[
        int(mined.file_offset[j]):int(mined.file_offset[j + 1])]) for j, p in enumerate(mined.paths)}
    assert got == want
    for path, reason in mined.skipped:
        assert reason in caplog.text and not os.path.exists(os.path.join(root, path + ".mined"))
    out = os.path.join(root, "device_copy")
    mined.write(out)
    assert read_tree(out) == want
    return want


def _mining_tables(ds):
    specimens = H.build_specimens(ds.primers, ds.specimens)
    return MatchTables(specimens, MatchParameters({synth.ITS1F: 5, synth.ITS4: 5}, 2, ds.search_len, True))


def _mining_block(ds):
    reads = [(b"%s_%d desc" % (ds.name.encode(), i), ds.read_str(i).encode(), ds.qual_str(i).encode())
             for i in range(ds.n_reads)]
    bases = b"".join(r[1] for r in reads)
    quals = b"".join(r[2] for r in reads)
    off = np.concatenate([[0], np.cumsum([len(r[1]) for r in reads])]).astype(np.uint64)
    titles = b"".join(r[0] for r in reads)
    t_off = np.concatenate([[0], np.cumsum([len(r[0]) for r in reads])]).astype(np.uint64)
    return reads, (bases, quals, off, titles, t_off)


def _small_mining():
    return synth.mining_reads(2, 3, 4, 3, 3, amplicon=160, seed=5)


@pytest.mark.parametrize("prefix", ["", "sample_", "p_"])
@pytest.mark.parametrize("flags", FLAG_SETS, ids=lambda f: " ".join(f) or "default")
def test_synthetic_batch_equals_mine_files(fsim, msim, tmp_path, monkeypatch, caplog, flags, prefix):
    ds = _small_mining()
    mt = _mining_tables(ds)
    m = Matcher(mt, binding=H.hostsim_binding())
    _reads, block = _mining_block(ds)
    res = m.match(PackedBatch([ds.read_str(i) for i in range(ds.n_reads)], clip=ds.search_len))
    rc, files, _bad, _need = sim_files(fsim, mt, block, res.records, True, prefix=prefix)
    assert rc == 0
    root = str(tmp_path / "tree")
    files.write(root)
    index = str(tmp_path / "index.txt")
    _write_index(index, ds.specimens)
    pf, npr, mi = _flags(flags)
    monkeypatch.setattr(specimine, "hw_best_grouped", _host_best_grouped(_oracle_distance))
    rc, mined, _bad = mine_sim(msim, files, index, pf, npr, mi)
    assert rc == 0
    want = assert_same_as_host(mined, root, files, index, flags, monkeypatch, caplog)
    if prefix == "p_":
        assert not mined.paths and len(mined.skipped) == len(ds.specimens)
        assert all(r.startswith("Could not find specimen p_") for _p, r in mined.skipped)
    else:
        assert len(mined.paths) == len(ds.specimens) and not mined.skipped
        if not npr or pf:
            assert any(want.values()), "the batch should give mined reads"


@pytest.mark.parametrize("name,run_name", [r for r in _golden_runs() if r[1] == "default"])
def test_golden_runs_equal_mine_files(fsim, msim, tmp_path, monkeypatch, caplog, name, run_name):
    g, params, matcher = _golden_matcher(name, run_name, H.hostsim_binding())
    reads = [(("%s x" % r[0]).encode(), r[1].encode(), r[2].encode()) for r in g["reads"]]
    bases = b"".join(r[1] for r in reads)
    block = (bases, b"".join(r[2] for r in reads), np.concatenate([[0], np.cumsum([len(r[1]) for r in reads])]).astype(np.uint64),
             b"".join(r[0] for r in reads), np.concatenate([[0], np.cumsum([len(r[0]) for r in reads])]).astype(np.uint64))
    res = matcher.match(PackedBatch([r[1] for r in g["reads"]], clip=params.search_len))
    rc, files, _bad, _need = sim_files(fsim, matcher.tables, block, res.records, True, prefix="")
    assert rc == 0
    root = str(tmp_path / "tree")
    files.write(root)
    index = str(tmp_path / "index.txt")
    _write_index(index, g["specimens"])
    monkeypatch.setattr(specimine, "hw_best_grouped", _host_best_grouped(_oracle_distance))
    for flags in FLAG_SETS + [["--partial-forward", "--min-identity", "0.5"]]:
        pf, npr, mi = _flags(flags)
        rc, mined, _bad = mine_sim(msim, files, index, pf, npr, mi)
        assert rc == 0
        assert_same_as_host(mined, root, files, index, flags, monkeypatch, caplog)


def test_multi_pair_pool_equals_mine_files_in_sorted_order(fsim, msim, tmp_path, monkeypatch, caplog):
    """Partial reads of one pool in two primer-pair directories (half of them without a forward primer): the virtual
    tree lists the pair directories in sorted path order, as glob patched to sorted order does on disk."""
    ds = _small_mining()
    mt = _mining_tables(ds)
    m = Matcher(mt, binding=H.hostsim_binding())
    _reads, block = _mining_block(ds)
    rec = m.match(PackedBatch([ds.read_str(i) for i in range(ds.n_reads)], clip=ds.search_len)).records.copy()
    part = np.nonzero(np.isin(rec["resolution"], (2, 3)))[0]
    rec["p1"][part[::2]] = -1
    rc, files, _bad, _need = sim_files(fsim, mt, block, rec, True, prefix="")
    assert rc == 0
    pairs = {p.split("/")[2] for p in files.paths if p.startswith("partial/")}
    assert len(pairs) > 1, pairs
    root = str(tmp_path / "tree")
    files.write(root)
    index = str(tmp_path / "index.txt")
    _write_index(index, ds.specimens)
    monkeypatch.setattr(specimine, "hw_best_grouped", _host_best_grouped(_oracle_distance))
    rc, mined, _bad = mine_sim(msim, files, index, True)
    assert rc == 0
    assert any(assert_same_as_host(mined, root, files, index, ["--partial-forward"], monkeypatch, caplog).values())


def test_validation_names_file_and_output(fsim, msim, tmp_path):
    ds = _small_mining()
    mt = _mining_tables(ds)
    m = Matcher(mt, binding=H.hostsim_binding())
    _reads, block = _mining_block(ds)
    res = m.match(PackedBatch([ds.read_str(i) for i in range(ds.n_reads)], clip=ds.search_len))
    rc, files, _bad, _need = sim_files(fsim, mt, block, res.records, True, prefix="")
    index = str(tmp_path / "index.txt")
    _write_index(index, ds.specimens)
    f = next(i for i, p in enumerate(files.paths) if p.startswith("partial/") and "/barcode_rev_" in p)
    o = int(np.searchsorted(files.offsets, files.file_offset[f])) + 1         # second output of that file
    a = int(files.offsets[o])
    data = files.data.copy()
    data[a] = ord(">")
    files.data = data
    rc, _mined, bad = mine_sim(msim, files, index)
    assert rc == 2 and bad == (f << 35 | 1 << 3 | 3)
    data[a] = ord("@")
    fo = files.file_offset.copy()
    files.file_offset = fo.copy()
    files.file_offset[f] += 1                                                   # not an output boundary
    rc, _mined, bad = mine_sim(msim, files, index)
    assert rc == 2 and bad >> 35 in (f - 1, f) and bad & 7 == 1
    files.file_offset = fo
    rc, mined, _bad = mine_sim(msim, files, index)
    assert rc == 0
    need = (int(mined.file_offset[-1]), len(mined.partial))
    if need[1]:
        assert mine_sim(msim, files, index, out_cap=(need[0] - 1, need[1]))[0] == 4
        assert mine_sim(msim, files, index, out_cap=(need[0], need[1] - 1))[0] == 4
    assert mine_sim(msim, files, index, out_cap=need)[0] == 0


RANK_LIMIT = 1 << 23                     # full reads of one group: the search key holds the winner's rank in 23 bits


def _rank_limit_files(tmp_path, n_full):
    """A tree of one pool-level full file of n_full one-base reads and one partial file, as numpy DeviceFiles, and its
    index."""
    from specimux_b200.engine import DeviceFiles
    rec = np.frombuffer(b"@r\nA\n+\nI\n", dtype=np.uint8)
    part = np.frombuffer(b"@p x\nACGT\n+\nIIII\n", dtype=np.uint8)
    data = np.concatenate([np.tile(rec, n_full), part])
    offsets = np.concatenate([np.arange(n_full + 1, dtype=np.int64) * len(rec), [n_full * len(rec) + len(part)]])
    file_off = np.array([0, n_full * len(rec), len(data)], dtype=np.int64)
    files = DeviceFiles(None, data, np.array([3 << 62, 1 << 62], dtype=np.uint64), file_off,
                        ["full/ITS/SP.fastq", "partial/ITS/ITS1F-ITS4/barcode_rev_ACGT.fastq"], None, offsets)
    index = str(tmp_path / "rank_index.txt")
    _write_index(index, [["SP", "ITS", "AAAA", "ITS1F", "ACGT", "ITS4"]])
    return files, index


def test_a_full_file_past_the_rank_field_is_refused(msim, tmp_path):
    files, index = _rank_limit_files(tmp_path, RANK_LIMIT + 1)
    rc, _mined, bad = mine_sim(msim, files, index)
    assert rc == 2 and bad == (0 << 35 | RANK_LIMIT << 3 | 6)
    files, index = _rank_limit_files(tmp_path, 3)
    rc, mined, _bad = mine_sim(msim, files, index, min_identity=0.0)
    assert rc == 0 and mined.paths == ["full/ITS/SP.fastq.mined"]


def test_virtual_tree_lists_in_sorted_order():
    t = specimine.VirtualTree(["partial/P/b-x/f.fastq", "partial/P/a-y/g.fastq", "full/P/s.fastq", "partial/P/.h/i.fastq"])
    assert t.listdir("partial/P/*") == ["partial/P/a-y", "partial/P/b-x"]
    assert t.isdir("partial/P") and t.exists("full/P/s.fastq") and not t.isdir("full/P/s.fastq")
    assert not t.exists("partial/Q")


def test_no_gpu_means_no_device_mining():
    lib = _lib.load()
    if lib.smx_device_count() > 0:
        pytest.skip("box has a GPU")
    n = C.c_uint64(0)
    z = np.zeros(2, dtype=np.uint64)
    g = np.zeros(1, dtype=np.uint32)
    rc = lib.smx_mine_device(None, None, 0, None, 0, _lib.ptr(z, _lib.u64p), 0, 0, None, None, None, None, 0,
                             _lib.ptr(g, _lib.u32p), 0.85, None, None, 0, 0, None, None, None, None, C.byref(n), C.byref(n),
                             None)
    assert rc == _lib.SMX_ERR_NO_DEVICE


def test_simulator_matcher_refuses_mine_device():
    m = Matcher(_mining_tables(_small_mining()), binding=H.hostsim_binding())
    with pytest.raises(RuntimeError, match="no device route"):
        m.mine_device(None, "index.txt")


# ---------------------------------------------------------------------------------------------------------------------
# GPU tier

def _tensors(block):
    import torch
    bases, quals, off, titles, t_off = block
    t = lambda x: torch.tensor(np.frombuffer(x, dtype=np.uint8).copy(), device="cuda")
    return (t(bases), t(quals), torch.tensor(off.astype(np.int64), device="cuda"), t(titles),
            torch.tensor(t_off.astype(np.int64), device="cuda"))


def _device_files(m, block, prefix="", fastq=True):
    b, q, o, t, to = _tensors(block)
    return m.demux_files_device(b, o, t, to, q, prefix=prefix, fastq=fastq)


@pytest.mark.gpu
@pytest.mark.parametrize("name,run_name", list(_golden_runs()))
def test_golden_runs_on_the_device_equal_mine_files(tmp_path, monkeypatch, caplog, name, run_name):
    g, params, m = _golden_matcher(name, run_name, None)
    reads = [(("%s x" % r[0]).encode(), r[1].encode(), r[2].encode()) for r in g["reads"]]
    block = (b"".join(r[1] for r in reads), b"".join(r[2] for r in reads),
             np.concatenate([[0], np.cumsum([len(r[1]) for r in reads])]).astype(np.uint64), b"".join(r[0] for r in reads),
             np.concatenate([[0], np.cumsum([len(r[0]) for r in reads])]).astype(np.uint64))
    files = _device_files(m, block)
    root = str(tmp_path / "tree")
    files.write(root)
    index = str(tmp_path / "index.txt")
    _write_index(index, g["specimens"])
    for flags in ([], ["--partial-forward", "--min-identity", "0.5"]):
        pf, npr, mi = _flags(flags)
        mined = m.mine_device(files, index, pf, npr, mi)
        assert_same_as_host(mined, root, files, index, flags, monkeypatch, caplog)


@pytest.mark.gpu
@pytest.mark.parametrize("flags", FLAG_SETS, ids=lambda f: " ".join(f) or "default")
def test_synthetic_batch_on_the_device_equals_mine_files_and_the_harness(msim, tmp_path, monkeypatch, caplog, flags):
    ds = synth.mining_reads(3, 8, 6, 3, 8, amplicon=640, seed=7)
    mt = _mining_tables(ds)
    _reads, block = _mining_block(ds)
    index = str(tmp_path / "index.txt")
    _write_index(index, ds.specimens)
    pf, npr, mi = _flags(flags)
    with Matcher(mt) as m:
        files = _device_files(m, block)
        root = str(tmp_path / "tree")
        files.write(root)
        mined = m.mine_device(files, index, pf, npr, mi)
        assert mined.device_ms[1] >= mined.device_ms[0] >= 0
        want = assert_same_as_host(mined, root, files, index, flags, monkeypatch, caplog)
        if not npr or pf:
            assert any(want.values())
        # the harness on the same files (copied to the host), with oracle distances
        import torch
        host = type(files)(None, files.data.cpu().numpy(), files.file_key, files.file_offset, files.paths,
                           files.record.cpu().numpy(), files.offsets.cpu().numpy())
        rc, sim, _bad = mine_sim(msim, host, index, pf, npr, mi)
        assert rc == 0
        assert mined.data.cpu().numpy().tobytes() == sim.data.tobytes()
        assert np.array_equal(mined.file_offset, sim.file_offset) and mined.paths == sim.paths
        assert np.array_equal(mined.partial.cpu().numpy(), sim.partial)
        assert np.array_equal(mined.winner.cpu().numpy(), sim.winner)
        assert np.array_equal(mined.distance.cpu().numpy(), sim.distance)


@pytest.mark.gpu
def test_multipool_batch_on_the_device_equals_mine_files(tmp_path, monkeypatch, caplog):
    from specimux_b200.orchestration import thresholds_for
    ds = synth.multipool(n_reads=30_000, seed=17)
    specimens = H.build_specimens(ds.primers, ds.specimens)
    k_idx, k_primers = thresholds_for(specimens)
    mt = MatchTables(specimens, MatchParameters(k_primers, k_idx, ds.search_len, True))
    _reads, block = _mining_block(ds)
    index = str(tmp_path / "index.txt")
    _write_index(index, ds.specimens)
    with Matcher(mt) as m:
        files = _device_files(m, block, prefix="sample_")
        root = str(tmp_path / "tree")
        files.write(root)
        for flags in ([], ["--partial-forward", "--min-identity", "0.2"]):
            pf, npr, mi = _flags(flags)
            assert_same_as_host(m.mine_device(files, index, pf, npr, mi), root, files, index, flags, monkeypatch, caplog)


@pytest.mark.gpu
def test_refusals_leave_the_matcher_usable_and_routes_interleave(tmp_path):
    import torch
    ds = synth.mining_reads(2, 4, 5, 3, 4, amplicon=500, seed=3)
    mt = _mining_tables(ds)
    _reads, block = _mining_block(ds)
    index = str(tmp_path / "index.txt")
    _write_index(index, ds.specimens)
    b, q, o, t, to = _tensors(block)
    with Matcher(mt) as m:
        files = m.demux_files_device(b, o, t, to, q)
        want = m.mine_device(files, index, True)
        assert want.partial.numel() > 0

        def check_usable():
            got = m.mine_device(m.demux_files_device(b, o, t, to, q), index, True)
            assert got.data.cpu().numpy().tobytes() == want.data.cpu().numpy().tobytes()
            assert m.match_device(b, o).records.shape[0] == files.result.records.shape[0]

        with pytest.raises(ValueError, match="FASTQ"):
            m.mine_device(m.demux_files_device(b, o, t, to, q, fastq=False), index)
        with pytest.raises(ValueError):
            m.mine_device("x", index)
        for attr, bad in (("data", files.data.cpu()), ("offsets", files.offsets.cpu()), ("offsets", files.offsets.to(torch.int32))):
            edited = type(files)(files.result, files.data, files.file_key, files.file_offset, files.paths, files.record,
                                 files.offsets)
            setattr(edited, attr, bad)
            with pytest.raises(ValueError):
                m.mine_device(edited, index)
        check_usable()
        # more than 64 distinct bytes in a full read: its sequence rewritten in place
        f = next(i for i, k in enumerate(files.file_key) if int(k) >> 62 == 3)
        offs = files.offsets.cpu().numpy()
        o0 = int(np.searchsorted(offs, files.file_offset[f]))
        a = int(offs[o0])
        rec = files.data[a:int(offs[o0 + 1])].cpu().numpy().tobytes()
        s = a + rec.index(b"\n") + 1
        data = files.data.clone()
        data[s:s + 70] = torch.tensor(list(range(33, 103)), dtype=torch.uint8)
        edited = type(files)(files.result, data, files.file_key, files.file_offset, files.paths, files.record, files.offsets)
        with pytest.raises(_lib.SmxError, match="file %d output 0 is a full read holding more than 64" % f):
            m.mine_device(edited, index, True)
        check_usable()
        # pointers that are not memory of the context's device, caught by the C call itself
        lib = _lib.load()
        _jobs, _skipped, (gf, gk, gpo, gp, mg), _distinct = mine_plan(files, index, True, False)
        file_off = np.ascontiguousarray(files.file_offset, dtype=np.uint64)
        host_off = files.offsets.cpu().numpy()
        host_out = np.zeros(1 << 20, dtype=np.uint8)
        e = lambda k, dt=torch.int64: torch.empty(k, dtype=dt, device="cuda")
        out, moff, part, win, dist = e(1 << 20, torch.uint8), e(len(_jobs) + 1), e(4096), e(4096), e(4096, torch.int32)
        nr, nb = C.c_uint64(0), C.c_uint64(0)

        def call(off_ptr, out_ptr):
            return lib.smx_mine_device(m._ctx, files.data.data_ptr(), files.data.numel(), off_ptr, files.offsets.numel() - 1,
                                       _lib.ptr(file_off, _lib.u64p), len(files.paths), len(gf), _lib.ptr(gf, _lib.u32p),
                                       _lib.ptr(gk, _lib.u8p), _lib.ptr(gpo, _lib.u32p), _lib.ptr(gp, _lib.u32p), len(_jobs),
                                       _lib.ptr(mg, _lib.u32p), 0.85, None, out_ptr, 1 << 20, 4096, moff.data_ptr(),
                                       part.data_ptr(), win.data_ptr(), dist.data_ptr(), C.byref(nr), C.byref(nb), None)
        assert call(host_off.ctypes.data, out.data_ptr()) == _lib.SMX_ERR_ARG
        assert "out_off is not memory of device" in lib.smx_last_error().decode()
        assert call(files.offsets.data_ptr(), host_out.ctypes.data) == _lib.SMX_ERR_ARG
        assert "out is not memory of device" in lib.smx_last_error().decode()
        assert call(files.offsets.data_ptr(), out.data_ptr()) == _lib.SMX_OK and nr.value == want.partial.numel()
        assert out[:nb.value].cpu().numpy().tobytes() == want.data.cpu().numpy().tobytes()
        check_usable()
        # a full file of more than 2^23 reads: the rank field of the search key cannot name the winner
        big, bindex = _rank_limit_files(tmp_path, RANK_LIMIT + 1)
        big.data, big.offsets = torch.tensor(big.data, device="cuda"), torch.tensor(big.offsets, device="cuda")
        with pytest.raises(_lib.SmxError, match="file 0 output %d is a full read beyond the 2\\^23" % RANK_LIMIT):
            m.mine_device(big, bindex)
        del big
        check_usable()
        # a full read longer than 4,096 nt
        long_ds = synth.mining_reads(1, 2, 2, 2, 1, amplicon=4300, seed=4)
        _r, lblock = _mining_block(long_ds)
        lindex = str(tmp_path / "long.txt")
        _write_index(lindex, long_ds.specimens)
        with Matcher(_mining_tables(long_ds)) as lm:
            lfiles = _device_files(lm, lblock)
            with pytest.raises(_lib.SmxError, match="is a full read longer than 4096 bytes"):
                lm.mine_device(lfiles, lindex)
        check_usable()


@pytest.mark.gpu
def test_side_stream_long_read_and_no_pool_level_files(tmp_path):
    import torch
    ds = synth.mining_reads(2, 3, 4, 3, 3, amplicon=400, seed=9)
    mt = _mining_tables(ds)
    reads, block = _mining_block(ds)
    # one more partial read of 190,000 nt holding a specimen's amplicon: mined, copied whole
    # a partial reverse read in forward orientation (its destroyed forward barcode first), the long run in front of it
    i = next(j for j in range(ds.n_reads) if ds.truth["kind"][j] == 1 and synth.ITS1F in ds.read_str(j))
    rng = np.random.default_rng(2)
    tail = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=190_000)].tobytes()
    big = tail + ds.read_str(i).encode()
    bases, quals, off, titles, t_off = block
    block = (bases + big, quals + b"5" * len(big), np.append(off, off[-1] + len(big)).astype(np.uint64),
             titles + b"big read", np.append(t_off, t_off[-1] + 8).astype(np.uint64))
    index = str(tmp_path / "index.txt")
    _write_index(index, ds.specimens)
    with Matcher(mt) as m:
        files = _device_files(m, block)
        want = m.mine_device(files, index, True)
        text = want.data.cpu().numpy().tobytes()
        assert b"@big_mined_reverse_" in text
        if tail[:1000] in files.data.cpu().numpy().tobytes():
            assert tail[:1000] in text
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            d2 = torch.zeros_like(files.data)
            torch.cuda._sleep(2_000_000)                 # the side stream is busy before the files are written
            d2.copy_(files.data)
            edited = type(files)(files.result, d2, files.file_key, files.file_offset, files.paths, files.record, files.offsets)
            got = m.mine_device(edited, index, True)
        assert got.data.cpu().numpy().tobytes() == text
        # no pool-level files: only partial reads
        part = synth.mining_reads(2, 3, 0, 3, 3, amplicon=300, seed=9)
        _r, pblock = _mining_block(part)
        pfiles = _device_files(m, pblock)
        assert not any(int(k) >> 62 == 3 for k in pfiles.file_key)
        none = m.mine_device(pfiles, index, True)
        assert none.paths == [] and none.data.numel() == 0 and list(none.file_offset) == [0] and none.skipped == []
        none.write(str(tmp_path / "t"))
        assert not os.path.exists(str(tmp_path / "t"))
