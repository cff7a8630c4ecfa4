"""Reads already in GPU memory: the device packer (smx_k_pack.cu) and Matcher.match_device.

CPU tier: the packer's per-thread work items (smx_pack.cuh) run as host loops (tests/packsim) and must reproduce the
host packer smx_pack_reads_fixed byte for byte; the validation names the first bad read.  GPU tier: match_device equals
Matcher.match(PackedBatch(reads, clip=search_len)) on the golden runs, edge batches, resident splits, sliced tensors,
side streams, and after refused calls."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers as H
from specimux_b200 import _lib, synth
from specimux_b200.engine import Matcher, PackedBatch
from specimux_b200.models import MatchParameters
from specimux_b200.orchestration import thresholds_for
from specimux_b200.tables import MatchTables

U64 = 0xFFFFFFFFFFFFFFFF
_packsim = None


def packsim(tmp_path_factory):
    """Builds (g++) and loads tests/packsim/packsim.cpp into a temporary directory."""
    global _packsim
    if _packsim is None:
        src = os.path.join(H.HERE, "packsim", "packsim.cpp")
        so = str(tmp_path_factory.mktemp("packsim") / "libpacksim.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unused-function", "-o", so, src])
        lib = C.CDLL(so)
        lib.packsim_validate.restype = C.c_uint64
        lib.packsim_validate.argtypes = [_lib.u64p, C.c_uint32, C.c_uint64]
        lib.packsim_pack.restype = C.c_uint64
        lib.packsim_pack.argtypes = [C.c_char_p, C.c_uint64, _lib.u64p, C.c_uint32, C.c_uint32, C.c_int, _lib.u32p, _lib.u32p,
                                     _lib.u32p, _lib.u64p, _lib.u32p, C.c_uint64, _lib.u64p, _lib.u32p]
        _packsim = lib
    return _packsim


@pytest.fixture(scope="module")
def sim(tmp_path_factory):
    return packsim(tmp_path_factory)


def _blob(reads):
    raw = [r if isinstance(r, bytes) else r.encode("latin-1") for r in reads]
    off = np.zeros(len(raw) + 1, dtype=np.uint64)
    np.cumsum([len(r) for r in raw], out=off[1:])
    return b"".join(raw), off


def _device_pack(sim, blob, off, clip, cuts):
    n = len(off) - 1
    stride = (2 * clip + 15) // 16
    packed2 = np.full(n * stride + len(cuts) - 1, 0xDEADBEEF, dtype=np.uint32)
    lengths = np.zeros(max(n, 1), dtype=np.uint32)
    off4 = np.full(max(n, 1), 7, dtype=np.uint64)
    cap4 = 2 * ((2 * clip + 7) // 8) * n + 1
    packed4 = np.full(cap4, 0xDEADBEEF, dtype=np.uint32)
    words4, flagged = C.c_uint64(0), C.c_uint32(0)
    cuts = np.asarray(cuts, dtype=np.uint32)
    key = sim.packsim_pack(blob, len(blob), _lib.ptr(off, _lib.u64p), n, clip, len(cuts) - 1, _lib.ptr(cuts, _lib.u32p),
                           _lib.ptr(packed2, _lib.u32p), _lib.ptr(lengths, _lib.u32p), _lib.ptr(off4, _lib.u64p),
                           _lib.ptr(packed4, _lib.u32p), cap4, C.byref(words4), C.byref(flagged))
    assert key == U64
    return packed2, lengths[:n], off4[:n], packed4[:words4.value], flagged.value


def _assert_same_as_host(sim, reads, clip=80, cuts=None):
    blob, off = _blob(reads)
    n = len(reads)
    host = PackedBatch.from_blob(blob, off, clip=clip)
    for lane_cuts in ([0, n],) + ((cuts,) if cuts else ()):
        packed2, lengths, off4, packed4, flagged = _device_pack(sim, blob, off, clip, lane_cuts)
        stride = host.stride
        at = 0
        for a, b in zip(lane_cuts[:-1], lane_cuts[1:]):           # each lane: its reads' words + the slack word
            words = (b - a) * stride + 1
            assert np.array_equal(packed2[at:at + words], host.packed2[a * stride:b * stride + 1]), (a, b)
            at += words
        assert np.array_equal(lengths, host.lengths[:n])
        assert flagged == host.n_flagged
        if flagged:
            assert np.array_equal(off4, host.off4[:n])
            assert np.array_equal(packed4, host.packed4)


def _reads_every_length(rng, alphabet="ACGT"):
    return ["".join(rng.choice(list(alphabet), size=n)) for n in range(261)]


def test_read_codes_match_the_encoding_table(sim):
    sim.packsim_read_code.argtypes = sim.packsim_read_code_rc.argtypes = [C.c_int]
    codes = {c: i for i, c in enumerate("ACGTRYSWKMBDHVN")}
    comp = dict(zip("ACGTRYSWKMBDHVN", "TGCAYRSWMKVHDBN"))
    for ch in range(256):
        want = codes.get(chr(ch), 15)
        want_rc = 0 if chr(ch) == "U" else codes.get(comp.get(chr(ch), ""), 15)
        assert (sim.packsim_read_code(ch), sim.packsim_read_code_rc(ch)) == (want, want_rc), ch


def test_every_length_and_twice_the_clip(sim):
    rng = np.random.default_rng(1)
    reads = _reads_every_length(rng)
    _assert_same_as_host(sim, reads, 80, [0, 100, 101, 261])
    for clip in (80, 200):
        edge = ["".join(rng.choice(list("ACGT"), size=2 * clip + d)) for d in (-1, 0, 1)]
        _assert_same_as_host(sim, edge + [e[:clip] + "N" + e[clip + 1:] for e in edge], clip, [0, 3, 6])


def test_long_empty_and_exotic_reads(sim):
    rng = np.random.default_rng(2)
    big = "".join(rng.choice(list("ACGT"), size=190_000))
    high = bytes(range(0x80, 0x100)) * 2
    reads = [big, "", "", "N" * 300, "acgt" * 50, "ACGU" * 40, "RYKMSWBDHVN" * 20, b"AC" + high + b"GT", "",
             big[:100] + "n" + big[100:], "ACGT" * 30 + "N", "x", big[:5000] + "Y" + big[5000:9000] + "R"]
    _assert_same_as_host(sim, reads, 80, [0, 1, 4, 9, 13])
    _assert_same_as_host(sim, reads, 1024)
    _assert_same_as_host(sim, ["", "", ""], 80, [0, 2, 3])


@pytest.mark.parametrize("n", [127, 128, 129, 2500])
def test_batch_sizes(sim, n):
    rng = np.random.default_rng(n)
    reads = []
    for i in range(n):
        s = rng.choice(list("ACGT"), size=int(rng.integers(0, 400)))
        if i % 7 == 3 and len(s):
            s[rng.integers(0, len(s))] = "N"
        reads.append("".join(s))
    _assert_same_as_host(sim, reads, 80, [0, n // 3, n // 3 + 1, n])


def test_validation_names_the_first_bad_read(sim):
    def key(off, n_bases):
        off = np.asarray(off, dtype=np.uint64)
        return sim.packsim_validate(_lib.ptr(off, _lib.u64p), len(off) - 1, n_bases)
    assert key([0, 5, 9, 9, 20], 20) == U64
    assert key([0, 5, 4, 9, 20], 20) == (1 << 2) | 1                 # read 1 ends before it starts
    assert key([0, 5, 9, 12, 21], 20) == (3 << 2) | 2                # read 3 ends past n_bases
    assert key([3, 5, 9, 12, 20], 20) == U64                         # a first offset above 0 is fine
    assert key([0, 5, 5 + (1 << 31), 5 + (1 << 31)], 1 << 33) == (1 << 2) | 3
    assert key([0, 5, 5 + (1 << 31) - 1], 1 << 33) == U64
    assert key([0, 5, 4, 30], 20) == (1 << 2) | 1                    # the first refused read wins


def test_import_stays_torch_free():
    code = ("import specimux_b200, specimux_b200.engine, specimux_b200.cli; import sys; "
            "assert 'torch' not in sys.modules")
    subprocess.check_call([sys.executable, "-c", code], cwd=H.ROOT)


def test_simulator_matcher_refuses_match_device():
    g = H.load_golden("fixture")
    run = g["runs"]["default"]
    specimens = H.build_specimens(g["primers"], g["specimens"])
    m = Matcher(MatchTables(specimens, H.params_from_run(run, specimens)), binding=H.hostsim_binding())
    with pytest.raises(RuntimeError, match="no device route"):
        m.match_device(None, None)


def test_no_gpu_means_no_device_match():
    lib = _lib.load()
    if lib.smx_device_count() > 0:
        pytest.skip("box has a GPU")
    n = C.c_uint64(0)
    rc = lib.smx_match_device(None, None, 0, None, 0, None, None, None, 0, C.byref(n), C.byref(n), None)
    assert rc == _lib.SMX_ERR_NO_DEVICE


# ---------------------------------------------------------------------------------------------------------------------
# GPU tier

def _tensors(reads, pad_front=0, pad_back=0):
    import torch
    blob, off = _blob(reads)
    full = torch.tensor(np.frombuffer(b"\x07" * pad_front + blob + b"\x07" * pad_back, dtype=np.uint8).copy(), device="cuda")
    return full, torch.tensor(off.astype(np.int64) + pad_front, device="cuda")


def _assert_equal(got, want, tag=""):
    host = got.to_host()
    assert host.n_matched == want.n_matched, tag
    assert np.array_equal(host.rec_offset, want.rec_offset), tag
    assert host.records.tobytes() == want.records.tobytes(), tag


def _golden_tables(name, run_name):
    g = H.load_golden(name)
    run = g["runs"][run_name]
    specimens = H.build_specimens(g["primers"], g["specimens"])
    args = H.make_args(run["flags"])
    mt = MatchTables(specimens, H.params_from_run(run, specimens), trim=args.trim, dereplicate=args.dereplicate,
                     prefilter=not args.disable_prefilter, min_length=args.min_length, max_length=args.max_length)
    return g, mt


@pytest.mark.gpu
@pytest.mark.parametrize("name,run_name", [(n, r) for n in H.golden_names() for r in H.load_golden(n)["runs"]])
def test_golden_runs_equal_host_route(name, run_name):
    g, mt = _golden_tables(name, run_name)
    reads = [r[1] for r in g["reads"]]
    bases, offsets = _tensors(reads)
    with Matcher(mt) as m:
        want = m.match(PackedBatch(reads, clip=mt.parameters.search_len))
        _assert_equal(m.match_device(bases, offsets), want, "%s/%s" % (name, run_name))


def _edge_batches():
    rng = np.random.default_rng(17)
    good = [r[1] for r in H.load_golden("fixture")["reads"]]

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


@pytest.mark.gpu
@pytest.mark.parametrize("name,reads", list(_edge_batches()), ids=[n for n, _ in _edge_batches()])
def test_edge_batches_equal_host_route(name, reads):
    g, mt = _golden_tables("fixture", "default")
    mt = MatchTables(mt.specimens, mt.parameters, trim="tails")
    bases, offsets = _tensors(reads)
    with Matcher(mt) as m:
        _assert_equal(m.match_device(bases, offsets), m.match(PackedBatch(reads, clip=mt.parameters.search_len)), name)


def _ont037_with_exotic(n, seed=99):
    ds = synth.ont037(n_reads=n, seed=seed, with_quals=False)
    specimens = H.build_specimens(ds.primers, ds.specimens)
    k_idx, k_primers = thresholds_for(specimens)
    mt = MatchTables(specimens, MatchParameters(k_primers, k_idx, ds.search_len, True))
    codes = np.frombuffer(b"ACGT", dtype=np.uint8)[ds.codes].copy()
    rng = np.random.default_rng(6)
    hits = rng.choice(codes.shape[0], size=codes.shape[0] // 5000, replace=False)
    codes[hits] = np.frombuffer(b"NRYn", dtype=np.uint8)[rng.integers(0, 4, size=hits.shape[0])]
    return mt, codes, ds.offsets.astype(np.uint64)


@pytest.mark.gpu
def test_resident_splits_equal_one_lane_host_route():
    import torch
    mt, codes, offs = _ont037_with_exotic(300_000)
    batch = PackedBatch.from_blob(codes.tobytes(), offs, clip=mt.parameters.search_len)
    assert batch.n_flagged > 0
    bases, offsets = torch.tensor(codes, device="cuda"), torch.tensor(offs.astype(np.int64), device="cuda")
    with Matcher(mt) as m:
        m.set_resident_split(1)
        m.set_pipeline_chunk(0)
        want = m.match(batch)
        for split in (1, 2, 3, 5):
            m.set_resident_split(split)
            got = m.match_device(bases, offsets)
            _assert_equal(got, want, "split %d" % split)
            assert got.device_ms[1] >= got.device_ms[0] > 0


@pytest.mark.gpu
def test_slice_of_a_larger_tensor_with_nonzero_first_offset():
    import torch
    g, mt = _golden_tables("synth_ont037", "default")
    reads = [r[1] for r in g["reads"]]
    reads[5] = reads[5][:40] + "N" + reads[5][41:]
    full, offsets = _tensors(reads, pad_front=1000, pad_back=333)
    bases = full[17:]                                   # a view: its data starts 17 bytes into the allocation
    offsets = offsets - 17
    assert int(offsets[0]) == 983 and bases.data_ptr() == full.data_ptr() + 17
    with Matcher(mt) as m:
        want = m.match(PackedBatch(reads, clip=mt.parameters.search_len))
        _assert_equal(m.match_device(bases, offsets.contiguous()), want)
        _assert_equal(m.match_device(full[1000:1000 + int(offsets[-1]) - 983], offsets - 983), want)


@pytest.mark.gpu
def test_ordered_after_work_on_the_callers_stream():
    import torch
    mt, codes, offs = _ont037_with_exotic(60_000, seed=3)
    want_batch = PackedBatch.from_blob(codes.tobytes(), offs, clip=mt.parameters.search_len)
    src = torch.tensor(codes, device="cuda")
    offsets = torch.tensor(offs.astype(np.int64), device="cuda")
    with Matcher(mt) as m:
        want = m.match(want_batch)
        torch.cuda.synchronize()
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            for _ in range(3):
                bases = torch.zeros_like(src)
                torch.cuda._sleep(2_000_000)           # keeps the side stream busy before the bases are written
                bases.copy_(src)
                _assert_equal(m.match_device(bases, offsets), want)


@pytest.mark.gpu
def test_bad_input_is_refused_and_the_context_stays_usable():
    import torch
    g, mt = _golden_tables("fixture", "default")
    reads = [r[1] for r in g["reads"]]
    bases, offsets = _tensors(reads)
    lib = _lib.load()
    n = len(reads)
    n_bases = bases.numel()
    with Matcher(mt) as m:
        want = m.match(PackedBatch(reads, clip=mt.parameters.search_len))
        cap = int(lib.smx_result_bound(m._ctx, n))
        rec = torch.empty((cap, 64), dtype=torch.uint8, device="cuda")
        ro = torch.empty(n + 1, dtype=torch.int32, device="cuda")
        n_rec, n_mat = C.c_uint64(0), C.c_uint64(0)

        def call(b_ptr, nb, o_ptr, rec_ptr=None, cap_=cap):
            return lib.smx_match_device(m._ctx, b_ptr, nb, o_ptr, n, 0, ro.data_ptr(),
                                        rec.data_ptr() if rec_ptr is None else rec_ptr, cap_, C.byref(n_rec), C.byref(n_mat), None)

        def check_usable():
            _assert_equal(m.match_device(bases, offsets), want)

        # offsets that descend: every offset still lies inside the bases tensor
        bad = offsets.clone()
        bad[7] = bad[9]
        assert call(bases.data_ptr(), n_bases, bad.data_ptr()) == _lib.SMX_ERR_ARG
        assert b"read 7 offsets descend" in lib.smx_last_error()
        check_usable()
        # seq_off[n] > n_bases: the tensor holds every byte, only n_bases is short
        assert call(bases.data_ptr(), n_bases - 1, offsets.data_ptr()) == _lib.SMX_ERR_ARG
        assert ("read %d" % (n - 1)).encode() in lib.smx_last_error()
        check_usable()
        # host memory where device memory belongs
        host_off = np.ascontiguousarray(offsets.cpu().numpy().astype(np.uint64))
        assert call(bases.data_ptr(), n_bases, host_off.ctypes.data) == _lib.SMX_ERR_ARG
        host_bases = np.frombuffer(bytes(bases.cpu().numpy()), dtype=np.uint8).copy()
        assert call(host_bases.ctypes.data, n_bases, offsets.data_ptr()) == _lib.SMX_ERR_ARG
        host_rec = np.zeros((cap, 64), dtype=np.uint8)
        assert call(bases.data_ptr(), n_bases, offsets.data_ptr(), rec_ptr=host_rec.ctypes.data) == _lib.SMX_ERR_ARG
        check_usable()
        # wrong dtype, shape, contiguity or device: ValueError before any C call
        for b, o in ((bases.to(torch.int8), offsets), (bases, offsets.to(torch.int32)), (bases, offsets.double()),
                     (bases.view(1, -1), offsets), (bases, offsets.view(1, -1)), (bases[::2], offsets),
                     (torch.stack([bases, bases], 1)[:, 0], offsets), (bases, torch.stack([offsets, offsets], 1)[:, 0]),
                     (bases.cpu(), offsets), (bases, offsets.cpu()), (bases, offsets[:1])):
            with pytest.raises(ValueError):
                m.match_device(b, o)
        check_usable()
        # too small a record capacity: the exact need, then success with it
        small = want.records.shape[0] - 1
        assert call(bases.data_ptr(), n_bases, offsets.data_ptr(), cap_=small) == _lib.SMX_ERR_CAPACITY
        assert n_rec.value == want.records.shape[0]
        assert call(bases.data_ptr(), n_bases, offsets.data_ptr(), cap_=n_rec.value) == _lib.SMX_OK
        assert rec[:n_rec.value].cpu().numpy().tobytes() == want.records.tobytes()
        assert np.array_equal(ro.cpu().numpy().view(np.uint32), want.rec_offset)
        assert n_mat.value == want.n_matched


@pytest.mark.gpu
def test_routes_interleave_on_one_matcher():
    import torch
    mt, codes, offs = _ont037_with_exotic(140_000, seed=8)
    batch = PackedBatch.from_blob(codes.tobytes(), offs, clip=mt.parameters.search_len)
    bases, offsets = torch.tensor(codes, device="cuda"), torch.tensor(offs.astype(np.int64), device="cuda")
    with Matcher(mt) as m:
        want = m.match(batch)
        m.upload(batch)
        m.run_resident()
        resident = m.download()
        assert resident.records.tobytes() == want.records.tobytes()
        for _ in range(2):
            _assert_equal(m.match_device(bases, offsets), want, "device")
            m.upload(batch)
            _assert_equal(m.match_device(bases, offsets), want, "device after upload")
            m.upload(batch)
            m.run_resident()
            got = m.download()
            assert got.records.tobytes() == want.records.tobytes() and np.array_equal(got.rec_offset, want.rec_offset)
            got = m.match(batch)
            assert got.records.tobytes() == want.records.tobytes() and np.array_equal(got.rec_offset, want.rec_offset)
