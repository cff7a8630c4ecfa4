"""Batching layer over the C ABI: pack reads, run the GPU path, hand back numpy records.

`Matcher` owns one device context (one per GPU; not re-entrant).  There is no CPU path: a
missing library raises ImportError, a missing GPU raises SmxError(SMX_ERR_NO_DEVICE).
"""
import ctypes as C
import os
import threading
from typing import List, Optional, Sequence

import numpy as np

from . import _lib


class PackedBatch:
    """Reads in the smx_batch encoding (2-bit stream + optional exact 4-bit side stream), held in
    pinned host memory.  `clip` (0 or >= search_len) stores only the first/last `clip` bases of
    longer reads -- the only bases the path looks at -- which cuts packing work and H2D bytes."""

    def __init__(self, bases: Sequence[str], clip: int = 0):
        n = len(bases)
        lens = np.fromiter((len(s) for s in bases), dtype=np.uint64, count=n)
        seq_off = np.zeros(n + 1, dtype=np.uint64)
        np.cumsum(lens, out=seq_off[1:])
        blob = "".join(bases).encode("latin-1", "replace")
        self._init_from_blob(blob, seq_off, clip)

    @classmethod
    def from_blob(cls, blob: bytes, seq_off: np.ndarray, clip: int = 0):
        self = cls.__new__(cls)
        self._init_from_blob(blob, np.ascontiguousarray(seq_off, dtype=np.uint64), clip)
        return self

    @classmethod
    def from_block(cls, block, clip: int = 0, reuse: "PackedBatch" = None):
        """Packs a native_io.ReadBlock straight from the reader's memory (no Python strings).
        `reuse`: a PackedBatch whose pinned buffers are recycled when they are large enough."""
        self = reuse if reuse is not None else cls.__new__(cls)
        self._init_from_blob(block.bases_ptr or b"", block.seq_off(), clip)
        return self

    @classmethod
    def reserve(cls, n_reads: int, clip: int):
        """An empty batch whose pinned buffers already hold `n_reads` clipped reads: a pipeline that re-packs into
        it (from_block(..., reuse=...)) then never allocates or frees pinned memory while the GPU is busy --
        cudaHostAlloc / cudaFreeHost synchronise with every device of the process."""
        self = cls.__new__(cls)
        if clip:
            stride = int(_lib.load().smx_pack_stride(clip))
            self._buffer(0, n_reads * stride + 1, np.uint32)
            for slot, dt in ((2, np.uint32), (3, np.uint64), (4, np.uint16)):
                self._buffer(slot, max(n_reads, 1), dt)
        self.n_reads = 0
        return self

    def _buffer(self, slot, count, dtype):
        """Pinned host buffer `slot`, grown geometrically and kept across repacks."""
        bufs = self.__dict__.setdefault("_bufs", {})
        hb = bufs.get(slot)
        if hb is None or len(hb.array) < count:
            if hb is not None:
                hb.free()
            hb = bufs[slot] = _lib.HostBuffer(max(int(count * 1.25), 1), dtype)
        return hb.array[:count]

    def _init_from_blob(self, blob, seq_off, clip):
        """blob: bytes, or the address of the concatenated bases.  Clipped batches (clip > 0) are packed at a fixed
        stride (no per-read offsets on the wire) with 16-bit lengths when every read is shorter than 65,536."""
        lib = _lib.load()
        n = len(seq_off) - 1
        seq_off = np.ascontiguousarray(seq_off, dtype=np.uint64)
        w2, w4 = C.c_uint64(0), C.c_uint64(0)
        lib.smx_pack_bound(_lib.ptr(seq_off, _lib.u64p), n, clip, C.byref(w2), C.byref(w4))
        self.n_reads = n
        self.clip = int(clip)
        self.stride = int(lib.smx_pack_stride(clip)) if clip else 0
        self.lengths = self._buffer(2, max(n, 1), np.uint32)
        self.off4 = self._buffer(3, max(n, 1), np.uint64)
        packed4 = np.zeros(int(w4.value), dtype=np.uint32)
        used4, flagged = C.c_uint64(0), C.c_uint32(0)
        src = blob if isinstance(blob, (bytes, bytearray)) else C.cast(C.c_void_p(int(blob)), C.c_char_p)
        if self.stride:
            self.packed2 = self._buffer(0, n * self.stride + 1, np.uint32)
            self.word_off = None
            l16 = self._buffer(4, max(n, 1), np.uint16)
            fit = C.c_int(0)
            _lib.check(lib.smx_pack_reads_fixed(src, _lib.ptr(seq_off, _lib.u64p), n, clip, _lib.ptr(self.packed2, _lib.u32p),
                                                _lib.ptr(self.lengths, _lib.u32p), _lib.ptr(l16, _lib.u16p), C.byref(fit),
                                                _lib.ptr(packed4, _lib.u32p), _lib.ptr(self.off4, _lib.u64p),
                                                C.byref(used4), C.byref(flagged)))
            self.lengths16 = l16 if fit.value else None
        else:
            self.packed2 = self._buffer(0, int(w2.value), np.uint32)
            self.word_off = self._buffer(1, max(n, 1), np.uint64)
            self.lengths16 = None
            _lib.check(lib.smx_pack_reads(src, _lib.ptr(seq_off, _lib.u64p), n, clip, _lib.ptr(self.packed2, _lib.u32p),
                                          _lib.ptr(self.word_off, _lib.u64p), _lib.ptr(self.lengths, _lib.u32p),
                                          _lib.ptr(packed4, _lib.u32p), _lib.ptr(self.off4, _lib.u64p),
                                          C.byref(used4), C.byref(flagged)))
        self.n_flagged = int(flagged.value)
        self.packed4 = packed4[:int(used4.value)].copy() if self.n_flagged else None
        self.h2d_bytes = (self.packed2.nbytes + (self.word_off.nbytes if self.word_off is not None else 0) +
                          (self.lengths16.nbytes if self.lengths16 is not None else self.lengths.nbytes) +
                          (self.packed4.nbytes + self.off4.nbytes if self.n_flagged else 0))

    def c_batch(self) -> "_lib.SmxBatch":
        b = _lib.SmxBatch()
        b.n_reads = self.n_reads
        b.clip_len = self.clip
        b.packed2 = _lib.ptr(self.packed2, _lib.u32p)
        b.packed2_words = len(self.packed2)
        b.stride_words = self.stride
        b.word_off = _lib.ptr(self.word_off, _lib.u64p) if self.word_off is not None else None
        b.lengths = _lib.ptr(self.lengths, _lib.u32p)
        b.lengths16 = _lib.ptr(self.lengths16, _lib.u16p) if self.lengths16 is not None else None
        if self.n_flagged:
            b.packed4 = _lib.ptr(self.packed4, _lib.u32p)
            b.packed4_words = len(self.packed4)
            b.off4 = _lib.ptr(self.off4, _lib.u64p)
        else:
            b.packed4 = None
            b.packed4_words = 0
            b.off4 = None
        return b


class BatchResult:
    def __init__(self, rec_offset, records, n_matched, primer_hits=None, endmask=None, barcode_hits=None, orient_hits=None):
        self.rec_offset = rec_offset
        self.records = records
        self.n_matched = n_matched
        self.primer_hits = primer_hits      # [2*n_primers, n_reads]
        self.endmask = endmask              # [2*n_primers, mask_words, n_reads] uint32
        self.barcode_hits = barcode_hits    # [total_barcode_slots, n_reads]
        self.orient_hits = orient_hits      # [2*n_primers, n_reads] uint8 (explicit orientation test, irregular reads)
        self.barcode_loc_hits = None        # detail="locations": every barcode hit at every primer end location


class DeviceBatchResult:
    """Result of Matcher.match_device, left in device memory: `records` is a torch.uint8 CUDA tensor [n_records, 64] of
    smx_record rows, `rec_offset` a torch.int32 CUDA tensor [n_reads + 1] (read r owns records
    [rec_offset[r], rec_offset[r + 1]))."""

    def __init__(self, records, rec_offset, n_matched: int, device_ms=(0.0, 0.0)):
        self.records = records
        self.rec_offset = rec_offset
        self.n_matched = n_matched
        self.device_ms = device_ms          # (pack kernels, whole call) in ms, CUDA events

    def to_host(self) -> BatchResult:
        """The same result as numpy arrays in host memory: what Matcher.match returns for the same reads packed with
        PackedBatch(reads, clip=search_len), byte for byte."""
        records = np.ascontiguousarray(self.records.cpu().numpy()).view(_lib.RECORD_DTYPE).reshape(-1)
        rec_offset = np.ascontiguousarray(self.rec_offset.cpu().numpy()).view(np.uint32)
        return BatchResult(rec_offset, records, self.n_matched)


def _file_paths(tables, keys, prefix: str, fastq: bool):
    """The relative path of each file key of smx_demux_device / smx_demux_files_device, named as smx_writer names the
    file: <top>/<pool>/<p1>-<p2>/<prefix><sample file id><ext>, and full/<pool>/<prefix><sample file id><ext> for the
    pool-level copies of full matches (top 3)."""
    from .constants import SampleId
    from .native_io import safe_file_id
    t = tables
    samples = ([safe_file_id(s) for s in t.specimen_ids], [safe_file_id(SampleId.PREFIX_FWD_MATCH + b) for b in t.b1],
               [safe_file_id(SampleId.PREFIX_REV_MATCH + b) for b in t.b2])
    ext = ".fastq" if fastq else ".fasta"
    out = []
    for key in (int(k) for k in keys):
        top, pool, p1, p2 = key >> 62, (key >> 52) & 1023, (key >> 44) & 255, (key >> 36) & 255
        kind, sample = (key >> 30) & 3, key & ((1 << 30) - 1)
        pool_dir = t.pools[pool - 1] if pool else "unknown"
        name = prefix + (samples[kind][sample] if kind < 3 else "unknown") + ext
        if top == 3:
            out.append("/".join(("full", pool_dir, name)))
        else:
            out.append("/".join((("full", "partial", "unknown")[top], pool_dir,
                                 "%s-%s" % (t.primer_names[p1 - 1] if p1 else "unknown", t.primer_names[p2 - 1] if p2 else "unknown"),
                                 name)))
    return out


class DeviceDemux:
    """Result of Matcher.demux_device, left in device memory: what the output-tree writer (native_io.TreeWriter) writes,
    without the header lines, grouped by the file it goes to.  Output i is record `record[i]` of `result`; its sequence
    is seq[offsets[i]:offsets[i + 1]] (trimmed, reverse-complemented where the record says so) and its qualities the same
    slice of `qual` (None for reads without qualities).  Destination g owns outputs [group_offset[g], group_offset[g + 1])
    and has the key group_key[g] (smx_demux_device, include/specimux_b200.h); within a destination the outputs keep
    record order.  The pool-level copies of full matches (full/<pool>/<sample>) are not groups of their own: such a file
    holds the full-match outputs (resolution full match or dereplicated full match) of that pool and specimen, in
    `record` order.  Matcher.demux_files_device gives the complete files instead: headers and pool-level copies included."""

    def __init__(self, result, seq, qual, offsets, record, group_key, group_offset, tables, device_ms=(0.0, 0.0)):
        self.result = result                # DeviceBatchResult of the records
        self.seq = seq                      # torch.uint8 CUDA tensor of every output's bases
        self.qual = qual                    # same for the qualities, or None
        self.offsets = offsets              # torch.int64 CUDA tensor, n_out + 1
        self.record = record                # torch.int64 CUDA tensor, n_out: the record of each output
        self.group_key = group_key          # numpy uint64, n_groups
        self.group_offset = group_offset    # numpy int64, n_groups + 1
        self.tables = tables
        self.device_ms = device_ms          # (copy kernels, whole call) in ms, CUDA events

    def groups(self, prefix: str = "", fastq: bool = True):
        """[(relative_path, start, stop)] per destination: the path of its file in the output tree, named as
        smx_writer names the primary files, and its outputs [start, stop)."""
        paths = _file_paths(self.tables, self.group_key, prefix, fastq)
        return [(p, int(self.group_offset[g]), int(self.group_offset[g + 1])) for g, p in enumerate(paths)]


class DeviceFiles:
    """Result of Matcher.demux_files_device: every file of the output tree this batch appends to, complete, in one
    device buffer.  File f is data[file_offset[f]:file_offset[f + 1]] and goes to `paths[f]` (relative to the output
    directory; pool-level copies of full matches included), in file-key order (smx_demux_files_device).  Output i is
    the formatted record of record `record[i]` of `result`, data[offsets[i]:offsets[i + 1]].  The bytes equal what
    native_io.TreeWriter appends to each file for the same records and reads."""

    def __init__(self, result, data, file_key, file_offset, paths, record, offsets, device_ms=(0.0, 0.0), fastq=True):
        self.result = result                # DeviceBatchResult of the records
        self.data = data                    # torch.uint8 CUDA tensor
        self.file_key = file_key            # numpy uint64, n_files
        self.file_offset = file_offset      # numpy int64, n_files + 1
        self.paths = paths                  # [str], n_files
        self.record = record                # torch.int64 CUDA tensor, n_outputs
        self.offsets = offsets              # torch.int64 CUDA tensor, n_outputs + 1
        self.device_ms = device_ms          # (copy kernels, whole call) in ms, CUDA events
        self.fastq = fastq                  # FASTQ records (else FASTA)

    def host_data(self):
        """`data` in host memory: one copy into pinned memory (a numpy array or bytes is returned as it is)."""
        if isinstance(self.data, (bytes, bytearray, np.ndarray)):
            return np.frombuffer(self.data, dtype=np.uint8) if not isinstance(self.data, np.ndarray) else self.data
        import torch
        host = torch.empty(self.data.shape, dtype=torch.uint8, pin_memory=True)
        host.copy_(self.data)
        return host.numpy()

    def write(self, output_dir):
        """Appends each file's bytes to <output_dir>/<path>, creating directories: the writer's append semantics, so that
        batch after batch builds the tree."""
        host = self.host_data()
        made = set()
        for f, path in enumerate(self.paths):
            full = os.path.join(output_dir, path)
            d = os.path.dirname(full)
            if d not in made:
                os.makedirs(d, exist_ok=True)
                made.add(d)
            with open(full, "ab") as fh:
                fh.write(memoryview(host[int(self.file_offset[f]):int(self.file_offset[f + 1])]))


class DeviceMined:
    """Result of Matcher.mine_device: the `.mined` files specimine writes for the pool-level full files of a DeviceFiles
    tree, complete, in one device buffer.  File j is data[file_offset[j]:file_offset[j + 1]] and goes to `paths[j]`
    (<full file path>.mined, relative to the tree's root); an empty range is a file with no mined reads, which specimine
    writes empty.  Mined record r rewrites the partial read of output `partial[r]` of the DeviceFiles; its best full read
    is output `winner[r]`, at edit distance `distance[r]`.  `skipped` lists the pool-level files specimine skips, with the
    message it logs."""

    def __init__(self, data, file_offset, paths, partial, winner, distance, skipped, device_ms=(0.0, 0.0)):
        self.data = data                    # torch.uint8 CUDA tensor
        self.file_offset = file_offset      # numpy int64, n_files + 1
        self.paths = paths                  # [str], n_files
        self.partial = partial              # torch.int64 CUDA tensor, n_records
        self.winner = winner                # torch.int64 CUDA tensor, n_records
        self.distance = distance            # torch.int32 CUDA tensor, n_records
        self.skipped = skipped              # [(pool-level file path, reason)]
        self.device_ms = device_ms          # (search kernels, whole call) in ms, CUDA events

    def write(self, output_dir):
        """Creates or truncates <output_dir>/<path> for every file and writes its bytes, as specimine opens it ("w")."""
        host = np.asarray(self.data.cpu() if hasattr(self.data, "cpu") else self.data, dtype=np.uint8)
        for j, path in enumerate(self.paths):
            full = os.path.join(output_dir, path)
            os.makedirs(os.path.dirname(full), exist_ok=True)
            with open(full, "wb") as fh:
                fh.write(memoryview(host[int(self.file_offset[j]):int(self.file_offset[j + 1])]))


def mine_plan(files, index_file: str, partial_forward: bool, no_partial_reverse: bool):
    """specimine's discovery over the pool-level full files of a DeviceFiles tree (specimine.select_in_tree) and the
    group table of smx_mine_device it gives: per .mined file its groups, forward before reverse as specimine.mine_files
    orders them, each the full file and its partial files.  Returns (jobs, skipped, (grp_file, grp_kind, grp_part_off,
    grp_part, mined_grp) as numpy arrays, the distinct partial files)."""
    from . import specimine
    pool_level = [p for p, k in zip(files.paths, files.file_key) if int(k) >> 62 == 3]
    jobs, skipped = specimine.select_in_tree(pool_level + [p for p in files.paths if p.startswith("partial/")], index_file,
                                             partial_forward, no_partial_reverse)
    index = {p: f for f, p in enumerate(files.paths)}
    grp_file, grp_kind, part_off, part, mined_grp = [], [], [0], [], [0]
    distinct = set()
    for path, by_kind in jobs:
        for kind in ("forward", "reverse"):
            if kind not in by_kind:
                continue
            grp_file.append(index[path])
            grp_kind.append(0 if kind == "forward" else 1)
            part.extend(index[p] for p in by_kind[kind])
            distinct.update(index[p] for p in by_kind[kind])
            part_off.append(len(part))
        mined_grp.append(len(grp_file))
    u32 = lambda x: np.ascontiguousarray(x, dtype=np.uint32)
    return jobs, skipped, (u32(grp_file), np.ascontiguousarray(grp_kind, dtype=np.uint8), u32(part_off), u32(part),
                           u32(mined_grp)), sorted(distinct)


def name_blob(tables):
    """The name tables of smx_demux_files_device in one blob: specimen ids, b1 ids, b2 ids, pools, primer names (UTF-8,
    as native_io.TreeWriter passes them).  Returns (bytes, uint64 offsets, uint32 counts)."""
    from .constants import SampleId
    tables_ = (list(tables.specimen_ids), [SampleId.PREFIX_FWD_MATCH + b for b in tables.b1],
               [SampleId.PREFIX_REV_MATCH + b for b in tables.b2], list(tables.pools), list(tables.primer_names))
    names = [s.encode("utf-8", "surrogateescape") for t in tables_ for s in t]
    off = np.zeros(len(names) + 1, dtype=np.uint64)
    np.cumsum([len(s) for s in names], out=off[1:])
    return b"".join(names), off, np.array([len(t) for t in tables_], dtype=np.uint32)


def _check_device_tensor(fn, name, t, dtype, device):
    """ValueError naming `fn` and `name` unless `t` is a 1-D contiguous torch tensor of `dtype` on cuda:`device`."""
    import torch
    if not isinstance(t, torch.Tensor):
        raise ValueError("%s: %s must be a torch tensor, not %s" % (fn, name, type(t).__name__))
    if t.dtype != dtype:
        raise ValueError("%s: %s must be %s, not %s" % (fn, name, dtype, t.dtype))
    if t.dim() != 1:
        raise ValueError("%s: %s must be 1-D, not %d-D" % (fn, name, t.dim()))
    if not t.is_contiguous():
        raise ValueError("%s: %s must be contiguous" % (fn, name))
    if t.device.type != "cuda" or t.device.index != device:
        raise ValueError("%s: %s is on %s, the Matcher on cuda:%d" % (fn, name, t.device, device))


def _capacity_retry(run, cap, need):
    """Runs a device route as `run(cap)` -> (rc, result) with the estimated capacity `cap`; when that is too small
    (SMX_ERR_CAPACITY), once more with `need()`, the exact size the first run reported.  Any other failure raises
    SmxError.  Returns the result."""
    rc, result = run(cap)
    if rc == _lib.SMX_ERR_CAPACITY:
        rc, result = run(need())
    _lib.check(rc)
    return result


class Matcher:
    """One device context.  `binding` lets the unit tests drive the same host code through the CPU
    kernel simulator (tests/hostsim); the product never passes it, and it is refused unless the test suite
    has opened the seam (SMX_TEST_SEAM=1, set by tests/conftest.py): there is no CPU execution route
    through the product API."""

    def __init__(self, tables, device: int = 0, binding=None):
        if binding is not None and os.environ.get("SMX_TEST_SEAM") != "1":
            raise RuntimeError("specimux_b200: the simulator binding is a test seam (SMX_TEST_SEAM=1); "
                               "the matching runs on the GPU only")
        self.tables = tables
        self.device = int(device)
        self._binding = binding
        self._ctx = C.c_void_p(None)
        self._lock = threading.Lock()
        if binding is None:
            self._lib = _lib.load()
            _lib.check(self._lib.smx_create(device, tables.tables_ref(), tables.params_ref(), C.byref(self._ctx)))
        else:
            self._lib = None

    def close(self):
        if self._lib is not None and self._ctx:
            self._lib.smx_destroy(self._ctx)
            self._ctx = C.c_void_p(None)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- results allocation ---------------------------------------------------------------
    def _alloc_results(self, n, detail, cap=None, reuse=False, compact=False):
        t = self.tables
        cap = int(cap if cap is not None else n + n // 8 + 1024)
        res = _lib.SmxResults()
        wire = compact == "wire"
        rec_dtype = _lib.RECORD16_DTYPE if wire else _lib.RECORD32_DTYPE if compact else _lib.RECORD_DTYPE
        rec_key = "rec16" if wire else "rec32" if compact else "rec"
        if reuse is not None and reuse is not False:
            # pinned pool reused across calls: the previous call's result arrays are overwritten.
            # reuse=True: one pool per Matcher; reuse=<dict>: a pool owned by the caller (lets several
            # results stay alive, e.g. while a writer thread still formats an earlier batch)
            pool = reuse if isinstance(reuse, dict) else self.__dict__.setdefault("_result_pool", {})
            # grown geometrically: every growth is a cudaHostAlloc + (later) cudaFreeHost, and both synchronise with
            # the devices -- batches of slightly different sizes must not reallocate each time
            if pool.get("n", -1) < n + 1:
                grown = n + 1 if "n" not in pool else n + n // 4 + 1024
                pool["n"], pool["off"] = grown, _lib.HostBuffer(grown, np.uint32)
            if pool.get("cap_" + rec_key, -1) < cap:
                grown = cap if ("cap_" + rec_key) not in pool else cap + cap // 4 + 1024
                pool["cap_" + rec_key], pool[rec_key] = grown, _lib.HostBuffer(grown, rec_dtype)
            rec_offset = pool["off"].array[:n + 1]
            records = pool[rec_key].array[:cap]
        else:
            rec_offset = np.empty(n + 1, dtype=np.uint32)
            records = np.empty(cap, dtype=rec_dtype)
        if wire:
            rec_offset = None                       # the last-of-read flags carry the grouping
            res.rec_offset = None
            res.records16 = records.ctypes.data
        else:
            res.rec_offset = _lib.ptr(rec_offset, _lib.u32p)
            if compact:
                res.records32 = records.ctypes.data
            else:
                res.records = records.ctypes.data
        res.records_cap = cap
        ph = em = bh = oh = None
        if detail:
            ph = np.zeros((2 * t.n_primers, n), dtype=_lib.PRIMER_HIT_DTYPE)
            em = np.zeros((2 * t.n_primers, t.mask_words, n), dtype=np.uint32)
            bh = np.zeros((max(t.total_barcode_slots, 1), n), dtype=_lib.BARCODE_HIT_DTYPE)
            res.primer_hits = ph.ctypes.data
            res.endmask_bits = em.ctypes.data
            oh = np.zeros((2 * t.n_primers, n), dtype=np.uint8)
            res.barcode_hits = bh.ctypes.data
            res.orient_hits = oh.ctypes.data
            lh = None
            if detail == "locations":
                lh = np.zeros(max(int(self.__dict__.get("_loc_cap", 0)), 64 * n + 1024), dtype=_lib.BARCODE_LOC_HIT_DTYPE)
                res.barcode_loc_hits = lh.ctypes.data
                res.barcode_loc_cap = len(lh)
            return res, rec_offset, records, ph, em, (bh, oh, lh)
        return res, rec_offset, records, ph, em, (bh, None, None)

    def _finish(self, res, rec_offset, records, ph, em, bh):
        bh, oh, lh = bh
        out = BatchResult(rec_offset, records[:int(res.n_records)], int(res.n_matched), ph, em, bh, oh)
        if lh is not None:
            out.barcode_loc_hits = lh[:min(int(res.n_barcode_loc_hits), len(lh))]
        return out

    def reserve_results(self, pool: dict, n: int, compact=False):
        """Sizes a caller-owned pinned result pool for batches of up to `n` reads ahead of the first match."""
        self._alloc_results(int(n), False, None, pool, compact)

    # -- whole path with host buffers (H2D + kernels + D2H) ---------------------------------
    def match(self, batch: PackedBatch, detail: bool = False, reuse=False, compact: bool = False) -> BatchResult:
        """`reuse=True` returns views into a pinned pool that the next reuse=True call overwrites;
        `reuse=<dict>` uses (and grows) a caller-owned pool instead.  `compact=True` returns 32-byte
        smx_record32 records (no location pairs); `compact="wire"` the 16-byte smx_record16 records in read
        order (what the output-tree writer needs; no rec_offset).  A context is not
        re-entrant: calls from several threads are serialised here."""
        with self._lock:
            return self._match_locked(batch, detail, reuse, compact)

    def _match_locked(self, batch, detail, reuse, compact=False):
        cb = batch.c_batch()
        cap = None
        while True:
            res, rec_offset, records, ph, em, bh = self._alloc_results(batch.n_reads, detail, cap, reuse, compact)
            if self._binding is not None:
                rc = self._binding.hostsim_match_batch(self.tables.tables_ref(), self.tables.params_ref(),
                                                       C.byref(cb), C.byref(res))
                if rc == _lib.SMX_ERR_CAPACITY:
                    cap = int(res.n_records)
                    continue
                if rc != 0:
                    raise _lib.SmxError(rc, self._binding.hostsim_last_error().decode())
            else:
                rc = self._lib.smx_match_batch(self._ctx, C.byref(cb), C.byref(res))
                if rc == _lib.SMX_ERR_CAPACITY:
                    cap = int(res.n_records)
                    continue
                _lib.check(rc)
            if detail == "locations" and int(res.n_barcode_loc_hits) > int(res.barcode_loc_cap):
                self._loc_cap = int(res.n_barcode_loc_hits) + 1024
                continue
            return self._finish(res, rec_offset, records, ph, em, bh)

    # -- whole path with reads already in device memory (packed there) -------------------------
    def _device_route(self, fn):
        if self._binding is not None:
            raise RuntimeError("%s needs the CUDA library: a Matcher on the kernel simulator has no device route" % fn)

    def match_device(self, bases, offsets) -> DeviceBatchResult:
        """Matches reads held in GPU memory without a copy to the host: `bases` is a 1-D contiguous torch.uint8 CUDA
        tensor of concatenated reads, `offsets` a 1-D contiguous torch.int64 CUDA tensor of n + 1 offsets into it, both
        on this Matcher's device.  The reads are packed on the device with clip = search_len and the work is ordered
        after what is already enqueued on torch.cuda.current_stream(device); the call returns when the result is
        written.  Records equal match(PackedBatch(reads, clip=search_len)) (see DeviceBatchResult.to_host)."""
        self._device_route("match_device")
        import torch
        _check_device_tensor("match_device", "bases", bases, torch.uint8, self.device)
        _check_device_tensor("match_device", "offsets", offsets, torch.int64, self.device)
        n = offsets.numel() - 1
        if n < 1 or n > 0xFFFFFFFF:
            raise ValueError("match_device: offsets must hold n + 1 entries for 1 <= n < 2^32 reads, not %d" % (n + 1))
        with self._lock:
            dev = torch.device("cuda", self.device)
            stream = torch.cuda.current_stream(dev).cuda_stream
            cap = int(self._lib.smx_result_bound(self._ctx, n))
            n_records, n_matched = C.c_uint64(0), C.c_uint64(0)
            ms = (C.c_float * 2)()

            def run(cap):
                records = torch.empty((cap, _lib.RECORD_DTYPE.itemsize), dtype=torch.uint8, device=dev)
                rec_offset = torch.empty(n + 1, dtype=torch.int32, device=dev)
                rc = self._lib.smx_match_device(self._ctx, bases.data_ptr() or None, bases.numel(), offsets.data_ptr(), n,
                                                stream, rec_offset.data_ptr(), records.data_ptr(), cap,
                                                C.byref(n_records), C.byref(n_matched), ms)
                return rc, (records, rec_offset)
            records, rec_offset = _capacity_retry(run, cap, lambda: int(n_records.value))
            return DeviceBatchResult(records[:int(n_records.value)], rec_offset, int(n_matched.value), (float(ms[0]), float(ms[1])))

    def demux_device(self, bases, offsets, quals=None) -> DeviceDemux:
        """match_device, then the demultiplexed output of its records, all in GPU memory: the trimmed, oriented
        sequences (and qualities) grouped by the file of the output tree each goes to (see DeviceDemux).  `quals`, when
        given, is a contiguous torch.uint8 CUDA tensor shaped like `bases`.  Ordered after the work already enqueued on
        torch.cuda.current_stream(device); returns when everything is written."""
        self._device_route("demux_device")
        import torch
        if quals is not None:
            _check_device_tensor("demux_device", "quals", quals, torch.uint8, self.device)
            if isinstance(bases, torch.Tensor) and quals.shape != bases.shape:
                raise ValueError("demux_device: quals must be shaped like bases %s, not %s" % (tuple(bases.shape), tuple(quals.shape)))
        return self._demux(self.match_device(bases, offsets), bases, offsets, quals)

    def _demux(self, result, bases, offsets, quals):
        import torch
        n_rec = int(result.records.shape[0])
        n = offsets.numel() - 1
        with self._lock:
            dev = torch.device("cuda", self.device)
            stream = torch.cuda.current_stream(dev).cuda_stream
            order = torch.empty(n_rec, dtype=torch.int64, device=dev)
            out_off = torch.empty(n_rec + 1, dtype=torch.int64, device=dev)
            group_key = torch.empty(n_rec, dtype=torch.int64, device=dev)
            group_off = torch.empty(n_rec + 1, dtype=torch.int64, device=dev)
            n_groups, n_bytes = C.c_uint64(0), C.c_uint64(0)
            ms = (C.c_float * 2)()
            cap = bases.numel()                 # enough unless a read gives several records: then once more, exactly

            def run(cap):
                seq = torch.empty(cap, dtype=torch.uint8, device=dev)
                qual = torch.empty(cap, dtype=torch.uint8, device=dev) if quals is not None else None
                rc = self._lib.smx_demux_device(
                    self._ctx, bases.data_ptr() or None, (quals.data_ptr() or None) if quals is not None else None, bases.numel(),
                    offsets.data_ptr(), n, result.records.data_ptr() or None, n_rec, stream, order.data_ptr() or None,
                    out_off.data_ptr(), seq.data_ptr() or None, qual.data_ptr() or None if qual is not None else None, cap,
                    group_key.data_ptr() or None, group_off.data_ptr(), C.byref(n_groups), C.byref(n_bytes), ms)
                return rc, (seq, qual)
            seq, qual = _capacity_retry(run, cap, lambda: int(n_bytes.value))
            g, total = int(n_groups.value), int(n_bytes.value)
            return DeviceDemux(result, seq[:total], qual[:total] if qual is not None else None, out_off, order,
                               group_key[:g].cpu().numpy().view(np.uint64), group_off[:g + 1].cpu().numpy(), self.tables,
                               (float(ms[0]), float(ms[1])))

    def demux_files_device(self, bases, offsets, titles, title_offsets, quals=None, prefix: str = "",
                           fastq: bool = True) -> DeviceFiles:
        """match_device, then every file of the output tree the records go to, complete and in GPU memory (see
        DeviceFiles): what native_io.TreeWriter(output_dir, prefix, fastq, tables) appends for the same reads.  `titles`
        is a 1-D contiguous torch.uint8 CUDA tensor of the reads' title lines (without '@' / '>') back to back and
        `title_offsets` a torch.int64 CUDA tensor of n + 1 offsets into it, as the native reader's block holds them;
        `quals` as for demux_device.  FASTQ output without `quals` writes 'I' for every base; FASTA output
        (fastq=False) ignores `quals`.  Ordered after the work already enqueued on torch.cuda.current_stream(device);
        returns when everything is written."""
        self._device_route("demux_files_device")
        import torch
        n = offsets.numel() - 1 if isinstance(offsets, torch.Tensor) else -1
        _check_device_tensor("demux_files_device", "titles", titles, torch.uint8, self.device)
        _check_device_tensor("demux_files_device", "title_offsets", title_offsets, torch.int64, self.device)
        if quals is not None:
            _check_device_tensor("demux_files_device", "quals", quals, torch.uint8, self.device)
            if isinstance(bases, torch.Tensor) and quals.shape != bases.shape:
                raise ValueError("demux_files_device: quals must be shaped like bases %s, not %s" % (tuple(bases.shape), tuple(quals.shape)))
        if title_offsets.numel() - 1 != n:
            raise ValueError("demux_files_device: title_offsets must hold n + 1 = %d entries, not %d" % (n + 1, title_offsets.numel()))
        result = self.match_device(bases, offsets)
        return self._demux_files(result, bases, offsets, titles, title_offsets, quals if fastq else None, prefix, fastq)

    def _demux_files(self, result, bases, offsets, titles, title_offsets, quals, prefix, fastq):
        import torch
        n_rec = int(result.records.shape[0])
        n = offsets.numel() - 1
        with self._lock:
            dev = torch.device("cuda", self.device)
            stream = torch.cuda.current_stream(dev).cuda_stream
            names = self.__dict__.get("_names_dev")
            if names is None:
                blob, off, counts = name_blob(self.tables)
                names = self._names_dev = (torch.tensor(np.frombuffer(blob, dtype=np.uint8).copy(), device=dev),
                                           torch.tensor(off.astype(np.int64), device=dev), counts,
                                           int(np.diff(off).max()) if len(off) > 1 else 0)
            name_bytes, name_off, counts, longest = names
            record = torch.empty(2 * n_rec, dtype=torch.int64, device=dev)
            out_off = torch.empty(2 * n_rec + 1, dtype=torch.int64, device=dev)
            file_key = torch.empty(2 * n_rec, dtype=torch.int64, device=dev)
            file_off = torch.empty(2 * n_rec + 1, dtype=torch.int64, device=dev)
            n_files, n_out, n_bytes = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
            ms = (C.c_float * 2)()
            # every record at most twice, each at most its read twice plus its title and the longest names: enough
            # unless a read gives several records -- then once more, exactly
            cap = 2 * ((2 if fastq else 1) * bases.numel() + titles.numel() + n_rec * (40 + 4 * longest))

            def run(cap):
                data = torch.empty(cap, dtype=torch.uint8, device=dev)
                rc = self._lib.smx_demux_files_device(
                    self._ctx, bases.data_ptr() or None, (quals.data_ptr() or None) if quals is not None else None,
                    bases.numel(), offsets.data_ptr(), n, titles.data_ptr() or None, titles.numel(), title_offsets.data_ptr(),
                    result.records.data_ptr() or None, n_rec, name_bytes.data_ptr() or None, name_bytes.numel(),
                    name_off.data_ptr(), _lib.ptr(counts, _lib.u32p), 1 if fastq else 0, stream, record.data_ptr() or None,
                    out_off.data_ptr(), data.data_ptr() or None, cap, file_key.data_ptr() or None, file_off.data_ptr(),
                    C.byref(n_files), C.byref(n_out), C.byref(n_bytes), ms)
                return rc, data
            data = _capacity_retry(run, cap, lambda: int(n_bytes.value))
            f, k, total = int(n_files.value), int(n_out.value), int(n_bytes.value)
            keys = file_key[:f].cpu().numpy().view(np.uint64)
            return DeviceFiles(result, data[:total], keys, file_off[:f + 1].cpu().numpy(), _file_paths(self.tables, keys, prefix, fastq),
                               record[:k], out_off[:k + 1], (float(ms[0]), float(ms[1])), fastq)

    def mine_device(self, files: DeviceFiles, index: str, partial_forward: bool = False, no_partial_reverse: bool = False,
                    min_identity: float = 0.85) -> DeviceMined:
        """specimine over the tree of a DeviceFiles in GPU memory: the `.mined` file of every pool-level full file
        (full/<pool>/<prefix><sample>.fastq) that `specimine --index index --fastq <that file>` would write on the tree
        files.write(dir) builds, byte for byte, with the flags meaning what they mean there (see DeviceMined).  `files`
        must be FASTQ (demux_files_device(..., fastq=True)).  Discovery is specimine's (specimine.select_in_tree), with
        the primer-pair directories of a pool taken in sorted path order; the search, the decisions and the records run on
        the device.  The scope is one DeviceFiles, the tree of one batch: mining across the DeviceFiles of several
        batches, and mining the primer-pair-level full files full/<pool>/<pair>/<sample>.fastq, are not done here.
        A pool-level full file holds at most 2^23 reads (the search key's rank field); a larger one raises SmxError.
        Memory: the first attempt sizes the output for every distinct partial read mined once at up to twice its
        record's size (2 x the partial files' bytes, plus record arrays of a 54-byte record minimum: about 2.4 x those
        bytes of device memory in all, for a short time), so that one search suffices in the usual case; a larger need
        (a partial read mined for several specimens) reruns the call once with the exact size.  Ordered after the work already enqueued on torch.cuda.current_stream(device); returns when everything is
        written."""
        self._device_route("mine_device")
        import torch
        if not isinstance(files, DeviceFiles):
            raise ValueError("mine_device: files must be a DeviceFiles, not %s" % type(files).__name__)
        if not files.fastq:
            raise ValueError("mine_device: specimine reads FASTQ; these DeviceFiles hold FASTA")
        _check_device_tensor("mine_device", "files.data", files.data, torch.uint8, self.device)
        _check_device_tensor("mine_device", "files.offsets", files.offsets, torch.int64, self.device)
        jobs, skipped, (grp_file, grp_kind, part_off, part, mined_grp), distinct = mine_plan(files, index, partial_forward,
                                                                                             no_partial_reverse)
        file_off = np.ascontiguousarray(files.file_offset, dtype=np.uint64)
        n_out = files.offsets.numel() - 1
        with self._lock:
            dev = torch.device("cuda", self.device)
            stream = torch.cuda.current_stream(dev).cuda_stream
            mined_off = torch.empty(len(jobs) + 1, dtype=torch.int64, device=dev)
            n_rec, n_bytes = C.c_uint64(0), C.c_uint64(0)
            ms = (C.c_float * 2)()
            # every partial read mined once, each record at most twice its size: enough unless a partial read is mined
            # for several specimens -- then once more, exactly.  A mined record holds at least 54 bytes.
            cap = 2 * sum(int(file_off[f + 1] - file_off[f]) for f in distinct) + 4096
            rec_cap = cap // 54 + 1

            def run(caps):
                cap, rec_cap = caps
                data = torch.empty(cap, dtype=torch.uint8, device=dev)
                partial = torch.empty(rec_cap, dtype=torch.int64, device=dev)
                winner = torch.empty(rec_cap, dtype=torch.int64, device=dev)
                dist = torch.empty(rec_cap, dtype=torch.int32, device=dev)
                rc = self._lib.smx_mine_device(
                    self._ctx, files.data.data_ptr() or None, files.data.numel(), files.offsets.data_ptr(), n_out,
                    _lib.ptr(file_off, _lib.u64p), len(files.paths), len(grp_file), _lib.ptr(grp_file, _lib.u32p),
                    _lib.ptr(grp_kind, _lib.u8p), _lib.ptr(part_off, _lib.u32p), _lib.ptr(part, _lib.u32p), len(jobs),
                    _lib.ptr(mined_grp, _lib.u32p), float(min_identity), stream, data.data_ptr(), cap, rec_cap,
                    mined_off.data_ptr(), partial.data_ptr(), winner.data_ptr(), dist.data_ptr(), C.byref(n_rec),
                    C.byref(n_bytes), ms)
                return rc, (data, partial, winner, dist)
            data, partial, winner, dist = _capacity_retry(run, (cap, rec_cap),
                                                          lambda: (max(int(n_bytes.value), 1), max(int(n_rec.value), 1)))
            r, total = int(n_rec.value), int(n_bytes.value)
            return DeviceMined(data[:total], mined_off.cpu().numpy(), [p + ".mined" for p, _f in jobs], partial[:r],
                               winner[:r], dist[:r], skipped, (float(ms[0]), float(ms[1])))

    # -- split form -------------------------------------------------------------------------
    def upload(self, batch: PackedBatch):
        self._resident_n = batch.n_reads
        cb = batch.c_batch()
        _lib.check(self._lib.smx_upload_batch(self._ctx, C.byref(cb)))

    def run_resident(self):
        _lib.check(self._lib.smx_run_resident(self._ctx))

    def download(self, detail: bool = False, reuse: bool = False) -> BatchResult:
        cap = None
        while True:
            res, rec_offset, records, ph, em, bh = self._alloc_results(self._resident_n, detail, cap, reuse)
            rc = self._lib.smx_download_results(self._ctx, C.byref(res))
            if rc == _lib.SMX_ERR_CAPACITY:
                cap = int(res.n_records)
                continue
            _lib.check(rc)
            return self._finish(res, rec_offset, records, ph, em, bh)

    def set_pipeline_chunk(self, reads_per_chunk: int):
        """Chunk size of the pipelined smx_match_batch (0 = always one shot)."""
        _lib.check(self._lib.smx_set_pipeline_chunk(self._ctx, int(reads_per_chunk)))

    def set_resident_split(self, n_sub_batches: int):
        """Sub-batches the resident form runs concurrently (1 = one lane, per-kernel times available)."""
        _lib.check(self._lib.smx_set_resident_split(self._ctx, int(n_sub_batches)))

    def last_chunk_count(self) -> int:
        return int(self._lib.smx_last_chunk_count(self._ctx))

    # slot 3 (once the separate start-recovery kernel) is the gap between stage 1 and stage 2: ~0
    KERNEL_NAMES = ("stage_windows", "primer_sliced", "primer_finish_start", "stage_gap", "barcode_tasks",
                    "select_fast", "select_general", "scan_compact", "rebase_offsets")

    def last_kernel_times(self):
        """{kernel: ms} of the last run_resident (CUDA events on the launching stream)."""
        ms = (C.c_float * len(self.KERNEL_NAMES))()
        n = self._lib.smx_last_kernel_times(self._ctx, ms, len(self.KERNEL_NAMES))
        return {k: float(ms[i]) for i, k in enumerate(self.KERNEL_NAMES[:n])}

    def last_deferred(self) -> int:
        return int(self._lib.smx_last_deferred(self._ctx))

    def flush_l2(self):
        _lib.check(self._lib.smx_flush_l2(self._ctx))

    def last_timing(self):
        total = C.c_float(0)
        stages = (C.c_float * 4)()
        _lib.check(self._lib.smx_last_timing(self._ctx, C.byref(total), stages))
        return float(total.value), [float(x) for x in stages]

    def last_launch_count(self) -> int:
        return int(self._lib.smx_last_launch_count(self._ctx))

    def last_useful_cells(self):
        """(stage 1, stage 2) bit-sliced DP cells evaluated by the last run_resident (5 LOP3 per cell)."""
        cells = (C.c_uint64 * 2)()
        _lib.check(self._lib.smx_last_useful_cells(self._ctx, cells))
        return int(cells[0]), int(cells[1])

    def last_work(self):
        cells = (C.c_uint64 * 2)()
        wcols = (C.c_uint64 * 2)()
        _lib.check(self._lib.smx_last_work(self._ctx, cells, wcols))
        return [int(x) for x in cells], [int(x) for x in wcols]
