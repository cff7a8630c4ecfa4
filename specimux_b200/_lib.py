"""ctypes binding of libspecimux_b200.so (include/specimux_b200.h).

Loading fails loudly when the library has not been built (`python -c "import __graft_entry__ as g;
g.build()"` or `make -C specimux_b200/csrc`); compute entry points fail loudly without a GPU.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# SMX_LIB_PATH: an alternative build of the same library (A/B of compile-time knobs, tools/ab_round.sh)
LIB_PATH = os.environ.get("SMX_LIB_PATH") or os.path.join(_HERE, "libspecimux_b200.so")

SMX_OK, SMX_ERR_ARG, SMX_ERR_CUDA, SMX_ERR_NO_DEVICE, SMX_ERR_CAPACITY, SMX_ERR_INTERNAL = range(6)
TRIM_CODES = {"none": 0, "primers": 1, "barcodes": 2, "tails": 3}
NONE = -(2 ** 31)

u8p, u16p, u32p, u64p, i32p = (C.POINTER(C.c_uint8), C.POINTER(C.c_uint16), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64),
                               C.POINTER(C.c_int32))


class SmxTables(C.Structure):
    _fields_ = [("n_primers", C.c_uint32), ("primer_seq", C.c_char_p), ("primer_rc", C.c_char_p),
                ("primer_off", u32p), ("primer_dir", u8p), ("primer_k", i32p), ("primer_file_index", i32p),
                ("pb_off", u32p), ("pb_barcode", u32p),
                ("n_b1", C.c_uint32), ("n_b2", C.c_uint32),
                ("b1_rc", C.c_char_p), ("b1_off", u32p), ("b2_rc", C.c_char_p), ("b2_off", u32p),
                ("n_pairs", C.c_uint32), ("pair_fwd", u32p), ("pair_rev", u32p), ("pair_pool", i32p),
                ("n_specimens", C.c_uint32), ("spec_b1", u32p), ("spec_b2", u32p),
                ("spec_p1_mask", u64p), ("spec_p2_mask", u64p), ("spec_pool", i32p)]


class SmxParams(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("search_len", "max_dist_index", "barcode_length", "preorient",
                                         "prefilter", "trim", "dereplicate_best", "min_length", "max_length")]


class SmxBatch(C.Structure):
    _fields_ = [("n_reads", C.c_uint32), ("packed2", u32p), ("packed2_words", C.c_uint64),
                ("word_off", u64p), ("lengths", u32p), ("packed4", u32p), ("packed4_words", C.c_uint64),
                ("off4", u64p), ("clip_len", C.c_uint32), ("stride_words", C.c_uint32), ("lengths16", u16p)]


class SmxResults(C.Structure):
    _fields_ = [("rec_offset", u32p), ("records", C.c_void_p), ("records_cap", C.c_uint64),
                ("n_records", C.c_uint64), ("n_matched", C.c_uint64), ("endmask_bits", C.c_void_p),
                ("primer_hits", C.c_void_p), ("barcode_hits", C.c_void_p), ("orient_hits", C.c_void_p),
                ("barcode_loc_hits", C.c_void_p), ("barcode_loc_cap", C.c_uint64), ("n_barcode_loc_hits", C.c_uint64),
                ("records32", C.c_void_p), ("records16", C.c_void_p)]


RECORD_DTYPE = np.dtype([("read", "<u4"), ("sample", "<i4"), ("trim_start", "<i4"), ("trim_end", "<i4"),
                         ("p1_loc", "<i4", (2,)), ("p2_loc", "<i4", (2,)), ("b1_loc", "<i4", (2,)),
                         ("b2_loc", "<i4", (2,)), ("pool", "<i2"), ("p1", "<i2"), ("p2", "<i2"),
                         ("dist", "i1", (4,)), ("resolution", "u1"), ("reverse", "u1"), ("trim_empty", "u1"),
                         ("candidate", "u1"), ("pad", "u1", (2,))])
PRIMER_HIT_DTYPE = np.dtype([("first_start", "<i4"), ("first_end", "<i4"), ("distance", "<i2"),
                             ("n_locations", "<u2")])
BARCODE_HIT_DTYPE = np.dtype([("end_mask", "<u8"), ("search_start", "<i4"), ("distance", "<i2"), ("barcode", "<u2")])
RECORD32_DTYPE = np.dtype([("read", "<u4"), ("sample", "<i4"), ("trim_start", "<i4"), ("trim_end", "<i4"),
                           ("pool", "<i2"), ("p1", "<i2"), ("p2", "<i2"), ("dist", "i1", (4,)), ("resolution", "u1"),
                           ("flags", "u1"), ("candidate", "u1"), ("pad", "u1", (3,))])
assert RECORD32_DTYPE.itemsize == 32
# smx_record16, the 16-byte wire form: records in read order, flags bit 5 = last record of its read
RECORD16_DTYPE = np.dtype([("sample", "<i4"), ("trim_start", "<u2"), ("trim_tail", "<u2"), ("pool", "<i2"), ("p1", "u1"),
                           ("p2", "u1"), ("dist_p1", "u1"), ("dist_p2", "u1"), ("dist_b", "u1"), ("flags", "u1")])
assert RECORD16_DTYPE.itemsize == 16
BARCODE_LOC_HIT_DTYPE = np.dtype([("read", "<u4"), ("slot", "<u2"), ("location", "<u2"), ("hit", BARCODE_HIT_DTYPE)])
assert BARCODE_LOC_HIT_DTYPE.itemsize == 24
assert RECORD_DTYPE.itemsize == 64 and PRIMER_HIT_DTYPE.itemsize == 12 and BARCODE_HIT_DTYPE.itemsize == 16

EXPORTS = ["smx_abi_version", "smx_last_error", "smx_device_count", "smx_create", "smx_destroy",
           "smx_result_bound", "smx_match_batch", "smx_upload_batch", "smx_run_resident",
           "smx_download_results", "smx_last_timing", "smx_last_launch_count", "smx_last_work",
           "smx_pairwise_nw", "smx_pack_bound", "smx_pack_reads", "smx_int_alu_peak", "smx_host_alloc",
           "smx_host_free", "smx_flush_l2", "smx_set_pipeline_chunk", "smx_last_chunk_count", "smx_last_deferred", "smx_last_kernel_times", "smx_set_resident_split",
           "smx_device_pci_bus_id", "smx_pack_stride", "smx_pack_reads_fixed", "smx_copy_peak", "smx_last_useful_cells", "smx_hw_distances",
           "smx_hw_best_grouped", "smx_match_device", "smx_demux_device",
           "smx_demux_files_device", "smx_mine_device"]


class SmxError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("libspecimux_b200 error %d: %s" % (code, message))
        self.code = code


_lib = None


def load():
    """The CUDA library.  Raises (never falls back) when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s not built: run `make -C specimux_b200/csrc` (or __graft_entry__.build()); "
                              "specimux_b200 has no CPU matching path" % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        lib.smx_last_error.restype = C.c_char_p
        lib.smx_result_bound.restype = C.c_uint64
        lib.smx_result_bound.argtypes = [C.c_void_p, C.c_uint32]
        lib.smx_create.argtypes = [C.c_int, C.POINTER(SmxTables), C.POINTER(SmxParams), C.POINTER(C.c_void_p)]
        lib.smx_destroy.argtypes = [C.c_void_p]
        lib.smx_destroy.restype = None
        for fn in ("smx_match_batch",):
            getattr(lib, fn).argtypes = [C.c_void_p, C.POINTER(SmxBatch), C.POINTER(SmxResults)]
        lib.smx_upload_batch.argtypes = [C.c_void_p, C.POINTER(SmxBatch)]
        lib.smx_run_resident.argtypes = [C.c_void_p]
        lib.smx_download_results.argtypes = [C.c_void_p, C.POINTER(SmxResults)]
        lib.smx_last_timing.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]
        lib.smx_last_launch_count.argtypes = [C.c_void_p]
        lib.smx_last_work.argtypes = [C.c_void_p, u64p, u64p]
        lib.smx_pairwise_nw.argtypes = [C.c_int, C.c_char_p, u32p, C.c_uint32, i32p]
        lib.smx_pack_bound.argtypes = [u64p, C.c_uint32, C.c_uint32, u64p, u64p]
        lib.smx_pack_bound.restype = None
        lib.smx_pack_reads.argtypes = [C.c_char_p, u64p, C.c_uint32, C.c_uint32, u32p, u64p, u32p, u32p, u64p, u64p, u32p]
        lib.smx_int_alu_peak.argtypes = [C.c_int, C.POINTER(C.c_double)]
        lib.smx_host_alloc.argtypes = [C.c_uint64]
        lib.smx_host_alloc.restype = C.c_void_p
        lib.smx_host_free.argtypes = [C.c_void_p]
        lib.smx_host_free.restype = None
        lib.smx_flush_l2.argtypes = [C.c_void_p]
        lib.smx_set_pipeline_chunk.argtypes = [C.c_void_p, C.c_uint32]
        lib.smx_last_chunk_count.argtypes = [C.c_void_p]
        lib.smx_last_deferred.argtypes = [C.c_void_p]
        lib.smx_last_kernel_times.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.c_int]
        lib.smx_last_deferred.restype = C.c_uint64
        lib.smx_set_resident_split.argtypes = [C.c_void_p, C.c_uint32]
        lib.smx_device_pci_bus_id.argtypes = [C.c_int, C.c_char_p, C.c_int]
        lib.smx_pack_stride.argtypes = [C.c_uint32]
        lib.smx_pack_stride.restype = C.c_uint32
        lib.smx_pack_reads_fixed.argtypes = [C.c_char_p, u64p, C.c_uint32, C.c_uint32, u32p, u32p, u16p, C.POINTER(C.c_int),
                                             u32p, u64p, u64p, u32p]
        lib.smx_copy_peak.argtypes = [C.c_int, C.c_uint64, C.POINTER(C.c_double)]
        lib.smx_last_useful_cells.argtypes = [C.c_void_p, u64p]
        lib.smx_hw_distances.argtypes = [C.c_int, C.c_char_p, u64p, i32p, C.c_uint32, C.c_char_p, u64p, C.c_uint32, i32p]
        lib.smx_hw_best_grouped.argtypes = [C.c_int, C.c_char_p, u64p, i32p, C.c_uint32, C.c_char_p, u64p, C.c_uint32,
                                             C.c_uint32, u32p, u64p, u32p, i32p, i32p, C.POINTER(C.c_float)]
        lib.smx_match_device.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_uint64, u64p, u64p, C.POINTER(C.c_float)]
        lib.smx_demux_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p,
                                         C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                                         C.c_void_p, C.c_void_p, u64p, u64p, C.POINTER(C.c_float)]
        lib.smx_demux_files_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32,
                                               C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p,
                                               C.c_uint64, C.c_void_p, u32p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, u64p, u64p, u64p,
                                               C.POINTER(C.c_float)]
        lib.smx_mine_device.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, u64p, C.c_uint64,
                                        C.c_uint32, u32p, C.POINTER(C.c_uint8), u32p, u32p, C.c_uint32, u32p, C.c_double,
                                        C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, u64p, u64p, C.POINTER(C.c_float)]
        if lib.smx_abi_version() != 3:
            raise ImportError("libspecimux_b200.so ABI version mismatch")
        _lib = lib
    return _lib


def check(rc):
    if rc != SMX_OK:
        raise SmxError(rc, load().smx_last_error().decode("utf-8", "replace"))


def ptr(arr, typ):
    return arr.ctypes.data_as(typ)


def source_id() -> str:
    """sha1 prefix over the sources libspecimux_b200.so is built from (csrc/*.cu|cuh|hpp, the Makefile, include/*.h): the
    identity a committed ncu capture is stamped with, so that bench.py quotes its figures only for the same code --
    independent of where and when the library was compiled."""
    import glob
    import hashlib
    here = os.path.dirname(os.path.abspath(__file__))
    files = sorted(glob.glob(os.path.join(here, "csrc", "*.cu")) + glob.glob(os.path.join(here, "csrc", "*.cuh")) +
                   glob.glob(os.path.join(here, "csrc", "*.hpp")) + [os.path.join(here, "csrc", "Makefile")] +
                   glob.glob(os.path.join(here, "..", "include", "*.h")))
    h = hashlib.sha1()
    for f in files:
        h.update(os.path.basename(f).encode())
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


class HostBuffer:
    """numpy view over pinned host memory (cudaHostAlloc through the library); falls back to ordinary
    pageable memory when no GPU driver is present (packing still works on a CPU-only box).

    The pinned block belongs to the views: it is released (cudaFreeHost) when the last numpy array that looks
    into it has gone, not when this object is dropped or `free()`d -- a result handed to another thread stays
    valid after the pool that produced it has grown a new buffer."""

    def __init__(self, count, dtype):
        import weakref
        dtype = np.dtype(dtype)
        self.nbytes = max(1, int(count) * dtype.itemsize)
        self.pinned = False
        try:
            lib = load()
            p = lib.smx_host_alloc(self.nbytes)
        except Exception:
            p = None
        if p:
            self.pinned = True
            raw = (C.c_char * self.nbytes).from_address(p)
            weakref.finalize(raw, lib.smx_host_free, p)
            self.array = np.frombuffer(raw, dtype=dtype, count=int(count))
        else:
            self.array = np.empty(int(count), dtype=dtype)

    def free(self):
        """Drops this object's own view (the memory goes when every other view has gone too)."""
        self.array = None


def bind_thread_to_gpu_numa_node(device: int):
    """Restricts the calling thread to the CPUs of the NUMA node `device` is attached to, so that the
    pinned buffers it allocates next (first touch) and its copies stay local to the GPU's PCIe root.
    Returns (node, n_cpus) or None when the topology is unknown (single node, containers, no sysfs)."""
    try:
        buf = C.create_string_buffer(32)
        if load().smx_device_pci_bus_id(device, buf, 32) != SMX_OK:
            return None
        bus = buf.value.decode().lower()
        with open("/sys/bus/pci/devices/%s/numa_node" % bus) as fh:
            node = int(fh.read().strip())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as fh:
            spec = fh.read().strip()
        cpus = set()
        for part in spec.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node, len(cpus)
    except (OSError, ValueError, AttributeError):
        return None
