"""specimine on the GPU: recover partial-barcode reads of a specimen by aligning the specimen's full-match reads
into them (reference: src/specimux/specimine.py).

The reference loops `edlib.align(full_seq, partial_seq, mode="HW", task="path", k=int(len(full) * (1 - min_identity)))`
over every (partial, full) pair and reads only `editDistance` from the result (specimine.py:226-248).  Here the whole
|full| x |partial| distance matrix comes from one call of the C ABI (smx_hw_distances: warp-cooperative multi-word
Myers, hand-written CUDA); file discovery, the identity rule (first full read with the strictly highest identity
>= --min-identity wins) and the output naming follow the reference.  No CPU path: without a GPU the call raises.

`--fastq` takes several files to mine a whole demultiplexed tree in one process (mine_files): every distinct partial
file is parsed once, every (specimen file, forward / reverse) pair becomes one group, and the groups go to the GPU in
few smx_hw_best_grouped calls, which keep only the best full read of every partial read.  Each file gets the
`.mined` file a run on it alone writes.
"""
import argparse
import copy
import ctypes
import glob
import logging
import os
import re
import sys
from typing import Dict, List, Optional, Tuple

import numpy as np

from . import _lib
from . import seqio

# at most this many int32 distances per GPU call (the matrix is cut along the partial reads)
_MATRIX_BUDGET = 32 << 20
# at most about this many bytes of input (full reads, partial reads, 20 bytes per text-list entry) per grouped GPU call
_GROUP_BUDGET = 64 << 20


def parse_arguments(argv=None):
    ap = argparse.ArgumentParser(description="Mine additional candidate sequences from partial matches.")
    ap.add_argument("--index", required=True, help="Path to specimen index file (same as used with specimux)")
    ap.add_argument("--fastq", required=True, nargs="+",
                    help="Path to full match FASTQ file for a specimen; several files are mined in one run, each "
                         "writing its own <file>.mined")
    ap.add_argument("--partial-forward", action="store_true", default=False,
                    help="Include forward partial matches (default: False)")
    ap.add_argument("--no-partial-reverse", action="store_true", default=False,
                    help="Exclude reverse partial matches (included by default)")
    ap.add_argument("--min-identity", type=float, default=0.85, help="Minimum alignment identity for a match (default: 0.85)")
    ap.add_argument("--debug", action="store_true", help="Enable debug logging")
    return ap.parse_args(argv)


def extract_specimen_id(fastq_path: str) -> str:
    """specimine.py:54-62: the file name minus `.fastq` (and minus the legacy `sample_` prefix)."""
    name = os.path.basename(fastq_path)
    m = re.match(r"(?:sample_)?(.+)\.fastq", name)
    if not m:
        raise ValueError(f"Could not extract specimen ID from filename: {name}")
    return m.group(1)


def find_barcodes(specimen_id: str, index_file: str) -> Tuple[Optional[str], Optional[str]]:
    """specimine.py:65-83: (FwIndex, RvIndex) of the specimen's row, upper-cased."""
    with open(index_file, "r") as fh:
        header = next(fh).strip().split("\t")
        col = lambda name, default: header.index(name) if name in header else default
        i_id, i_fw, i_rv = col("SampleID", 0), col("FwIndex", 2), col("RvIndex", 4)
        for line in fh:
            fields = line.strip().split("\t")
            if len(fields) > max(i_id, i_fw, i_rv) and fields[i_id] == specimen_id:
                return fields[i_fw].upper(), fields[i_rv].upper()
    logging.error(f"Could not find specimen {specimen_id} in index file")
    return None, None


def detect_input_level(fastq_path: str) -> Tuple[str, str, Optional[str]]:
    """specimine.py:86-117: (output root, pool, primer pair or None) from .../full/<pool>[/<pair>]/<specimen>.fastq."""
    parts = os.path.abspath(fastq_path).split(os.sep)
    if "full" not in parts:
        raise ValueError(f"Could not find 'full' directory in path: {fastq_path}")
    at = parts.index("full")
    below = parts[at + 1:-1]
    if len(below) not in (1, 2):
        raise ValueError(f"Unexpected path structure: {fastq_path}")
    return os.sep.join(parts[:at]), below[0], (below[1] if len(below) == 2 else None)


def _partials_in(directory: str, fwd_barcode: str, rev_barcode: str, found: Dict[str, List[str]], exists=None,
                 isdir=None) -> None:
    """specimine.py:120-150: barcode_fwd_<b1>.fastq / barcode_rev_<b2>.fastq (or the legacy sample_ names)."""
    exists, isdir = exists or os.path.exists, isdir or os.path.isdir
    if not isdir(directory):
        return
    for kind, tag, barcode in (("forward", "fwd", fwd_barcode), ("reverse", "rev", rev_barcode)):
        if not barcode:
            continue
        for name in (f"barcode_{tag}_{barcode}.fastq", f"sample_barcode_{tag}_{barcode}.fastq"):
            path = os.path.join(directory, name)
            if exists(path):
                found[kind].append(path)
                break


def derive_partial_match_filenames(fastq_path: str, fwd_barcode: str, rev_barcode: str, exists=None, isdir=None,
                                   listdir=None) -> Dict[str, List[str]]:
    """specimine.py:153-194: the partial files next to a pool-level or primer-pair-level full-match file.  `exists`,
    `isdir` and `listdir` (a glob of one directory's entries) default to os.path.exists, os.path.isdir and glob.glob."""
    isdir, listdir = isdir or os.path.isdir, listdir or glob.glob
    found: Dict[str, List[str]] = {"forward": [], "reverse": []}
    root, pool, pair = detect_input_level(fastq_path)
    if pair is not None:
        _partials_in(os.path.join(root, "partial", pool, pair), fwd_barcode, rev_barcode, found, exists, isdir)
    else:
        pool_dir = os.path.join(root, "partial", pool)
        if isdir(pool_dir):
            for d in listdir(os.path.join(pool_dir, "*")):
                if isdir(d):
                    _partials_in(d, fwd_barcode, rev_barcode, found, exists, isdir)
    if fwd_barcode and not found["forward"]:
        logging.warning(f"No forward partial match files found for barcode: {fwd_barcode}")
    if rev_barcode and not found["reverse"]:
        logging.warning(f"No reverse partial match files found for barcode: {rev_barcode}")
    return {k: v for k, v in found.items() if v}


class VirtualTree:
    """A tree of relative file paths (an output tree held in memory, such as DeviceFiles.paths) seen through the file
    system calls discovery makes, rooted at '/': a path is looked up as '/<relative path>' and the partial files come
    back relative.  Directory listings are in sorted path order (on disk glob's order depends on the file system)."""

    def __init__(self, paths):
        self.files = set(paths)
        kids: Dict[str, set] = {}
        for p in self.files:
            parts = p.split("/")
            for i in range(1, len(parts)):
                kids.setdefault("/".join(parts[:i]), set()).add("/".join(parts[:i + 1]))
        self.children = {d: sorted(k) for d, k in kids.items()}

    def exists(self, path: str) -> bool:
        return path in self.files or path in self.children

    def isdir(self, path: str) -> bool:
        return path in self.children

    def listdir(self, pattern: str) -> List[str]:
        d = os.path.dirname(pattern)
        return [c for c in self.children.get(d, []) if not os.path.basename(c).startswith(".")]

def _blob(seqs: List[str]):
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    np.cumsum([len(s) for s in seqs], out=off[1:])
    return "".join(seqs).encode("latin-1", "replace"), off


def hw_distances(patterns: List[str], max_dist: List[int], texts: List[str], device: int = 0) -> np.ndarray:
    """[len(patterns), len(texts)] int32: HW edit distance of pattern i in text j, -1 when above max_dist[i].
    One smx_hw_distances call per slab of texts (GPU only)."""
    lib = _lib.load()
    out = np.empty((len(patterns), len(texts)), dtype=np.int32)
    if not patterns or not texts:
        return out
    pblob, poff = _blob(patterns)
    pk = np.asarray(max_dist, dtype=np.int32)
    per = max(1, _MATRIX_BUDGET // max(1, len(patterns)))
    for lo in range(0, len(texts), per):
        hi = min(len(texts), lo + per)
        tblob, toff = _blob(texts[lo:hi])
        slab = np.empty((len(patterns), hi - lo), dtype=np.int32)
        _lib.check(lib.smx_hw_distances(device, pblob, _lib.ptr(poff, _lib.u64p), _lib.ptr(pk, _lib.i32p), len(patterns),
                                        tblob, _lib.ptr(toff, _lib.u64p), hi - lo, _lib.ptr(slab, _lib.i32p)))
        out[:, lo:hi] = slab
    return out


def hw_best_grouped(patterns: List[str], max_dist: List[int], texts: List[str], grp_pat_off: np.ndarray,
                    grp_txt_off: np.ndarray, grp_txt_idx: np.ndarray, device: int = 0):
    """Best pattern of every text-list entry of every group (one smx_hw_best_grouped call, GPU only): group g owns
    patterns [grp_pat_off[g], grp_pat_off[g + 1]) and entries [grp_txt_off[g], grp_txt_off[g + 1]), entry e names
    texts[grp_txt_idx[e]].  Returns (best_pat, best_dist, device_ms): per entry the index within the group of the
    pattern with the smallest distance / length (ties to the first; distances above max_dist and empty patterns never
    win) and its distance, -1 / -1 when none qualifies."""
    lib = _lib.load()
    pblob, poff = _blob(patterns)
    tblob, toff = _blob(texts)
    pk = np.asarray(max_dist, dtype=np.int32)
    gp = np.ascontiguousarray(grp_pat_off, dtype=np.uint32)
    gt = np.ascontiguousarray(grp_txt_off, dtype=np.uint64)
    gi = np.ascontiguousarray(grp_txt_idx, dtype=np.uint32)
    best_pat = np.full(len(gi), -1, dtype=np.int32)
    best_dist = np.full(len(gi), -1, dtype=np.int32)
    ms = ctypes.c_float(0.0)
    _lib.check(lib.smx_hw_best_grouped(device, pblob, _lib.ptr(poff, _lib.u64p), _lib.ptr(pk, _lib.i32p), len(patterns),
                                       tblob, _lib.ptr(toff, _lib.u64p), len(texts), len(gp) - 1, _lib.ptr(gp, _lib.u32p),
                                       _lib.ptr(gt, _lib.u64p), _lib.ptr(gi, _lib.u32p), _lib.ptr(best_pat, _lib.i32p),
                                       _lib.ptr(best_dist, _lib.i32p), ctypes.byref(ms)))
    return best_pat, best_dist, float(ms.value)


def _max_dist(full_seqs: List[str], min_identity: float) -> List[int]:
    return [int(len(s) * (1 - min_identity)) for s in full_seqs]          # specimine.py:238


def _rewrite_mined(partial, best: np.ndarray, kind: str):
    """The partial records with a best identity (not -inf), as copies with the reference's id / description rewrite
    (specimine.py:246-262); copies, because a partial record may be mined for several specimens."""
    mined = []
    for rec, b in zip(partial, best):
        if b == -np.inf:
            continue
        b = float(b)
        out = copy.copy(rec)
        out.id = f"{rec.id}_mined_{kind}_{b:.2f}"
        out.description = f"{rec.description} mined_{kind} identity={b:.2f}"
        mined.append(out)
    return mined


def mine_sequences(full_match_file: str, partial_match_files: Dict[str, List[str]], min_identity: float, device: int = 0):
    """specimine.py:205-268.  Returns the mined partial records (id / description rewritten) in the reference's order."""
    full = list(seqio.parse(full_match_file, "fastq"))
    if not full:
        logging.error(f"No sequences found in full match file: {full_match_file}")
        return []
    logging.info(f"Loaded {len(full)} sequences from full match file")
    full_seqs = [str(r.seq) for r in full]
    full_len = np.array([len(s) for s in full_seqs], dtype=np.float64)
    max_dist = _max_dist(full_seqs, min_identity)
    mined = []
    for kind, files in partial_match_files.items():
        logging.info(f"Processing {kind} partial matches from {len(files)} file(s)")
        partial = []
        for path in files:
            logging.debug(f"  Loading: {path}")
            partial.extend(seqio.parse(path, "fastq"))
        logging.info(f"Found {len(partial)} sequences across all {kind} partial match files")
        dist = hw_distances(full_seqs, max_dist, [str(r.seq) for r in partial], device)
        # identity = 1 - d / len(full) where the alignment exists (specimine.py:197-202, :243-244); the first full read
        # with the strictly highest identity >= min_identity (and > 0, the initial best) wins (:246-248)
        with np.errstate(divide="ignore", invalid="ignore"):
            ident = 1 - (dist / full_len[:, None])
        ok = (dist != -1) & (ident >= min_identity) & (ident > 0)
        ident = np.where(ok, ident, -np.inf)
        hits = _rewrite_mined(partial, ident.max(axis=0), kind)
        mined.extend(hits)
        logging.info(f"Matched {len(hits)}/{len(partial)} sequences from {kind} partial matches")
    return mined


def _select_partials(fastq: str, index: str, partial_forward: bool, no_partial_reverse: bool, exists=None, isdir=None,
                     listdir=None) -> Tuple[Optional[Dict[str, List[str]]], str]:
    """main()'s discovery for one file: (the selected partial files by kind, "") or, where a run on this file alone
    would stop, (None, the message it logs).  exists / isdir / listdir as for derive_partial_match_filenames."""
    specimen = extract_specimen_id(fastq)
    logging.info(f"Processing specimen: {specimen}")
    fwd, rev = find_barcodes(specimen, index)
    if not (fwd and rev):
        return None, f"Could not find specimen {specimen} in index file"
    logging.info(f"Found barcodes - Forward: {fwd}, Reverse: {rev}")
    files = derive_partial_match_filenames(fastq, fwd, rev, exists, isdir, listdir)
    for kind, paths in files.items():
        logging.info(f"Found {len(paths)} {kind} partial match file(s)")
        for p in paths:
            logging.debug(f"  - {p}")
    if not partial_forward:
        files.pop("forward", None)
    if no_partial_reverse:
        files.pop("reverse", None)
    if not files:
        logging.error("No partial match files found or selected")
        return None, "No partial match files found or selected"
    return files, ""


def select_in_tree(paths: List[str], index: str, partial_forward: bool = False, no_partial_reverse: bool = False):
    """Discovery over a tree held as relative paths (VirtualTree) for its pool-level full files, full/<pool>/<name>.fastq:
    returns ([(full path, {kind: [partial paths]})] in the order given, [(full path, reason)] for the files a run on
    them alone would stop on, with the message it logs).  Partial paths are relative, as in `paths`."""
    tree = VirtualTree(paths)
    jobs, skipped = [], []
    for p in paths:
        parts = p.split("/")
        if len(parts) != 3 or parts[0] != "full" or not p.endswith(".fastq"):
            continue
        try:
            files, reason = _select_partials("/" + p, index, partial_forward, no_partial_reverse, tree.exists, tree.isdir,
                                             tree.listdir)
        except ValueError as e:
            logging.error(str(e))
            files, reason = None, str(e)
        if files is None:
            logging.error(f"Skipping {p}")
            skipped.append((p, reason))
        else:
            jobs.append((p, files))
    return jobs, skipped


def mine_files(fastqs: List[str], index: str, partial_forward: bool = False, no_partial_reverse: bool = False,
               min_identity: float = 0.85, device: int = 0) -> int:
    """Mines every file of `fastqs` and writes <file>.mined for each, with the bytes a run on that file alone writes.
    Every distinct partial file is parsed once; each (file, kind) is one group of hw_best_grouped, and groups go to
    the GPU in calls of about _GROUP_BUDGET bytes.  A file a single run would stop on is logged with the same message
    and skipped.  Returns the number of skipped files."""
    jobs, failed = [], 0
    for fastq in fastqs:
        try:
            files, _reason = _select_partials(fastq, index, partial_forward, no_partial_reverse)
        except ValueError as e:
            logging.error(str(e))
            files = None
        if files is None:
            logging.error(f"Skipping {fastq}")
            failed += 1
            continue
        full = [str(r.seq) for r in seqio.parse(fastq, "fastq")]
        if not full:
            logging.error(f"No sequences found in full match file: {fastq}")
        jobs.append((fastq, files, full))

    partial_cache: Dict[str, list] = {}
    partial_bytes: Dict[str, int] = {}

    def records(path):
        if path not in partial_cache:
            logging.debug(f"  Loading: {path}")
            partial_cache[path] = list(seqio.parse(path, "fastq"))
            partial_bytes[path] = sum(len(r.seq) for r in partial_cache[path])
        return partial_cache[path]

    groups = [(j, kind, paths) for j, (_, files, full) in enumerate(jobs) if full for kind, paths in files.items()]
    mined: Dict[Tuple[int, str], list] = {}
    total_ms, lo = 0.0, 0
    while lo < len(groups):
        # one call: groups in order while the call's input stays within the budget (at least one group)
        seen, cost, hi = set(), 0, lo
        while hi < len(groups):
            j, _, paths = groups[hi]
            add = sum(len(s) for s in jobs[j][2])
            for p in paths:
                recs = records(p)
                add += 20 * len(recs) + (0 if p in seen else partial_bytes[p])
            if hi > lo and cost + add > _GROUP_BUDGET:
                break
            seen.update(paths)
            cost += add
            hi += 1
        texts, base = [], {}
        patterns, max_dist, gp, gt, gi = [], [], [0], [0], []
        for j, kind, paths in groups[lo:hi]:
            full = jobs[j][2]
            patterns.extend(full)
            max_dist.extend(_max_dist(full, min_identity))
            gp.append(len(patterns))
            for p in paths:
                if p not in base:
                    base[p] = len(texts)
                    texts.extend(str(r.seq) for r in records(p))
                gi.extend(range(base[p], base[p] + len(records(p))))
            gt.append(len(gi))
        best_pat, best_dist, ms = hw_best_grouped(patterns, max_dist, texts, np.array(gp, dtype=np.uint32),
                                                  np.array(gt, dtype=np.uint64), np.array(gi, dtype=np.uint32), device)
        total_ms += ms
        for g, (j, kind, paths) in enumerate(groups[lo:hi]):
            full_len = np.array([len(s) for s in jobs[j][2]], dtype=np.float64)
            partial = [r for p in paths for r in records(p)]
            i, d = best_pat[gt[g]:gt[g + 1]], best_dist[gt[g]:gt[g + 1]]
            # the winner's identity, as mine_sequences computes it; when it fails the tests every other candidate does
            ident = 1 - (d / full_len[np.maximum(i, 0)])
            best = np.where((i >= 0) & (ident >= min_identity) & (ident > 0), ident, -np.inf)
            mined[(j, kind)] = _rewrite_mined(partial, best, kind)
            logging.info(f"{jobs[j][0]}: matched {len(mined[(j, kind)])}/{len(partial)} sequences from {kind} partial matches")
        lo = hi
    logging.info(f"Grouped search: {len(groups)} group(s), {len(partial_cache)} partial file(s), {total_ms:.1f} ms on the device")
    for j, (fastq, files, _) in enumerate(jobs):
        out_recs = [r for kind in files for r in mined.get((j, kind), [])]
        out = f"{fastq}.mined"
        write_fastq(out_recs, out)
        logging.info(f"Wrote {len(out_recs)} sequences to {out}")
    return failed


def fastq_title(rec) -> str:
    """Title line Biopython's FASTQ writer gives a record (Bio.SeqIO.QualityIO.FastqPhredWriter.write_record): the
    description when it already starts with the id, else "<id> <description>"; newlines become spaces."""
    clean = lambda s: s.replace("\n", " ").replace("\r", " ")
    ident = clean(rec.id) if rec.id else ""
    desc = clean(rec.description or "")
    if desc and desc.split(None, 1)[0] == ident:
        return desc
    return f"{ident} {desc}" if desc else ident


def write_fastq(records, path: str) -> int:
    with open(path, "w") as fh:
        for rec in records:
            qtext = rec.qual if getattr(rec, "qual", None) is not None else "".join(
                chr(q + 33) for q in rec.letter_annotations["phred_quality"])
            fh.write("@%s\n%s\n+\n%s\n" % (fastq_title(rec), str(rec.seq), qtext))
    return len(records)


def main(argv=None):
    args = parse_arguments(argv)
    logging.basicConfig(level=logging.DEBUG if args.debug else logging.INFO, format="%(asctime)s - %(levelname)s - %(message)s")
    if len(args.fastq) > 1:
        if mine_files(args.fastq, args.index, args.partial_forward, args.no_partial_reverse, args.min_identity):
            sys.exit(1)
        return
    fastq = args.fastq[0]
    specimen = extract_specimen_id(fastq)
    logging.info(f"Processing specimen: {specimen}")
    fwd, rev = find_barcodes(specimen, args.index)
    if not (fwd and rev):
        sys.exit(1)
    logging.info(f"Found barcodes - Forward: {fwd}, Reverse: {rev}")
    files = derive_partial_match_filenames(fastq, fwd, rev)
    for kind, paths in files.items():
        logging.info(f"Found {len(paths)} {kind} partial match file(s)")
        for p in paths:
            logging.debug(f"  - {p}")
    if not args.partial_forward:
        files.pop("forward", None)
    if args.no_partial_reverse:
        files.pop("reverse", None)
    if not files:
        logging.error("No partial match files found or selected")
        sys.exit(1)
    mined = mine_sequences(fastq, files, args.min_identity)
    logging.info(f"Found {len(mined)} mined sequences")
    out = f"{fastq}.mined"
    write_fastq(mined, out)
    logging.info(f"Wrote {len(mined)} sequences to {out}")


if __name__ == "__main__":
    main()
