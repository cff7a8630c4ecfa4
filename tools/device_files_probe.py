#!/usr/bin/env python3
"""Probe of the complete output files in GPU memory: config 2 (synth.ont037, 765k reads, with qualities and titles; 1 in
2000 bases replaced by IUPAC / lower-case / U letters) held as CUDA tensors, formatted three ways, alternating after
warm-up:
  (a) Matcher.demux_files_device: host clock around the call, plus the CUDA-event times of the copy kernels and of the
      call;
  (b) Matcher.demux_files_device, then DeviceFiles.write into a fresh directory on tmpfs (/dev/shm);
  (c) Matcher.match_device, then records, bases, qualities and titles copied to pinned host memory, then the native
      writer (native_io.TreeWriter) writing the tree of the same reads (a reader block) into a fresh tmpfs directory.
The trees of (b) and (c) must be identical, file by file.  The copy kernels' bytes moved (every output byte written
once and read once -- sequence and quality bytes from the reads, header bytes from the titles and name tables) over
their CUDA-event time is set against 7.7 TB/s.  Prints the card name and power limit read in the same run and one JSON
object; --out writes it to a file too.

    python tools/device_files_probe.py --steps 5 --out profiles/device_files_probe.json
"""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from device_input_probe import _card  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def same_trees(a, b):
    """True when the two directories hold the same relative paths with the same bytes."""
    def files(root):
        out = {}
        for d, _s, fs in os.walk(root):
            for f in fs:
                p = os.path.join(d, f)
                out[os.path.relpath(p, root)] = p
        return out
    fa, fb = files(a), files(b)
    if fa.keys() != fb.keys():
        return False
    for k in fa:
        with open(fa[k], "rb") as x, open(fb[k], "rb") as y:
            if x.read() != y.read():
                return False
    return True


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reads", type=int, default=765_000)
    ap.add_argument("--steps", type=int, default=5, help="timed calls of each route (alternating)")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--tmpfs", default="/dev/shm")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    from specimux_b200 import native_io, synth
    from specimux_b200.engine import Matcher
    from specimux_b200.models import MatchParameters
    from specimux_b200.orchestration import thresholds_for
    from specimux_b200.tables import MatchTables
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers as H

    ds = synth.ont037(n_reads=a.reads, with_quals=True)
    specimens = H.build_specimens(ds.primers, ds.specimens)
    k_idx, k_primers = thresholds_for(specimens)
    mt = MatchTables(specimens, MatchParameters(k_primers, k_idx, ds.search_len, True))
    codes = np.frombuffer(b"ACGT", dtype=np.uint8)[ds.codes].copy()
    rng = np.random.default_rng(2024)
    hits = rng.choice(codes.shape[0], size=codes.shape[0] // 2000, replace=False)
    codes[hits] = np.frombuffer(b"NRYnacgtUuKM", dtype=np.uint8)[rng.integers(0, 12, size=hits.shape[0])]
    qtext = (ds.quals + 33).astype(np.uint8)
    card = _card(a.device)

    # the reads go through the native reader once: its block feeds route (c) and gives the titles of (a) and (b)
    work = tempfile.mkdtemp(prefix="files_probe_", dir=a.tmpfs)
    fq = os.path.join(work, "reads.fastq")
    with open(fq, "wb") as fh:
        off = ds.offsets
        for i in range(ds.n_reads):
            fh.write(b"@read_%d runid=probe ch=%d\n%s\n+\n%s\n" % (i, i % 512, codes[off[i]:off[i + 1]].tobytes(),
                                                                  qtext[off[i]:off[i + 1]].tobytes()))
    rd = native_io.FastxReader(fq, True)
    blk = rd.next_block(ds.n_reads + 1)
    os.remove(fq)
    assert blk.n_reads == ds.n_reads
    import ctypes as C
    v = blk._view
    t_off = np.ctypeslib.as_array(v.title_off, shape=(ds.n_reads + 1,)).astype(np.int64)
    titles_h = np.frombuffer(C.string_at(v.titles, int(t_off[-1])), dtype=np.uint8).copy()

    dev = torch.device("cuda", a.device)
    bases, quals = torch.tensor(codes, device=dev), torch.tensor(qtext, device=dev)
    offsets = torch.tensor(ds.offsets.astype(np.int64), device=dev)
    titles, title_offsets = torch.tensor(titles_h, device=dev), torch.tensor(t_off, device=dev)
    h_bases = torch.empty(bases.shape, dtype=torch.uint8, pin_memory=True)
    h_quals = torch.empty(quals.shape, dtype=torch.uint8, pin_memory=True)
    h_titles = torch.empty(titles.shape, dtype=torch.uint8, pin_memory=True)
    tree_b, tree_c = os.path.join(work, "b"), os.path.join(work, "c")

    def route_a():
        t = time.perf_counter()
        r = m.demux_files_device(bases, offsets, titles, title_offsets, quals)
        return time.perf_counter() - t, r

    def route_b():
        shutil.rmtree(tree_b, ignore_errors=True)
        t = time.perf_counter()
        r = m.demux_files_device(bases, offsets, titles, title_offsets, quals)
        r.write(tree_b)
        return time.perf_counter() - t, r

    def route_c():
        shutil.rmtree(tree_c, ignore_errors=True)
        t = time.perf_counter()
        res = m.match_device(bases, offsets)
        h_bases.copy_(bases)
        h_quals.copy_(quals)
        h_titles.copy_(titles)
        recs = res.to_host().records
        with native_io.TreeWriter(tree_c, "", True, mt) as wr:
            wr.write(blk, recs)
        return time.perf_counter() - t, len(recs)

    sa, sb, sc, dms = [], [], [], []
    with Matcher(mt, device=a.device) as m:
        for _ in range(a.warmup):
            route_a(); route_b(); route_c()
        for _ in range(a.steps):
            s, got = route_a()
            sa.append(s)
            dms.append(got.device_ms)
            s, _files = route_b()
            sb.append(s)
            s, n_rec = route_c()
            sc.append(s)
        identical = same_trees(tree_b, tree_c)
    assert identical, "routes (b) and (c) built different trees"
    total = int(got.data.numel())
    n_files = len(got.paths)
    n_pool = sum(1 for p in got.paths if p.startswith("full/") and p.count("/") == 2)
    med = lambda v: float(np.median(v)) * 1e3
    copy_ms = float(np.median([x[0] for x in dms]))
    moved = 2 * total
    out = dict(card, config="ont037", reads=int(ds.n_reads), bases=int(codes.shape[0]), substituted_bases=int(hits.shape[0]),
               title_bytes=int(titles_h.shape[0]), records=int(n_rec), outputs=int(got.record.numel()), files=n_files,
               pool_level_files=n_pool, output_bytes=total, steps=a.steps, warmup=a.warmup, identical_b_c=identical,
               demux_files_device_ms=dict(host_clock_median=med(sa), host_clock_min=float(min(sa)) * 1e3,
                                          copy_kernels_median=copy_ms, device_call_median=float(np.median([x[1] for x in dms]))),
               device_files_and_write_ms=dict(host_clock_median=med(sb), host_clock_min=float(min(sb)) * 1e3),
               host_writer_route_ms=dict(host_clock_median=med(sc), host_clock_min=float(min(sc)) * 1e3),
               copy_kernels=dict(bytes_moved=moved, bytes_per_s=moved / (copy_ms * 1e-3),
                                 share_of_7_7_TBps=moved / (copy_ms * 1e-3) / HBM_BYTES_PER_S),
               per_step=dict(demux_files_device_s=sa, demux_files_device_device_ms=dms, device_files_and_write_s=sb,
                             host_writer_route_s=sc))
    rd.close()
    shutil.rmtree(work, ignore_errors=True)
    print("%s, power limit %s" % (card["gpu"], card.get("power_limit")))
    print(json.dumps(out))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
