#!/usr/bin/env python3
"""Probe of specimine in GPU memory: seeded reads of synth.mining_reads (one amplicon per specimen, full reads with both
barcodes, partial reads with one barcode destroyed, unrelated reads with one barcode) held as CUDA tensors, demultiplexed
and mined two ways, alternating after warm-up:
  (a) Matcher.demux_files_device, then Matcher.mine_device: host clock around both, with the CUDA-event times of the
      search kernels and of the mine_device call;
  (b) Matcher.demux_files_device, then DeviceFiles.write into a fresh tmpfs directory (/dev/shm), then an in-process
      specimine.mine_files over the tree's pool-level full files.
The `.mined` files of (a) and (b) must be identical, file by file.  In a separate pass torch.profiler gives the k_hw_best
kernel time of one call of each route (mean of --reps calls after a warm-up); both search the same pairs.  Shapes: the
config-2 plate, 8 x 96 specimens, with (full, partial, unrelated) reads of (16, 4, 32) as BASELINE.md section 5, and a
larger one.  Prints the card name and power limit read in the same run and one JSON object; --out writes it too.

    python tools/device_mine_probe.py --steps 5 --out profiles/r7_device_mine_probe.json
"""
import argparse
import glob
import json
import logging
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
from mine_probe import _kernel_ms  # noqa: E402

SHAPES = {"section5": dict(n_fwd=8, n_rev=96, n_full=16, n_partial=4, n_other=32),
          "large": dict(n_fwd=8, n_rev=96, n_full=64, n_partial=16, n_other=128)}


def mined_files(root):
    out = {}
    for p in glob.glob(os.path.join(root, "**", "*.mined"), recursive=True):
        with open(p, "rb") as fh:
            out[os.path.relpath(p, root)] = fh.read()
    return out


def run_shape(name, shape, a, m_cls, work):
    import torch
    from specimux_b200 import specimine, synth
    from specimux_b200.models import MatchParameters
    from specimux_b200.tables import MatchTables
    import helpers as H

    t0 = time.perf_counter()
    ds = synth.mining_reads(seed=a.seed, **shape)
    gen_s = time.perf_counter() - t0
    specimens = H.build_specimens(ds.primers, ds.specimens)
    mt = MatchTables(specimens, MatchParameters({synth.ITS1F: 5, synth.ITS4: 5}, 2, ds.search_len, True))
    index = os.path.join(work, name + "_index.txt")
    with open(index, "w") as fh:
        fh.write("SampleID\tPrimerPool\tFwIndex\tFwPrimer\tRvIndex\tRvPrimer\n")
        for row in ds.specimens:
            fh.write("\t".join(row) + "\n")
    dev = torch.device("cuda", a.device)
    codes = np.frombuffer(b"ACGT", dtype=np.uint8)[ds.codes].copy()
    titles = [b"read_%d runid=probe ch=%d" % (i, i % 512) for i in range(ds.n_reads)]
    t_off = np.concatenate([[0], np.cumsum([len(t) for t in titles])]).astype(np.int64)
    bases = torch.tensor(codes, device=dev)
    quals = torch.tensor((ds.quals + 33).astype(np.uint8), device=dev)
    offsets = torch.tensor(ds.offsets.astype(np.int64), device=dev)
    tt = torch.tensor(np.frombuffer(b"".join(titles), dtype=np.uint8).copy(), device=dev)
    to = torch.tensor(t_off, device=dev)
    tree_b, out_a = os.path.join(work, name + "_b"), os.path.join(work, name + "_a")
    m = m_cls(mt, a.device)

    def route_a():
        t = time.perf_counter()
        files = m.demux_files_device(bases, offsets, tt, to, quals)
        mined = m.mine_device(files, index)
        torch.cuda.synchronize()
        return time.perf_counter() - t, (files, mined)

    def route_b():
        shutil.rmtree(tree_b, ignore_errors=True)
        t = time.perf_counter()
        files = m.demux_files_device(bases, offsets, tt, to, quals)
        files.write(tree_b)
        pool = [os.path.join(tree_b, p) for p, k in zip(files.paths, files.file_key) if int(k) >> 62 == 3]
        specimine.mine_files(pool, index)
        return time.perf_counter() - t, (files, pool)

    for _ in range(a.warmup):
        route_a()
        route_b()
    ta, tb, dev_ms = [], [], []
    for _ in range(a.steps):
        t, (files, mined) = route_a()
        ta.append(t)
        dev_ms.append(mined.device_ms)
        t, _r = route_b()
        tb.append(t)
    shutil.rmtree(out_a, ignore_errors=True)
    mined.write(out_a)
    got, want = mined_files(out_a), mined_files(tree_b)
    identical = got == want
    n_pool = sum(1 for k in files.file_key if int(k) >> 62 == 3)

    # kernel time of one call of each route's search, in a pass of its own
    files = m.demux_files_device(bases, offsets, tt, to, quals)
    ka = _kernel_ms(lambda: m.mine_device(files, index), ["k_hw_best"], a.reps)
    pool = [os.path.join(tree_b, p) for p, k in zip(files.paths, files.file_key) if int(k) >> 62 == 3]
    kb = _kernel_ms(lambda: specimine.mine_files(pool, index), ["k_hw_best"], a.reps)
    m.close()
    med = lambda x: float(np.median(x)) * 1e3
    return {"shape": shape, "reads": int(ds.n_reads), "bases": int(ds.offsets[-1]), "generate_s": round(gen_s, 1),
            "pool_level_files": n_pool, "mined_files": len(got), "mined_records": int(mined.partial.numel()),
            "mined_bytes": int(mined.data.numel()), "skipped": len(mined.skipped),
            "a_demux_files_plus_mine_device_ms": {"median": med(ta), "all": [round(x * 1e3, 2) for x in ta]},
            "a_mine_device_event_ms": {"search_kernels": float(np.median([d[0] for d in dev_ms])),
                                       "whole_call": float(np.median([d[1] for d in dev_ms]))},
            "b_demux_files_write_mine_files_ms": {"median": med(tb), "all": [round(x * 1e3, 2) for x in tb]},
            "speedup_b_over_a": round(med(tb) / med(ta), 2),
            "k_hw_best_kernel_ms": {"a_mine_device": round(ka, 3), "b_mine_files": round(kb, 3)},
            "mined_identical": identical}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=5, help="timed calls of each route (alternating)")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--reps", type=int, default=3, help="profiled calls of each route's search")
    ap.add_argument("--shapes", default="section5,large")
    ap.add_argument("--seed", type=int, default=41)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--tmpfs", default="/dev/shm")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    logging.basicConfig(level=logging.WARNING)
    logging.getLogger().setLevel(logging.CRITICAL)               # specimine logs per file; not part of the timing
    from specimux_b200.engine import Matcher
    card = _card(a.device)
    print(card)
    work = tempfile.mkdtemp(prefix="mine_probe_", dir=a.tmpfs if os.path.isdir(a.tmpfs) else None)
    res = {"card": card, "shapes": {}}
    try:
        for name in a.shapes.split(","):
            res["shapes"][name] = run_shape(name, SHAPES[name], a, Matcher, work)
            print(name, json.dumps(res["shapes"][name]))
    finally:
        shutil.rmtree(work, ignore_errors=True)
    ok = all(s["mined_identical"] for s in res["shapes"].values())
    res["all_mined_identical"] = ok
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
