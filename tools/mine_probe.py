#!/usr/bin/env python3
"""Probe of tree-wide specimine: a seeded synthetic demultiplexed tree of config-2 shape (8 x 96 specimens under
full/ITS/, partial files under partial/ITS/ITS1F-ITS4/, ~700-nt amplicons with 7 % errors per read), mined three ways:
  (a) one `specimine` process per file, as users ran it before --fastq took several files,
  (b) one multi-file `specimine` process over the same N files,
  (c) one multi-file `specimine` process over the whole tree.
Every `.mined` file of the N files must be byte-identical across the three routes.  Then, in this process and on the
pairs of the whole tree, the kernel time of the grouped search (k_hw_best, smx_hw_best_grouped) against the all-pairs
matrix of smx_hw_distances (k_hw_distance, one call per group as a single-file run makes), from torch.profiler, as
DP cells (sum of m * n over (full, partial) pairs) per second.  Prints the card name and power limit and one JSON
object; --out writes it to a file too.

    python tools/mine_probe.py --files 16 --out profiles/mine_probe.json
"""
import argparse
import filecmp
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, ROOT)


def _specimine(index, files, workdir):
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    t = time.perf_counter()
    subprocess.run([sys.executable, "-m", "specimux_b200.specimine", "--index", index, "--fastq"] + files,
                   check=True, cwd=workdir, env=env, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    return time.perf_counter() - t


def _collect(files, dest):
    os.makedirs(dest, exist_ok=True)
    for i, f in enumerate(files):
        shutil.move(f + ".mined", os.path.join(dest, "%04d.mined" % i))


def _groups(paths, index):
    """(full reads, partial reads) of every (file, kind) group of a default-flag run (reverse partials only)."""
    from specimux_b200 import seqio, specimine
    out = []
    for p in paths:
        files, _reason = specimine._select_partials(p, index, False, False)
        full = [str(r.seq) for r in seqio.parse(p, "fastq")]
        for kind, fs in files.items():
            out.append((full, [str(r.seq) for f in fs for r in seqio.parse(f, "fastq")]))
    return out


def _kernel_ms(fn, names, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()                                                          # warm-up: module load, every class launched once
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if any(n in e.key for n in names))
    return us / 1e3 / reps


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--files", type=int, default=16, help="N: files of routes (a) and (b)")
    ap.add_argument("--n-fwd", type=int, default=8)
    ap.add_argument("--n-rev", type=int, default=96)
    ap.add_argument("--full-reads", type=int, default=16, help="reads per full-match file")
    ap.add_argument("--partial-reads", type=int, default=4, help="reads per specimen in each partial file")
    ap.add_argument("--other-reads", type=int, default=32, help="unrelated reads in each partial file")
    ap.add_argument("--amplicon", type=int, default=700)
    ap.add_argument("--reps", type=int, default=3, help="profiled repetitions of each kernel comparison")
    ap.add_argument("--seed", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from specimux_b200 import specimine, synth
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    torch.cuda.init()
    res = {"gpu": gpu[0] if gpu else "unknown", "files": args.files, "specimens": args.n_fwd * args.n_rev,
           "full_reads": args.full_reads, "partial_reads_per_specimen": args.partial_reads, "other_reads": args.other_reads,
           "amplicon": args.amplicon, "seed": args.seed}
    print("GPU (name, power limit):", res["gpu"])
    tmp = tempfile.mkdtemp(prefix="mine_probe_")
    try:
        tree = os.path.join(tmp, "tree")
        os.makedirs(tree)
        paths = synth.specimine_tree(tree, args.n_fwd, args.n_rev, args.full_reads, args.partial_reads, args.other_reads,
                                     args.amplicon, seed=args.seed)
        index = os.path.join(tree, "index.txt")
        # spread the N files over the plate: specimens of different reverse barcodes share no partial file
        step = max(1, len(paths) // args.files)
        sample = paths[::step][:args.files]
        ta = sum(_specimine(index, [p], tmp) for p in sample)
        _collect(sample, os.path.join(tmp, "a"))
        tb = _specimine(index, sample, tmp)
        _collect(sample, os.path.join(tmp, "b"))
        tc = _specimine(index, paths, tmp)
        n_hits = 0
        for i, p in enumerate(sample):
            fa, fb = os.path.join(tmp, "a", "%04d.mined" % i), os.path.join(tmp, "b", "%04d.mined" % i)
            if not (filecmp.cmp(fa, fb, shallow=False) and filecmp.cmp(fa, p + ".mined", shallow=False)):
                raise SystemExit("route outputs differ for %s" % p)
            with open(fa) as fh:
                n_hits += sum(1 for _ in fh) // 4
        res.update({"identical_mined_files": len(sample), "mined_reads_in_sample": n_hits,
                    "route_a_s": ta, "route_b_s": tb, "route_c_s": tc,
                    "route_a_s_per_specimen": ta / len(sample), "route_b_s_per_specimen": tb / len(sample),
                    "route_c_s_per_specimen": tc / len(paths)})

        groups = _groups(paths, index)
        pairs = sum(len(f) * len(t) for f, t in groups)
        cells = sum(sum(len(a) for a in f) * sum(len(b) for b in t) for f, t in groups)
        patterns, ks, texts, gp, gt, gi = [], [], [], [0], [0], []
        for f, t in groups:
            patterns += f
            ks += [int(len(s) * 0.15) for s in f]
            gp.append(len(patterns))
            gi += range(len(texts), len(texts) + len(t))
            texts += t
            gt.append(len(gi))
        gp, gt, gi = np.array(gp, dtype=np.uint32), np.array(gt, dtype=np.uint64), np.array(gi, dtype=np.uint32)
        dev = []

        def grouped():
            dev.append(specimine.hw_best_grouped(patterns, ks, texts, gp, gt, gi)[2])

        def matrix():
            for f, t in groups:
                specimine.hw_distances(f, [int(len(s) * 0.15) for s in f], t)
        ms_g = _kernel_ms(grouped, ["k_hw_best"], args.reps)
        ms_m = _kernel_ms(matrix, ["k_hw_distance"], args.reps)
        # same winners as the host argmin over the matrix (one pass, outside the timing)
        bp, bd, _ = specimine.hw_best_grouped(patterns, ks, texts, gp, gt, gi)
        for g, (f, t) in enumerate(groups):
            d = specimine.hw_distances(f, [int(len(s) * 0.15) for s in f], t).astype(np.float64)
            m = np.array([len(s) for s in f], dtype=np.float64)[:, None]
            r = np.where(d >= 0, d / m, np.inf)
            want = np.where(np.isfinite(r.min(axis=0)), r.argmin(axis=0), -1)
            if not (bp[gt[g]:gt[g + 1]] == want).all():
                raise SystemExit("grouped winners differ from the matrix argmin in group %d" % g)
        res.update({"groups": len(groups), "pairs": pairs, "dp_cells": cells,
                    "grouped_kernel_ms": ms_g, "grouped_device_ms_events": float(np.median(dev)),
                    "matrix_kernel_ms": ms_m,
                    "grouped_gcells_per_s": cells / ms_g / 1e6, "matrix_gcells_per_s": cells / ms_m / 1e6,
                    "grouped_speedup_per_cell": ms_m / ms_g})
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
