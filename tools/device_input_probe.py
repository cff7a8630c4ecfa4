#!/usr/bin/env python3
"""Probe of reads that are already in GPU memory: config 2 (synth.ont037, 765k reads) with 1 in 5000 bases replaced by
N / R / Y / n, held as CUDA tensors (uint8 bases, int64 offsets), matched two ways, alternating after warm-up:
  (a) Matcher.match_device: host clock around the call, plus the CUDA-event times it reports (pack kernels, whole call);
  (b) the host route on the same reads: copy bases and offsets to pinned host memory, PackedBatch.from_blob with
      clip = search_len, Matcher.match (pinned result pool reused, as the file pipeline does).
Records, offsets and matched counts of the two routes must be identical.  Prints the card name and power limit read in
the same run and one JSON object; --out writes it to a file too.

    python tools/device_input_probe.py --steps 10 --out profiles/device_input_probe.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, ROOT)


def _card(device):
    import torch
    info = {"gpu": torch.cuda.get_device_name(device)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        info.update(nvidia_smi_name=name, power_limit=power, max_sm_clock=clock)
    except (OSError, ValueError, subprocess.SubprocessError):
        info.update(power_limit="unknown")
    return info


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reads", type=int, default=765_000)
    ap.add_argument("--steps", type=int, default=10, help="timed calls of each route (alternating)")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    from specimux_b200 import synth
    from specimux_b200.engine import Matcher, PackedBatch
    from specimux_b200.models import MatchParameters
    from specimux_b200.orchestration import thresholds_for
    from specimux_b200.tables import MatchTables
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers as H

    ds = synth.ont037(n_reads=a.reads, with_quals=False)
    specimens = H.build_specimens(ds.primers, ds.specimens)
    k_idx, k_primers = thresholds_for(specimens)
    mt = MatchTables(specimens, MatchParameters(k_primers, k_idx, ds.search_len, True))
    codes = np.frombuffer(b"ACGT", dtype=np.uint8)[ds.codes].copy()
    rng = np.random.default_rng(2024)
    hits = rng.choice(codes.shape[0], size=codes.shape[0] // 5000, replace=False)
    codes[hits] = np.frombuffer(b"NRYn", dtype=np.uint8)[rng.integers(0, 4, size=hits.shape[0])]
    dev = torch.device("cuda", a.device)
    bases = torch.tensor(codes, device=dev)
    offsets = torch.tensor(ds.offsets.astype(np.int64), device=dev)
    h_bases = torch.empty(bases.shape, dtype=torch.uint8, pin_memory=True)
    h_offsets = torch.empty(offsets.shape, dtype=torch.int64, pin_memory=True)
    torch.cuda.synchronize(dev)
    card = _card(a.device)
    clip = ds.search_len
    pool = {}

    def device_route():
        t = time.perf_counter()
        r = m.match_device(bases, offsets)
        return time.perf_counter() - t, r

    def host_route():
        t = time.perf_counter()
        h_bases.copy_(bases)
        h_offsets.copy_(offsets)
        batch = PackedBatch.from_blob(h_bases.numpy().ctypes.data, h_offsets.numpy().view(np.uint64), clip=clip)
        r = m.match(batch, reuse=pool)
        return time.perf_counter() - t, r, batch.n_flagged

    dev_s, dev_ms, host_s = [], [], []
    with Matcher(mt, device=a.device) as m:
        for _ in range(a.warmup):
            device_route()
            host_route()
        for _ in range(a.steps):
            s, got = device_route()
            dev_s.append(s)
            dev_ms.append(got.device_ms)
            s, want, n_flagged = host_route()
            host_s.append(s)
            back = got.to_host()
            assert back.n_matched == want.n_matched
            assert np.array_equal(back.rec_offset, want.rec_offset)
            assert back.records.tobytes() == want.records.tobytes()
    med = lambda v: float(np.median(v)) * 1e3
    out = dict(card, config="ont037", reads=int(ds.n_reads), bases=int(codes.shape[0]), search_len=clip,
               substituted_bases=int(hits.shape[0]), flagged_reads=int(n_flagged), records=int(want.records.shape[0]),
               matched=int(want.n_matched), steps=a.steps, warmup=a.warmup, identical=True,
               match_device_ms=dict(host_clock_median=med(dev_s), host_clock_min=float(min(dev_s)) * 1e3,
                                    pack_kernels_median=float(np.median([x[0] for x in dev_ms])),
                                    device_call_median=float(np.median([x[1] for x in dev_ms]))),
               host_route_ms=dict(host_clock_median=med(host_s), host_clock_min=float(min(host_s)) * 1e3),
               per_step=dict(match_device_s=dev_s, match_device_device_ms=dev_ms, host_route_s=host_s))
    print("%s, power limit %s" % (card["gpu"], card.get("power_limit")))
    print(json.dumps(out))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
