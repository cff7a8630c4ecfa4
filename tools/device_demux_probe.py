#!/usr/bin/env python3
"""Probe of the demultiplexed output in GPU memory: config 2 (synth.ont037, 765k reads, with qualities; 1 in 2000 bases
replaced by IUPAC / lower-case / U letters) held as CUDA tensors, demultiplexed three ways, alternating after warm-up:
  (a) Matcher.demux_device: host clock around the call, plus the CUDA-event times of the copy kernels and of the call;
  (b) Matcher.match_device, then the same output built with plain torch ops on the device: the destination key and a
      stable torch.sort, a repeat_interleave gather with descending indices for reversed records, a lookup-table
      complement;
  (c) Matcher.match_device, then records, bases and qualities copied to pinned host memory, then the native writer
      (libspecimux_io) formatting the records in console form (stdout sent to /dev/null) from a block of the same reads.
(a) and (b) must give identical bytes, offsets, record order and groups.  The copy kernels' bytes moved (every output
byte read once and written once, sequences and qualities) over their CUDA-event time is set against 7.7 TB/s.  Prints
the card name and power limit read in the same run and one JSON object; --out writes it to a file too.

    python tools/device_demux_probe.py --steps 10 --out profiles/device_demux_probe.json
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from device_input_probe import _card  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def torch_demux(res, bases, offsets, quals, tables):
    """Route (b): DeviceDemux's arrays from DeviceBatchResult records with torch ops only."""
    import torch
    rec = res.records
    n = rec.shape[0]
    i32, i16 = rec.view(torch.int32), rec.view(torch.int16)
    read, sample, ts, te = i32[:, 0].long(), i32[:, 1].long(), i32[:, 2].long(), i32[:, 3].long()
    pool, p1, p2 = i16[:, 24].long(), i16[:, 25].long(), i16[:, 26].long()
    resol, rev, empty = rec[:, 58].long(), rec[:, 59] != 0, rec[:, 60] != 0
    live = ~empty
    res_eff = torch.where(empty, torch.full_like(resol, 5), resol)
    top = torch.where(res_eff == 5, 2, torch.where((res_eff == 2) | (res_eff == 3), 1, 0))
    kind = torch.where((res_eff == 1) | (res_eff == 4) | (res_eff == 6), 0,
                       torch.where(res_eff == 2, 1, torch.where(res_eff == 3, 2, 3)))
    field = lambda x: torch.where(live & (x >= 0), x + 1, 0)
    smp = torch.where(kind < 3, sample, 0)
    key = (top << 62) | (field(pool) << 52) | (field(p1) << 44) | (field(p2) << 36) | (kind << 30) | smp
    order = torch.sort(key ^ (-(1 << 63)), stable=True).indices            # unsigned order of the 64-bit key
    start = offsets[read]
    L = offsets[read + 1] - start
    s = torch.clamp(torch.where(ts < 0, ts + L, ts), min=0)
    s = torch.minimum(s, L)
    e = torch.minimum(torch.clamp(torch.where(te < 0, te + L, te), min=0), L)
    e = torch.maximum(e, s)
    s, e = torch.where(live, s, 0), torch.where(live, e, L)
    first = torch.where(rev, start + L - 1 - s, start + s)[order]
    lens = (e - s)[order]
    step = torch.where(rev, -1, 1)[order]
    out_off = torch.zeros(n + 1, dtype=torch.int64, device=rec.device)
    torch.cumsum(lens, 0, out=out_off[1:])
    total = int(out_off[-1])
    pos = torch.arange(total, device=rec.device) - torch.repeat_interleave(out_off[:-1], lens, output_size=total)
    src = torch.repeat_interleave(first, lens, output_size=total) + pos * torch.repeat_interleave(step, lens, output_size=total)
    lut = torch.arange(256, dtype=torch.uint8, device=rec.device)
    lut[torch.tensor(list(b"ACGTMRWSYKVHDBXNacgtmrwsykvhdbxnUu"), device=rec.device)] = \
        torch.tensor(list(b"TGCAKYWSRMBDHVXNtgcakywsrmbdhvxnAa"), dtype=torch.uint8, device=rec.device)
    seq = bases[src]
    seq = torch.where(torch.repeat_interleave(rev[order], lens, output_size=total), lut[seq.long()], seq)
    qual = quals[src]
    k = key[order]
    starts = torch.nonzero(torch.cat([torch.ones(1, dtype=torch.bool, device=rec.device), k[1:] != k[:-1]])).flatten()
    return order, out_off, seq, qual, k[starts], torch.cat([starts, torch.tensor([n], device=rec.device)])


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reads", type=int, default=765_000)
    ap.add_argument("--steps", type=int, default=10, help="timed calls of each route (alternating)")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--device", type=int, default=0)
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
    dev = torch.device("cuda", a.device)
    bases, quals = torch.tensor(codes, device=dev), torch.tensor(qtext, device=dev)
    offsets = torch.tensor(ds.offsets.astype(np.int64), device=dev)
    h_bases = torch.empty(bases.shape, dtype=torch.uint8, pin_memory=True)
    h_quals = torch.empty(quals.shape, dtype=torch.uint8, pin_memory=True)
    card = _card(a.device)

    # route (c) formats from a reader block of the same reads (the writer takes its reads from the native reader)
    tmp = tempfile.mkdtemp(prefix="demux_probe_")
    fq = os.path.join(tmp, "reads.fastq")
    with open(fq, "wb") as fh:
        off = ds.offsets
        for i in range(ds.n_reads):
            fh.write(b"@r%d\n%s\n+\n%s\n" % (i, codes[off[i]:off[i + 1]].tobytes(), qtext[off[i]:off[i + 1]].tobytes()))
    rd = native_io.FastxReader(fq, True)
    blk = rd.next_block(ds.n_reads + 1)
    os.remove(fq)
    assert blk.n_reads == ds.n_reads
    devnull = os.open(os.devnull, os.O_WRONLY)

    def route_a():
        t = time.perf_counter()
        r = m.demux_device(bases, offsets, quals)
        return time.perf_counter() - t, r

    def route_b():
        t = time.perf_counter()
        res = m.match_device(bases, offsets)
        r = torch_demux(res, bases, offsets, quals, mt)
        torch.cuda.synchronize(dev)
        return time.perf_counter() - t, r

    def route_c():
        t = time.perf_counter()
        res = m.match_device(bases, offsets)
        h_bases.copy_(bases)
        h_quals.copy_(quals)
        recs = res.to_host().records
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(devnull, 1)
        try:
            with native_io.TreeWriter(None, "", True, mt) as wr:
                wr.write(blk, recs)
        finally:
            os.dup2(saved, 1)
            os.close(saved)
        return time.perf_counter() - t, len(recs)

    sa, sb, sc, dms = [], [], [], []
    with Matcher(mt, device=a.device) as m:
        for _ in range(a.warmup):
            route_a(); route_b(); route_c()
        for _ in range(a.steps):
            s, got = route_a()
            sa.append(s)
            dms.append(got.device_ms)
            s, want = route_b()
            sb.append(s)
            s, n_rec = route_c()
            sc.append(s)
            order, out_off, seq, qual, gkey, goff = want
            assert torch.equal(got.record, order) and torch.equal(got.offsets, out_off)
            assert torch.equal(got.seq, seq) and torch.equal(got.qual, qual)
            assert np.array_equal(got.group_key.view(np.int64), gkey.cpu().numpy()) and np.array_equal(got.group_offset, goff.cpu().numpy())
    total = int(got.offsets[-1])
    med = lambda v: float(np.median(v)) * 1e3
    copy_ms = float(np.median([x[0] for x in dms]))
    moved = 2 * 2 * total                       # sequences and qualities, each read once and written once
    out = dict(card, config="ont037", reads=int(ds.n_reads), bases=int(codes.shape[0]), substituted_bases=int(hits.shape[0]),
               records=int(n_rec), outputs=int(got.record.numel()), groups=len(got.group_key), output_bytes=total,
               steps=a.steps, warmup=a.warmup, identical_a_b=True,
               demux_device_ms=dict(host_clock_median=med(sa), host_clock_min=float(min(sa)) * 1e3,
                                    copy_kernels_median=copy_ms, device_call_median=float(np.median([x[1] for x in dms]))),
               torch_ops_route_ms=dict(host_clock_median=med(sb), host_clock_min=float(min(sb)) * 1e3),
               host_writer_route_ms=dict(host_clock_median=med(sc), host_clock_min=float(min(sc)) * 1e3),
               copy_kernels=dict(bytes_moved=moved, bytes_per_s=moved / (copy_ms * 1e-3),
                                 share_of_7_7_TBps=moved / (copy_ms * 1e-3) / HBM_BYTES_PER_S),
               per_step=dict(demux_device_s=sa, demux_device_device_ms=dms, torch_ops_route_s=sb, host_writer_route_s=sc))
    os.close(devnull)
    rd.close()
    os.rmdir(tmp)
    print("%s, power limit %s" % (card["gpu"], card.get("power_limit")))
    print(json.dumps(out))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
