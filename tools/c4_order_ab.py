"""Config 4 (combined sequence PSSM + averaged 7-channel profile, computed background) in both orders, one process.

Builds bench.py's shard (bench.make_device_shard / make_tables_fn), times device.BackgroundFusedScan sequence-first
and structure-first alternately (--rounds x --steps each, after a warm-up), checks that both return the same hits bit
for bit (positions, float32 and float64 score bits), and prints one JSON line: median and spread of ms per step per
order, bytes per step from shapes and counters, and the card's name and power limit.  --trace FILE adds a
torch.profiler kernel breakdown of a few steps per order, taken in a separate pass after the timing.

    python tools/c4_order_ab.py [--symbols 1000000000] [--rounds 3] [--steps 20] [--trace out.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--symbols", type=int, default=1_000_000_000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--threshold", type=float, default=None)
    ap.add_argument("--trace", default=None)
    args = ap.parse_args()

    import torch
    import bench
    from rnascan_b200 import device as dev, _lib

    device = torch.device("cuda", 0)
    torch.cuda.set_device(device)
    shard = bench.make_device_shard(args.symbols, 4000, "c4", device)
    n, codes, prof = shard["n"], shard["codes"], shard["prof"]
    tables = bench.make_tables_fn("c4")
    tq = tables(np.zeros(8, np.int64))[1]
    W = tq.shape[0]
    thr = bench.THRESHOLD if args.threshold is None else args.threshold
    absmax = dev.ProfileStream.from_device(prof, n).absrow_max()
    cap = max(1 << 16, n // 256)
    jobs = {"sequence_first": dev.BackgroundFusedScan(n, device, capacity=cap, structure_first=False),
            "structure_first": dev.BackgroundFusedScan(n, device, capacity=cap, structure_first=True)}
    stream = torch.cuda.current_stream()

    def step(job):
        job.launch(codes, prof, _lib.RS_F32, W, tq, lambda c: tables(c)[0], thr, absmax)

    for job in jobs.values():
        for _ in range(5):
            step(job)
    torch.cuda.synchronize()
    times = {k: [] for k in jobs}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for name, job in jobs.items():
            e0.record(stream)
            for _ in range(args.steps):
                step(job)
            e1.record(stream)
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / args.steps)

    res = {k: j.results() for k, j in jobs.items()}
    if any(r is None for r in res.values()):
        raise SystemExit("candidate buffer overflowed")
    (p0, q0, s0), (p1, q1, s1) = res["sequence_first"], res["structure_first"]
    same = (np.array_equal(p0, p1) and np.array_equal(q0.view(np.uint32), q1.view(np.uint32))
            and np.array_equal(s0.view(np.uint64), s1.view(np.uint64)))
    sf = jobs["sequence_first"].hb.cand_counters.cpu().numpy()
    out = {"card": card(), "symbols": n, "W": W, "minscore": thr, "hits": int(len(p0)), "bit_equal": bool(same),
           "steps": args.steps, "rounds": args.rounds,
           "ms_per_step": {k: {"median": float(np.median(v)), "min": float(min(v)), "max": float(max(v)),
                               "spread": float((max(v) - min(v)) / np.median(v)), "rounds": v}
                           for k, v in times.items()},
           # from shapes and counters: symbols read twice (histogram, sequence scan), 28 B of profile rows + W
           # symbols per scored candidate (sequence first); symbols + rows once (structure first)
           "bytes_per_step": {"sequence_first": int(2 * n + int(sf[1]) * W * 28 + int(sf[0]) * 8),
                              "structure_first": int(29 * n + n)},
           "sequence_candidates": int(sf[0]), "structure_scores_computed": int(sf[1])}
    out["speedup"] = out["ms_per_step"]["structure_first"]["median"] / out["ms_per_step"]["sequence_first"]["median"]

    if args.trace:
        from torch.profiler import profile, ProfilerActivity
        breakdown = {}
        for name, job in jobs.items():
            with profile(activities=[ProfilerActivity.CUDA]) as pr:
                for _ in range(5):
                    step(job)
                torch.cuda.synchronize()
            agg = {}
            for e in pr.events():
                if e.device_type == torch.autograd.DeviceType.CUDA:
                    agg[e.name[:80]] = agg.get(e.name[:80], 0.0) + (e.time_range.end - e.time_range.start) / 5
            breakdown[name] = dict(sorted(agg.items(), key=lambda kv: -kv[1]))
        with open(args.trace, "w") as fh:
            json.dump({"unit": "us per step", "card": out["card"], "kernels": breakdown}, fh, indent=1)
    print(json.dumps(out))
    if not same:
        raise SystemExit("the two orders disagree")


if __name__ == "__main__":
    main()
