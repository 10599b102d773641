"""Batched scan of a motif collection over one FASTA symbol stream (device.scan_onehot_many, rs_scan_onehot_many)
beside the per-motif scans it replaces (device.scan_seq / scan_struct_onehot, one call per motif).

Streams: synth.rna_codes / synth.struct_codes, 125 M symbols (records of ~2500), and 1 G symbols (the same
stream tiled 8 times); both are larger than the 126 MB L2.  Motifs: M in {8, 32, 256} synth.pfm_rows PSSMs of
W 7..12 at m = 6 (RNA) and m = STRUCT_THR (structure; printed hit rates show how the two compare).
CUDA events around each Python call (hit download included), 2 warm-ups, median and spread of REPS runs (the
per-motif loop at 1 G symbols and 256 motifs: one run).  Hits per motif are checked identical.  The kernel
split (k-mer table build / count pass / offsets / write pass) comes from one torch.profiler run per shape.
Achieved symbol rate = passes x n bytes / kernel time; table-row L2 bytes per position = 2 passes x
ceil(M_group / 32) x 4 B.  Last, the CLI's --stats scan_s for `-p <256-motif file> seqs.fa` over a generated
100 Mnt FASTA, batched and with the per-motif loop forced.

    python tools/multi_fasta_perf.py [--json out.json] [--skip-cli]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rnascan_b200 import device, synth  # noqa: E402

REPS = 5
STRUCT_THR = 4.0


def card():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def timed(fn, reps):
    out, ms = None, []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return out, ms


def stats(ms):
    return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms)), "n": len(ms)}


def kernel_split(fn):
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    split = {"table_build": 0.0, "count": 0.0, "offsets": 0.0, "write": 0.0}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        name, us = ev.name, ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
        if "kmer_mask_build" in name:
            split["table_build"] += us / 1e3
        elif "multi_scan_kernel" in name:
            split["write" if "true" in name or "Lb1E" in name else "count"] += us / 1e3
        elif "multi_offsets" in name or "multi_bases" in name:
            split["offsets"] += us / 1e3
    return split


def shapes(kind, n_small):
    rng = np.random.default_rng(1 if kind == "rna" else 2)
    lengths = synth.record_lengths(n_small, max(1, n_small // 2500), rng)
    codes, offsets = (synth.rna_codes if kind == "rna" else synth.struct_codes)(lengths, rng)
    return codes, offsets, lengths


def run_kernels(res):
    for kind in ("rna", "struct"):
        A = 4 if kind == "rna" else 7
        thr = 6.0 if kind == "rna" else STRUCT_THR
        codes, offsets, lengths = shapes(kind, 125_000_000 - 50_000)
        for scale in (1, 8):
            big = np.tile(codes, scale) if scale > 1 else codes
            stream = device.SymbolStream(big, kind=kind)
            n = stream.n
            for M in (8, 32, 256):
                rng = np.random.default_rng(M)
                tables = [synth.pssm_table(synth.pfm_rows(int(w), A, rng)) for w in rng.integers(7, 13, size=M)]
                batched = lambda: device.scan_onehot_many(stream, tables, thr)
                timed(batched, 2)
                (motif, pos, sc, bases), ms_b = timed(batched, REPS)
                per = device.scan_seq if kind == "rna" else device.scan_struct_onehot
                loop = lambda: [per(stream, t, thr) for t in tables]
                timed(lambda: per(stream, tables[0], thr), 2)
                loop_reps = 1 if (scale == 8 and M == 256) else 3
                ref, ms_l = timed(loop, loop_reps)
                same = all(np.array_equal(pos[bases[m]:bases[m + 1]], ref[m][0]) and
                           np.array_equal(sc[bases[m]:bases[m + 1]], ref[m][1]) for m in range(M))
                split = kernel_split(batched)
                kern = split["count"] + split["write"]
                groups = (M + 255) // 256
                words = sum((min(256, M - 256 * g) + 31) // 32 for g in range(groups))
                row = {"kind": kind, "n": n, "M": M, "threshold": thr, "hits": int(bases[-1]),
                       "hits_per_position_per_motif": int(bases[-1]) / n / M,
                       "batched": stats(ms_b), "per_motif_loop": stats(ms_l), "identical": bool(same),
                       "speedup": float(np.median(ms_l) / np.median(ms_b)), "kernel_split_ms": split,
                       "symbol_GBps_count_plus_write": 2 * groups * n / (kern * 1e-3) / 1e9 if kern > 0 else None,
                       "table_L2_bytes_per_position": 2 * words * 4}
                print(json.dumps(row), flush=True)
                res["kernels"].append(row)
            del stream
            torch.cuda.empty_cache()


def run_cli(res):
    from rnascan_b200 import pfmutil, rnascan as ms
    tmp = tempfile.mkdtemp(prefix="multi_fasta_perf_")
    rng = np.random.default_rng(7)
    lengths = synth.record_lengths(100_000_000, 40_000, rng)
    codes, _ = synth.rna_codes(lengths, rng)
    text = synth.to_text(codes, "rna").decode().split("\n")[:-1]
    fasta = os.path.join(tmp, "seqs.fa")
    with open(fasta, "w") as fh:
        for k, r in enumerate(text):
            fh.write(">rec%d synthetic record %d\n%s\n" % (k, k, r))
    pfms = []
    for w in rng.integers(7, 13, size=256):
        rows = synth.pfm_rows(int(w), 4, rng)
        pfms.append({c: rows[:, i].tolist() for i, c in enumerate("ACGU")})
    pfm = os.path.join(tmp, "coll256.pfm")
    pfmutil.write_multi_pfm(["m%d" % i for i in range(256)], pfms, pfm)
    real = ms._batched_fasta_hits
    for label, router in (("batched", real), ("per_motif_loop", lambda *a, **k: None), ("batched_again", real)):
        ms._batched_fasta_hits = router
        ms._BATCH_CACHE.clear()
        st = os.path.join(tmp, label + ".json")
        t0 = time.perf_counter()
        with open(os.devnull, "w") as null:
            saved, saved_err = sys.stdout, sys.stderr
            sys.stdout, sys.stderr = null, null
            try:
                ms.main(["-p", pfm, "-C", "0.01", "-m", "6", fasta, "--stats", st])
            finally:
                sys.stdout, sys.stderr = saved, saved_err
        wall = time.perf_counter() - t0
        with open(st) as fh:
            line = json.loads(fh.readline())
        row = {"run": label, "wall_s": wall, "scan_s": line["phases_s"].get("scan_s"), "total_s": line["total_s"],
               "batched_motifs": line.get("batched_motifs")}
        print(json.dumps(row), flush=True)
        res["cli"].append(row)
    ms._batched_fasta_hits = real


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default=None)
    ap.add_argument("--skip-cli", action="store_true")
    a = ap.parse_args()
    device.require_cuda()
    name, limit = card()
    res = {"card": name, "power_limit": limit, "kernels": [], "cli": []}
    print(json.dumps({"card": name, "power_limit": limit}), flush=True)
    run_kernels(res)
    if not a.skip_cli:
        run_cli(res)
    if a.json:
        with open(a.json, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
