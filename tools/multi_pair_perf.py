"""Batched scan of a motif-pair collection in the combined mode over two FASTA symbol streams
(device.scan_onehot_many on the sequence stream + device.scan_pair_onehot_many on both) beside the per-pair chain
it replaces (device.scan_seq + device.scan_pair_onehot, one of each per pair).

Streams: synth.rna_codes and synth.struct_codes over one record_lengths draw (separators coincide), 125 M
symbols each (records of ~2500), and 1 G symbols each (the same pair tiled 8 times); every stream is larger than
the 126 MB L2.  Motif pairs: M in {8, 32, 256}, both PSSMs of one W in 7..12, at m = 6 and m = STRUCT_THR.
CUDA events around each Python call (hit download included), 2 warm-ups, median and spread of REPS runs (the
per-pair loop at 1 G symbols and 256 pairs: one run).  Hits and both scores per pair are checked identical.  The
kernel split (k-mer table builds / count pass / offsets / write pass, sequence-only and pair kernels apart) comes
from one torch.profiler run per shape.  Last, the CLI's --stats scan_s for `-p <256> -q <256> seqs.fa structs.fa`
over a generated 100 Mnt pair of FASTA files, batched and with the per-pair loop forced.

    python tools/multi_pair_perf.py [--json out.json] [--skip-cli]
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from rnascan_b200 import device, synth  # noqa: E402
from multi_fasta_perf import STRUCT_THR, card, stats, timed  # noqa: E402

REPS = 5


def kernel_split(fn):
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    split = {"table_build": 0.0, "seq_count": 0.0, "seq_write": 0.0, "pair_count": 0.0, "pair_write": 0.0,
             "offsets": 0.0}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        name, us = ev.name, ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
        if "kmer_mask_build" in name:
            split["table_build"] += us / 1e3
        elif "multi_scan_kernel<" in name:            # multi_scan_kernel<A, PAIR, WRITE>
            args = [a.strip() for a in name.split("<", 1)[1].split(">", 1)[0].split(",")]
            key = ("pair_" if args[1] == "true" else "seq_") + ("write" if args[2] == "true" else "count")
            split[key] += us / 1e3
        elif "multi_offsets" in name or "multi_bases" in name:
            split["offsets"] += us / 1e3
    return split


def make_pair(n_small):
    rng = np.random.default_rng(3)
    lengths = synth.record_lengths(n_small, max(1, n_small // 2500), rng)
    seq, _ = synth.rna_codes(lengths, rng, n_frac=0.0)
    st, _ = synth.struct_codes(lengths, rng)
    return seq, st


def run_kernels(res):
    seq, st = make_pair(125_000_000 - 50_000)
    for scale in (1, 8):
        ss = device.SymbolStream(np.tile(seq, scale) if scale > 1 else seq, kind="rna")
        sq = device.SymbolStream(np.tile(st, scale) if scale > 1 else st, kind="struct")
        n = ss.n
        for thr in (6.0, STRUCT_THR):
            for M in (8, 32, 256):
                rng = np.random.default_rng(M)
                widths = rng.integers(7, 13, size=M)
                ts = [synth.pssm_table(synth.pfm_rows(int(w), 4, rng)) for w in widths]
                tq = [synth.pssm_table(synth.pfm_rows(int(w), 7, rng)) for w in widths]

                def batched():
                    return device.scan_onehot_many(ss, ts, thr), device.scan_pair_onehot_many(ss, sq, ts, tq, thr)

                def loop():
                    return [(device.scan_seq(ss, a, thr), device.scan_pair_onehot(ss, sq, a, b, thr))
                            for a, b in zip(ts, tq)]
                timed(batched, 2)
                (one, pair), ms_b = timed(batched, REPS)
                timed(lambda: (device.scan_seq(ss, ts[0], thr), device.scan_pair_onehot(ss, sq, ts[0], tq[0], thr)), 2)
                ref, ms_l = timed(loop, 1 if (scale == 8 and M == 256) else 3)
                _, pos1, sc1, b1 = one
                _, pos2, sa2, sb2, b2 = pair
                same = all(np.array_equal(pos1[b1[m]:b1[m + 1]], ref[m][0][0]) and
                           np.array_equal(sc1[b1[m]:b1[m + 1]], ref[m][0][1]) and
                           np.array_equal(pos2[b2[m]:b2[m + 1]], ref[m][1][0]) and
                           np.array_equal(sa2[b2[m]:b2[m + 1]], ref[m][1][1]) and
                           np.array_equal(sb2[b2[m]:b2[m + 1]], ref[m][1][2]) for m in range(M))
                row = {"n": n, "M": M, "threshold": thr, "seq_hits": int(b1[-1]), "joint_hits": int(b2[-1]),
                       "batched": stats(ms_b), "per_pair_loop": stats(ms_l), "identical": bool(same),
                       "speedup": float(np.median(ms_l) / np.median(ms_b)), "kernel_split_ms": kernel_split(batched)}
                print(json.dumps(row), flush=True)
                res["kernels"].append(row)
        del ss, sq
        torch.cuda.empty_cache()


def run_cli(res):
    from rnascan_b200 import pfmutil, rnascan as ms
    tmp = tempfile.mkdtemp(prefix="multi_pair_perf_")
    rng = np.random.default_rng(7)
    lengths = synth.record_lengths(100_000_000, 40_000, rng)
    paths = {}
    for kind, fn in (("rna", synth.rna_codes), ("struct", synth.struct_codes)):
        codes, _ = fn(lengths, rng) if kind == "struct" else fn(lengths, rng, n_frac=0.0)
        text = synth.to_text(codes, kind).decode().split("\n")[:-1]
        paths[kind] = os.path.join(tmp, kind + ".fa")
        with open(paths[kind], "w") as fh:
            for k, r in enumerate(text):
                fh.write(">rec%d synthetic record %d\n%s\n" % (k, k, r))
    pfm = {"rna": [], "struct": []}
    for w in rng.integers(7, 13, size=256):
        for kind, letters in (("rna", "ACGU"), ("struct", "BEHLMRT")):
            rows = synth.pfm_rows(int(w), len(letters), rng)
            pfm[kind].append({c: rows[:, i].tolist() for i, c in enumerate(letters)})
    files = {}
    for kind in pfm:
        files[kind] = os.path.join(tmp, kind + "256.pfm")
        pfmutil.write_multi_pfm(["m%d" % i for i in range(256)], pfm[kind], files[kind])
    real = ms._batched_pair_hits
    for label, router in (("batched", real), ("per_pair_loop", lambda *a, **k: None), ("batched_again", real)):
        ms._batched_pair_hits = router
        ms._BATCH_CACHE.clear()
        st = os.path.join(tmp, label + ".json")
        t0 = time.perf_counter()
        with open(os.devnull, "w") as null:
            saved, saved_err = sys.stdout, sys.stderr
            sys.stdout, sys.stderr = null, null
            try:
                ms.main(["-p", files["rna"], "-q", files["struct"], "-C", "0.01", "-m", "6", paths["rna"],
                         paths["struct"], "--stats", st])
            finally:
                sys.stdout, sys.stderr = saved, saved_err
        wall = time.perf_counter() - t0
        with open(st) as fh:
            line = json.loads(fh.readline())
        row = {"run": label, "wall_s": wall, "scan_s": line["phases_s"].get("scan_s"), "total_s": line["total_s"],
               "batched_motifs": line.get("batched_motifs")}
        print(json.dumps(row), flush=True)
        res["cli"].append(row)
    ms._batched_pair_hits = real


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
