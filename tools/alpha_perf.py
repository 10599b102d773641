"""Kernel times of the alphabet scans (rs_scores_dense_alpha, rs_scan_alpha at m = 6) for A in {5, 20, 31} and
W in {7, 12}, beside the BEHLMRT kernels (rs_scores_dense_struct, rs_scan_struct_onehot) on a stream of the same
length.  The stream (default 512 M symbols, larger than the 126 MB L2, so every pass reads HBM) is drawn on the
device: uniform letter indices, about a fifth of them lower case, one separator per ~2500 symbols.
CUDA events around each call, 3 warm-ups, median of 10.  Rates: positions per second, and bytes per second
counting 1 B/position for hit scans (the symbols) and 9 B/position for dense fp64 output.

    python tools/alpha_perf.py [--n 512000000] [--json alpha_perf.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rnascan_b200 import _lib, device, synth  # noqa: E402
from rnascan_b200._lib import lib, check  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def codes_for(raw, sep, A, lower):
    """Alphabet-layout (or, with lower = 8, structure-layout) codes: index raw % A, `lower` bit on ~1/5."""
    c = (raw % A) | ((raw >= 205).to(torch.uint8) * lower)
    c[sep] = _lib.RS_SEP
    return c


def timed(fn, reps=10, warm=3):
    for _ in range(warm):
        fn()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512_000_000)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    device.require_cuda()
    n = args.n
    npad = device.padded_count(n)
    g = torch.Generator(device="cuda").manual_seed(7)
    raw = torch.randint(0, 256, (npad,), dtype=torch.uint8, device="cuda", generator=g)
    sep = torch.arange(2499, npad, 2500, device="cuda")
    raw[n:] = 0
    out = torch.empty(n, dtype=torch.float64, device="cuda")
    cap = n // 16
    hb = device.HitBuffers(n, cap, "cuda", want_seq=False, want_struct=True)
    st = device._stream()
    name, limit = card()
    print("# %s, power limit %s, n = %d symbols, median of 10 after 3 warm-ups" % (name, limit, n))
    rows = []

    def record(what, A, W, ms, bpp, hits=None):
        r = {"kernel": what, "A": A, "W": W, "ms": round(ms, 4), "gpos_s": round(n / ms / 1e6, 2),
             "gb_s": round(n * bpp / ms / 1e6, 1)}
        if hits is not None:
            r["hits"] = hits
        rows.append(r)
        print("%-22s A=%2d W=%2d  %8.3f ms  %7.2f Gpos/s  %7.1f GB/s%s"
              % (what, A, W, ms, r["gpos_s"], r["gb_s"], "" if hits is None else "  hits=%d" % hits))

    rng = np.random.default_rng(3)
    for W in (7, 12):
        for A in (7, 5, 20, 31):
            struct = A == 7                                    # the BEHLMRT kernels on a structure stream
            codes = codes_for(raw, sep, A, 8 if struct else _lib.RS_ALPHA_LOWER)
            codes[n:] = _lib.RS_SEP
            table = np.ascontiguousarray(synth.pssm_table(synth.pfm_rows(W, A, rng)))
            if struct:
                dense = lambda: check(lib.rs_scores_dense_struct(codes.data_ptr(), n, table.ctypes.data, W,
                                                                 out.data_ptr(), st))
                scan = lambda: check(lib.rs_scan_struct_onehot(codes.data_ptr(), n, table.ctypes.data, W, 6.0, cap,
                                                               hb.pos.data_ptr(), hb.struct.data_ptr(),
                                                               hb.counters.data_ptr(), hb.work.data_ptr(),
                                                               hb.work_bytes, st))
            else:
                dense = lambda: check(lib.rs_scores_dense_alpha(codes.data_ptr(), n, table.ctypes.data, W, A,
                                                                out.data_ptr(), st))
                scan = lambda: check(lib.rs_scan_alpha(codes.data_ptr(), n, table.ctypes.data, W, A, 6.0, cap,
                                                       hb.pos.data_ptr(), hb.struct.data_ptr(), hb.counters.data_ptr(),
                                                       hb.work.data_ptr(), hb.work_bytes, st))
            label = "struct" if struct else "alpha"
            if W == 7 and A in (7, 31):                        # background counts: 1 B/position
                counts = torch.zeros(32, dtype=torch.int64, device="cuda")
                hist = lib.rs_hist if struct else lib.rs_hist_alpha
                record("hist_" + label, A, 0, timed(lambda: check(hist(codes.data_ptr(), n, counts.data_ptr(), st))),
                       1.0)
            record("dense_" + label, A, W, timed(dense), 9.0)
            ms = timed(scan)
            hits = int(hb.counters[0].item())
            if hits > cap:
                raise SystemExit("hit buffer overflow: %d hits" % hits)
            record("scan_" + label + " m=6", A, W, ms, 1.0, hits)
            del codes
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as fh:
            json.dump({"gpu": name, "power_limit": limit, "n": n, "rows": rows}, fh, indent=1)


if __name__ == "__main__":
    main()
