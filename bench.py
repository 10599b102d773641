#!/usr/bin/env python
"""Benchmark of the rnascan_b200 hot path (contract: see the task statement / DESIGN.md).

    python bench.py --gpus 1 --steps 10 --warmup 3              # this framework (default)
    python bench.py ... --dump-outputs DIR                      # also write the last timed step's results as .npy
    python bench.py --impl reference --gpus 1 --steps 3 ...     # the reference's CPU path
    torchrun ... bench.py --gpus N ...                          # one rank per GPU, the 1 Gnt split N ways

Workload (default "c4", BASELINE.json configs[3] -- the configuration the north-star's
HBM-fraction target is quoted on): combined sequence-PSSM + averaged 7-channel structure
profile scan of 1 Gnt in total (one GPU holds all of it: 29 GB; N GPUs hold 1/N each -- strong
scaling; --n-per-gpu fixes the per-GPU share instead), W = 7, m = 6, sequence background
computed from the data (histogram -> all-reduce of the integer counts -> log-odds on the
host), structure background = the reference's example 3'UTR table.  A step is ONE pass of
the whole path over the rank's shard:   histogram -> [all-reduce] -> PSSM -> fused scan ->
ordered hit compaction.  `--workload c2` / `c3` time the sequence-only and one-hot
structure scans (BASELINE.json configs[1], configs[2]) the same way.

All positions/s figures count scored positions = sum over records of max(0, L - W + 1).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

W_MOTIF = 7
THRESHOLD = 6.0
SS_BG = {"B": 0.0163181097311479, "E": 0.272087789050946, "H": 0.153012079123538,
         "L": 0.204624685341275, "M": 0.0196001330531237, "R": 0.196989713257981,
         "T": 0.137367490441988}       # example/3p_UTR_background_structural_context.txt
ALGO_BYTES = {"c4": 29.0, "c2": 1.0, "c3": 5.0, "c5": 29.0}     # SURVEY.md section 8(d), per scored position
N_MOTIFS_C5 = 256
OTHERS_N = 125_000_000          # symbols per GPU of the side runs (configs 2, 3, 5) and of weak-scaling shards
DUMP_ENTRY_BYTES = 48 << 20     # --dump-outputs: per-hit / per-window arrays beyond this are sampled (64 MB in all)


# ----------------------------------------------------------------------------- helpers
def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def recorded_traffic(workload, n_symbols):
    """DRAM bytes per launch of the workload's dominant kernel from the committed ncu capture
    (profiles/traffic.json, written by tools/ncu_summary.py --traffic), for the same shard size; else None."""
    try:
        with open(os.path.join(REPO, "profiles", "traffic.json")) as fh:
            db = json.load(fh)
        for key, rec in db.items():              # keys: "<workload>" or "<workload>@<size tag>"
            if key.split("@")[0] == workload and abs(rec["symbols_per_gpu"] - n_symbols) <= 0.001 * n_symbols:
                return rec["traffic"], rec["source"]
    except Exception:
        pass
    return None, None


def measured_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled every ~10 ms through NVML while the benchmark runs
    (in-process, so even millisecond-long timed regions get samples); falls back to an
    `nvidia-smi -lms 200` child process when NVML cannot be loaded."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        threading.Thread.__init__(self, daemon=True)
        self.index, self.proc = index, None
        self.sm, self.mx, self.reasons = [], [], set()
        self._stop_flag = threading.Event()

    def _nvml_loop(self):
        import pynvml as nv
        nv.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = self.index
        if vis:
            try:
                idx = int(vis.split(",")[self.index])
            except (ValueError, IndexError):
                pass
        h = nv.nvmlDeviceGetHandleByIndex(idx)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        flags = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self._stop_flag.is_set():
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
            self.mx.append(float(mx))
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            for name, bit in flags.items():
                if r & bit:
                    self.reasons.add(name)
            time.sleep(0.01)

    def _smi_loop(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        self.proc = subprocess.Popen(
            ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
             "--format=csv,noheader,nounits", "-lms", "200"],
            stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        for line in self.proc.stdout:
            r = [c.strip() for c in line.split(",")]
            try:
                self.sm.append(float(r[0])); self.mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)

    def run(self):
        try:
            self._nvml_loop()
        except Exception:
            try:
                self._smi_loop()
            except Exception:
                pass

    def stop(self):
        self._stop_flag.set()
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None,
                "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


# ----------------------------------------------------------------------------- synthetic shard
def record_layout(n_symbols, seed):
    """Record lengths (lognormal, SURVEY 8d) filling ~n_symbols stream slots incl. separators."""
    from rnascan_b200 import synth
    rng = np.random.default_rng(seed)
    n_records = max(1, int(round(n_symbols / 3334.0)))
    lengths = synth.record_lengths(n_symbols - n_records, n_records, rng)
    offsets, total = synth.layout(lengths)
    return lengths, offsets, total


def scored_positions(lengths, W):
    return int(np.maximum(lengths - W + 1, 0).sum())


def dump_outputs(directory, entries, fixed, seed=0):
    """Write every array as <directory>/<name>.npy: float32 stays float32, anything else becomes float64.
    `entries` holds arrays of one length (one element per hit or per window).  When they would take more than
    DUMP_ENTRY_BYTES, each is cut to the same seeded sample of elements, in ascending order, and the sampled
    indices are written as `sample_index`.  The `fixed` arrays are small and are written whole.  Arrays may be
    numpy arrays or tensors; a device tensor is sampled on the device and only the sample is copied to the host."""
    def as_float(a):
        a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
        return a.astype(np.float32 if a.dtype == np.float32 else np.float64, copy=False)

    def take(a, idx):
        if not hasattr(a, "cpu"):
            return np.asarray(a)[idx]
        import torch
        return a[torch.from_numpy(idx).to(a.device)]
    n = len(next(iter(entries.values())))
    per_entry = sum(4 if str(a.dtype).endswith("float32") else 8 for a in entries.values())
    if n * per_entry > DUMP_ENTRY_BYTES:
        idx = np.sort(np.random.default_rng(seed).choice(n, DUMP_ENTRY_BYTES // (per_entry + 8), replace=False))
        entries = {name: take(a, idx) for name, a in entries.items()}
        entries["sample_index"] = idx
    out = {name: as_float(a) for name, a in list(entries.items()) + list(fixed.items())}
    os.makedirs(directory, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def make_device_shard(n_symbols, seed, workload, device):
    """Synthetic shard generated on the device with torch (plumbing only): symbol codes with
    separators + N runs, and (c4) float32 profile rows = Dirichlet(0.2) smoothed by a
    length-5 box filter, re-normalised, separator rows zero."""
    import torch
    from rnascan_b200 import device as dev
    lengths, offsets, n = record_layout(n_symbols, seed)
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    npad = dev.padded_count(n)
    sep_idx = torch.from_numpy(offsets + lengths).to(device)
    if workload == "c3":
        p = torch.tensor([SS_BG[c] for c in "BEHLMRT"], device=device, dtype=torch.float64)
        change = torch.rand(n, device=device, generator=g) >= 0.8
        change[0] = True
        draws = torch.multinomial(p.float(), int(change.sum().item()), replacement=True, generator=g)
        codes = draws[torch.cumsum(change, 0) - 1].to(torch.uint8)
    else:
        cdf = torch.tensor([0.27, 0.49, 0.71], device=device)
        codes = torch.bucketize(torch.rand(n, device=device, generator=g), cdf).to(torch.uint8)
        n_runs = int(n * 0.001 / 25.5)
        if n_runs:
            starts = torch.randint(0, n, (n_runs,), device=device, generator=g)
            runlen = torch.randint(1, 51, (n_runs,), device=device, generator=g)
            mark = torch.zeros(n + 64, device=device, dtype=torch.int32)
            mark.index_add_(0, starts, torch.ones_like(starts, dtype=torch.int32))
            mark.index_add_(0, torch.clamp(starts + runlen, max=n + 63), -torch.ones_like(starts, dtype=torch.int32))
            codes[torch.cumsum(mark[:n], 0) > 0] = 0x0C
            del mark
    full = torch.full((npad,), 0xFF, dtype=torch.uint8, device=device)
    full[:n] = codes
    full[sep_idx] = 0xFF
    del codes
    prof = None
    if workload in ("c4", "c5"):
        prof = torch.zeros((npad, 7), dtype=torch.float32, device=device)
        step = 1 << 24
        for a in range(0, n, step):
            b = min(n, a + step)
            lo, hi = max(0, a - 2), min(n, b + 2)
            gam = torch._standard_gamma(torch.full((hi - lo, 7), 0.2, device=device), generator=g)
            gam = gam / gam.sum(1, keepdim=True).clamp_min(1e-30)
            sm = torch.nn.functional.avg_pool1d(gam.t().unsqueeze(0), 5, stride=1, padding=2,
                                                count_include_pad=False)[0].t()
            sm = sm / sm.sum(1, keepdim=True).clamp_min(1e-30)
            prof[a:b] = sm[a - lo:a - lo + (b - a)]
            del gam, sm
        prof[sep_idx] = 0.0
    torch.cuda.synchronize()
    return {"codes": full, "prof": prof, "n": n, "lengths": lengths, "offsets": offsets}


def make_tables_fn(workload, seed=102, pure_python=False):
    """PFMs (Dirichlet(0.3) rows, pseudocount 0.01) and the counts -> log-odds tables step,
    done with the product's own PFM preprocessing (rnascan_b200.motifs).  pure_python=True (the reference
    arm) builds the same tables with motifs.log_odds' Python arithmetic so that the CUDA library is never
    loaded in that process (the two are bit-identical, tests/test_host_cpu.py)."""
    from rnascan_b200 import motifs, synth

    def log_odds_rows(prob_arr, bgn):
        if not pure_python:
            return motifs.log_odds_table(prob_arr, bgn)
        out = np.empty_like(prob_arr)                   # Python's math.log(p / b, 2), as Biopython's log_odds
        for i in range(prob_arr.shape[0]):
            for a in range(prob_arr.shape[1]):
                pr, b = float(prob_arr[i, a]), float(bgn[a])
                out[i, a] = math.log(pr / b, 2) if pr > 0 else float("-inf")
        return out

    rng = np.random.default_rng(seed)
    pfm_seq = synth.pfm_rows(W_MOTIF, 4, rng)               # columns A,C,G,U
    pfm_str = synth.pfm_rows(W_MOTIF, 7, np.random.default_rng(seed + 1))   # columns B,E,H,L,M,R,T
    rna, chan = "GAUC", "EHTBLRM"                           # alphabet.letters orders
    seq_counts = {l: pfm_seq[:, "ACGU".index(l)].tolist() for l in rna}
    str_counts = {l: pfm_str[:, "BEHLMRT".index(l)].tolist() for l in chan}
    str_pssm = motifs.log_odds(motifs.normalize_counts(str_counts, chan, 0.01), chan,
                               {l: SS_BG[l] for l in chan})
    tq = np.array([str_pssm[l] for l in "BEHLMRT"], np.float64).T.copy()
    seq_prob = motifs.normalize_counts(seq_counts, rna, 0.01)
    str_prob_uniform = motifs.normalize_counts(str_counts, chan, 0.01)

    seq_prob_arr = np.array([seq_prob[l] for l in "ACGU"], np.float64).T.copy()
    str_prob_arr = np.array([str_prob_uniform[l] for l in "BEHLMRT"], np.float64).T.copy()

    def seq_table(counts8):
        # rnascan.py:445-457: p = (count + 1) / (sum(count) + |A|), keys in "GAUC" order; Biopython
        # re-normalises the background (sum in dict order) before log2(p / b).  log_odds_table is
        # the library's host helper, bit-identical to motifs.log_odds (tests/test_host_cpu.py).
        c = {"A": int(counts8[0]), "C": int(counts8[1]), "G": int(counts8[2]), "U": int(counts8[3])}
        total = 4 + sum(c[l] for l in rna)
        bg = {l: (float(c[l]) + 1) / total for l in rna}
        norm = sum(bg.values())
        return log_odds_rows(seq_prob_arr, np.array([bg[l] / norm for l in "ACGU"]))

    def struct_table_computed(counts8):
        c = {l: int(counts8["BEHLMRT".index(l)]) for l in chan}
        total = 7 + sum(c.values())
        bg = {l: (float(c[l]) + 1) / total for l in chan}
        norm = sum(bg.values())
        return log_odds_rows(str_prob_arr, np.array([bg[l] / norm for l in "BEHLMRT"]))

    if workload == "c4":
        return lambda counts8: (seq_table(counts8), tq)
    if workload == "c5":
        # 256 motif pairs, W ~ U{7..12} (same W for the two PFMs of a pair), Dirichlet(0.3) rows
        r5 = np.random.default_rng(seed + 5)
        widths = r5.integers(7, 13, size=N_MOTIFS_C5)
        seq_probs, tqs = [], []
        for w in widths:
            ps = synth.pfm_rows(int(w), 4, r5)
            pq = synth.pfm_rows(int(w), 7, r5)
            seq_probs.append(motifs.normalize_counts({l: ps[:, "ACGU".index(l)].tolist() for l in rna}, rna, 0.01))
            sp = motifs.log_odds(motifs.normalize_counts({l: pq[:, "BEHLMRT".index(l)].tolist() for l in chan},
                                                         chan, 0.01), chan, {l: SS_BG[l] for l in chan})
            tqs.append(np.array([sp[l] for l in "BEHLMRT"], np.float64).T.copy())

        prob_arrays = [np.array([prob[l] for l in "ACGU"], np.float64).T.copy() for prob in seq_probs]
        stacked = np.concatenate(prob_arrays, axis=0)       # all motifs' rows: one helper call per step
        stride = int(max(widths))
        row_of = np.concatenate([m * stride + np.arange(w) for m, w in enumerate(widths)])
        qs = np.zeros((N_MOTIFS_C5, stride, 7), np.float64)
        for m, t in enumerate(tqs):
            qs[m, :t.shape[0]] = t

        def batched(counts8):
            c = {"A": int(counts8[0]), "C": int(counts8[1]), "G": int(counts8[2]), "U": int(counts8[3])}
            total = 4 + sum(c[l] for l in rna)
            bg = {l: (float(c[l]) + 1) / total for l in rna}
            norm = sum(bg.values())                         # Biopython re-normalises the background
            bgn = np.array([bg[l] / norm for l in "ACGU"])
            ss = np.zeros((N_MOTIFS_C5 * stride, 4), np.float64)
            ss[row_of] = log_odds_rows(stacked, bgn)   # == motifs.log_odds per motif, bit for bit
            return ss.reshape(N_MOTIFS_C5, stride, 4), qs
        batched.widths = np.asarray(widths, np.int32)
        batched.lists = lambda counts8: ([t[:w] for t, w in zip(batched(counts8)[0], widths)], tqs)
        return batched
    if workload == "c2":
        fn = lambda counts8: (seq_table(counts8), None)
        fn.seq_prob = seq_prob_arr
        return fn
    return lambda counts8: (None, struct_table_computed(counts8))


# ----------------------------------------------------------------------------- this framework
def run_b200(args):
    import torch
    import torch.distributed as dist
    from rnascan_b200 import device as dev

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    dev.require_cuda()
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=device, timeout=datetime.timedelta(seconds=180))
    if args.n_per_gpu:
        n_main, scaling = args.n_per_gpu, "weak"
    elif args.workload in ("c4", "c5"):
        n_main, scaling = args.n_total // world, "strong"          # BASELINE config 4/5: 1 Gnt in total
    else:
        n_main, scaling = OTHERS_N, "weak"                          # configs 2/3: ~100 Mnt per GPU
    out = measure(args, args.workload, args.steps, (rank, world, local, device), True, n_main)
    out["scaling"] = scaling
    if world == 1 and not args.no_others:
        # the other BASELINE.json configurations, briefly, so that one bench line shows them all
        others = {}
        for wl in ("c2", "c3", "c5", "c4"):
            if wl == args.workload:
                continue
            torch.cuda.empty_cache()
            o = measure(args, wl, 5, (rank, world, local, device), False, OTHERS_N)
            others[wl] = {"workload": o["config"]["workload"], "value": o["value"], "unit": o["unit"],
                          "ms_per_step": o["ms_per_step"], "kernel": o["roofline"]["kernel"],
                          "kernel_ms": o["roofline"]["kernel_ms"], "bound": o["roofline"]["bound"],
                          "achieved": o["roofline"]["achieved"], "roofline_unit": o["roofline"]["unit"],
                          "frac": o["roofline"]["frac"], "symbols": o["config"]["symbols_per_gpu"]}
            for key in ("frac_executed", "achieved_executed"):
                if key in o["roofline"]:
                    others[wl][key] = o["roofline"][key]
            if "e2e" in o:
                others[wl]["e2e"] = o["e2e"]["value"]
            if "motif_positions_per_s" in o:
                others[wl]["motif_positions_per_s_G"] = o["motif_positions_per_s"]
        out["other_workloads"] = others
    if rank == 0:
        if not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_port_baseline(args.workload)
        emit(out)
    if world > 1:
        dist.destroy_process_group()


def measure(args, wl, steps, ctx, full, n_target):
    """Time `steps` steps of workload `wl` on this rank's shard of ~n_target symbols; returns the JSON object."""
    import torch
    import torch.distributed as dist
    from rnascan_b200 import device as dev, _lib
    from rnascan_b200.device import lib, check, _ptr

    rank, world, local, device = ctx
    shard = make_device_shard(n_target, 4000 + rank, wl, device)
    n, codes, prof = shard["n"], shard["codes"], shard["prof"]
    positions = scored_positions(shard["lengths"], W_MOTIF)
    tables = make_tables_fn(wl)
    stream = torch.cuda.current_stream()
    sptr = stream.cuda_stream
    counts = torch.zeros(8, dtype=torch.int64, device=device)
    counts_host = torch.zeros(8, dtype=torch.int64).pin_memory()
    hb = dev.HitBuffers(n, max(1 << 16, n // 256), device)
    # C3: every window's float64 score (the calculate() result) for the device-resident figure; the end-to-end leg
    # brings back what rnascan prints -- round(score, 3) as int32 thousandths, 4 B per position
    dense_out = torch.empty(n, dtype=torch.float64, device=device) if wl == "c3" else None
    milli_out = torch.empty(n, dtype=torch.int32, device=device) if wl == "c3" else None
    absmax = 1.0
    if wl in ("c4", "c5"):
        absmax = dev.ProfileStream.from_device(prof, n).absrow_max()
    if wl == "c5":
        c5_widths = tables.widths
        c5_motif = torch.empty(hb.capacity, dtype=torch.int32, device=device)
        c5_counters = torch.zeros(2 * N_MOTIFS_C5, dtype=torch.int64, device=device)
        c5_bases = torch.zeros(N_MOTIFS_C5 + 1, dtype=torch.int64, device=device)
        hb.work_bytes = int(lib.rs_scan_batched_workspace_bytes(n, N_MOTIFS_C5, int(c5_widths.max()), hb.capacity))
        hb.work = torch.empty(hb.work_bytes, dtype=torch.uint8, device=device)
        check(lib.rs_set_batched_path({"auto": 0, "cuda": 1, "tensor": 2}[args.c5_path]))
    launches = [0]
    c3_milli = [False]
    bgscan = None
    if wl == "c4" and not args.serial_bg:
        # the structure-only candidate scan overlaps histogram -> all-reduce -> host log-odds (side stream);
        # rs_refine_hits_seq applies the sequence PSSM to the candidates (device.BackgroundFusedScan)
        bgscan = dev.BackgroundFusedScan(n, device, capacity=hb.capacity)
        if os.environ.get("RS_BENCH_COUNT_IN_KERNEL") in ("0", "1"):         # experiment switch (tools/gpu_r2p.sh)
            bgscan.count_in_kernel = os.environ["RS_BENCH_COUNT_IN_KERNEL"] == "1"
        hb = bgscan.hb
        tq_fixed = tables(np.zeros(8, np.int64))[1]

    ohscan = None
    if wl == "c2" and not args.serial_bg:
        # the device selects candidates with a provisional table while the host builds the exact one
        ohscan = dev.BackgroundOneHotScan(n, "rna", device, capacity=hb.capacity)
        hb = ohscan.hb

    def all_reduce(t):
        if world > 1:
            dist.all_reduce(t)

    def step(thr=THRESHOLD, job=None):
        job = job or bgscan
        if job is not None:
            job.launch(codes, prof, _lib.RS_F32, W_MOTIF, tq_fixed, lambda c: tables(c)[0], thr, absmax,
                       all_reduce if world > 1 else None)
            launches[0] += job.launches
            return
        if ohscan is not None:
            ohscan.launch(codes, tables.seq_prob, lambda c: tables(c)[0], THRESHOLD, all_reduce if world > 1 else None)
            launches[0] += ohscan.launches
            return
        counts.zero_()
        check((lib.rs_hist if wl == "c3" else lib.rs_hist_rna)(_ptr(codes), n, _ptr(counts), sptr)); launches[0] += 1
        all_reduce(counts)                                  # the path's only collective
        counts_host.copy_(counts, non_blocking=True)
        stream.synchronize()
        ts, tq = tables(counts_host.numpy())
        if wl == "c4":
            check(lib.rs_scan_fused(_ptr(codes), _ptr(prof), _lib.RS_F32, n, ts.ctypes.data, tq.ctypes.data,
                                    W_MOTIF, THRESHOLD, absmax, _lib.RS_MODE_AND, hb.capacity, _ptr(hb.pos),
                                    _ptr(hb.seq), _ptr(hb.struct), _ptr(hb.counters), _ptr(hb.work),
                                    hb.work_bytes, sptr))
            launches[0] += 2                                # scan, ordering
        elif wl == "c5":
            M, stride = tq.shape[0], tq.shape[1]            # ts, tq: (256, stride, 4|7) stacked tables
            check(lib.rs_scan_batched(_ptr(codes), _ptr(prof), _lib.RS_F32, n, M, c5_widths.ctypes.data,
                                      ts.ctypes.data, tq.ctypes.data, stride, THRESHOLD, absmax, _lib.RS_MODE_AND,
                                      hb.capacity, _ptr(c5_motif), _ptr(hb.pos), _ptr(hb.seq), _ptr(hb.struct),
                                      _ptr(c5_counters), _ptr(c5_bases), _ptr(hb.work), hb.work_bytes, sptr))
            launches[0] += 4 * M
        elif wl == "c2":
            check(lib.rs_scan_seq(_ptr(codes), n, ts.ctypes.data, W_MOTIF, THRESHOLD, hb.capacity, _ptr(hb.pos),
                                  _ptr(hb.seq), _ptr(hb.counters), _ptr(hb.work), hb.work_bytes, sptr))
            launches[0] += 3                                # decision table, scan, finish (segment scan + expansion)
        else:
            if c3_milli[0]:
                check(lib.rs_scores_dense_struct_milli(_ptr(codes), n, tq.ctypes.data, W_MOTIF, _ptr(milli_out), sptr))
            else:
                check(lib.rs_scores_dense_struct(_ptr(codes), n, tq.ctypes.data, W_MOTIF, _ptr(dense_out), sptr))
            launches[0] += 1

    def flush(scrub):
        # L2 flush between individually timed steps: 512 MB written, then 256 MB of it read back.  The write alone
        # would leave the 126 MB L2 full of DIRTY lines whose write-back the next step's first kernel pays for
        # (measured: the histogram's 125 MB read took 36 us behind it instead of 22 us); after the read pass L2 holds
        # clean lines of unrelated data -- the step starts cold and is billed only its own traffic.
        scrub.fill_(1)
        scrub[: 256 << 20].view(torch.int64).sum()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0 and full:
        sampler.start()                  # covers warm-up + timed region + e2e (all under load)
    for _ in range(max(args.warmup, 3)):
        step()
    # settle: a timed region of 20 sub-millisecond steps right after a cold start is at the mercy of clock ramps and
    # of the collective's first launches; keep stepping (untimed) for about 0.3 s.  The count is a function of the
    # nominal shard size only, so every rank runs the same number of steps (each holds an all-reduce).
    settle = 0
    if full:
        nominal = args.n_per_gpu or (args.n_total // world if wl in ("c4", "c5") else OTHERS_N)
        per_step_s = {"c4": 4.7e-12, "c5": 56e-12, "c2": 1.0e-12, "c3": 3.1e-12}[wl] * nominal
        settle = int(min(1000, max(0, 0.3 / max(per_step_s, 1e-6))))
        for _ in range(settle):
            step()
    # a garbage-collector pause on ONE rank is a visible fraction of a 12 ms timed region (20 sub-millisecond steps,
    # max over ranks): collect now, keep the collector off until the region is over
    import gc
    gc.collect()
    gc.disable()
    barrier()
    launches[0] = 0
    per_step = N_MOTIFS_C5 if wl == "c5" else 1      # upper bound on profiled launches per step
    check(lib.rs_prof_begin(max(steps, 1) * per_step))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    input_bytes = n * (29 if wl in ("c4", "c5") else 1)
    flush_l2 = input_bytes < 512 * 1024 * 1024       # inputs that could sit in the 126 MB L2: flush between steps
    if flush_l2:
        # every step timed on its own event pair; between steps (untimed) a 512 MB buffer is overwritten
        scrub = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=device)
        pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in pairs:
            flush(scrub)
            a.record(stream)
            step()
            b.record(stream)
        barrier()
        ms_total = sum(a.elapsed_time(b) for a, b in pairs)
        del scrub
    else:
        e0.record(stream)
        for _ in range(steps):
            step()
        e1.record(stream)
        barrier()
        ms_total = e0.elapsed_time(e1)
    gc.enable()
    kms = np.zeros(max(steps, 1) * per_step, np.float32)
    nrec = np.zeros(1, np.int32)
    check(lib.rs_prof_end(kms.ctypes.data, len(kms), nrec.ctypes.data))
    kernel_ms = float(kms[:int(nrec[0])].sum()) / steps if nrec[0] else float("nan")
    n_launch = launches[0]
    hits = int(hb.counters[0].item()) if wl in ("c4", "c2") else None
    rejected = None
    if ohscan is not None:
        # candidates the exact table turned down (position -1, dropped by results()): none at N = 1, a few
        # per cent at N > 1 where the decision pass starts from the shard's own counts with 0.05 of slack
        rejected = int(hb.counters[1].item())
        hits -= rejected
        if ohscan.rescanned:
            raise SystemExit("shard composition outside the slack: the timed steps re-scanned (not the overlapped path)")
    if bgscan is not None and int(hb.cand_counters[0].item()) > hb.capacity:
        raise SystemExit("candidate buffer overflowed: %d > %d" % (int(hb.cand_counters[0].item()), hb.capacity))
    if wl == "c5":
        hits = int(c5_bases[-1].item())
    if full and rank == 0 and args.dump_outputs:
        # the last timed step's results as a caller of the path receives them, before the legs below reuse the buffers
        found = None if wl == "c3" else (int(c5_bases[-1].item()) if wl == "c5" else int(hb.counters[0].item()))
        if found is not None and found > hb.capacity:
            raise SystemExit("hit buffer overflowed: %d > %d" % (found, hb.capacity))
        if bgscan is not None:
            pos, sq, sb = bgscan.results()
            entries, counts8 = {"position": pos, "seq_score": sq, "struct_score": sb}, bgscan.counts_host.numpy()
        elif ohscan is not None:
            pos, sq, _ = ohscan.results()
            entries, counts8 = {"position": pos, "seq_score": sq}, ohscan.counts_host.numpy()[:8]
        elif wl == "c3":
            entries, counts8 = {"score": dense_out[:max(0, n - W_MOTIF + 1)]}, counts_host.numpy()
        else:
            entries, counts8 = {"position": hb.pos[:found], "seq_score": hb.seq[:found]}, counts_host.numpy()
            if wl != "c2":
                entries["struct_score"] = hb.struct[:found]
            if wl == "c5":
                entries["motif"] = c5_motif[:found]
        fixed = {"background_counts": counts8}
        if wl == "c5":
            fixed["motif_bases"] = c5_bases
        dump_outputs(args.dump_outputs, entries, fixed)

    # ---- optional device timeline of a few more steps (CUPTI through torch.profiler; never part of a bench value)
    if full and args.trace and rank == 0:
        from torch.profiler import profile, ProfilerActivity
        scrub = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=device) if flush_l2 else None
        with profile(activities=[ProfilerActivity.CUDA]) as prof_run:
            for _ in range(8):
                if scrub is not None:
                    flush(scrub)
                step()
            torch.cuda.synchronize()
        del scrub
        evs = sorted(((e.time_range.start, e.time_range.end, e.name) for e in prof_run.events()
                      if e.device_type == torch.autograd.DeviceType.CUDA), key=lambda t: t[0])
        t_first = evs[0][0] if evs else 0
        with open(args.trace, "w") as fh:
            json.dump({"workload": wl, "unit": "us", "note": "kernel / memset / memcpy intervals on the device, 8 steps, "
                       "CUPTI via torch.profiler; gap_before = idle time since the previous interval ended",
                       "events": [{"start": a - t_first, "dur": b - a, "gap_before": (a - evs[k - 1][1]) if k else 0.0,
                                   "name": nm[:90]} for k, (a, b, nm) in enumerate(evs)]}, fh, indent=0)

    # ---- sustained: keep stepping for a couple of seconds (power / clock regime of a long job)
    sustained = None
    if full and not flush_l2 and args.sustain_seconds > 0:
        # every rank must run the SAME number of steps (each step holds one all-reduce): agree on the slowest rank's time
        agreed = torch.tensor([ms_total], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(agreed, op=dist.ReduceOp.MAX)
        k_s = max(steps, int(math.ceil(args.sustain_seconds * 1e3 / max(float(agreed.item()) / steps, 1e-3))))
        e0.record(stream)
        for _ in range(k_s):
            step()
        e1.record(stream)
        barrier()
        sustained = {"steps": k_s, "ms": e0.elapsed_time(e1)}

    # ---- threshold sweep (c4): what the scan costs when more windows pass the filter
    sweep = None
    if full and wl == "c4" and bgscan is not None and not args.no_sweep:
        sweep = []
        job = dev.BackgroundFusedScan(n, device, capacity=max(1 << 16, n // 16))
        for thr in (6.0, 2.0, 0.0):
            for _ in range(2):
                step(thr, job)
            barrier()
            e0.record(stream)
            for _ in range(3):
                step(thr, job)
            e1.record(stream)
            barrier()
            cand, resc = (int(v) for v in job.hb.cand_counters.cpu().numpy())
            sweep.append({"minscore": thr, "ms_per_step": e0.elapsed_time(e1) / 3, "hits": int(job.hb.counters[0].item()),
                          "structure_candidates": cand, "windows_rescored_fp64": resc,
                          "overflow": cand > job.hb.capacity})
        del job
        torch.cuda.empty_cache()

    # ---- end to end: host buffers -> device -> results back on the host, every step
    e2e = None
    e2e_extra = {}
    k2 = max(2, min(steps, 5))
    h_codes = torch.empty(codes.shape, dtype=torch.uint8).pin_memory()
    h_codes.copy_(codes)
    if args.no_e2e:
        pass
    elif wl == "c4":
        e2e, e2e_extra = e2e_c4(args, dev, shard, h_codes, tables, absmax, hits, all_reduce, barrier, (rank, world, device),
                                full)
    else:
        # plain copy-in / step / copy-out through the same C-ABI calls
        h_prof = None
        if wl == "c5":
            h_prof = torch.empty(prof.shape, dtype=torch.float32).pin_memory()
            h_prof.copy_(prof)
        h_out = torch.empty(milli_out.shape, dtype=milli_out.dtype).pin_memory() if wl == "c3" else None
        c3_milli[0] = wl == "c3"
        h_pos = torch.empty(hb.capacity, dtype=torch.int64).pin_memory()
        h_sc = torch.empty(hb.capacity, dtype=torch.float64).pin_memory()
        io = [0, 0]

        def e2e_step():
            codes.copy_(h_codes, non_blocking=True); io[0] = codes.numel()
            if h_prof is not None:
                prof.copy_(h_prof, non_blocking=True); io[0] += prof.numel() * 4
            step()
            if wl == "c3":
                h_out.copy_(milli_out, non_blocking=True); io[1] = milli_out.numel() * 4
                stream.synchronize()
            else:
                stream.synchronize()
                found = int(c5_bases[-1].item()) if wl == "c5" else int(hb.counters[0].item())
                k = min(found, hb.capacity)
                h_pos[:k].copy_(hb.pos[:k], non_blocking=True)
                h_sc[:k].copy_((hb.struct if wl == "c5" else hb.seq)[:k], non_blocking=True)
                stream.synchronize()
                io[1] = 64 + 16 + k * (20 if wl == "c5" else 12)
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(k2):
            e2e_step()
        e1.record(stream)
        torch.cuda.synchronize()
        ms_e2e = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3) / k2
        e2e = {"ms": ms_e2e, "h2d": io[0], "d2h": io[1],
               "api": "pinned host streams -> device -> C-ABI step -> pinned host results"}
        del h_prof, h_out
    del h_codes
    clocks = sampler.stop() if (rank == 0 and full) else None

    # ---- max over ranks, totals
    stats = torch.tensor([ms_total, kernel_ms, e2e["ms"] if e2e else 0.0], device=device, dtype=torch.float64)
    tot = torch.tensor([positions, n], device=device, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot)
    ms_total, kernel_ms, ms_e2e = (float(v) for v in stats.cpu())
    all_positions, all_n = (int(v) for v in tot.cpu())
    ms_step = ms_total / steps
    peak, peak_src = measured_peaks()
    achieved = ALGO_BYTES[wl] * positions / (kernel_ms * 1e-3) / 1e9
    out = {
        "metric": "scored positions/sec", "value": all_positions / (ms_step * 1e-3) / 1e9, "unit": "Gpos/s",
        "n_gpus": world, "steps": steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,      # run_b200 sets `scaling`
        "dtype": "f32 filter + f64 exact re-score (sequence: f64 accumulate -> f32)" if wl == "c4" else
                 ("f64 accumulate -> f32" if wl == "c2" else ("f64" if wl == "c3" else
                                                              "f32 filter + f64 exact re-score, per motif")),
        "data": "synthetic (SURVEY.md 8d shapes; generated on device, seed 4000+rank)",
        "config": {"workload": {"c4": "C4 seq PSSM + averaged 7-channel structure profile, fused AND scan",
                                "c2": "C2 sequence-only scan", "c3": "C3 one-hot structure scan, every position: dense f64 scores on the device; e2e returns round(x, 3) as int32 thousandths",
                                "c5": "C5 batched %d motif pairs (W 7-12), seq + averaged structure" % N_MOTIFS_C5}[wl],
                   "symbols_per_gpu": n, "records_per_gpu": int(len(shard["lengths"])),
                   "scored_positions_total": all_positions, "W": W_MOTIF, "minscore": THRESHOLD,
                   "background": (("computed every step: the structure-only candidate scan counts the letters itself "
                                   "(rs_scan_fused_candidates_counting) -> all-reduce(int64[8]) -> host log-odds; the sequence "
                                   "PSSM is applied to the candidates afterwards (rs_scan_fused_resolve)")
                                  if (bgscan is not None and bgscan.count_in_kernel) else
                                  "computed every step: histogram -> all-reduce(int64[8]) -> host log-odds on a side "
                                  "stream, overlapped with the structure-only candidate scan; the sequence PSSM is "
                                  "applied to the candidates afterwards (rs_scan_fused_resolve)") if bgscan is not None else
                                 ("computed every step: histogram -> all-reduce(int64[8]); the device scans with a provisional "
                                  "log-odds table while the counts go to the host, the exact host table decides and scores "
                                  "the candidates (rs_scan_onehot_begin/_finish)" if ohscan is not None else
                                  "computed: histogram -> all-reduce(int64[8]) -> host log-odds, every step"),
                   "l2_policy": ("L2 flushed between timed steps (512 MB overwrite, then 256 MB read back so that no dirty lines of the flush remain; untimed); inputs %.2f GB per GPU"
                                 if flush_l2 else "inputs (%.2f GB per GPU) exceed the 126 MB L2") % (input_bytes / 1e9),
                   "parallelism": "shard%d (contiguous record ranges per GPU, no data-path collective)" % world,
                   "untimed_steps_before_the_timed_region": max(args.warmup, 3) + settle},
        "gpu_launches": n_launch,
        "roofline": {"bound": "hbm", "kernel": {"c4": "fused_filter_kernel<7>", "c2": "kmer_scan_kernel<7>",
                                               "c3": "dense_w_kernel<7,7,0>",
                                               "c5": "fused_filter_kernel<W> x %d motifs" % N_MOTIFS_C5}[wl],
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "peak_source": peak_src, "algorithmic_bytes_per_position": ALGO_BYTES[wl],
                     "kernel_ms": kernel_ms, "kernel_share_of_step": kernel_ms / ms_step,
                     "traffic": recorded_traffic(wl, n)[0], "traffic_source": recorded_traffic(wl, n)[1],
                     "note": "peak = a device-to-device COPY (half reads, half writes); a read-only stream like this "
                             "kernel's can run a few per cent above it"},
        "clocks": clocks,
    }
    if hits is not None:
        out["hits_rank0"] = hits
    if rejected is not None:
        out["rejected_candidates_rank0"] = rejected
    if wl == "c5":
        out["motif_positions_per_s"] = out["value"] * N_MOTIFS_C5
        took = int(lib.rs_last_batched_path())
        out["config"]["c5_path"] = {1: "cuda-core loop (one fused scan per motif)", 2: "tcgen05 GEMM filter + exact re-score"}[took]
        if took == 2:
            # 2 * 96 (K, padded window x 8 channels) * 256 motifs flop per position on the tensor cores
            flops = 2.0 * 96 * 256 * positions
            tf = flops / (kernel_ms * 1e-3) / 1e12
            try:
                with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as fh:
                    tpeak = float(json.load(fh)["bf16_tflops_sustained"])
                src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
            except Exception:
                tpeak, src = 1400.0, "fallback (B200_PROFILING.md ~1.4 PFLOP/s sustained)"
            # SURVEY.md 8(d)'s ALGORITHMIC figure: 2 * 7 channels * W_m * 256 motifs (no padding of W to 12, no
            # eighth channel); `achieved`/`frac` below use it -- the padded figure the MMAs execute is given beside it
            w_mean = float(np.mean(c5_widths))
            flops_alg = 2.0 * 7 * w_mean * N_MOTIFS_C5 * positions
            tf_alg = flops_alg / (kernel_ms * 1e-3) / 1e12
            out["roofline"] = {"bound": "tensor", "kernel": "batched_tc_kernel", "achieved": tf_alg, "peak": tpeak,
                               "unit": "TFLOP/s", "frac": tf_alg / tpeak, "peak_source": src,
                               "flop_per_position_algorithmic": 2.0 * 7 * w_mean * N_MOTIFS_C5,
                               "achieved_executed": tf, "frac_executed": tf / tpeak,
                               "flop_per_position_executed": 2.0 * 96 * 256, "kernel_ms": kernel_ms,
                               "kernel_share_of_step": kernel_ms / ms_step, "traffic": recorded_traffic(wl, n)[0],
                               "traffic_source": recorded_traffic(wl, n)[1],
                               "hbm_GBps_algorithmic": 29.0 * positions / (kernel_ms * 1e-3) / 1e9}
        else:
            out["roofline"]["note"] = ("CUDA-core path re-reads the streams once per motif: physical traffic is %d x "
                                       "the algorithmic 29 B/position" % N_MOTIFS_C5)
    if e2e:
        out["e2e"] = {"value": all_positions / (ms_e2e * 1e-3) / 1e9, "unit": "Gpos/s",
                      "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": e2e["d2h"],
                      "ms_per_step": ms_e2e,
                      "link_GBps": (e2e["h2d"] + e2e["d2h"]) / (ms_e2e * 1e-3) / 1e9,
                      "api": e2e["api"]}
        for key in ("form", "bytes_per_position", "guard_band_score_units"):
            if key in e2e:
                out["e2e"][key] = e2e[key]
        for key in ("candidates", "structure_candidates", "filter_pass", "launches", "host_prep_s_untimed", "hits"):
            if key in e2e:
                out["e2e"][key + "_rank0"] = e2e[key]
        out.update(e2e_extra)
    if sustained is not None:
        st = torch.tensor([sustained["ms"]], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(st, op=dist.ReduceOp.MAX)
        ms_s = float(st.item()) / sustained["steps"]
        out["sustained"] = {"steps": sustained["steps"], "seconds": float(st.item()) * 1e-3, "ms_per_step": ms_s,
                            "value": all_positions / (ms_s * 1e-3) / 1e9, "unit": "Gpos/s"}
    if sweep is not None:
        for row in sweep:
            row["value_rank0"] = positions / (row["ms_per_step"] * 1e-3) / 1e9
        out["threshold_sweep_rank0"] = sweep
    out["consistency_timed_region_s"] = ms_total * 1e-3
    if wl == "c5":
        check(lib.rs_set_batched_path(0))
    return out


def e2e_c4(args, dev, shard, h_codes, tables, absmax, hits_dev, all_reduce, barrier, ctx, full):
    """End-to-end legs of config 4: HOST buffers in, host hit arrays out, copies inside the timed region.

    e2e       the rows as a profile pack holds them (rnascan_b200/pack.py): 8-byte quantised filter rows (symbol
              included) in pinned memory + the exact rows in ordinary host memory; device.HostProfileScanner sends
              only the filter form over the link (8 B/position), counts the background in the same pass, gathers the
              exact rows of the candidates on the host and resolves them on the device -- same hits as the
              device-resident scan (checked).
    e2e_f32   round 1's pipeline for comparison (float32 rows over the link, 29 B/position), on a prefix.
    e2e_api   the public scan API: rnascan_b200.rnascan.scan_main(<directory with a pack>) on a prefix."""
    import torch
    rank, world, device = ctx
    n, prof, lengths, offsets = shard["n"], shard["prof"], shard["lengths"], shard["offsets"]
    stream = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k2 = max(2, min(args.steps, 3))
    extra = {}

    # the parsed input on the host: exact rows (float32-representable by construction, SURVEY.md 8d) ...
    t0 = time.perf_counter()
    rows_host = np.empty((n, 7), np.float32)
    bounce = torch.empty((1 << 23, 7), dtype=torch.float32).pin_memory()
    for a in range(0, n, 1 << 23):
        b = min(n, a + (1 << 23))
        bounce[:b - a].copy_(prof[a:b])
        rows_host[a:b] = bounce[:b - a].numpy()
    del bounce
    codes_np = h_codes.numpy()[:n]
    # ... and their filter form (what `rnascan --pack` leaves on disk), built by the product's host quantiser
    hp = dev.HostProfile(rows_host)
    tq = tables(np.zeros(8, np.int64))[1]
    # which quantised form: 4 bytes per position when its guard band (here ~2 score units) leaves the threshold
    # selective, else 8 bytes (guard ~0.2); `--e2e-form` forces one
    guard4 = dev.q4_guard(tq, max(hp.stats()[3], 1e-300))
    form = args.e2e_form if args.e2e_form != "auto" else ("q4" if guard4 <= 0.4 * THRESHOLD else "q8")
    width = 4 if form == "q4" else 8
    q8 = torch.empty((n, width), dtype=torch.uint8).pin_memory()
    ok = hp.make_q4(codes_np, out=q8.numpy()) if form == "q4" else hp.make_q8(codes_np, out=q8.numpy())
    if not ok:
        raise SystemExit("synthetic rows do not fit the quantised form")
    prep_s = time.perf_counter() - t0
    seq_fn = lambda c: tables(c)[0]
    # 128 MB per copy whatever the form (16 M rows of 8 bytes, 32 M rows of 4): the link runs a few per cent faster on
    # larger transfers (measured with 4-byte rows: 51.5 / 53.1 / 53.9 GB/s at 32 / 64 / 128 MB per copy)
    chunk_rows = int(os.environ.get("RS_BENCH_E2E_CHUNK_ROWS", (128 << 20) // width))
    sc = dev.HostProfileScanner(n, W_MOTIF, form, chunk_rows=chunk_rows, device=device)
    ar = all_reduce if world > 1 else None

    def run():
        return sc.run(None, q8, rows_host, tq, seq_fn, THRESHOLD, absmax, q8_scale=hp.q8_scale, all_reduce=ar)
    res = run()
    barrier()
    t0 = time.perf_counter()
    e0.record(stream)
    for _ in range(k2):
        res = run()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3) / k2
    if hits_dev is not None and len(res[0]) != hits_dev:
        raise SystemExit("e2e hit count %d != device-resident hit count %d" % (len(res[0]), hits_dev))
    e2e = {"ms": ms, "h2d": sc.h2d_bytes, "d2h": sc.d2h_bytes, "hits": int(len(res[0])),
           "api": "rnascan_b200.device.HostProfileScanner.run: pinned %d-byte quantised rows (7 channels + symbol) -> "
                  "device filter (+ background counts)%s -> candidate positions -> host gather of the exact rows -> "
                  "device resolve -> host hit arrays"
                  % (width, " -> sequence table applied to the candidates' packed symbols on the device" if form == "q4" else ""),
           "form": form, "bytes_per_position": width, "guard_band_score_units": guard4 if form == "q4" else None,
           "candidates": sc.n_candidates, "structure_candidates": sc.n_struct_candidates or sc.n_candidates,
           "filter_pass": sc.n_filter_pass, "launches": sc.launches, "host_prep_s_untimed": prep_s}
    del sc, q8
    if not full:
        return e2e, extra

    # ---- round 1's float32 pipeline on a prefix, for comparison
    n_pre = min(n, OTHERS_N)
    ends = offsets + lengths
    k_full = int(np.searchsorted(ends, n_pre, side="right"))
    pos_pre = int(np.maximum(lengths[:k_full] - W_MOTIF + 1, 0).sum())
    if k_full < len(lengths):
        pos_pre += max(0, n_pre - int(offsets[k_full]) - W_MOTIF + 1) if offsets[k_full] < n_pre else 0
    h_prof = torch.empty((n_pre, 7), dtype=torch.float32).pin_memory()
    h_prof.copy_(prof[:n_pre])
    torch.cuda.synchronize()
    pipe = dev.HostFusedScanner(n_pre, W_MOTIF, device=device)
    for _ in range(2):
        pipe.run(h_codes, h_prof, tables, THRESHOLD, absrow_max=absmax)
    barrier()
    t0 = time.perf_counter()
    for _ in range(k2):
        pipe.run(h_codes, h_prof, tables, THRESHOLD, absrow_max=absmax)
    torch.cuda.synchronize()
    ms32 = (time.perf_counter() - t0) * 1e3 / k2
    extra["e2e_f32"] = {"value": pos_pre / (ms32 * 1e-3) / 1e9, "unit": "Gpos/s", "symbols": n_pre,
                        "h2d_bytes_per_step": pipe.h2d_bytes, "d2h_bytes_per_step": pipe.d2h_bytes, "ms_per_step": ms32,
                        "api": "rnascan_b200.device.HostFusedScanner.run (float32 rows over the link, round 1's e2e)"}
    del h_prof, pipe

    # ---- the public API on a directory that holds a profile pack
    if world == 1 and not args.no_api:
        try:
            extra["e2e_api"] = e2e_api(dev, rows_host, lengths, offsets, tq, prof, device)
        except Exception as exc:                       # reported, never fatal for the bench line
            extra["e2e_api"] = {"error": "%s: %s" % (type(exc).__name__, exc)}
    return e2e, extra


def e2e_api(dev, rows_host, lengths, offsets, tq, prof, device, target_rows=32_000_000):
    """rnascan_b200.rnascan.scan_main(directory) -- the reference's own entry point (rnascan.py:335-413) -- on a
    directory whose averaged profiles are present as a pack (what a first `rnascan --pack` run leaves behind):
    map the pack, send the quantised rows, gather + resolve, build the result frame.  Hits are checked against
    the device-resident structure-only scan of the same rows."""
    import argparse as ap
    import shutil
    import tempfile
    import torch
    from rnascan_b200 import pack, rnascan as ms
    from rnascan_b200.BioAddons.Alphabet import ContextualSecondaryStructure
    from rnascan_b200.BioAddons.motifs import matrix
    k = max(1, int(np.searchsorted(offsets + lengths, target_rows, side="right")))
    k = min(k, len(lengths))
    m = int(offsets[k - 1] + lengths[k - 1] + 1)
    rows64 = rows_host[:m].astype(np.float64)
    hp = dev.HostProfile(rows64)
    sep = np.zeros(m, np.uint8)
    sep[offsets[:k] + lengths[:k]] = 0xFF
    if not (hp.make_q8(sep) and hp.make_q4(sep)):
        raise RuntimeError("rows do not fit the quantised form")
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    tmp = tempfile.mkdtemp(prefix="rnascan_b200_bench_", dir=base)
    try:
        t0 = time.perf_counter()
        pack.write(tmp, None, rows64, lengths[:k], hp.stats(), hp.q8, hp.q8_scale,
                   names=["structure.rec%d.txt" % i for i in range(k)], q4=hp.q4)
        write_s = time.perf_counter() - t0
        del rows64, hp
        alphabet = ContextualSecondaryStructure()
        pssm = {"bench_struct": matrix.ExtendedPositionSpecificScoringMatrix(
            alphabet, {l: tq[:, "BEHLMRT".index(l)].tolist() for l in alphabet.letters})}
        ns = ap.Namespace(minscore=THRESHOLD, debug=False, pack=False)
        positions = int(np.maximum(lengths[:k] - W_MOTIF + 1, 0).sum())
        t0 = time.perf_counter()
        frame = ms.scan_main(tmp, pssm, alphabet, None, ns)
        first_s = time.perf_counter() - t0
        times = []
        for _ in range(4):
            t0 = time.perf_counter()
            frame = ms.scan_main(tmp, pssm, alphabet, None, ns)
            times.append(time.perf_counter() - t0)
        # the same rows, device-resident, structure only
        st = dev.SymbolStream.__new__(dev.SymbolStream)
        codes = torch.zeros(dev.padded_count(m), dtype=torch.uint8, device=device)
        codes[torch.from_numpy(offsets[:k] + lengths[:k]).to(device)] = 0xFF
        codes[m:] = 0xFF
        st.codes, st.n, st.kind = codes, m, None
        st.offsets, st.lengths = offsets[:k], lengths[:k]
        pf = dev.ProfileStream.from_device(prof, m)
        pos, _, sc = dev.scan_fused(st, pf, None, tq, THRESHOLD)
        same = (len(frame) == len(pos) and
                np.array_equal(np.asarray(frame["LogOdds"], np.float64).view(np.uint64), sc.view(np.uint64)))
        if not same:
            raise RuntimeError("scan_main over the pack found %d hits, the device-resident scan %d (or scores differ)"
                               % (len(frame), len(pos)))
        sec = float(np.median(times))
        return {"value": positions / sec / 1e9, "unit": "Gpos/s", "ms_per_call": sec * 1e3, "symbols": m, "records": k,
                "calls_ms": [round(first_s * 1e3, 2)] + [round(t * 1e3, 2) for t in times],
                "calls_note": "value = median of calls 2..5; call 1 maps the pack (page faults) and allocates, call 2 "
                              "copies the quantised section into page-locked memory once (pack.page_locked), later calls ship chunks straight from it",
                "hits": int(len(frame)), "pack_bytes": os.path.getsize(pack.pack_path(tmp)), "pack_write_s": write_s,
                "pack_on": "tmpfs" if base else "disk",
                "api": "rnascan_b200.rnascan.scan_main(<directory holding rnascan_b200.pack>, pssm, alphabet, None, args): "
                       "map the pack -> quantised rows to the device -> filter -> gather exact float64 rows -> resolve "
                       "-> result DataFrame; identical hits and scores to the device-resident scan (checked)"}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


# ----------------------------------------------------------------------------- CPU legs
def host_sample(n_symbols, workload, seed=4999, min_records=1):
    """A bounded host-side sample of the same synthetic workload (numpy generator)."""
    from rnascan_b200 import synth
    rng = np.random.default_rng(seed)
    n_records = max(1, min_records, int(round(n_symbols / 3334.0)))
    lengths = synth.record_lengths(n_symbols - n_records, n_records, rng)
    if workload == "c3":
        codes, offsets = synth.struct_codes(lengths, rng)
        return lengths, offsets, codes, None
    codes, offsets = synth.rna_codes(lengths, rng)
    rows = synth.profile_rows(len(codes), rng, lengths=lengths) if workload in ("c4", "c5") else None
    return lengths, offsets, codes, rows


def cpu_port_baseline(workload, n_symbols=None):
    """The C oracle (oracle/pwm_oracle.c, a port of the reference's loops) over whole records
    with all host threads: the most the reference's C kernel could do if it were driven per
    record instead of per window.  Reported, not the target."""
    from oracle import oracle as orc
    from rnascan_b200 import synth
    L = orc.lib()
    cores = int(L.orc_get_threads())
    if n_symbols is None:
        n_symbols = 1_000_000 if workload == "c5" else 16_000_000
    lengths, offsets, codes, rows = host_sample(n_symbols, "c4" if workload == "c5" else workload)
    positions = scored_positions(lengths, W_MOTIF)
    tables = make_tables_fn(workload)

    def one_pass():
        if workload == "c3":
            counts = np.array([(codes == k).sum() for k in range(8)], np.int64)
            _, tq = tables(counts)
            sc = orc.alpha_scores(synth.to_text(codes, "struct"), tq, "BEHLMRT")
            nh = int(np.isfinite(sc).sum())
        else:
            text = synth.to_text(codes, "rna")
            counts = np.zeros(8, np.int64)
            cnt = np.zeros(4, np.int64)
            L.orc_count_letters(text, len(text), b"ACGU", 4, cnt.ctypes.data)
            counts[:4] = cnt
            ts, tq = tables.lists(counts) if workload == "c5" else tables(counts)
            if workload == "c5":
                nh = 0
                for ts_m, tq_m in zip(ts, tq):
                    a = orc.seq_scores(text, ts_m, threads=True)
                    b = orc.profile_scores(rows, tq_m)
                    nh += int(((a.astype(np.float64) > THRESHOLD) & (b > THRESHOLD)).sum())
            else:
                a = orc.seq_scores(text, ts, threads=True)
                keep = a.astype(np.float64) > THRESHOLD
                if workload == "c4":
                    b = orc.profile_scores(rows, tq)
                    keep &= b > THRESHOLD
                nh = int(keep.sum())
        return nh

    # about 10-30 s of CPU work: repeat the pass over the sample until ~1.5 s of wall time on all host threads
    t0 = time.perf_counter()
    nh = one_pass()
    first = time.perf_counter() - t0
    passes = 1 + int(min(40, max(0, math.ceil(1.5 / max(first, 1e-3)) - 1)))
    for _ in range(passes - 1):
        one_pass()
    dt = time.perf_counter() - t0
    return {"value": positions * passes / dt / 1e9, "unit": "Gpos/s", "cores": cores, "kind": "port",
            "sample": "%d symbols (%d scored positions) of the same synthetic workload x %d passes, whole-record C "
                      "loops on %d threads, %.2f s of wall time = %.0f s of CPU work, %d hits per pass"
                      % (len(codes), positions, passes, cores, dt, dt * cores, nh)}


def run_reference(args):
    """The reference's own CPU path, driven the way the reference drives it (oracle/ref_driver.py):
    one _pwm.calculate call per window from Biopython-style search(), the pandas .iloc loop of
    scan_averaged_structure, multiprocessing.Pool over records."""
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    from oracle import ref_driver
    wl = args.workload
    cores = os.cpu_count() or 1
    tables = make_tables_fn(wl, pure_python=True)       # the CUDA library is never loaded in this process
    target_s = float(os.environ.get("RNASCAN_REF_STEP_SECONDS", "5"))
    # size the per-step sample from a calibration pass through the SAME Pool fan-out (load imbalance
    # between records included), so that one step takes about target_s seconds on this box
    rate1 = ref_driver.calibrate(wl, tables, W_MOTIF, THRESHOLD)          # windows/s on one core
    n_cal = int(max(300 if wl == "c5" else 2000, min(5_000_000, rate1 * cores * 1.0)))
    lengths, offsets, codes, rows = host_sample(n_cal, wl, seed=5998, min_records=8 * cores)
    t0 = time.perf_counter()
    ref_driver.run_step(wl, lengths, offsets, codes, rows, tables, W_MOTIF, THRESHOLD, cores)
    rate = scored_positions(lengths, W_MOTIF) / max(time.perf_counter() - t0, 1e-6)      # windows/s, all cores
    n_symbols = int(max(300 if wl == "c5" else 2000, min(50_000_000, rate * target_s)))
    # the reference parallelises over records only: keep >= 8 records per core in the sample
    lengths, offsets, codes, rows = host_sample(n_symbols, wl, seed=5999, min_records=8 * cores)
    positions = scored_positions(lengths, W_MOTIF)
    times = []
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        nh = ref_driver.run_step(wl, lengths, offsets, codes, rows, tables, W_MOTIF, THRESHOLD, cores)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    ms_step = 1e3 * sum(times) / len(times)
    value = positions / (ms_step * 1e-3) / 1e9
    sample = ("%d symbols / %d records / %d scored positions per step of the same synthetic workload; "
              "%s; Pool(%d); %d hits" % (len(codes), len(lengths), positions, ref_driver.describe(wl), cores, nh))
    out = {"impl": "reference", "metric": "scored positions/sec", "value": value, "unit": "Gpos/s",
           "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
           "higher_is_better": True,
           "scaling": "strong" if (not args.n_per_gpu and wl in ("c4", "c5")) else "weak",     # as the b200 arm reports it
           "vs_baseline": None,
           "dtype": "f64 accumulate -> f32 (sequence), f64 (structure)", "data": "synthetic (bounded sample)",
           "config": {"workload": {"c4": "C4 seq PSSM + averaged 7-channel structure profile",
                                   "c2": "C2 sequence-only scan", "c3": "C3 one-hot structure scan",
                                   "c5": "C5 batched 256 motif pairs, one reference run per pair"}[wl],
                      "W": W_MOTIF, "minscore": THRESHOLD, "sample_symbols": len(codes)},
           "gpu_launches": 0,
           "cpu_baseline": {"value": value, "unit": "Gpos/s", "cores": cores,
                            "kind": ref_driver.kind(), "sample": sample},
           "e2e": {"value": value, "unit": "Gpos/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


_REAL_STDOUT = None


def emit(obj):
    """The ONE JSON line of the contract, on the process's original stdout."""
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


def main():
    # native libraries (NCCL's version banner, for one) write to fd 1: keep stdout for the JSON line only
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4", choices=["c4", "c2", "c3", "c5"])
    ap.add_argument("--n-total", type=int, default=1_000_000_000, dest="n_total",
                    help="symbols of the whole job, split evenly over the GPUs (config 4: 1 Gnt)")
    ap.add_argument("--n-per-gpu", type=int, default=0, dest="n_per_gpu",
                    help="fix the per-GPU share instead (weak scaling)")
    ap.add_argument("--sustain-seconds", type=float, default=2.0, dest="sustain_seconds",
                    help="after the K timed steps, keep stepping for this long and report it as `sustained`")
    ap.add_argument("--trace", default="", help="also write a device timeline of 8 extra steps to this JSON file")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", dest="no_e2e",
                    help="skip the host-buffer end-to-end leg (e.g. for shards too large to pin on the host)")
    ap.add_argument("--serial-bg", action="store_true", dest="serial_bg",
                    help="c4/c2: histogram -> host tables -> scan, strictly in sequence (no overlap)")
    ap.add_argument("--e2e-form", default="auto", choices=["auto", "q4", "q8"], dest="e2e_form",
                    help="quantised row form of the end-to-end leg (auto: 4 bytes when its guard band allows)")
    ap.add_argument("--no-sweep", action="store_true", dest="no_sweep", help="skip the threshold sweep (c4)")
    ap.add_argument("--no-api", action="store_true", dest="no_api", help="skip the scan_main(pack directory) leg")
    ap.add_argument("--no-others", action="store_true", dest="no_others",
                    help="skip the brief runs of the other configurations (other_workloads)")
    ap.add_argument("--c5-path", default="auto", choices=["auto", "cuda", "tensor"], dest="c5_path")
    ap.add_argument("--dump-outputs", default="", metavar="DIR", dest="dump_outputs",
                    help="after the timed steps, write what the last one computed on rank 0's shard as DIR/<name>.npy "
                         "(float32 / float64, at most 64 MB: larger per-hit or per-window outputs are a seeded sample)")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
