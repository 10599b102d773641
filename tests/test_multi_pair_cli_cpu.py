"""Host logic of the batched combined mode over two FASTA inputs (rnascan._batched_pair_hits) without a GPU: the
device layer is the CPU oracle (tests/oracle_backend.py), the stand-in for scan_onehot_many of
test_multi_cli_cpu.py and the stand-in for scan_pair_onehot_many below, so routing, stderr order, the background
histograms and the sharded gather are checked against the per-pair loop."""
import json
import os
import subprocess
import sys

import pytest

from oracle_backend import install
from test_cli_gpu import MULTI_CASES, run_cli
from test_multi_cli_cpu import FAKE, fake_scan_onehot_many

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEQ_PFM = "tests/golden/inputs/multi/multi_seq.pfm"
STRUCT_PFM = "tests/golden/inputs/multi/multi_struct.pfm"
FA, SS_FA = "tests/golden/inputs/mixed.fa", "tests/golden/inputs/mixed_struct.fa"

PAIR_FAKE = r'''
def fake_scan_pair_onehot_many(seq_stream, struct_stream, seq_tables, struct_tables, threshold, capacity=None):
    """The per-pair oracle scans laid out as rs_scan_pair_onehot_many returns them."""
    import numpy as np
    from rnascan_b200 import device
    if not np.isfinite(threshold) or any(len(a) != len(b) or len(a) > 16 for a, b in zip(seq_tables, struct_tables)):
        raise ValueError("outside scan_pair_onehot_many")
    motif, pos, sq, st, bases = [], [], [], [], [0]
    for m, (a, b) in enumerate(zip(seq_tables, struct_tables)):
        p, x, y = device.scan_pair_onehot(seq_stream, struct_stream, a, b, threshold)
        motif.append(np.full(len(p), m, np.int32)); pos.append(p); sq.append(x); st.append(y)
        bases.append(bases[-1] + len(p))
    return (np.concatenate(motif), np.concatenate(pos), np.concatenate(sq).astype(np.float32),
            np.concatenate(st).astype(np.float64), np.array(bases, np.int64))
'''
exec(PAIR_FAKE)


def install_pair(monkeypatch):
    """The oracle backend, both batched stand-ins, the pair router's inputs counted as device-resident; returns the
    list of the pair router's results (True: batched)."""
    from rnascan_b200 import device, rnascan as ms
    install(monkeypatch)
    monkeypatch.setattr(device, "scan_onehot_many", fake_scan_onehot_many, raising=False)
    monkeypatch.setattr(device, "scan_pair_onehot_many", fake_scan_pair_onehot_many, raising=False)
    monkeypatch.setattr(ms, "_pair_on_device", lambda a, b: True)
    calls = []
    real = ms._batched_pair_hits

    def router(*a, **kw):
        out = real(*a, **kw)
        calls.append(out is not None)
        return out
    monkeypatch.setattr(ms, "_batched_pair_hits", router)
    return calls


def _forced_loop(monkeypatch, argv):
    from rnascan_b200 import rnascan as ms
    with monkeypatch.context() as mp:
        mp.setattr(ms, "_batched_pair_hits", lambda *a, **kw: None)
        ms._BATCH_CACHE.clear()
        return run_cli(argv)


def _write_fasta(path, records):
    with open(path, "w") as fh:
        for rid, text in records:
            fh.write(">%s d\n%s\n" % (rid, text))


def _read_fasta(path):
    records = []
    with open(path) as fh:
        for line in fh:
            line = line.rstrip("\n")
            if line.startswith(">"):
                records.append([line[1:].split()[0], ""])
            elif records:
                records[-1][1] += line
    return records


@pytest.fixture()
def odd_inputs(tmp_path):
    """Structure FASTA files that do not line up with mixed.fa's: other record lengths, and a pair of inputs with
    duplicate ids."""
    seq, st = _read_fasta(os.path.join(REPO, FA)), _read_fasta(os.path.join(REPO, SS_FA))
    ids = [i for i, _ in seq]
    seq_texts, st_texts = [t for _, t in seq], [t for _, t in st]
    short = str(tmp_path / "short_struct.fa")
    _write_fasta(short, [(i, t[:-1] if len(t) > 3 else t) for i, t in zip(ids, st_texts)])
    dup_seq, dup_st = str(tmp_path / "dup.fa"), str(tmp_path / "dup_struct.fa")
    _write_fasta(dup_seq, [(ids[0], seq_texts[0])] + list(zip(ids, seq_texts)))
    _write_fasta(dup_st, [(ids[0], st_texts[0])] + list(zip(ids, st_texts)))
    return {"short": short, "dup_seq": dup_seq, "dup_struct": dup_st}


def _cases(odd):
    both = ["-p", SEQ_PFM, "-q", STRUCT_PFM, "-C", "0.01"]
    return [
        (both + ["-u", "-m", "-1", FA, SS_FA], True),
        (both + ["-m", "0", FA, SS_FA], True),                                               # computed backgrounds
        (both + ["-b", "tests/golden/inputs/bg_seq_custom.txt", "-B", "tests/golden/inputs/bg_struct_example.txt",
                 "-m", "0.5", FA, SS_FA], True),
        (both + ["-u", "-m", " -inf", FA, SS_FA], False),                                    # every-position output
        (both + ["-u", "-t", "ACGUACGUAGCUAGCUAGCUAGC,EEEEEHHHHHHHHLLLLLLLRRR"], False),      # -t
        (both + ["-g", FA, SS_FA], None),                                              # --bgonly: no scan
        (["-p", "tests/golden/inputs/test_seq_pfm.txt", "-q", "tests/golden/inputs/test_struct_pfm.txt", "-C",
          "0.01", "-u", FA, SS_FA], None),                                                   # one motif pair
        (both + ["-u", "-m", "-1", FA, odd["short"]], False),                                # records differ
        (both + ["-u", "-m", "-1", odd["dup_seq"], odd["dup_struct"]], False),               # duplicate ids
        (MULTI_CASES["multi_rnass_avg"]["argv"], None),                                      # profile directory
    ]


def test_routing_and_output_equal_the_per_pair_loop(odd_inputs, in_repo, monkeypatch):
    import warnings
    from rnascan_b200 import rnascan as ms
    for argv, batched in _cases(odd_inputs):
        with monkeypatch.context() as mp:
            calls = install_pair(mp)
            profile_calls = []
            real_profile = ms._batched_profile_hits
            mp.setattr(ms, "_batched_profile_hits", lambda *a, **k: profile_calls.append(1) or real_profile(*a, **k))
            with warnings.catch_warnings():
                warnings.simplefilter("always")
                ms._BATCH_CACHE.clear()
                got = run_cli(argv)
                ms.REFERENCE_COMPAT = False
                want = _forced_loop(mp, argv)
                ms.REFERENCE_COMPAT = False
        if "--reference-compat" in argv:
            assert True not in calls and profile_calls, argv   # a directory is the profile router's shape only
        else:
            assert calls == ([] if batched is None else [batched]), argv
        assert got == want, argv                      # stdout, stderr lines (in the reference's order), exit code
        assert got[2] == 0 and got[0], argv


def test_golden_collection_through_the_batched_path(in_repo, monkeypatch):
    calls = install_pair(monkeypatch)
    out, _, code = run_cli(MULTI_CASES["multi_rnass_fasta"]["argv"])
    with open(os.path.join(REPO, "tests", "golden", "cli", "multi_rnass_fasta.stdout")) as fh:
        assert out == fh.read() and code == 0
    assert calls == [True]


def test_each_input_is_counted_once_per_run(in_repo, monkeypatch):
    """A collection with computed backgrounds: one histogram per input, however many pairs print them."""
    from rnascan_b200 import device
    calls = install_pair(monkeypatch)
    real = device.histogram
    counted = []
    monkeypatch.setattr(device, "histogram", lambda stream: counted.append(stream.kind) or real(stream))
    argv = ["-p", SEQ_PFM, "-q", STRUCT_PFM, "-C", "0.01", "-m", "0", FA, SS_FA]
    got = run_cli(argv)
    assert calls == [True] and sorted(counted) == ["rna", "struct"]
    assert sum("Calculating background" in line for line in got[1]) == 2 * MULTI_CASES["multi_rnass_fasta"]["runs"]
    assert _forced_loop(monkeypatch, argv) == got


_WORKER = r"""
import contextlib, io, json, os, sys, warnings
sys.path.insert(0, %(repo)r)
sys.path.insert(0, os.path.join(%(repo)r, "tests"))
os.chdir(%(repo)r)
import oracle_backend
from rnascan_b200 import device, rnascan as ms, shard
%(fake)s
%(pair_fake)s

class Patch(object):
    def setattr(self, obj, name, value, raising=True):
        setattr(obj, name, value)


oracle_backend.install(Patch())
device.scan_onehot_many = fake_scan_onehot_many
device.scan_pair_onehot_many = fake_scan_pair_onehot_many
ms._pair_on_device = lambda a, b: True
real = ms._batched_pair_hits
routed = []
ms._batched_pair_hits = lambda *a, **k: routed.append(1) or real(*a, **k)
rank, size = shard.init("gloo")
res = {}
for name, argv in %(cases)r:
    ms._BATCH_CACHE.clear()
    out, err = io.StringIO(), io.StringIO()
    with contextlib.redirect_stdout(out), contextlib.redirect_stderr(err), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ms.main(list(argv))
    res[name] = out.getvalue()
import torch.distributed as dist
dist.destroy_process_group()
if rank == 0:
    print(json.dumps({"out": res, "routed": len(routed)}))
elif any(res.values()):
    print(json.dumps({"out": "rank %%d wrote output" %% rank}))
"""


def test_two_ranks_equal_one_process(tmp_path, in_repo, monkeypatch):
    """torchrun with 2 gloo ranks: each rank scans its pieces, rank 0 prints the golden stdout of the collection."""
    cases = [("multi_rnass_fasta", MULTI_CASES["multi_rnass_fasta"]["argv"]),
             ("computed_bg", ["-p", SEQ_PFM, "-q", STRUCT_PFM, "-C", "0.01", "-m", "0", FA, SS_FA])]
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % {"repo": REPO, "fake": FAKE, "pair_fake": PAIR_FAKE, "cases": cases})
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", OMP_NUM_THREADS="1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29563", str(script)],
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-3000:]
    res = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert res["routed"] == 2
    with open(os.path.join(REPO, "tests", "golden", "cli", "multi_rnass_fasta.stdout")) as fh:
        assert res["out"]["multi_rnass_fasta"] == fh.read()
    install_pair(monkeypatch)
    assert res["out"]["computed_bg"] == _forced_loop(monkeypatch, cases[1][1])[0]


def test_scan_many_combined_equals_combine_of_scan_main(odd_inputs, in_repo, monkeypatch):
    """Columns, dtypes and values of every pair's frame, also where a pair has no joint window (its structure
    columns keep the dtypes of the structure-only hits), for inputs that do not line up and at -inf."""
    import argparse
    import warnings
    from rnascan_b200 import rnascan as ms
    from rnascan_b200.BioAddons.Alphabet import ContextualSecondaryStructure
    install_pair(monkeypatch)
    rna, structure = ms.IUPAC.IUPACUnambiguousRNA(), ContextualSecondaryStructure()
    seq_pssms = [ms._quiet(ms.load_motif, b, 0.01, rna, None) for b in ms.pfm_blocks(SEQ_PFM)]
    struct_pssms = [ms._quiet(ms.load_motif, b, 0.01, structure, None) for b in ms.pfm_blocks(STRUCT_PFM)]
    empty_joint = 0
    for ss, thr in ((SS_FA, -1.0), (SS_FA, 0.5), (SS_FA, float("-inf")), (odd_inputs["short"], 0.0)):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            frames = ms.scan_many_combined(FA, ss, seq_pssms, struct_pssms, thr)
            ns = argparse.Namespace(minscore=thr, debug=False)
            for sp, qp, frame in zip(seq_pssms, struct_pssms, frames):
                want = ms.combine(ms._quiet(ms.scan_main, FA, sp, rna, None, ns),
                                  ms._quiet(ms.scan_main, ss, qp, structure, None, ns))
                assert list(frame.columns) == list(want.columns)
                assert list(frame.dtypes) == list(want.dtypes)
                for col in want.columns:
                    assert frame[col].tolist() == want[col].tolist()
                empty_joint += len(want) == 0
    assert empty_joint > 0
