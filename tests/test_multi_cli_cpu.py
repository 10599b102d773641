"""Host logic of the batched FASTA scan of motif collections (rnascan._batched_fasta_hits) without a GPU: the
device layer is the CPU oracle (tests/oracle_backend.py) plus the stand-in for scan_onehot_many below, so
routing, stderr order and the sharded gather are checked against the per-motif loop."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle_backend import install
from test_cli_gpu import MULTI_CASES, run_cli

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEQ_PFM = "tests/golden/inputs/multi/multi_seq.pfm"
STRUCT_PFM = "tests/golden/inputs/multi/multi_struct.pfm"
FA, SS_FA = "tests/golden/inputs/mixed.fa", "tests/golden/inputs/mixed_struct.fa"

FAKE = r'''
def fake_scan_onehot_many(stream, tables, threshold, capacity=None):
    """The per-motif oracle scans laid out as rs_scan_onehot_many returns them."""
    import numpy as np
    from rnascan_b200 import device
    if stream.kind not in ("rna", "struct") or not np.isfinite(threshold) or max(len(t) for t in tables) > 16:
        raise ValueError("outside scan_onehot_many")
    fn = device.scan_seq if stream.kind == "rna" else device.scan_struct_onehot
    motif, pos, scores, bases = [], [], [], [0]
    for m, t in enumerate(tables):
        p, s = fn(stream, t, threshold)
        motif.append(np.full(len(p), m, np.int32)); pos.append(p); scores.append(s)
        bases.append(bases[-1] + len(p))
    return (np.concatenate(motif), np.concatenate(pos), np.concatenate(scores), np.array(bases, np.int64))
'''
exec(FAKE)


def install_batched(monkeypatch):
    """The oracle backend, the stand-in for scan_onehot_many, and its streams counted as device-resident."""
    from rnascan_b200 import device, rnascan as ms
    install(monkeypatch)
    monkeypatch.setattr(device, "scan_onehot_many", fake_scan_onehot_many, raising=False)
    monkeypatch.setattr(ms, "_on_device", lambda batches: True)
    calls = []
    real = ms._batched_fasta_hits

    def router(*a, **kw):
        out = real(*a, **kw)
        calls.append(out is not None)
        return out
    monkeypatch.setattr(ms, "_batched_fasta_hits", router)
    return calls


def _forced_loop(monkeypatch, argv):
    from rnascan_b200 import rnascan as ms
    with monkeypatch.context() as mp:
        mp.setattr(ms, "_batched_fasta_hits", lambda *a, **kw: None)
        ms._BATCH_CACHE.clear()
        return run_cli(argv)


@pytest.mark.parametrize("argv,batched", [
    (["-p", SEQ_PFM, "-C", "0.01", "-m", "0.5", FA], True),
    (["-q", STRUCT_PFM, "-C", "0.01", "-m", "0", SS_FA], True),
    (["-p", SEQ_PFM, "-C", "0.01", "-u", "-m", "-1", FA], True),
    (["-q", STRUCT_PFM, "-C", "0.01", "-B", "tests/golden/inputs/bg_struct_example.txt", "-m", "2", SS_FA], True),
    (["-p", SEQ_PFM, "-C", "0.01", "-m", " -inf", FA], False),                  # every-position output
    (["-p", SEQ_PFM, "-C", "0.01", "-t", "ACGUACGUAGCUAGCUAGCUAGC"], False),     # -t
    (["-p", SEQ_PFM, "-C", "0.01", "-g", FA], None),                           # --bgonly: no scan
    (["-p", "tests/golden/inputs/test_seq_pfm.txt", "-C", "0.01", FA], None),  # one motif: not a collection
    (MULTI_CASES["multi_rnass_fasta"]["argv"], False),                          # two FASTA inputs
    (MULTI_CASES["multi_ss_avg"]["argv"], False),                               # profile directory
])
def test_routing_and_output_equal_the_per_motif_loop(argv, batched, in_repo, monkeypatch):
    import warnings
    from rnascan_b200 import rnascan as ms
    calls = install_batched(monkeypatch)
    with warnings.catch_warnings():
        warnings.simplefilter("always")
        ms._BATCH_CACHE.clear()
        got = run_cli(argv)
        ms.REFERENCE_COMPAT = False
        want = _forced_loop(monkeypatch, argv)
        ms.REFERENCE_COMPAT = False
    assert calls == ([] if batched is None else [batched])
    assert got == want                                # stdout, stderr lines (in the reference's order), exit code


def test_wide_motifs_fall_back(in_repo, monkeypatch, tmp_path):
    from rnascan_b200 import pfmutil
    rng = np.random.default_rng(1)
    pfms = [{c: rng.dirichlet(np.ones(4))[i:i + 1].tolist() * W for i, c in enumerate("ACGU")} for W in (6, 17)]
    path = str(tmp_path / "wide.pfm")
    pfmutil.write_multi_pfm(["a", "b"], pfms, path)
    calls = install_batched(monkeypatch)
    got = run_cli(["-p", path, "-C", "0.01", "-m", "0", FA])
    assert calls == [False]
    assert got == _forced_loop(monkeypatch, ["-p", path, "-C", "0.01", "-m", "0", FA])


def test_golden_collections_through_the_batched_path(in_repo, monkeypatch):
    calls = install_batched(monkeypatch)
    for name in ("multi_rna_mixed", "multi_ss_fasta"):
        out, _, code = run_cli(MULTI_CASES[name]["argv"])
        with open(os.path.join(REPO, "tests", "golden", "cli", name + ".stdout")) as fh:
            assert out == fh.read() and code == 0
    assert calls == [True, True]


_WORKER = r"""
import contextlib, io, json, os, sys, warnings
sys.path.insert(0, %(repo)r)
sys.path.insert(0, os.path.join(%(repo)r, "tests"))
os.chdir(%(repo)r)
import oracle_backend
from rnascan_b200 import device, rnascan as ms, shard
%(fake)s

class Patch(object):
    def setattr(self, obj, name, value, raising=True):
        setattr(obj, name, value)


oracle_backend.install(Patch())
device.scan_onehot_many = fake_scan_onehot_many
ms._on_device = lambda batches: True
real = ms._batched_fasta_hits
routed = []
ms._batched_fasta_hits = lambda *a, **k: routed.append(1) or real(*a, **k)
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
    """torchrun with 2 gloo ranks: each rank scans its pieces, one gather, rank 0 prints what one process
    prints (the golden stdout of the collection)."""
    cases = [(name, MULTI_CASES[name]["argv"]) for name in ("multi_rna_mixed", "multi_ss_fasta")]
    cases.append(("rna_u", ["-p", SEQ_PFM, "-C", "0.01", "-u", "-m", "-1", FA]))
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % {"repo": REPO, "fake": FAKE, "cases": cases})
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", OMP_NUM_THREADS="1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29561", str(script)],
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-3000:]
    res = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert res["routed"] == 3
    install_batched(monkeypatch)
    for name, argv in cases:
        assert res["out"][name] == _forced_loop(monkeypatch, argv)[0], name
