"""Motif-pair collections in the combined mode over two FASTA inputs through the batched scans
(rnascan._batched_pair_hits -> device.scan_onehot_many + device.scan_pair_onehot_many): stdout and stderr must
equal the per-pair loop's, and scan_many_combined must equal combine(scan_main, scan_main) per pair."""
import argparse
import json
import os
import warnings

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

pytest.importorskip("torch")

from test_cli_gpu import CLI, INP, MULTI_CASES, run_cli  # noqa: E402


def _run(argv):
    with warnings.catch_warnings():
        warnings.simplefilter("always")
        return run_cli(argv)


def test_golden_collection_goes_through_the_batched_scans(in_repo, monkeypatch):
    from rnascan_b200 import device, rnascan as ms
    calls = {"per_motif": 0, "pair_many": 0}
    for name in ("scan_seq", "scan_onehot_bg", "scan_pair_onehot"):
        real = getattr(device, name)
        monkeypatch.setattr(device, name, lambda *a, _real=real, **k: calls.__setitem__(
            "per_motif", calls["per_motif"] + 1) or _real(*a, **k))
    real_many = device.scan_pair_onehot_many
    monkeypatch.setattr(device, "scan_pair_onehot_many", lambda *a, **k: calls.__setitem__(
        "pair_many", calls["pair_many"] + 1) or real_many(*a, **k))
    ms._BATCH_CACHE.clear()
    out, _, code = _run(MULTI_CASES["multi_rnass_fasta"]["argv"])
    with open(os.path.join(CLI, "multi_rnass_fasta.stdout")) as fh:
        assert out == fh.read()
    n_batches = len(ms._cached_batches(os.path.join(INP, "mixed.fa"), ms.IUPAC.IUPACUnambiguousRNA()))
    assert code == 0 and calls == {"per_motif": 0, "pair_many": n_batches}


def _pair_files(root, k, rng):
    """A multi-PFM file of sequence motifs and one of structure motifs; about one pair in four has two widths."""
    from rnascan_b200 import pfmutil
    M = int(rng.integers(2, 13))
    seq, struct = [], []
    for _ in range(M):
        W = int(rng.integers(4, 17))
        W2 = W if rng.random() > 0.25 else int(rng.integers(4, 17))
        for out, letters, width in ((seq, "ACGU", W), (struct, "BEHLMRT", W2)):
            rows = rng.dirichlet(0.4 * np.ones(len(letters)), size=width)
            rows[rng.random(rows.shape) < 0.05] = 0.0                    # zero counts
            out.append({c: [round(float(v), 4) for v in rows[:, i]] for i, c in enumerate(letters)})
    paths = [os.path.join(root, "c%d_%s.pfm" % (k, side)) for side in ("seq", "struct")]
    pfmutil.write_multi_pfm(["s%d_%d" % (k, i) for i in range(M)], seq, paths[0])
    pfmutil.write_multi_pfm(["q%d_%d" % (k, i) for i in range(M)], struct, paths[1])
    return paths


def _fasta_pair(root, rng, shorten=False, duplicate=False):
    """A sequence FASTA and a structure FASTA with the same ids and record lengths (or, `shorten`, structure records
    one letter shorter; `duplicate`, one id twice)."""
    from rnascan_b200 import synth
    lengths = synth.record_lengths(60_000, 30, rng).tolist() + [0, 2]
    ids = ["r%d" % i for i in range(len(lengths))]
    if duplicate:
        ids[5] = ids[2]
    paths = [os.path.join(root, "pair%s%s_%s.fa" % ("_short" if shorten else "", "_dup" if duplicate else "", kind))
             for kind in ("seq", "struct")]
    with open(paths[0], "w") as fs, open(paths[1], "w") as fq:
        for rid, ln in zip(ids, lengths):
            s = "".join(rng.choice(list("ACGUTNacgu"), size=ln, p=[.23, .23, .23, .2, .03, .02, .02, .02, .01, .01]))
            q = "".join(rng.choice(list("BEHLMRTehx"), size=ln - (shorten and ln > 3),
                                   p=[.02, .25, .15, .2, .03, .2, .1, .02, .02, .01]))
            fs.write(">%s desc\n%s\n" % (rid, s))
            fq.write(">%s desc\n%s\n" % (rid, q))
    return paths


def _both_ways(monkeypatch, argv, state):
    from rnascan_b200 import rnascan as ms
    got = {}
    for loop in (False, True):
        state["loop"] = loop
        ms._BATCH_CACHE.clear()
        got[loop] = _run(argv)
    return got


def _patch_router(monkeypatch):
    from rnascan_b200 import rnascan as ms
    real = ms._batched_pair_hits
    state = {"loop": False, "batched": 0, "declined": 0}

    def router(*a, **kw):
        if state["loop"]:
            return None                                   # the per-pair loop
        out = real(*a, **kw)
        state["batched" if out is not None else "declined"] += 1
        return out
    monkeypatch.setattr(ms, "_batched_pair_hits", router)
    return state


def test_generated_collections_equal_the_per_pair_loop(tmp_path, in_repo, monkeypatch):
    from rnascan_b200 import rnascan as ms
    rng = np.random.default_rng(77)
    root = str(tmp_path)
    fa, ss = _fasta_pair(root, rng)
    bg = {}
    for side, letters in (("seq", "ACGU"), ("struct", "BEHLMRT")):
        p = rng.dirichlet(np.ones(len(letters)))
        bg[side] = os.path.join(root, side + "_bg.txt")
        with open(bg[side], "w") as fh:
            fh.write(repr({c: float(v) for c, v in zip(letters, p)}))
    state = _patch_router(monkeypatch)
    for k in range(30):
        seq_pfm, struct_pfm = _pair_files(root, k, rng)
        bgs = [[], ["-b", bg["seq"], "-B", bg["struct"]], ["-u"]][k % 3]
        thr = ["-1", "0", "2"][(k // 3) % 3] if k < 29 else "1000"               # the last one: no joint hit
        argv = ["-p", seq_pfm, "-q", struct_pfm, "-C", "0.01", "-m", thr] + bgs + [fa, ss]
        monkeypatch.setattr(ms, "NATIVE_WRITER_MIN_ROWS", 1 if k % 4 != 1 else 10 ** 12)
        got = _both_ways(monkeypatch, argv, state)
        assert state["batched"] == k + 1, argv
        assert got[False] == got[True], argv
        assert got[False][2] == 0


@pytest.mark.parametrize("shape", ["shorten", "duplicate"])
def test_inputs_that_do_not_line_up_take_the_loop(shape, tmp_path, in_repo, monkeypatch):
    rng = np.random.default_rng(5)
    fa, ss = _fasta_pair(str(tmp_path), rng, **{shape: True})
    seq_pfm, struct_pfm = _pair_files(str(tmp_path), 0, rng)
    state = _patch_router(monkeypatch)
    got = _both_ways(monkeypatch, ["-p", seq_pfm, "-q", struct_pfm, "-C", "0.01", "-u", "-m", "0", fa, ss], state)
    assert state == {"loop": True, "batched": 0, "declined": 1}
    assert got[False] == got[True] and got[False][2] == 0


def test_scan_many_combined_equals_combine_of_scan_main_per_pair(in_repo):
    from rnascan_b200 import rnascan as ms
    from rnascan_b200.BioAddons.Alphabet import ContextualSecondaryStructure
    rna, structure = ms.IUPAC.IUPACUnambiguousRNA(), ContextualSecondaryStructure()
    fa, ss = os.path.join(INP, "mixed.fa"), os.path.join(INP, "mixed_struct.fa")
    bg_seq = ms._quiet(ms.compute_background, fa, rna, False)
    bg_struct = ms._quiet(ms.compute_background, ss, structure, False)
    seq_pssms = [ms._quiet(ms.load_motif, b, 0.01, rna, bg_seq)
                 for b in ms.pfm_blocks(os.path.join(INP, "multi", "multi_seq.pfm"))]
    struct_pssms = [ms._quiet(ms.load_motif, b, 0.01, structure, bg_struct)
                    for b in ms.pfm_blocks(os.path.join(INP, "multi", "multi_struct.pfm"))]
    for thr in (-1.0, 0.5, float("-inf")):
        frames = ms.scan_many_combined(fa, ss, seq_pssms, struct_pssms, thr)
        ns = argparse.Namespace(minscore=thr, debug=False)
        assert len(frames) == len(seq_pssms)
        for sp, qp, frame in zip(seq_pssms, struct_pssms, frames):
            want = ms.combine(ms._quiet(ms.scan_main, fa, sp, rna, None, ns),
                              ms._quiet(ms.scan_main, ss, qp, structure, None, ns))
            assert list(frame.columns) == list(want.columns)
            assert list(frame.dtypes) == list(want.dtypes)
            for col in want.columns:
                assert frame[col].tolist() == want[col].tolist()


def test_stats_record_the_batched_pairs(tmp_path, in_repo):
    from rnascan_b200 import rnascan as ms
    ms._BATCH_CACHE.clear()
    stats = str(tmp_path / "stats.json")
    _run(MULTI_CASES["multi_rnass_fasta"]["argv"] + ["--stats", stats])
    with open(stats) as fh:
        line = json.loads(fh.readline())
    assert line["batched_motifs"] == MULTI_CASES["multi_rnass_fasta"]["runs"]
    assert line["scored_positions"] > 0
