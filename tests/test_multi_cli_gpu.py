"""Motif collections over a FASTA input through the batched scan (rnascan._batched_fasta_hits ->
device.scan_onehot_many): stdout and stderr must equal the per-motif loop's, and scan_many_fasta must equal
scan_main per motif."""
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


def _spy(monkeypatch):
    """Counts per-motif scan calls and batched-router results."""
    from rnascan_b200 import device, rnascan as ms
    calls = {"per_motif": 0, "batched": 0}
    for name in ("scan_seq", "scan_struct_onehot", "scan_onehot_bg"):
        real = getattr(device, name)

        def wrapped(*a, _real=real, **k):
            calls["per_motif"] += 1
            return _real(*a, **k)
        monkeypatch.setattr(device, name, wrapped)
    real_router = ms._batched_fasta_hits

    def router(*a, **k):
        out = real_router(*a, **k)
        calls["batched"] += out is not None
        return out
    monkeypatch.setattr(ms, "_batched_fasta_hits", router)
    return calls


@pytest.mark.parametrize("name", ["multi_rna_mixed", "multi_ss_fasta"])
def test_golden_collections_go_through_the_batched_scan(name, in_repo, monkeypatch):
    from rnascan_b200 import rnascan as ms
    calls = _spy(monkeypatch)
    ms._BATCH_CACHE.clear()
    out, _, code = _run(MULTI_CASES[name]["argv"])
    with open(os.path.join(CLI, name + ".stdout")) as fh:
        assert out == fh.read()
    assert code == 0 and calls == {"per_motif": 0, "batched": 1}


def _collection(root, k, rng, kind):
    from rnascan_b200 import pfmutil
    letters = "ACGU" if kind == "rna" else "BEHLMRT"
    M = int(rng.integers(2, 12))
    pfms = []
    for _ in range(M):
        W = int(rng.integers(4, 17))
        rows = rng.dirichlet(0.4 * np.ones(len(letters)), size=W)
        rows[rng.random(rows.shape) < 0.05] = 0.0                        # zero counts
        pfms.append({c: [round(float(v), 4) for v in rows[:, i]] for i, c in enumerate(letters)})
    path = os.path.join(root, "coll%d.pfm" % k)
    pfmutil.write_multi_pfm(["m%d_%d" % (k, i) for i in range(M)], pfms, path)
    return path


def _fasta(root, kind, rng):
    from rnascan_b200 import synth
    path = os.path.join(root, kind + ".fa")
    lengths = synth.record_lengths(60_000, 30, rng)
    with open(path, "w") as fh:
        for i, ln in enumerate(lengths.tolist()):
            if kind == "rna":
                s = "".join(rng.choice(list("ACGUTNacgu"), size=ln, p=[.23, .23, .23, .2, .03, .02, .02, .02, .01, .01]))
            else:
                s = "".join(rng.choice(list("BEHLMRTehx"), size=ln, p=[.02, .25, .15, .2, .03, .2, .1, .02, .02, .01]))
            fh.write(">r%d desc %d\n%s\n" % (i, i, s))
        fh.write(">empty\n\n>short\n%s\n" % ("AC" if kind == "rna" else "BE"))
    return path


def test_generated_collections_equal_the_per_motif_loop(tmp_path, in_repo, monkeypatch):
    from rnascan_b200 import rnascan as ms
    rng = np.random.default_rng(2024)
    root = str(tmp_path)
    fastas = {kind: _fasta(root, kind, rng) for kind in ("rna", "struct")}
    bg_files = {}
    for kind, letters in (("rna", "ACGU"), ("struct", "BEHLMRT")):
        p = rng.dirichlet(np.ones(len(letters)))
        bg_files[kind] = os.path.join(root, kind + "_bg.txt")
        with open(bg_files[kind], "w") as fh:
            fh.write(repr({c: float(v) for c, v in zip(letters, p)}))
    cases = []
    for k in range(40):
        kind = "rna" if k % 2 == 0 else "struct"
        flag = "-p" if kind == "rna" else "-q"
        bg = [[], ["-B", bg_files[kind]] if kind == "struct" else ["-b", bg_files[kind]], ["-u"]][k % 3]
        thr = ["0", "0.5", "6"][(k // 3) % 3] if k < 39 else "1000"                # the last one: no hit at all
        cases.append([flag, _collection(root, k, rng, kind), "-C", "0.01", "-m", thr] + bg + [fastas[kind]])
    real = ms._batched_fasta_hits
    state = {"loop": False, "batched": 0}

    def router(*a, **kw):
        if state["loop"]:
            return None                                   # the per-motif loop
        out = real(*a, **kw)
        state["batched"] += out is not None
        return out
    monkeypatch.setattr(ms, "_batched_fasta_hits", router)
    for k, argv in enumerate(cases):
        monkeypatch.setattr(ms, "NATIVE_WRITER_MIN_ROWS", 1 if k % 4 != 1 else 10 ** 12)
        got = {}
        for loop in (False, True):
            state["loop"] = loop
            ms._BATCH_CACHE.clear()
            got[loop] = _run(argv)
        assert state["batched"] == k + 1, argv
        assert got[False] == got[True], argv


def test_scan_many_fasta_equals_scan_main_per_motif(in_repo):
    from rnascan_b200 import rnascan as ms
    from rnascan_b200.BioAddons.Alphabet import ContextualSecondaryStructure
    rna, structure = ms.IUPAC.IUPACUnambiguousRNA(), ContextualSecondaryStructure()
    for alphabet, fasta, pfm in ((rna, "mixed.fa", "multi_seq.pfm"), (structure, "mixed_struct.fa", "multi_struct.pfm")):
        path = os.path.join(INP, fasta)
        blocks = ms.pfm_blocks(os.path.join(INP, "multi", pfm))
        bg = ms._quiet(ms.compute_background, path, alphabet, False)
        pssms = [ms._quiet(ms.load_motif, b, 0.01, alphabet, bg) for b in blocks]
        for thr in (-1.0, 0.5, float("-inf")):
            frames = ms.scan_many_fasta(path, pssms, alphabet, thr)
            ns = argparse.Namespace(minscore=thr, debug=False)
            assert len(frames) == len(pssms)
            for pssm, frame in zip(pssms, frames):
                want = ms._quiet(ms.scan_main, path, pssm, alphabet, None, ns)
                assert list(frame.columns) == list(want.columns)
                assert list(frame.dtypes) == list(want.dtypes)
                for col in want.columns:
                    assert frame[col].tolist() == want[col].tolist()


def test_stats_record_the_batched_motifs(tmp_path, in_repo):
    from rnascan_b200 import rnascan as ms
    ms._BATCH_CACHE.clear()
    stats = str(tmp_path / "stats.json")
    _run(MULTI_CASES["multi_rna_mixed"]["argv"] + ["--stats", stats])
    with open(stats) as fh:
        line = json.loads(fh.readline())
    assert line["batched_motifs"] == MULTI_CASES["multi_rna_mixed"]["runs"]
    assert line["scored_positions"] > 0
