"""Differential test against the REFERENCE ITSELF on randomly generated inputs.

For every seed a small input set is drawn -- FASTA records with DNA letters, lower case, N runs, empty and
too-short records; matching one-hot structure contexts; averaged-profile files for some of the records; PFMs
with zero cells; thresholds from -inf upwards; pseudocounts; background options.  The reference's own
``rnascan.rnascan.main()`` (unmodified, with oracle/bio_shim standing in for Biopython and the reference's
compiled ``_pwm.c``) was run on each of them by tests/golden/make_golden_fuzz.py; its stdout, exit code and
argv are stored in tests/golden/fuzz.  Here the inputs are drawn again from the seed and
``rnascan_b200.rnascan.main()`` runs on them with the device entry points swapped for the CPU oracle
(tests/oracle_backend.py).  stdout must be byte-identical (averaged-profile runs under ``--reference-compat``,
see INTEGRATION.md section 0), exit codes equal.  A seed the reference crashed on (it has a few: merging with an
empty structure frame raises KeyError) has no stored output and skips itself -- there is nothing to be
identical to.

This pins the HOST logic -- record handling, background arithmetic, PFM preprocessing, frame assembly with all
the pandas dtype artefacts, TSV text -- far beyond the fixed golden files; the kernels are pinned to the same
oracle, and to the same stored outputs, by the -m gpu tests.
"""
import contextlib
import io
import json
import os
import warnings

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FUZZ = os.path.join(REPO, "tests", "golden", "fuzz")


@pytest.fixture(scope="module")
def reference():
    """{seed: {"argv", "exit", "mode"}} of the reference's runs; its stdout is FUZZ/<seed>.stdout."""
    with open(os.path.join(FUZZ, "cases.json")) as fh:
        return json.load(fh)


def run_ours(argv):
    from rnascan_b200 import rnascan as ms
    out, err = io.StringIO(), io.StringIO()
    code = 0
    ms._BATCH_CACHE.clear()
    with contextlib.redirect_stdout(out), contextlib.redirect_stderr(err), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        try:
            ms.main(list(argv))
        except SystemExit as e:
            code = e.code or 0
    ms.REFERENCE_COMPAT = False
    return out.getvalue(), code


def draw_inputs(rng, root):
    """Files of one random case; returns a dict of paths."""
    os.makedirs(root, exist_ok=True)
    n_rec = int(rng.integers(1, 7))
    recs = []
    for r in range(n_rec):
        n = int(rng.choice([0, 2, 5, 12, 30, 60, 140], p=[.06, .06, .08, .2, .25, .2, .15]))
        seq = rng.choice(list("ACGU"), size=n, p=[.27, .22, .22, .29])
        if n > 8 and rng.random() < 0.3:
            a = int(rng.integers(0, n - 3))
            seq[a:a + int(rng.integers(1, 4))] = "N"
        seq = "".join(seq)
        if rng.random() < 0.3:
            seq = seq.replace("U", "T")
        if rng.random() < 0.2:
            seq = seq.lower()
        title = "r%d" % r + ("" if rng.random() < 0.5 else " some description %d" % r)
        recs.append((title, seq))
    paths = {"fa": os.path.join(root, "seqs.fa"), "ss": os.path.join(root, "structs.fa"),
             "dir": os.path.join(root, "profiles")}
    with open(paths["fa"], "w") as fh:
        for title, seq in recs:
            fh.write(">%s\n" % title)
            for k in range(0, len(seq), 50):
                fh.write(seq[k:k + 50] + "\n")
    with open(paths["ss"], "w") as fh:
        for title, seq in recs:
            st, cur = [], "E"
            for _ in range(len(seq)):
                if rng.random() > 0.7:
                    cur = str(rng.choice(list("EHTBLRM")))
                st.append(cur)
            st = "".join(st)
            if st and rng.random() < 0.2:
                st = st[:len(st) // 2].lower() + st[len(st) // 2:]
            fh.write(">%s\n%s\n" % (title, st))
    os.makedirs(paths["dir"], exist_ok=True)
    n_prof = 0
    for title, seq in recs:
        if len(seq) == 0 or (rng.random() < 0.25 and n_prof > 0):
            continue
        w = rng.dirichlet(0.4 * np.ones(7), size=len(seq))
        w[w < 0.03] = 0.0
        w /= np.maximum(w.sum(axis=1, keepdims=True), 1e-300)
        with open(os.path.join(paths["dir"], "structure.%s.txt" % title.split()[0]), "w") as fh:
            fh.write("PO\tB\tE\tH\tL\tM\tR\tT\n")
            for i in range(len(seq)):
                fh.write(str(i) + "".join("\t" + str(float(v)) for v in w[i]) + "\n")
        n_prof += 1
    if n_prof == 0:                                # the reference raises IOError on an empty directory
        with open(os.path.join(paths["dir"], "structure.extra.txt"), "w") as fh:
            fh.write("PO\tB\tE\tH\tL\tM\tR\tT\n0\t0.1\t0.2\t0.1\t0.2\t0.1\t0.2\t0.1\n")
    W = int(rng.integers(2, 9))
    for key, letters in (("pfm_seq", "ACGU"), ("pfm_struct", "BEHLMRT")):
        rows = rng.dirichlet(0.5 * np.ones(len(letters)), size=W)
        if rng.random() < 0.4:
            rows[rows < 0.05] = 0.0
        order = list(letters)
        rng.shuffle(order)                         # header letters may come in any order (rnascan.py:242-244)
        paths[key] = os.path.join(root, key + ".txt")
        with open(paths[key], "w") as fh:
            fh.write("PO\t" + "\t".join(order) + "\n")
            for i in range(W):
                fh.write("%d\t%s\n" % (i + 1, "\t".join(repr(round(float(rows[i, letters.index(l)]), 4)) for l in order)))
    paths["bg_seq"] = os.path.join(root, "bg_seq.txt")
    with open(paths["bg_seq"], "w") as fh:
        fh.write(repr({"A": 0.28, "C": 0.21, "G": 0.22, "U": 0.29}))
    paths["bg_struct"] = os.path.join(root, "bg_struct.txt")
    with open(paths["bg_struct"], "w") as fh:
        fh.write(repr({"E": 0.27, "H": 0.15, "T": 0.14, "B": 0.02, "L": 0.2, "R": 0.2, "M": 0.02}))
    return paths


def draw_argv(rng, p):
    mode = str(rng.choice(["rna", "ss", "rnass", "ss_avg", "rnass_avg", "testseq_rna", "testseq_ss", "testseq_rnass"],
                          p=[.2, .15, .15, .15, .2, .05, .05, .05]))
    if mode.startswith("testseq"):                 # -t: one sequence (and / or structure) on the command line
        n = int(rng.integers(1, 40))
        seq = "".join(rng.choice(list("ACGTUacgun"), size=n))
        st = "".join(rng.choice(list("EHTBLRMe"), size=n))
        thr = str(rng.choice([" -inf", " -2", "0", "1"]))
        argv = ["-m", thr, "-C", str(rng.choice(["0", "0.01"]))]
        if mode == "testseq_rna":
            argv += ["-p", p["pfm_seq"], "-t", seq]
        elif mode == "testseq_ss":
            argv += ["-q", p["pfm_struct"], "-t", st]
        else:
            argv += ["-p", p["pfm_seq"], "-q", p["pfm_struct"], "-t", seq + "," + st]
        return mode, argv, []
    thr = rng.choice([" -inf", " -4", " -1", "0", "0.5", "1.5", "3", "6"])
    argv = ["-m", str(thr), "-C", str(rng.choice(["0", "0.01", "0.5"]))]
    bg = str(rng.choice(["computed", "uniform", "file"]))
    if mode in ("rna", "rnass", "rnass_avg"):
        argv += ["-p", p["pfm_seq"]]
    if mode in ("ss", "rnass", "ss_avg", "rnass_avg"):
        argv += ["-q", p["pfm_struct"]]
    if mode in ("ss_avg", "rnass_avg") and bg == "computed":
        bg = "file"                                # a directory has no structure background to compute
    if bg == "uniform":
        argv += ["-u"]
    elif bg == "file":
        if "-p" in argv:
            argv += ["-b", p["bg_seq"]]
        if "-q" in argv:
            argv += ["-B", p["bg_struct"]]
    if mode == "rna":
        argv += [p["fa"]]
    elif mode == "ss":
        argv += [p["ss"]]
    elif mode == "rnass":
        argv += [p["fa"], p["ss"]]
    elif mode == "ss_avg":
        argv += [p["dir"]]
    else:
        argv += [p["fa"], p["dir"]]
    compat = ["--reference-compat"] if mode.endswith("avg") else []
    if mode in ("rna", "ss") and bg == "computed" and rng.random() < 0.25:
        argv = ["--bgonly"] + argv                 # print the background dictionary and exit (rnascan.py:512-515)
    return mode, argv, compat


@pytest.mark.parametrize("seed", range(90))
def test_reference_and_rnascan_b200_print_the_same_bytes(seed, reference, tmp_path, monkeypatch):
    from oracle_backend import install
    rng = np.random.default_rng(9000 + seed)
    paths = draw_inputs(rng, str(tmp_path / "case"))
    mode, argv, compat = draw_argv(rng, paths)
    case = reference.get(str(seed))
    if case is None:
        pytest.skip("the reference raised on this input")
    placeholders = {v: "{%s}" % k for k, v in paths.items()}
    assert [placeholders.get(a, a) for a in argv] + compat == case["argv"], "the seed no longer draws the stored case"
    with open(os.path.join(FUZZ, "%d.stdout" % seed)) as fh:
        want = fh.read()
    install(monkeypatch)
    got, got_code = run_ours(argv + compat)
    assert got_code == case["exit"], (mode, argv)
    assert got == want, (mode, argv)
