"""Host-side logic of the product (no GPU needed): PFM -> log-odds, sequence handling, argument
parsing, pfmutil, shard planning, and that the C-ABI library loads and exports every symbol
declared in include/rnascan_b200.h."""
import copy
import os
import re
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INP = os.path.join(REPO, "tests", "golden", "inputs")


def same(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b)) and \
        np.array_equal(a[~np.isnan(a)], b[~np.isnan(b)])


# ----------------------------------------------------------------------------- C ABI
def test_library_exports_every_declared_symbol():
    from rnascan_b200 import _lib
    header = open(os.path.join(REPO, "include", "rnascan_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = sorted(set(re.findall(r"\b(rs_[a-z0-9_]+)\s*\(", header)))
    assert declared, "no declarations found"
    for name in declared:
        assert hasattr(_lib.lib, name), "library lacks %s" % name
    assert sorted(_lib.EXPORTS) == declared, "ctypes signatures and header differ"
    assert _lib.lib.rs_version() >= 100
    assert _lib.lib.rs_padded_count(0) == 256 and _lib.lib.rs_padded_count(257) == 768
    assert _lib.lib.rs_scan_workspace_bytes(1 << 20, 1000) > 0


def test_host_encoders_match_the_reference_switch():
    from rnascan_b200 import device, _lib
    codes, off, ln = device.pack_texts(["ACGUTacgutNn-x", "", "Rr"], "rna")
    assert codes.tolist() == [0, 1, 2, 3, 3, 0, 1, 2, 3, 3, 12, 12, 12, 12, 255, 255, 12, 12, 255]
    assert off.tolist() == [0, 15, 16] and ln.tolist() == [14, 0, 2]
    codes, _, _ = device.pack_texts(["BEHLMRTbehlmrtXx."], "struct")
    assert codes.tolist() == [0, 1, 2, 3, 4, 5, 6, 8, 9, 10, 11, 12, 13, 14, 15, 15, 15, 255]
    assert _lib.RS_SEP == 255


def test_no_cpu_fallback_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from rnascan_b200 import device, _lib
    with pytest.raises(_lib.RnascanCudaError):
        device.SymbolStream(np.zeros(8, np.uint8))
    from rnascan_b200.BioAddons.motifs import _pwm
    with pytest.raises(_lib.RnascanCudaError):
        _pwm.calculate("ACGUACGU", np.zeros((4, 4)))


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(REPO, "rnascan_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                text = open(os.path.join(root, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "liboracle" not in text, f


# ----------------------------------------------------------------------------- PFM -> PSSM
def test_pfm2pssm_matches_the_reference(golden_api, in_repo):
    from rnascan_b200 import rnascan as ms
    from rnascan_b200.seq import IUPAC
    from rnascan_b200.BioAddons.Alphabet import ContextualSecondaryStructure
    for name, g in golden_api["pssm"].items():
        alpha = IUPAC.IUPACUnambiguousRNA() if g["alphabet"] == "GAUC" else ContextualSecondaryStructure()
        assert alpha.letters == g["alphabet"]
        bg = g["background"]
        if bg is not None:
            bg = {l: bg[l] for l in g["alphabet"]}
        pm = ms.pfm2pssm(g["file"], g["pseudocount"], alpha, bg)
        assert list(pm.keys()) == list(g["alphabet"])
        assert pm.length == len(g["values"][g["alphabet"][0]])
        for letter in g["alphabet"]:
            assert same(pm[letter], g["values"][letter]), (name, letter)


def test_pssm_object(golden_api, in_repo):
    from rnascan_b200 import rnascan as ms
    from rnascan_b200.seq import IUPAC
    pm = ms.pfm2pssm(os.path.join(INP, "SLBP_pfm_assembled_normalized_seq.txt"), 0,
                     IUPAC.IUPACUnambiguousRNA(), None)
    assert pm.length == 18 and len(pm.consensus) == 18
    assert str(pm.consensus)[5:9] == "CUCU" or len(str(pm.consensus)) == 18
    t = pm.table("ACGU")
    assert t.shape == (18, 4) and t[0, 3] == pm["U"][0]
    loaded = ms.load_motif(os.path.join(INP, "test_seq_pfm.txt"), 0, IUPAC.IUPACUnambiguousRNA(), None)
    assert list(loaded) == ["test_seq_pfm"]


def test_wrong_alphabet_pfm_raises_keyerror(in_repo):
    from rnascan_b200 import rnascan as ms
    from rnascan_b200.BioAddons.Alphabet import ContextualSecondaryStructure
    with pytest.raises(KeyError):
        ms.load_motif(os.path.join(INP, "test_seq_pfm.txt"), 0, ContextualSecondaryStructure(), None)


# ----------------------------------------------------------------------------- sequences
def test_preprocess_seq_cases_of_the_reference():
    # /root/reference/tests/preprocess_seq_test.py:13-53
    from rnascan_b200 import rnascan as ms
    from rnascan_b200.seq import Seq, SeqRecord, IUPAC, SingleLetterAlphabet
    from rnascan_b200.BioAddons.Alphabet import ContextualSecondaryStructure
    rna, dna = IUPAC.IUPACUnambiguousRNA(), IUPAC.IUPACUnambiguousDNA()
    cases = [(Seq("GATTACA", dna), rna, "GAUUACA"), (Seq("GAUUACA", rna), rna, "GAUUACA"),
             (Seq("GAUUACA", rna), dna, "GAUUACA"), (Seq("GATTACA", dna), dna, "GATTACA"),
             (Seq("GAUUACA", SingleLetterAlphabet()), rna, "GAUUACA"),
             (Seq("KHIL", ContextualSecondaryStructure()), rna, "KHIL"),
             (Seq("gattaca", SingleLetterAlphabet()), rna, "GAUUACA")]
    for s, alpha, want in cases:
        assert str(ms.preprocess_seq(SeqRecord(s), alpha)) == want
    with pytest.raises(TypeError):
        ms.preprocess_seq("GATTACA", rna)


def test_parse_sequences_and_batches():
    # /root/reference/tests/motif_scan_test.py:18-25
    from rnascan_b200 import rnascan as ms
    recs = list(ms.parse_sequences([os.path.join(INP, "test.fa")]))
    assert [r.id for r in recs] == ["read1", "read2"]
    assert all(str(r.seq) == "UUUUGCUCUGUAUAUA" for r in recs)
    recs = list(ms.parse_sequences(os.path.join(INP, "mixed.fa")))
    assert [r.id for r in recs] == ["rec1", "rec2", "rec3", "rec4", "rec5", "rec6"]
    assert recs[0].description == "rec1 first record, DNA letters" and len(recs[4].seq) == 0
    assert len(recs[5].seq) == 400                       # wrapped lines are joined
    assert [len(b) for b in ms.batch_iterator(iter(range(1, 8)), 3)] == [3, 3, 1]
    assert list(ms.batch_iterator(iter([]), 3)) == []


def test_gzip_fasta(tmp_path):
    import gzip
    from rnascan_b200 import rnascan as ms
    p = tmp_path / "x.fa.gz"
    with gzip.open(p, "wt") as fh:
        fh.write(">a desc\nACGT\nAC\n>b\n\n")
    recs = list(ms.parse_sequences(str(p)))
    assert [(r.id, r.description, str(r.seq)) for r in recs] == [("a", "a desc", "ACGTAC"), ("b", "b", "")]


# ----------------------------------------------------------------------------- CLI arguments
def test_getoptions_and_mode_guess(capsys):
    from rnascan_b200 import rnascan as ms
    a = ms.getoptions(["-p", "x.pfm", "in.fa"])
    assert (a.minscore, a.cores, a.pseudocount, a.uniform_background, a.bgonly, a.debug) == \
        (6, 8, 0, False, False, False)
    assert ms._guess_seq_type(a) == "RNA"
    assert ms._guess_seq_type(ms.getoptions(["-q", "x.pfm", "in.fa"])) == "SS"
    assert ms._guess_seq_type(ms.getoptions(["-p", "a", "-q", "b", "s.fa", "t.fa"])) == "RNASS"
    assert ms._guess_seq_type(ms.getoptions(["-p", "a", "-q", "b", "-t", "ACGU,EEEE"])) == "RNASS"
    assert ms.getoptions(["-p", "a", "-m", " -inf", "x.fa"]).minscore == float("-inf")
    with pytest.raises(SystemExit):
        ms.getoptions(["in.fa"])
    with pytest.raises(SystemExit):
        ms.getoptions(["-p", "a", "-u", "-b", "bg.txt", "x.fa"])
    with pytest.raises(SystemExit):
        ms._guess_seq_type(ms.getoptions(["-p", "a", "-q", "b", "only_one.fa"]))
    capsys.readouterr()


def test_load_background_file_and_uniform(in_repo, capsys):
    from rnascan_b200 import rnascan as ms
    bg = ms.load_background(os.path.join(INP, "bg_seq_custom.txt"), False)
    assert bg == {"A": 0.3, "C": 0.2, "G": 0.2, "U": 0.3}
    assert ms.load_background(None, True) is None
    err = capsys.readouterr().err
    assert "Reading custom background probabilities from" in err


# ----------------------------------------------------------------------------- pfmutil
def test_pfmutil_matches_the_reference(golden_api, tmp_path):
    from rnascan_b200 import pfmutil as pu
    V = golden_api["pfmutil"]
    struct = pu.read_pfm(os.path.join(INP, "SLBP_pfm_assembled_normalized_struct.txt"))
    seq = pu.read_pfm(os.path.join(INP, "test_seq_pfm.txt"))
    assert struct == V["read_struct"]
    assert pu.format_pfm(struct) == V["format_struct"] and pu.format_pfm(seq) == V["format_seq"]
    assert pu.norm_pfm(seq) == V["norm_seq"]
    assert [pu.is_normalized(seq), pu.is_normalized(pu.norm_pfm(seq)), pu.is_normalized(struct)] == V["is_normalized"]
    assert pu.pfm_from_IUPAC("ACGURYSWKMBDHVN") == V["from_IUPAC"]
    assert pu.pfm_from_string("EHLLRT", pu.FULL_STRUCT_ALPHABET) == V["from_string"]
    with pytest.raises(Exception):
        pu.pfm_from_string("EHX", pu.FULL_STRUCT_ALPHABET)
    assert pu.pfm_to_pwm(pu.norm_pfm(seq), 20) == V["to_pwm_seq_20"]
    assert pu.reduce_pfm_alphabet(struct) == V["reduce_struct"]
    f = str(tmp_path / "multi.txt")
    pu.write_multi_pfm(["m1", "m2"], [seq, struct], f)
    assert open(f).read() == V["multi_text"]
    got = [[i, copy.deepcopy(pfm)] for i, pfm in pu.multi_pfm_iter(f)]
    assert got == V["multi_iter"]
    g = str(tmp_path / "one.txt")
    pu.write_pfm(struct, g)
    assert pu.read_pfm(g) == struct


# ----------------------------------------------------------------------------- sharding
def _check_plan(lengths, R, W):
    from rnascan_b200 import shard
    plan = shard.plan_shards(lengths, R, W)
    assert len(plan) == R
    own = [np.zeros(max(L, 1), int) for L in lengths]
    cnt = [np.zeros(max(L, 1), int) for L in lengths]
    order = []
    for pieces in plan:
        for (r, a, b, o) in pieces:
            order.append((r, a))
            L = lengths[r]
            last = o >= b
            hi = (b - W + 1) if last else o
            assert 0 <= a <= b <= L
            if not last:
                assert b == min(L, o + W - 1)
            own[r][a:max(a, hi)] += 1
            cnt[r][a:a + shard.owned_symbols((r, a, b, o))] += 1
    assert order == sorted(order)
    for r, L in enumerate(lengths):
        nw = max(0, L - W + 1)
        assert (own[r][:nw] == 1).all() and (own[r][nw:L] == 0).all()
        assert (cnt[r][:L] == 1).all()
    return plan


def test_shard_plan_owns_every_window_once():
    rng = np.random.default_rng(0)
    for trial in range(300):
        n = int(rng.integers(1, 30))
        lengths = rng.integers(0, 200, size=n).tolist()
        if trial % 5 == 0:
            lengths[int(rng.integers(0, n))] = 5000
        _check_plan(lengths, int(rng.integers(1, 9)), int(rng.integers(1, 20)))
    _check_plan([], 4, 7)
    _check_plan([0, 0, 0], 2, 7)
    plan = _check_plan([1_000_000], 8, 7)                 # one long record is split 8 ways
    loads = [sum(b - a for (_, a, b, _) in p) for p in plan]
    assert max(loads) - min(loads) <= 16 and all(len(p) == 1 for p in plan)


_WORKER = r"""
import os, sys, json
sys.path.insert(0, %(repo)r)
import numpy as np
import torch.distributed as dist
from rnascan_b200 import shard, synth
rank, size = shard.init("gloo")
rng = np.random.default_rng(5)
lengths = synth.record_lengths(200000, 40, rng)
codes, offsets = synth.rna_codes(lengths, rng, n_frac=0.01)
W = 7
plan = shard.plan_shards(lengths, size, W)
counts = np.zeros(8, np.int64)
starts = []
for piece in plan[rank]:
    r, a, b, o = piece
    seg = codes[offsets[r] + a: offsets[r] + b]
    k = shard.owned_symbols(piece)
    counts += np.bincount(seg[:k][seg[:k] < 8], minlength=8)      # stand-in for rs_hist on this rank's shard
    hi = (b - W + 1) if o >= b else o
    starts.extend((r, i) for i in range(a, max(a, hi)))
total = shard.allreduce_counts(counts)
gathered = shard.gather_objects(starts)
if rank == 0:
    flat = [x for part in gathered for x in part]
    want_counts = np.bincount(codes[codes < 8], minlength=8)
    want = [(r, i) for r, L in enumerate(lengths.tolist()) for i in range(max(0, L - W + 1))]
    print(json.dumps({"counts_ok": bool((total == want_counts).all()), "order_ok": flat == want,
                      "n": len(flat), "size": size}))
dist.destroy_process_group()
"""


def test_two_rank_gloo_allreduce_and_ordered_gather(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % {"repo": REPO})
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", OMP_NUM_THREADS="1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29533", str(script)],
                         capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    import json
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    res = json.loads(line)
    assert res == {"counts_ok": True, "order_ok": True, "n": res["n"], "size": 2} and res["n"] > 100000


def test_numpy_strided_dot_is_the_pinned_arithmetic(oracle):
    """The averaged-profile oracle pins OpenBLAS' strided ddot arithmetic; check that numpy on
    THIS machine still computes it that way (skip, not fail, on a different BLAS build)."""
    rng = np.random.default_rng(3)
    prof = np.asfortranarray(rng.random((200, 7)))
    tab = np.asfortranarray(rng.normal(size=(5, 7)) * 3)
    got = oracle.profile_scores(np.ascontiguousarray(prof), np.ascontiguousarray(tab))
    want = oracle.profile_scores_py(prof, tab)
    if not np.array_equal(got, want):
        pytest.skip("this machine's BLAS uses a different ddot kernel than the one the golden vectors pin")


def test_c_log_odds_helper_is_bit_identical_to_the_python_path():
    from rnascan_b200 import motifs
    rng = np.random.default_rng(11)
    letters = "GAUC"
    for trial in range(50):
        W = int(rng.integers(1, 13))
        counts = {l: rng.dirichlet(0.3 * np.ones(4), size=W)[:, k].tolist() for k, l in enumerate(letters)}
        if trial % 4 == 0:
            counts["A"][0] = 0.0
        pc = 0.0 if trial % 4 == 0 else 0.01
        prob = motifs.normalize_counts(counts, letters, pc)
        bgv = rng.dirichlet(np.ones(4))
        bg = {l: float(bgv[k]) for k, l in enumerate(letters)}
        want = motifs.log_odds(prob, letters, bg)
        total = sum(bg.values())
        bgn = np.array([bg[l] / total for l in letters])
        got = motifs.log_odds_table(np.array([prob[l] for l in letters]).T, bgn)
        for k, l in enumerate(letters):
            assert same(got[:, k], want[l])


# ----------------------------------------------------------------------------- dot-bracket annotation
def test_structure_annotation_matches_the_reference_tool():
    """tests/golden/dotbracket.json holds the output of the reference's own C++ program
    (scripts/parse_secondary_structure.cpp) for 400+ structures."""
    import json
    from rnascan_b200 import structure
    with open(os.path.join(REPO, "tests", "golden", "dotbracket.json")) as fh:
        cases = json.load(fh)
    got = structure.parse_many([c[0] for c in cases])
    assert got == [c[1] for c in cases]
    assert set("".join(got)) == set("BEHLMRT")
    assert structure.parse("..((...))..") == "EELLHHHRREE"
    for bad in ("((..)", "())(", "((.x.))"):
        with pytest.raises(ValueError):
            structure.parse(bad)
    assert structure.parse_many([]) == []


def test_structure_annotation_fuzz_against_the_reference_binary(tmp_path):
    """tests/golden/dotbracket_fuzz.txt.gz holds the output of the reference's own C++ program for the seeded
    structures below; when the program is built (oracle/Makefile, `make ref`) it is also run on them here."""
    import gzip
    import random
    from rnascan_b200 import structure
    binary = os.path.join(REPO, "oracle", "_ref", "parse_secondary_structure")
    rnd = random.Random(5)

    def rand_struct(n):
        s, depth = [], 0
        while len(s) < n:
            r, rem = rnd.random(), n - len(s)
            if depth >= rem:
                s.append(")"); depth -= 1
            elif r < 0.3:
                s.append(".")
            elif r < 0.68 and rem > depth + 1:
                s.append("("); depth += 1
            elif depth > 0:
                s.append(")"); depth -= 1
            else:
                s.append(".")
        return "".join(s)
    structs = [s for s in (rand_struct(rnd.randint(1, 300)) for _ in range(3000)) if "." in s]
    fi, fo = tmp_path / "in.txt", tmp_path / "out.txt"
    fi.write_text("\n".join(structs) + "\n")
    with gzip.open(os.path.join(REPO, "tests", "golden", "dotbracket_fuzz.txt.gz"), "rt") as fh:
        want = fh.read()
    if os.path.exists(binary):
        subprocess.check_call([binary, str(fi), str(fo)])
        assert fo.read_text() == want
    assert len(structs) == 2989 and want.split("\n")[:-1] == structure.parse_many(structs)
    # file interface of the tool
    out2 = tmp_path / "out2.txt"
    structure.parse_file(str(fi), str(out2))
    assert out2.read_text() == want


def test_structure_annotation_is_linear_time():
    """The reference is O(L^2) (nested pair search, enclosing-pair scan); 2 M nested symbols here."""
    import time
    from rnascan_b200 import structure
    n = 1_000_000
    s = "(" * n + "...." + ")" * n
    t0 = time.perf_counter()
    a = structure.parse(s)
    assert time.perf_counter() - t0 < 5.0
    assert a == "L" * n + "HHHH" + "R" * n


def test_profile_averaging_matches_the_reference():
    """struct_pfm_from_aligned + norm_pfm (the post-RNAfold half of run_folding) against outputs of the
    reference's own functions, and the profile text format the scan reads back."""
    import json
    from rnascan_b200 import structure, pfmutil
    with open(os.path.join(REPO, "tests", "golden", "averaging.json")) as fh:
        cases = json.load(fh)
    for c in cases:
        assert structure.struct_pfm_from_aligned(c["sequences"]) == c["counts"]
        prof = structure.profile_from_aligned(c["sequences"])
        assert prof == c["profile"]
        assert pfmutil.format_pfm(prof) == c["text"]
    with pytest.raises(KeyError):
        structure.struct_pfm_from_aligned(["EEX-", "EEH-"])
    # fragments -> annotate -> align -> average
    prof = structure.profile_from_fragments(11, [(-3, "((...))"), (2, "..((...))"), (4, "(....)")])
    assert all(abs(sum(prof[l][i] for l in prof) - 1.0) < 1e-12 for i in range(11))
    assert prof["L"][0] == 1.0 and prof["E"][2] == 0.5


# ----------------------------------------------------------------------------- native hits.tab writer
def test_native_writer_text_equals_pandas_to_csv():
    """rs_host_format_hits vs DataFrame.to_csv on random rows: float32 text, widened float32,
    Python round(x, 3) of float64, unrounded float64 (incl. huge/small magnitudes), csv quoting."""
    import io
    import pandas as pd
    from rnascan_b200 import rnascan as ms
    rng = np.random.default_rng(0)
    n, W = 5000, 5
    ids = ["id%d" % k for k in range(7)] + ['we"ird', "tab\there"]
    descs = ["desc %d" % k for k in range(7)] + ['has "quotes" inside', ""]
    blobs = ms._StringBlobs(ids, descs)
    rec = np.sort(rng.integers(0, len(ids), size=n))
    start0 = rng.integers(0, 10_000_000, size=n)
    raw = rng.choice(np.frombuffer(b"ACGUN", np.uint8), size=4096)
    tpos = rng.integers(0, 4096 - W, size=n)
    frags = [raw[p:p + W].tobytes().decode() for p in tpos]
    f32 = np.round((rng.normal(size=n) * 30).astype(np.float32), 3)
    f32[:5] = [0.0, -0.0, 0.001, 123456.7, -999.999]
    f64 = rng.normal(size=n) * 30
    f64[:8] = [0.0005, 2.0005, 1e-7, -1.7976931348623157e308, 1234567.891, 2.5, -0.00049, 1e15]

    def frame(scores):
        return pd.DataFrame({"Sequence_ID": np.array(ids, object)[rec], "Description": np.array(descs, object)[rec],
                             "Motif_ID": "m", "Start": start0 + 1, "End": start0 + W, "Sequence": frags,
                             "LogOdds": scores, "Match_ID": np.arange(1, n + 1)})

    def csv(df):
        b = io.StringIO()
        df.to_csv(b, sep="\t", index=False, header=False)
        return b.getvalue()
    for kind, arr, col in ((0, f32, f32), (1, f32, f32.astype(object)),
                           (2, f64, np.array([round(v, 3) for v in f64.tolist()], dtype=object))):
        got = ms._native_rows(n, 1, rec, blobs, None, "m", None, start0, W, raw, None, tpos, kind,
                              np.ascontiguousarray(arr), None, None)
        assert got == csv(frame(col)), kind
    # combined rows: float32 + unrounded float64 + their sum
    got = ms._native_rows(n, 1, rec, blobs, None, "ms", "mq", start0, W, raw, None, tpos, 0, f32, 3, f64)
    df = pd.DataFrame({"Sequence_ID": np.array(ids, object)[rec], "Description.Seq": np.array(descs, object)[rec],
                       "Motif_ID.Seq": "ms", "Start": start0 + 1, "End": start0 + W, "Sequence.Seq": frags,
                       "LogOdds.Seq": f32, "Description.Struct": "", "Motif_ID.Struct": "mq",
                       "Sequence.Struct": ".", "LogOdds.Struct": f64})
    df["LogOdds.SeqStruct"] = df["LogOdds.Seq"] + df["LogOdds.Struct"]
    df["Match_ID"] = np.arange(1, n + 1)
    assert got == csv(df)
    # out-of-range float32 text is declined (the caller falls back to pandas)
    bad = f32.copy()
    bad[3] = 3e9
    assert ms._native_rows(n, 1, rec, blobs, None, "m", None, start0, W, raw, None, tpos, 0, bad, None, None) is None


# ----------------------------------------------------------------------------- native FASTA ingest
@pytest.mark.parametrize("min_chunk", [None, "48"], ids=["one-chunk", "many-chunks"])
def test_native_fasta_ingest_equals_the_python_parser(tmp_path, monkeypatch, min_chunk):
    """rs_host_fasta_index/_fill vs the Biopython-semantics Python parser (seq.iter_fasta + preprocess_seq +
    pack_texts) on hostile FASTA text: CRLF / lone CR, blank lines, leading junk, blanks inside lines,
    lower case, T/U, ambiguity codes, empty records, empty titles, no trailing newline, gzip.
    "many-chunks": the buffer is cut into up to 8 pieces at record starts and parsed on threads."""
    if min_chunk:
        monkeypatch.setenv("RNASCAN_FASTA_MIN_CHUNK", min_chunk)
        monkeypatch.setenv("RNASCAN_HOST_THREADS", "8")
    import gzip
    import random
    from rnascan_b200 import rnascan as ms, device
    from rnascan_b200.seq import IUPAC
    from rnascan_b200.BioAddons.Alphabet import ContextualSecondaryStructure
    rnd = random.Random(3)

    def fake(k):
        out = ["junk before the first record\n", "more junk\n"] if k % 3 == 0 else []
        for r in range(rnd.randint(0, 12)):
            title = rnd.choice(["", "id%d" % r, "id%d some words\t tabbed " % r, "  leading blank %d" % r,
                                "id%d\x1c odd" % r])
            out.append(">" + title + rnd.choice(["\n", "\r\n", "\r", " \n", "\t\n"]))
            for _ in range(rnd.randint(0, 6)):
                line = "".join(rnd.choice("ACGTUacgtunNRY-BEHLMRTbehlmrt. ") for _ in range(rnd.randint(0, 70)))
                out.append(line + rnd.choice(["\n", "\r\n", "\r", "  \n", "\n\n"]))
        text = "".join(out)
        return text[:-1] if (k % 4 == 0 and text.endswith("\n")) else text

    def python_path(path, alphabet, kind):
        recs = list(ms.parse_sequences(path))
        texts = [str(ms.preprocess_seq(r, alphabet)) for r in recs]
        codes, off, ln = device.pack_texts(texts, kind)
        return [r.id for r in recs], [r.description for r in recs], texts, codes, off, ln

    for k in range(40):
        path = str(tmp_path / ("f%d.fa%s" % (k, ".gz" if k % 5 == 0 else "")))
        data = fake(k).encode("ascii")
        if path.endswith(".gz"):
            with gzip.open(path, "wb") as fh:
                fh.write(data)
        else:
            with open(path, "wb") as fh:
                fh.write(data)
        for alphabet, kind in ((IUPAC.IUPACUnambiguousRNA(), "rna"), (ContextualSecondaryStructure(), "struct")):
            ids, descs, texts, codes, off, ln = python_path(path, alphabet, kind)
            data_b = ms._read_fasta_bytes(path)
            buf = np.frombuffer(data_b, np.uint8)
            sizes = np.zeros(3, np.int64)
            from rnascan_b200 import _lib
            _lib.check(_lib.lib.rs_host_fasta_index(buf.ctypes.data if len(buf) else 0, len(buf), sizes[0:].ctypes.data,
                                                    sizes[1:].ctypes.data, sizes[2:].ctypes.data))
            n_rec, n_sym, n_title = (int(v) for v in sizes)
            assert n_rec == len(ids) and n_sym == int(ln.sum())
            text = np.empty(max(n_sym + n_rec, 1), np.uint8); cds = np.empty(max(n_sym + n_rec, 1), np.uint8)
            o = np.zeros(max(n_rec, 1), np.int64); l = np.zeros(max(n_rec, 1), np.int64)
            titles = np.empty(max(n_title, 1), np.uint8); toff = np.zeros(n_rec + 1, np.int64)
            _lib.check(_lib.lib.rs_host_fasta_fill(buf.ctypes.data if len(buf) else 0, len(buf), 0 if kind == "rna" else 1,
                                                   text.ctypes.data, cds.ctypes.data, o.ctypes.data, l.ctypes.data,
                                                   titles.ctypes.data, toff.ctypes.data))
            assert np.array_equal(cds[:n_sym + n_rec], codes), (k, kind)
            assert np.array_equal(o[:n_rec], off) and np.array_equal(l[:n_rec], ln)
            assert text[:n_sym + n_rec].tobytes().decode() == "".join(t + "\n" for t in texts)
            blob = titles[:n_title].tobytes().decode()
            got_desc = [blob[a:b] for a, b in zip(toff[:-1].tolist(), toff[1:].tolist())]
            assert got_desc == descs
            assert [(d.split(None, 1) or [""])[0] for d in got_desc] == ids


# ----------------------------------------------------------------------------- native profile ingest
def _pandas_column(tokens):
    """What pandas.read_csv makes of the tokens as ONE tab-separated float column (its default converter)."""
    import io
    import pandas as pd
    return pd.read_csv(io.StringIO("x\n" + "\n".join(tokens) + "\n"), sep="\t", dtype={"x": np.float64})["x"].to_numpy()


def test_native_number_conversion_equals_pandas_default_converter():
    """rs_host_parse_doubles restates pandas' precise_xstrtod (not correctly rounded!): bit-identical to
    pd.read_csv on profile-like values, random doubles of every magnitude and over-long digit strings."""
    import random
    from rnascan_b200 import _lib
    rng = np.random.default_rng(20261018)
    vals = []
    counts = rng.integers(0, 21, size=(60_000, 7)).astype(float)
    counts /= np.maximum(counts.sum(1, keepdims=True), 1)               # what run_folding writes: normalised counts
    vals += counts.ravel().tolist()
    vals += rng.random(150_000).tolist()
    vals += (10.0 ** rng.uniform(-320, 308, 100_000)).tolist()
    vals += (-(10.0 ** rng.uniform(-30, 30, 20_000))).tolist()
    vals += [0.0, -0.0, 1.0, 1e-5, 5e-324, 2.2250738585072014e-308, 1.7976931348623157e308, 0.1, 0.2, 0.3, 1 / 3]
    tokens = [repr(v) for v in vals]
    rnd = random.Random(7)
    for _ in range(60_000):
        tokens.append("0." + "".join(rnd.choice("0123456789") for _ in range(rnd.randint(1, 25))))
    for _ in range(30_000):
        tokens.append("".join(rnd.choice("0123456789") for _ in range(rnd.randint(1, 15))) + "." +
                      "".join(rnd.choice("0123456789") for _ in range(rnd.randint(0, 9))))
    tokens += ["1e5", "1E-3", "+.5", "5.", "-12.50e+2", "007", "123456789012345", ".000000000000000000001", "1e-400", "3e-700"]
    want = _pandas_column(tokens)
    text = "\n".join(tokens).encode()
    got = np.zeros(len(tokens), np.float64)
    ok = np.zeros(len(tokens), np.uint8)
    n_out = np.zeros(1, np.int64)
    _lib.check(_lib.lib.rs_host_parse_doubles(text, len(text), got.ctypes.data, len(got), n_out.ctypes.data,
                                              ok.ctypes.data))
    assert int(n_out[0]) == len(tokens) and ok.all()
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
    # the converter is genuinely pandas', not strtod: a large share of these tokens convert differently
    exact = np.array([float(t) for t in tokens])
    assert (got.view(np.uint64) != exact.view(np.uint64)).mean() > 0.2
    # tokens the native converter must decline (pandas decides what they are)
    bad = ["", "-", "e5", "1e", "nan", "inf", "1,5", " 1.0", "1.0 ", "0x10", "1e999999", "1234567890123456", "1e400", "--1"]
    text = "\n".join(bad).encode()
    ok = np.ones(len(bad), np.uint8)
    got = np.zeros(len(bad), np.float64)
    _lib.check(_lib.lib.rs_host_parse_doubles(text, len(text), got.ctypes.data, len(got), n_out.ctypes.data,
                                              ok.ctypes.data))
    assert int(n_out[0]) == len(bad) and not ok.any()


def test_native_profile_reader_equals_pandas(tmp_path):
    """rs_host_profiles_* (through rnascan._read_profiles_packed) == pd.read_csv per file (rnascan._read_profile),
    bit for bit, on plain files, permuted/extra columns, CRLF / CR line ends, blank lines, no final newline;
    hostile files (quotes, NaN words, ragged rows, duplicate columns, blanks) fall back to pandas."""
    from rnascan_b200 import pfmutil, rnascan
    rng = np.random.default_rng(5)
    files, kinds = [], []

    def write(name, text, kind, binary=False):
        path = str(tmp_path / ("structure.%s.txt" % name))
        with open(path, "wb") as fh:
            fh.write(text if binary else text.encode())
        files.append(path)
        kinds.append(kind)

    def table(L, order="BEHLMRT", extra=None, eol="\n", final_eol=True, blank_every=0):
        rows = rng.integers(0, 30, size=(L, 7)).astype(float)
        rows /= np.maximum(rows.sum(1, keepdims=True), 1)
        cols = ["PO"] + list(order) + ([extra] if extra else [])
        lines = ["\t".join(cols)]
        for i in range(L):
            vals = {c: repr(float(rows[i, "BEHLMRT".index(c)])) for c in "BEHLMRT"}
            f = [str(i)] + [vals[c] for c in order] + (["7"] if extra else [])
            lines.append("\t".join(f))
            if blank_every and i % blank_every == 0:
                lines.append("")
        return eol.join(lines) + (eol if final_eol else "")

    for k in range(6):                                            # what pfmutil.write_pfm produces
        rows = rng.random((int(rng.integers(1, 400)), 7))
        pfm = {c: [float(v) for v in rows[:, j]] for j, c in enumerate("BEHLMRT")}
        path = str(tmp_path / ("structure.w%d.txt" % k))
        pfmutil.write_pfm(pfm, path)
        files.append(path); kinds.append("native")
    write("perm", table(50, order="TRMLHEB"), "native")
    write("extra", table(40, extra="Z"), "native")
    write("crlf", table(30, eol="\r\n"), "native")
    write("cr", table(30, eol="\r"), "native")
    write("noeol", table(20, final_eol=False), "native")
    write("blank", "\n\n" + table(25, blank_every=4), "native")
    write("ints", "PO\tB\tE\tH\tL\tM\tR\tT\n0\t1\t0\t0\t0\t0\t0\t0\n1\t0\t0\t1\t0\t0\t0\t0\n", "native")
    write("exp", "PO\tB\tE\tH\tL\tM\tR\tT\n0\t1e-05\t2.5E-3\t0.1\t0.2\t0.3\t.25\t5.\n", "native")
    write("quoted", 'PO\tB\tE\tH\tL\tM\tR\tT\n0\t"0.25"\t0.2\t0.3\t0.1\t0.1\t0.05\t0.0\n1\t0.5\t0.5\t0\t0\t0\t0\t0\n', "pandas")
    write("nanword", "PO\tB\tE\tH\tL\tM\tR\tT\n0\tnan\t0.2\t0.3\t0.1\t0.1\t0.05\t0.0\n1\t0.5\tNA\t0\t0\t0\t0\tinf\n", "pandas")
    write("missing", "PO\tB\tE\tH\tL\tM\tR\tT\n0\t0.1\t\t0.3\t0.1\t0.1\t0.1\t0.3\n", "pandas")
    write("short", "PO\tB\tE\tH\tL\tM\tR\tT\n0\t0.1\t0.2\t0.3\t0.1\t0.1\t0.1\n", "pandas")
    write("spaces", "PO\tB\tE\tH\tL\tM\tR\tT\n0\t 0.1\t0.2 \t0.3\t0.1\t0.1\t0.1\t0.1\n", "pandas")
    write("bigint", "PO\tB\tE\tH\tL\tM\tR\tT\n0\t12345678901234567\t0\t0\t0\t0\t0\t0\n", "pandas")
    packed, lengths = rnascan._read_profiles_packed(files, threads=4)
    off = 0
    for path, L in zip(files, lengths.tolist()):
        want = rnascan._read_profile(path)
        assert want.shape == (L, 7), path
        got = packed[off:off + L]
        nan = np.isnan(want)
        assert np.array_equal(np.isnan(got), nan), path
        assert np.array_equal(got[~nan].view(np.uint64), want[~nan].view(np.uint64)), path
        assert not packed[off + L].any()                           # separator row
        off += L + 1
    assert off == packed.shape[0]
    # which files the native reader really took (the others went through pandas)
    import ctypes
    from rnascan_b200 import _lib
    arr = (ctypes.c_char_p * len(files))(*[os.fsencode(f) for f in files])
    handle = ctypes.c_void_p()
    rows = np.zeros(len(files), np.int64)
    _lib.check(_lib.lib.rs_host_profiles_open(ctypes.cast(arr, ctypes.c_void_p), len(files), 2, ctypes.byref(handle),
                                              rows.ctypes.data))
    offs = np.concatenate([[0], np.cumsum(np.maximum(rows, 0)[:-1] + 1)]).astype(np.int64)
    out = np.zeros((int(np.maximum(rows, 0).sum()) + len(files), 7))
    status = np.zeros(len(files), np.int32)
    _lib.check(_lib.lib.rs_host_profiles_fill(handle, 2, out.ctypes.data, offs.ctypes.data, status.ctypes.data))
    _lib.lib.rs_host_profiles_close(handle)
    took = [(r >= 0 and s == 0) for r, s in zip(rows.tolist(), status.tolist())]
    assert took == [k == "native" for k in kinds], list(zip(files, took, kinds))


def test_background_shift_bounds_the_score_difference_between_two_backgrounds():
    """device._background_shift: W x it bounds |score(b_local) - score(b_global)| for every window (the slack the
    sharded one-hot scan verifies before trusting a decision pass started from the shard's own counts)."""
    import math
    from rnascan_b200 import device
    rng = np.random.default_rng(11)
    for A in (4, 7):
        for _ in range(50):
            local = np.zeros(8, np.int64); glob = np.zeros(8, np.int64)
            local[:A] = rng.integers(0, 10_000, A)
            glob[:A] = local[:A] + rng.integers(0, 50_000, A)
            shift = device._background_shift(local, glob, A)
            def bg(c):
                b = [(float(c[k]) + 1) / (float(sum(int(v) for v in c[:A])) + A) for k in range(A)]
                t = sum(b)
                return [v / t for v in b]
            bl, bgl = bg(local), bg(glob)
            worst = max(abs(math.log2(bl[k]) - math.log2(bgl[k])) for k in range(A))
            assert worst <= shift <= worst * 1.001 + 1e-9
    same = np.array([5, 6, 7, 8, 0, 0, 0, 0], np.int64)
    assert device._background_shift(same, same, 4) < 1e-9


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the reference's own CPU call pattern on a bounded sample) prints exactly ONE JSON
    line on stdout with the contract's keys; no GPU involved."""
    import json
    env = dict(os.environ, RNASCAN_REF_STEP_SECONDS="0.3")
    proc = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "1",
                           "--warmup", "0", "--workload", "c2"], capture_output=True, text=True, env=env, timeout=600)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [l for l in proc.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, proc.stdout
    out = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "gpu_launches", "cpu_baseline", "e2e"):
        assert key in out, key
    assert out["impl"] == "reference" and out["gpu_launches"] == 0 and out["value"] > 0
    assert out["cpu_baseline"]["kind"] in ("reference", "port") and out["cpu_baseline"]["cores"] >= 1
    assert out["e2e"]["h2d_bytes_per_step"] == 0 and out["e2e"]["value"] == out["value"]
    assert "workload" in out["config"]


def test_bench_dump_outputs_keeps_float32_and_samples_large_outputs(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: float32 stays float32, anything else is written as float64; per-hit arrays above
    the cap are cut to one seeded, ascending sample (written as sample_index), the same on every run and for
    numpy arrays and tensors alike -- so that the dumps of two builds can be compared."""
    import torch
    import bench
    load = lambda d: {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}
    bench.dump_outputs(str(tmp_path / "small"), {"position": np.arange(10), "seq_score": np.ones(10, np.float32)},
                       {"counts": np.arange(8)})
    got = load(tmp_path / "small")
    assert sorted(got) == ["counts", "position", "seq_score"] and got["position"].tolist() == list(range(10))
    assert got["seq_score"].dtype == np.float32 and got["position"].dtype == got["counts"].dtype == np.float64
    monkeypatch.setattr(bench, "DUMP_ENTRY_BYTES", 12000)
    pos, sc = np.arange(5000) * 3, np.arange(5000, dtype=np.float32)      # 5000 entries of 12 bytes
    bench.dump_outputs(str(tmp_path / "a"), {"position": pos, "seq_score": sc}, {"counts": np.arange(8)})
    bench.dump_outputs(str(tmp_path / "b"), {"position": torch.from_numpy(pos), "seq_score": torch.from_numpy(sc)},
                       {"counts": torch.arange(8)})
    a, b = load(tmp_path / "a"), load(tmp_path / "b")
    idx = a["sample_index"]
    assert idx.dtype == np.float64 and len(idx) == 12000 // (12 + 8) and (np.diff(idx) > 0).all()
    assert np.array_equal(a["position"], idx * 3) and np.array_equal(a["seq_score"], idx.astype(np.float32))
    assert a["position"].nbytes + a["seq_score"].nbytes + idx.nbytes <= 12000
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) and a[k].dtype == b[k].dtype for k in a)


def test_pfm_reader_without_pandas_equals_pandas_or_declines(tmp_path):
    """rnascan._read_pfm_counts (PFM tables without importing pandas) must give exactly what
    pd.read_csv(...).drop(first column).to_dict("list") gives -- same keys, same Python types, same bits --
    or decline (None) and leave the file to pandas.  Random tables in many number formats, plus the oddities
    it has to decline."""
    import pandas as pd
    from rnascan_b200 import rnascan as ms
    rng = np.random.default_rng(77)

    def token(kind):
        v = float(rng.random()) * float(rng.choice([1.0, 1e-3, 37.0, 1e5]))
        if kind == 0:
            return repr(v)
        if kind == 1:
            return "%.17g" % v
        if kind == 2:
            return "%.4f" % v
        if kind == 3:
            return "%d" % int(v * 10)
        if kind == 4:
            return "%.3e" % v
        if kind == 5:
            return "-" + repr(v)
        if kind == 6:
            return ("%.6f" % v).lstrip("0") or "0"          # ".123456"
        if kind == 7:
            return "%d." % int(v)
        return str(rng.choice(["nan", "inf", "", " 0.5", "0.5 ", "1e400", "0x10", "1,5", "12345678901234567890", "abc"]))

    n_equal = n_declined = 0
    for case in range(400):
        ncol = int(rng.integers(2, 9))
        nrow = int(rng.integers(1, 9))
        letters = list(rng.permutation(list("ACGUBEHLMRT"))[:ncol - 1])
        header = ["PO"] + letters
        odd = rng.random() < 0.25
        col_kind = [int(rng.integers(0, 8)) for _ in range(ncol)]
        lines = ["\t".join(header)]
        for r in range(nrow):
            fields = [str(r + 1)]
            for c in range(1, ncol):
                kind = col_kind[c] if rng.random() < 0.8 else int(rng.integers(0, 8))
                if odd and rng.random() < 0.1:
                    kind = 8
                fields.append(token(kind))
            lines.append("\t".join(fields))
        text = "\n".join(lines) + ("\n" if rng.random() < 0.8 else "")
        if rng.random() < 0.1:
            text = text.replace("\n", "\r\n")
        if rng.random() < 0.05:
            text = text.replace("\n", "\n\n", 1)                     # a blank line (pandas skips it)
        if odd and rng.random() < 0.2:
            text = text.replace("\t", "\t\t", 1)                     # a ragged header or row
        path = tmp_path / ("pfm%d.txt" % case)
        path.write_bytes(text.encode("ascii"))
        got = ms._read_pfm_counts(str(path))
        if got is None:
            n_declined += 1
            continue
        table = pd.read_csv(str(path), sep="\t")
        want = table.drop(columns=table.columns[0]).to_dict(orient="list")
        assert list(got) == list(want), (case, text)
        for name in got:
            assert len(got[name]) == len(want[name]), (case, name, text)
            for a, b in zip(got[name], want[name]):
                assert type(a) is type(b), (case, name, a, b, text)
                if isinstance(a, float):
                    assert np.float64(a).view(np.uint64) == np.float64(b).view(np.uint64), (case, name, a, b)
                else:
                    assert a == b
        n_equal += 1
    assert n_equal > 200 and n_declined > 20, (n_equal, n_declined)
    # a multi-PFM block goes through the same reader
    block = ms._PfmBlock("m1", "PO\tA\tC\tG\tU\n1\t0.1\t0.2\t0.3\t0.4\n", "x.multi")
    assert ms._read_pfm_counts(block) == {"A": [0.1], "C": [0.2], "G": [0.3], "U": [0.4]}
