"""Host side of scoring single-letter alphabets other than GAUC and BEHLMRT: the alphabet-layout encoder
(rs_host_encode_alpha) against a Python restatement, the alphabet rules, and the host logic of scan_main /
compute_background on such alphabets -- in one process and over two gloo ranks -- with the device functions
replaced by oracle stand-ins defined here (tests/oracle_backend.py provides the rest of the stand-in device)."""
import argparse
import json
import os
import subprocess
import sys
import warnings

import numpy as np
import pytest

from oracle import oracle as orc
from oracle_backend import install
from rnascan_b200 import device, pfmutil, rnascan as ms, seq, _lib

ALPHABETS = ["HSTC", "EHIMP", "ACDFGIK", "ACDEFGHIKLMNPQRSTVWY", "ABCDEFGHIJKLMNOPQRSTUVWXYZ*-.@#"]
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def make_alphabet(letters):
    return type("Alpha", (seq.SingleLetterAlphabet,), {"letters": letters})()


def layout(byte, letters):
    """The alphabet layout of rnascan_b200.h, restated."""
    c = chr(byte)
    if c in letters:
        return letters.index(c)
    if "a" <= c <= "z" and c.upper() in letters:
        return letters.index(c.upper()) | _lib.RS_ALPHA_LOWER
    return _lib.RS_ALPHA_OTHER


# ----------------------------------------------------------------------------- encoder + rules
@pytest.mark.parametrize("letters", ALPHABETS)
def test_encoder_matches_layout(letters):
    text = bytes(range(256)).decode("latin-1")
    codes, off, ln = device.pack_texts([text, letters.lower() + letters, ""], device.AlphaKind(letters))
    assert codes[0:256].tolist() == [layout(b, letters) for b in range(256)]
    assert codes[256] == _lib.RS_SEP and codes[-1] == _lib.RS_SEP and off.tolist() == [0, 257, 257 + 2 * len(letters) + 1]
    second = codes[257:257 + 2 * len(letters)]
    assert second.tolist() == [layout(ord(c), letters) for c in letters.lower() + letters]
    assert ((codes[:-1] & 31) != 31).sum() == sum(c in letters or c.upper() in letters for c in text) + 2 * len(letters)


@pytest.mark.parametrize("letters", ["", "ab", "Ab", "AA", "A" * 32, "".join(chr(65 + k) for k in range(32)),
                                     "ABé", None])
def test_unsupported_alphabets_name_the_rule(letters):
    with pytest.raises(NotImplementedError, match="1 to 31 distinct single ASCII characters"):
        device.AlphaKind(letters)
    with pytest.raises(NotImplementedError, match="1 to 31"):
        ms._kind_of(make_alphabet(letters))


def test_encoder_rejects_bad_letters():
    codes = np.zeros(4, np.uint8)
    for letters in (b"ab", b"AA", b"", b"A" * 32, b"\xe9"):
        rc = _lib.lib.rs_host_encode_alpha(b"ABCD", 4, letters, len(letters), codes.ctypes.data)
        assert rc == _lib.RS_ERR_INVALID and _lib.last_error()


def test_kinds_of_alphabets():
    from rnascan_b200.BioAddons.Alphabet import ContextualSecondaryStructure
    assert ms._kind_of(seq.IUPAC.IUPACUnambiguousRNA()) == "rna"
    assert ms._kind_of(ContextualSecondaryStructure()) == "struct"
    assert ms._kind_of(make_alphabet("TRMLHEB")) == "struct"
    assert ms._kind_of(seq.SecondaryStructure()) == device.AlphaKind("HSTC")
    assert ms._kind_of(make_alphabet("BEH")) == device.AlphaKind("BEH")


def test_pwm_scan_fwd_limits():
    pwm = {chr(65 + k): [0.0] for k in range(32)}
    with pytest.raises(NotImplementedError, match="up to 31"):
        pfmutil.pwm_scan_fwd(pwm, "ABC")


# ----------------------------------------------------------------------------- oracle stand-ins
def _alpha_text(stream, A):
    """Codes -> text over stand-in letters '!'.. ('!' + A - 1) (none of them a-z); lower case, other and separator
    symbols -> the letter / newline, which is what the oracle's upper-casing makes of them."""
    lut = np.full(256, ord("\n"), np.uint8)
    for k in range(A):
        lut[k] = lut[k | _lib.RS_ALPHA_LOWER] = 0x21 + k
    return lut[stream.host_codes()].tobytes(), bytes(range(0x21, 0x21 + A))


def dense_alpha(stream, table):
    import torch
    t = device._alpha_table(table)
    text, letters = _alpha_text(stream, t.shape[1])
    return torch.from_numpy(orc.alpha_scores(text, t, letters))


def scan_alpha(stream, table, threshold, capacity=None):
    sc = dense_alpha(stream, table).numpy()
    pos = orc.search_hits(sc, threshold).astype(np.int64)
    return pos, sc[pos]


def install_alpha(monkeypatch):
    """oracle_backend.install plus the alphabet kernels' stand-ins."""
    import torch
    install(monkeypatch)
    rest = device.histogram

    def histogram(stream):
        if isinstance(stream.kind, device.AlphaKind):
            c = stream.host_codes()
            return torch.from_numpy(np.array([(c == k).sum() for k in range(len(stream.kind.letters))], np.int64))
        return rest(stream)
    monkeypatch.setattr(device, "histogram", histogram)
    monkeypatch.setattr(device, "dense_alpha", dense_alpha)
    monkeypatch.setattr(device, "scan_alpha", scan_alpha)


def random_texts(letters, n_records, seed, long_record=0):
    rng = np.random.default_rng(seed)
    pool = list(letters) + [c.lower() for c in letters] + list("0189")
    lengths = rng.integers(1, 400, size=n_records).tolist()
    if long_record:
        lengths[n_records // 2] = long_record
    return ["".join(rng.choice(pool, size=ln)) for ln in lengths]


def write_fasta(path, texts):
    with open(path, "w") as fh:
        for k, t in enumerate(texts):
            fh.write(">r%d desc %d\n" % (k, k))
            for a in range(0, len(t), 70):
                fh.write(t[a:a + 70] + "\n")


def oracle_rows(texts, table, letters, thr):
    rows = []
    for k, t in enumerate(texts):
        rows += [("r%d" % k, "r%d desc %d" % (k, k)) + tuple(r)
                 for r in orc.scan_rows("mot", t, orc.alpha_scores(t, table, letters), thr)]
    return rows


def frame_rows(df):
    if len(df) == 0:
        return []
    return list(zip(df["Sequence_ID"], df["Description"], df["Motif_ID"], df["Start"].tolist(), df["End"].tolist(),
                    df["Sequence"], df["LogOdds"].tolist()))


def run_case(fasta, texts, letters, W, thr):
    """scan_main + compute_background of one FASTA: (frame rows, background) and what the oracle gives."""
    from rnascan_b200.BioAddons.motifs.matrix import ExtendedPositionSpecificScoringMatrix
    rng = np.random.default_rng(W)
    table = rng.normal(size=(W, len(letters)))
    alphabet = make_alphabet(letters)
    pm = ExtendedPositionSpecificScoringMatrix(alphabet, {c: table[:, k].tolist() for k, c in enumerate(letters)})
    ms._BATCH_CACHE.clear()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        df = ms.scan_main(fasta, {"mot": pm}, alphabet, None, argparse.Namespace(minscore=thr, debug=False))
        bg = ms.compute_background(fasta, alphabet, verbose=False)
    got = (frame_rows(df), list(bg.items()))
    want = (oracle_rows(texts, table, letters, thr), list(orc.background(texts, letters).items()))
    return got, want


@pytest.mark.parametrize("letters", ALPHABETS)
@pytest.mark.parametrize("batch_symbols", [None, 2000])
def test_scan_main_and_background_host_logic(tmp_path, monkeypatch, letters, batch_symbols):
    install_alpha(monkeypatch)
    if batch_symbols:
        monkeypatch.setattr(ms, "MAX_BATCH_SYMBOLS", batch_symbols)
    texts = random_texts(letters, 30, seed=len(letters))
    fasta = str(tmp_path / "in.fa")
    write_fasta(fasta, texts)
    for W, thr in ((1, float("-inf")), (6, 0.5), (40, 1.0)):
        got, want = run_case(fasta, texts, letters, W, thr)
        assert got == want, (letters, W, thr)
        assert W == 40 or len(want[0]) > 0


_RANK_WORKER = r"""
import json, os, sys
sys.path.insert(0, %(repo)r)
sys.path.insert(0, os.path.join(%(repo)r, "tests"))
os.chdir(%(repo)r)
import test_alphabets_cpu as t
import torch.distributed as dist
from rnascan_b200 import rnascan as ms, shard


class Patch(object):
    def setattr(self, obj, name, value):
        setattr(obj, name, value)


t.install_alpha(Patch())
rank, size = shard.init("gloo")
bad = []
for letters in %(alphabets)r:
    texts = t.random_texts(letters, 9, seed=3, long_record=5000)   # the long record is split over the ranks
    fasta = %(tmp)r + "/in_%%d.fa" %% len(letters)
    if rank == 0:
        t.write_fasta(fasta, texts)
    dist.barrier()
    for W, thr in ((1, float("-inf")), (6, 0.5), (40, 1.0)):
        got, want = t.run_case(fasta, texts, letters, W, thr)
        if rank == 0 and got != want:
            bad.append("%%s/%%d" %% (letters, W))
        if rank != 0 and (got[0] or got[1] != want[1]):
            bad.append("%%s/%%d:rank%%d" %% (letters, W, rank))
allbad = [None] * size
dist.all_gather_object(allbad, bad)
if rank == 0:
    print(json.dumps({"bad": [b for part in allbad for b in part], "size": size}))
dist.destroy_process_group()
"""


def test_scan_main_sharded_over_two_ranks(tmp_path):
    """torchrun with 2 ranks (gloo): records split over ranks with overlap, background counts all-reduced,
    rank 0 gathers the hits -- the same frame and background as the oracle."""
    script = tmp_path / "rank_worker.py"
    script.write_text(_RANK_WORKER % {"repo": REPO, "alphabets": ["EHIMP", "ACDEFGHIKLMNPQRSTVWY"],
                                      "tmp": str(tmp_path)})
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", OMP_NUM_THREADS="1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29561", str(script)],
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-3000:]
    res = json.loads([line for line in out.stdout.splitlines() if line.startswith("{")][-1])
    assert res == {"bad": [], "size": 2}
