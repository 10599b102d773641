"""GPU parity of the alphabet kernels (rs_scores_dense_alpha / rs_scan_alpha / rs_hist_alpha) and of the Python
API on top of them, for single-letter alphabets other than GAUC and BEHLMRT, against the CPU oracle
(oracle.alpha_scores / search_hits / background / scan_rows: matrix.py:25-43, rnascan.py:258-275, :440-465)
-- bit-exact scores and identical hit sets."""
import argparse
import os
import warnings

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from oracle import oracle as orc  # noqa: E402
from test_kernels_gpu import assert_same_float, _bits  # noqa: E402

ALPHABETS = {
    "HSTC": "HSTC",                                       # Bio.Alphabet.SecondaryStructure
    "EHIMP": "EHIMP",                                     # pfmutil.reduce_pfm_alphabet
    "a7": "ACDFGIK",                                      # 7 letters, not BEHLMRT: the structure instantiations
    "a8": "ACDFGIKN",                                     # the smallest TS = 32 alphabet
    "protein": "ACDEFGHIKLMNPQRSTVWY",
    "a26": "ABCDEFGHIJKLMNOPQRSTUVWXYZ",
    "a31": "ABCDEFGHIJKLMNOPQRSTUVWXYZ*-.@#",
}
NON_LETTERS = "0123456789"                                # in none of the alphabets above
WIDTHS = [1, 7, 12, 16, 33, 64]


@pytest.fixture(scope="module")
def dev():
    from rnascan_b200 import device
    device.require_cuda()
    return device


def make_alphabet(letters):
    from rnascan_b200 import seq
    return type("Alpha_" + "".join(c if c.isalnum() else "_" for c in letters), (seq.SingleLetterAlphabet,),
                {"letters": letters})()


def random_texts(letters, total, n_records, seed, lower=0.2, other=0.005):
    """Records over `letters`, a share of them lower case (where the letter has a case), a few non-letters."""
    from rnascan_b200 import synth
    rng = np.random.default_rng(seed)
    lengths = synth.record_lengths(total, n_records, rng) if n_records > 1 else np.array([total], np.int64)
    upper = np.frombuffer(letters.encode("ascii"), np.uint8)
    pool = np.concatenate([upper, np.frombuffer(letters.lower().encode("ascii"), np.uint8)])
    texts = []
    for ln in lengths.tolist():
        k = rng.integers(0, len(upper), size=ln)
        b = np.where(rng.random(ln) < lower, pool[len(upper) + k], upper[k])
        bad = rng.random(ln) < other
        b[bad] = np.frombuffer(NON_LETTERS.encode("ascii"), np.uint8)[rng.integers(0, 10, size=int(bad.sum()))]
        texts.append(b.astype(np.uint8).tobytes().decode("ascii"))
    return texts


def random_table(W, A, seed, zero_frac=0.05):
    """Log-odds (W, A): some -inf entries (zero probabilities) so that -inf windows occur."""
    from rnascan_b200 import synth
    rng = np.random.default_rng(seed)
    pfm = synth.pfm_rows(W, A, rng, alpha=1.0)
    pfm[rng.random(pfm.shape) < zero_frac] = 0.0
    top = pfm.argmax(axis=1)
    pfm[np.arange(W), top] += 0.1                         # no all-zero row
    pfm[0, (top[0] + 1) % A] = 0.0                        # at least one -inf entry
    return synth.pssm_table(pfm, pseudocount=0.0)


def oracle_stream_scores(texts, table, letters):
    """Oracle scores of the packed stream (records + one separator each, as the device lays them out)."""
    return orc.alpha_scores("\n".join(texts) + "\n", table, letters)


# ----------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("name", sorted(ALPHABETS))
@pytest.mark.parametrize("W", WIDTHS)
def test_dense_and_scan_match_oracle(dev, name, W):
    letters = ALPHABETS[name]
    kind = dev.AlphaKind(letters)
    texts = random_texts(letters, 60_000, 40, seed=W * 31 + len(letters))
    table = random_table(W, len(letters), seed=W + 7 * len(letters))
    stream = dev.SymbolStream.from_texts(texts, kind)
    want = oracle_stream_scores(texts, table, letters)
    got = dev.dense_alpha(stream, table).cpu().numpy()
    assert_same_float(got, want)
    assert np.isnan(want).any() and np.isfinite(want).any()
    assert np.isneginf(want).any() or len(letters) == 1
    finite = want[np.isfinite(want)]
    attained = float(finite[len(finite) // 3])
    for thr in (float("-inf"), 0.0, 6.0, attained):
        pos, sc = dev.scan_alpha(stream, table, thr)
        hits = orc.search_hits(want, thr)
        assert np.array_equal(pos, hits), (name, W, thr)
        assert np.array_equal(_bits(sc), _bits(want[hits]))
    pos, _ = dev.scan_alpha(stream, table, attained)
    assert not np.isin(np.nonzero(want == attained)[0], pos).any()      # strict '>'


@pytest.mark.parametrize("name", ["EHIMP", "protein", "a31"])
def test_many_tiles(dev, name):
    """One stream of 12 M symbols: every tile and CTA of the persistent kernels, the histogram's grid stride."""
    letters = ALPHABETS[name]
    texts = random_texts(letters, 12_000_000, 300, seed=5)
    stream = dev.SymbolStream.from_texts(texts, dev.AlphaKind(letters))
    for W in (12, 33):
        table = random_table(W, len(letters), seed=W)
        want = oracle_stream_scores(texts, table, letters)
        assert_same_float(dev.dense_alpha(stream, table).cpu().numpy(), want)
        thr = float(np.quantile(want[np.isfinite(want)], 0.99))
        pos, sc = dev.scan_alpha(stream, table, thr)
        hits = orc.search_hits(want, thr)
        assert len(hits) > 1000 and np.array_equal(pos, hits)
        assert np.array_equal(_bits(sc), _bits(want[hits]))
    counts = dev.histogram(stream).cpu().numpy()
    bg = orc.background(texts, letters)
    total = len(letters) + int(counts.sum())
    assert [(float(int(c)) + 1) / total for c in counts] == list(bg.values())


@pytest.mark.parametrize("name", sorted(ALPHABETS))
@pytest.mark.parametrize("n", [1, 15, 16, 17, 100_003])
def test_histogram_counts_upper_case_only(dev, name, n):
    letters = ALPHABETS[name]
    text = random_texts(letters, n, 1, seed=n)[0]
    stream = dev.SymbolStream.from_texts([text], dev.AlphaKind(letters))
    counts = dev.histogram(stream).cpu().numpy()
    assert counts.dtype == np.int64 and len(counts) == len(letters)
    assert counts.tolist() == [text.count(c) for c in letters]


# ----------------------------------------------------------------------------- API
def test_calculate_and_search_types(dev):
    from rnascan_b200.BioAddons.motifs.matrix import ExtendedPositionSpecificScoringMatrix
    for letters in (ALPHABETS["HSTC"], ALPHABETS["protein"]):
        table = random_table(5, len(letters), seed=len(letters))
        pm = ExtendedPositionSpecificScoringMatrix(make_alphabet(letters),
                                                  {c: table[:, k].tolist() for k, c in enumerate(letters)})
        text = random_texts(letters, 400, 1, seed=3)[0]
        want = orc.alpha_scores(text, table, letters)
        got = pm.calculate(text)
        assert isinstance(got, list) and all(type(v) is float for v in got)
        assert_same_float(np.array(got), want)
        one = pm.calculate(text[:5])
        assert type(one) is float
        assert_same_float(np.array([one]), want[:1])
        assert pm.calculate(text[:4]) == []
        for thr in (float("-inf"), 0.0):
            hits = list(pm.search(text, threshold=thr))
            assert all(type(p) is int and type(s) is float for p, s in hits)
            idx = orc.search_hits(want, thr)
            assert [p for p, _ in hits] == idx.tolist()
            assert np.array_equal(_bits(np.array([s for _, s in hits], np.float64)), _bits(want[idx]))


@pytest.mark.parametrize("A", [8, 13, 20, 31])
def test_pwm_scan_fwd_wide_alphabets(dev, A):
    from rnascan_b200 import pfmutil
    letters = "abcdefghijklmnopqrstuvwxyzABCDE"[:A]           # case-sensitive keys are fine here
    rng = np.random.default_rng(A)
    pwm = {c: rng.normal(size=9).tolist() for c in letters}
    seq = "".join(rng.choice(list(letters), size=500))
    want = []
    for i in range(len(seq) - 9 + 1):
        score = 0.0
        for j in range(9):
            score += pwm[seq[i + j]][j]
        want.append(score)
    got = pfmutil.pwm_scan_fwd(pwm, seq)
    assert all(type(v) is float for v in got)
    assert np.array_equal(_bits(np.array(got)), _bits(np.array(want)))
    with pytest.raises(KeyError):
        pfmutil.pwm_scan_fwd(pwm, seq[:20] + "Z" + seq[20:])


def write_fasta(path, texts):
    with open(path, "w") as fh:
        for k, t in enumerate(texts):
            fh.write(">rec%d some description %d\n" % (k, k))
            for a in range(0, len(t), 60):
                fh.write(t[a:a + 60] + "\n")


def oracle_rows(texts, motif_id, table, letters, thr):
    rows = []
    for k, t in enumerate(texts):
        scores = orc.alpha_scores(t, table, letters)
        rows += [("rec%d" % k, "rec%d some description %d" % (k, k)) + tuple(r)
                 for r in orc.scan_rows(motif_id, t, scores, thr)]
    return rows


def frame_rows(df):
    if len(df) == 0:
        return []
    return list(zip(df["Sequence_ID"], df["Description"], df["Motif_ID"], df["Start"].tolist(),
                    df["End"].tolist(), df["Sequence"], df["LogOdds"].tolist()))


@pytest.mark.parametrize("name", ["HSTC", "EHIMP", "protein", "a31"])
@pytest.mark.parametrize("batch_symbols", [None, 5000])
def test_scan_main_fasta_matches_oracle(dev, tmp_path, monkeypatch, name, batch_symbols):
    from rnascan_b200 import rnascan as ms
    from rnascan_b200.BioAddons.motifs.matrix import ExtendedPositionSpecificScoringMatrix
    letters = ALPHABETS[name]
    alphabet = make_alphabet(letters)
    texts = random_texts(letters, 30_000, 25, seed=len(letters))
    fasta = str(tmp_path / "in.fa")
    write_fasta(fasta, texts)
    table = random_table(8, len(letters), seed=1)
    pm = ExtendedPositionSpecificScoringMatrix(alphabet, {c: table[:, k].tolist() for k, c in enumerate(letters)})
    if batch_symbols:
        monkeypatch.setattr(ms, "MAX_BATCH_SYMBOLS", batch_symbols)
        monkeypatch.setattr(ms, "NATIVE_INGEST", False)
    ms._BATCH_CACHE.clear()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for thr in (float("-inf"), 2.0):
            df = ms.scan_main(fasta, {"mot": pm}, alphabet, None, argparse.Namespace(minscore=thr, debug=False))
            assert frame_rows(df) == oracle_rows(texts, "mot", table, letters, thr)
        bg = ms.compute_background(fasta, alphabet, verbose=False)
    want = orc.background(texts, letters)
    assert list(bg) == list(letters) and dict(bg) == want
    ms._BATCH_CACHE.clear()


def test_ehimp_pssm_from_reduced_pfm_scans_fasta(dev, tmp_path):
    """BEHLMRT PFM -> pfmutil.reduce_pfm_alphabet -> write_pfm -> pfm2pssm (EHIMP) -> scan_main on a FASTA,
    with a background computed from the same FASTA."""
    from rnascan_b200 import pfmutil, rnascan as ms
    rng = np.random.default_rng(11)
    pfm = {c: [float(v) for v in rng.random(9)] for c in "BEHLMRT"}
    path = str(tmp_path / "reduced.txt")
    pfmutil.write_pfm(pfmutil.reduce_pfm_alphabet(pfm), path)
    alphabet = make_alphabet("EHIMP")
    texts = random_texts("EHIMP", 20_000, 12, seed=2)
    fasta = str(tmp_path / "in.fa")
    write_fasta(fasta, texts)
    ms._BATCH_CACHE.clear()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        bg = ms.compute_background(fasta, alphabet, verbose=False)
        assert dict(bg) == orc.background(texts, "EHIMP")
        pssm = ms.load_motif(path, 0.01, alphabet, bg)
        motif_id, pm = list(pssm.items())[0]
        table = pm.table("EHIMP")
        assert np.isfinite(table).all() and pm.length == 9
        df = ms.scan_main(fasta, pssm, alphabet, bg, argparse.Namespace(minscore=1.0, debug=False))
    want = oracle_rows(texts, motif_id, table, "EHIMP", 1.0)
    assert len(want) > 10 and frame_rows(df) == want
    ms._BATCH_CACHE.clear()
