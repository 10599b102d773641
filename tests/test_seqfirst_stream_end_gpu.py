"""The sequence-first combined scan reads each candidate's profile rows as the 16-byte pieces of the window's aligned
span.  A hit whose window ends at the last row of the stream (rows allocated with exactly rs_padded_count(n), as
ProfileStream does) must be found with the exact scores, at every alignment of the window's first byte."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("W", [7, 16])
@pytest.mark.parametrize("n", [40_000, 40_001, 40_002, 40_003])
def test_seqfirst_hit_ending_at_the_last_row(oracle, dtype, W, n):
    from rnascan_b200 import device, synth
    device.require_cuda()
    rng = np.random.default_rng(n + 100 * W)
    codes = rng.integers(0, 4, size=n).astype(np.uint8)
    rows = synth.profile_rows(n, rng).astype(dtype)
    ts = synth.pssm_table(synth.pfm_rows(W, 4, rng))
    tq = synth.pssm_table(synth.pfm_rows(W, 7, rng), background=[synth.SS_P[c] for c in "BEHLMRT"])
    last = n - W
    codes[last:] = ts.argmax(axis=1)                          # the best-scoring window ends at the last row
    rows[last:] = 0.0
    rows[last + np.arange(W), tq.argmax(axis=1)] = 1.0
    pf = device.ProfileStream(rows)
    assert pf.rows.shape[0] == device.padded_count(n)

    a = oracle.seq_scores(synth.to_text(codes, "rna"), ts)
    with np.errstate(all="ignore"):
        b = oracle.profile_scores(rows, tq)
    thr = float(np.nextafter(min(np.float64(a[last]), b[last]), -np.inf))
    with np.errstate(invalid="ignore"):
        want = np.nonzero((a.astype(np.float64) > thr) & (b > thr))[0]
    assert want[-1] == last

    pos, sq, sb = device.scan_fused(device.SymbolStream(codes), pf, ts, tq, thr)
    assert np.array_equal(pos, want)
    assert np.array_equal(sq.view(np.uint32), a[want].view(np.uint32))
    assert np.array_equal(sb.view(np.uint64), b[want].view(np.uint64))
