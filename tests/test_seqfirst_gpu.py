"""GPU parity of the sequence-first combined scan (rs_scan_fused in RS_MODE_AND for W <= 16, and
device.BackgroundFusedScan): the sequence scan runs first and only the windows that pass it have their
profile rows scored.  Positions and both scores must equal the oracle and the structure-first path bit for bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def dev():
    from rnascan_b200 import device
    device.require_cuda()
    return device


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


def _case(dev, total, n_records, seed, dtype, W, zero=False, n_frac=0.01):
    from rnascan_b200 import synth
    rng = np.random.default_rng(seed)
    lengths = synth.record_lengths(total, n_records, rng)
    codes, off = synth.rna_codes(lengths, rng, n_frac=n_frac)
    rows = synth.profile_rows(len(codes), rng, lengths=lengths)
    pfm = synth.pfm_rows(W, 7, rng)
    if zero:
        # -inf log-odds meet exact zeros in the rows: 0 * -inf = NaN -> 0 in the reference's nan_to_num
        pfm[pfm < 0.05] = 0.0
        rows = rows.astype(np.float64)
        rows[rows < 0.08] = 0.0
        rows /= np.maximum(rows.sum(axis=1, keepdims=True), 1e-300)
    rows = rows.astype(np.float32).astype(dtype)
    tq = synth.pssm_table(pfm, background=[synth.SS_P[c] for c in "BEHLMRT"], pseudocount=0.0 if zero else 0.01)
    prob = synth.pfm_rows(W, 4, rng)
    return dev.SymbolStream(codes, off, lengths), dev.ProfileStream(rows), codes, rows, tq, prob


def _seq_table_fn(prob):
    from rnascan_b200 import synth

    def fn(counts8):
        bg = (np.asarray(counts8[:4], np.float64) + 1) / (float(np.sum(counts8[:4])) + 4)
        return synth.pssm_table(prob, background=list(bg / bg.sum()))
    return fn


def _oracle(oracle, codes, rows, ts, tq, thr):
    from rnascan_b200 import synth
    with np.errstate(all="ignore"):
        b = oracle.profile_scores(rows, tq)
    a = oracle.seq_scores(synth.to_text(codes, "rna"), ts)
    with np.errstate(invalid="ignore"):
        wpos = np.nonzero((a.astype(np.float64) > thr) & (b > thr))[0]
    return wpos, a[wpos], b[wpos], a, b


def _bg_scan(dev, st, pf, tq, fn, thr, structure_first, capacity=None, all_reduce=None):
    job = dev.BackgroundFusedScan(st.n, st.codes.device, capacity, structure_first=structure_first)
    W = tq.shape[0]
    absmax = pf.absrow_max()
    launches = 0
    while True:
        job.launch(st.codes, pf.rows, pf.dtype, W, tq, fn, thr, absmax, all_reduce)
        launches += 1
        res = job.results()
        if res is not None:
            return res, job, launches
        job.grow()


def _same(got, want):
    p, q, s = got
    wp, wq, ws = want
    assert np.array_equal(p, wp)
    assert np.array_equal(_bits(q), _bits(wq)) and np.array_equal(_bits(s), _bits(ws))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("W", [1, 5, 7, 8, 9, 12, 16])
@pytest.mark.parametrize("thr", [6.0, 2.0, 0.0, -1.5])
def test_seqfirst_matches_oracle_and_structure_first(dev, oracle, dtype, W, thr):
    st, pf, codes, rows, tq, prob = _case(dev, 300_000, 90, 1000 + 10 * W + int(thr * 4), dtype, W)
    fn = _seq_table_fn(prob)
    counts = np.array([(codes == k).sum() for k in range(8)], np.int64)
    ts = fn(counts)
    want = _oracle(oracle, codes, rows, ts, tq, thr)[:3]
    _same(dev.scan_fused(st, pf, ts, tq, thr), want)                 # rs_scan_fused routes W <= 16 here
    (p, q, s), job, _ = _bg_scan(dev, st, pf, tq, fn, thr, structure_first=False)
    _same((p, q, s), want)
    assert job.launches == 5 and np.array_equal(job.counts_host.numpy(), counts)
    if dtype == np.float32:
        _same(_bg_scan(dev, st, pf, tq, fn, thr, structure_first=True)[0], want)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("W", [7, 12])
def test_seqfirst_threshold_on_an_exact_score(dev, oracle, dtype, W):
    """A threshold equal to a hit's score excludes it (strict >); one ulp below includes it."""
    st, pf, codes, rows, tq, prob = _case(dev, 200_000, 50, 77 + W, dtype, W)
    fn = _seq_table_fn(prob)
    ts = fn(np.array([(codes == k).sum() for k in range(8)], np.int64))
    wpos, wq, ws, a, b = _oracle(oracle, codes, rows, ts, tq, 0.0)
    assert len(wpos) > 10
    k = wpos[len(wpos) // 2]
    for t in (float(min(a[k], b[k])), float(np.nextafter(min(np.float64(a[k]), b[k]), -np.inf))):
        want = _oracle(oracle, codes, rows, ts, tq, t)[:3]
        _same(dev.scan_fused(st, pf, ts, tq, t), want)
        _same(_bg_scan(dev, st, pf, tq, fn, t, structure_first=False)[0], want)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_seqfirst_inf_table_meets_zero_rows(dev, oracle, dtype):
    st, pf, codes, rows, tq, prob = _case(dev, 250_000, 60, 5, dtype, 7, zero=True)
    assert np.isinf(tq).any() and (rows == 0).any()
    fn = _seq_table_fn(prob)
    ts = fn(np.array([(codes == k).sum() for k in range(8)], np.int64))
    for thr in (0.0, -3.0):
        want = _oracle(oracle, codes, rows, ts, tq, thr)[:3]
        _same(dev.scan_fused(st, pf, ts, tq, thr), want)
        _same(_bg_scan(dev, st, pf, tq, fn, thr, structure_first=False)[0], want)


@pytest.mark.parametrize("W", [5, 12])
def test_seqfirst_dense_warps_short_records_and_regrow(dev, oracle, W):
    """A very low threshold puts hundreds of candidates into one warp's segments (the dense expansion path);
    N runs, separators, records shorter than W and the stream end are in the input; a tiny capacity forces
    the overflow -> grow -> relaunch cycle."""
    from rnascan_b200 import synth
    rng = np.random.default_rng(31 + W)
    lengths = np.concatenate([rng.integers(1, W + 1, size=200), synth.record_lengths(400_000, 40, rng)])
    rng.shuffle(lengths)
    codes, off = synth.rna_codes(lengths, rng, n_frac=0.02)
    rows = synth.profile_rows(len(codes), rng, lengths=lengths).astype(np.float32)
    tq = synth.pssm_table(synth.pfm_rows(W, 7, rng), background=[synth.SS_P[c] for c in "BEHLMRT"])
    fn = _seq_table_fn(synth.pfm_rows(W, 4, rng))
    st, pf = dev.SymbolStream(codes, off, lengths), dev.ProfileStream(rows)
    ts = fn(np.array([(codes == k).sum() for k in range(8)], np.int64))
    thr = -20.0
    want = _oracle(oracle, codes, rows, ts, tq, thr)[:3]
    assert len(want[0]) > 100_000            # far more than 256 candidates in a warp's 28-32 K positions
    _same(dev.scan_fused(st, pf, ts, tq, thr, capacity=100), want)
    got, job, launches = _bg_scan(dev, st, pf, tq, fn, thr, structure_first=False, capacity=1000)
    _same(got, want)
    assert launches > 1 and int(job.hb.cand_counters[0].item()) >= len(want[0])


def test_seqfirst_sharded_with_stub_all_reduce(dev, oracle):
    """Two ranks simulated by a stub all_reduce that adds a fixed second shard's counts: the exact table comes
    from the global counts, whatever this shard's own composition."""
    st, pf, codes, rows, tq, prob = _case(dev, 300_000, 80, 91, np.float32, 7)
    other = np.array([900_000, 10, 10, 900_000, 0, 0, 0, 0], np.int64)     # a far-off composition

    def all_reduce(t):
        t.add_(torch.from_numpy(other).to(t.device))

    fn = _seq_table_fn(prob)
    mine = np.array([(codes == k).sum() for k in range(8)], np.int64)
    ts = fn(mine + other)
    want = _oracle(oracle, codes, rows, ts, tq, 1.0)[:3]
    got, job, _ = _bg_scan(dev, st, pf, tq, fn, 1.0, structure_first=False, all_reduce=all_reduce)
    _same(got, want)
    assert np.array_equal(job.counts_host.numpy(), mine + other)
    _same(_bg_scan(dev, st, pf, tq, fn, 1.0, structure_first=True, all_reduce=all_reduce)[0], want)
