"""GPU parity of device.scan_pair_onehot_many (rs_scan_pair_onehot_many): many (sequence, structure) motif pairs
over an RNA stream and the structure stream that lines up with it must give, pair by pair, exactly the hits and
both scores of scan_pair_onehot run per pair and of the CPU oracle (oracle.seq_scores / alpha_scores +
search_hits on each stream, ANDed: rnascan.py:263 twice and the combine() join, rnascan.py:416-434)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from oracle import oracle as orc  # noqa: E402


@pytest.fixture(scope="module")
def dev():
    from rnascan_b200 import device
    device.require_cuda()
    return device


def make_pair(dev, total, n_records, seed, lower=0.1, other=0.002):
    """An RNA stream and a structure stream over the same record lengths (separators coincide), with empty and
    1-3 symbol records, invalid symbols placed independently in each stream and lower-case structure letters."""
    from rnascan_b200 import synth
    rng = np.random.default_rng(seed)
    lengths = synth.record_lengths(total, n_records, rng) if n_records > 1 else np.array([total], np.int64)
    lengths = np.concatenate([lengths, [0, 0, 3, 2, 1]])
    rng.shuffle(lengths)
    seq, offsets = synth.rna_codes(lengths, rng, n_frac=0.0)
    st, offsets2 = synth.struct_codes(lengths, rng)
    assert np.array_equal(offsets, offsets2) and np.array_equal(seq == 0xFF, st == 0xFF)
    letters = seq != 0xFF
    seq[letters & (rng.random(len(seq)) < other)] = 0x0C
    bad = letters & (rng.random(len(st)) < other)
    st[bad] = 0x0F
    st[letters & ~bad & (rng.random(len(st)) < lower)] |= 8
    return (dev.SymbolStream(seq, offsets, lengths, kind="rna"), dev.SymbolStream(st, offsets, lengths, kind="struct"),
            seq, st)


def make_tables(widths, seed, bg_seq=None, bg_struct=None, pseudocount=0.01):
    from rnascan_b200 import synth
    rng = np.random.default_rng(seed)
    ts = [synth.pssm_table(synth.pfm_rows(int(W), 4, rng), bg_seq, pseudocount) for W in widths]
    tq = [synth.pssm_table(synth.pfm_rows(int(W), 7, rng), bg_struct, pseudocount) for W in widths]
    return ts, tq


def oracle_pair(seq, st, ts, tq, thr):
    from rnascan_b200 import synth
    a = orc.seq_scores(synth.to_text(seq, "rna"), ts)
    b = orc.alpha_scores(synth.to_text(st, "struct").upper(), tq, "BEHLMRT")   # lower case scores as upper
    both = np.intersect1d(orc.search_hits(a, thr), orc.search_hits(b, thr)).astype(np.int64)
    return both, a[both], b[both]


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


def check(dev, pair, ts, tq, thr, oracle=True, capacity=None):
    ss, sq, seq, st = pair
    motif, pos, a, b, bases = dev.scan_pair_onehot_many(ss, sq, ts, tq, thr, capacity=capacity)
    assert a.dtype == np.float32 and b.dtype == np.float64
    assert len(bases) == len(ts) + 1 and bases[0] == 0 and bases[-1] == len(pos)
    for m in range(len(ts)):
        lo, hi = int(bases[m]), int(bases[m + 1])
        assert (motif[lo:hi] == m).all()
        rp, ra, rb = dev.scan_pair_onehot(ss, sq, ts[m], tq[m], thr)
        assert np.array_equal(pos[lo:hi], rp), m
        assert np.array_equal(bits(a[lo:hi]), bits(ra)), m
        assert np.array_equal(bits(b[lo:hi]), bits(rb)), m
        if oracle:
            op, oa, ob = oracle_pair(seq, st, ts[m], tq[m], thr)
            assert np.array_equal(pos[lo:hi], op), m
            assert np.array_equal(bits(a[lo:hi]), bits(oa)), m
            assert np.array_equal(bits(b[lo:hi]), bits(ob)), m
    return motif, pos, a, b, bases


@pytest.mark.parametrize("M", [1, 2, 31, 32, 33, 256, 257, 600])
def test_collection_sizes(dev, M):
    pair = make_pair(dev, 40_000, 20, seed=M)
    widths = np.random.default_rng(M).integers(1, 17, size=M)
    ts, tq = make_tables(widths, seed=100 + M)
    *_, bases = check(dev, pair, ts, tq, 1.0, oracle=M <= 33)
    assert bases[-1] > 0


def test_mixed_widths_1_to_16_and_warp_range_boundaries(dev):
    pair = make_pair(dev, 300_001, 7, seed=3)              # > 200 warp ranges of 1024 positions
    ts, tq = make_tables(list(range(1, 17)) * 3, seed=4)
    for thr in (-2.0, 0.0, 1.5, 3.0):
        motif, *_ = check(dev, pair, ts, tq, thr)
        for lo, hi in ((0, 5), (5, 8), (8, 16)):           # all three exactness regimes give joint hits
            assert np.isin(motif % 16, np.arange(lo, hi)).any(), (thr, lo, hi)


def test_infinite_and_nan_cells(dev):
    pair = make_pair(dev, 30_000, 5, seed=5)
    widths = [3, 5, 6, 8, 9, 12, 16]
    ts, tq = make_tables(widths, seed=6)
    ts_ninf, tq_ninf = make_tables(widths, seed=7, pseudocount=0)       # zero counts: -inf cells
    for t in ts_ninf:
        t[::2, 1] = -np.inf
    for t in tq_ninf:
        t[1::2, 2] = -np.inf
    zs, zq = np.ones(4), np.ones(7)
    zs[2] = zq[3] = 0.0                                                 # zero background: +inf / NaN cells
    with np.errstate(divide="ignore", invalid="ignore"):
        ts_pinf, tq_pinf = make_tables(widths, seed=8, bg_seq=zs, bg_struct=zq, pseudocount=0)
    ts_pinf[0][1, 3] = np.nan
    tq_pinf[3][5, 0] = np.nan
    # each kind of special cell on one side, an ordinary table on the other, and both sides special
    all_s = ts_ninf + ts + ts_pinf + ts_pinf
    all_q = tq + tq_ninf + tq + tq_pinf
    *_, bases = check(dev, pair, all_s, all_q, 0.5)
    assert bases[-1] > 0


def test_threshold_on_and_one_ulp_below_a_joint_score(dev):
    pair = make_pair(dev, 20_000, 3, seed=9)
    ts, tq = make_tables([4, 5, 7, 8, 9, 14], seed=10)
    for m in range(len(ts)):
        pos, a, b = dev.scan_pair_onehot(pair[0], pair[1], ts[m], tq[m], -1e9)
        k = len(pos) // 2
        sa, sb = float(a[k]), float(b[k])
        for thr in (sa, float(np.nextafter(np.float32(sa), np.float32(-np.inf))), sb, np.nextafter(sb, -np.inf)):
            *_, bases = check(dev, pair, ts, tq, thr)
            assert bases[-1] > 0


def test_capacity_overflow_regrows(dev):
    pair = make_pair(dev, 50_000, 4, seed=11)
    ts, tq = make_tables([4, 6, 10, 12], seed=12)
    *_, bases = check(dev, pair, ts, tq, -3.0, oracle=False, capacity=100)
    assert bases[-1] > 100


def test_empty_streams(dev):
    ss = dev.SymbolStream(np.zeros(0, np.uint8), np.zeros(0, np.int64), np.zeros(0, np.int64), kind="rna")
    sq = dev.SymbolStream(np.zeros(0, np.uint8), np.zeros(0, np.int64), np.zeros(0, np.int64), kind="struct")
    ts, tq = make_tables([5, 9], seed=13)
    motif, pos, a, b, bases = dev.scan_pair_onehot_many(ss, sq, ts, tq, 0.0)
    assert len(pos) == len(motif) == len(a) == len(b) == 0 and list(bases) == [0, 0, 0]


def test_invalid_arguments(dev):
    ss, sq, _, _ = make_pair(dev, 1000, 1, seed=14)
    ts, tq = make_tables([5], seed=1)
    with pytest.raises(ValueError):
        dev.scan_pair_onehot_many(ss, sq, *make_tables([17], seed=1), 0.0)
    with pytest.raises(ValueError):
        dev.scan_pair_onehot_many(ss, sq, ts, make_tables([6], seed=1)[1], 0.0)         # unequal pair widths
    with pytest.raises(ValueError):
        dev.scan_pair_onehot_many(ss, sq, ts, tq, float("-inf"))
    with pytest.raises(ValueError):
        dev.scan_pair_onehot_many(sq, ss, ts, tq, 0.0)                                   # stream kinds swapped
    short = dev.SymbolStream(sq.host_codes()[:500], kind="struct")
    with pytest.raises(ValueError):
        dev.scan_pair_onehot_many(ss, short, ts, tq, 0.0)                                # lengths differ
    from rnascan_b200 import _lib
    w = np.array([5], np.int32)
    s4, s7 = np.zeros((1, 5, 4)), np.zeros((1, 5, 7))
    assert _lib.lib.rs_scan_pair_onehot_many_workspace_bytes(10, 1, 17) < 0
    assert _lib.lib.rs_scan_pair_onehot_many_workspace_bytes(1 << 32, 1, 5) < 0
    assert _lib.lib.rs_scan_pair_onehot_many(0, 0, 0, 1, w.ctypes.data, s4.ctypes.data, 0, 5, 0.0, 0, 0, 0, 0, 0, 0,
                                             0, 0, 0) == _lib.RS_ERR_INVALID              # no structure tables
    w6 = np.array([6], np.int32)
    assert _lib.lib.rs_scan_pair_onehot_many(0, 0, 0, 1, w6.ctypes.data, s4.ctypes.data, s7.ctypes.data, 5, 0.0, 0,
                                             0, 0, 0, 0, 0, 0, 0, 0) == _lib.RS_ERR_INVALID  # width > stride
    assert _lib.lib.rs_scan_pair_onehot_many(0, 0, 0, 1, w.ctypes.data, s4.ctypes.data, s7.ctypes.data, 5,
                                             float("nan"), 0, 0, 0, 0, 0, 0, 0, 0, 0) == _lib.RS_ERR_INVALID


def test_100m_symbol_pair(dev):
    pair = make_pair(dev, 100_000_000, 40_000, seed=15, lower=0.05, other=0.0005)
    widths = np.random.default_rng(16).integers(4, 17, size=24)
    ts, tq = make_tables(widths, seed=17)
    *_, bases = check(dev, pair, ts, tq, 3.0, oracle=False)
    assert bases[-1] > 0
