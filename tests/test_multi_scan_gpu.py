"""GPU parity of device.scan_onehot_many (rs_scan_onehot_many): many one-hot PSSMs over one symbol stream must
give, motif by motif, exactly the hits and scores of scan_seq / scan_struct_onehot run per motif and of the CPU
oracle (oracle.seq_scores / alpha_scores + search_hits: _pwm.c:34-68, matrix.py:25-43, rnascan.py:263)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from oracle import oracle as orc  # noqa: E402

A_OF = {"rna": 4, "struct": 7}


@pytest.fixture(scope="module")
def dev():
    from rnascan_b200 import device
    device.require_cuda()
    return device


def make_stream(dev, kind, total, n_records, seed, lower=0.1, other=0.002, empty=0):
    """Records of `kind` (lower-case structure letters, invalid symbols N / X, `empty` empty records)."""
    from rnascan_b200 import synth
    rng = np.random.default_rng(seed)
    lengths = synth.record_lengths(total, n_records, rng) if n_records > 1 else np.array([total], np.int64)
    lengths = np.concatenate([lengths, np.zeros(empty, np.int64), [3, 1]])       # empty and short records
    rng.shuffle(lengths)
    codes, offsets = (synth.rna_codes if kind == "rna" else synth.struct_codes)(lengths, rng)
    letters = codes != 0xFF
    bad = letters & (rng.random(len(codes)) < other)
    codes[bad] = 0x0C if kind == "rna" else 0x0F
    if kind == "struct":
        low = letters & ~bad & (rng.random(len(codes)) < lower)
        codes[low] |= 8
    return dev.SymbolStream(codes, offsets, lengths, kind=kind), codes


def make_tables(kind, widths, seed, bg=None, pseudocount=0.01):
    from rnascan_b200 import synth
    rng = np.random.default_rng(seed)
    A = A_OF[kind]
    return [synth.pssm_table(synth.pfm_rows(int(W), A, rng), bg, pseudocount) for W in widths]


def per_motif(dev, stream, kind, tables, thr):
    fn = dev.scan_seq if kind == "rna" else dev.scan_struct_onehot
    return [fn(stream, t, thr) for t in tables]


def oracle_hits(codes, kind, table, thr):
    from rnascan_b200 import synth
    text = synth.to_text(codes, kind)
    if kind == "rna":
        sc = orc.seq_scores(text, table)
    else:                                  # lower-case letters score as their upper case (matrix.py:36-41)
        sc = orc.alpha_scores(text.upper(), table, "BEHLMRT")
    pos = orc.search_hits(sc, thr).astype(np.int64)
    return pos, sc[pos]


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


def check(dev, stream, codes, kind, tables, thr, oracle=True, capacity=None):
    motif, pos, scores, bases = dev.scan_onehot_many(stream, tables, thr, capacity=capacity)
    assert scores.dtype == (np.float32 if kind == "rna" else np.float64)
    assert len(bases) == len(tables) + 1 and bases[0] == 0 and bases[-1] == len(pos)
    ref = per_motif(dev, stream, kind, tables, thr)
    assert np.array_equal(np.diff(bases), [len(p) for p, _ in ref])
    for m, (rp, rs) in enumerate(ref):
        a, b = int(bases[m]), int(bases[m + 1])
        assert (motif[a:b] == m).all()
        assert np.array_equal(pos[a:b], rp), m
        assert np.array_equal(bits(scores[a:b]), bits(rs)), m
        if oracle:
            op, osc = oracle_hits(codes, kind, tables[m], thr)
            assert np.array_equal(pos[a:b], op), m
            assert np.array_equal(bits(scores[a:b]), bits(osc)), m
    return motif, pos, scores, bases


@pytest.mark.parametrize("kind", ["rna", "struct"])
@pytest.mark.parametrize("M", [1, 2, 31, 32, 33, 256, 257, 600])
def test_collection_sizes(dev, kind, M):
    stream, codes = make_stream(dev, kind, 40_000, 20, seed=M, empty=2)
    widths = np.random.default_rng(M).integers(4, 13, size=M)
    tables = make_tables(kind, widths, seed=100 + M)
    check(dev, stream, codes, kind, tables, 3.0, oracle=M <= 33)


@pytest.mark.parametrize("kind", ["rna", "struct"])
def test_mixed_widths_1_to_16_and_warp_range_boundaries(dev, kind):
    stream, codes = make_stream(dev, kind, 300_001, 7, seed=3)     # > 200 warp ranges of 1024 positions
    widths = list(range(1, 17)) * 3
    tables = make_tables(kind, widths, seed=4)
    for thr in (-2.0, 0.0, 2.5, 6.0):
        check(dev, stream, codes, kind, tables, thr)


@pytest.mark.parametrize("kind", ["rna", "struct"])
def test_infinite_and_nan_cells(dev, kind):
    A = A_OF[kind]
    stream, codes = make_stream(dev, kind, 30_000, 5, seed=5)
    widths = [3, 6, 8, 9, 12, 16]
    ninf = make_tables(kind, widths, seed=6, pseudocount=0)              # zero counts: -inf cells
    for t in ninf:
        t[::2, 1] = -np.inf
    zero_bg = np.ones(A)
    zero_bg[2] = 0.0                                                      # zero background: +inf / NaN cells
    with np.errstate(divide="ignore", invalid="ignore"):
        pinf = make_tables(kind, widths, seed=7, bg=zero_bg, pseudocount=0)
    pinf[0][1, 3] = np.nan
    pinf[3][10 % pinf[3].shape[0], 0] = np.nan
    check(dev, stream, codes, kind, ninf + pinf, 1.0)


@pytest.mark.parametrize("kind", ["rna", "struct"])
def test_threshold_on_and_one_ulp_below_an_exact_score(dev, kind):
    stream, codes = make_stream(dev, kind, 20_000, 3, seed=8)
    tables = make_tables(kind, [5, 8, 9, 14], seed=9)
    for t in tables:
        pos, sc = per_motif(dev, stream, kind, [t], -1e9)[0]
        s = float(sc[len(sc) // 2])
        below = float(np.nextafter(np.float32(s), np.float32(-np.inf))) if kind == "rna" else np.nextafter(s, -np.inf)
        for thr in (s, below):
            check(dev, stream, codes, kind, tables, thr)


@pytest.mark.parametrize("kind", ["rna", "struct"])
def test_capacity_overflow_regrows(dev, kind):
    stream, codes = make_stream(dev, kind, 50_000, 4, seed=10)
    tables = make_tables(kind, [6, 10, 12], seed=11)
    motif, pos, scores, bases = check(dev, stream, codes, kind, tables, -5.0, oracle=False, capacity=100)
    assert bases[-1] > 100


@pytest.mark.parametrize("kind", ["rna", "struct"])
def test_invalid_arguments(dev, kind):
    stream, _ = make_stream(dev, kind, 1000, 1, seed=12)
    with pytest.raises(ValueError):
        dev.scan_onehot_many(stream, make_tables(kind, [17], seed=1), 0.0)
    with pytest.raises(ValueError):
        dev.scan_onehot_many(stream, make_tables(kind, [5], seed=1), float("-inf"))
    from rnascan_b200 import _lib
    t = np.zeros((1, 5, 4))
    w = np.array([5], np.int32)
    assert _lib.lib.rs_scan_onehot_many(5, 0, 0, 1, w.ctypes.data, t.ctypes.data, 5, 0.0, 0, 0, 0, 0, 0, 0, 0, 0,
                                        0) == _lib.RS_ERR_INVALID
    assert _lib.lib.rs_scan_onehot_many_workspace_bytes(4, 10, 1, 17) < 0


@pytest.mark.parametrize("kind", ["rna", "struct"])
def test_100m_symbol_stream(dev, kind):
    stream, codes = make_stream(dev, kind, 100_000_000, 40_000, seed=13, lower=0.05, other=0.0005)
    widths = np.random.default_rng(14).integers(7, 13, size=24)
    tables = make_tables(kind, widths, seed=15)
    check(dev, stream, codes, kind, tables, 6.0 if kind == "rna" else 4.0, oracle=False)
