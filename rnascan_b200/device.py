"""Device-buffer plumbing between the Python host API and the C ABI.

PyTorch is used for exactly three things: allocating device / pinned-host memory, host<->
device copies and CUDA streams.  All arithmetic happens in librnascan_b200.so.

Layout in HBM (see DESIGN.md):
  symbol stream   uint8[rs_padded_count(n)]      records concatenated, one 0xFF separator
                                                  after every record, padding = 0xFF
  profile stream  float32|float64[padded][7]      rows aligned 1:1 with the symbol stream
                                                  (separator rows are zeros), channels
                                                  B,E,H,L,M,R,T
  hits            int64 pos[], float32 seq[], float64 struct[]   (structure of arrays)
"""
import ctypes
import os
import time

import numpy as np
import torch

from . import _lib
from ._lib import lib, check, RnascanCudaError

CHANNELS = "BEHLMRT"        # device channel order == profile file column order
HOST_THREADS = max(1, min(32, os.cpu_count() or 1))
RNA_COLUMNS = "ACGU"        # device column order of sequence tables (matrix.py:57 sorts)


def require_cuda():
    if not torch.cuda.is_available():
        raise RnascanCudaError(
            "rnascan_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def padded_count(n):
    return int(lib.rs_padded_count(int(n)))


MAX_ALPHA_LETTERS = 31


class AlphaKind(object):
    """Stream kind of any other alphabet: the "alphabet" layout of rnascan_b200.h, letter k of `letters` (in
    the caller's column order) has index k.  Supported: 1..31 distinct single ASCII characters, none of them a
    lower-case a-z (text is scored upper-cased but counted case-sensitively, so a lower-case letter would need
    two indices in one code); NotImplementedError names the rule otherwise."""

    def __init__(self, letters):
        letters = "".join(letters) if letters is not None else ""
        if not (1 <= len(letters) <= MAX_ALPHA_LETTERS and len(set(letters)) == len(letters)
                and all(ord(c) < 128 and not "a" <= c <= "z" for c in letters)):
            raise NotImplementedError(
                "GPU scoring supports GAUC, BEHLMRT and alphabets of 1 to %d distinct single ASCII characters "
                "without lower-case a-z (got %r)" % (MAX_ALPHA_LETTERS, letters))
        self.letters = letters

    def __eq__(self, other):
        return isinstance(other, AlphaKind) and other.letters == self.letters

    def __ne__(self, other):
        return not self == other

    def __hash__(self):
        return hash(("alpha", self.letters))

    def __repr__(self):
        return "AlphaKind(%r)" % self.letters


# --------------------------------------------------------------------------- packing (host)
def pack_texts(texts, kind):
    """Encode a list of record strings into one symbol stream (host, numpy).  `kind`: "rna", "struct" or an
    AlphaKind.

    Returns (codes uint8[n_total], offsets int64[R], lengths int64[R]); record r occupies
    codes[offsets[r] : offsets[r]+lengths[r]] and is followed by one separator.
    """
    if isinstance(kind, AlphaKind):
        letters = kind.letters.encode("ascii")

        def enc(src, n, dst):
            return lib.rs_host_encode_alpha(src, n, letters, len(letters), dst)
    else:
        enc = lib.rs_host_encode_rna if kind == "rna" else lib.rs_host_encode_struct
    lengths = np.fromiter((len(t) for t in texts), dtype=np.int64, count=len(texts))
    offsets = np.zeros(len(texts), dtype=np.int64)
    if len(texts) > 1:
        np.cumsum(lengths[:-1] + 1, out=offsets[1:])
    total = int(lengths.sum() + len(texts))
    raw = "\n".join(texts).encode("latin-1", "replace") + b"\n" if texts else b""
    assert len(raw) == total
    src = np.frombuffer(raw, dtype=np.uint8)
    codes = np.empty(total, dtype=np.uint8)
    if total:
        check(enc(src.ctypes.data, total, codes.ctypes.data))
        codes[offsets + lengths] = _lib.RS_SEP
    return codes, offsets, lengths


def pack_profiles(profiles, dtype=np.float64):
    """Concatenate (L_r, 7) arrays with one zero separator row after each."""
    lengths = np.fromiter((p.shape[0] for p in profiles), dtype=np.int64, count=len(profiles))
    total = int(lengths.sum() + len(profiles))
    out = np.zeros((total, len(CHANNELS)), dtype=dtype)
    off = 0
    for p in profiles:
        out[off:off + p.shape[0]] = p
        off += p.shape[0] + 1
    return out


class SymbolStream(object):
    """A symbol stream resident in HBM."""

    def __init__(self, codes, offsets=None, lengths=None, device=None, kind=None):
        require_cuda()
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        self.kind = kind                 # "rna" | "struct" | AlphaKind | None (unknown: generic kernels)
        self.n = int(codes.shape[0])
        self.offsets = np.zeros(1, np.int64) if offsets is None else np.asarray(offsets, np.int64)
        self.lengths = np.array([self.n], np.int64) if lengths is None else np.asarray(lengths, np.int64)
        npad = padded_count(self.n)
        host = torch.empty(npad, dtype=torch.uint8, pin_memory=True)
        hv = host.numpy()
        hv[:self.n] = codes
        hv[self.n:] = _lib.RS_SEP
        self.codes = host.to(device or "cuda", non_blocking=True)
        self._host = host            # keep the pinned buffer alive until the copy is done

    @classmethod
    def from_texts(cls, texts, kind, device=None):
        codes, offsets, lengths = pack_texts(texts, kind)
        return cls(codes, offsets, lengths, device, kind=kind)

    def host_codes(self):
        """The encoded symbols as a host uint8 array (the pinned upload buffer)."""
        return self._host.numpy()[:self.n]

    def locate(self, pos):
        """stream position -> (record index, 0-based start within the record)."""
        pos = np.asarray(pos, dtype=np.int64)
        rec = np.searchsorted(self.offsets, pos, side="right") - 1
        return rec, pos - self.offsets[rec]


class ProfileStream(object):
    """A 7-channel profile stream resident in HBM, row-aligned with a SymbolStream."""

    def __init__(self, rows, device=None):
        require_cuda()
        rows = np.ascontiguousarray(rows)
        if rows.dtype not in (np.float32, np.float64):
            rows = rows.astype(np.float64)
        if rows.ndim != 2 or rows.shape[1] != len(CHANNELS):
            raise ValueError("profile must have shape (L, 7) in channel order %s" % CHANNELS)
        self.n = int(rows.shape[0])
        self.dtype = _lib.RS_F32 if rows.dtype == np.float32 else _lib.RS_F64
        npad = padded_count(self.n)
        tdt = torch.float32 if rows.dtype == np.float32 else torch.float64
        host = torch.zeros((npad, len(CHANNELS)), dtype=tdt, pin_memory=True)
        host.numpy()[:self.n] = rows
        self.rows = host.to(device or "cuda", non_blocking=True)
        self._host = host
        self._stats = None

    @classmethod
    def from_device(cls, tensor, n):
        """Wrap an already-resident (padded, 7) tensor (used by bench.py)."""
        self = cls.__new__(cls)
        self.n = int(n)
        self.dtype = _lib.RS_F32 if tensor.dtype == torch.float32 else _lib.RS_F64
        self.rows = tensor
        self._host = None
        self._stats = None
        return self

    def stats(self):
        """(max abs row sum, #non-finite, #negative) -- computed once on the device."""
        if self._stats is None:
            st = torch.empty(3, dtype=torch.float64, device=self.rows.device)
            check(lib.rs_profile_stats(_ptr(self.rows), self.dtype, self.n, _ptr(st), _stream()))
            self._stats = tuple(float(v) for v in st.cpu().numpy())
        return self._stats

    def absrow_max(self):
        mx, bad, neg = self.stats()
        return float("nan") if (bad or neg) else mx

    def shadow(self):
        """float32 round-to-nearest copy of float64 rows, resident beside them (the batched scan's tensor-core
        filter reads it; candidates are re-scored from the float64 rows).  None for float32 streams or when
        the host copy is gone."""
        if self.dtype != _lib.RS_F64 or self._host is None:
            return None
        if getattr(self, "_shadow", None) is None:
            h32 = torch.empty(self._host.shape, dtype=torch.float32, pin_memory=True)
            check(lib.rs_host_rows_to_f32(self._host.numpy().ctypes.data, self._host.numel(), h32.numpy().ctypes.data,
                                          HOST_THREADS))
            self._shadow = h32.to(self.rows.device, non_blocking=True)
            self._shadow_host = h32
        return self._shadow


# --------------------------------------------------------------------------- kernels
def _table(table, cols):
    t = np.ascontiguousarray(table, dtype=np.float64)
    if t.ndim != 2:
        raise ValueError("position-weight matrix has incorrect rank (%d expected 2)" % t.ndim)
    if t.shape[1] != cols:
        raise ValueError("position-weight matrix should have %d columns (%d columns found)"
                         % (cols, t.shape[1]))
    if not 1 <= t.shape[0] <= _lib.RS_MAX_W:
        raise ValueError("motif width %d outside [1, %d]" % (t.shape[0], _lib.RS_MAX_W))
    return t


def histogram(stream):
    """int64[8] exact counts of symbols 0..7 whose 'not counted' bit is clear; for an AlphaKind stream
    int64[A], the counts of its A letters in upper case."""
    kind = getattr(stream, "kind", None)
    if isinstance(kind, AlphaKind):
        counts = torch.zeros(32, dtype=torch.int64, device=stream.codes.device)
        check(lib.rs_hist_alpha(_ptr(stream.codes), stream.n, _ptr(counts), _stream()))
        return counts[:len(kind.letters)]
    counts = torch.zeros(8, dtype=torch.int64, device=stream.codes.device)
    fn = lib.rs_hist_rna if getattr(stream, "kind", None) == "rna" else lib.rs_hist
    check(fn(_ptr(stream.codes), stream.n, _ptr(counts), _stream()))
    return counts


def dense_seq(stream, table):
    t = _table(table, 4)
    W = t.shape[0]
    nout = max(0, stream.n - W + 1)
    out = torch.empty(max(nout, 1), dtype=torch.float32, device=stream.codes.device)
    check(lib.rs_scores_dense_seq(_ptr(stream.codes), stream.n, t.ctypes.data, W, _ptr(out), _stream()))
    return out[:nout]


def dense_struct(stream, table):
    t = _table(table, 7)
    W = t.shape[0]
    nout = max(0, stream.n - W + 1)
    out = torch.empty(max(nout, 1), dtype=torch.float64, device=stream.codes.device)
    check(lib.rs_scores_dense_struct(_ptr(stream.codes), stream.n, t.ctypes.data, W, _ptr(out), _stream()))
    return out[:nout]


def _alpha_table(table):
    t = np.ascontiguousarray(table, dtype=np.float64)
    if t.ndim != 2 or not 1 <= t.shape[1] <= MAX_ALPHA_LETTERS:
        raise ValueError("position-weight matrix must be (width, 1..%d letters)" % MAX_ALPHA_LETTERS)
    return _table(t, t.shape[1])


def dense_alpha(stream, table):
    """float64 score of every window of an alphabet-layout stream (rs_scores_dense_alpha); table (W, A), column k
    = letter index k of the stream's codes."""
    t = _alpha_table(table)
    W, A = t.shape
    nout = max(0, stream.n - W + 1)
    out = torch.empty(max(nout, 1), dtype=torch.float64, device=stream.codes.device)
    check(lib.rs_scores_dense_alpha(_ptr(stream.codes), stream.n, t.ctypes.data, W, A, _ptr(out), _stream()))
    return out[:nout]


def dense_struct_milli(stream, table):
    """int32 thousandths of Python's round(score, 3) for every window (rs_scores_dense_struct_milli), W <= 16."""
    t = _table(table, 7)
    W = t.shape[0]
    nout = max(0, stream.n - W + 1)
    out = torch.empty(max(nout, 1), dtype=torch.int32, device=stream.codes.device)
    check(lib.rs_scores_dense_struct_milli(_ptr(stream.codes), stream.n, t.ctypes.data, W, _ptr(out), _stream()))
    return out[:nout]


def scan_struct_every_position(stream, table):
    """The -m -inf scan of a structure stream as it is PRINTED: (pos, round(score, 3) in thousandths, int32) for
    every window with a finite score (NaN and -inf windows are never reported, SURVEY.md H5); 4 bytes per
    position come back from the device instead of 8.  None when the form does not apply (W > 16, a score
    outside its range): the caller uses scan_struct_onehot."""
    t = _table(table, 7)
    if t.shape[0] > 16:
        return None
    host = torch.empty(max(stream.n - t.shape[0] + 1, 0), dtype=torch.int32, pin_memory=True)
    if host.numel() == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int32)
    host.copy_(dense_struct_milli(stream, t))
    m = host.numpy()
    if (m == _lib.RS_MILLI_RANGE).any():
        return None
    pos = np.nonzero((m > _lib.RS_MILLI_RANGE) | (m == _lib.RS_MILLI_NEG0))[0].astype(np.int64)
    return pos, m[pos]


def dense_profile(profile, table, stream=None):
    t = _table(table, 7)
    W = t.shape[0]
    nout = max(0, profile.n - W + 1)
    out = torch.empty(max(nout, 1), dtype=torch.float64, device=profile.rows.device)
    codes = None if stream is None else stream.codes
    check(lib.rs_scores_dense_profile(_ptr(profile.rows), profile.dtype, profile.n, _ptr(codes),
                                      t.ctypes.data, W, _ptr(out), _stream()))
    return out[:nout]


class HitBuffers(object):
    """Caller-owned output + workspace for one thresholded scan (reusable)."""

    def __init__(self, n, capacity, device, want_seq=True, want_struct=True):
        self.capacity = int(capacity)
        cap = max(self.capacity, 1)
        self.pos = torch.empty(cap, dtype=torch.int64, device=device)
        self.seq = torch.empty(cap, dtype=torch.float32, device=device) if want_seq else None
        self.struct = torch.empty(cap, dtype=torch.float64, device=device) if want_struct else None
        self.counters = torch.zeros(2, dtype=torch.int64, device=device)
        self.cand_counters = torch.zeros(2, dtype=torch.int64, device=device)   # first pass of two-pass scans
        self.work_bytes = int(lib.rs_scan_workspace_bytes(int(n), self.capacity))
        self.work = torch.empty(self.work_bytes, dtype=torch.uint8, device=device)


def _run_thresholded(n, device, launch, want_seq, want_struct, capacity=None):
    """Run `launch(buffers)`; grow the hit buffers and re-run if they overflowed."""
    cap = int(capacity) if capacity else max(4096, n // 256)
    while True:
        hb = HitBuffers(n, cap, device, want_seq, want_struct)
        launch(hb)
        found, rescored = (int(v) for v in hb.counters.cpu().numpy())
        if found <= cap:
            pos = hb.pos[:found].cpu().numpy()
            seq = hb.seq[:found].cpu().numpy() if want_seq else None
            st = hb.struct[:found].cpu().numpy() if want_struct else None
            return pos, seq, st, rescored
        cap = found


def scan_seq(stream, table, threshold, capacity=None):
    """Ordered (pos int64[], score float32[]) of windows with score > threshold."""
    t = _table(table, 4)
    W = t.shape[0]
    threshold = float(threshold)
    if threshold == float("-inf"):
        sc = dense_seq(stream, t).cpu().numpy()
        with np.errstate(invalid="ignore"):
            pos = np.nonzero(sc.astype(np.float64) > threshold)[0].astype(np.int64)
        return pos, sc[pos]

    def launch(hb):
        check(lib.rs_scan_seq(_ptr(stream.codes), stream.n, t.ctypes.data, W, threshold, hb.capacity,
                              _ptr(hb.pos), _ptr(hb.seq), _ptr(hb.counters), _ptr(hb.work),
                              hb.work_bytes, _stream()))
    pos, seq, _, _ = _run_thresholded(stream.n, stream.codes.device, launch, True, False, capacity)
    return pos, seq


def scan_struct_onehot(stream, table, threshold, capacity=None):
    t = _table(table, 7)
    W = t.shape[0]
    threshold = float(threshold)
    if threshold == float("-inf"):
        sc = dense_struct(stream, t).cpu().numpy()
        with np.errstate(invalid="ignore"):
            pos = np.nonzero(sc > threshold)[0].astype(np.int64)
        return pos, sc[pos]

    def launch(hb):
        check(lib.rs_scan_struct_onehot(_ptr(stream.codes), stream.n, t.ctypes.data, W, threshold,
                                        hb.capacity, _ptr(hb.pos), _ptr(hb.struct), _ptr(hb.counters),
                                        _ptr(hb.work), hb.work_bytes, _stream()))
    pos, _, st, _ = _run_thresholded(stream.n, stream.codes.device, launch, False, True, capacity)
    return pos, st


def scan_alpha(stream, table, threshold, capacity=None):
    """Ordered (pos int64[], score float64[]) of the windows of an alphabet-layout stream with score > threshold
    (rs_scan_alpha); table as for dense_alpha."""
    t = _alpha_table(table)
    W, A = t.shape
    threshold = float(threshold)
    if threshold == float("-inf"):
        sc = dense_alpha(stream, t).cpu().numpy()
        with np.errstate(invalid="ignore"):
            pos = np.nonzero(sc > threshold)[0].astype(np.int64)
        return pos, sc[pos]

    def launch(hb):
        check(lib.rs_scan_alpha(_ptr(stream.codes), stream.n, t.ctypes.data, W, A, threshold, hb.capacity,
                                _ptr(hb.pos), _ptr(hb.struct), _ptr(hb.counters), _ptr(hb.work), hb.work_bytes,
                                _stream()))
    pos, _, st, _ = _run_thresholded(stream.n, stream.codes.device, launch, False, True, capacity)
    return pos, st


def scan_pair_onehot(seq_stream, struct_stream, seq_table, struct_table, threshold, capacity=None):
    """Windows where the sequence score AND the structure score exceed the threshold."""
    ts, tq = _table(seq_table, 4), _table(struct_table, 7)
    if ts.shape[0] != tq.shape[0]:
        raise ValueError("sequence and structure motifs must have the same width")
    if seq_stream.n != struct_stream.n:
        raise ValueError("sequence and structure streams differ in length")
    W = ts.shape[0]
    threshold = float(threshold)
    if threshold == float("-inf"):
        a = dense_seq(seq_stream, ts).cpu().numpy()
        b = dense_struct(struct_stream, tq).cpu().numpy()
        with np.errstate(invalid="ignore"):
            pos = np.nonzero((a.astype(np.float64) > threshold) & (b > threshold))[0].astype(np.int64)
        return pos, a[pos], b[pos]

    def launch(hb):
        check(lib.rs_scan_pair_onehot(_ptr(seq_stream.codes), _ptr(struct_stream.codes), seq_stream.n,
                                      ts.ctypes.data, tq.ctypes.data, W, threshold, hb.capacity,
                                      _ptr(hb.pos), _ptr(hb.seq), _ptr(hb.struct), _ptr(hb.counters),
                                      _ptr(hb.work), hb.work_bytes, _stream()))
    pos, sq, st, _ = _run_thresholded(seq_stream.n, seq_stream.codes.device, launch, True, True, capacity)
    return pos, sq, st


def scan_fused(stream, profile, seq_table, struct_table, threshold, capacity=None, return_stats=False):
    """Sequence PSSM + averaged profile in one pass.

    seq_table=None  -> RS_MODE_STRUCT: hits where the profile score > threshold
    seq_table given -> RS_MODE_AND:    hits where both scores > threshold
    Returns (pos, seq_scores|None, struct_scores[, n_rescored]).
    """
    tq = _table(struct_table, 7)
    W = tq.shape[0]
    mode = _lib.RS_MODE_STRUCT if seq_table is None else _lib.RS_MODE_AND
    ts = None if seq_table is None else _table(seq_table, 4)
    if ts is not None and ts.shape[0] != W:
        raise ValueError("sequence and structure motifs must have the same width")
    if stream.n != profile.n:
        raise ValueError("symbol stream and profile stream differ in length")
    threshold = float(threshold)
    if threshold == float("-inf"):
        b = dense_profile(profile, tq, stream).cpu().numpy()
        with np.errstate(invalid="ignore"):
            keep = b > threshold
            if ts is not None:
                a = dense_seq(stream, ts).cpu().numpy()
                keep &= a.astype(np.float64) > threshold
        pos = np.nonzero(keep)[0].astype(np.int64)
        out = (pos, a[pos] if ts is not None else None, b[pos])
        return out + (0,) if return_stats else out
    absmax = profile.absrow_max()

    def launch(hb):
        check(lib.rs_scan_fused(_ptr(stream.codes), _ptr(profile.rows), profile.dtype, stream.n,
                                0 if ts is None else ts.ctypes.data, tq.ctypes.data, W, threshold,
                                absmax, mode, hb.capacity, _ptr(hb.pos), _ptr(hb.seq), _ptr(hb.struct),
                                _ptr(hb.counters), _ptr(hb.work), hb.work_bytes, _stream()))
    pos, sq, st, resc = _run_thresholded(stream.n, stream.codes.device, launch, ts is not None, True,
                                         capacity)
    return (pos, sq, st, resc) if return_stats else (pos, sq, st)


def refine_hits_seq(stream, pos, struct_scores, seq_table, threshold):
    """Keep, in order, the candidate windows `pos` (ascending stream positions, e.g. the hits of a
    structure-only scan) whose sequence score also exceeds `threshold` (rs_refine_hits_seq).
    Returns (pos, seq_scores float32, struct_scores | None)."""
    ts = _table(seq_table, 4)
    dev = stream.codes.device
    pos = np.ascontiguousarray(pos, np.int64)
    k = len(pos)
    hb = HitBuffers(stream.n, k, dev, True, struct_scores is not None)
    if k:
        hb.pos[:k].copy_(torch.from_numpy(pos))
        if struct_scores is not None:
            hb.struct[:k].copy_(torch.from_numpy(np.ascontiguousarray(struct_scores, np.float64)))
    hb.cand_counters[0] = k
    check(lib.rs_refine_hits_seq(_ptr(stream.codes), stream.n, ts.ctypes.data, ts.shape[0], float(threshold),
                                 _ptr(hb.cand_counters), hb.capacity, _ptr(hb.pos), _ptr(hb.seq), _ptr(hb.struct),
                                 _ptr(hb.counters), _ptr(hb.work), hb.work_bytes, _stream()))
    found = int(hb.counters[0].item())
    return (hb.pos[:found].cpu().numpy(), hb.seq[:found].cpu().numpy(),
            hb.struct[:found].cpu().numpy() if struct_scores is not None else None)


class BackgroundFusedScan(object):
    """Combined scan of device-resident streams whose sequence background is computed from the
    same data (BASELINE config 4: "computed background").

    The reference runs compute_background over the whole input, then builds the log-odds, then
    scans (rnascan.py:507-521).  Only the SEQUENCE table depends on those counts (the averaged
    profile mode cannot compute a structure background, rnascan.py:533-540), and combine() is an
    AND of two separately thresholded result sets (rnascan.py:416-434).

    W <= 16 (sequence first): histogram -> (all-reduce) -> counts to the host -> exact sequence table ->
    rs_scan_fused_seqfirst_counted, which reads the profile rows of the windows whose sequence score
    passes and of no other (a fraction of a per cent of the 28 B per position at typical thresholds).

    W > 16, or structure_first=True (kept for A/B measurements): the structure-only candidate scan
    starts at once on the caller's stream while histogram -> all-reduce -> counts D2H run on a side
    stream; rs_scan_fused_resolve then keeps the candidates whose sequence score passes too.

    Both orders give results identical to histogram -> tables -> rs_scan_fused(RS_MODE_AND).
    """

    def __init__(self, n, device=None, capacity=None, structure_first=False):
        require_cuda()
        self.device = torch.device(device or "cuda")
        self.n = int(n)
        self.structure_first = bool(structure_first)
        self.side = torch.cuda.Stream(device=self.device, priority=-1)
        self.counts = torch.zeros(8, dtype=torch.int64, device=self.device)
        self.counts_host = torch.zeros(8, dtype=torch.int64).pin_memory()
        self.ready = torch.cuda.Event()
        self.hb = HitBuffers(self.n, int(capacity) if capacity else max(1 << 16, self.n // 256), self.device)
        self.launches = 0
        # Very long streams: the histogram's second read of the symbols (1 of 30 B per position, competing with the scan
        # for HBM) costs more than waiting for the counts until the scan has finished -- the scan kernel then counts
        # the letters itself (rs_scan_fused_candidates_counting).  Measured: a gain from ~4 * 10^8 symbols on (DESIGN.md 3.1).
        self.count_in_kernel = self.n >= self.COUNT_IN_KERNEL_FROM

    COUNT_IN_KERNEL_FROM = 400_000_000

    def launch(self, codes, profile_rows, profile_dtype, W, struct_table, seq_table_fn, threshold,
               absrow_max, all_reduce=None):
        """Enqueue one whole pass.  codes / profile_rows: device tensors (padded); seq_table_fn(counts
        int64[8]) -> (W, 4) table.  The host blocks only until the COUNTS are on the host (side
        stream); the caller's stream keeps running.  Read the outcome with results()."""
        n, hb = self.n, self.hb
        tq = _table(struct_table, 7)
        main = torch.cuda.current_stream(self.device)
        if W <= self.SEQUENCE_FIRST_MAX_W and not self.structure_first:
            return self._launch_sequence_first(codes, profile_rows, profile_dtype, W, tq, seq_table_fn, threshold,
                                               all_reduce, main)
        self.side.wait_stream(main)                         # inputs ready; previous pass finished with the buffers
        # the big kernel first, so that the host-side cost of the side-stream calls (the collective above
        # all) is spent while the device is already busy
        tiles = ctypes.c_int64(0)
        if self.count_in_kernel and profile_dtype == _lib.RS_F32 and W <= 24 and n >= W and \
                filter_applies(tq, threshold, absrow_max):
            self.counts.zero_()
            check(lib.rs_scan_fused_candidates_counting(_ptr(codes), _ptr(profile_rows), profile_dtype, n, tq.ctypes.data, W,
                                                        float(threshold), float(absrow_max), hb.capacity,
                                                        _ptr(hb.cand_counters), _ptr(self.counts), _ptr(hb.work),
                                                        hb.work_bytes, ctypes.addressof(tiles), main.cuda_stream))
            if all_reduce is not None:
                all_reduce(self.counts)                     # the path's only collective
            self.counts_host.copy_(self.counts, non_blocking=True)
            main.synchronize()
            ts = _table(seq_table_fn(self.counts_host.numpy()), 4)
            if ts.shape[0] != W:
                raise ValueError("sequence and structure motifs must have the same width")
            check(lib.rs_scan_fused_resolve(_ptr(codes), n, ts.ctypes.data, W, float(threshold), tiles.value,
                                            hb.capacity, _ptr(hb.pos), _ptr(hb.seq), _ptr(hb.struct),
                                            _ptr(hb.counters), _ptr(hb.work), hb.work_bytes, main.cuda_stream))
            self.launches = 2          # candidate scan (+ counts), sequence check + ordering
            return ts
        check(lib.rs_set_reserved_sms(1 if all_reduce is not None else 0))    # room for the collective's kernel
        try:
            check(lib.rs_scan_fused_candidates(_ptr(codes), _ptr(profile_rows), profile_dtype, n, tq.ctypes.data, W,
                                               float(threshold), float(absrow_max), hb.capacity,
                                               _ptr(hb.cand_counters), _ptr(hb.work), hb.work_bytes,
                                               ctypes.addressof(tiles), main.cuda_stream))
        finally:
            lib.rs_set_reserved_sms(0)
        with torch.cuda.stream(self.side):
            self.counts.zero_()
            check(lib.rs_hist_rna(_ptr(codes), n, _ptr(self.counts), self.side.cuda_stream))
            if all_reduce is not None:
                all_reduce(self.counts)                     # the path's only collective
            self.counts_host.copy_(self.counts, non_blocking=True)
            self.ready.record(self.side)
        self.ready.synchronize()
        ts = _table(seq_table_fn(self.counts_host.numpy()), 4)
        if ts.shape[0] != W:
            raise ValueError("sequence and structure motifs must have the same width")
        check(lib.rs_scan_fused_resolve(_ptr(codes), n, ts.ctypes.data, W, float(threshold), tiles.value,
                                        hb.capacity, _ptr(hb.pos), _ptr(hb.seq), _ptr(hb.struct),
                                        _ptr(hb.counters), _ptr(hb.work), hb.work_bytes, main.cuda_stream))
        main.wait_stream(self.side)
        self.launches = 3          # hist, candidate scan, sequence check + ordering
        return ts

    SEQUENCE_FIRST_MAX_W = 16

    def _launch_sequence_first(self, codes, profile_rows, profile_dtype, W, tq, seq_table_fn, threshold, all_reduce,
                               main):
        n, hb = self.n, self.hb
        self.counts.zero_()
        check(lib.rs_hist_rna(_ptr(codes), n, _ptr(self.counts), main.cuda_stream))
        if all_reduce is not None:
            all_reduce(self.counts)                         # the path's only collective
        self.counts_host.copy_(self.counts, non_blocking=True)
        self.ready.record(main)
        self.ready.synchronize()
        ts = _table(seq_table_fn(self.counts_host.numpy()), 4)
        if ts.shape[0] != W:
            raise ValueError("sequence and structure motifs must have the same width")
        check(lib.rs_scan_fused_seqfirst_counted(_ptr(codes), _ptr(profile_rows), profile_dtype, n, ts.ctypes.data,
                                                 tq.ctypes.data, W, float(threshold), hb.capacity, _ptr(hb.pos),
                                                 _ptr(hb.seq), _ptr(hb.struct), _ptr(hb.cand_counters),
                                                 _ptr(hb.counters), _ptr(hb.work), hb.work_bytes, main.cuda_stream))
        self.launches = 5          # hist, decision table, sequence scan, finish (profile rows), compaction
        return ts

    def results(self):
        """(pos, seq_scores, struct_scores) on the host, or None when the candidate buffer overflowed
        (grow() and launch again)."""
        hb = self.hb
        cand = int(hb.cand_counters[0].item())
        if cand > hb.capacity:
            return None
        found = int(hb.counters[0].item())
        return (hb.pos[:found].cpu().numpy(), hb.seq[:found].cpu().numpy(), hb.struct[:found].cpu().numpy())

    def grow(self):
        cand = int(self.hb.cand_counters[0].item())
        self.hb = HitBuffers(self.n, max(cand, 2 * self.hb.capacity), self.device)


def scan_fused_bg(stream, profile, struct_table, seq_table_fn, threshold, all_reduce=None, capacity=None):
    """histogram + combined scan in one overlapped pass (see BackgroundFusedScan).
    Returns (pos, seq_scores, struct_scores, counts int64[8])."""
    if stream.n != profile.n:
        raise ValueError("symbol stream and profile stream differ in length")
    if float(threshold) == float("-inf"):
        raise ValueError("scan_fused_bg needs a finite threshold (use histogram() + scan_fused for -inf)")
    W = _table(struct_table, 7).shape[0]
    job = BackgroundFusedScan(stream.n, stream.codes.device, capacity)
    absmax = profile.absrow_max()
    while True:
        job.launch(stream.codes, profile.rows, profile.dtype, W, struct_table, seq_table_fn, threshold,
                   absmax, all_reduce)
        res = job.results()
        if res is not None:
            return res + (job.counts_host.numpy().copy(),)
        job.grow()


def _background_shift(local8, global8, A):
    """max over letters of |log2(b_local / b_global)| for backgrounds b = (count + 1) / (sum + A) renormalised
    (rnascan.py:445-457): a window score computed with one background differs from the other by at most W
    times this."""
    import math
    worst = 0.0
    bl = [(float(local8[c]) + 1) / (float(sum(int(v) for v in local8[:A])) + A) for c in range(A)]
    bg = [(float(global8[c]) + 1) / (float(sum(int(v) for v in global8[:A])) + A) for c in range(A)]
    sl, sg = sum(bl), sum(bg)
    for c in range(A):
        worst = max(worst, abs(math.log2((bl[c] / sl) / (bg[c] / sg))))
    return worst * (1 + 1e-9) + 1e-12


class BackgroundOneHotScan(object):
    """Thresholded one-hot scan (sequence or structure contexts, W <= 16) whose background is computed
    from the same data (BASELINE config 2: default `rnascan -p pfm seqs.fa`).

    Reference order: compute_background -> log-odds -> scan (rnascan.py:507-521).  The exact log-odds
    need the host (Python's math.log); waiting for them would idle the device between the histogram and
    the scan.  Here the device derives a provisional table from the counts itself and selects candidate
    windows with a safety margin (rs_scan_onehot_begin) while the counts travel to
    the host and `table_fn` builds the exact table; rs_scan_onehot_finish then decides and scores every
    candidate with the exact table.  Results are identical to histogram -> table -> rs_scan_seq."""

    def __init__(self, n, kind, device=None, capacity=None):
        require_cuda()
        self.device = torch.device(device or "cuda")
        self.n, self.kind = int(n), kind
        self.A = 4 if kind == "rna" else 7
        self.side = torch.cuda.Stream(device=self.device, priority=-1)
        self.counts = torch.zeros(8, dtype=torch.int64, device=self.device)
        self.counts_next = torch.zeros(8, dtype=torch.int64, device=self.device)   # unsharded: zeroed by the device
        self.counts_global = torch.zeros(8, dtype=torch.int64, device=self.device)
        self.counts_host = torch.zeros(16, dtype=torch.int64).pin_memory()      # [0:8] global, [8:16] this shard
        self.note = torch.zeros(8, dtype=torch.int64).pin_memory()    # written by the device: (tag << 48) | count
        self.epoch = 0
        self._clean = True                                   # self.counts holds zeros
        self.counted = torch.cuda.Event()
        self.rescanned = False
        self.ready = torch.cuda.Event()
        self.hb = HitBuffers(self.n, int(capacity) if capacity else max(1 << 16, self.n // 256), self.device,
                             kind == "rna", kind != "rna")
        self.launches = 4          # hist, decision table (k-mers), scan, finish

    def launch(self, codes, prob, table_fn, threshold, all_reduce=None, extra_margin=0.0, shard_margin=0.05):
        """codes: device tensor (padded); prob: (W, A) probabilities in device column order;
        table_fn(counts int64[8]) -> exact (W, A) log-odds table.  Returns that table."""
        n, hb, A = self.n, self.hb, self.A
        prob = _table(prob, A)
        W = prob.shape[0]
        main = torch.cuda.current_stream(self.device)
        if all_reduce is None:
            return self._launch_unsharded(codes, prob, table_fn, threshold, extra_margin, main)
        self.counts.zero_()
        self._clean = False
        check((lib.rs_hist_rna if A == 4 else lib.rs_hist)(_ptr(codes), n, _ptr(self.counts), main.cuda_stream))
        self.counted.record(main)
        # Sharded runs: the decision pass starts from THIS shard's counts with `shard_margin` of extra slack
        # while the all-reduce and the trip to the host run beside it; the slack is verified below against
        # the global counts (a shard whose composition differs more is re-scanned from the global counts).
        sharded = all_reduce is not None
        slack = float(extra_margin) + (float(shard_margin) if sharded else 0.0)
        check(lib.rs_set_reserved_sms(1 if sharded else 0))                   # room for the collective's kernel
        try:
            check(lib.rs_scan_onehot_begin(A, _ptr(codes), n, _ptr(self.counts), prob.ctypes.data, W, float(threshold),
                                           slack, hb.capacity, _ptr(hb.work), hb.work_bytes, main.cuda_stream))
        finally:
            lib.rs_set_reserved_sms(0)
        with torch.cuda.stream(self.side):                  # counts -> (all ranks) -> host, beside the scan
            self.side.wait_event(self.counted)
            self.counts_host[8:].copy_(self.counts, non_blocking=True)          # local
            if sharded:
                self.counts_global.copy_(self.counts)
                all_reduce(self.counts_global)              # the path's only collective
                self.counts_host[:8].copy_(self.counts_global, non_blocking=True)
            else:
                self.counts_host[:8].copy_(self.counts, non_blocking=True)
            self.ready.record(self.side)
        self.ready.synchronize()
        ch = self.counts_host.numpy()
        table = _table(table_fn(ch[:8]), A)
        if table.shape[0] != W:
            raise ValueError("table_fn returned a table of another width")
        self.rescanned = False
        if sharded and W * _background_shift(ch[8:], ch[:8], A) > float(shard_margin) * 0.999:
            # this shard's composition is too far from the global one for the slack: decide from global counts
            main.wait_stream(self.side)
            check(lib.rs_scan_onehot_begin(A, _ptr(codes), n, _ptr(self.counts_global), prob.ctypes.data, W,
                                           float(threshold), float(extra_margin), hb.capacity, _ptr(hb.work),
                                           hb.work_bytes, main.cuda_stream))
            self.rescanned = True
        check(lib.rs_scan_onehot_finish(A, _ptr(codes), n, table.ctypes.data, W, float(threshold), hb.capacity,
                                        _ptr(hb.pos), _ptr(hb.seq if A == 4 else hb.struct), _ptr(hb.counters),
                                        _ptr(hb.work), hb.work_bytes, main.cuda_stream))
        main.wait_stream(self.side)
        return table

    NOTIFY_TIMEOUT_S = 20.0

    def _launch_unsharded(self, codes, prob, table_fn, threshold, extra_margin, main):
        """One device, no collective: no side stream, no copy, no event.  The first kernel of the decision pass
        stores the counts, tagged with this launch's number, into the pinned host buffer
        (rs_scan_onehot_begin_notify); the host spins until all eight words carry the tag, builds the exact table while the scan runs and queues the finish behind it.  The same
        kernel zeroes the OTHER counter array, the next launch's histogram target."""
        n, hb, A = self.n, self.hb, self.A
        W = prob.shape[0]
        sptr = main.cuda_stream
        if not self._clean:
            self.counts.zero_()
        self._clean = False                                  # until the device has zeroed the next target
        check((lib.rs_hist_rna if A == 4 else lib.rs_hist)(_ptr(codes), n, _ptr(self.counts), sptr))
        self.epoch = self.epoch % 65535 + 1                  # 1..65535; the buffer starts as zeros
        ch, note = self.counts_host.numpy(), self.note.numpy().view(np.uint64)
        check(lib.rs_scan_onehot_begin_notify(A, _ptr(codes), n, _ptr(self.counts), prob.ctypes.data, W,
                                              float(threshold), float(extra_margin), hb.capacity, _ptr(hb.work),
                                              hb.work_bytes, self.note.data_ptr(), self.epoch,
                                              _ptr(self.counts_next), sptr))
        self.counts, self.counts_next = self.counts_next, self.counts
        self._clean = True
        tag, spins, t0 = np.uint64(self.epoch), 0, None
        shift = np.uint64(48)
        while not ((note >> shift) == tag).all():
            spins += 1
            if spins & 0x3FF == 0:                           # every 1024 polls: look at the clock
                now = time.perf_counter()
                t0 = t0 or now
                if now - t0 > self.NOTIFY_TIMEOUT_S:
                    torch.cuda.synchronize(self.device)      # surfaces a device error if that is the cause
                    raise RuntimeError("the device never reported the background counts")
        ch[:8] = (note & np.uint64((1 << 48) - 1)).astype(np.int64)
        ch[8:] = ch[:8]
        table = _table(table_fn(ch[:8]), A)
        if table.shape[0] != W:
            raise ValueError("table_fn returned a table of another width")
        self.rescanned = False
        check(lib.rs_scan_onehot_finish(A, _ptr(codes), n, table.ctypes.data, W, float(threshold), hb.capacity,
                                        _ptr(hb.pos), _ptr(hb.seq if A == 4 else hb.struct), _ptr(hb.counters),
                                        _ptr(hb.work), hb.work_bytes, sptr))
        return table

    def results(self):
        """(pos, scores, n_false_candidates) on the host, or None when the hit buffer overflowed
        (grow() and launch again)."""
        hb = self.hb
        found, false_cand = (int(v) for v in hb.counters.cpu().numpy())
        if found > hb.capacity:
            return None
        pos = hb.pos[:found].cpu().numpy()
        sc = (hb.seq if self.A == 4 else hb.struct)[:found].cpu().numpy()
        if false_cand:                                      # candidates the exact table rejected
            keep = pos >= 0
            pos, sc = pos[keep], sc[keep]
        return pos, sc, false_cand

    def grow(self):
        found = int(self.hb.counters[0].item())
        self.hb = HitBuffers(self.n, max(found, 2 * self.hb.capacity), self.device, self.A == 4, self.A != 4)


def scan_onehot_bg(stream, prob, table_fn, threshold, all_reduce=None, capacity=None, extra_margin=0.0):
    """histogram + thresholded one-hot scan with the host round trip hidden (see BackgroundOneHotScan).
    Returns (pos, scores, counts int64[8], n_false_candidates)."""
    if float(threshold) == float("-inf"):
        raise ValueError("scan_onehot_bg needs a finite threshold")
    kind = stream.kind or "struct"
    job = BackgroundOneHotScan(stream.n, kind, stream.codes.device, capacity)
    while True:
        job.launch(stream.codes, prob, table_fn, threshold, all_reduce, extra_margin)
        res = job.results()
        if res is not None:
            return res[0], res[1], job.counts_host.numpy()[:8].copy(), res[2]
        job.grow()


def scan_batched(stream, profile, seq_tables, struct_tables, threshold, capacity=None, path=0):
    """Many motif pairs over the same resident streams (BASELINE config 5).

    seq_tables: list of (W_m, 4) arrays or None (structure-only); struct_tables: list of
    (W_m, 7) arrays.  Returns (motif int32[], pos int64[], seq float32[]|None, struct
    float64[], bases int64[M+1]) with hits grouped by motif, ordered by position."""
    M = len(struct_tables)
    if M == 0:
        raise ValueError("no motifs")
    if seq_tables is not None and len(seq_tables) != M:
        raise ValueError("sequence and structure motif lists differ in length")
    widths, qs, stride = _pack_tables(struct_tables, 7)
    ss = None
    if seq_tables is not None:
        seq_widths, ss, _ = _pack_tables(seq_tables, 4)
        differ = np.nonzero(seq_widths != widths)[0]
        if len(differ):
            raise ValueError("motif %d: sequence and structure widths differ" % differ[0])
    if stream.n != profile.n:
        raise ValueError("symbol stream and profile stream differ in length")
    threshold = float(threshold)
    if threshold == float("-inf"):
        raise ValueError("scan_batched needs a finite threshold (use the dense entry points for -inf)")
    mode = _lib.RS_MODE_STRUCT if ss is None else _lib.RS_MODE_AND
    absmax = profile.absrow_max()
    dev = stream.codes.device
    cap = int(capacity) if capacity else max(1 << 16, stream.n // 64)
    counters = torch.zeros(2 * M, dtype=torch.int64, device=dev)
    bases = torch.zeros(M + 1, dtype=torch.int64, device=dev)
    check(lib.rs_set_batched_path(int(path)))
    # float64 rows (parsed text): the tensor-core filter runs on their float32 shadow
    shadow = profile.shadow() if (path != 1 and M >= 32 or path == 2) and hasattr(profile, "shadow") else None
    while True:
        hb = HitBuffers(stream.n, cap, dev)
        hb.work_bytes = int(lib.rs_scan_batched_workspace_bytes(stream.n, M, stride, cap))
        hb.work = torch.empty(hb.work_bytes, dtype=torch.uint8, device=dev)
        motif = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
        if shadow is not None:
            check(lib.rs_scan_batched_shadow(_ptr(stream.codes), _ptr(shadow), _ptr(profile.rows), stream.n, M,
                                             widths.ctypes.data, 0 if ss is None else ss.ctypes.data, qs.ctypes.data,
                                             stride, threshold, absmax, mode, cap, _ptr(motif), _ptr(hb.pos),
                                             _ptr(hb.seq), _ptr(hb.struct), _ptr(counters), _ptr(bases), _ptr(hb.work),
                                             hb.work_bytes, _stream()))
        else:
            check(lib.rs_scan_batched(_ptr(stream.codes), _ptr(profile.rows), profile.dtype, stream.n, M,
                                      widths.ctypes.data, 0 if ss is None else ss.ctypes.data, qs.ctypes.data,
                                      stride, threshold, absmax, mode, cap, _ptr(motif), _ptr(hb.pos),
                                      _ptr(hb.seq), _ptr(hb.struct), _ptr(counters), _ptr(bases), _ptr(hb.work),
                                      hb.work_bytes, _stream()))
        b = bases.cpu().numpy()
        total = int(b[-1])
        if total <= cap:
            lib.rs_set_batched_path(0)
            return (motif[:total].cpu().numpy(), hb.pos[:total].cpu().numpy(),
                    hb.seq[:total].cpu().numpy() if ss is not None else None,
                    hb.struct[:total].cpu().numpy(), b)
        cap = total


MANY_MAX_W = 16                 # widest motif scan_onehot_many takes


def _pack_tables(tables, A):
    """(widths int32[M], packed, stride): the checked (W_m, A) tables zero-padded into one (M, stride, A) float64
    array, stride = the widest W_m, as the grouped scans read them."""
    ts = [_table(t, A) for t in tables]
    widths = np.array([t.shape[0] for t in ts], dtype=np.int32)
    stride = int(widths.max())
    packed = np.zeros((len(ts), stride, A), np.float64)
    for m, t in enumerate(ts):
        packed[m, :t.shape[0]] = t
    return widths, packed, stride


def _run_many(dev, M, work_bytes, cap, score_dtypes, launch):
    """Run `launch(cap, work, bases, motif, pos, *scores)` of a grouped one-hot scan with output buffers for `cap`
    hits (one score buffer per dtype of `score_dtypes`); re-run with the exact capacity if the hits overflowed.
    Returns (motif, pos, *scores, bases) on the host."""
    if work_bytes < 0:
        check(_lib.RS_ERR_INVALID)
    work = torch.empty(max(work_bytes, 1), dtype=torch.uint8, device=dev)
    bases = torch.zeros(M + 1, dtype=torch.int64, device=dev)
    while True:
        out = [torch.empty(max(cap, 1), dtype=dt, device=dev) for dt in (torch.int32, torch.int64) + score_dtypes]
        launch(cap, work, bases, *out)
        b = bases.cpu().numpy()
        total = int(b[-1])
        if total <= cap:
            return tuple(t[:total].cpu().numpy() for t in out) + (b,)
        cap = total


def scan_onehot_many(stream, tables, threshold, capacity=None):
    """Many one-hot PSSMs over one FASTA symbol stream in one call (rs_scan_onehot_many).

    stream.kind "rna": tables (W_m, 4) in ACGU order, float32 scores as scan_seq; "struct": (W_m, 7) in
    BEHLMRT order, float64 scores as scan_struct_onehot.  Widths 1..16, finite threshold.  Returns
    (motif int32[], pos int64[], scores, bases int64[M+1]) with hits grouped by motif, ordered by position:
    bases[m] .. bases[m+1] is motif m's slice, identical to the per-motif scan."""
    if stream.kind not in ("rna", "struct"):
        raise ValueError("scan_onehot_many takes RNA or structure streams (kind %r)" % (stream.kind,))
    A = 4 if stream.kind == "rna" else 7
    M = len(tables)
    if M == 0:
        raise ValueError("no motifs")
    widths, packed, stride = _pack_tables(tables, A)
    if widths.max() > MANY_MAX_W:
        raise ValueError("scan_onehot_many takes motifs up to %d wide (%d found)" % (MANY_MAX_W, widths.max()))
    threshold = float(threshold)
    if not np.isfinite(threshold):
        raise ValueError("scan_onehot_many needs a finite threshold")
    work_bytes = int(lib.rs_scan_onehot_many_workspace_bytes(A, stream.n, M, stride))

    def launch(cap, work, bases, motif, pos, scores):
        check(lib.rs_scan_onehot_many(A, _ptr(stream.codes), stream.n, M, widths.ctypes.data, packed.ctypes.data,
                                      stride, threshold, cap, _ptr(motif), _ptr(pos),
                                      _ptr(scores) if A == 4 else 0, 0 if A == 4 else _ptr(scores), _ptr(bases),
                                      _ptr(work), work_bytes, _stream()))
    cap = int(capacity) if capacity else max(1 << 16, stream.n // 16)
    return _run_many(stream.codes.device, M, work_bytes, cap, (torch.float32 if A == 4 else torch.float64,), launch)


def scan_pair_onehot_many(seq_stream, struct_stream, seq_tables, struct_tables, threshold, capacity=None):
    """Many (sequence, structure) motif pairs over an RNA stream and the structure stream that lines up with it,
    in one call (rs_scan_pair_onehot_many).

    seq_tables[m] (W_m, 4) in ACGU order and struct_tables[m] (W_m, 7) in BEHLMRT order share one width, 1..16;
    the threshold is finite.  Returns (motif int32[], pos int64[], seq_scores float32[], struct_scores float64[],
    bases int64[M+1]): pair m's slice bases[m] .. bases[m+1], in position order, is exactly what
    scan_pair_onehot returns for that pair."""
    if seq_stream.kind != "rna" or struct_stream.kind != "struct":
        raise ValueError("scan_pair_onehot_many takes an RNA stream and a structure stream (kinds %r, %r)"
                         % (seq_stream.kind, struct_stream.kind))
    if seq_stream.n != struct_stream.n:
        raise ValueError("sequence and structure streams differ in length")
    M = len(seq_tables)
    if M == 0 or len(struct_tables) != M:
        raise ValueError("need as many structure tables as sequence tables (%d, %d), at least one"
                         % (M, len(struct_tables)))
    widths, packed_s, stride = _pack_tables(seq_tables, 4)
    struct_widths, packed_q, _ = _pack_tables(struct_tables, 7)
    if not np.array_equal(widths, struct_widths):
        raise ValueError("sequence and structure motifs of a pair must have the same width")
    if widths.max() > MANY_MAX_W:
        raise ValueError("scan_pair_onehot_many takes motifs up to %d wide (%d found)" % (MANY_MAX_W, widths.max()))
    threshold = float(threshold)
    if not np.isfinite(threshold):
        raise ValueError("scan_pair_onehot_many needs a finite threshold")
    n = seq_stream.n
    work_bytes = int(lib.rs_scan_pair_onehot_many_workspace_bytes(n, M, stride))

    def launch(cap, work, bases, motif, pos, seq, struct):
        check(lib.rs_scan_pair_onehot_many(_ptr(seq_stream.codes), _ptr(struct_stream.codes), n, M,
                                           widths.ctypes.data, packed_s.ctypes.data, packed_q.ctypes.data, stride,
                                           threshold, cap, _ptr(motif), _ptr(pos), _ptr(seq), _ptr(struct),
                                           _ptr(bases), _ptr(work), work_bytes, _stream()))
    cap = int(capacity) if capacity else max(1 << 16, n // 16)
    return _run_many(seq_stream.codes.device, M, work_bytes, cap, (torch.float32, torch.float64), launch)


# --------------------------------------------------------------------------- host-buffer pipeline
class _HitOverflow(Exception):
    def __init__(self, found):
        Exception.__init__(self, "hit buffer overflow")
        self.found = int(found)


class HostFusedScanner(object):
    """Combined sequence + averaged-profile scan of HOST-resident streams.

    The reference-facing call for data that lives in host memory (what the CLI has after
    parsing): the symbol stream (1 B/symbol) goes to the device first so the background
    histogram -- which the log-odds tables depend on -- is known early; the profile stream
    (28 B/row) follows in chunks on a copy stream while the previous chunk is being scanned
    on the compute stream (double buffering).  Chunks overlap by W-1 rows so every window
    is scored exactly once.  All device buffers are allocated once and reused.
    """

    def __init__(self, n, W, chunk_rows=1 << 23, device=None, hits_per_row=1.0 / 64):
        require_cuda()
        self.device = torch.device(device or "cuda")
        self.n, self.W = int(n), int(W)
        self.chunk = max(256, int(chunk_rows) // 256 * 256)
        self.starts = list(range(0, max(self.n - self.W + 1, 1), self.chunk)) if self.n >= self.W else []
        rows = padded_count(min(self.chunk + self.W - 1, max(self.n, 1))) + 256
        self.codes = torch.empty(padded_count(self.n) + 1024, dtype=torch.uint8, device=self.device)
        self.prof = [torch.empty((rows, len(CHANNELS)), dtype=torch.float32, device=self.device)
                     for _ in range(2)]
        self.counts = torch.zeros(8, dtype=torch.int64, device=self.device)
        self.counts_host = torch.zeros(8, dtype=torch.int64).pin_memory()
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.loaded = [torch.cuda.Event() for _ in range(2)]
        self.freed = [torch.cuda.Event() for _ in range(2)]
        cap = max(4096, int(self.chunk * hits_per_row))
        self.hb = [HitBuffers(self.chunk + self.W, cap, self.device) for _ in self.starts]
        if self.hb:                      # one workspace serves all chunks (they run in order)
            for hb in self.hb[1:]:
                hb.work = self.hb[0].work
        self.h2d_bytes = 0
        self.d2h_bytes = 0

    def run(self, h_codes, h_prof, make_tables, threshold, mode=_lib.RS_MODE_AND, absrow_max=1.0,
            all_reduce=None):
        """h_codes: pinned uint8[>= n]; h_prof: pinned float32[>= n, 7];
        make_tables(counts int64[8]) -> (seq_table | None, struct_table).
        Returns (pos, seq_scores, struct_scores) as numpy arrays, positions ascending.  A chunk whose hits do
        not fit its buffer makes the buffers grow and the pass run again."""
        while True:
            try:
                return self._run_once(h_codes, h_prof, make_tables, threshold, mode, absrow_max, all_reduce)
            except _HitOverflow as over:
                cap = int(over.found * 1.25) + 1024
                self.hb = [HitBuffers(self.chunk + self.W, cap, self.device) for _ in self.starts]
                for hb in self.hb[1:]:
                    hb.work = self.hb[0].work

    def _run_once(self, h_codes, h_prof, make_tables, threshold, mode, absrow_max, all_reduce):
        n, W = self.n, self.W
        comp = torch.cuda.current_stream(self.device)
        self.h2d_bytes = self.d2h_bytes = 0
        # -- pass 1: symbols -> device, exact background counts
        self.codes[:n].copy_(h_codes[:n], non_blocking=True)
        self.codes[n:].fill_(_lib.RS_SEP)
        self.h2d_bytes += n
        self.copy_stream.wait_stream(comp)
        # profile chunks start flowing while the histogram runs
        order = self.starts
        def load(k):
            c0 = order[k]
            rows = min(self.chunk + W - 1, n - c0)
            slot = k & 1
            with torch.cuda.stream(self.copy_stream):
                if k >= 2:
                    self.copy_stream.wait_event(self.freed[slot])
                self.prof[slot][:rows].copy_(h_prof[c0:c0 + rows], non_blocking=True)
                self.loaded[slot].record(self.copy_stream)
            self.h2d_bytes += rows * 28
            return rows
        pending = {}
        for k in range(min(2, len(order))):
            pending[k] = load(k)
        self.counts.zero_()
        check(lib.rs_hist_rna(_ptr(self.codes), n, _ptr(self.counts), comp.cuda_stream))
        if all_reduce is not None:
            all_reduce(self.counts)
        self.counts_host.copy_(self.counts, non_blocking=True)
        comp.synchronize()
        self.d2h_bytes += 64
        ts, tq = make_tables(self.counts_host.numpy())
        tq = _table(tq, 7)
        ts = None if ts is None else _table(ts, 4)
        # -- pass 2: scan chunk k while chunk k+1 is in flight
        for k, c0 in enumerate(order):
            rows = pending.pop(k)
            slot = k & 1
            comp.wait_event(self.loaded[slot])
            hb = self.hb[k]
            check(lib.rs_scan_fused(_ptr(self.codes) + c0, _ptr(self.prof[slot]), _lib.RS_F32, rows,
                                    0 if ts is None else ts.ctypes.data, tq.ctypes.data, W, float(threshold),
                                    float(absrow_max), mode, hb.capacity, _ptr(hb.pos), _ptr(hb.seq),
                                    _ptr(hb.struct), _ptr(hb.counters), _ptr(hb.work), hb.work_bytes,
                                    comp.cuda_stream))
            self.freed[slot].record(comp)
            if k + 2 < len(order):
                pending[k + 2] = load(k + 2)
        comp.synchronize()
        # -- results back to the host
        pos_l, seq_l, str_l = [], [], []
        for k, c0 in enumerate(order):
            hb = self.hb[k]
            found = int(hb.counters[0].item())
            self.d2h_bytes += 16
            if found > hb.capacity:
                raise _HitOverflow(found)
            if found:
                pos_l.append(hb.pos[:found].cpu().numpy() + c0)
                str_l.append(hb.struct[:found].cpu().numpy())
                if ts is not None:
                    seq_l.append(hb.seq[:found].cpu().numpy())
                self.d2h_bytes += found * (20 if ts is not None else 16)
        pos = np.concatenate(pos_l) if pos_l else np.zeros(0, np.int64)
        st = np.concatenate(str_l) if str_l else np.zeros(0, np.float64)
        sq = (np.concatenate(seq_l) if seq_l else np.zeros(0, np.float32)) if ts is not None else None
        return pos, sq, st


# --------------------------------------------------------------------------- exact rows on the host: filter + gather + resolve

def _np_ptr(a):
    return 0 if a is None else a.ctypes.data


class HostProfile(object):
    """Averaged-profile rows that stay in HOST memory, row-aligned with a symbol stream.

    `rows`: (n, 7) float64 (what pd.read_table gives the reference, rnascan.py:296-297) or float32,
    C-contiguous numpy array or memmap, channels B,E,H,L,M,R,T, separator rows zero.  Only a FILTER
    FORM of them travels to the device (include/rnascan_b200.h, rs_filter_profile): the rows themselves
    when they are float32, their float32 shadow when they are float64, or the 8-byte quantised form
    `q8` (n, 8) uint8 with `q8_scale` when one is supplied (profile packs) or built with make_q8()."""

    def __init__(self, rows, q8=None, q8_scale=None, stats=None, q4=None):
        if rows.dtype not in (np.float32, np.float64):
            rows = np.ascontiguousarray(rows, dtype=np.float64)
        if rows.ndim != 2 or rows.shape[1] != len(CHANNELS):
            raise ValueError("profile must have shape (L, 7) in channel order %s" % CHANNELS)
        if not rows.flags["C_CONTIGUOUS"]:
            rows = np.ascontiguousarray(rows)
        self.rows = rows
        self.n = int(rows.shape[0])
        self.dtype = _lib.RS_F32 if rows.dtype == np.float32 else _lib.RS_F64
        self.q8, self.q8_scale = q8, q8_scale
        self.q4 = q4                                 # (n, 4) uint8 view of the 4-byte quantised rows (make_q4)
        self.page_locked = None                      # (fn(form) -> pinned tensor | None, {form: array it stands for})
        self._stats = None if stats is None else tuple(float(v) for v in stats)

    def stats(self):
        """(max abs row sum, #non-finite, #negative, max |value|), computed once on host threads."""
        if self._stats is None:
            out = np.zeros(4, np.float64)
            check(lib.rs_host_rows_stats(_np_ptr(self.rows), self.dtype, self.n, HOST_THREADS, out.ctypes.data))
            self._stats = tuple(float(v) for v in out)
        return self._stats

    def absrow_max(self):
        mx, bad, neg, _ = self.stats()
        return float("nan") if (bad or neg) else mx

    def make_q8(self, codes=None, out=None):
        """Build the quantised filter form (byte 7 = codes[r], 0 when codes is None).  Returns False --
        and leaves q8 unset -- when the rows do not fit it (negative / non-finite entries)."""
        mx, bad, neg, vmax = self.stats()
        if bad or neg or self.n == 0:
            return False
        scale = vmax if vmax > 0 else 1.0
        q8 = np.empty((self.n, 8), np.uint8) if out is None else out
        n_bad = ctypes.c_int64(0)
        check(lib.rs_host_quantize_q8(_np_ptr(self.rows), self.dtype, self.n, _np_ptr(codes), float(scale),
                                      q8.ctypes.data, HOST_THREADS, ctypes.byref(n_bad)))
        if n_bad.value:
            return False
        self.q8, self.q8_scale = q8, float(scale)
        return True


def _make_q4(self, codes=None, out=None):
    """Build the 4-byte quantised filter form (seven floored 4-bit channels + the symbol in the top nibble).
    `out`: a (n, 4) uint8 array to fill.  Returns False when the rows do not fit it."""
    mx, bad, neg, vmax = self.stats()
    if bad or neg or self.n == 0:
        return False
    scale = vmax if vmax > 0 else 1.0
    q4 = np.empty((self.n, 4), np.uint8) if out is None else out
    n_bad = ctypes.c_int64(0)
    check(lib.rs_host_quantize_q4(_np_ptr(self.rows), self.dtype, self.n, _np_ptr(codes), float(scale),
                                  q4.ctypes.data, HOST_THREADS, ctypes.byref(n_bad)))
    if n_bad.value:
        return False
    self.q4, self.q8_scale = q4, float(scale)
    return True


HostProfile.make_q4 = _make_q4


def q4_guard(struct_table, scale):
    """The 4-bit form's guard band in score units: scale / 15 times the sum of the table's positive entries (rows
    with -inf count their positive part)."""
    t = np.asarray(struct_table, np.float64)
    return float(scale) / 15.0 * float(np.where(np.isfinite(t) & (t > 0), t, 0.0).sum())


def filter_applies(struct_table, threshold, absrow_max):
    """Can the fp32 filter kernels decide candidates for this scan?  (Else: the exact fp64 kernel.)"""
    t = np.asarray(struct_table, np.float64)
    return bool(t.shape[0] <= 24 and np.isfinite(float(threshold)) and np.isfinite(absrow_max) and
                0 <= absrow_max < 1e30 and not np.isnan(t).any() and not (t == np.inf).any())


def pick_filter_form(hp, struct_table, threshold):
    """The smallest filter form whose guard band leaves the threshold selective: 4 bytes per position when that
    form's band is at most 0.4 of a positive threshold, else 8 bytes; rows without a quantised form go as float32
    (their own dtype, or the float32 shadow of float64 rows)."""
    if hp.q4 is not None and threshold > 0 and q4_guard(struct_table, hp.q8_scale) <= 0.4 * threshold:
        return "q4"
    if hp.q8 is not None:
        return "q8"
    return "f32" if hp.dtype == _lib.RS_F32 else "shadow"


class HostProfileScanner(object):
    """Averaged-profile scan (optionally AND the sequence PSSM) of HOST-resident streams through
    rs_filter_profile -> rs_host_gather_windows -> rs_resolve_candidates.

    Chunks of the filter form go to the device double-buffered on a copy stream while the previous chunk is
    being filtered; candidate positions come back, their exact rows are gathered from host memory and one
    small launch decides and scores them in the reference's arithmetic.  Bytes over the link per position:
    8 (quantised rows, symbol included) or 1 + 28 (float32 rows / shadow) instead of 1 + 56.  All device and
    pinned buffers are allocated once; run() may be called repeatedly (bench.py) and regrows the candidate
    buffers when a threshold lets more windows through than they hold."""

    def __init__(self, n, W, form, chunk_rows=1 << 23, device=None, cand_per_row=1.0 / 256):
        require_cuda()
        if form not in ("f32", "shadow", "q8", "q4"):
            raise ValueError("form must be 'f32', 'shadow', 'q8' or 'q4'")
        self.device = torch.device(device or "cuda")
        self.n, self.W, self.form = int(n), int(W), form
        self.chunk = max(256, int(chunk_rows) // 256 * 256)
        self.starts = list(range(0, max(self.n - self.W + 1, 1), self.chunk)) if self.n >= self.W else []
        self.quantised = form in ("q8", "q4")     # the rows carry the symbols: no separate symbol stream
        if self.quantised and not self.starts and self.n > 0:
            self.starts = [0]                       # nothing to scan, but the symbols still count
        self.rows_max = padded_count(min(self.chunk + self.W - 1, max(self.n, 1))) + 256
        cols, tdt = ((8 if form == "q8" else 4), torch.uint8) if self.quantised else (len(CHANNELS), torch.float32)
        self.cols, self.tdt = cols, tdt
        self.dbuf = [torch.empty((self.rows_max, cols), dtype=tdt, device=self.device) for _ in range(2)]
        # Rows past the end of a chunk must read as separators.  A full chunk always ends at the same row, so the
        # rows behind it are set ONCE here; only a shorter (last) chunk needs them set again after its copy -- a
        # fill kernel between every two copies on the copy stream kept the copy engine from running back to back.
        self.full_rows = min(self.chunk + self.W - 1, max(self.n, 1))
        if self.quantised:
            for b in self.dbuf:
                b.fill_(0xFF)
        self.stage = None                           # pinned staging, made on first use with a pageable source
        self.codes = None if self.quantised else torch.empty(padded_count(self.n) + 1024, dtype=torch.uint8,
                                                             device=self.device)
        self.counts = torch.zeros(8, dtype=torch.int64, device=self.device)
        self.counts_host = torch.zeros(8, dtype=torch.int64, pin_memory=True)
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.loaded = [torch.cuda.Event() for _ in range(2)]
        self.freed = [torch.cuda.Event() for _ in range(2)]
        self.cap = max(4096, int(self.chunk * cand_per_row))
        self._alloc_cand()
        self.h2d_bytes = self.d2h_bytes = 0
        self.n_candidates = self.n_filter_pass = self.n_struct_candidates = 0
        self.launches = 0

    def _alloc_cand(self):
        k = max(len(self.starts), 1)
        self.cand = torch.empty((k, self.cap), dtype=torch.int64, device=self.device)
        # 4-bit rows: every candidate's packed symbols, for the sequence table that arrives after the filter pass
        self.cand_sym = torch.empty((k, self.cap), dtype=torch.int64, device=self.device) if self.form == "q4" else None
        self.cand_counters = torch.zeros((k, 2), dtype=torch.int64, device=self.device)
        self.cand_counters_host = torch.zeros((k, 2), dtype=torch.int64, pin_memory=True)
        self.work_bytes = int(lib.rs_filter_workspace_bytes(self.chunk + self.W + 256, self.cap))
        self.work = torch.empty(self.work_bytes, dtype=torch.uint8, device=self.device)

    # -- chunk k of the filter form -> device buffer k & 1 (copy stream)
    def _load(self, k, src):
        c0 = self.starts[k]
        rows = min(self.chunk + self.W - 1, self.n - c0)
        slot = k & 1
        if isinstance(src, torch.Tensor):           # pinned host tensor of the filter form: straight from it
            piece = src[c0:c0 + rows]
        else:                                       # numpy / memmap: through pinned staging (and, for float64
            if self.stage is None:                  # rows, the conversion to the float32 shadow on the way)
                self.stage = [torch.empty((self.rows_max, self.cols), dtype=self.tdt, pin_memory=True)
                              for _ in range(2)]
            if k >= 2:
                self.loaded[slot].synchronize()     # the previous copy out of this staging buffer is done
            st = self.stage[slot].numpy()
            part = src[c0:c0 + rows]
            if part.dtype == np.float64:
                part = np.ascontiguousarray(part)
                check(lib.rs_host_rows_to_f32(part.ctypes.data, rows * self.cols, st.ctypes.data, HOST_THREADS))
            elif part.flags["C_CONTIGUOUS"] and part.dtype == st.dtype:
                check(lib.rs_host_copy(st.ctypes.data, part.ctypes.data, part.nbytes, HOST_THREADS))
            else:
                np.copyto(st[:rows], part)
            piece = self.stage[slot][:rows]
        with torch.cuda.stream(self.copy_stream):
            if k >= 2:
                self.copy_stream.wait_event(self.freed[slot])
            self.dbuf[slot][:rows].copy_(piece, non_blocking=True)
            if self.quantised and rows != self.full_rows:      # a short chunk: separators behind it (see __init__)
                self.dbuf[slot][rows:rows + 512].fill_(0xFF)
            self.loaded[slot].record(self.copy_stream)
        self.h2d_bytes += rows * self.cols * (1 if self.quantised else 4)
        return rows

    def run(self, codes, filt_src, exact_rows, struct_table, seq, threshold, absrow_max, q8_scale=1.0,
            all_reduce=None, exact_codes=None):
        """codes: uint8[n] host symbols (numpy or pinned tensor; ignored for 'q8', whose rows carry them);
        filt_src: the filter form on the host -- float32 / float64 (n, 7) or uint8 (n, 8), numpy, memmap or
        pinned tensor; exact_rows: (n, 7) float32 | float64 numpy array or memmap the candidates are gathered
        from; seq: None (structure only), a (W, 4) table, or a callable counts int64[8] -> table (background
        computed from the data, rnascan.py:507-511: the counts are taken on the device in the same pass);
        exact_codes: host symbols for the gather when `codes` is None ('q8': byte 7 of filt_src serves).
        Returns (pos int64[], seq float32[] | None, struct float64[]), positions ascending."""
        n, W = self.n, self.W
        tq = _table(struct_table, 7)
        if tq.shape[0] != W:
            raise ValueError("structure table width differs from the scanner's")
        threshold = float(threshold)
        comp = torch.cuda.current_stream(self.device)
        deferred_seq = callable(seq)
        ts = None if (seq is None or deferred_seq) else _table(seq, 4)
        fmt = {"f32": _lib.RS_ROWS_F32, "shadow": _lib.RS_ROWS_F32_SHADOW, "q8": _lib.RS_ROWS_Q8,
               "q4": _lib.RS_ROWS_Q4}[self.form]
        want_sym = self.form == "q4" and deferred_seq
        while True:
            self.h2d_bytes = self.d2h_bytes = 0
            self.launches = 0
            self.copy_stream.wait_stream(comp)
            if not self.quantised:
                h = codes if isinstance(codes, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(codes))
                self.codes[:n].copy_(h[:n], non_blocking=True)
                self.codes[n:].fill_(_lib.RS_SEP)
                self.h2d_bytes += n
            if deferred_seq:
                self.counts.zero_()
                if not self.quantised:
                    check(lib.rs_hist_rna(_ptr(self.codes), n, _ptr(self.counts), comp.cuda_stream))
                    self.launches += 1
            pending = {}
            for k in range(min(2, len(self.starts))):
                pending[k] = self._load(k, filt_src)
            for k, c0 in enumerate(self.starts):
                rows = pending.pop(k)
                slot = k & 1
                comp.wait_event(self.loaded[slot])
                count_rows = min(self.chunk, n - c0)
                want_counts = deferred_seq and self.quantised
                check(lib.rs_filter_profile(0 if self.quantised else _ptr(self.codes) + c0, _ptr(self.dbuf[slot]),
                                            fmt, float(q8_scale), rows, 0 if ts is None else ts.ctypes.data,
                                            tq.ctypes.data, W, threshold, float(absrow_max), c0, count_rows,
                                            _ptr(self.counts) if want_counts else 0, self.cap, _ptr(self.cand[k]),
                                            _ptr(self.cand_sym[k]) if want_sym else 0,
                                            _ptr(self.cand_counters[k]), _ptr(self.work), self.work_bytes,
                                            comp.cuda_stream))
                self.launches += 2                  # filter + ordering
                self.freed[slot].record(comp)
                if k + 2 < len(self.starts):
                    pending[k + 2] = self._load(k + 2, filt_src)
            if deferred_seq and all_reduce is None:
                self.counts_host.copy_(self.counts, non_blocking=True)
                self.d2h_bytes += 64
            self.cand_counters_host.copy_(self.cand_counters, non_blocking=True)
            comp.synchronize()
            cc = self.cand_counters_host.numpy()[:len(self.starts)]
            self.d2h_bytes += cc.size * 8
            found = cc[:, 0].copy() if len(self.starts) else np.zeros(0, np.int64)     # (cc views the pinned buffer)
            if len(found) and int(found.max()) > self.cap:
                self.cap = int(found.max() * 1.25) + 1024
                self._alloc_cand()
                continue
            break
        if deferred_seq and all_reduce is not None:
            # the path's only collective -- outside the regrow loop: every rank calls it exactly once per run
            all_reduce(self.counts)
            self.counts_host.copy_(self.counts, non_blocking=True)
            comp.synchronize()
            self.d2h_bytes += 64
        self.n_filter_pass = int(cc[:, 1].sum()) if len(self.starts) else 0
        if deferred_seq:
            ts = _table(seq(self.counts_host.numpy()), 4)
            if ts.shape[0] != W:
                raise ValueError("sequence and structure motifs must have the same width")
        if want_sym and len(found) and int(found.sum()):
            # thin the candidates with the sequence table ON THE DEVICE (their symbols came with them) before
            # anything is gathered on the host; survivors replace the candidates of their chunk, in order
            wb = int(lib.rs_refine_packed_workspace_bytes(self.cap))
            rwork = torch.empty(wb, dtype=torch.uint8, device=self.device)
            kept = torch.empty_like(self.cand)
            for k, f in enumerate(found.tolist()):
                if f:
                    check(lib.rs_refine_candidates_packed(_ptr(self.cand[k]), _ptr(self.cand_sym[k]), int(f),
                                                          ts.ctypes.data, W, threshold, _ptr(kept[k]),
                                                          _ptr(self.cand_counters[k]), _ptr(rwork), wb, comp.cuda_stream))
                    self.launches += 2
            self.cand_counters_host.copy_(self.cand_counters, non_blocking=True)
            comp.synchronize()
            self.n_struct_candidates = int(found.sum())
            found = np.where(found > 0, self.cand_counters_host.numpy()[:len(self.starts), 0], 0)
            self.cand, kept = kept, self.cand
        parts = [self.cand[k, :int(f)].cpu().numpy() for k, f in enumerate(found.tolist()) if f]
        cand = np.concatenate(parts) if parts else np.zeros(0, np.int64)
        self.d2h_bytes += cand.size * 8
        self.n_candidates = int(cand.size)
        if ts is not None and ts.shape[0] != W:
            raise ValueError("sequence and structure motifs must have the same width")
        return self._resolve(cand, codes if exact_codes is None else exact_codes, filt_src, exact_rows, ts, tq,
                             threshold)

    RESOLVE_BATCH = 1 << 20

    def _resolve(self, cand, codes, filt_src, exact_rows, ts, tq, threshold):
        W = self.W
        dtype = _lib.RS_F32 if exact_rows.dtype == np.float32 else _lib.RS_F64
        ftype = torch.float32 if dtype == _lib.RS_F32 else torch.float64
        if codes is None and self.form == "q8":     # the symbols ride in byte 7 of the quantised rows
            q = filt_src.numpy() if isinstance(filt_src, torch.Tensor) else np.asarray(filt_src)
            code_ptr, code_stride = q.ctypes.data + 7, 8
        elif codes is None and self.form == "q4":   # ... or in the top nibble of the 4-byte rows
            q = filt_src.numpy() if isinstance(filt_src, torch.Tensor) else np.asarray(filt_src)
            code_ptr, code_stride = q.ctypes.data, -4
        elif codes is None:
            code_ptr, code_stride = 0, 1
        else:
            c = codes.numpy() if isinstance(codes, torch.Tensor) else np.ascontiguousarray(codes)
            code_ptr, code_stride = c.ctypes.data, 1
        pos_l, seq_l, str_l = [], [], []
        comp = torch.cuda.current_stream(self.device)
        for a in range(0, len(cand), self.RESOLVE_BATCH):
            part = np.ascontiguousarray(cand[a:a + self.RESOLVE_BATCH])
            k = len(part)
            h_rows = torch.empty((k, W, len(CHANNELS)), dtype=ftype, pin_memory=True)
            h_codes = torch.empty((k, W), dtype=torch.uint8, pin_memory=True)
            check(lib.rs_host_gather_windows(exact_rows.ctypes.data, dtype, exact_rows.shape[0], code_ptr, code_stride,
                                             part.ctypes.data, k, W, h_rows.numpy().ctypes.data,
                                             h_codes.numpy().ctypes.data, HOST_THREADS))
            d_rows = h_rows.to(self.device, non_blocking=True)
            d_codes = h_codes.to(self.device, non_blocking=True)
            d_pos = torch.from_numpy(part).to(self.device, non_blocking=True)
            self.h2d_bytes += h_rows.numel() * h_rows.element_size() + h_codes.numel() + k * 8
            out_pos = torch.empty(k, dtype=torch.int64, device=self.device)
            out_seq = torch.empty(k, dtype=torch.float32, device=self.device) if ts is not None else None
            out_str = torch.empty(k, dtype=torch.float64, device=self.device)
            counters = torch.zeros(2, dtype=torch.int64, device=self.device)
            wb = int(lib.rs_resolve_workspace_bytes(k))
            work = torch.empty(wb, dtype=torch.uint8, device=self.device)
            check(lib.rs_resolve_candidates(_ptr(d_pos), k, _ptr(d_rows), dtype, _ptr(d_codes),
                                            0 if ts is None else ts.ctypes.data, tq.ctypes.data, W, threshold,
                                            _ptr(out_pos), _ptr(out_seq), _ptr(out_str), _ptr(counters), _ptr(work),
                                            wb, comp.cuda_stream))
            self.launches += 2
            hits = int(counters[0].item())
            pos_l.append(out_pos[:hits].cpu().numpy())
            str_l.append(out_str[:hits].cpu().numpy())
            if ts is not None:
                seq_l.append(out_seq[:hits].cpu().numpy())
            self.d2h_bytes += 16 + hits * (20 if ts is not None else 16)
        pos = np.concatenate(pos_l) if pos_l else np.zeros(0, np.int64)
        st = np.concatenate(str_l) if str_l else np.zeros(0, np.float64)
        sq = (np.concatenate(seq_l) if seq_l else np.zeros(0, np.float32)) if ts is not None else None
        return pos, sq, st


def scan_profile_host(codes, hp, seq, struct_table, threshold, all_reduce=None, chunk_rows=1 << 23, form=None,
                      return_scanner=False):
    """Averaged-profile scan of host-resident rows (a HostProfile) through the filter + gather + resolve
    path; same results as scan_fused(SymbolStream(codes), ProfileStream(hp.rows), ...).  `codes`: uint8[n]
    host symbols (None: no separators, structure-only).  Falls back to the exact fp64 kernel when the fp32
    filter does not apply (-m -inf, W > 24, +inf / NaN tables, negative or non-finite rows)."""
    tq = _table(struct_table, 7)
    W = tq.shape[0]
    n = hp.n
    threshold = float(threshold)
    if codes is None:
        codes = np.zeros(n, np.uint8)
    if not filter_applies(tq, threshold, hp.absrow_max()) or n < W:
        stream = SymbolStream(codes, kind="rna")
        profile = ProfileStream(hp.rows)
        if callable(seq):
            counts = histogram(stream)
            if all_reduce is not None:
                all_reduce(counts)
            seq = seq(counts.cpu().numpy())
        out = scan_fused(stream, profile, seq, tq, threshold)
        return out + (None,) if return_scanner else out
    if form is None:
        form = pick_filter_form(hp, tq, threshold)
    sc = HostProfileScanner(n, W, form, chunk_rows=min(int(chunk_rows), max(n, 256)))
    src = {"q8": hp.q8, "q4": hp.q4}.get(form, hp.rows)
    if hp.page_locked is not None and form in ("q8", "q4") and src is hp.page_locked[1][form]:
        locked = hp.page_locked[0](form)            # the pack's own section, untouched: maybe held in pinned memory
        if locked is not None:
            src = locked
    out = sc.run(codes, src, hp.rows, tq, seq, threshold, hp.absrow_max(),
                 q8_scale=hp.q8_scale if form in ("q8", "q4") else 1.0, all_reduce=all_reduce)
    return out + (sc,) if return_scanner else out
