"""The reference's scan API and CLI (rnascan/rnascan.py) on the B200 kernels.

Same function names, arguments, stderr messages and hits.tab output as the reference; the
per-window Python loops (Biopython ``search`` -> ``_pwm.calculate``, ``_py_calculate``, the
pandas double loop of ``scan_averaged_structure``) and the ``multiprocessing.Pool`` fan-out
are replaced by one kernel launch over ALL records of a file: records are packed into a
single symbol stream (include/rnascan_b200.h), scanned in one pass, and the ordered hit list
is mapped back to (record, start) on the host.  Each function cites the reference lines it
mirrors.  There is no CPU fallback: without the CUDA library / a device the scans raise.

Result frames reproduce the reference's dtypes (float32 sequence scores rounded in float32,
Python-float structure scores, object columns when a record has no hit, ...) because the
TSV text written by ``to_csv`` depends on them (SURVEY.md H8, a17).
"""
from __future__ import print_function

import argparse
import ast
import glob
import os
import os.path
import re
import sys
import time
import warnings
from collections import defaultdict

import numpy as np


class _LazyPandas(object):
    """pandas on first use.  A FASTA scan needs it neither for its PFMs (_read_pfm_counts) nor for hits.tab (the
    native writer): importing it costs 1-3 s of a run whose device work is milliseconds.  Profile directories,
    -t, empty results and anything unusual still go through pandas, exactly as before."""

    def __getattr__(self, name):
        import pandas
        globals()["pd"] = pandas
        return getattr(pandas, name)


pd = _LazyPandas()

from . import motifs
from . import seq as _seq
from .BioAddons.Alphabet import ContextualSecondaryStructure
from .BioAddons.motifs import matrix
from .seq import IUPAC, RNAAlphabet, Seq, SeqRecord  # noqa: F401  (re-exported names)
from .version import __version__

HIT_COLUMNS = ["Motif_ID", "Start", "End", "Sequence", "LogOdds"]


class _Stats(object):
    """--stats: where a run's time goes and what the device achieved (the reference has only the tic/toc of
    rnascan.py:569-575).  Phases are wall-clock seconds on the host; `kernel_ms` are the durations of the main
    scan kernels measured with CUDA events inside the library (rs_prof_begin / rs_prof_end)."""

    def __init__(self):
        self.on = False
        self.phases = defaultdict(float)
        self.counts = defaultdict(int)
        self.notes = {}

    def reset(self, on):
        self.__init__()
        self.on = bool(on)

    class _Timer(object):
        def __init__(self, stats, name):
            self.stats, self.name = stats, name

        def __enter__(self):
            self.t0 = time.perf_counter()

        def __exit__(self, *exc):
            self.stats.phases[self.name] += time.perf_counter() - self.t0

    def phase(self, name):
        return self._Timer(self, name)

    def add(self, name, value):
        self.counts[name] += int(value)


STATS = _Stats()
MAX_BATCH_SYMBOLS = 1 << 30          # symbols per device batch when scanning a FASTA file


def getoptions(argv=None):
    """argparse definition of rnascan.py:44-105 (same flags, defaults and checks)."""
    desc = "Scan sequence for motif binding sites. Results sent to STDOUT."
    parser = argparse.ArgumentParser(description=desc)
    parser.add_argument("fastafiles", metavar="FASTA", nargs="*",
                        help="Input sequence and structure FASTA files")
    pfm_grp = parser.add_argument_group("PFM options")
    pfm_grp.add_argument("-p", "--pfm_seq", dest="pfm_seq", type=str, help="Sequence PFM")
    pfm_grp.add_argument("-q", "--pfm_struct", dest="pfm_struct", type=str, help="Structure PFM")
    parser.add_argument("-C", "--pseudocount", type=float, dest="pseudocount", default=0,
                        help="Pseudocount for normalizing PFM. [%(default)s]")
    parser.add_argument("-m", "--minscore", type=float, dest="minscore", default=6,
                        help="Minimum score for motif hits. [%(default)s]")
    parser.add_argument("-t", "--testseq", dest="testseq", default=None,
                        help=("Supply a test sequence to scan. FASTA files will be ignored. Can "
                              "supply sequence and structure as single string separated by  comma."))
    parser.add_argument("-c", "--cores", type=int, default=8, dest="cores",
                        help="Accepted for compatibility; the scan runs on the GPU and the result "
                             "does not depend on it [%(default)s]")
    bg_grp = parser.add_argument_group("Background frequency options")
    bg_grp.add_argument("-u", "--uniformbg", action="store_true", default=False,
                        dest="uniform_background",
                        help=("Use uniform background for calculating log-odds [%(default)s]. "
                              "Default is to compute background from input sequences. This option "
                              "is mutually exclusive with -B."))
    bg_grp.add_argument("-g", "--bgonly", action="store_true", default=False, dest="bgonly",
                        help=("Compute background probabilities from input sequences (STDOUT) and "
                              "exit. Useful for getting background probabilities from a superset of "
                              "sequences. Then, these values can be subsequently supplied using -b. "
                              "[%(default)s]"))
    bg_grp.add_argument("-b", "--bg_seq", default=None, dest="bg_seq",
                        help="Load file of pre-computed background probabilities for nucleotide sequences")
    bg_grp.add_argument("-B", "--bg_struct", default=None, dest="bg_struct",
                        help="Load file of pre-computed background probabilities for structure contexts")
    parser.add_argument("--pack", action="store_true", default=False, dest="pack",
                        help="(rnascan_b200) After parsing a directory of averaged structure profiles, leave "
                             "a binary pack (rnascan_b200.pack) in it; later scans of the unchanged directory "
                             "map the pack instead of parsing the text [%(default)s]")
    parser.add_argument("--reference-compat", action="store_true", default=False, dest="reference_compat",
                        help="(rnascan_b200) Averaged structure profiles: pair profile and PSSM columns by "
                             "position (B,E,H,L,M,R,T against E,H,T,B,L,R,M) as the unmodified reference does on "
                             "Python >= 3.6, instead of by label [%(default)s]")
    parser.add_argument("--stats", dest="stats", default=None, metavar="FILE",
                        help="(rnascan_b200) Write one JSON line with the run's phase times, scored positions, "
                             "Gpos/s and the device kernels' achieved GB/s to FILE ('-' = STDERR)")
    parser.add_argument("-v", "--version", action="version", version="%(prog)s " + __version__)
    parser.add_argument("-x", "--debug", action="store_true", default=False, dest="debug",
                        help="Reference debug mode (no process pool there; here it only changes the "
                             "Sequence_ID of averaged-structure hits as in the reference) [%(default)s]")
    args = parser.parse_args(argv)
    if not (args.pfm_seq or args.pfm_struct):
        parser.error("Must specify PFMs with -p and/or -q")
    if args.uniform_background and (args.bg_seq or args.bg_struct):
        parser.error("You cannot set uniform and custom background options at the same time\n")
    return args


_QUIET = 0


def eprint(*args, **kwargs):
    if _rank() == 0 and not _QUIET:       # under torchrun only rank 0 talks
        print(*args, file=sys.stderr, **kwargs)


def _rank():
    from . import shard
    return shard.world()[0]


def _world_size():
    from . import shard
    return shard.world()[1]


###############################################################################
# Sequence functions
###############################################################################
def _guess_seq_type(args):
    """RNA, SS or RNASS from the number of inputs and PFMs (rnascan.py:114-137)."""
    if len(args.fastafiles) == 2:
        if not (args.pfm_seq or args.pfm_struct):
            eprint("Missing PFMs")
            sys.exit(1)
        return "RNASS"
    if args.pfm_seq and args.pfm_struct and not args.testseq:
        eprint("Can't specify two PFMs with one input file")
        sys.exit(1)
    if args.pfm_seq and args.pfm_struct and args.testseq:
        return "RNASS"
    if args.pfm_seq:
        return "RNA"
    if args.pfm_struct:
        return "SS"
    eprint("Must specify PFMs with -p and/or -q")
    sys.exit(1)


def batch_iterator(iterator, batch_size):
    """Lists of up to `batch_size` entries of `iterator` (rnascan.py:140-167); a None entry
    ends the iteration like exhaustion does."""
    iterator = iter(iterator)
    done = False
    while not done:
        batch = []
        while len(batch) < batch_size:
            entry = next(iterator, None)
            if entry is None:
                done = True
                break
            batch.append(entry)
        if batch:
            yield batch


def parse_sequences(fasta_file):
    """SeqRecord iterator over one FASTA path or a list of paths; .gz/.bz2 transparently
    (rnascan.py:170-174)."""
    return _seq.parse_fasta(fasta_file)


def preprocess_seq(seqrec, alphabet):
    """RNA target alphabet + non-RNA input -> transcribe (T->U, t->u) and upper-case;
    anything else passes through (rnascan.py:177-204).  Returns a Seq."""
    if not _seq.is_seqrecord(seqrec):
        raise TypeError("SeqRecord object must be supplied")
    if _seq.is_ambiguous_rna_alphabet(alphabet) and not _seq.is_rna_alphabet(seqrec.seq.alphabet):
        out = seqrec.seq.transcribe()
        out.alphabet = alphabet
        return out.upper()
    return seqrec.seq


###############################################################################
# PFM functions
###############################################################################
def load_motif(pfm_file, *args):
    """{motif_id: PSSM} for one PFM file; motif_id = file name without extension
    (rnascan.py:210-235, messages included)."""
    motifs_set = {}
    eprint("Loading PFM %s" % pfm_file, end="")
    tic = time.time()
    try:
        if isinstance(pfm_file, _PfmBlock):
            motif_id = pfm_file.motif_id
        else:
            motif_id = os.path.splitext(os.path.basename(pfm_file))[0]
        motifs_set[motif_id] = pfm2pssm(pfm_file, *args)
    except ValueError:
        eprint("\nFailed to load motif %s" % pfm_file)
    except KeyError:
        eprint("\nFailed to load motif %s" % pfm_file)
        eprint("Check that you are using the correct --type")
        raise
    except Exception:
        eprint("Unexpected error: %s" % sys.exc_info()[0])
        raise
    eprint("\b.", end="")
    sys.stderr.flush()
    eprint("done in %0.2f seconds!" % (float(time.time() - tic)))
    eprint("Found %d motifs" % len(motifs_set))
    if len(motifs_set) == 0:
        raise ValueError("No motifs found.")
    return motifs_set


def pfm2pssm(pfm_file, pseudocount, alphabet, background=None):
    """PFM file -> normalize(pseudocount) -> log_odds(background) -> PSSM
    (rnascan.py:238-252).  The first column is dropped; header letters may come in any order."""
    counts = _pfm_counts(pfm_file)
    values = motifs.Motif(alphabet=alphabet, counts=counts).pssm(pseudocount, background)
    return matrix.ExtendedPositionSpecificScoringMatrix(alphabet, values)


def _pfm_counts(pfm_file):
    """{letter: column values} of a PFM table, first column dropped: what
    ``pd.read_csv(f, sep="\\t").drop(columns=first).to_dict(orient="list")`` gives (rnascan.py:242-245)."""
    counts = _read_pfm_counts(pfm_file)
    if counts is None:
        table = pd.read_csv(pfm_file.open() if isinstance(pfm_file, _PfmBlock) else pfm_file, sep="\t")
        counts = table.drop(columns=table.columns[0]).to_dict(orient="list")
    return counts


_PLAIN_INT = re.compile(r"^[+-]?[0-9]{1,15}$")


def _read_pfm_counts(pfm_file):
    """The same dictionary without pandas, for tables in the plain format -- a header of unique names, every row
    with as many tab-separated fields as the header, every value a plain decimal number -- or None (then pandas
    reads the file: quotes, blanks, NaN, ragged rows, index inference, ... are its business).  Numbers are
    converted as pandas converts them: its default converter is not correctly rounded, rs_host_parse_doubles
    restates it bit for bit (tests/test_host_cpu.py); an all-integer column stays int64 as in pandas."""
    from . import _lib
    try:
        if isinstance(pfm_file, _PfmBlock):
            text = pfm_file.text
        else:
            with open(pfm_file, "r", newline="") as handle:
                text = handle.read()
    except (OSError, UnicodeDecodeError):
        return None
    if not text.isascii() or '"' in text or "\r" in text.replace("\r\n", "\n") or "\x00" in text:
        return None
    lines = [ln for ln in text.replace("\r\n", "\n").split("\n") if ln != ""]
    if len(lines) < 2:
        return None
    names = lines[0].split("\t")
    if len(names) < 2 or len(set(names)) != len(names) or any(n == "" or n != n.strip() for n in names):
        return None
    if any(_PLAIN_INT.match(n) or n.startswith("Unnamed") for n in names):
        return None
    rows = [ln.split("\t") for ln in lines[1:]]
    if any(len(r) != len(names) for r in rows):
        return None
    counts = {}
    for c in range(1, len(names)):
        tokens = [r[c] for r in rows]
        if any(t == "" or t != t.strip() for t in tokens):
            return None
        if all(_PLAIN_INT.match(t) for t in tokens):
            counts[names[c]] = [int(t) for t in tokens]          # an int64 column
            continue
        blob = "\n".join(tokens).encode("ascii")
        out = np.zeros(len(tokens), np.float64)
        ok = np.zeros(len(tokens), np.uint8)
        n_out = np.zeros(1, np.int64)
        if _lib.lib.rs_host_parse_doubles(blob, len(blob), out.ctypes.data, len(out), n_out.ctypes.data,
                                          ok.ctypes.data) != 0 or int(n_out[0]) != len(tokens):
            return None
        values = out.tolist()
        for k, t in enumerate(tokens):
            if not ok[k]:
                if not _PLAIN_INT.match(t):
                    return None                                   # not a number the converter takes: pandas decides
                values[k] = float(int(t))                         # an integer token in a float column (exact)
        counts[names[c]] = values
    return counts


class _PfmBlock(object):
    """One motif of a multi-PFM file (pfmutil.write_multi_pfm layout, pfmutil.py:89-133 of the reference),
    standing in for the single-PFM file the reference would be run with: same table text, so the same parse."""

    def __init__(self, motif_id, text, source):
        self.motif_id, self.text, self.source = motif_id, text, source

    def open(self):
        import io
        return io.StringIO(self.text)

    def __str__(self):
        return "%s#%s" % (self.source, self.motif_id)


def pfm_blocks(path):
    """The motifs of a multi-PFM file as _PfmBlock objects, or None when `path` is an ordinary PFM file
    (first line does not start with '#').  Layout per block: ``#<id>``, ``#PO<TAB>letters``, one row per
    position, blank line."""
    if not isinstance(path, str) or not os.path.isfile(path):
        return None
    with open(path) as handle:
        lines = handle.read().splitlines()
    if not lines or not lines[0].startswith("#"):
        return None
    blocks, k = [], 0
    while k < len(lines):
        if not lines[k].startswith("#"):
            k += 1
            continue
        if k + 1 >= len(lines) or not lines[k + 1].startswith("#"):
            raise ValueError("%s: block '%s' lacks its '#PO<TAB>letters' line" % (path, lines[k]))
        motif_id, header = lines[k][1:].rstrip(), lines[k + 1][1:].rstrip()
        k += 2
        rows = []
        while k < len(lines) and not lines[k].startswith("#"):
            if lines[k].strip():
                rows.append(lines[k].rstrip())
            k += 1
        blocks.append(_PfmBlock(motif_id, "\n".join([header] + rows) + "\n", path))
    return blocks


###############################################################################
# Packed record batches (host side of the device layout)
###############################################################################
class _Batch(object):
    """Records (or, when the input is sharded over ranks, pieces of records) of one input
    packed into a symbol stream resident in HBM.

    ids/descriptions describe ALL records of the batch's input range; `record` maps each
    packed text to its record, `piece_start` is its offset inside that record and `own`
    the number of leading window starts / symbols this rank owns (shard.plan_shards).
    `counts`: the owned symbol counts (compute_background), taken once per batch."""
    counts = None

    def __init__(self, ids, descriptions, texts, kind, record=None, piece_start=None, own=None,
                 full_texts=None):
        from . import device
        self.ids, self.descriptions, self.texts, self.kind = ids, descriptions, texts, kind
        self.full_texts = texts if full_texts is None else full_texts     # one per record
        n = len(texts)
        self.record = np.arange(n, dtype=np.int64) if record is None else np.asarray(record, np.int64)
        self.piece_start = np.zeros(n, np.int64) if piece_start is None else np.asarray(piece_start, np.int64)
        self.own = None if own is None else np.asarray(own, np.int64)
        self.stream = device.SymbolStream.from_texts(texts, kind)

    @classmethod
    def from_pieces(cls, ids, descriptions, text, codes, offsets, lengths, kind, pieces):
        """This rank's pieces (shard.plan_shards: (record, start, stop, own_stop)) cut out of the natively parsed
        arrays of the whole input -- slices of `codes` / `text`, no Python strings."""
        from . import device, _lib
        n = len(pieces)
        rec = np.array([p[0] for p in pieces], np.int64)
        a = np.array([p[1] for p in pieces], np.int64)
        b = np.array([p[2] for p in pieces], np.int64)
        o = np.array([p[3] for p in pieces], np.int64)
        ln = b - a
        poff = np.zeros(n, np.int64)
        if n > 1:
            np.cumsum(ln[:-1] + 1, out=poff[1:])
        total = int(ln.sum() + n)
        pcodes = np.full(total, _lib.RS_SEP, np.uint8)
        ptext = np.full(total, ord("\n"), np.uint8)
        for k in range(n):
            src = int(offsets[rec[k]] + a[k])
            pcodes[poff[k]:poff[k] + ln[k]] = codes[src:src + ln[k]]
            ptext[poff[k]:poff[k] + ln[k]] = text[src:src + ln[k]]
        self = cls.__new__(cls)
        self.ids, self.descriptions, self.kind = ids, descriptions, kind
        self.texts = _LazyTexts(ptext, poff, ln)
        self.full_texts = _LazyTexts(text, np.asarray(offsets, np.int64), np.asarray(lengths, np.int64))
        self.record, self.piece_start = rec, a
        self.own = np.where(o >= b, b, o) - a
        self.stream = device.SymbolStream(pcodes, poff, ln, kind=kind)
        return self

    def overlap_counts(self):
        """Counts (int64[8], int64[A] for an alphabet kind: the bins of device.histogram) of the symbols this rank
        holds but does not own (the overlap tails of split records); the device histogram minus these is the
        owned count."""
        bins = 8 if self.kind in ("rna", "struct") else len(self.kind.letters)
        counts = np.zeros(bins, np.int64)
        if self.own is None:
            return counts
        host = self.stream.host_codes()
        for k in np.nonzero(self.own < self.stream.lengths)[0]:
            a = self.stream.offsets[k] + self.own[k]
            tail = host[a:self.stream.offsets[k] + self.stream.lengths[k]]
            counts += np.bincount(tail[tail < bins], minlength=bins)[:bins]
        return counts

    def locate(self, pos):
        """stream positions -> (keep mask, record index, 0-based start in the record)."""
        if len(pos) == 0:
            z = np.zeros(0, np.int64)
            return np.zeros(0, bool), z, z
        piece, start = self.stream.locate(pos)
        keep = np.ones(len(pos), bool) if self.own is None else start < self.own[piece]
        return keep, self.record[piece], start + self.piece_start[piece]

    def __len__(self):
        return len(self.texts)


class _LazyTexts(object):
    """List-like view of the records of a packed text buffer; strings are made on demand."""

    def __init__(self, raw, offsets, lengths):
        self.raw, self.offsets, self.lengths = raw, offsets, lengths

    def __len__(self):
        return len(self.offsets)

    def __getitem__(self, k):
        if isinstance(k, slice):
            return [self[i] for i in range(*k.indices(len(self)))]
        o, n = int(self.offsets[k]), int(self.lengths[k])
        return self.raw[o:o + n].tobytes().decode("ascii")

    def __iter__(self):
        return (self[k] for k in range(len(self)))


def _record_text(batches):
    """(uint8 text, offsets) of the whole records of `batches` (under torchrun: of the whole input, which every
    rank holds) laid out one after the other with one separator each: byte offsets[r] + i is letter i of
    record r.  Hit fragments are cut from it without a Python loop."""
    if len(batches) == 1 and isinstance(batches[0].full_texts, _LazyTexts):
        return batches[0].full_texts.raw, batches[0].full_texts.offsets
    texts = [t for b in batches for t in b.full_texts]
    offsets = np.zeros(len(texts), np.int64)
    if len(texts) > 1:
        np.cumsum([len(t) + 1 for t in texts[:-1]], out=offsets[1:])
    joined = ("\n".join(texts) + "\n") if texts else ""
    return np.frombuffer(joined.encode("latin-1", "replace"), dtype=np.uint8), offsets


def _read_fasta_bytes(fasta_file):
    """The bytes fileinput would feed the parser (rnascan.py:173: .gz/.bz2 transparently, several
    files chained)."""
    import bz2
    import gzip
    paths = [fasta_file] if isinstance(fasta_file, str) else list(fasta_file)
    chunks = []
    for path in paths:
        ext = os.path.splitext(path)[1]
        opener = gzip.open if ext == ".gz" else (bz2.open if ext == ".bz2" else open)
        with opener(path, "rb") as fh:
            chunks.append(fh.read())
    return b"\n".join(chunks)


def _native_batch(fasta_file, alphabet):
    """Parse + pre-process + encode a FASTA input in one native pass (rs_host_fasta_*); None when
    the input is not plain ASCII or too large for one batch (the Python parser handles those)."""
    from . import device
    native = _native_parse(fasta_file, alphabet, MAX_BATCH_SYMBOLS)
    if native is None:
        return None
    text, codes, off, ln, ids, descs, kind = native
    n_rec = len(ids)
    batch = _Batch.__new__(_Batch)
    batch.ids, batch.descriptions, batch.kind = ids, descs, kind
    batch.texts = batch.full_texts = _LazyTexts(text, off, ln)
    batch.record = np.arange(n_rec, dtype=np.int64)
    batch.piece_start = np.zeros(n_rec, np.int64)
    batch.own = None
    batch.stream = device.SymbolStream(codes, off if n_rec else None, ln if n_rec else None, kind=kind) \
        if n_rec else device.SymbolStream(np.zeros(0, np.uint8), np.zeros(0, np.int64), np.zeros(0, np.int64), kind=kind)
    return batch


def _native_parse(fasta_file, alphabet, max_symbols=None):
    """(text uint8[], codes uint8[], offsets, lengths, ids, descriptions, kind) of a FASTA input from the native
    two-pass parser, records laid out one after the other with one separator each; None when it does not
    apply (non-ASCII input, DNA target alphabet, an alphabet other than GAUC and BEHLMRT, unreadable file, more
    than `max_symbols`)."""
    from . import _lib
    rna_target = _seq.is_ambiguous_rna_alphabet(alphabet)
    kind = _kind_of(alphabet)
    if kind == "rna" and not rna_target:
        return None                                   # DNA target alphabets: no transcription (not a CLI path)
    if kind not in ("rna", "struct"):
        return None                                   # other alphabets: the Python parser (not a CLI path)
    try:
        data = _read_fasta_bytes(fasta_file)
    except (OSError, EOFError):
        return None
    if not data.isascii():
        return None
    buf = np.frombuffer(data, dtype=np.uint8)
    sizes = np.zeros(3, np.int64)
    _lib.check(_lib.lib.rs_host_fasta_index(buf.ctypes.data if len(buf) else 0, len(buf), sizes[0:].ctypes.data,
                                            sizes[1:].ctypes.data, sizes[2:].ctypes.data))
    n_rec, n_sym, n_title = (int(v) for v in sizes)
    if max_symbols is not None and n_sym + n_rec > max_symbols:
        return None
    text = np.empty(max(n_sym + n_rec, 1), np.uint8)
    codes = np.empty(max(n_sym + n_rec, 1), np.uint8)
    off = np.zeros(max(n_rec, 1), np.int64)
    ln = np.zeros(max(n_rec, 1), np.int64)
    titles = np.empty(max(n_title, 1), np.uint8)
    toff = np.zeros(n_rec + 1, np.int64)
    _lib.check(_lib.lib.rs_host_fasta_fill(buf.ctypes.data if len(buf) else 0, len(buf), 0 if kind == "rna" else 1,
                                           text.ctypes.data, codes.ctypes.data, off.ctypes.data, ln.ctypes.data,
                                           titles.ctypes.data, toff.ctypes.data))
    text, codes, off, ln = text[:n_sym + n_rec], codes[:n_sym + n_rec], off[:n_rec], ln[:n_rec]
    blob = titles[:n_title].tobytes().decode("ascii")
    descs = [blob[a:b] for a, b in zip(toff[:-1].tolist(), toff[1:].tolist())]
    ids = [(d.split(None, 1) or [""])[0] for d in descs]
    return text, codes, off, ln, ids, descs, kind


NATIVE_INGEST = True                 # tests switch it off to exercise the Python parser


def _kind_of(alphabet):
    """Stream kind of a target alphabet: "rna" (nucleotides), "struct" (BEHLMRT) or a device.AlphaKind for any
    other alphabet (NotImplementedError, naming the rule, for one the device layouts cannot hold)."""
    from . import device
    if _seq.is_nucleotide_alphabet(alphabet):
        return "rna"
    if sorted(alphabet.letters or "") == sorted(device.CHANNELS):
        return "struct"
    return device.AlphaKind(alphabet.letters)


def _sharded_batch(fasta_file, alphabet, rank, size):
    """This rank's share of the input: contiguous pieces balanced by total length, split
    records overlapping by RS_MAX_W - 1 symbols (enough for any motif width).  The file is parsed and encoded
    natively on host threads (rs_host_fasta_*: no Python object per record); only this rank's pieces are
    packed and uploaded.  Inputs outside the native parser's scope go through the Python parser."""
    from . import shard, _lib
    if NATIVE_INGEST:
        native = _native_parse(fasta_file, alphabet)
        if native is not None:
            text, codes, off, ln, ids, descs, kind = native
            plan = shard.plan_shards(ln.tolist(), size, _lib.RS_MAX_W)
            mine = plan[rank]
            return _Batch.from_pieces(ids, descs, text, codes, off, ln, kind, mine)
    ids, descs, texts = [], [], []
    for rec in parse_sequences(fasta_file):
        ids.append(rec.id)
        descs.append(rec.description)
        texts.append(str(preprocess_seq(rec, alphabet)))
    plan = shard.plan_shards([len(t) for t in texts], size, _lib.RS_MAX_W)
    mine = plan[rank]
    piece_texts = [texts[r][a:b] for (r, a, b, o) in mine]
    own = [(b if o >= b else o) - a for (r, a, b, o) in mine]
    return _Batch(ids, descs, piece_texts, _kind_of(alphabet), record=[p[0] for p in mine],
                  piece_start=[p[1] for p in mine], own=own, full_texts=texts)


def _record_batches(fasta_file, alphabet, max_symbols=None):
    """Parse + preprocess a FASTA input and yield _Batch objects of bounded size."""
    size = _world_size()
    if size > 1:
        yield _sharded_batch(fasta_file, alphabet, _rank(), size)
        return
    if NATIVE_INGEST and max_symbols is None:
        batch = _native_batch(fasta_file, alphabet)
        if batch is not None:
            if len(batch.ids):
                yield batch
            return
    max_symbols = max_symbols or MAX_BATCH_SYMBOLS
    ids, descs, texts, size = [], [], [], 0
    for rec in parse_sequences(fasta_file):
        text = str(preprocess_seq(rec, alphabet))
        if texts and size + len(text) + 1 > max_symbols:
            yield _Batch(ids, descs, texts, _kind_of(alphabet))
            ids, descs, texts, size = [], [], [], 0
        ids.append(rec.id)
        descs.append(rec.description)
        texts.append(text)
        size += len(text) + 1
    if texts:
        yield _Batch(ids, descs, texts, _kind_of(alphabet))


def _columns(kind):
    """Device column order of a stream kind: the order of tables and histogram bins."""
    from . import device
    if kind == "rna":
        return device.RNA_COLUMNS
    return device.CHANNELS if kind == "struct" else kind.letters


def _table_for(pm, kind):
    return pm.table(_columns(kind))


def _first_motif(pssm):
    return list(pssm.items())[0]


def _fragments(raw, pos, width):
    """Python str of the `width` letters starting at each stream position."""
    if len(pos) == 0:
        return []
    windows = np.lib.stride_tricks.sliding_window_view(raw, width)[pos]
    return np.ascontiguousarray(windows).view("S%d" % width).ravel().astype("U%d" % width).tolist()


def _round3_f32(scores):
    """round(numpy.float32, 3) elementwise: float32 arithmetic, as rnascan.py:273 gets it."""
    return np.round(np.asarray(scores, dtype=np.float32), 3)


def _round3_f64(scores):
    """round(float, 3) elementwise with Python's exact decimal rounding.  int32 input = the same values already
    rounded on the device, in thousandths (device.scan_struct_every_position)."""
    scores = np.asarray(scores)
    if scores.dtype == np.int32:
        from . import _lib
        return [-0.0 if k == _lib.RS_MILLI_NEG0 else k / 1000.0 for k in scores.tolist()]
    return [round(v, 3) for v in scores.astype(np.float64).tolist()]


###############################################################################
# Motif scan functions
###############################################################################
def scan(pssm, seq, alphabet, minscore):
    """[motif_id, Start (1-based), End, fragment, round(score, 3)] for every window of `seq`
    whose score is > minscore (rnascan.py:258-275)."""
    motif_id, pm = _first_motif(pssm)
    width = len(pm.consensus)
    results = []
    for position, score in pm.search(seq, threshold=minscore, both=False):
        end_position = position + width
        results.append([motif_id, position + 1, end_position, str(seq[position:end_position]),
                        round(score, 3)])
    return results


def scan_all(seqrecord, pssm, alphabet, *args):
    """DataFrame of the hits of one record (rnascan.py:278-286)."""
    sequence = preprocess_seq(seqrecord, alphabet)
    final = pd.DataFrame(scan(pssm, sequence, alphabet, *args), columns=HIT_COLUMNS)
    return final.sort_values(["Start", "Motif_ID"])


def _scan_all(a_b):
    return scan_all(*a_b)


def _read_profile(struct_file):
    """(L, 7) float64 rows in B,E,H,L,M,R,T order from a ``structure.<id>.txt`` profile
    (pfmutil.format_pfm layout).  Channels are matched BY LABEL (SURVEY.md H6)."""
    from . import device
    table = pd.read_csv(struct_file, sep="\t")
    del table["PO"]
    return np.ascontiguousarray(table[list(device.CHANNELS)].to_numpy(dtype=np.float64))


def _read_profiles_packed(files, threads=None):
    """All profiles of `files` as ONE packed (sum L + len(files), 7) float64 array in B,E,H,L,M,R,T order
    (a zero separator row after each profile, the layout device.ProfileStream uploads) plus their lengths.
    Plain files are read and converted natively on host threads (rs_host_profiles_*: pandas' own number
    conversion restated, bit-identical rows); anything else goes through `_read_profile` (pandas)."""
    import ctypes
    from . import _lib
    n = len(files)
    lengths = np.zeros(n, np.int64)
    if n == 0:
        return np.zeros((0, 7), np.float64), lengths
    threads = int(threads or min(32, os.cpu_count() or 1))
    arr = (ctypes.c_char_p * n)(*[os.fsencode(f) for f in files])
    handle = ctypes.c_void_p()
    rows = np.zeros(n, np.int64)
    _lib.check(_lib.lib.rs_host_profiles_open(ctypes.cast(arr, ctypes.c_void_p), n, threads, ctypes.byref(handle),
                                              rows.ctypes.data))
    try:
        fallback = {k: _read_profile(files[k]) for k in np.nonzero(rows < 0)[0].tolist()}
        for k, prof in fallback.items():
            rows[k] = prof.shape[0]
        offsets = np.zeros(n, np.int64)
        if n > 1:
            np.cumsum(rows[:-1] + 1, out=offsets[1:])
        packed = np.zeros((int(rows.sum()) + n, 7), np.float64)
        status = np.zeros(n, np.int32)
        _lib.check(_lib.lib.rs_host_profiles_fill(handle, threads, packed.ctypes.data, offsets.ctypes.data,
                                                  status.ctypes.data))
    finally:
        _lib.lib.rs_host_profiles_close(handle)
    for k in range(n):
        if k in fallback:
            packed[offsets[k]:offsets[k] + rows[k]] = fallback[k]
        elif status[k] != 0:                  # a field pandas must judge: re-read this one file with pandas
            prof = _read_profile(files[k])
            if prof.shape[0] != rows[k]:
                raise ValueError("%s: pandas sees %d rows, the native reader %d" % (files[k], prof.shape[0], rows[k]))
            packed[offsets[k]:offsets[k] + rows[k]] = prof
    lengths[:] = rows
    return packed, lengths


def _averaged_frame(motif_id, starts, width, scores):
    """Frame built the way pd.DataFrame(list of Series) builds it in the reference
    (rnascan.py:311-315): object columns; no columns at all when there is no hit."""
    if len(starts) == 0:
        return pd.DataFrame([])
    starts = np.asarray(starts, dtype=np.int64)
    data = {
        "Motif_ID": np.array([motif_id] * len(starts), dtype=object),
        "Start": (starts + 1).astype(object),
        "End": (starts + width).astype(object),
        "Sequence": np.array(["."] * len(starts), dtype=object),
        "LogOdds": np.asarray(scores, dtype=np.float64).astype(object),
    }
    return pd.DataFrame(data, columns=HIT_COLUMNS)


def scan_averaged_structure(struct_file, pssm, minscore):
    """Hits of a structure PSSM on one averaged 7-channel profile (rnascan.py:293-315):
    score_i = sum_j nan_to_num(dot(profile[i+j], pssm[j])) in float64, unrounded, > minscore."""
    from . import device
    motif_id, pm = _first_motif(pssm)
    rows = _read_profile(struct_file)
    tq = _structure_table(pm)
    width = tq.shape[0]
    if rows.shape[0] < width:
        return pd.DataFrame([])
    # the float64 rows stay on the host: a float32 shadow is filtered on the device, the few windows near
    # the threshold are re-scored from the exact rows (device.scan_profile_host)
    pos, _, scores = device.scan_profile_host(None, device.HostProfile(rows), None, tq, minscore)
    return _averaged_frame(motif_id, pos, width, scores)


def _scan_averaged_structure(a_b):
    return scan_averaged_structure(*a_b)


REFERENCE_COMPAT = False             # --reference-compat: pair profile columns and PSSM columns by POSITION


def _structure_table(pm):
    """(W, 7) table in device channel order from a PSSM object or a plain {letter: values}.

    Channels are matched BY LABEL (profile column "H" meets the PSSM's "H" column).  The unmodified reference
    on Python >= 3.6 pairs them by position instead (rnascan.py:300-307: ``pd.DataFrame(pm)`` has its columns
    in ``alphabet.letters`` order E,H,T,B,L,R,M while the profile file has B,E,H,L,M,R,T -- SURVEY.md H6);
    REFERENCE_COMPAT reproduces that pairing, for diffing against upstream output (profile files in the
    pfmutil.format_pfm column order)."""
    from . import device
    if REFERENCE_COMPAT:
        letters = list(getattr(getattr(pm, "alphabet", None), "letters", None) or pm.keys())
        return np.array([list(pm[c]) for c in letters], dtype=np.float64).T.copy()
    return np.array([list(pm[c]) for c in device.CHANNELS], dtype=np.float64).T.copy()


def _add_sequence_id(df, seq_id, description):
    df["Sequence_ID"] = seq_id
    df["Description"] = description


def _add_match_id(df):
    df["Match_ID"] = list(range(1, df.shape[0] + 1))


def _assemble_fasta_frame(n_records, rec, ids, descriptions, motif_id, start0, width, fragments,
                          logodds):
    """The frame pd.concat() of the reference's per-record frames would give
    (rnascan.py:284-286,401-408): typed columns when every record has a hit, object columns
    (Python ints / Python floats widened from the column dtype) as soon as one record has
    none, because an empty per-record frame has object columns."""
    n = len(rec)
    rec = np.asarray(rec, dtype=np.int64)
    per_record = np.bincount(rec, minlength=n_records) if n_records else np.zeros(0, np.int64)
    any_empty = bool((per_record == 0).any())
    start = np.asarray(start0, dtype=np.int64) + 1
    end = np.asarray(start0, dtype=np.int64) + width
    ids_arr = np.array(ids, dtype=object)[rec] if n else np.array([], dtype=object)
    desc_arr = np.array(descriptions, dtype=object)[rec] if n else np.array([], dtype=object)
    first = np.concatenate([[0], np.cumsum(per_record)[:-1]]) if n_records else np.zeros(0, np.int64)
    index = np.arange(n, dtype=np.int64) - first[rec] if n else np.zeros(0, np.int64)
    if any_empty:
        start, end = start.astype(object), end.astype(object)
        logodds = np.asarray(logodds).astype(object) if not isinstance(logodds, list) \
            else np.array(logodds, dtype=object)
    elif isinstance(logodds, list):
        logodds = np.array(logodds, dtype=np.float64)
    frame = pd.DataFrame({
        "Sequence_ID": ids_arr, "Description": desc_arr,
        "Motif_ID": np.array([motif_id] * n, dtype=object),
        "Start": start, "End": end,
        "Sequence": np.array(fragments, dtype=object) if n else np.array([], dtype=object),
        "LogOdds": logodds,
    }, index=index)
    return frame


def _scan_batch(batch, table, kind, minscore):
    """(stream positions, scores) of one motif's hits in a packed batch."""
    from . import device
    if kind == "rna":
        return device.scan_seq(batch.stream, table, minscore)
    if kind != "struct":
        return device.scan_alpha(batch.stream, table, minscore)
    every = None
    if minscore == float("-inf"):                       # every position: the device rounds, 4 B per window come back
        every = device.scan_struct_every_position(batch.stream, table)
    return every if every is not None else device.scan_struct_onehot(batch.stream, table, minscore)


def _scan_batches(batches, scan, widths, dtypes):
    """The hits of `scan` over the device batches of an input, gathered (_gather): the columns (record index over
    all batches, 0-based start, column...), None on ranks other than 0 under torchrun.  A device batch is a
    _Batch or a lined-up (sequence, structure) pair of them, located by its structure batch; `scan(batch)`
    returns (stream positions, column...) of its hits, `dtypes` are the dtypes of those columns and `widths` the
    widths of the motifs it scores."""
    parts, n_records = [], 0
    for batch in batches:
        where = batch[1] if isinstance(batch, tuple) else batch
        with STATS.phase("scan_s"):
            pos, *columns = scan(batch)
        lengths = where.stream.lengths
        STATS.add("scored_positions", sum(int(np.maximum(lengths - w + 1, 0).sum()) for w in widths))
        keep, rec, start0 = where.locate(pos)
        parts.append((rec[keep] + n_records, start0[keep]) + tuple(c[keep] for c in columns))
        n_records += len(where.ids)
    empty = (np.zeros(0, np.int64), np.zeros(0, np.int64)) + tuple(np.zeros(0, dt) for dt in dtypes)
    return _gather(parts or [empty])


def _gather(parts):
    """The hit arrays of a scan -- one (rec, start0, scores, ...) tuple per device batch -- concatenated column
    by column.  Under torchrun every rank's columns are gathered on rank 0 and concatenated in rank order
    (= record order, shard.plan_shards); the other ranks get None."""
    from . import shard
    columns = [_concat(col) for col in zip(*parts)]
    if _world_size() == 1:
        return columns
    ranks = shard.gather_arrays(columns)
    return None if ranks is None else [_concat(col) for col in zip(*ranks)]


def _concat(arrays):
    """np.concatenate keeping the dtype of the scores: the device-rounded thousandths (int32) of the
    every-position structure scan turn into floats only next to the float scores of a batch or rank where that
    form did not apply."""
    if len(arrays) == 1:
        return arrays[0]
    if len({a.dtype for a in arrays}) > 1:
        arrays = [np.array(_round3_f64(a), np.float64) if a.dtype == np.int32 else a for a in arrays]
    return np.concatenate(arrays)


NATIVE_WRITER_MIN_ROWS = 1           # from this many rows on, a table with arrays is printed natively (no DataFrame)
NATIVE_CHUNK_ROWS = 4_000_000        # rows formatted per call (bounds the text buffer to ~0.5 GB)
_HEADER = ["Sequence_ID", "Description", "Motif_ID", "Start", "End", "Sequence", "LogOdds", "Match_ID"]
_COMBINED_HEADER = ["Sequence_ID", "Description.Seq", "Motif_ID.Seq", "Start", "End", "Sequence.Seq", "LogOdds.Seq",
                    "Description.Struct", "Motif_ID.Struct", "Sequence.Struct", "LogOdds.Struct",
                    "LogOdds.SeqStruct", "Match_ID"]


class _HitTable(object):
    """The rows of one hits.tab.  `frame()` builds the DataFrame the reference prints for them.  A table with
    arrays can also be printed without one (rs_host_format_hits*): row r is the hit at 0-based `start0[r]` of
    record `rec[r]` (`ids` / `descs` per record), its fragment is `width` letters of `text` from `text_pos[r]`
    (no text: "."), its score `scores[r]`, printed as score_kind `kind` says.  Combined rows (`motif_b` set)
    add the structure side: `text_b` (None: "."), `kind_b` / `scores_b` and per-record `sdescs` (None: empty).
    A result only pandas can print (-t, the merge fallback, some directory shapes) has the frame only."""

    def __init__(self, frame, rec=None, start0=None, ids=(), descs=(), motif=None, width=0, text=None,
                 text_pos=None, kind=0, scores=None, motif_b=None, text_b=None, kind_b=0, scores_b=None,
                 sdescs=None):
        self.frame, self.rec, self.start0, self.ids, self.descs = frame, rec, start0, ids, descs
        self.motif, self.width, self.text, self.text_pos = motif, width, text, text_pos
        self.kind, self.scores = kind, scores
        self.motif_b, self.text_b, self.kind_b, self.scores_b, self.sdescs = motif_b, text_b, kind_b, scores_b, sdescs

    def write(self, out):
        """hits.tab on `out`: natively when the table has arrays, at least max(1, NATIVE_WRITER_MIN_ROWS) rows and
        only values the native formatter covers; through pandas otherwise."""
        if self.rec is None or len(self.rec) < max(1, NATIVE_WRITER_MIN_ROWS) or not self._write_native(out):
            frame = self.frame()
            _add_match_id(frame)
            frame.to_csv(out, sep="\t", index=False)

    def _write_native(self, out):
        """False (nothing written) when the formatter declines the first chunk; a later chunk it declines raises."""
        blobs = _StringBlobs(self.ids, self.descs)
        sblobs = None if self.sdescs is None else _StringBlobs(self.ids, self.sdescs)
        scores = _writer_scores(self.kind, self.scores)
        scores_b = None if self.motif_b is None else _writer_scores(self.kind_b, self.scores_b)
        for a in range(0, len(self.rec), NATIVE_CHUNK_ROWS):
            b = min(len(self.rec), a + NATIVE_CHUNK_ROWS)
            text = _native_rows(b - a, 1 + a, self.rec[a:b], blobs, sblobs, self.motif, self.motif_b, self.start0[a:b],
                                self.width, self.text, self.text_b, self.text_pos[a:b], self.kind, scores[a:b],
                                self.kind_b, None if scores_b is None else scores_b[a:b])
            if text is None:
                if a:
                    raise ValueError("hit score outside the text formats of the native hits.tab writer")
                return False
            if not a:
                _emit(out, "\t".join(_HEADER if self.motif_b is None else _COMBINED_HEADER) + "\n")
            _emit(out, text)
        return True


def _writer_scores(kind, scores):
    """`scores` in the dtype rs_host_format_hits* reads for score_kind `kind`: 0 / 1 float32 rounded to three
    decimals, 4 int32 thousandths, 2 / 3 float64."""
    kind &= 0xFF
    if kind <= 1:
        return _round3_f32(scores)
    return np.ascontiguousarray(scores, np.int32 if kind == 4 else np.float64)


def _fasta_table(motif_id, width, kind, batches, rec, start0, scores):
    """The _HitTable of a single-modality FASTA scan (modes RNA / SS) from its hits: record index over all
    `batches`, 0-based start, scores as the device returned them."""
    ids = [i for b in batches for i in b.ids]
    descs = [d for b in batches for d in b.descriptions]
    text, offsets = _record_text(batches)
    text_pos = offsets[rec] + start0

    def frame():
        if not ids:
            return pd.DataFrame()
        logodds = _round3_f32(scores) if kind == "rna" else _round3_f64(scores)
        return _assemble_fasta_frame(len(ids), rec, ids, descs, motif_id, start0, width,
                                     _fragments(text, text_pos, width), logodds)
    if kind == "rna":                      # float32 text unless a record has no hit (H8, a17)
        score_kind = 1 if (np.bincount(rec, minlength=len(ids)) == 0).any() else 0
    else:                                  # 4: thousandths rounded on the device
        score_kind = 4 if scores.dtype == np.int32 else 2
    return _HitTable(frame, rec, start0, ids, descs, motif_id, width, text, text_pos, score_kind, scores)


class _StringBlobs(object):
    """Per-record id and description strings as (utf-8 blob, offsets) pairs for the C writer."""

    def __init__(self, ids, descs):
        self.id_blob, self.id_off = self._pack(ids)
        self.desc_blob, self.desc_off = self._pack(descs)

    @staticmethod
    def _pack(strings):
        enc = [s.encode("utf-8") for s in strings]
        off = np.zeros(len(enc) + 1, np.int64)
        if enc:
            np.cumsum([len(e) for e in enc], out=off[1:])
        return b"".join(enc), off


def _native_rows(n_rows, match_first, rec, blobs, sblobs, motif_a, motif_b, start0, width, text_a, text_b,
                 text_pos, kind_a, scores_a, kind_b, scores_b):
    """Text of n_rows hits.tab rows from arrays (single-modality when motif_b is None, combined
    otherwise); None when the native formatter declines."""
    from . import _lib
    if n_rows == 0:
        return ""
    rec = np.ascontiguousarray(rec, np.int64)
    start0 = np.ascontiguousarray(start0, np.int64)
    text_pos = np.ascontiguousarray(text_pos, np.int64)
    text_a = None if text_a is None else np.ascontiguousarray(text_a, np.uint8)
    text_b = None if text_b is None else np.ascontiguousarray(text_b, np.uint8)
    ptr = lambda a: 0 if a is None else a.ctypes.data
    capacity = int(n_rows) * 160 + 4096
    written = np.zeros(1, np.int64)
    while True:
        out = np.empty(capacity, np.uint8)
        if motif_b is None:
            rc = _lib.lib.rs_host_format_hits(
                n_rows, match_first, rec.ctypes.data, blobs.id_blob, blobs.id_off.ctypes.data, blobs.desc_blob,
                blobs.desc_off.ctypes.data, motif_a.encode("utf-8"), start0.ctypes.data, width, ptr(text_a),
                text_pos.ctypes.data, kind_a, scores_a.ctypes.data, out.ctypes.data, capacity, written.ctypes.data)
        else:
            rc = _lib.lib.rs_host_format_hits_combined(
                n_rows, match_first, rec.ctypes.data, blobs.id_blob, blobs.id_off.ctypes.data, blobs.desc_blob,
                blobs.desc_off.ctypes.data, None if sblobs is None else sblobs.desc_blob,
                0 if sblobs is None else sblobs.desc_off.ctypes.data, motif_a.encode("utf-8"),
                motif_b.encode("utf-8"), start0.ctypes.data, width, ptr(text_a), ptr(text_b), text_pos.ctypes.data,
                kind_a, scores_a.ctypes.data, kind_b, scores_b.ctypes.data, out.ctypes.data, capacity,
                written.ctypes.data)
        if rc == _lib.RS_ERR_WORKSPACE:
            capacity = int(written[0]) + 64
            continue
        if rc != _lib.RS_OK:
            return None
        return out[:int(written[0])].tobytes().decode("utf-8", "replace")


def _emit(out, text):
    """Write to a text stream, through its binary buffer when it has one (sys.stdout)."""
    if hasattr(out, "buffer"):
        out.flush()
        out.buffer.write(text.encode("utf-8"))
    else:
        out.write(text)


def _scan_fasta_hits(fasta_file, pssm, alphabet, minscore, found=None):
    """All records of a FASTA input in one (or a few) kernel launches, as a _HitTable (None on ranks other than
    0 under torchrun).  `found`: this motif's _Found hits from the batched scan of its motif collection
    (_batched_fasta_hits); the input is then not scanned again."""
    eprint("Scanning sequences ")
    motif_id, pm = _first_motif(pssm)
    kind = _kind_of(alphabet)
    batches = _cached_batches(fasta_file, alphabet)
    if found is None:
        table = _table_for(pm, kind)
        found = _Found(_scan_batches(batches, lambda batch: _scan_batch(batch, table, kind, minscore),
                                     [table.shape[0]], [np.float64]))
    eprint("Processed %d sequences" % sum(len(b.ids) for b in batches))
    return None if found.hits is None else _fasta_table(motif_id, pm.length, kind, batches, *found.hits)


class _Found(object):
    """One motif's (pair's) hits from a batched scan, in record coordinates: the columns (record index, 0-based
    start, scores) -- (record index, 0-based start, sequence scores, structure scores) for joint hits -- on rank
    0, None on the other ranks under torchrun."""

    def __init__(self, hits):
        self.hits = hits


def _fasta_many_hits(batches, kind, tables, minscore):
    """Hits of every table on the FASTA input `batches` from one device.scan_onehot_many call per batch: one
    (record index, 0-based start, scores) tuple per table, or None per table on ranks other than 0.  Under
    torchrun each rank scans its own pieces and the whole collection makes ONE _gather."""
    from . import device

    def scan(batch):
        motif, pos, scores, _ = device.scan_onehot_many(batch.stream, tables, minscore)
        return pos, scores, motif
    dtypes = [np.float32 if kind == "rna" else np.float64, np.int32]
    return _by_motif(_scan_batches(batches, scan, [t.shape[0] for t in tables], dtypes), len(tables))


def _by_motif(hits, n_motifs):
    """Gathered (rec, start0, scores..., motif) columns -> one (rec, start0, scores...) tuple per motif, in record
    order; None per motif on ranks other than 0."""
    if hits is None:
        return [None] * n_motifs
    order = np.argsort(hits[-1], kind="stable")       # rank order (= record order) within each motif
    cols = [c[order] for c in hits]
    cut = np.searchsorted(cols[-1], np.arange(n_motifs + 1))
    return [tuple(c[a:b] for c in cols[:-1]) for a, b in zip(cut[:-1], cut[1:])]


def _pair_many_hits(seq_batches, struct_batches, seq_tables, struct_tables, minscore):
    """Joint hits of every (sequence, structure) table pair on two FASTA inputs that line up (_lined_up) from one
    device.scan_pair_onehot_many call per device batch: one (record index, 0-based start, sequence scores,
    structure scores) tuple per pair, or None per pair on ranks other than 0; one _gather for the collection."""
    from . import device

    def scan(pair):
        motif, pos, seq_sc, scores, _ = device.scan_pair_onehot_many(pair[0].stream, pair[1].stream, seq_tables,
                                                                     struct_tables, minscore)
        return pos, seq_sc, scores, motif
    hits = _scan_batches(list(zip(seq_batches, struct_batches)), scan, [t.shape[0] for t in seq_tables],
                         [np.float32, np.float64, np.int32])
    return _by_motif(hits, len(seq_tables))


def _scan_fasta_hits_computed_bg(fasta_file, pfm_file, pseudocount, alphabet, minscore):
    """compute_background -> load_motif -> scan (rnascan.py:507-521) for a FASTA input whose background is
    computed from the same data, without idling the device between the three: the decision pass starts from
    a provisional table the device derives from its own counts while the counts travel to the host, the
    exact log-odds are built there (Python's math.log, as Biopython does) and the finish pass decides every
    candidate with them (device.BackgroundOneHotScan; results identical to the serial order).
    Returns (bg, pssm, _HitTable), or None when this shape of run takes the serial path."""
    from . import device
    kind = _kind_of(alphabet)
    if kind not in ("rna", "struct"):
        return None
    columns = _columns(kind)
    if not np.isfinite(minscore) or any(letter not in columns for letter in alphabet.letters):
        return None
    batches = _cached_batches(fasta_file, alphabet)
    if len(batches) != 1 or batches[0].own is not None or batches[0].stream.n == 0:
        return None
    batch = batches[0]
    try:
        counts = _pfm_counts(pfm_file)
        norm = motifs.normalize_counts(motifs.Motif(alphabet=alphabet, counts=counts).counts, alphabet.letters,
                                       pseudocount)
        prob = np.array([norm[c] for c in columns], dtype=np.float64).T.copy()
    except Exception:
        return None                       # the serial path reports what is wrong with the PFM
    if not (1 <= prob.shape[0] <= 16) or not np.isfinite(prob).all():
        return None
    state = {}

    def table_fn(counts8):
        state["bg"] = _background_from_counts(np.asarray(counts8, np.int64), len(batch.ids), alphabet, True)
        state["pssm"] = load_motif(pfm_file, pseudocount, alphabet, state["bg"])
        return _table_for(_first_motif(state["pssm"])[1], kind)

    eprint("Calculating background probabilities...")
    with STATS.phase("scan_s"):
        pos, scores, _, _ = device.scan_onehot_bg(batch.stream, prob, table_fn, minscore)
    STATS.add("scored_positions", int(np.maximum(batch.stream.lengths - prob.shape[0] + 1, 0).sum()))
    motif_id, pm = _first_motif(state["pssm"])
    eprint("Scanning sequences ")
    keep, rec, start0 = batch.locate(pos)
    table = _fasta_table(motif_id, pm.length, kind, batches, rec[keep], start0[keep], scores[keep])
    eprint("Processed %d sequences" % len(table.ids))
    return state["bg"], state["pssm"], table


# one parsed + uploaded input is reused by compute_background and the scan that follows it
_BATCH_CACHE = {}


def _cache_key(fasta_file, alphabet):
    paths = [fasta_file] if isinstance(fasta_file, str) else list(fasta_file)
    try:
        stamp = tuple((os.path.abspath(p), os.path.getmtime(p), os.path.getsize(p)) for p in paths)
    except OSError:
        return None
    return (stamp, _kind_of(alphabet), _seq.is_ambiguous_rna_alphabet(alphabet))


def _count_input(key, batches):
    """--stats: every input counts once per run, however often it is looked up."""
    seen = STATS.notes.setdefault("_inputs", set())
    if key is None or key not in seen:
        seen.add(key)
        STATS.add("symbols", sum(int(b.stream.lengths.sum()) for b in batches))
        STATS.add("records", sum(len(b.ids) for b in batches))


def _cached_batches(fasta_file, alphabet):
    key = _cache_key(fasta_file, alphabet)
    if key is not None and key in _BATCH_CACHE:
        _count_input(key, _BATCH_CACHE[key])
        return _BATCH_CACHE[key]
    with STATS.phase("ingest_fasta_s"):
        batches = list(_record_batches(fasta_file, alphabet))
    _count_input(key, batches)
    if key is not None:
        while len(_BATCH_CACHE) >= 2:                      # sequence + structure input of one run
            _BATCH_CACHE.pop(next(iter(_BATCH_CACHE)))
        if sum(b.stream.n for b in batches) <= MAX_BATCH_SYMBOLS:
            _BATCH_CACHE[key] = batches
    return batches


def _profile_files(directory):
    structures = glob.glob(directory + "/structure.*.txt")
    if len(structures) == 0:
        raise IOError("No averaged structure files found")
    return structures


def _load_profile_dir(directory, write_pack=False):
    """This rank's share of the profiles of a directory as one packed stream:
    (this rank's paths, all paths, HostProfile, lengths).  A valid ``rnascan_b200.pack`` (pack.py) is
    mapped instead of parsing the text; `write_pack` leaves one behind after parsing."""
    from . import device, shard, pack
    rank, size = shard.world()
    pk = pack.read(directory)
    try:
        files = _profile_files(directory)
    except IOError:
        if pk is None:
            raise
        files = [directory + os.sep + nm for nm in pk.names]            # a pack standing for the text files
    else:
        if size > 1:
            files = shard.broadcast_object(files)      # one canonical order (os.listdir order is per process)
        if pk is not None and not pack.matches(pk, files):
            pk = None
    n_files = len(files)
    lo, hi = 0, n_files
    if size > 1:
        sizes = pk.lengths.tolist() if pk is not None else [os.path.getsize(f) for f in files]
        mine = [r for (r, a, b, o) in shard.plan_shards(sizes, size, 1)[rank] if a == 0]    # W = 1: whole files
        lo, hi = (mine[0], mine[-1] + 1) if mine else (0, 0)
    if pk is not None:
        lengths = pk.lengths[lo:hi]
        r0 = int(pk.offsets[lo]) if hi > lo else 0
        r1 = int(pk.offsets[hi - 1] + pk.lengths[hi - 1] + 1) if hi > lo else 0
        hp = device.HostProfile(pk.rows[r0:r1], q8=None if pk.q8 is None else pk.q8[r0:r1], q8_scale=pk.q8_scale,
                                stats=pk.stats, q4=None if pk.q4 is None else pk.q4[r0:r1])
        if size == 1:                                  # repeated scans of one pack: a pinned copy of the section (pack.py)
            hp.page_locked = (pk.page_locked, {"q8": hp.q8, "q4": hp.q4})
        return files[lo:hi], files, hp, lengths
    packed, lengths = _read_profiles_packed(files[lo:hi])
    hp = device.HostProfile(packed)
    if write_pack and size == 1 and n_files:
        sep = np.zeros(packed.shape[0], np.uint8)
        sep[np.cumsum(lengths + 1) - 1] = device._lib.RS_SEP
        ok = hp.make_q8(sep) and hp.make_q4(sep)
        try:
            pack.write(directory, files, packed, lengths, hp.stats(), hp.q8 if ok else None, hp.q8_scale,
                       q4=hp.q4 if ok else None)
        except OSError as exc:
            eprint("Could not write %s: %s" % (pack.pack_path(directory), exc))
    return files[lo:hi], files, hp, lengths


def _profile_dir_streams(directory, debug, seq_batches, write_pack):
    """The packed streams of a profile directory: (this rank's files, the ids of ALL files, HostProfile, lengths,
    this rank's ids, offsets, codes).
    `codes` holds separators only, or -- with `seq_batches` (combined mode) -- the sequence symbols of the
    record with the same id, aligned row by row; rows beyond the shorter of the two get an invalid symbol (no
    joint window exists there).  Cached per directory while a motif collection is being scanned."""
    from . import device
    key = (os.path.abspath(directory), bool(debug), None if seq_batches is None else id(seq_batches))
    if key in _PROFILE_DIR_CACHE:
        return _PROFILE_DIR_CACHE[key]
    with STATS.phase("ingest_profiles_s"):
        files, all_files, hp, lengths = _load_profile_dir(directory, write_pack)
    n_files = len(all_files)
    STATS.add("profile_rows", int(lengths.sum()))
    STATS.add("profile_files", len(files))
    STATS.notes["profile_source"] = "pack" if isinstance(hp.rows, np.memmap) else "text"
    # rnascan.py:299-301: the id is what stands between "structure." and ".txt" (the full path in debug mode)
    cut = len(os.path.dirname(files[0])) + 1 + 10 if files else 0     # "<directory>/structure."
    names = list(files) if debug else [path[cut:-4] for path in files]
    n_prof = len(files)
    offsets = np.zeros(n_prof, np.int64)
    if n_prof > 1:
        np.cumsum(lengths[:-1] + 1, out=offsets[1:])
    codes = np.zeros(int(lengths.sum() + n_prof), np.uint8)
    if seq_batches is not None:
        by_id = {}
        for batch in seq_batches:
            for rid, text in zip(batch.ids, batch.full_texts):
                by_id.setdefault(rid, text)
        for k, name in enumerate(names):
            seg = codes[offsets[k]:offsets[k] + lengths[k]]
            seg[:] = device._lib.RS_RNA_OTHER
            text = by_id.get(name)
            if text is not None:
                sym = device.pack_texts([text], "rna")[0][:-1]
                m = min(len(sym), len(seg))
                seg[:m] = sym[:m]
    if n_prof:
        codes[offsets + lengths] = device._lib.RS_SEP
    if len(codes) and hp.q8 is not None and seq_batches is not None:
        q8 = np.array(hp.q8)                          # the pack's rows carry no sequence: add the symbols
        q8[:, 7] = codes
        hp.q8 = q8
        if hp.q4 is not None:
            q4 = np.array(hp.q4)
            q4[:, 3] = (q4[:, 3] & 0x0F) | ((codes & 0x0F) << 4)
            hp.q4 = q4
    all_names = list(all_files) if debug else [path[cut:-4] for path in all_files]
    out = (files, all_names, hp, lengths, names, offsets, codes)
    if _PROFILE_DIR_CACHE_ON[0]:
        _PROFILE_DIR_CACHE[key] = out
    return out


def _scan_profile_dir(directory, pssm, minscore, debug, seq_batches=None, seq_pm=None, seq_hits=None,
                      write_pack=False, found=None):
    """All ``structure.<id>.txt`` profiles of a directory in one pass (rnascan.py:348-375), as a _HitTable (None
    on ranks other than 0 under torchrun).
    With `seq_batches`/`seq_pm` (combined mode) the sequence PSSM is evaluated on the same windows and only
    those passing BOTH thresholds come back: the rows of the combined hits.tab, whose sequence side is the
    table `seq_hits` of the sequence scan.  The float64 rows stay on the host: the device filters a float32
    shadow or the pack's 8-byte quantised rows and re-scores the few windows near the threshold from the exact
    rows (device.scan_profile_host).  `found`: the _Found hits of this motif (pair) from the batched scan of a
    motif collection (_batched_profile_hits).  Under torchrun every rank takes a contiguous range of files
    balanced by size and rank 0 gathers the hits."""
    from . import device, shard
    eprint("Scanning averaged secondary structures ")
    motif_id, pm = _first_motif(pssm)
    tq = _structure_table(pm)
    width = tq.shape[0]
    rank, size = shard.world()
    files, all_names, hp, lengths, names, offsets, codes = _profile_dir_streams(directory, debug, seq_batches,
                                                                                write_pack)
    n_files = len(all_names)
    seq = None if seq_batches is None else _table_for(seq_pm, "rna")
    STATS.add("scored_positions", int(np.maximum(lengths - width + 1, 0).sum()))
    if found is not None:                 # this motif (pair) was scanned in the collection's batched pass
        hits = found.hits
    else:
        rec = start0 = np.zeros(0, np.int64)
        scores, seq_scores = np.zeros(0, np.float64), np.zeros(0, np.float32)
        if len(codes):
            with STATS.phase("scan_s"):
                pos, seq_scores, scores, scanner = device.scan_profile_host(codes, hp, seq, tq, minscore,
                                                                            return_scanner=True)
            if scanner is not None:
                STATS.notes["profile_filter_form"] = scanner.form
                STATS.add("h2d_bytes", scanner.h2d_bytes)
                STATS.add("candidates", scanner.n_candidates)
            rec = np.searchsorted(offsets, pos, side="right") - 1
            start0 = pos - offsets[rec]
        first = all_names.index(names[0]) if names else 0      # this rank's files are a contiguous range
        hits = _gather([(rec + first, start0) + (() if seq is None else (seq_scores,))
                        + (np.asarray(scores, np.float64),)])
    # Combined mode without a single joint hit: the reference's merge still needs the STRUCTURE frame's columns,
    # which exist iff some window passes the structure threshold on its own (else its merge raises KeyError, and
    # so does ours): one structure-only pass settles it -- only in this corner, on every rank when sharded.
    any_struct_hits = None
    if seq is not None:
        need = len(hits[0]) == 0 if rank == 0 else None
        if size > 1:
            need = shard.broadcast_object(need)
        if need:
            local = bool(len(codes)) and len(device.scan_profile_host(codes, hp, None, tq, minscore)[0]) > 0
            ranks = shard.gather_objects(local) if size > 1 else [local]
            any_struct_hits = bool(ranks and any(ranks))
    eprint("Processed %d sequences" % n_files)
    if hits is None:                      # only rank 0 prints
        return None
    rec, start0, scores = hits[0], hits[1], hits[-1]
    if seq is None:
        frame = lambda: _averaged_dir_frame(all_names, rec, motif_id, start0, width, scores)
        shape = _dir_frame_shape(np.bincount(rec, minlength=n_files))
        if shape not in ("hit", "hit,empty"):       # first file without hits (another column order), or no hit
            return _HitTable(frame)
        # Start / End print as floats when some file has no hit; the scores unrounded
        return _HitTable(frame, rec, start0, all_names, [""] * n_files, motif_id, width, None, start0,
                         3 | (0x100 if shape == "hit,empty" else 0), scores)
    first_has_hits = None
    if n_files > 1 and len(lengths):
        # combined mode: `rec` only knows the windows where BOTH scores pass, but the column order of the
        # reference's structure frame -- and with it that of the merged output -- follows the first file's own
        # structure hits: one small structure-only scan of that file settles it
        head = device.HostProfile(np.ascontiguousarray(hp.rows[:int(lengths[0])]))
        first_has_hits = len(device.scan_profile_host(None, head, None, tq, minscore)[0]) > 0

    def frame():
        return combine(seq_hits.frame(), _averaged_dir_frame(all_names, rec, motif_id, start0, width, scores,
                                                             first_has_hits, any_struct_hits))
    if first_has_hits is False:           # unusual column order: pandas prints it
        return _HitTable(frame)
    # the joint windows in the order of the inner join, whose left side is the sequence frame: sequence record,
    # then Start
    text, text_offsets = _record_text(seq_batches)
    index = {rid: k for k, rid in enumerate(seq_hits.ids)}
    seq_rec = np.array([index.get(nm, -1) for nm in all_names], np.int64)[rec]
    keep = seq_rec >= 0
    order = np.lexsort((start0[keep], seq_rec[keep]))
    seq_rec, seq_start0 = seq_rec[keep][order], start0[keep][order]
    return _HitTable(frame, seq_rec, seq_start0, seq_hits.ids, seq_hits.descs, seq_hits.motif, width, text,
                     text_offsets[seq_rec] + seq_start0, seq_hits.kind, hits[2][keep][order], motif_id, None, 3,
                     scores[keep][order])


_DIR_PROTOTYPES = {}


def _dir_frame_prototype(shape):
    """One-row stand-ins for the per-file frames of the reference -- "hit": pd.DataFrame(list of Series), "empty":
    pd.DataFrame([]) -- with the id columns added, concatenated in the order `shape` names and the last two
    columns moved to the front, all through the reference's own pandas calls.  Column order and dtypes of the
    result depend on nothing else, so each of the five shapes is worked out once per process."""
    proto = _DIR_PROTOTYPES.get(shape)
    if proto is None:
        parts = []
        for kind in (shape.split(",") if shape else []):
            part = pd.DataFrame([pd.Series(["m", 1, 2, ".", 0.5], index=HIT_COLUMNS)]) if kind == "hit" \
                else pd.DataFrame([])
            _add_sequence_id(part, "id", "")
            parts.append(part)
        proto = pd.concat(parts) if parts else pd.DataFrame()
        cols = proto.columns.tolist()
        proto = _DIR_PROTOTYPES[shape] = proto[cols[-2:] + cols[:-2]]
    return proto


def _dir_frame_shape(hits_per_file, first_has_hits=None, any_struct_hits=None):
    """Which per-file frames the reference concatenates, as far as the result's columns and dtypes go: "hit" (every
    file has one), "hit,empty" / "empty,hit" (some file has none; the first file's frame decides the column order),
    "empty" (no hit anywhere), "" (no file).  `hits_per_file`: the number of hits of each file, in file order."""
    if not len(hits_per_file):
        return ""
    n = int(hits_per_file.sum())
    any_empty = bool((hits_per_file == 0).any())
    if n == 0 and any_struct_hits and first_has_hits is None:
        first_has_hits = len(hits_per_file) == 1   # a single file: it is the one with the structure hits
    if n == 0 and not first_has_hits and not any_struct_hits:
        return "empty"
    if not any_empty:
        return "hit"
    if first_has_hits is None:
        first_has_hits = hits_per_file[0] > 0
    return "hit,empty" if first_has_hits else "empty,hit"


def _averaged_dir_frame(all_names, rec, motif_id, start0, width, scores, first_has_hits=None, any_struct_hits=None):
    """The frame the reference gets for a directory (rnascan.py:348-375, 408-413): one frame per file built
    by pd.DataFrame(list of Series) -- or, for a file without hits, pd.DataFrame([]) with only the two id
    columns -- then pd.concat and the last two columns moved to the front.  What pandas makes of that mix
    (column order follows the first file's frame; Start/End turn float when any file had no hit; only the id
    columns remain when no file had one) is learnt from one-row prototypes run through the same calls, then
    applied to the whole result at once.  Hit i is in file `all_names[rec[i]]`."""
    rec = np.asarray(rec, np.int64)
    n = len(rec)
    proto = _dir_frame_prototype(_dir_frame_shape(np.bincount(rec, minlength=len(all_names)), first_has_hits,
                                                  any_struct_hits))
    data = {"Sequence_ID": np.array(all_names, dtype=object)[rec], "Description": np.array([""] * n, dtype=object),
            "Motif_ID": np.array([motif_id] * n, dtype=object), "Start": np.asarray(start0, np.int64) + 1,
            "End": np.asarray(start0, np.int64) + width, "Sequence": np.array(["."] * n, dtype=object),
            "LogOdds": np.asarray(scores, dtype=np.float64)}
    frame = pd.DataFrame({c: data[c] for c in proto.columns})
    for c in ("Start", "End", "LogOdds"):
        if c in frame.columns and n:
            frame[c] = frame[c].astype(proto[c].dtype)
    return frame


def scan_main(fasta_file, pssm, alphabet, bg, args):
    """Scan one input -- a SeqRecord, a directory of averaged profiles or a FASTA file -- and
    return the hit frame with Sequence_ID and Description in front (rnascan.py:335-413)."""
    table = _scan_table(fasta_file, pssm, alphabet, args)
    return pd.DataFrame() if table is None else table.frame()


def _scan_table(fasta_file, pssm, alphabet, args, found=None):
    """scan_main's scan as a _HitTable (None on ranks other than 0 under torchrun); `found`: the _Found hits of
    this motif from the batched scan of its collection."""
    if _seq.is_seqrecord(fasta_file):
        final = scan_all(fasta_file, pssm, alphabet, args.minscore)
        _add_sequence_id(final, "testseq", "")
        cols = final.columns.tolist()
        final = final[cols[-2:] + cols[:-2]]
        eprint("Processed 1 sequences")
        return _HitTable(lambda: final)
    if os.path.isdir(fasta_file):
        return _scan_profile_dir(fasta_file, pssm, args.minscore, args.debug, write_pack=getattr(args, "pack", False),
                                 found=found)
    return _scan_fasta_hits(fasta_file, pssm, alphabet, args.minscore, found)


def combine(seq_results, struct_results):
    """Inner join of the two hit sets on Sequence_ID, Start, End; the combined score is the
    sum of the two (rnascan.py:416-434).  A hit exists only where BOTH scans reported one."""
    keys = ["Sequence_ID", "Start", "End"]
    left, right = seq_results, struct_results
    for key in keys[1:]:                     # pandas >= 2 refuses int64-vs-object merge keys
        if key in left and key in right and left[key].dtype != right[key].dtype:
            left, right = left.copy(), right.copy()
            left[key], right[key] = left[key].astype(object), right[key].astype(object)
    result = pd.merge(left, right, on=keys)
    result.rename(columns={"Description_x": "Description.Seq", "Description_y": "Description.Struct",
                           "Sequence_x": "Sequence.Seq", "Sequence_y": "Sequence.Struct",
                           "Motif_ID_x": "Motif_ID.Seq", "Motif_ID_y": "Motif_ID.Struct",
                           "LogOdds_x": "LogOdds.Seq", "LogOdds_y": "LogOdds.Struct"}, inplace=True)
    result["LogOdds.SeqStruct"] = result["LogOdds.Seq"] + result["LogOdds.Struct"]
    return result


###############################################################################
# Background functions
###############################################################################
def compute_background(fastas, alphabet, verbose=True):
    """p(letter) = (count + 1) / (sum(counts) + |alphabet|) over all records, counted on the
    device (exact integers), keys in ``alphabet.letters`` order (rnascan.py:440-465).
    Counting is case-sensitive on the pre-processed sequence: lower-case structure letters
    are scored but not counted (SURVEY.md H11)."""
    from . import device
    eprint("Calculating background probabilities...")
    kind = _kind_of(alphabet)
    if any(letter not in _columns(kind) for letter in alphabet.letters):
        raise NotImplementedError("GPU background counting of nucleotides supports the letters A, C, G, U only "
                                  "(alphabet %r)" % (alphabet.letters,))
    counts = np.zeros(8 if kind in ("rna", "struct") else len(kind.letters), dtype=np.int64)
    n_records = 0
    for batch in _cached_batches(fastas, alphabet):
        if batch.counts is None:
            batch.counts = device.histogram(batch.stream).cpu().numpy() - batch.overlap_counts()
        counts += batch.counts
        n_records += len(batch.ids)
    counts = _allreduce_counts(counts)
    return _background_from_counts(counts, n_records, alphabet, verbose)


def _background_from_counts(counts, n_records, alphabet, verbose=True):
    """(count + 1) / (total + |alphabet|) per letter, messages and checks of rnascan.py:454-465."""
    columns = _columns(_kind_of(alphabet))
    content = defaultdict(int)
    total = len(alphabet.letters)
    if n_records:
        for letter in alphabet.letters:
            amount = int(counts[columns.index(letter)])
            content[letter] += amount
            total += amount
    pct_sum = 0
    for letter, count in content.items():
        content[letter] = (float(count) + 1) / total
        if content[letter] <= 0.05:
            warnings.warn("Letter %s has low content: %0.2f" % (letter, content[letter]), Warning)
        pct_sum += content[letter]
    if verbose:
        eprint(dict(content))
    assert abs(1.0 - pct_sum) < 0.0001, "Background sums to %f" % pct_sum
    return content


def _allreduce_counts(counts):
    """Sum the integer background counts over all ranks when running under torchrun (the
    path's only collective); identity in a single process."""
    from . import shard
    return shard.allreduce_counts(counts)


def load_background(bg_file, uniform, *args):
    """Dict-literal background file, else computed from the input, else None = uniform
    (rnascan.py:468-484)."""
    if bg_file:
        eprint("Reading custom background probabilities from %s" % bg_file)
        with open(bg_file, "r") as fin:
            bg = ast.literal_eval(fin.read())
            eprint(dict(bg))
    elif not uniform:
        bg = compute_background(*args)
    else:
        bg = None
    return bg


###############################################################################
# Main
###############################################################################
def _unique_ids(batches):
    """The record ids of an input, or None when an id repeats (duplicate ids join across records)."""
    ids = [i for b in batches for i in b.ids]
    return ids if len(set(ids)) == len(ids) else None


def _lined_up(seq_batches, struct_batches):
    """(sequence text, structure text, record offsets) when the two FASTA inputs of the combined mode can be
    scanned together -- unique ids, the same ids in the same order and the same whole-record lengths, so that
    every window lines up -- else None (the inputs are then scanned apart and merged as the reference does)."""
    ids = _unique_ids(seq_batches)
    if ids is None or [i for b in struct_batches for i in b.ids] != ids:
        return None
    seq_text, offsets = _record_text(seq_batches)
    struct_text, struct_offsets = _record_text(struct_batches)
    if len(struct_text) != len(seq_text) or not np.array_equal(struct_offsets, offsets):
        return None
    return seq_text, struct_text, offsets


def _combined_hits(seq_file, struct_file, seq_pssm, struct_pssm, seq_hits, args, found=None):
    """The table of the combined mode (rnascan.py:416-434) on top of `seq_hits`, the sequence scan's table; None
    on ranks other than 0 under torchrun.  The structure side is scanned ON THE DEVICE only where the sequence
    score also passes (the inner join keeps nothing else): one fused launch instead of a second full scan +
    merge.  Where the two inputs cannot be scanned together (-t, different motif widths, duplicate ids, inputs
    that do not line up) the structure input is scanned on its own and merged as the reference does.
    `found`: the pair's joint _Found hits from the batched scan of its collection."""
    from . import device
    _, seq_pm = _first_motif(seq_pssm)
    motif_id, pm = _first_motif(struct_pssm)
    width = pm.length
    structure = ContextualSecondaryStructure()

    def merged():
        struct_hits = _scan_table(struct_file, struct_pssm, structure, args)
        return None if struct_hits is None else _HitTable(lambda: combine(seq_hits.frame(), struct_hits.frame()))
    if _seq.is_seqrecord(struct_file) or seq_pm.length != width:
        return merged()
    seq_batches = _cached_batches(seq_file, IUPAC.IUPACUnambiguousRNA())
    ids = _unique_ids(seq_batches)
    if ids is None:
        return merged()
    if os.path.isdir(struct_file):
        return _scan_profile_dir(struct_file, struct_pssm, args.minscore, args.debug, seq_batches, seq_pm, seq_hits,
                                 getattr(args, "pack", False), found)
    struct_batches = _cached_batches(struct_file, structure)
    lined = _lined_up(seq_batches, struct_batches)
    if lined is None:
        return merged()
    seq_text, struct_text, offsets = lined
    eprint("Scanning sequences ")
    if found is None:
        ts, tq = _table_for(seq_pm, "rna"), _table_for(pm, "struct")
        found = _Found(_scan_batches(
            list(zip(seq_batches, struct_batches)),
            lambda pair: device.scan_pair_onehot(pair[0].stream, pair[1].stream, ts, tq, args.minscore),
            [width], [np.float32, np.float64]))
    eprint("Processed %d sequences" % sum(len(qb.ids) for qb in struct_batches))
    if found.hits is None:
        return None
    rec, start0, seq_scores, scores = found.hits
    text_pos = offsets[rec] + start0
    struct_descs = [d for b in struct_batches for d in b.descriptions]

    def frame():                          # the structure frame of the joint windows: the join keeps the same rows
        struct = pd.DataFrame() if not ids else _assemble_fasta_frame(
            len(ids), rec, ids, struct_descs, motif_id, start0, width, _fragments(struct_text, text_pos, width),
            _round3_f64(scores))
        return combine(seq_hits.frame(), struct)
    return _HitTable(frame, rec, start0, seq_hits.ids, seq_hits.descs, seq_hits.motif, width, seq_text, text_pos,
                     seq_hits.kind, seq_scores, motif_id, struct_text, 2, scores, struct_descs)


_PROFILE_DIR_CACHE = {}              # directory -> _profile_dir_streams result while a motif collection is scanned
_PROFILE_DIR_CACHE_ON = [False]


def _multi_pfm_pairs(args):
    """[(sequence PFM | None, structure PFM | None)] when -p and/or -q name a multi-PFM file, else None.
    Two multi-PFM files pair up block by block; an ordinary PFM file on the other side serves every pair."""
    seq_blocks = pfm_blocks(args.pfm_seq) if args.pfm_seq else None
    struct_blocks = pfm_blocks(args.pfm_struct) if args.pfm_struct else None
    if seq_blocks is None and struct_blocks is None:
        return None
    if seq_blocks is not None and struct_blocks is not None and len(seq_blocks) != len(struct_blocks):
        eprint("The multi-PFM files hold %d and %d motifs" % (len(seq_blocks), len(struct_blocks)))
        sys.exit(1)
    count = len(seq_blocks if seq_blocks is not None else struct_blocks)
    seq_side = seq_blocks if seq_blocks is not None else [args.pfm_seq] * count
    struct_side = struct_blocks if struct_blocks is not None else [args.pfm_struct] * count
    return list(zip(seq_side, struct_side))


def _run_multi(args, seq_type, rank, pairs):
    """A motif collection: the output is the concatenation of what one reference run per motif (pair) prints
    (rnascan.py:490-567 once per PFM).  Inputs are parsed and uploaded once; with a directory of averaged
    profiles all pairs are scanned in ONE batched pass (rs_scan_batched: tensor cores from 32 motifs on)."""
    import copy
    _PROFILE_DIR_CACHE.clear()
    _PROFILE_DIR_CACHE_ON[0] = True
    try:
        pre = None
        if not args.bgonly:
            pre = (_batched_profile_hits(args, seq_type, pairs) or _batched_fasta_hits(args, seq_type, pairs)
                   or _batched_pair_hits(args, seq_type, pairs))
        for k, (seq_pfm, struct_pfm) in enumerate(pairs):
            one = copy.copy(args)
            one.pfm_seq, one.pfm_struct = seq_pfm, struct_pfm
            _run(one, seq_type, rank, None if pre is None else pre[k])
            if args.bgonly:
                break
    finally:
        _PROFILE_DIR_CACHE_ON[0] = False
        _PROFILE_DIR_CACHE.clear()


def _quiet(fn, *a, **kw):
    """Run `fn` with this module's stderr messages (and low-content warnings) suppressed."""
    global _QUIET
    _QUIET += 1
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            return fn(*a, **kw)
    finally:
        _QUIET -= 1


def _side_tables(args, pfms, alphabet, bg_file, table, fasta=None):
    """`table(pssm)` for the PSSM of every PFM of one side of a motif collection, with that side's background
    (`bg_file`, uniform, or computed over `fasta`), all loaded quietly; None when anything raises (the per-motif
    runs then report it)."""
    bg_input = () if fasta is None else (fasta, alphabet, False)
    try:
        bg = _quiet(load_background, bg_file, args.uniform_background, *bg_input)
        return [table(_first_motif(_quiet(load_motif, pfm, args.pseudocount, alphabet, bg))[1]) for pfm in pfms]
    except Exception:
        return None


def _batched_profile_hits(args, seq_type, pairs):
    """Hits of every motif pair on a directory of averaged profiles from one device.scan_batched call: a
    (None, _Found) per pair, or None when this run does not have that shape (the per-motif scans then run one
    after the other)."""
    from . import device
    if args.testseq or _world_size() > 1 or len(pairs) < 2 or not np.isfinite(args.minscore):
        return None
    struct_file = args.fastafiles[-1] if args.fastafiles else None
    if seq_type not in ("SS", "RNASS") or not struct_file or not os.path.isdir(struct_file):
        return None
    if not (args.bg_struct or args.uniform_background):
        return None                       # an averaged-profile run cannot compute a structure background
    tqs = _side_tables(args, [q for _, q in pairs], ContextualSecondaryStructure(), args.bg_struct, _structure_table)
    if tqs is None:
        return None
    tss = seq_batches = None
    if seq_type == "RNASS":
        rna = IUPAC.IUPACUnambiguousRNA()
        seq_file = args.fastafiles[0]
        tss = _side_tables(args, [p for p, _ in pairs], rna, args.bg_seq, lambda pm: _table_for(pm, "rna"), seq_file)
        if tss is None or any(a.shape[0] != b.shape[0] for a, b in zip(tss, tqs)):
            return None
        try:
            seq_batches = _cached_batches(seq_file, rna)
        except Exception:
            return None                   # the per-motif run reports what is wrong
        if _unique_ids(seq_batches) is None:
            return None
    if max(t.shape[0] for t in tqs) > 24:
        return None
    files, all_names, hp, lengths, names, offsets, codes = _profile_dir_streams(
        struct_file, args.debug, seq_batches, getattr(args, "pack", False))
    if not len(codes) or not device.filter_applies(np.concatenate(tqs), args.minscore, hp.absrow_max()):
        return None
    hits = _profile_collection_hits(offsets, lengths, codes, hp, tss, tqs, args.minscore)
    STATS.notes["batched_motifs"] = len(pairs)
    return [(None, _Found(h)) for h in hits]


def _profile_collection_hits(offsets, lengths, codes, hp, seq_tables, struct_tables, minscore):
    """Hits of every motif (pair) on the streams of a profile directory (_profile_dir_streams) from one
    device.scan_batched call: per motif (pair), the columns (file index, 0-based start, scores) -- (file index,
    0-based start, sequence scores, structure scores) with `seq_tables`."""
    from . import device
    with STATS.phase("scan_s"):
        stream = device.SymbolStream(codes, offsets, lengths)
        profile = device.ProfileStream(hp.rows)
        motif, pos, sq, st, bases = device.scan_batched(stream, profile, seq_tables, struct_tables, minscore)
    out = []
    for a, b in zip(bases[:-1].tolist(), bases[1:].tolist()):
        rec = np.searchsorted(offsets, pos[a:b], side="right") - 1
        out.append((rec, pos[a:b] - offsets[rec]) + (() if sq is None else (sq[a:b],)) + (st[a:b],))
    return out


MULTI_FASTA_MIN_MOTIFS = 2           # motif collections from this size on are scanned over a FASTA input in one pass


def _on_device(batches):
    """True when every batch's stream is resident on a CUDA device (what the batched kernel reads)."""
    return all(b.stream.codes.is_cuda for b in batches)


def _pair_on_device(seq_batches, struct_batches):
    """True when the streams of both inputs are resident on a CUDA device (what the pair kernel reads).  Kept apart
    from _on_device so that replacing one check (as the CPU tests do) opens only its own route."""
    return all(b.stream.codes.is_cuda for b in list(seq_batches) + list(struct_batches))


def _fasta_inputs(args, pairs, n_inputs):
    """The `n_inputs` FASTA inputs of a motif collection run that a batched FASTA route can take -- no -t or
    --bgonly, at least MULTI_FASTA_MIN_MOTIFS motifs, a finite -m, no directory -- else None."""
    if args.testseq or args.bgonly or len(pairs) < MULTI_FASTA_MIN_MOTIFS or not np.isfinite(args.minscore):
        return None
    files = (args.fastafiles or [])[:n_inputs]
    if len(files) < n_inputs or any(os.path.isdir(f) for f in files):
        return None
    return files


def _batched_fasta_hits(args, seq_type, pairs):
    """Hits of every motif of a collection scanned over one FASTA input (modes RNA / SS) by
    device.scan_onehot_many: a (_Found, None) (RNA) or (None, _Found) (SS) per motif, or None when this run does
    not have that shape (the per-motif scans then run one after the other).  The background is taken once,
    quietly; every _run still prints its own messages."""
    from . import device
    files = _fasta_inputs(args, pairs, 1)
    if seq_type not in ("RNA", "SS") or files is None:
        return None
    if seq_type == "RNA":
        alphabet, kind, bg_file, pfms = IUPAC.IUPACUnambiguousRNA(), "rna", args.bg_seq, [p for p, _ in pairs]
    else:
        alphabet, kind, bg_file, pfms = ContextualSecondaryStructure(), "struct", args.bg_struct, [q for _, q in pairs]
    batches = _cached_batches(files[0], alphabet)
    if not _on_device(batches):
        return None
    tables = _side_tables(args, pfms, alphabet, bg_file, lambda pm: _table_for(pm, kind), files[0])
    if tables is None or max(t.shape[0] for t in tables) > device.MANY_MAX_W:
        return None
    found = [_Found(h) for h in _fasta_many_hits(batches, kind, tables, args.minscore)]
    STATS.notes["batched_motifs"] = len(pairs)
    return [(f, None) if kind == "rna" else (None, f) for f in found]


def scan_many_fasta(fasta_file, pssms, alphabet, minscore):
    """Scan a FASTA file with MANY motifs in one batched pass per device batch.

    pssms: a list of ``{motif_id: PSSM}`` as load_motif returns them, for the RNA or the
    ContextualSecondaryStructure alphabet.  Returns one DataFrame per motif, equal to what
    scan_main(fasta_file, pssm, alphabet, bg, args) returns for that motif (empty frames on ranks other than 0
    under torchrun).  Motifs wider than 16 and a threshold of -inf are scanned one motif at a time."""
    from . import device
    kind = _kind_of(alphabet)
    if kind not in ("rna", "struct"):
        raise NotImplementedError("scan_many_fasta takes the RNA or the ContextualSecondaryStructure alphabet")
    pms = [_first_motif(p) for p in pssms]
    tables = [_table_for(pm, kind) for _, pm in pms]
    batches = _cached_batches(fasta_file, alphabet)
    many = [k for k, t in enumerate(tables) if t.shape[0] <= device.MANY_MAX_W] if np.isfinite(minscore) else []
    hits = dict(zip(many, _fasta_many_hits(batches, kind, [tables[k] for k in many], minscore))) if many else {}
    frames = []
    for k, (motif_id, pm) in enumerate(pms):
        if k in hits:
            table = None if hits[k] is None else _fasta_table(motif_id, pm.length, kind, batches, *hits[k])
        else:
            table = _quiet(_scan_fasta_hits, fasta_file, pssms[k], alphabet, minscore)
        frames.append(pd.DataFrame() if table is None else table.frame())
    return frames


def _batched_pair_hits(args, seq_type, pairs):
    """Hits of every motif pair of a collection in the combined mode over two FASTA inputs (RNASS): the sequence
    motifs' hits from device.scan_onehot_many and the joint hits of the equal-width pairs from
    device.scan_pair_onehot_many, one call of each per device batch.  A (_Found, _Found) per pair -- (_Found, None)
    for a pair of unequal widths --, or None when this run does not have that shape (the per-pair scans then run
    one after the other).  Both backgrounds are taken once, quietly; every _run still prints its own messages."""
    from . import device
    files = _fasta_inputs(args, pairs, 2)
    if seq_type != "RNASS" or files is None:
        return None
    seq_file, struct_file = files
    rna, structure = IUPAC.IUPACUnambiguousRNA(), ContextualSecondaryStructure()
    seq_batches = _cached_batches(seq_file, rna)
    struct_batches = _cached_batches(struct_file, structure)
    if not _pair_on_device(seq_batches, struct_batches) or len(seq_batches) != len(struct_batches):
        return None
    if _lined_up(seq_batches, struct_batches) is None:
        return None
    ts = _side_tables(args, [p for p, _ in pairs], rna, args.bg_seq, lambda pm: _table_for(pm, "rna"), seq_file)
    tq = None if ts is None else _side_tables(args, [q for _, q in pairs], structure, args.bg_struct,
                                              lambda pm: _table_for(pm, "struct"), struct_file)
    if tq is None or max(t.shape[0] for t in ts + tq) > device.MANY_MAX_W:
        return None
    same = [k for k in range(len(ts)) if ts[k].shape[0] == tq[k].shape[0]]
    seq_hits = _fasta_many_hits(seq_batches, "rna", ts, args.minscore)
    joint = dict(zip(same, _pair_many_hits(seq_batches, struct_batches, [ts[k] for k in same],
                                           [tq[k] for k in same], args.minscore))) if same else {}
    STATS.notes["batched_motifs"] = len(pairs)
    return [(_Found(h), _Found(joint[k]) if k in joint else None) for k, h in enumerate(seq_hits)]


def scan_many_combined(seq_file, struct_file, seq_pssms, struct_pssms, minscore):
    """The combined mode over two FASTA files for MANY motif pairs.

    seq_pssms / struct_pssms: lists of ``{motif_id: PSSM}`` as load_motif returns them (RNA and
    ContextualSecondaryStructure alphabets), paired by position.  Returns one DataFrame per pair, equal to
    combine(scan_main(seq_file, seq_pssm, rna, None, args), scan_main(struct_file, struct_pssm, structure, None,
    args)) for that pair -- columns, dtypes and values -- (empty frames on ranks other than 0 under torchrun).
    Each input is scanned with all its motifs in one batched pass per device batch (scan_many_fasta) and the two
    frames of a pair are joined as the reference joins them: the structure frame's dtypes depend on which records
    have a structure-only hit, which the joint windows alone do not tell.  Any widths and any two inputs are taken;
    a threshold of -inf and motifs wider than 16 are scanned one motif at a time."""
    if len(seq_pssms) != len(struct_pssms):
        raise ValueError("sequence and structure motif lists differ in length")
    seq = scan_many_fasta(seq_file, seq_pssms, IUPAC.IUPACUnambiguousRNA(), minscore)
    struct = scan_many_fasta(struct_file, struct_pssms, ContextualSecondaryStructure(), minscore)
    if _rank() != 0:
        return [pd.DataFrame() for _ in seq_pssms]
    return [combine(a, b) for a, b in zip(seq, struct)]


def scan_many(struct_dir, struct_pssms, minscore, seq_file=None, seq_pssms=None, debug=False):
    """Scan a directory of averaged profiles with MANY motifs in one batched pass (BASELINE config 5).

    struct_pssms (and seq_pssms, for the combined mode) are lists of ``{motif_id: PSSM}`` as load_motif
    returns them.  Returns one DataFrame per motif (pair): what scan_main(struct_dir, ...) returns for that
    structure motif alone -- limited, with seq_pssms, to the windows whose sequence score passes too, with
    an extra ``LogOdds.Seq`` column."""
    if seq_pssms is not None and len(seq_pssms) != len(struct_pssms):
        raise ValueError("sequence and structure motif lists differ in length")
    seq_batches = None
    if seq_pssms is not None:
        seq_batches = _cached_batches(seq_file, IUPAC.IUPACUnambiguousRNA())
    files, all_names, hp, lengths, names, offsets, codes = _profile_dir_streams(struct_dir, debug, seq_batches, False)
    pms = [_first_motif(p) for p in struct_pssms]
    tqs = [_structure_table(pm) for _, pm in pms]
    tss = None if seq_pssms is None else [_table_for(_first_motif(p)[1], "rna") for p in seq_pssms]
    frames = []
    for (motif_id, _), tq, hits in zip(pms, tqs, _profile_collection_hits(offsets, lengths, codes, hp, tss, tqs,
                                                                          minscore)):
        frame = _averaged_dir_frame(all_names, hits[0], motif_id, hits[1], tq.shape[0], hits[-1])
        if tss is not None and len(frame.columns) > 2:
            frame["LogOdds.Seq"] = _round3_f32(hits[2])
        frames.append(frame)
    return frames


class _CleanStdout(object):
    """Under torchrun native libraries write to file descriptor 1 (NCCL prints its version banner there), which
    would end up in hits.tab: for the duration of a multi-rank run fd 1 is pointed at stderr and sys.stdout at
    a private duplicate of the real stdout, so that only what this module prints reaches it."""

    def __enter__(self):
        # (a caller that has replaced sys.stdout -- a test harness capturing it -- keeps its object)
        self.active = int(os.environ.get("WORLD_SIZE", "1")) > 1 and sys.stdout is sys.__stdout__
        if not self.active:
            return self
        try:
            sys.stdout.flush()
            self.saved_fd = os.dup(1)
            os.dup2(2, 1)
            self.saved_stdout = sys.stdout
            sys.stdout = os.fdopen(os.dup(self.saved_fd), "w")
        except (OSError, ValueError, AttributeError):      # stdout is not a real file (captured by a test harness)
            self.active = False
        return self

    def __exit__(self, *exc):
        if not self.active:
            return False
        try:
            sys.stdout.flush()
            sys.stdout.close()
        finally:
            sys.stdout = self.saved_stdout
            os.dup2(self.saved_fd, 1)
            os.close(self.saved_fd)
        return False


def main(argv=None):
    from . import shard
    brought_its_own_group = shard.initialized()          # a caller's process group is left alone
    with _CleanStdout():
        try:
            return _main(argv)
        finally:
            if not brought_its_own_group:
                shard.finalize()


def _main(argv=None):
    tic = time.time()
    from . import shard
    rank, _ = shard.init()                # joins the torchrun rendezvous if there is one
    t_init = time.time() - tic            # importing torch + the rendezvous: reported by --stats
    args = getoptions(argv)
    global REFERENCE_COMPAT
    REFERENCE_COMPAT = bool(args.reference_compat)
    STATS.reset(args.stats)
    if STATS.on:
        from . import _lib
        STATS.phases["import_and_rendezvous_s"] = t_init
        with STATS.phase("cuda_context_s"):
            import torch
            if torch.cuda.is_available():
                torch.cuda.init()
                torch.zeros(1, device="cuda")
        _lib.lib.rs_prof_begin(4096)
    seq_type = _guess_seq_type(args)
    pairs = _multi_pfm_pairs(args)
    if pairs is None:
        _run(args, seq_type, rank)
    else:
        _run_multi(args, seq_type, rank, pairs)
    runtime = float(time.time() - tic)
    if STATS.on:
        _write_stats(args.stats, seq_type, runtime)
    if runtime > 60:
        eprint("Done in %0.4f minutes!" % (runtime / 60))
    else:
        eprint("Done in %0.4f seconds!" % (runtime))


def _run(args, seq_type, rank, precomputed=None):
    """One reference run (rnascan.py:490-567): backgrounds, motifs, scans, hits.tab on STDOUT.
    `precomputed`: (sequence side, structure side) of this motif (pair) from the batched scans of its collection,
    each a _Found or None where that side is scanned here."""
    seq_found, struct_found = precomputed or (None, None)
    bg = None
    seq_file = struct_file = None
    seq_pssm = seq_hits = table = None
    fusable = (_world_size() == 1 and not args.testseq and not args.bgonly and not args.uniform_background
               and precomputed is None)

    if args.testseq:
        testseq_stack = args.testseq.split(",")[::-1]

    if seq_type in ["RNA", "RNASS"]:
        rna = IUPAC.IUPACUnambiguousRNA()
        fused = None
        if args.testseq:
            seq_file = SeqRecord(Seq(testseq_stack.pop()))
        else:
            seq_file = args.fastafiles[0]
            if fusable and not args.bg_seq and not os.path.isdir(seq_file):
                fused = _scan_fasta_hits_computed_bg(seq_file, args.pfm_seq, args.pseudocount, rna, args.minscore)
            if fused is not None:
                bg, seq_pssm, seq_hits = fused
            else:
                bg = load_background(args.bg_seq, args.uniform_background, seq_file, rna, not args.bgonly)
        if args.bgonly:
            if rank == 0:
                print(dict(bg))
            sys.exit()
        if fused is None:                 # else: background, motif and scan were done in one overlapped pass
            seq_pssm = load_motif(args.pfm_seq, args.pseudocount, rna, bg)
            seq_hits = _scan_table(seq_file, seq_pssm, rna, args, seq_found)
        table = seq_hits

    if seq_type in ["SS", "RNASS"]:
        structure = ContextualSecondaryStructure()
        fused = None
        if args.testseq:
            struct_file = SeqRecord(Seq(testseq_stack.pop()))
        elif seq_type == "SS":
            struct_file = args.fastafiles[0]
        else:
            struct_file = args.fastafiles[1]
        if seq_type == "SS" and fusable and not args.bg_struct and not os.path.isdir(struct_file):
            fused = _scan_fasta_hits_computed_bg(struct_file, args.pfm_struct, args.pseudocount, structure,
                                                 args.minscore)
        if fused is not None:
            bg, struct_pssm, table = fused
        elif not args.testseq:
            bg = load_background(args.bg_struct, args.uniform_background, struct_file, structure,
                                 not args.bgonly)
        if args.bgonly:
            if rank == 0:
                print(dict(bg))
            sys.exit()
        if fused is None:
            struct_pssm = load_motif(args.pfm_struct, args.pseudocount, structure, bg)
            if seq_type == "RNASS":
                table = _combined_hits(seq_file, struct_file, seq_pssm, struct_pssm, seq_hits, args, struct_found)
            else:
                table = _scan_table(struct_file, struct_pssm, structure, args, struct_found)

    t_out = time.perf_counter()
    if rank == 0:
        table.write(sys.stdout)
    STATS.phases["output_s"] += time.perf_counter() - t_out


def _write_stats(dest, seq_type, runtime):
    """One JSON line: phases, sizes, throughput.  `device_GBps` relates the bytes the scan kernels have to read
    at least (1 B per symbol; + 28 B per float32 profile row or 8 B per quantised row altogether) to the time
    their main kernels took."""
    import json
    from . import _lib
    kms = np.zeros(4096, np.float32)
    nrec = np.zeros(1, np.int32)
    _lib.lib.rs_prof_end(kms.ctypes.data, len(kms), nrec.ctypes.data)
    kernel_ms = float(kms[:int(nrec[0])].sum())
    c, ph = STATS.counts, STATS.phases
    positions = c.get("scored_positions", 0)
    form = STATS.notes.get("profile_filter_form")
    per_row = {"q4": 4.0, "q8": 8.0, "f32": 29.0, "shadow": 29.0}.get(form, 0.0)
    dev_bytes = c.get("symbols", 0) * 1.0 + c.get("profile_rows", 0) * per_row
    out = {"mode": seq_type, "world_size": _world_size(), "total_s": runtime,
           "phases_s": {k: round(v, 6) for k, v in sorted(ph.items())},
           "records": c.get("records", 0), "symbols": c.get("symbols", 0), "profile_rows": c.get("profile_rows", 0),
           "scored_positions": positions,
           "gpos_per_s_total": positions / runtime / 1e9 if runtime > 0 else None,
           "gpos_per_s_scan_phase": positions / ph["scan_s"] / 1e9 if ph.get("scan_s") else None,
           "main_kernel_launches": int(nrec[0]), "main_kernel_ms": kernel_ms,
           "gpos_per_s_kernels": positions / (kernel_ms * 1e-3) / 1e9 if kernel_ms > 0 else None,
           "device_GBps": dev_bytes / (kernel_ms * 1e-3) / 1e9 if kernel_ms > 0 else None,
           "h2d_bytes": c.get("h2d_bytes", 0), "candidates": c.get("candidates", 0)}
    out.update({k: v for k, v in STATS.notes.items() if not k.startswith("_")})
    line = json.dumps(out) + "\n"
    if _rank() != 0:
        return
    if dest == "-":
        sys.stderr.write(line)
    else:
        with open(dest, "a") as fh:
            fh.write(line)


if __name__ == "__main__":
    main()
