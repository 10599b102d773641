"""PFM helpers with the reference's names and file formats (rnascan/pfmutil.py).

A PFM here is ``{letter: [value per position]}``.  The tab-separated layout written by
``format_pfm`` -- header ``PO`` + the letters in sorted order, then one ``pos<TAB>values``
row per position with values printed by ``str(float)`` -- is also the on-disk format of
run_folding's averaged structure profiles (``structure.<id>.txt``, pfmutil.py:61-80), i.e.
the input of the averaged-profile scan.

``pwm_scan_fwd`` (pfmutil.py:205-221) runs on the GPU.
"""
import csv
from itertools import groupby
from math import log

RNA_ALPHABET = ["A", "C", "G", "U"]
FULL_STRUCT_ALPHABET = ["B", "E", "H", "L", "M", "R", "T"]
REDUCED_STRUCT_ALPHABET = ["E", "H", "I", "M", "P"]


def _iupac_table():
    groups = {"A": "A", "C": "C", "G": "G", "U": "U", "R": "AG", "Y": "CU", "S": "CG", "W": "AU",
              "K": "GU", "M": "AC", "B": "CGU", "D": "AGU", "H": "ACU", "V": "ACG", "N": "ACGU"}
    table = {}
    for code, members in groups.items():
        share = 1.0 / len(members)
        table[code] = {base: (share if base in members else 0.0) for base in RNA_ALPHABET}
    return table


IUPAC_to_pfm = _iupac_table()


def _letters_and_length(pfm):
    letters = sorted(pfm.keys())
    return letters, len(pfm[letters[0]])


def read_pfm(pfmfile):
    """Tab-separated PFM: header row names the letters (first cell ignored); the first cell
    of every following row is the position and is dropped."""
    with open(pfmfile) as handle:
        rows = csv.reader(handle, delimiter="\t")
        letters = next(rows)[1:]
        pfm = {letter: [] for letter in letters}
        for row in rows:
            for letter, cell in zip(letters, row[1:]):
                pfm[letter].append(float(cell))
    return pfm


def _format_rows(pfm, letters, length):
    lines = []
    for pos in range(length):
        if pfm[letters[0]][pos] is None:
            break
        lines.append(str(pos) + "".join("\t" + str(pfm[letter][pos]) for letter in letters) + "\n")
    return lines


def format_pfm(pfm):
    letters, length = _letters_and_length(pfm)
    head = "PO" + "".join("\t" + letter for letter in letters) + "\n"
    return head + "".join(_format_rows(pfm, letters, length))


def write_pfm(pfm, pfmoutfile):
    with open(pfmoutfile, "w") as handle:
        handle.write(format_pfm(pfm))


def multi_pfm_iter(filename):
    """(id, pfm) per block of a multi-PFM file: two '#' lines (``#id`` then ``#PO<TAB>letters``)
    followed by the rows.  As in the reference the SAME dict object is re-filled for every
    block, so copy it if you keep it."""
    identifier, letters, pfm = "", [], {}
    with open(filename) as handle:
        for is_header, block in groupby(handle, lambda line: line[0] == "#"):
            if is_header:
                header = [line.rstrip()[1:] for line in block]
                identifier = header[0]
                letters = header[1].split("\t")[1:]
            else:
                for letter in letters:
                    pfm[letter] = []
                for line in block:
                    cells = line.rstrip().split("\t")
                    for letter, cell in zip(letters, cells[1:]):
                        pfm[letter].append(float(cell))
                yield identifier, pfm


def write_multi_pfm(idlist, pfmlist, outfile):
    with open(outfile, "w") as handle:
        for identifier, pfm in zip(idlist, pfmlist):
            letters, length = _letters_and_length(pfm)
            handle.write("#" + identifier + "\n")
            handle.write("#PO" + "".join("\t" + letter for letter in letters) + "\n")
            handle.write("".join(_format_rows(pfm, letters, length)))
            handle.write("\n")


def norm_pfm(pfm):
    letters, length = _letters_and_length(pfm)
    out = {letter: [None] * length for letter in letters}
    for pos in range(length):
        total = 0
        for letter in letters:
            total = total + pfm[letter][pos]
        for letter in letters:
            out[letter][pos] = pfm[letter][pos] / float(total)
    return out


def is_normalized(pfm, epsilon=1e-6):
    letters, length = _letters_and_length(pfm)
    for pos in range(length):
        total = 0
        for letter in letters:
            total = total + pfm[letter][pos]
        if abs(1 - total) > epsilon:
            return False
    return True


def pfm_from_IUPAC(iupac):
    pfm = {base: [0.0] * len(iupac) for base in RNA_ALPHABET}
    for i, code in enumerate(iupac):
        for base in RNA_ALPHABET:
            pfm[base][i] = IUPAC_to_pfm[code][base]
    return pfm


def pfm_from_string(string, alphabet):
    pfm = {base: [0.0] * len(string) for base in alphabet}
    for i, base in enumerate(string):
        if base not in alphabet:
            raise Exception("char " + base + " not in alphabet " + str(alphabet))
        pfm[base][i] = 1.0
    return pfm


def pfm_to_pwm(pfm, num_sites):
    """log2 odds against a uniform background with the (p*n + 1/A)/(n + 1) small-sample
    correction (pfmutil.py:187-203)."""
    letters, length = _letters_and_length(pfm)
    uniform = 1.0 / len(letters)
    pwm = {letter: [None] * length for letter in letters}
    for pos in range(length):
        for letter in letters:
            corrected = (float(pfm[letter][pos]) * num_sites + uniform) / (num_sites + 1)
            pwm[letter][pos] = log(corrected / uniform, 2)
    return pwm


def pwm_scan_fwd(pwm, seq):
    """Forward-strand score of every window: sum_j pwm[seq[i+j]][j] as Python floats in j
    order (pfmutil.py:205-221).  Case-SENSITIVE; a letter that is not a key of `pwm`
    raises KeyError, as the reference's dict lookup does.  Scored on the GPU (sequential
    fp64 adds, so the values are bit-identical to the Python loop)."""
    import numpy as np
    from . import device

    letters, length = _letters_and_length(pwm)
    seq = str(seq)
    if len(seq) - length + 1 <= 0:
        return []
    if len(letters) > device.MAX_ALPHA_LETTERS or any(len(letter) != 1 or ord(letter) > 255 for letter in letters):
        raise NotImplementedError("GPU scoring supports alphabets of up to %d single-byte letters"
                                  % device.MAX_ALPHA_LETTERS)
    lut = np.full(256, device._lib.RS_ALPHA_OTHER, np.uint8)      # case-sensitive: each key has its own index
    for k, letter in enumerate(letters):
        lut[ord(letter)] = k
    raw = np.frombuffer(seq.encode("latin-1", "replace"), np.uint8)
    codes = lut[raw]
    bad = np.nonzero(codes == device._lib.RS_ALPHA_OTHER)[0]
    if len(bad):
        raise KeyError(seq[int(bad[0])])
    stream = device.SymbolStream(codes)
    if len(letters) <= 7:                                         # the structure kernels, table padded to 7 columns
        table = np.zeros((length, 7), np.float64)
        for k, letter in enumerate(letters):
            table[:, k] = pwm[letter]
        scores = device.dense_struct(stream, table).cpu().numpy()
    else:
        table = np.array([pwm[letter] for letter in letters], np.float64).T
        scores = device.dense_alpha(stream, table).cpu().numpy()
    return [float(v) for v in scores]


def reduce_pfm_alphabet(pfm):
    """BEHLMRT -> EHIMP: paired = L + R, internal = B + T (pfmutil.py:223-240)."""
    letters, length = _letters_and_length(pfm)
    assert letters == FULL_STRUCT_ALPHABET
    reduced = {letter: [None] * length for letter in REDUCED_STRUCT_ALPHABET}
    for letter in ("E", "H", "M"):
        reduced[letter] = pfm[letter]
    reduced["P"] = [sum(pair) for pair in zip(pfm["L"], pfm["R"])]
    reduced["I"] = [sum(pair) for pair in zip(pfm["B"], pfm["T"])]
    return reduced
