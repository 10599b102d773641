"""Same module path and class as the reference (rnascan/BioAddons/motifs/matrix.py:14-81),
without the Biopython base class and with the scoring loops on the GPU.

``ExtendedPositionSpecificScoringMatrix`` is a dict ``{letter: [log-odds per position]}``
in ``alphabet.letters`` order with ``.alphabet``, ``.length``, ``.consensus``,
``.calculate()`` and ``.search()`` -- the members rnascan uses from Biopython's
``PositionSpecificScoringMatrix``.
"""
import numpy as np

from ... import device
from ...seq import Seq, is_nucleotide_alphabet
from . import _pwm


class ExtendedPositionSpecificScoringMatrix(dict):

    _pwm = _pwm

    def __init__(self, alphabet, values):
        dict.__init__(self)
        self.length = None
        for letter in alphabet.letters:
            column = list(values[letter])
            if self.length is None:
                self.length = len(column)
            elif self.length != len(column):
                raise Exception("data has inconsistent lengths")
            self[letter] = column
        self.alphabet = alphabet
        self._letters = sorted(self.alphabet.letters)

    # ---- tables in device column order ------------------------------------------------
    def table(self, columns):
        """(length, len(columns)) float64 array, one column per letter of `columns`."""
        return np.array([self[letter] for letter in columns], dtype=np.float64).T.copy()

    @property
    def consensus(self):
        sequence = ""
        for i in range(self.length):
            maximum = float("-inf")
            best = None
            for letter in self.alphabet.letters:
                value = self[letter][i]
                if value > maximum:
                    maximum, best = value, letter
            if best is None:                # every entry NaN/-inf: Biopython keeps going
                best = sequence[-1] if sequence else self.alphabet.letters[0]
            sequence += best
        return Seq(sequence, self.alphabet)

    # ---- scoring ----------------------------------------------------------------------
    def _is_structure(self):
        return sorted(self.alphabet.letters) == sorted(device.CHANNELS)

    def _py_calculate(self, sequence, m, n):
        """Generic-alphabet scores as a list of Python floats (matrix.py:25-43), on the GPU:
        the structure-context kernels for BEHLMRT, the alphabet kernels for any other
        alphabet device.AlphaKind accepts (NotImplementedError otherwise)."""
        if n - m + 1 <= 0:
            return []
        if self._is_structure():
            stream = device.SymbolStream.from_texts([sequence], "struct")
            out = device.dense_struct(stream, self.table(device.CHANNELS)).cpu().numpy()
        else:
            kind = device.AlphaKind(self.alphabet.letters)
            stream = device.SymbolStream.from_texts([sequence], kind)
            out = device.dense_alpha(stream, self.table(kind.letters)).cpu().numpy()
        return [float(v) for v in out[:n - m + 1]]

    def _calculate(self, sequence, m, n):
        if not is_nucleotide_alphabet(self.alphabet):
            return self._py_calculate(sequence, m, n)
        letters = "".join(sorted(self.alphabet.letters))
        logodds = [[self[letter][i] for letter in letters] for i in range(m)]
        return self._pwm.calculate(sequence, np.array(logodds, dtype=np.float64).reshape(m, 4))

    def calculate(self, sequence):
        """Scores of every window; a scalar when there is exactly one (matrix.py:68-81)."""
        sequence = str(sequence)
        m = self.length
        n = len(sequence)
        scores = self._calculate(sequence, m, n)
        if len(scores) == 1:
            return scores[0]
        return scores

    def search(self, sequence, threshold=0.0, both=False):
        """(position, score) for every window whose score is > threshold, in order
        (Biopython <= 1.77 ``search`` as called at rnascan.py:263; NaN and -inf windows
        are never reported).  Only the forward strand is supported."""
        if both:
            raise ValueError("reverse-complement search is undefined for this alphabet; "
                             "call search(..., both=False) as rnascan does")
        text = str(sequence)
        if len(text) < self.length:
            return
        if is_nucleotide_alphabet(self.alphabet):
            stream = device.SymbolStream.from_texts([text], "rna")
            pos, score = device.scan_seq(stream, self.table(device.RNA_COLUMNS), threshold)
            for p, s in zip(pos.tolist(), score):
                yield (p, s)                       # s is numpy.float32, as in the reference
        else:
            if self._is_structure():
                stream = device.SymbolStream.from_texts([text], "struct")
                pos, score = device.scan_struct_onehot(stream, self.table(device.CHANNELS), threshold)
            else:
                kind = device.AlphaKind(self.alphabet.letters)
                stream = device.SymbolStream.from_texts([text], kind)
                pos, score = device.scan_alpha(stream, self.table(kind.letters), threshold)
            for p, s in zip(pos.tolist(), score.tolist()):
                yield (p, s)                       # Python float
