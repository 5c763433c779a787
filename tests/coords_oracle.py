"""ctypes binding of tests/coords_oracle.cpp, the CPU restatement of the alignment coordinates. TEST INFRASTRUCTURE:
imported only by tests/. The library is compiled on first use into the system's temporary directory (named after a
hash of the source and flags), so the repository tree is never written."""
from __future__ import annotations

import ctypes
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "coords_oracle.cpp")
_FLAGS = ["-std=c++17", "-O3", "-fopenmp", "-fPIC", "-shared"]


class CoordsOracle:
    def __init__(self, lib, matrix_of):
        self.lib = lib
        self.matrix_of = matrix_of  # blosum -> 21x21 int8 table (the oracle's)
        lib.sw4c_gotoh_coords_batch.restype = ctypes.c_long

    @staticmethod
    def _p(a):
        return a.ctypes.data_as(ctypes.c_void_p)

    def coords(self, blosum, q, subjects, gop, gex, threads=0) -> np.ndarray:
        """(score, qb, qe, rb, re) of q against each subject (a list of code arrays, or a dbformat.SequenceDB): int32
        array of shape (n, 5), as sw4_alignment_coordinates defines them."""
        q = np.ascontiguousarray(q, dtype=np.uint8)
        if hasattr(subjects, "chars"):
            chars = np.ascontiguousarray(subjects.chars, dtype=np.uint8)
            offsets = np.ascontiguousarray(subjects.offsets, dtype=np.uint64)
            lengths = np.ascontiguousarray(subjects.lengths, dtype=np.int32)
        else:
            seqs = [np.asarray(s, dtype=np.uint8) for s in subjects]
            lengths = np.array([len(s) for s in seqs], dtype=np.int32)
            offsets = np.zeros(len(seqs) + 1, dtype=np.uint64)
            offsets[1:] = np.cumsum(lengths)
            chars = np.ascontiguousarray(np.concatenate(seqs + [np.zeros(1, np.uint8)]), dtype=np.uint8)
        matrix = np.ascontiguousarray(self.matrix_of(blosum), dtype=np.int8).reshape(441)
        n = len(lengths)
        out = np.empty((max(n, 1), 5), dtype=np.int32)
        failed = self.lib.sw4c_gotoh_coords_batch(self._p(matrix), self._p(q), len(q), self._p(chars), self._p(offsets),
                                                  self._p(lengths), ctypes.c_long(n), gop, gex, self._p(out), threads)
        assert failed == 0
        return out[:n]


def load(oracle) -> CoordsOracle:
    """`oracle`: the tests.oracle_lib.Oracle whose substitution tables are used."""
    gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    src = open(_SRC, "rb").read()
    tag = hashlib.sha1(src + " ".join([gxx or ""] + _FLAGS).encode()).hexdigest()[:16]
    lib = os.path.join(tempfile.gettempdir(), f"sw4_coords_oracle_{os.getuid()}_{tag}.so")
    if not os.path.exists(lib):
        if not gxx:
            raise RuntimeError("no host C++ compiler for tests/coords_oracle.cpp")
        fd, tmp = tempfile.mkstemp(suffix=".so", dir=tempfile.gettempdir())
        os.close(fd)
        try:
            subprocess.run([gxx] + _FLAGS + ["-o", tmp, _SRC], check=True)
            os.replace(tmp, lib)  # atomic: concurrent test processes never load a half-written library
        finally:
            if os.path.exists(tmp):
                os.remove(tmp)
    return CoordsOracle(ctypes.CDLL(lib), oracle.matrix)
