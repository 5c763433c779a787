"""ctypes binding of tests/pssm_oracle.cpp, the CPU restatement of scores, coordinates and traceback of PSSM queries.
TEST INFRASTRUCTURE: imported only by tests/. The library is compiled on first use into the system's temporary
directory (named after a hash of the source and flags), so the repository tree is never written."""
from __future__ import annotations

import ctypes
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

from tests.traceback_oracle import Traceback, cigar_of

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "pssm_oracle.cpp")
_FLAGS = ["-std=c++17", "-O3", "-fopenmp", "-fPIC", "-shared"]


def _subjects(subjects):
    if hasattr(subjects, "chars"):
        return (np.ascontiguousarray(subjects.chars, dtype=np.uint8), np.ascontiguousarray(subjects.offsets, dtype=np.uint64),
                np.ascontiguousarray(subjects.lengths, dtype=np.int32))
    seqs = [np.asarray(s, dtype=np.uint8) for s in subjects]
    lengths = np.array([len(s) for s in seqs], dtype=np.int32)
    offsets = np.zeros(len(seqs) + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum(lengths)
    return np.ascontiguousarray(np.concatenate(seqs + [np.zeros(1, np.uint8)]), dtype=np.uint8), offsets, lengths


class PssmOracle:
    def __init__(self, lib):
        self.lib = lib
        lib.sw4p_coords_batch.restype = ctypes.c_long
        lib.sw4p_traceback_batch.restype = ctypes.c_long

    @staticmethod
    def _p(a):
        return a.ctypes.data_as(ctypes.c_void_p)

    def coords(self, pssm, subjects, gop, gex, threads=0) -> np.ndarray:
        """(score, qb, qe, rb, re) of the PSSM query ((qlen, 21) int8) against each subject (code arrays or a
        dbformat.SequenceDB): int32 array of shape (n, 5). Column 0 is the scan's score."""
        P = np.ascontiguousarray(pssm, dtype=np.int8)
        chars, offsets, lengths = _subjects(subjects)
        n = len(lengths)
        out = np.empty((max(n, 1), 5), dtype=np.int32)
        failed = self.lib.sw4p_coords_batch(self._p(P), len(P), self._p(chars), self._p(offsets), self._p(lengths),
                                            ctypes.c_long(n), gop, gex, self._p(out), threads)
        assert failed == 0
        return out[:n]

    def traceback(self, pssm, q, subjects, gop, gex, threads=0, coords=None) -> Traceback:
        """Coordinates, counts and CIGAR of the PSSM query (residue codes q for the identities) against each subject."""
        P = np.ascontiguousarray(pssm, dtype=np.int8)
        q = np.ascontiguousarray(q, dtype=np.uint8)
        assert P.shape == (len(q), 21)
        chars, offsets, lengths = _subjects(subjects)
        n = len(lengths)
        if coords is None:
            coords = self.coords(P, subjects, gop, gex, threads)
        coords = np.ascontiguousarray(coords, dtype=np.int32).reshape(-1, 5)
        room = np.where(coords[:, 0] > 0, (coords[:, 2] - coords[:, 1] + 1) + (coords[:, 4] - coords[:, 3] + 1), 0)
        ops_offsets = np.zeros(n + 1, dtype=np.uint64)
        ops_offsets[1:] = np.cumsum(room)
        ops = np.zeros(max(int(ops_offsets[-1]), 1), dtype=np.uint8)
        counts = np.zeros((max(n, 1), 4), dtype=np.int32)
        failed = self.lib.sw4p_traceback_batch(self._p(P), self._p(q), self._p(chars), self._p(offsets), ctypes.c_long(n),
                                               self._p(coords), gop, gex, self._p(ops), self._p(ops_offsets), self._p(counts),
                                               threads)
        assert failed == 0
        cigars = [cigar_of(ops[int(ops_offsets[k]):int(ops_offsets[k]) + int(counts[k, 0])].tobytes()) for k in range(n)]
        return Traceback(coords[:n].copy(), counts[:n].copy(), cigars)


def load() -> PssmOracle:
    gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    src = open(_SRC, "rb").read()
    tag = hashlib.sha1(src + " ".join([gxx or ""] + _FLAGS).encode()).hexdigest()[:16]
    lib = os.path.join(tempfile.gettempdir(), f"sw4_pssm_oracle_{os.getuid()}_{tag}.so")
    if not os.path.exists(lib):
        if not gxx:
            raise RuntimeError("no host C++ compiler for tests/pssm_oracle.cpp")
        fd, tmp = tempfile.mkstemp(suffix=".so", dir=tempfile.gettempdir())
        os.close(fd)
        try:
            subprocess.run([gxx] + _FLAGS + ["-o", tmp, _SRC], check=True)
            os.replace(tmp, lib)  # atomic: concurrent test processes never load a half-written library
        finally:
            if os.path.exists(tmp):
                os.remove(tmp)
    return PssmOracle(ctypes.CDLL(lib))
