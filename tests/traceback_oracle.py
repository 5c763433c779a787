"""ctypes binding of tests/traceback_oracle.cpp, the CPU restatement of the alignment traceback. TEST INFRASTRUCTURE:
imported only by tests/. The library is compiled on first use into the system's temporary directory (named after a
hash of the source and flags), so the repository tree is never written. The coordinates come from tests/coords_oracle."""
from __future__ import annotations

import ctypes
import hashlib
import os
import shutil
import subprocess
import tempfile
from dataclasses import dataclass

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "traceback_oracle.cpp")
_FLAGS = ["-std=c++17", "-O3", "-fopenmp", "-fPIC", "-shared"]


def cigar_of(ops: bytes) -> str:
    """Run-length encoding of a column string such as b"==X=ID" -> "2=1X1=1I1D"."""
    if not ops:
        return ""
    a = np.frombuffer(ops, dtype=np.uint8)
    starts = np.concatenate([[0], np.nonzero(a[1:] != a[:-1])[0] + 1])
    runs = np.diff(np.concatenate([starts, [len(a)]]))
    return "".join(f"{int(r)}{chr(a[s])}" for s, r in zip(starts, runs))


@dataclass
class Traceback:
    coordinates: np.ndarray  # (n, 5) int32, as coords_oracle
    counts: np.ndarray       # (n, 4) int32: length, identities, positives, gaps
    cigars: list             # str per pair


class TracebackOracle:
    def __init__(self, lib, coords_oracle):
        self.lib = lib
        self.coords_oracle = coords_oracle
        lib.sw4t_traceback_batch.restype = ctypes.c_long

    @staticmethod
    def _p(a):
        return a.ctypes.data_as(ctypes.c_void_p)

    def traceback(self, blosum, q, subjects, gop, gex, threads=0, coords=None) -> Traceback:
        """Coordinates, counts and CIGAR of q against each subject (a list of code arrays, or a dbformat.SequenceDB),
        as sw4_alignment_traceback defines them. `coords` (from coords_oracle) may be passed when already known."""
        q = np.ascontiguousarray(q, dtype=np.uint8)
        if hasattr(subjects, "chars"):
            chars = np.ascontiguousarray(subjects.chars, dtype=np.uint8)
            offsets = np.ascontiguousarray(subjects.offsets, dtype=np.uint64)
            n = len(subjects.lengths)
        else:
            seqs = [np.asarray(s, dtype=np.uint8) for s in subjects]
            offsets = np.zeros(len(seqs) + 1, dtype=np.uint64)
            offsets[1:] = np.cumsum([len(s) for s in seqs])
            chars = np.ascontiguousarray(np.concatenate(seqs + [np.zeros(1, np.uint8)]), dtype=np.uint8)
            n = len(seqs)
        if coords is None:
            coords = self.coords_oracle.coords(blosum, q, subjects, gop, gex, threads)
        coords = np.ascontiguousarray(coords, dtype=np.int32).reshape(-1, 5)
        room = np.where(coords[:, 0] > 0, (coords[:, 2] - coords[:, 1] + 1) + (coords[:, 4] - coords[:, 3] + 1), 0)
        ops_offsets = np.zeros(n + 1, dtype=np.uint64)
        ops_offsets[1:] = np.cumsum(room)
        ops = np.zeros(max(int(ops_offsets[-1]), 1), dtype=np.uint8)
        counts = np.zeros((max(n, 1), 4), dtype=np.int32)
        matrix = np.ascontiguousarray(self.coords_oracle.matrix_of(blosum), dtype=np.int8).reshape(441)
        failed = self.lib.sw4t_traceback_batch(self._p(matrix), self._p(q), self._p(chars), self._p(offsets), ctypes.c_long(n),
                                               self._p(coords), gop, gex, self._p(ops), self._p(ops_offsets), self._p(counts),
                                               threads)
        assert failed == 0
        cigars = [cigar_of(ops[int(ops_offsets[k]):int(ops_offsets[k]) + int(counts[k, 0])].tobytes()) for k in range(n)]
        return Traceback(coords[:n].copy(), counts[:n].copy(), cigars)


def load(coords_oracle) -> TracebackOracle:
    """`coords_oracle`: the tests.coords_oracle.CoordsOracle that provides the coordinates and substitution tables."""
    gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    src = open(_SRC, "rb").read()
    tag = hashlib.sha1(src + " ".join([gxx or ""] + _FLAGS).encode()).hexdigest()[:16]
    lib = os.path.join(tempfile.gettempdir(), f"sw4_traceback_oracle_{os.getuid()}_{tag}.so")
    if not os.path.exists(lib):
        if not gxx:
            raise RuntimeError("no host C++ compiler for tests/traceback_oracle.cpp")
        fd, tmp = tempfile.mkstemp(suffix=".so", dir=tempfile.gettempdir())
        os.close(fd)
        try:
            subprocess.run([gxx] + _FLAGS + ["-o", tmp, _SRC], check=True)
            os.replace(tmp, lib)  # atomic: concurrent test processes never load a half-written library
        finally:
            if os.path.exists(tmp):
                os.remove(tmp)
    return TracebackOracle(ctypes.CDLL(lib), coords_oracle)
