"""ctypes binding of tests/topk_harness.cu, which runs the device top-k of cudasw4_b200/csrc/topk.cuh through the
engine's own dispatch (topk_enqueue). TEST INFRASTRUCTURE: imported only by tests/. The library is compiled on first
use with nvcc into the system's temporary directory (named after a hash of the harness, topk.cuh and the flags), so the
repository tree is never written. Loading it needs no GPU; only run() does."""
from __future__ import annotations

import ctypes
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "topk_harness.cu")
_TOPK = os.path.join(os.path.dirname(_HERE), "cudasw4_b200", "csrc", "topk.cuh")
_FLAGS = ["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-shared"]

REFUSED = -1


class TopkHarness:
    def __init__(self, lib):
        self.lib = lib
        lib.topk_h_shift_for.argtypes = [ctypes.c_longlong]
        lib.topk_h_pass1_blocks.argtypes = [ctypes.c_longlong, ctypes.c_int, ctypes.c_int]
        lib.topk_h_run.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_longlong, ctypes.c_int,
                                   ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        self.max_candidates = lib.topk_h_max_candidates()
        self.large_blocks = lib.topk_h_large_blocks()

    def shift_for(self, max_score: int) -> int:
        return self.lib.topk_h_shift_for(max_score)

    def pass1_blocks(self, n: int, k: int, sm_count: int) -> int:
        return self.lib.topk_h_pass1_blocks(n, k, sm_count)

    def uses_large_path(self, k: int) -> bool:
        return bool(self.lib.topk_h_uses_large_path(k))

    def sm_count(self) -> int:
        n = self.lib.topk_h_sm_count()
        if n <= 0:
            raise RuntimeError("no CUDA device for the top-k harness")
        return n

    def run(self, scores, k: int, max_score: int, sm_count: int, global_ids=None):
        """(scores[k], ids[k], count, kernel launches) from topk_enqueue, or REFUSED when it refuses max_score."""
        scores = np.ascontiguousarray(scores, dtype=np.int32)
        ids = None if global_ids is None else np.ascontiguousarray(global_ids, dtype=np.int32)
        assert 1 <= k <= len(scores) and (ids is None or len(ids) == len(scores))
        out_s = np.empty(k, np.int32)
        out_i = np.empty(k, np.int32)
        count = ctypes.c_int(0)
        launches = ctypes.c_int(0)
        rc = self.lib.topk_h_run(scores.ctypes.data, len(scores), k, max_score, sm_count,
                                 None if ids is None else ids.ctypes.data, out_s.ctypes.data, out_i.ctypes.data,
                                 ctypes.addressof(count), ctypes.addressof(launches))
        if rc == REFUSED:
            return REFUSED
        if rc != 0:
            raise RuntimeError(f"CUDA error {rc} in the top-k harness")
        return out_s, out_i, count.value, launches.value


def load() -> TopkHarness:
    nvcc = shutil.which("nvcc") or ("/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else None)
    if not nvcc:
        raise RuntimeError("nvcc not found: tests/topk_harness.cu cannot be built")
    host = ["-ccbin", "/usr/bin/g++"] if os.path.exists("/usr/bin/g++") else []
    flags = _FLAGS + host
    digest = hashlib.sha1()
    for path in (_SRC, _TOPK):
        with open(path, "rb") as f:
            digest.update(f.read())
    digest.update(" ".join([nvcc] + flags).encode())
    lib = os.path.join(tempfile.gettempdir(), f"sw4_topk_harness_{os.getuid()}_{digest.hexdigest()[:16]}.so")
    if not os.path.exists(lib):
        fd, tmp = tempfile.mkstemp(suffix=".so", dir=tempfile.gettempdir())
        os.close(fd)
        try:
            subprocess.run([nvcc] + flags + ["-o", tmp, _SRC], check=True)
            os.replace(tmp, lib)  # atomic: concurrent test processes never load a half-written library
        finally:
            if os.path.exists(tmp):
                os.remove(tmp)
    return TopkHarness(ctypes.CDLL(lib))
