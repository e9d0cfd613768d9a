"""
ORACLE -- TEST INFRASTRUCTURE ONLY.  Builds oracle/_ref/libcrf_decode_ref.so from oracle/csrc/crf_decode_ref.c (gcc + OpenMP)
and binds it with ctypes.  `oracle/_ref/` is git-ignored (it still travels to the GPU box with the gpurun snapshot).
The reference itself has no C/C++ sources to compile (SURVEY.md section 0), so `_ref/` only ever holds this restatement.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc", "crf_decode_ref.c")
OUT = os.path.join(HERE, "_ref", "libcrf_decode_ref.so")
_lib = None


def build(force=False):
    """Path of an up-to-date library, compiled if needed: into oracle/_ref/, or into a temporary directory where the tree
    cannot be written (bench.py may run from a read-only one)."""
    if not force and os.path.exists(OUT) and os.path.getmtime(OUT) >= os.path.getmtime(SRC):
        return OUT
    out = OUT
    try:
        os.makedirs(os.path.dirname(OUT), exist_ok=True)
    except OSError:
        pass
    if not os.access(os.path.dirname(OUT), os.W_OK):
        out = os.path.join(tempfile.mkdtemp(prefix="crf_decode_ref_"), os.path.basename(OUT))
    subprocess.run(["gcc", "-O2", "-fopenmp", "-shared", "-fPIC", "-o", out, SRC, "-lm"], check=True)
    return out


def load():
    global _lib
    if _lib is None:
        lib = ctypes.CDLL(build())
        lib.crf_decode_ref.restype = ctypes.c_int
        lib.crf_decode_ref.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                       ctypes.c_float, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        _lib = lib
    return _lib


def decode(scores_ntc, state_len, blank_score=2.0, qscale=1.0, qbias=0.0):
    """C counterpart of crf_oracle.decode_native: (moves, sequence, qstring) uint8 [N, T]."""
    x = np.ascontiguousarray(scores_ntc, dtype=np.float32)
    n, t, c = x.shape
    assert c == 4 ** (state_len + 1)
    outs = [np.zeros((n, t), dtype=np.uint8) for _ in range(3)]
    rc = load().crf_decode_ref(x.ctypes.data, n, t, state_len, blank_score, qscale, qbias, *(o.ctypes.data for o in outs))
    if rc != 0:
        raise MemoryError("crf_decode_ref failed")
    return tuple(outs)
