"""ctypes front end of tests/kmer_correct_oracle.c, the CPU restatement of the correcting walk (DESIGN.md §10).

TEST INFRASTRUCTURE ONLY: imported by tests/test_kmer_correct.py and tools/kmer_bench.py.  The C file is compiled into
a temporary directory on first use, so nothing is written into the tree (which may be read-only).
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "kmer_correct_oracle.c")

_lib = None
_tmp = None   # kept alive for as long as the library is loaded


def lib():
    global _lib, _tmp
    if _lib is None:
        _tmp = tempfile.TemporaryDirectory(prefix="kbbq_kmer_correct_oracle_")
        so = os.path.join(_tmp.name, "libkmer_correct_oracle.so")
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-Wall", "-Wextra", "-std=c11", "-shared",
                               "-o", so, SRC])
        _lib = C.CDLL(so)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def kmer_corrections(seq, L, k=23, min_count=0):
    """Errors found by the correcting walk (DESIGN.md §10) -> (bits u32[ceil(N*L/32)], hist u64[256], t), as
    kmer_errors returns them."""
    seq = np.ascontiguousarray(seq, dtype=np.uint8).ravel()
    N = seq.size // L
    bits = np.zeros((N * L + 31) // 32, np.uint32)
    hist = np.zeros(256, np.uint64)
    t = C.c_int(0)
    st = lib().oracle_kmer_corrections(_p(seq), C.c_int64(N), C.c_int(L), C.c_int(k), C.c_int(min_count), _p(bits),
                                       _p(hist), C.byref(t))
    if st:
        raise RuntimeError("oracle_kmer_corrections: bad argument or out of memory")
    return bits, hist, t.value


def kmer_correct_lookups(seq, L, k=23, min_count=0):
    """The table lookups the kernel of the correcting walk makes on the batch (t >= 2): its valid windows and the
    windows the walks score."""
    seq = np.ascontiguousarray(seq, dtype=np.uint8).ravel()
    n = C.c_uint64(0)
    if lib().oracle_kmer_correct_lookups(_p(seq), C.c_int64(seq.size // L), C.c_int(L), C.c_int(k), C.c_int(min_count),
                                         C.byref(n)):
        raise RuntimeError("oracle_kmer_correct_lookups: bad argument or out of memory")
    return n.value
