"""ctypes front end of tests/kmer_oracle.c, the CPU restatement of the k-mer error rule (DESIGN.md section 10).

TEST INFRASTRUCTURE ONLY: imported by tests/test_kmer.py and tools/kmer_bench.py.  The C file is compiled into a
temporary directory on first use, so nothing is written into the tree (which may be read-only).
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "kmer_oracle.c")

_lib = None
_tmp = None   # kept alive for as long as the library is loaded


def lib():
    global _lib, _tmp
    if _lib is None:
        _tmp = tempfile.TemporaryDirectory(prefix="kbbq_kmer_oracle_")
        so = os.path.join(_tmp.name, "libkmer_oracle.so")
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-Wall", "-Wextra", "-std=c11", "-shared",
                               "-o", so, SRC])
        _lib = C.CDLL(so)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def kmer_errors(seq, L, k=23, min_count=0):
    """Errors from the batch's k-mer counts -> (bits u32[ceil(N*L/32)], hist u64[256], t): the 1-bit map of
    kbbq_host_mismatch_bits, the count histogram and the threshold used."""
    seq = np.ascontiguousarray(seq, dtype=np.uint8).ravel()
    N = seq.size // L
    bits = np.zeros((N * L + 31) // 32, np.uint32)
    hist = np.zeros(256, np.uint64)
    t = C.c_int(0)
    st = lib().oracle_kmer_errors(_p(seq), C.c_int64(N), C.c_int(L), C.c_int(k), C.c_int(min_count), _p(bits),
                                  _p(hist), C.byref(t))
    if st:
        raise RuntimeError("oracle_kmer_errors: bad argument or out of memory")
    return bits, hist, t.value
