"""ctypes binding of libkbbq_b200.so (include/kbbq_b200.h).

This is the only door between the Python API mirror and the CUDA kernels.  There is no CPU
fallback: if the shared library is missing, or a compute entry point is called without a CUDA
device, the call raises -- it never silently computes on the host.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libkbbq_b200.so")

NQ = 43
FLAG_QUAL_RANGE, FLAG_BAD_BASE, FLAG_RG_RANGE, FLAG_SEGMENTS = 1, 2, 4, 8
FLAG_KMER_FULL = 16
KMER_BOUNDARIES, KMER_CORRECT = 0, 1   # k-mer error rules (include/kbbq_b200.h)
APPLY_BASES_CHECKED = 0x10   # kbbq_apply path flag: skip the base check (include/kbbq_b200.h)
E_DATA = -4
E_UNSUPPORTED = -12

_lib = None

# name -> (restype, argtypes); must list every symbol include/kbbq_b200.h declares
_vp, _i, _i64, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_size_t
SIGNATURES = {
    "kbbq_abi_version": (_i, []),
    "kbbq_strerror": (C.c_char_p, [_i]),
    "kbbq_last_cuda_error": (C.c_char_p, []),
    "kbbq_pos_table_elems": (_i64, [_i, _i]),
    "kbbq_din_table_elems": (_i64, [_i]),
    "kbbq_workspace_bytes": (_i, [_i64, _i, _i, C.POINTER(_sz)]),
    "kbbq_build": (_i, [_vp] * 5 + [_i64, _i, _i, _i] + [_vp] * 4 + [_vp, _sz, _vp, _i, _vp]),
    "kbbq_marginals": (_i, [_vp, _vp, _i, _i] + [_vp] * 5 + [_vp]),
    "kbbq_delta_q": (_i, [_vp, _vp, _vp, _i64, _vp, _vp]),
    "kbbq_get_delta_qs": (_i, [_vp] * 9 + [_i, _i, _i, _i] + [_vp] * 4 + [_vp]),
    "kbbq_apply": (_i, [_vp] * 4 + [_i64, _i, _i, _i] + [_vp] * 5 + [_i, _i, _vp, _vp, _sz, _vp, _i, _vp]),
    "kbbq_recalibrate_host": (_i, [_vp] * 5 + [_i64, _i, _i, _i] + [_vp] * 3 + [C.POINTER(_i), _i]),
    "kbbq_recalibrate_host_multi": (_i, [_vp] * 5 + [_i64, _i, _i, _i] + [_vp] * 3 + [C.POINTER(_i), C.POINTER(_i), _i]),
    "kbbq_recalibrate_fastq": (_i, [C.c_char_p, C.c_char_p, _i, _i, _i, _i, _i, C.POINTER(_i64), C.POINTER(_i), C.POINTER(_i)]),
    "kbbq_host_release": (_i, [_i]),
    "kbbq_session_create": (_i, [_i, _i, _i, _i, _i64, _i64, _i, C.POINTER(_vp)]),
    "kbbq_session_destroy": (None, [_vp]),
    "kbbq_session_chunk_reads": (_i64, [_vp]),
    "kbbq_session_reset": (_i, [_vp]),
    "kbbq_session_build_chunk": (_i, [_vp] * 6 + [_i64, _i]),
    "kbbq_session_build_range": (_i, [_vp] * 6 + [_i64]),
    "kbbq_session_tables": (_i, [_vp, _vp]),
    "kbbq_session_set_tables": (_i, [_vp, _vp]),
    "kbbq_session_tables_dev": (_i, [_vp, C.POINTER(_vp), C.POINTER(_i64), C.POINTER(_vp)]),
    "kbbq_session_model": (_i, [_vp, _vp]),
    "kbbq_session_apply_resident": (_i, [_vp, _i64, _vp]),
    "kbbq_session_apply_chunk": (_i, [_vp] * 5 + [_i64, _vp]),
    "kbbq_session_flush": (_i, [_vp]),
    "kbbq_session_sync": (_i, [_vp, C.POINTER(_i)]),
    "kbbq_session_traffic": (_i, [_vp, C.POINTER(_i64), C.POINTER(_i64)]),
    "kbbq_build_host": (_i, [_vp] * 5 + [_i64, _i, _i, _i] + [_vp] * 4 + [C.POINTER(_i), _i]),
    "kbbq_apply_host": (_i, [_vp] * 4 + [_i64, _i, _i, _i] + [_vp] * 5 + [_i, _i, _vp, C.POINTER(_i), _i]),
    "kbbq_get_delta_qs_host": (_i, [_vp] * 9 + [_i, _i, _i, _i] + [_vp] * 4 + [_i]),
    "kbbq_delta_q_host": (_i, [_vp, _vp, _vp, _i64, _vp, _i]),
    "kbbq_posterior_q_real": (_i, [_vp, _vp, _vp, _i64, _vp, _vp]),
    "kbbq_posterior_q_real_host": (_i, [_vp, _vp, _vp, _i64, _vp, _i]),
    "kbbq_calibration_counts": (_i, [_vp] * 5 + [_i64, _vp, _vp, _vp]),
    "kbbq_calibration_counts_host": (_i, [_vp] * 5 + [_i64, _vp, _vp, _i]),
    "kbbq_bam_workspace_bytes": (_i, [_i64, _i, _i, C.POINTER(_sz)]),
    "kbbq_build_bam": (_i, [_vp] * 8 + [_i64, _i, _i, _i] + [_vp] * 4 + [_vp, _sz, _vp, _vp]),
    "kbbq_apply_bam": (_i, [_vp] * 4 + [_i64, _i, _i, _i] + [_vp] * 5 + [_i, _i, _vp, _vp, _sz, _vp, _vp]),
    "kbbq_build_bam_host": (_i, [_vp] * 8 + [_i64, _i, _i, _i] + [_vp] * 4 + [_vp, _i]),
    "kbbq_apply_bam_host": (_i, [_vp] * 4 + [_i64, _i, _i, _i] + [_vp] * 5 + [_i, _i, _vp, _vp, _i]),
    "kbbq_marginals_host": (_i, [_vp, _vp, _i, _i] + [_vp] * 5 + [_i]),
    "kbbq_synth_reads": (_i, [C.c_uint64, _i64, _i64, _i, _i] + [_vp] * 5 + [_vp]),
    "kbbq_launch_count": (_i64, []),
    "kbbq_fastq_open": (_i, [C.c_char_p, _i, C.POINTER(_vp)]),
    "kbbq_fastq_open_mem": (_i, [_vp, _sz, _i, C.POINTER(_vp)]),
    "kbbq_fastq_close": (None, [_vp]),
    "kbbq_fastq_num_reads": (_i64, [_vp]),
    "kbbq_fastq_read_len": (_i, [_vp]),
    "kbbq_fastq_pack": (_i, [_vp, _i64, _i64, _vp, _vp, _i]),
    "kbbq_fastq_name": (_i, [_vp, _i64, C.POINTER(C.c_char_p), C.POINTER(_i)]),
    "kbbq_fastq_infer": (_i, [_vp, _i, _vp, _vp, C.POINTER(_i), _i]),
    "kbbq_fastq_rg_key": (_i, [_vp, _i, C.POINTER(C.c_char_p), C.POINTER(_i)]),
    "kbbq_fastq_check_names": (_i, [_vp, _vp, _i64, _i, C.POINTER(_i64)]),
    "kbbq_fastq_write": (_i, [_i, _vp, _i64, _i64, _vp, _i]),
    "kbbq_fastq_format_size": (_i, [_vp, _i64, _i64, _i, C.POINTER(_i64)]),
    "kbbq_fastq_format": (_i, [_vp, _i64, _i64, _vp, _vp, _i64, _i]),
    "kbbq_host_mismatch_bits": (_i, [_vp, _vp, _i64, _vp, _i]),
    "kbbq_expand_mismatch_bits": (_i, [_vp, _vp, _i64, _vp, _vp]),
    "kbbq_host_last_traffic": (_i, [_i, C.POINTER(_i64), C.POINTER(_i64)]),
    "kbbq_host_pack_mode": (_i, [_i]),
    "kbbq_host_pack_nibbles": (_i, [_vp, _vp, _i64, _vp, _i, _vp]),
    "kbbq_expand_nibbles": (_i, [_vp, _i64, _vp, _vp, _vp]),
    "kbbq_plan_info": (_i, [_i, _i, _i, _i, _i, C.POINTER(_i)]),
    "kbbq_segment_rows_bound": (_i64, [_i64, _i]),
    "kbbq_segment_table_elems": (_i64, [_i]),
    "kbbq_segmented_supported": (_i, [_i, _i, _i]),
    "kbbq_segment_plan": (_i, [_vp, _vp, _i64, _i, _vp, _vp, _vp, _vp]),
    "kbbq_segment_rows": (_i, [_vp, _vp, _i64, _i, _vp, _vp]),
    "kbbq_segment_pad": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp]),
    "kbbq_unsegment_rows": (_i, [_vp, _vp, _i64, _i, _i64, _vp, _vp]),
    "kbbq_build_segmented": (_i, [_vp] * 4 + [_i64, _i, _i, _i] + [_vp] * 4 + [_vp, _sz, _vp, _vp]),
    "kbbq_apply_segmented": (_i, [_vp] * 3 + [_i64, _i, _i, _i] + [_vp] * 5 + [_i, _i, _vp, _vp, _sz, _vp, _vp]),
    "kbbq_apply_segmented_flags": (_i, [_vp] * 3 + [_i64, _i, _i, _i] + [_vp] * 5 + [_i, _i, _vp, _vp, _sz, _vp, _i, _vp]),
    "kbbq_kmer_table_bytes": (_i, [_i64, _i, _i, C.POINTER(C.c_uint64), C.POINTER(_sz)]),
    "kbbq_kmer_clear": (_i, [_vp, C.c_uint64, _vp]),
    "kbbq_kmer_count": (_i, [_vp, _i64, _i, _i, _vp, C.c_uint64, _vp, _vp]),
    "kbbq_kmer_histogram": (_i, [_vp, C.c_uint64, _vp, _vp]),
    "kbbq_kmer_flag": (_i, [_vp, _i64, _i, _i, _vp, C.c_uint64, _i, _vp, _vp, _vp]),
    "kbbq_kmer_min_count": (_i, [_vp]),
    "kbbq_kmer_errors_host": (_i, [_vp, _i64, _i, _i, _i, _vp, _vp, C.POINTER(_i), _i]),
    "kbbq_recalibrate_kmer_host": (_i, [_vp] * 4 + [_i64, _i, _i, _i, _i, _i] + [_vp] * 3 + [C.POINTER(_i), C.POINTER(_i), _i]),
    "kbbq_kmer_stream_plan": (_i, [C.c_uint64, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "kbbq_kmer_sieve": (_i, [_vp, _i64, _i, _i, _vp, C.c_uint64, _vp, C.c_uint64, _vp, _vp]),
    "kbbq_kmer_count_present": (_i, [_vp, _i64, _i, _i, _vp, C.c_uint64, _vp, _vp, _vp]),
    "kbbq_kmer_histogram_sieved": (_i, [_vp, C.c_uint64, _vp, _vp, _vp]),
    "kbbq_kmer_flag_sieved": (_i, [_vp, _i64, _i, _i, _vp, C.c_uint64, _i, _vp, _vp, _vp]),
    "kbbq_session_kmer_begin": (_i, [_vp, _i, _i64, C.c_uint64, C.c_uint64]),
    "kbbq_session_kmer_sieve": (_i, [_vp, _vp, _i64]),
    "kbbq_session_kmer_count": (_i, [_vp, _vp, _i64]),
    "kbbq_session_kmer_threshold": (_i, [_vp, _i, _vp, C.POINTER(_i)]),
    "kbbq_session_build_chunk_kmer": (_i, [_vp] * 5 + [_i64]),
    "kbbq_session_kmer_sizes": (_i, [_vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "kbbq_kmer_correct": (_i, [_vp, _i64, _i, _i, _vp, C.c_uint64, _i, _vp, _vp, _vp]),
    "kbbq_kmer_errors_rule_host": (_i, [_vp, _i64, _i, _i, _i, _i, _vp, _vp, C.POINTER(_i), _i]),
    "kbbq_recalibrate_kmer_rule_host": (_i, [_vp] * 4 + [_i64, _i, _i, _i, _i, _i, _i] + [_vp] * 3 + [C.POINTER(_i), C.POINTER(_i), _i]),
    "kbbq_session_kmer_rule": (_i, [_vp, _i]),
}


class KbbqNativeError(RuntimeError):
    """The CUDA library is missing, or a CUDA / argument error came back from it."""


class DoesNotFit(ValueError):
    """The reads and the k-mer table of a single-batch call do not fit the GPU's free memory (KBBQ_E_UNSUPPORTED):
    the streamed path (Session.kmer_*) handles such inputs."""


def lib():
    """Load libkbbq_b200.so (once). Raises if it has not been built -- there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise KbbqNativeError(
                "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or make -C kbbq-py_b200/csrc). kbbq_b200 has no CPU fallback." % LIB_PATH)
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc, status=0):
    if rc == 0:
        return
    if rc == E_DATA:
        raise_for_status(status)
    L = lib()
    msg = L.kbbq_strerror(rc).decode()
    if rc == -2:
        msg += ": " + L.kbbq_last_cuda_error().decode()
    raise KbbqNativeError("libkbbq_b200: %s (%d)" % (msg, rc))


def raise_for_status(status):
    """Map the device status word onto the exceptions the reference raises for the same input."""
    if status & FLAG_QUAL_RANGE:
        # kbbq/recalibrate.py:115-119: a quality > 42 indexes past the 43-row tables
        raise IndexError("quality score out of range for the covariate tables (max 42)")
    if status & FLAG_BAD_BASE:
        # kbbq/compare_reads.py:224: Dinucleotide.vecget returns None for a non-ACGT dinucleotide
        raise TypeError("sequence contains a base outside A, C, G, T, N")
    if status & FLAG_RG_RANGE:
        raise IndexError("read group index out of range")
    if status & FLAG_SEGMENTS:
        raise ValueError("malformed span table of a segmented batch")
    if status & FLAG_KMER_FULL:
        raise MemoryError("the k-mer table is full")


def ptr(a):
    """Host pointer of a C-contiguous numpy array (None -> NULL)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


def u8(a):
    return np.ascontiguousarray(a, dtype=np.uint8)


def i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def _opt(a, dtype=np.uint8):
    """An optional array argument: None stays None (NULL), anything else becomes a contiguous array of `dtype`."""
    return None if a is None else np.ascontiguousarray(a, dtype=dtype)


def plan_info(L, R=1, minscore=6, arrays=3, max_smem=0):
    """Shared-memory plan of the build (arrays=3) / apply (arrays=2) kernel, or None for the generic path."""
    out = (C.c_int * 10)()
    if lib().kbbq_plan_info(L, R, minscore, arrays, max_smem, out) != 0:
        return None
    keys = ("G", "lanes", "ng", "threads", "nprod", "kps", "stages", "drep", "smem", "table_bytes")
    return dict(zip(keys, out))


DEVICE = int(os.environ.get("KBBQ_DEVICE", os.environ.get("LOCAL_RANK", "0")))


def _dev(device):
    """The device of a call: `device`, or DEVICE when it is None."""
    return DEVICE if device is None else int(device)


# ---- host-buffer wrappers (numpy in, numpy out) ---------------------------------------------

def build_host(seq, qual, corr, rg, second, L, R, minscore=6, device=None):
    seq, qual, corr = u8(seq).ravel(), u8(qual).ravel(), u8(corr).ravel()
    N = seq.size // L
    assert seq.size == qual.size == corr.size == N * L
    rg = _opt(rg, np.uint16)
    second = _opt(second)
    pe, pt = np.zeros((R, NQ, 2 * L), np.int64), np.zeros((R, NQ, 2 * L), np.int64)
    de, dt = np.zeros((R, NQ, 16), np.int64), np.zeros((R, NQ, 16), np.int64)
    st = C.c_int(0)
    rc = lib().kbbq_build_host(ptr(seq), ptr(qual), ptr(corr), ptr(rg), ptr(second), N, L, R, minscore,
                               ptr(pe), ptr(pt), ptr(de), ptr(dt), C.byref(st), _dev(device))
    check(rc, st.value)
    return pe, pt, de, dt


def marginals_host(pos_errs, pos_total, device=None):
    pos_errs, pos_total = i64(pos_errs), i64(pos_total)
    R, nq, L2 = pos_total.shape
    assert nq == NQ
    q_e, q_t = np.zeros((R, NQ), np.int64), np.zeros((R, NQ), np.int64)
    g_e, g_t, mq = np.zeros(R, np.int64), np.zeros(R, np.int64), np.zeros(R, np.int64)
    check(lib().kbbq_marginals_host(ptr(pos_errs), ptr(pos_total), L2 // 2, R, ptr(q_e), ptr(q_t),
                                    ptr(g_e), ptr(g_t), ptr(mq), _dev(device)))
    return mq, g_e, g_t, q_e, q_t


def delta_q_host(prior_q, numerrs, numtotal, device=None):
    prior_q, numerrs, numtotal = i64(prior_q), i64(numerrs), i64(numtotal)
    out = np.zeros(prior_q.shape, np.int64)
    check(lib().kbbq_delta_q_host(ptr(prior_q), ptr(numerrs), ptr(numtotal), prior_q.size, ptr(out), _dev(device)))
    return out


def posterior_q_real_host(prior_q, numerrs, numtotal, device=None):
    """MAP quality for real-valued priors (the read-group table of a recalibration report)."""
    prior_q = np.ascontiguousarray(prior_q, dtype=np.float64)
    numerrs, numtotal = i64(numerrs), i64(numtotal)
    out = np.zeros(prior_q.shape, np.int64)
    check(lib().kbbq_posterior_q_real_host(ptr(prior_q), ptr(numerrs), ptr(numtotal), prior_q.size, ptr(out),
                                           _dev(device)))
    return out


def calibration_counts_host(qual, err=None, seq=None, corr=None, skip=None, device=None):
    """-> (total int64[256], errs int64[256]): bases and errors per quality, skipped bases left out."""
    qual = u8(qual).ravel()
    arrs = [_opt(a) for a in (err, seq, corr, skip)]
    for a in arrs:
        assert a is None or a.size == qual.size
    total, errs = np.zeros(256, np.int64), np.zeros(256, np.int64)
    check(lib().kbbq_calibration_counts_host(ptr(qual), *[ptr(a) for a in arrs], qual.size, ptr(total), ptr(errs),
                                             _dev(device)))
    return total, errs


def build_bam_host(seq, qual, err, skip, rg, flags, aln_start, aln_end, L, R, minscore=6, tables=None, device=None):
    """BAM-side tally on packed host arrays (kbbq_build_bam_host); `tables` = (pe, pt, de, dt) to add to."""
    seq, qual, err = u8(seq).ravel(), u8(qual).ravel(), u8(err).ravel()
    skip = _opt(skip)
    N = seq.size // L
    assert seq.size == qual.size == err.size == N * L
    flags = _opt(flags)
    rg, aln_start, aln_end = _opt(rg, np.uint16), _opt(aln_start, np.uint16), _opt(aln_end, np.uint16)
    if tables is None:
        tables = (np.zeros((R, NQ, 2 * L), np.int64), np.zeros((R, NQ, 2 * L), np.int64),
                  np.zeros((R, NQ, 16), np.int64), np.zeros((R, NQ, 16), np.int64))
    pe, pt, de, dt = tables
    st = C.c_int(0)
    rc = lib().kbbq_build_bam_host(ptr(seq), ptr(qual), ptr(err), ptr(skip), ptr(rg), ptr(flags), ptr(aln_start),
                                   ptr(aln_end), N, L, R, minscore, ptr(pe), ptr(pt), ptr(de), ptr(dt), C.byref(st),
                                   _dev(device))
    check(rc, st.value)
    return pe, pt, de, dt


def apply_bam_host(seq, qual, rg, flags, L, R, meanq, rgdq, qdq, posdq, dindq, minscore=6, device=None):
    seq, qual = u8(seq).ravel(), u8(qual).ravel()
    N = seq.size // L
    flags = _opt(flags)
    rg = _opt(rg, np.uint16)
    meanq, rgdq, qdq, posdq, dindq = [i64(a) for a in (meanq, rgdq, qdq, posdq, dindq)]
    nq, ndin1 = qdq.shape[1], dindq.shape[2]
    assert posdq.shape == (R, nq, 2 * L) and dindq.shape[:2] == (R, nq)
    out = np.zeros((N, L), np.uint8)
    st = C.c_int(0)
    rc = lib().kbbq_apply_bam_host(ptr(seq), ptr(qual), ptr(rg), ptr(flags), N, L, R, minscore, ptr(meanq), ptr(rgdq),
                                   ptr(qdq), ptr(posdq), ptr(dindq), nq, ndin1, ptr(out), C.byref(st), _dev(device))
    check(rc, st.value)
    return out


def get_delta_qs_host(meanq, rg_errs, rg_total, q_errs, q_total, pos_errs, pos_total, din_errs, din_total,
                      device=None):
    arrs = [i64(a) for a in (meanq, rg_errs, rg_total, q_errs, q_total, pos_errs, pos_total, din_errs, din_total)]
    R, nq = arrs[4].shape
    ncyc, ndin = arrs[6].shape[2], arrs[8].shape[2]
    rgdq, qdq = np.zeros(R, np.int64), np.zeros((R, nq), np.int64)
    posdq, dindq = np.zeros((R, nq, ncyc), np.int64), np.zeros((R, nq, ndin + 1), np.int64)
    check(lib().kbbq_get_delta_qs_host(*[ptr(a) for a in arrs], R, nq, ncyc, ndin, ptr(rgdq), ptr(qdq),
                                       ptr(posdq), ptr(dindq), _dev(device)))
    return rgdq, qdq, posdq, dindq


def apply_host(seq, qual, rg, second, L, R, meanq, rgdq, qdq, posdq, dindq, minscore=6, device=None):
    seq, qual = u8(seq).ravel(), u8(qual).ravel()
    N = seq.size // L
    rg = _opt(rg, np.uint16)
    second = _opt(second)
    meanq, rgdq, qdq, posdq, dindq = [i64(a) for a in (meanq, rgdq, qdq, posdq, dindq)]
    nq, ndin1 = qdq.shape[1], dindq.shape[2]
    assert posdq.shape == (R, nq, 2 * L) and dindq.shape[:2] == (R, nq)
    out = np.zeros((N, L), np.uint8)
    st = C.c_int(0)
    rc = lib().kbbq_apply_host(ptr(seq), ptr(qual), ptr(rg), ptr(second), N, L, R, minscore, ptr(meanq),
                               ptr(rgdq), ptr(qdq), ptr(posdq), ptr(dindq), nq, ndin1, ptr(out),
                               C.byref(st), _dev(device))
    check(rc, st.value)
    return out


def device_list(devices=None):
    """Devices of the whole-path entry points: an explicit list, else KBBQ_DEVICES ("0,1,2,3"), else [DEVICE]."""
    if devices is None:
        env = os.environ.get("KBBQ_DEVICES", "").strip()
        devices = [int(x) for x in env.split(",") if x.strip() != ""] if env else [DEVICE]
    elif isinstance(devices, int):
        devices = [devices]
    devices = [int(d) for d in devices]
    if not devices:
        raise ValueError("empty device list")
    return devices


def recalibrate_host(seq, qual, corr, rg, second, L, R, minscore=6, want_tables=False, device=None, out=None,
                     devices=None):
    """Whole path on host buffers; returns out_qual [N, L] u8 (and tables / deltas if asked).
    devices: several GPUs of this box share the reads (kbbq_recalibrate_host_multi); the result is the same."""
    seq, qual, corr = u8(seq).ravel(), u8(qual).ravel(), u8(corr).ravel()
    N = seq.size // L
    rg = _opt(rg, np.uint16)
    second = _opt(second)
    if out is None:
        out = np.zeros((N, L), np.uint8)
    tables = deltas = None
    if want_tables:
        tables = np.zeros(2 * R * NQ * 2 * L + 2 * R * NQ * 16, np.int64)
        deltas = np.zeros(2 * R + R * NQ * (1 + 2 * L + 17), np.int64)
    st = C.c_int(0)
    devs = device_list(devices if devices is not None else device)
    dev_arr = (C.c_int * len(devs))(*devs)
    rc = lib().kbbq_recalibrate_host_multi(ptr(seq), ptr(qual), ptr(corr), ptr(rg), ptr(second), N, L, R, minscore,
                                           ptr(out), ptr(tables), ptr(deltas), C.byref(st), dev_arr, len(devs))
    check(rc, st.value)
    if not want_tables:
        return out
    npos, ndin = R * NQ * 2 * L, R * NQ * 16
    tabs = (tables[:npos].reshape(R, NQ, 2 * L), tables[npos:2 * npos].reshape(R, NQ, 2 * L),
            tables[2 * npos:2 * npos + ndin].reshape(R, NQ, 16), tables[2 * npos + ndin:].reshape(R, NQ, 16))
    return out, tabs, split_deltas(deltas, L, R)


def kmer_table_bytes(N, L, k):
    """-> (capacity, bytes) of the default k-mer table for N reads of length L."""
    cap, nbytes = C.c_uint64(0), C.c_size_t(0)
    check(lib().kbbq_kmer_table_bytes(N, L, k, C.byref(cap), C.byref(nbytes)))
    return cap.value, nbytes.value


def kmer_min_count(hist):
    """The automatic threshold of a 256-bin count histogram (kbbq_kmer_min_count)."""
    hist = np.ascontiguousarray(hist, dtype=np.uint64)
    assert hist.size == 256
    return int(lib().kbbq_kmer_min_count(ptr(hist)))


def kmer_stream_plan(windows, budget_bytes):
    """-> (filter_words, capacity) of a sieved k-mer table for `windows` windows within budget_bytes
    (kbbq_kmer_stream_plan); ValueError when not even the smallest table fits."""
    f, cap = C.c_uint64(0), C.c_uint64(0)
    rc = lib().kbbq_kmer_stream_plan(windows, budget_bytes, C.byref(f), C.byref(cap))
    if rc == E_UNSUPPORTED:
        raise ValueError("a sieved k-mer table for %d windows does not fit %.3f GB" % (windows, budget_bytes / 1e9))
    check(rc)
    return f.value, cap.value


def _kmer_check(rc, status, N, L, k, device):
    if rc == E_UNSUPPORTED:
        nbytes = kmer_table_bytes(N, L, k)[1]
        raise DoesNotFit("%d reads x %d bp with a %.1f GB k-mer table (k = %d) do not fit the free memory of GPU %d"
                         % (N, L, nbytes / 1e9, k, device))
    check(rc, status)


def kmer_errors_host(seq, L, k=23, min_count=0, device=None, rule=KMER_BOUNDARIES):
    """Errors from the batch's k-mer counts (kbbq_kmer_errors_rule_host) by `rule` (KMER_BOUNDARIES or KMER_CORRECT)
    -> (bits u32[ceil(N*L/32)], hist u64[256], t)."""
    seq = u8(seq).ravel()
    N = seq.size // L
    assert seq.size == N * L
    bits = np.zeros((N * L + 31) // 32, np.uint32)
    hist = np.zeros(256, np.uint64)
    t = C.c_int(0)
    dev = _dev(device)
    rc = lib().kbbq_kmer_errors_rule_host(ptr(seq), N, L, k, min_count, rule, ptr(bits), ptr(hist), C.byref(t), dev)
    _kmer_check(rc, FLAG_KMER_FULL, N, L, k, dev)   # a full table is the only data error of this entry point
    return bits, hist, t.value


def recalibrate_kmer_host(seq, qual, rg, second, L, R, minscore=6, k=23, min_count=0, want_tables=False, device=None,
                          correct=False):
    """The whole path with the errors found from the reads' k-mer counts (kbbq_recalibrate_kmer_rule_host; correct:
    by the correcting walk instead of the boundary rule) -> (out_qual [N, L] u8, t), or (out_qual, t, tables, deltas)
    as recalibrate_host's with want_tables."""
    seq, qual = u8(seq).ravel(), u8(qual).ravel()
    N = seq.size // L
    assert seq.size == qual.size == N * L
    rg = _opt(rg, np.uint16)
    second = _opt(second)
    out = np.zeros((N, L), np.uint8)
    tables = deltas = None
    if want_tables:
        tables = np.zeros(2 * R * NQ * 2 * L + 2 * R * NQ * 16, np.int64)
        deltas = np.zeros(2 * R + R * NQ * (1 + 2 * L + 17), np.int64)
    t, st = C.c_int(0), C.c_int(0)
    dev = _dev(device)
    rule = KMER_CORRECT if correct else KMER_BOUNDARIES
    rc = lib().kbbq_recalibrate_kmer_rule_host(ptr(seq), ptr(qual), ptr(rg), ptr(second), N, L, R, minscore, k,
                                               min_count, rule, ptr(out), ptr(tables), ptr(deltas), C.byref(t),
                                               C.byref(st), dev)
    _kmer_check(rc, st.value, N, L, k, dev)
    if not want_tables:
        return out, t.value
    npos, ndin = R * NQ * 2 * L, R * NQ * 16
    tabs = (tables[:npos].reshape(R, NQ, 2 * L), tables[npos:2 * npos].reshape(R, NQ, 2 * L),
            tables[2 * npos:2 * npos + ndin].reshape(R, NQ, 16), tables[2 * npos + ndin:].reshape(R, NQ, 16))
    return out, t.value, tabs, split_deltas(deltas, L, R)


def split_deltas(deltas, L, R):
    """[meanq R | rgdq R | qdq R*43 | posdq R*43*2L | dindq R*43*17] -> the five arrays"""
    npos = R * NQ * 2 * L
    o = 0
    meanq = deltas[o:o + R]; o += R
    rgdq = deltas[o:o + R]; o += R
    qdq = deltas[o:o + R * NQ].reshape(R, NQ); o += R * NQ
    posdq = deltas[o:o + npos].reshape(R, NQ, 2 * L); o += npos
    dindq = deltas[o:].reshape(R, NQ, 17)
    return meanq, rgdq, qdq, posdq, dindq


class Session:
    """kbbq_session: the two passes of the path on one device, fed chunk by chunk from host arrays
    (include/kbbq_b200.h).  resident_reads > 0 keeps that many reads in HBM between the passes."""

    def __init__(self, L, R=1, minscore=6, chunk_reads=0, resident_reads=0, device=None, host_threads=0):
        self.L, self.R = int(L), int(R)
        self.device = _dev(device)
        h = C.c_void_p()
        check(lib().kbbq_session_create(self.device, self.L, self.R, minscore, chunk_reads, resident_reads,
                                        host_threads, C.byref(h)))
        self.h = h
        self.chunk_reads = int(lib().kbbq_session_chunk_reads(h))
        self.ntab = 2 * R * NQ * 2 * L + 2 * R * NQ * 16
        self._keep = []   # output arrays still being written by the device

    def close(self):
        if self.h:
            lib().kbbq_session_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def reset(self):
        check(lib().kbbq_session_reset(self.h))

    def build_chunk(self, seq, qual, corr, rg=None, second=None, keep=False):
        seq, qual, corr = u8(seq).ravel(), u8(qual).ravel(), u8(corr).ravel()
        n = seq.size // self.L
        rg = _opt(rg, np.uint16)
        second = _opt(second)
        check(lib().kbbq_session_build_chunk(self.h, ptr(seq), ptr(qual), ptr(corr), ptr(rg), ptr(second), n, int(keep)))

    def build_range(self, seq, qual, corr, rg=None, second=None):
        """Pass 1 of reads that lie contiguously in host memory: cut into chunks by the session and pipelined across
        them (kbbq_session_build_range).  Returns the number of chunks added."""
        seq, qual, corr = u8(seq).ravel(), u8(qual).ravel(), u8(corr).ravel()
        n = seq.size // self.L
        rg = _opt(rg, np.uint16)
        second = _opt(second)
        check(lib().kbbq_session_build_range(self.h, ptr(seq), ptr(qual), ptr(corr), ptr(rg), ptr(second), n))
        return -(-n // self.chunk_reads)

    def tables(self):
        t = np.zeros(self.ntab, np.int64)
        check(lib().kbbq_session_tables(self.h, ptr(t)))
        return t

    def set_tables(self, t):
        t = i64(t).ravel()
        assert t.size == self.ntab
        check(lib().kbbq_session_set_tables(self.h, ptr(t)))

    def tables_dev(self):
        """(device pointer, element count, cudaStream_t) of the session's table buffer"""
        p, n, st = C.c_void_p(), C.c_int64(), C.c_void_p()
        check(lib().kbbq_session_tables_dev(self.h, C.byref(p), C.byref(n), C.byref(st)))
        return p.value, n.value, st.value

    def flush(self):
        check(lib().kbbq_session_flush(self.h))

    def model(self, want_deltas=False):
        d = np.zeros(2 * self.R + self.R * NQ * (1 + 2 * self.L + 17), np.int64) if want_deltas else None
        check(lib().kbbq_session_model(self.h, ptr(d)))
        return split_deltas(d, self.L, self.R) if want_deltas else None

    def apply_resident(self, chunk, out):
        assert out.dtype == np.uint8 and out.flags["C_CONTIGUOUS"]
        self._keep.append(out)
        check(lib().kbbq_session_apply_resident(self.h, chunk, ptr(out)))

    def apply_chunk(self, seq, qual, rg, second, out):
        seq, qual = u8(seq).ravel(), u8(qual).ravel()
        n = seq.size // self.L
        rg = _opt(rg, np.uint16)
        second = _opt(second)
        assert out.dtype == np.uint8 and out.flags["C_CONTIGUOUS"] and out.size >= n * self.L
        self._keep.append(out)
        check(lib().kbbq_session_apply_chunk(self.h, ptr(seq), ptr(qual), ptr(rg), ptr(second), n, ptr(out)))

    def sync(self):
        st = C.c_int(0)
        rc = lib().kbbq_session_sync(self.h, C.byref(st))
        self._keep = []
        check(rc, st.value)

    def traffic(self):
        a, b = C.c_int64(), C.c_int64()
        check(lib().kbbq_session_traffic(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    # ---- `kbbq recalibrate -r` in chunks: a sieved k-mer table (include/kbbq_b200.h, kbbq_session_kmer_*) ----

    def kmer_begin(self, k, windows, filter_words=0, capacity=0):
        """Allocate and clear the filter and the table for k-mers of length k; 0 sizes them by kbbq_kmer_stream_plan
        of `windows` (the input's windows) from the free memory.  ValueError when that does not fit."""
        self.k = int(k)
        rc = lib().kbbq_session_kmer_begin(self.h, self.k, int(windows), filter_words, capacity)
        if rc == E_UNSUPPORTED:
            what = ("%d filter words and %d slots (%.2f GB)" % (filter_words, capacity, (8 * filter_words + 16 * capacity) / 1e9)
                    if filter_words else "the smallest sieved table for %d windows" % windows)
            raise ValueError("k-mer table (k = %d): %s do not fit the free memory of GPU %d" % (self.k, what, self.device))
        check(rc)

    def kmer_sizes(self):
        """-> (filter_words, capacity) the k-mer buffers were given."""
        f, cap = C.c_uint64(0), C.c_uint64(0)
        check(lib().kbbq_session_kmer_sizes(self.h, C.byref(f), C.byref(cap)))
        return f.value, cap.value

    def kmer_sieve(self, seq):
        """Pass A over one chunk (every chunk of the input)."""
        seq = u8(seq).ravel()
        check(lib().kbbq_session_kmer_sieve(self.h, ptr(seq), seq.size // self.L))

    def kmer_count(self, seq):
        """Pass B over one chunk (every chunk again, after pass A).  MemoryError, naming the table's size, when the
        table filled in pass A."""
        seq = u8(seq).ravel()
        rc = lib().kbbq_session_kmer_count(self.h, ptr(seq), seq.size // self.L)
        if rc == E_DATA:
            self._kmer_full()
        check(rc)

    def _kmer_full(self):
        f, cap = self.kmer_sizes()
        raise MemoryError("the sieved k-mer table (k = %d) of %d slots (%.2f GB) is full: more distinct repeated "
                          "k-mers than it holds" % (self.k, cap, 16 * cap / 1e9))

    def kmer_threshold(self, min_count=0):
        """-> (t, hist u64[256]): the exact histogram and the threshold (min_count when > 0, else the first valley).
        MemoryError, naming the table's size, when it filled."""
        hist = np.zeros(256, np.uint64)
        t = C.c_int(0)
        rc = lib().kbbq_session_kmer_threshold(self.h, int(min_count), ptr(hist), C.byref(t))
        if rc == E_DATA:
            self._kmer_full()
        check(rc)
        return t.value, hist

    def kmer_rule(self, rule):
        """The rule build_chunk_kmer flags by (KMER_BOUNDARIES or KMER_CORRECT), from kmer_begin until the first
        build_chunk_kmer."""
        check(lib().kbbq_session_kmer_rule(self.h, int(rule)))

    def build_chunk_kmer(self, seq, qual, rg=None, second=None):
        """Pass 1 of the build for a chunk, its errors flagged from the k-mer table."""
        seq, qual = u8(seq).ravel(), u8(qual).ravel()
        rg = _opt(rg, np.uint16)
        second = _opt(second)
        check(lib().kbbq_session_build_chunk_kmer(self.h, ptr(seq), ptr(qual), ptr(rg), ptr(second), seq.size // self.L))
