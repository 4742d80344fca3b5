"""Mirror of the reference's kbbq/recalibrate.py -- the driver of the FASTQ recalibration path.

Same functions, signatures, return order and exceptions; the per-read Python loops of the
reference (kbbq/recalibrate.py:56-119 and :141-156) become one packed batch handed to the CUDA
kernels through the C ABI (include/kbbq_b200.h).
"""
import sys

import numpy as np

from . import _native
from . import compare_reads as utils
from .batch import ReadBatch
from .gatk import applybqsr


def find_corrected_sites(uncorr_read, corr_read):
    """reference: kbbq/recalibrate.py:13-20 -- raw character comparison of one read pair."""
    assert corr_read.name.startswith(uncorr_read.name)
    uncorr_seq = np.array(list(uncorr_read.sequence), dtype=np.str_)
    corr_seq = np.array(list(corr_read.sequence), dtype=np.str_)
    return (uncorr_seq != corr_seq)


def _tables_from_batch(batch, minscore=6):
    if batch.N == 0:
        # the reference returns zero-length arrays when there are no reads (kbbq/recalibrate.py:45-54)
        z = np.zeros(0, dtype=np.int64)
        return (utils.p_to_q(z.astype(float)), z.copy(), z.copy(), np.zeros((0, 43), np.int64),
                np.zeros((0, 43), np.int64), np.zeros((0, 43, 0), np.int64), np.zeros((0, 43, 0), np.int64),
                np.zeros((0, 43, 16), np.int64), np.zeros((0, 43, 16), np.int64))
    pe, pt, de, dt = _native.build_host(batch.seq, batch.qual, batch.corr, batch.rg, batch.second,
                                        batch.L, batch.R, minscore)
    meanq, rg_e, rg_t, q_e, q_t = _native.marginals_host(pe, pt)
    return meanq, rg_e, rg_t, q_e, q_t, pe, pt, de, dt


def fastq_to_covariate_arrays(fastq, infer_rg=False, minscore=6, maxscore=42):
    """reference: kbbq/recalibrate.py:22-121.

    -> (meanq, rg_errs, rg_total, q_errs, q_total, pos_errs, pos_total, dinuc_errs, dinuc_total),
    fresh int64 arrays of shapes [R], [R], [R], [R,43], [R,43], [R,43,2L], [R,43,2L], [R,43,16] x2.
    """
    if maxscore != 42:
        raise NotImplementedError("only maxscore = 42 is supported")
    batch = ReadBatch.from_fastq(fastq, infer_rg)
    return _tables_from_batch(batch, minscore)


STREAM_ABOVE_BYTES = 4 << 30      # larger FASTQ files go through the device in batches (host memory stays bounded)
STREAM_BATCH_READS = 8_000_000


def _stdout_fd():
    """Descriptor of sys.stdout, or None when it is not a real file (a StringIO, a capture object)."""
    try:
        fd = sys.stdout.fileno()
    except (AttributeError, OSError, ValueError):
        return None
    sys.stdout.flush()
    return fd


def _packed_batches(total, batch_reads, pack):
    """pack(lo, m) for the batches [lo, lo + m) of reads [0, total), in order; the next batch is tokenised on a worker
    thread (native code, GIL released) while the caller hands this one to the GPU, so host memory holds two."""
    from concurrent.futures import ThreadPoolExecutor
    starts = list(range(0, total, batch_reads))
    if not starts:
        return
    with ThreadPoolExecutor(1) as pool:
        nxt = pool.submit(pack, starts[0], min(batch_reads, total - starts[0]))
        for i in range(len(starts)):
            cur = nxt.result()
            if i + 1 < len(starts):
                nxt = pool.submit(pack, starts[i + 1], min(batch_reads, total - starts[i + 1]))
            yield cur


def _apply_pass(sess, reads, rg, second, batch_reads):
    """Pass 2 of a streaming session whose model is built: every read of `reads` packed again, applied and printed."""
    L = reads.L
    fd = _stdout_fd()
    for lo, m, seq, qual in _packed_batches(reads.N, batch_reads, lambda lo, m: (lo, m) + reads.pack(lo, m)):
        out = np.empty((m, L), np.uint8)
        sess.apply_chunk(seq, qual, rg[lo:lo + m], second[lo:lo + m], out)
        sess.sync()   # raises the reference's exception for bad input; `out` is complete
        if fd is not None:
            reads.write(fd, out, lo, m)
        else:
            txt = (out + np.uint8(33)).astype(np.uint8)
            sys.stdout.write(''.join('@%s\n%s\n+\n%s\n' % (reads.name(lo + i), seq[i].tobytes().decode(),
                                                          txt[i].tobytes().decode('latin-1')) for i in range(m)))


def _recalibrate_fastq_streamed(fastq, infer_rg, batch_reads, devices=None):
    """The two passes of kbbq/recalibrate.py:123-156 over batches of `batch_reads` reads through a session
    (kbbq_session_*, csrc/host_api.cu): pass 1 packs a batch from the indexed files and hands it to the session,
    which uploads it and adds it to the tables on the GPU while the next batch is being packed; the model runs
    once; pass 2 packs each batch again, applies and prints it.  Host memory holds two batches (plus 8 bytes of
    index per read); the result is the one of the single-batch path.  Pass 1 covers the reads both files have
    (zip() in the reference stops at the shorter one), pass 2 every read of fastq[0] (kbbq/recalibrate.py:141)."""
    from . import fastx
    reads, fixed = fastx.NativeFastq(fastq[0]), fastx.NativeFastq(fastq[1])
    n_build = min(reads.N, fixed.N)
    reads.check_names(fixed, n_build)
    if reads.N == 0:
        return
    if reads.L < 0 or (n_build and fixed.L != reads.L):
        raise ValueError("operands could not be broadcast together: reads of unequal length")
    rg, second, keys = reads.infer(infer_rg)
    L, R = reads.L, max(1, len(keys))
    device = _native.device_list(devices)[0]
    with _native.Session(L, R, 6, chunk_reads=batch_reads, resident_reads=0, device=device) as sess:
        for lo, m, seq, qual, corr in _packed_batches(n_build, batch_reads,
                                                      lambda lo, m: (lo, m) + reads.pack(lo, m) + fixed.pack(lo, m)[:1]):
            sess.build_chunk(seq, qual, corr, rg[lo:lo + m], second[lo:lo + m])
        fixed.close()
        sess.model()
        _apply_pass(sess, reads, rg, second, batch_reads)
    reads.close()


def _fastq_size(path):
    """Size of the FASTQ text of a regular file (a gzip file is taken at four times its size: the streaming decision
    is about the inflated reads); 0 for anything else (pipes, process substitution)."""
    import os
    try:
        if not os.path.isfile(path):
            return 0
        size = os.path.getsize(path)
        with open(path, "rb") as fh:
            gz = fh.read(2) == b"\x1f\x8b"
        return 4 * size if gz else size
    except OSError:
        return 0


def recalibrate_fastq(fastq, infer_rg=False, devices=None):
    """Recalibrate fastq[0] given its corrected twin fastq[1]; FASTQ to stdout
    (reference: kbbq/recalibrate.py:123-156: name without comment, sequence, '+', chr(q + 33)).
    devices: GPUs of this box that share the reads (default: KBBQ_DEVICES, else one); the output is the same."""
    import os
    batch_reads = int(os.environ.get("KBBQ_BATCH_READS", "0"))
    if batch_reads <= 0 and _fastq_size(fastq[0]) > STREAM_ABOVE_BYTES:
        batch_reads = STREAM_BATCH_READS
    if batch_reads > 0:
        return _recalibrate_fastq_streamed(fastq, infer_rg, batch_reads, devices)
    devs = _native.device_list(devices)
    fd = _stdout_fd()
    if fd is not None and len(devs) == 1:
        # the whole path in native code: tokenise, upload, build, model, apply, download, format -- pipelined per chunk
        import ctypes as C
        from . import fastx
        n, nrg, st = C.c_int64(0), C.c_int(0), C.c_int(0)
        rc = _native.lib().kbbq_recalibrate_fastq(str(fastq[0]).encode(), str(fastq[1]).encode(), 1 if infer_rg else 0, 6, fd,
                                                  devs[0], 0, C.byref(n), C.byref(nrg), C.byref(st))
        if rc == 0:
            return
        if rc != _native.E_UNSUPPORTED:
            if rc == _native.E_DATA:
                _native.check(rc, st.value)
            fastx._check(rc, str(fastq[0]))
    batch = ReadBatch.from_fastq(fastq, infer_rg)
    if batch.N == 0:
        return
    if batch.N_all != batch.N:
        # fastq[0] holds more reads than the corrected file: the tables come from the pairs, every read is written
        batch.source.close()
        return _recalibrate_fastq_streamed(fastq, infer_rg, STREAM_BATCH_READS, devices)
    out = _native.recalibrate_host(batch.seq, batch.qual, batch.corr, batch.rg, batch.second,
                                   batch.L, batch.R, 6, devices=devices)
    # native formatter straight to the stdout descriptor when there is one; text fallback otherwise
    # (e.g. sys.stdout replaced by an in-memory stream)
    w = sys.stdout
    try:
        fd = w.fileno()
    except (AttributeError, OSError, ValueError):
        fd = None
    if fd is not None and batch.source is not None:
        w.flush()
        batch.source.write(fd, out, 0, batch.N)
        return
    qual_txt = (out + np.uint8(33)).astype(np.uint8)
    seq = batch.seq
    chunks = []
    for i, name in enumerate(batch.names):
        chunks.append('@%s\n%s\n+\n%s\n' % (name, seq[i].tobytes().decode(), qual_txt[i].tobytes().decode('latin-1')))
        if len(chunks) >= 4096:
            w.write(''.join(chunks))
            chunks = []
    w.write(''.join(chunks))


def _recalibrate_reads_streamed(reads, infer_rg, k, min_count, batch_reads, device, correct=False, devices=None):
    """recalibrate_reads through a streaming session, for files of any size (DESIGN.md §10, "Streaming"): two passes
    over every batch fill a sieved k-mer table that only holds the k-mers seen at least twice (A: sieve, B: count),
    the threshold is taken from its histogram -- the exact one --, a third pass flags and builds, the model runs once
    and a fourth pass applies and prints, as _recalibrate_fastq_streamed does.  Host memory holds two batches (plus
    the index of the file); the output is the single-batch path's, byte for byte.  correct: the third pass flags by
    the correcting walk.  devices: several GPUs, the first `device`, each holding one partition of the table split by
    key (DESIGN.md §10, "Several GPUs"): the same output with room for n times the k-mers.  When `device` cannot read
    the others' memory the table stays whole on `device`."""
    if reads.L < 0:
        raise ValueError("%s: reads of unequal length are not supported on this path" % reads.path)
    rg, second, keys = reads.infer(infer_rg)
    N, L, R = reads.N, reads.L, max(1, len(keys))

    def seq_only(lo, m):
        return reads.pack(lo, m)[0]

    with _native.Session(L, R, 6, chunk_reads=batch_reads, resident_reads=0, device=device) as sess:
        windows = N * max(0, L - k + 1)
        try:
            sess.kmer_begin(k, windows, devices=devices)
        except _native.PeerUnreachable:
            sess.kmer_begin(k, windows)
        if correct:
            sess.kmer_rule(_native.KMER_CORRECT)
        for seq in _packed_batches(N, batch_reads, seq_only):
            sess.kmer_sieve(seq)
        for seq in _packed_batches(N, batch_reads, seq_only):
            sess.kmer_count(seq)
        sess.kmer_threshold(min_count)
        for lo, m, seq, qual in _packed_batches(N, batch_reads, lambda lo, m: (lo, m) + reads.pack(lo, m)):
            sess.build_chunk_kmer(seq, qual, rg[lo:lo + m], second[lo:lo + m])
        sess.model()
        _apply_pass(sess, reads, rg, second, batch_reads)


def recalibrate_reads(path, infer_rg=False, k=23, min_count=0, devices=None, correct=False):
    """Recalibrate the reads of one FASTQ file with the errors found from their own k-mer counts (kbbq.kmer); FASTQ to
    stdout as recalibrate_fastq prints it, on the first of `devices`.  The file is one batch unless KBBQ_BATCH_READS
    is set, the file is larger than STREAM_ABOVE_BYTES, or the batch and its k-mer table do not fit the GPU: then it
    streams through in batches (_recalibrate_reads_streamed), with the same output, and with its k-mer table split
    across every GPU of `devices`.  correct: find the errors by correcting each read against its trusted k-mers
    (DESIGN.md §10, "The correcting walk") instead of by the boundaries of the uncovered runs."""
    import os
    from . import fastx
    if not 1 <= k <= 31:
        raise ValueError("k must be in 1..31, got %d" % k)
    if min_count < 0:
        raise ValueError("min_count must be >= 0, got %d" % min_count)
    batch_reads = int(os.environ.get("KBBQ_BATCH_READS", "0"))
    if batch_reads <= 0 and _fastq_size(path) > STREAM_ABOVE_BYTES:
        batch_reads = STREAM_BATCH_READS
    devs = _native.device_list(devices)
    device = devs[0]
    # the option is passed on only when set: without it both drivers are called exactly as before it existed
    opts = {"correct": True} if correct else {}
    stream_opts = dict(opts, devices=devs) if len(devs) > 1 else opts
    reads = fastx.NativeFastq(path)
    try:
        if reads.N == 0:
            return
        if batch_reads > 0:
            return _recalibrate_reads_streamed(reads, infer_rg, k, min_count, batch_reads, device, **stream_opts)
        seq, qual = reads.pack()   # ValueError for reads of unequal length, as on the -f path
        rg, second, keys = reads.infer(infer_rg)
        L, R = reads.L, max(1, len(keys))
        try:
            out, _ = _native.recalibrate_kmer_host(seq, qual, rg, second, L, R, 6, k, min_count, device=device, **opts)
        except _native.DoesNotFit:
            del seq, qual
            return _recalibrate_reads_streamed(reads, infer_rg, k, min_count, STREAM_BATCH_READS, device, **stream_opts)
        fd = _stdout_fd()
        if fd is not None:
            reads.write(fd, out)
            return
        txt = (out + np.uint8(33)).astype(np.uint8)
        sys.stdout.write(''.join('@%s\n%s\n+\n%s\n' % (reads.name(i), seq[i].tobytes().decode(),
                                                      txt[i].tobytes().decode('latin-1')) for i in range(reads.N)))
    finally:
        reads.close()


def recalibrate_bam(bam, use_oq=False, set_oq=False):
    """Not implemented in the reference either (kbbq/recalibrate.py:158-164)."""
    raise NotImplementedError('Recalibrating a bam is not yet implemented. \
        Try converting your BAM to a FASTQ file with the samtools fastq command.')


def recalibrate(bam, fastq, infer_rg=False, use_oq=False, set_oq=False, gatkreport=None, devices=None, reads=None,
                kmer_size=23, min_count=0, kmer_correct=False):
    """reference: kbbq/recalibrate.py:166-174 (devices: see recalibrate_fastq).  reads: one FASTQ file whose errors
    come from its own k-mer counts (recalibrate_reads) instead of a corrected twin; kmer_correct: found by the
    correcting walk."""
    if gatkreport is not None:
        raise NotImplementedError('GATKreport reading / creation is not yet supported.')
    elif bam is not None:
        recalibrate_bam(bam, use_oq, set_oq)
    elif fastq is not None:
        recalibrate_fastq(fastq, infer_rg=infer_rg, devices=devices)
    elif reads is not None:
        opts = {"correct": True} if kmer_correct else {}   # as in recalibrate_reads: passed on only when set
        recalibrate_reads(reads, infer_rg=infer_rg, k=kmer_size, min_count=min_count, devices=devices, **opts)
    else:
        raise ValueError("A BAM or FASTQ file should be provided for recalibration.")
