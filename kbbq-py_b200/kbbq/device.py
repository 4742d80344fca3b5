"""Device-resident driver of the hot path: torch tensors in HBM, kernels through the C ABI.

torch is plumbing only (allocation, streams, torch.distributed); every kernel launched here is
one of libkbbq_b200.so's.  This is what a batch driver (and bench.py) uses when the packed reads
already live on the GPU; the host-buffer path is kbbq._native.recalibrate_host.

Multi-GPU (SURVEY.md section 8e): reads shard by rank, each rank builds partial int64 tables, ONE
all-reduce (sum) over the packed table buffer makes them global, every rank recomputes the deltas
deterministically from the reduced integers (so no broadcast is needed) and applies them to its
own shard.  Integer sums make the result independent of the number of ranks.
"""
import ctypes as C
import weakref

import torch

from . import _native
from . import parallel

NQ = _native.NQ


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _on_device(fn):
    """Run a method with self.device current: the C ABI launches on, and uploads its constants to, the
    CURRENT device, while the stream and the pointers handed over belong to self.device."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *args, **kwargs):
        with torch.cuda.device(self.device):
            return fn(self, *args, **kwargs)
    return wrapper


class SegmentedBatch:
    """A batch in the segmented HBM layout (include/kbbq_b200.h, "Segmented batch layout"): rows sorted by
    2 * rg + second, spans padded to 16 rows.  seq / qual / corr: u8 [rows_bound, L]; seg: the span table;
    dest: int32 [N], row of read i."""

    def __init__(self, seq, qual, corr, seg, dest, n_reads, rows_bound):
        self.seq, self.qual, self.corr, self.seg, self.dest = seq, qual, corr, seg, dest
        self.N, self.rows_bound = n_reads, rows_bound


class DeviceRecalibrator:
    """Owns the tables, model buffers and workspace for batches of up to `max_reads` reads."""

    def __init__(self, L, R=1, max_reads=0, minscore=6, device=None, process_group=None):
        if not torch.cuda.is_available():
            raise _native.KbbqNativeError("no CUDA device: kbbq_b200 has no CPU fallback")
        self.lib = _native.lib()
        self.L, self.R, self.minscore = int(L), int(R), int(minscore)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.pg = process_group
        npos, ndin = R * NQ * 2 * L, R * NQ * 16
        with torch.cuda.device(self.device):
            # one packed buffer [pos_errs | pos_total | din_errs | din_total]: one collective sums it
            self.tables = torch.zeros(2 * npos + 2 * ndin, dtype=torch.int64, device=self.device)
            self.pos_errs = self.tables[:npos].view(R, NQ, 2 * L)
            self.pos_total = self.tables[npos:2 * npos].view(R, NQ, 2 * L)
            self.din_errs = self.tables[2 * npos:2 * npos + ndin].view(R, NQ, 16)
            self.din_total = self.tables[2 * npos + ndin:].view(R, NQ, 16)
            self.q_errs = torch.zeros(R, NQ, dtype=torch.int64, device=self.device)
            self.q_total = torch.zeros(R, NQ, dtype=torch.int64, device=self.device)
            self.rg_errs = torch.zeros(R, dtype=torch.int64, device=self.device)
            self.rg_total = torch.zeros(R, dtype=torch.int64, device=self.device)
            self.meanq = torch.zeros(R, dtype=torch.int64, device=self.device)
            self.rgdq = torch.zeros(R, dtype=torch.int64, device=self.device)
            self.qdq = torch.zeros(R, NQ, dtype=torch.int64, device=self.device)
            self.posdq = torch.zeros(R, NQ, 2 * L, dtype=torch.int64, device=self.device)
            self.dindq = torch.zeros(R, NQ, 17, dtype=torch.int64, device=self.device)
            self.status = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.workspace = None
        self.ws_reads = -1
        self._ensure_workspace(max_reads)
        # base arrays built since the last reset (a weak reference and torch's version counter of each): any base
        # outside ACGTN in them has already set the status word, so applying them again skips the base check
        self._built = []

    @_on_device
    def _ensure_workspace(self, n_reads):
        if n_reads <= self.ws_reads:
            return
        nbytes = C.c_size_t(0)
        _native.check(self.lib.kbbq_workspace_bytes(n_reads, self.L, self.R, C.byref(nbytes)))
        self.workspace = torch.empty(max(nbytes.value, 256), dtype=torch.uint8, device=self.device)
        self.ws_bytes = nbytes.value
        self.ws_reads = n_reads

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def reset(self):
        self.tables.zero_()
        self.status.zero_()
        self._built = []

    @staticmethod
    def _version(t):
        try:
            return t._version
        except RuntimeError:   # inference-mode tensors keep no version counter
            return None

    def _remember_built(self, seq):
        v = self._version(seq)
        self._built = [(r, w) for r, w in self._built if r() is not None and r() is not seq]
        if v is not None:
            self._built.append((weakref.ref(seq), v))

    def _bases_checked(self, seq):
        """True when `seq` is a tensor this recalibrator built since its last reset and that torch has not written
        to since: the build flagged any base outside ACGTN in this status word, the apply need not look again."""
        v = self._version(seq)
        return v is not None and any(r() is seq and w == v for r, w in self._built)

    @_on_device
    def build(self, seq, qual, corr, rg=None, second=None, path=0):
        """Accumulate one batch into the tables (kbbq_build). Tensors: u8 [N, L] (rg int16/uint16 [N])."""
        N = seq.numel() // self.L
        self._ensure_workspace(N)
        rc = self.lib.kbbq_build(_p(seq), _p(qual), _p(corr), _p(rg), _p(second), N, self.L, self.R, self.minscore,
                                 _p(self.pos_errs), _p(self.pos_total), _p(self.din_errs), _p(self.din_total),
                                 _p(self.workspace), self.ws_bytes, _p(self.status), path, self._stream())
        _native.check(rc)
        self._remember_built(seq)

    @_on_device
    def build_from_bits(self, seq, qual, bits, corr_scratch, rg=None, second=None):
        """build() when the corrected reads arrive as the 1-bit-per-base mismatch map of
        kbbq_host_mismatch_bits (int32 tensor): it is expanded into `corr_scratch` (u8, like seq) first."""
        _native.check(self.lib.kbbq_expand_mismatch_bits(_p(seq), _p(bits), seq.numel(), _p(corr_scratch), self._stream()))
        self.build(seq, qual, corr_scratch, rg, second)

    @_on_device
    def segment(self, seq, qual, corr=None, rg=None, second=None):
        """Rewrite a batch into the segmented layout on the device (kbbq_segment_plan / _rows / _pad).
        Several read groups then run at the one-read-group speed of the kernels (build_segmented /
        apply_segmented); unsegment() brings recalibrated qualities back into read order."""
        N, L, R = seq.numel() // self.L, self.L, self.R
        if not self.lib.kbbq_segmented_supported(L, R, self.minscore):
            raise _native.KbbqNativeError("no shared-memory plan for L=%d, R=%d: use build() / apply()" % (L, R))
        rows = int(self.lib.kbbq_segment_rows_bound(N, R))
        dev, st = self.device, self._stream()
        seg = torch.empty(int(self.lib.kbbq_segment_table_elems(R)), dtype=torch.int32, device=dev)
        dest = torch.empty(max(N, 1), dtype=torch.int32, device=dev)
        _native.check(self.lib.kbbq_segment_plan(_p(rg), _p(second), N, R, _p(seg), _p(dest), _p(self.status), st))
        outs = []
        for src in (seq, qual, corr):
            if src is None:
                outs.append(None)
                continue
            dst = torch.empty(rows * L + 16, dtype=torch.uint8, device=dev)
            _native.check(self.lib.kbbq_segment_rows(_p(src), _p(dest), N, L, _p(dst), st))
            outs.append(dst)
        _native.check(self.lib.kbbq_segment_pad(_p(seg), R, L, _p(outs[0]), _p(outs[1]), _p(outs[2]), st))
        return SegmentedBatch(outs[0], outs[1], outs[2], seg, dest, N, rows)

    @_on_device
    def build_segmented(self, sb):
        """kbbq_build on a segmented batch (kbbq_build_segmented)."""
        self._ensure_workspace(sb.rows_bound)
        rc = self.lib.kbbq_build_segmented(_p(sb.seq), _p(sb.qual), _p(sb.corr), _p(sb.seg), sb.rows_bound, self.L, self.R,
                                           self.minscore, _p(self.pos_errs), _p(self.pos_total), _p(self.din_errs),
                                           _p(self.din_total), _p(self.workspace), self.ws_bytes, _p(self.status),
                                           self._stream())
        _native.check(rc)
        self._remember_built(sb.seq)

    @_on_device
    def apply_segmented(self, sb, out_seg):
        """kbbq_apply on a segmented batch; out_seg: u8 [rows_bound, L] in the segmented order."""
        self._ensure_workspace(sb.rows_bound)
        flags = _native.APPLY_BASES_CHECKED if self._bases_checked(sb.seq) else 0
        rc = self.lib.kbbq_apply_segmented_flags(_p(sb.seq), _p(sb.qual), _p(sb.seg), sb.rows_bound, self.L, self.R,
                                                 self.minscore, _p(self.meanq), _p(self.rgdq), _p(self.qdq),
                                                 _p(self.posdq), _p(self.dindq), NQ, 17, _p(out_seg), _p(self.workspace),
                                                 self.ws_bytes, _p(self.status), flags, self._stream())
        _native.check(rc)

    @_on_device
    def unsegment(self, sb, out_seg, out):
        """out row i = out_seg row dest[i] (kbbq_unsegment_rows)."""
        _native.check(self.lib.kbbq_unsegment_rows(_p(out_seg), _p(sb.dest), sb.N, self.L, sb.rows_bound, _p(out),
                                                   self._stream()))

    def allreduce(self):
        """Sum the partial tables over all ranks: the one collective of the path."""
        parallel.allreduce_tables(self.tables, self.pg)

    @_on_device
    def model(self):
        """marginals + meanq + hierarchical delta tables (kbbq_marginals, kbbq_get_delta_qs)."""
        L, R = self.L, self.R
        _native.check(self.lib.kbbq_marginals(_p(self.pos_errs), _p(self.pos_total), L, R, _p(self.q_errs),
                                              _p(self.q_total), _p(self.rg_errs), _p(self.rg_total),
                                              _p(self.meanq), self._stream()))
        _native.check(self.lib.kbbq_get_delta_qs(_p(self.meanq), _p(self.rg_errs), _p(self.rg_total),
                                                 _p(self.q_errs), _p(self.q_total), _p(self.pos_errs),
                                                 _p(self.pos_total), _p(self.din_errs), _p(self.din_total),
                                                 R, NQ, 2 * L, 16, _p(self.rgdq), _p(self.qdq), _p(self.posdq),
                                                 _p(self.dindq), self._stream()))

    @_on_device
    def apply(self, seq, qual, out, rg=None, second=None, path=0):
        """Write recalibrated qualities of one batch into `out` (kbbq_apply).  A batch that was not built here since
        the last reset (or was changed since) has its bases checked: one outside ACGTN raises at check_status()."""
        N = seq.numel() // self.L
        self._ensure_workspace(N)
        if self._bases_checked(seq):
            path |= _native.APPLY_BASES_CHECKED
        rc = self.lib.kbbq_apply(_p(seq), _p(qual), _p(rg), _p(second), N, self.L, self.R, self.minscore,
                                 _p(self.meanq), _p(self.rgdq), _p(self.qdq), _p(self.posdq), _p(self.dindq),
                                 NQ, 17, _p(out), _p(self.workspace), self.ws_bytes, _p(self.status), path,
                                 self._stream())
        _native.check(rc)

    @_on_device
    def build_bam(self, seq, qual, err, skip=None, rg=None, flags=None, aln_start=None, aln_end=None, fast=True):
        """Accumulate a batch of aligned reads (kbbq_build_bam): err / skip u8 [N, L] from the host's CIGAR
        walk, flags u8 [N] (bit 0 read 2, bit 1 reverse strand), aln_start / aln_end int16 [N]."""
        N = seq.numel() // self.L
        ws = self._bam_workspace(N) if fast else None
        rc = self.lib.kbbq_build_bam(_p(seq), _p(qual), _p(err), _p(skip), _p(rg), _p(flags), _p(aln_start),
                                     _p(aln_end), N, self.L, self.R, self.minscore, _p(self.pos_errs),
                                     _p(self.pos_total), _p(self.din_errs), _p(self.din_total), _p(ws),
                                     0 if ws is None else ws.numel(), _p(self.status), self._stream())
        _native.check(rc)

    @_on_device
    def _bam_workspace(self, n_reads):
        """Canonical copies of a BAM batch + the build / apply workspace (kbbq_bam_workspace_bytes)."""
        if n_reads > getattr(self, "bam_ws_reads", -1):
            nbytes = C.c_size_t(0)
            _native.check(self.lib.kbbq_bam_workspace_bytes(n_reads, self.L, self.R, C.byref(nbytes)))
            self.bam_ws = torch.empty(max(nbytes.value, 256), dtype=torch.uint8, device=self.device)
            self.bam_ws_reads = n_reads
        return self.bam_ws

    @_on_device
    def apply_bam(self, seq, qual, out, rg=None, flags=None, fast=True):
        """Recalibrated qualities of a batch of aligned reads (kbbq_apply_bam)."""
        N = seq.numel() // self.L
        ws = self._bam_workspace(N) if fast else None
        rc = self.lib.kbbq_apply_bam(_p(seq), _p(qual), _p(rg), _p(flags), N, self.L, self.R, self.minscore,
                                     _p(self.meanq), _p(self.rgdq), _p(self.qdq), _p(self.posdq), _p(self.dindq),
                                     NQ, 17, _p(out), _p(ws), 0 if ws is None else ws.numel(), _p(self.status),
                                     self._stream())
        _native.check(rc)

    @_on_device
    def check_status(self):
        """Synchronise and raise the reference's exception for any data error seen on the device."""
        st = int(self.status.item())
        if st:
            _native.raise_for_status(st)

    def covariate_arrays(self):
        """The reference's 9-tuple (kbbq/recalibrate.py:121) as host numpy arrays."""
        self.model()
        return tuple(t.cpu().numpy().copy() for t in (self.meanq, self.rg_errs, self.rg_total, self.q_errs,
                                                      self.q_total, self.pos_errs, self.pos_total,
                                                      self.din_errs, self.din_total))

    def delta_qs(self):
        return tuple(t.cpu().numpy().copy() for t in (self.rgdq, self.qdq, self.posdq, self.dindq))


def calibration_counts(qual, err=None, seq=None, corr=None, skip=None, total=None, errs=None):
    """Bases and errors per quality of device-resident reads (kbbq_calibration_counts, the counting
    step of kbbq/benchmark.py:76-91).  error = err != 0, or seq != corr when `err` is None; bases with
    a non-zero `skip` byte are left out.  Accumulates into int64[256] tensors `total` / `errs`
    (allocated when None) and returns them, so batches -- and, after an all-reduce, ranks -- add up."""
    lib = _native.lib()
    dev = qual.device
    torch.cuda.set_device(dev)
    if total is None:
        total = torch.zeros(256, dtype=torch.int64, device=dev)
    if errs is None:
        errs = torch.zeros(256, dtype=torch.int64, device=dev)
    rc = lib.kbbq_calibration_counts(_p(qual), _p(err), _p(seq), _p(corr), _p(skip), qual.numel(), _p(total),
                                     _p(errs), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    _native.check(rc)
    return total, errs


def synth_reads(seed, first_read, n, L, R, device=None, want_corr=True):
    """Counter-based synthetic reads generated on the GPU (kbbq_synth_reads): bench / test input."""
    lib = _native.lib()
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    torch.cuda.set_device(dev)
    seq = torch.empty(n, L, dtype=torch.uint8, device=dev)
    qual = torch.empty(n, L, dtype=torch.uint8, device=dev)
    corr = torch.empty(n, L, dtype=torch.uint8, device=dev)
    rg = torch.empty(n, dtype=torch.int16, device=dev)
    second = torch.empty(n, dtype=torch.uint8, device=dev)
    rc = lib.kbbq_synth_reads(seed, first_read, n, L, R, _p(seq), _p(qual), _p(corr), _p(rg), _p(second),
                              C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    _native.check(rc)
    return seq, qual, corr, rg, second
