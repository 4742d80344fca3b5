"""`kbbq recalibrate -r` streamed through the GPU in chunks: the sieved k-mer table (kbbq_kmer_sieve / _count_present /
_histogram_sieved / _flag_sieved), its sizing rule, the session entry points (kbbq_session_kmer_*) and the driver.
Every GPU comparison is bit for bit: against the C oracle, against an exact table of the same reads, and against the
single-batch path.  Which false-positive singletons the sieved table holds depends on the schedule; nothing checked
here does."""
import ctypes as C
import importlib.util
import os
import sys

import numpy as np
import pytest

E_ARG = -1


@pytest.fixture(scope="module")
def kmer_oracle():
    """tests/kmer_oracle.py, loaded by path (it compiles tests/kmer_oracle.c into a temporary directory)."""
    spec = importlib.util.spec_from_file_location(
        "kmer_oracle", os.path.join(os.path.dirname(os.path.abspath(__file__)), "kmer_oracle.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def batch(k, L, seed=3, lower=0.001):
    """Every k-mer of an 8 kb genome ~25 times, 1 % substitutions, N bases and a few lowercase bytes.
    -> seq, qual, second, N"""
    from kbbq import synth
    G = 8000
    n = (25 * G // (L - k + 1)) & ~1
    s = seed + 31 * k + L
    seq, qual, _, second = synth.genome_reads(s, G, n, L, 0.01, 0.003)
    low = np.random.default_rng(s + 1).random(seq.shape) < lower
    seq[low] = seq[low] | 0x20
    return seq, qual, second, n


# ---- CPU: the sizing rule -------------------------------------------------------------------------------------------

def _pow2(x):
    return x >= 1 and x & (x - 1) == 0


@pytest.mark.parametrize("windows", [0, 1, 1000, 1_280_000_000, 48_000_000 * 128])
@pytest.mark.parametrize("budget", [4 << 20, 1 << 30, 160 << 30])
def test_stream_plan(windows, budget):
    from kbbq import _native
    exact = _native.kmer_table_bytes(windows, 1, 1)[0]
    F, cap = _native.kmer_stream_plan(windows, budget)
    assert _pow2(F) and _pow2(cap)
    assert 8 * F + 16 * cap <= budget
    assert cap <= exact
    # the filter: the largest power of two with 8 F <= min(W, budget / 4) bytes, at least one word
    lim = min(windows, budget // 4)
    assert 8 * F <= lim < 16 * F or (F == 1 and lim < 8)
    # the table: the exact capacity when it fits, else the largest power of two that does
    assert cap == exact or 16 * 2 * cap > budget - 8 * F


def test_stream_plan_refuses_below_minimum():
    from kbbq import _native
    L = _native.lib()
    f, cap = C.c_uint64(), C.c_uint64()
    W = 10_000_000
    # 2 MiB: a quarter for the filter (65536 words), the rest holds 65536 slots (KBBQ_KMER_MIN_SLOTS)
    assert L.kbbq_kmer_stream_plan(W, 2 << 20, C.byref(f), C.byref(cap)) == 0
    assert cap.value == 65536 and f.value == 65536
    # 1 MiB: the filter takes 256 KiB, and 49152 slots are fewer than the smallest table
    assert L.kbbq_kmer_stream_plan(W, 1 << 20, C.byref(f), C.byref(cap)) == _native.E_UNSUPPORTED
    assert L.kbbq_kmer_stream_plan(W, 0, C.byref(f), C.byref(cap)) == _native.E_UNSUPPORTED
    # a small input needs only its exact table
    assert L.kbbq_kmer_stream_plan(10, 8 + 16 * 16, C.byref(f), C.byref(cap)) == 0 and cap.value == 16
    assert L.kbbq_kmer_stream_plan(W, 1 << 30, None, C.byref(cap)) == E_ARG
    with pytest.raises(ValueError, match="does not fit"):
        _native.kmer_stream_plan(W, 1000)


# ---- CPU: argument and order checks that need no device -------------------------------------------------------------

def test_device_entry_points_check_arguments():
    from kbbq import _native
    L = _native.lib()
    p = C.c_void_p(1 << 20)   # never dereferenced: every call below returns before touching the device
    z = C.c_void_p(None)
    assert L.kbbq_kmer_sieve(p, 4, 50, 23, p, 1024, p, 1024, z, z) == E_ARG           # no status word
    assert L.kbbq_kmer_sieve(p, 4, 50, 23, p, 1000, p, 1024, p, z) == E_ARG           # filter not a power of two
    assert L.kbbq_kmer_sieve(p, 4, 50, 23, p, 1024, p, 1000, p, z) == E_ARG           # table not a power of two
    assert L.kbbq_kmer_sieve(p, 4, 50, 32, p, 1024, p, 1024, p, z) == E_ARG           # k > 31
    assert L.kbbq_kmer_sieve(p, 4, 50, 23, z, 1024, p, 1024, p, z) == E_ARG           # no filter
    assert L.kbbq_kmer_sieve(p, 4, 50, 23, C.c_void_p((1 << 20) + 4), 1024, p, 1024, p, z) == E_ARG   # misaligned
    assert L.kbbq_kmer_sieve(z, 0, 50, 23, p, 1024, p, 1024, p, z) == 0               # nothing to do
    assert L.kbbq_kmer_sieve(z, 4, 20, 23, p, 1024, p, 1024, p, z) == 0               # L < k: no windows
    assert L.kbbq_kmer_count_present(p, 4, 50, 23, p, 1024, z, p, z) == E_ARG         # no window counter
    assert L.kbbq_kmer_count_present(p, 4, 50, 0, p, 1024, p, p, z) == E_ARG
    assert L.kbbq_kmer_count_present(z, 0, 50, 23, p, 1024, p, p, z) == 0
    assert L.kbbq_kmer_histogram_sieved(p, 1024, p, z, z) == E_ARG                    # no histogram
    assert L.kbbq_kmer_histogram_sieved(p, 1024, z, p, z) == E_ARG                    # no window counter
    assert L.kbbq_kmer_histogram_sieved(p, 1023, p, p, z) == E_ARG
    assert L.kbbq_kmer_flag_sieved(p, 4, 50, 23, p, 1024, 0, p, p, z) == E_ARG        # t = 0
    assert L.kbbq_kmer_flag_sieved(p, 4, 50, 23, p, 1024, 1, p, z, z) == E_ARG        # t = 1, no status
    assert L.kbbq_kmer_flag_sieved(z, 0, 50, 23, p, 1024, 1, p, p, z) == 0


def test_session_entry_points_check_arguments():
    from kbbq import _native
    L = _native.lib()
    z = C.c_void_p(None)
    assert L.kbbq_session_kmer_begin(z, 23, 100, 0, 0) == E_ARG
    assert L.kbbq_session_kmer_sieve(z, z, 0) == E_ARG
    assert L.kbbq_session_kmer_count(z, z, 0) == E_ARG
    assert L.kbbq_session_kmer_threshold(z, 0, z, None) == E_ARG
    assert L.kbbq_session_build_chunk_kmer(z, z, z, z, z, 0) == E_ARG
    assert L.kbbq_session_kmer_sizes(z, None, None) == E_ARG


# ---- CPU: which driver recalibrate_reads takes ----------------------------------------------------------------------

@pytest.fixture
def small_fastq(tmp_path):
    from kbbq import synth
    seq, qual, _, second = synth.genome_reads(4, 2000, 40, 60, 0.01)
    path = str(tmp_path / "reads.fq")
    synth.write_reads_fastq(path, seq, qual, second)
    return path


def _spy_streamed(monkeypatch):
    from kbbq import recalibrate
    seen = []
    monkeypatch.setattr(recalibrate, "_recalibrate_reads_streamed",
                        lambda reads, infer_rg, k, min_count, batch_reads, device:
                        seen.append(dict(N=reads.N, infer_rg=infer_rg, k=k, min_count=min_count,
                                         batch_reads=batch_reads, device=device)))
    return seen


def test_driver_streams_under_batch_reads(monkeypatch, small_fastq):
    from kbbq import _native, recalibrate
    seen = _spy_streamed(monkeypatch)
    monkeypatch.setattr(_native, "recalibrate_kmer_host", lambda *a, **kw: pytest.fail("single batch taken"))
    monkeypatch.setenv("KBBQ_BATCH_READS", "7")
    recalibrate.recalibrate_reads(small_fastq, infer_rg=True, k=15, min_count=2, devices=[0])
    assert seen == [dict(N=40, infer_rg=True, k=15, min_count=2, batch_reads=7, device=0)]


def test_driver_streams_large_files(monkeypatch, small_fastq):
    from kbbq import _native, recalibrate
    seen = _spy_streamed(monkeypatch)
    monkeypatch.setattr(_native, "recalibrate_kmer_host", lambda *a, **kw: pytest.fail("single batch taken"))
    monkeypatch.delenv("KBBQ_BATCH_READS", raising=False)
    monkeypatch.setattr(recalibrate, "STREAM_ABOVE_BYTES", 100)
    recalibrate.recalibrate_reads(small_fastq)
    assert [s["batch_reads"] for s in seen] == [recalibrate.STREAM_BATCH_READS]


def test_driver_streams_when_the_batch_does_not_fit(monkeypatch, small_fastq):
    from kbbq import _native, recalibrate
    seen = _spy_streamed(monkeypatch)

    def refuse(*a, **kw):
        raise _native.DoesNotFit("does not fit")
    monkeypatch.setattr(_native, "recalibrate_kmer_host", refuse)
    monkeypatch.delenv("KBBQ_BATCH_READS", raising=False)
    recalibrate.recalibrate_reads(small_fastq, k=21)
    assert [(s["k"], s["batch_reads"]) for s in seen] == [(21, recalibrate.STREAM_BATCH_READS)]


def test_driver_single_batch_otherwise(monkeypatch, small_fastq, capfd):
    from kbbq import _native, recalibrate
    seen = _spy_streamed(monkeypatch)
    calls = []

    def fake(seq, qual, rg, second, L, R, minscore, k, min_count, device=None):
        calls.append((seq.shape, k, min_count))
        return np.full(seq.shape, 30, np.uint8), 4
    monkeypatch.setattr(_native, "recalibrate_kmer_host", fake)
    monkeypatch.delenv("KBBQ_BATCH_READS", raising=False)
    recalibrate.recalibrate_reads(small_fastq, k=19, min_count=3)
    assert calls == [((40, 60), 19, 3)] and seen == []
    assert capfd.readouterr().out.count("\n") == 160


def test_streamed_driver_refuses_unequal_lengths(tmp_path, monkeypatch):
    from kbbq import recalibrate
    path = tmp_path / "ragged.fq"
    path.write_text("@a/1\nACGTACGT\n+\nIIIIIIII\n@a/2\nACGTAC\n+\nIIIIII\n")
    monkeypatch.setenv("KBBQ_BATCH_READS", "1")
    with pytest.raises(ValueError, match="unequal length"):
        recalibrate.recalibrate_reads(str(path))


# ---- GPU: the device entry points on torch buffers ------------------------------------------------------------------

class DevSieve:
    """A batch on the device and the exact table of its reads (kbbq_kmer_count), for sieved runs of any size."""

    def __init__(self, seq, L, k):
        import torch
        from kbbq import _native
        self.torch, self.lib, self.native = torch, _native.lib(), _native
        self.N, self.L, self.k = seq.shape[0], L, k
        self.seq = torch.from_numpy(np.ascontiguousarray(seq).ravel()).cuda()
        self.stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        self.exact_cap = _native.kmer_table_bytes(self.N, L, k)[0]
        table = self.buf(2 * self.exact_cap)
        status = torch.zeros(1, dtype=torch.int32, device="cuda")
        self.ok(self.lib.kbbq_kmer_clear(self.p(table), self.exact_cap, self.stream))
        self.ok(self.lib.kbbq_kmer_count(self.p(self.seq), self.N, L, k, self.p(table), self.exact_cap, self.p(status),
                                         self.stream))
        assert int(status.cpu()[0]) == 0
        self.exact = self.entries(table)

    def buf(self, n):
        return self.torch.empty(n, dtype=self.torch.int64, device="cuda")

    def p(self, t, off=0):
        return C.c_void_p(t.data_ptr() + off)

    def ok(self, rc):
        self.native.check(rc)

    @staticmethod
    def entries(table):
        t = table.cpu().numpy().view(np.uint64).reshape(-1, 2)
        t = t[t[:, 0] != np.uint64(2 ** 64 - 1)]
        return t[np.argsort(t[:, 0])]

    def run(self, filter_words, cap, chunks, min_count):
        """Sieve and count-present over the chunks (read counts), histogram, threshold, flags.
        -> (hist, t, bits, entries, status, windows)"""
        torch, lib, L, k = self.torch, self.lib, self.L, self.k
        filt = torch.zeros(filter_words, dtype=torch.int64, device="cuda")
        table = self.buf(2 * cap)
        status = torch.zeros(1, dtype=torch.int32, device="cuda")
        windows = torch.zeros(1, dtype=torch.int64, device="cuda")
        hist = torch.zeros(256, dtype=torch.int64, device="cuda")
        bits = torch.full(((self.N * L + 31) // 32,), -1, dtype=torch.int32, device="cuda")
        self.ok(lib.kbbq_kmer_clear(self.p(table), cap, self.stream))
        assert sum(chunks) == self.N
        for count in (False, True):
            r0 = 0
            for n in chunks:
                s = self.p(self.seq, r0 * L)
                if count:
                    self.ok(lib.kbbq_kmer_count_present(s, n, L, k, self.p(table), cap, self.p(windows),
                                                        self.p(status), self.stream))
                else:
                    self.ok(lib.kbbq_kmer_sieve(s, n, L, k, self.p(filt), filter_words, self.p(table), cap,
                                                self.p(status), self.stream))
                r0 += n
        self.ok(lib.kbbq_kmer_histogram_sieved(self.p(table), cap, self.p(windows), self.p(hist), self.stream))
        h = hist.cpu().numpy().astype(np.uint64)
        t = min_count or self.native.kmer_min_count(h)
        self.ok(lib.kbbq_kmer_flag_sieved(self.p(self.seq), self.N, L, k, self.p(table), cap, t, self.p(bits),
                                          self.p(status), self.stream))
        return (h, t, bits.cpu().numpy().view(np.uint32), self.entries(table), int(status.cpu()[0]),
                int(windows.cpu()[0]))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [15, 23, 31])
@pytest.mark.parametrize("L", [33, 100, 151])
@pytest.mark.parametrize("min_count", [0, 1, 3])
def test_gpu_sieved_matches_oracle(kmer_oracle, k, L, min_count):
    from kbbq import _native
    seq, _, _, n = batch(k, L)
    want_bits, want_hist, want_t = kmer_oracle.kmer_errors(seq, L, k, min_count)
    assert want_bits.any() or min_count == 1   # t = 1: every valid window is solid
    d = DevSieve(seq, L, k)
    exact_keys, exact_counts = d.exact[:, 0], d.exact[:, 1]
    W = int(exact_counts.sum())
    planned = _native.kmer_stream_plan(W, 2 << 20)   # 2 MiB: the smallest table, far below the exact rule's
    assert planned[1] < d.exact_cap
    for filter_words, cap in ((1, d.exact_cap), (1 << 10, d.exact_cap), planned):
        for chunks in ([n], [1, 33, n - 34]):
            hist, t, bits, ent, status, windows = d.run(filter_words, cap, chunks, min_count)
            where = (filter_words, cap, chunks)
            assert status == 0, where
            assert windows == W, where
            assert np.array_equal(hist, want_hist), where
            assert t == want_t, where
            assert np.array_equal(bits, want_bits), where
            # every key seen twice or more is there with its exact count; any other key present was seen once
            assert (ent[:, 1] >= 1).all(), where
            i = np.searchsorted(exact_keys, ent[:, 0])
            assert (i < exact_keys.size).all() and np.array_equal(exact_keys[i], ent[:, 0]), where
            assert np.array_equal(ent[:, 1], exact_counts[i]), where
            assert np.isin(exact_keys[exact_counts >= 2], ent[:, 0]).all(), where
            if filter_words == 1:   # one filter word: almost every key seen once is a false positive
                assert (ent[:, 1] == 1).sum() > 0.9 * (exact_counts == 1).sum(), where


@pytest.mark.gpu
def test_gpu_sieve_full_table():
    """A sieved table too small for the repeated k-mers raises KBBQ_FLAG_KMER_FULL."""
    from kbbq import _native
    seq, _, _, n = batch(23, 100)
    d = DevSieve(seq, 100, 23)
    status = d.run(1 << 10, 64, [n], 3)[4]
    assert status & _native.FLAG_KMER_FULL


# ---- GPU: sessions --------------------------------------------------------------------------------------------------

def _session_run(seq, qual, rg, second, L, R, k, min_count, chunk):
    """The streamed path through a Session -> (out, tables, deltas, t, hist)"""
    from kbbq import _native
    n = seq.shape[0]
    with _native.Session(L, R, 6, chunk_reads=chunk, resident_reads=0) as s:
        s.kmer_begin(k, n * max(0, L - k + 1))
        C_ = s.chunk_reads
        spans = [(lo, min(C_, n - lo)) for lo in range(0, n, C_)]
        for lo, m in spans:
            s.kmer_sieve(seq[lo:lo + m])
        for lo, m in spans:
            s.kmer_count(seq[lo:lo + m])
        t, hist = s.kmer_threshold(min_count)
        for lo, m in spans:
            s.build_chunk_kmer(seq[lo:lo + m], qual[lo:lo + m], rg[lo:lo + m], second[lo:lo + m])
        deltas = s.model(want_deltas=True)
        tables = s.tables()
        out = np.zeros((n, L), np.uint8)
        for lo, m in spans:
            s.apply_chunk(seq[lo:lo + m], qual[lo:lo + m], rg[lo:lo + m], second[lo:lo + m], out[lo:lo + m])
        s.sync()
    return out, tables, deltas, t, hist


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [16, 1000, "all"])
@pytest.mark.parametrize("R", [1, 3])
@pytest.mark.parametrize("k,L,min_count", [(23, 150, 0), (15, 100, 1), (31, 151, 3)])
def test_gpu_session_matches_single_batch(kmer_oracle, chunk, R, k, L, min_count):
    from kbbq import _native
    seq, qual, second, n = batch(k, L, seed=9, lower=0.0)   # lowercase is a bad base to the build
    rg = (np.arange(n) // 2 % R).astype(np.uint16)
    chunk = n if chunk == "all" else chunk
    want_out, want_t, want_tabs, want_deltas = _native.recalibrate_kmer_host(seq, qual, rg, second, L, R, 6, k,
                                                                             min_count, want_tables=True)
    out, tables, deltas, t, hist = _session_run(seq, qual, rg, second, L, R, k, min_count, chunk)
    assert t == want_t == kmer_oracle.kmer_errors(seq, L, k, min_count)[2]
    assert np.array_equal(hist, kmer_oracle.kmer_errors(seq, L, k, min_count)[1])
    assert np.array_equal(out, want_out)
    assert np.array_equal(tables, np.concatenate([a.ravel() for a in want_tabs]))
    for a, b in zip(deltas, want_deltas):
        assert np.array_equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("capacity", [64, 1 << 12])
def test_gpu_session_full_table_raises_memory_error(capacity):
    """A table that fills in pass A is reported when pass B starts, not after it."""
    from kbbq import _native
    seq, _, _, n = batch(23, 100)
    with _native.Session(100, 1, 6, chunk_reads=512, resident_reads=0) as s:
        s.kmer_begin(23, n * 78, filter_words=1024, capacity=capacity)
        assert s.kmer_sizes() == (1024, capacity)
        for lo in range(0, n, 512):
            s.kmer_sieve(seq[lo:lo + 512])
        with pytest.raises(MemoryError, match="%d slots" % capacity):
            s.kmer_count(seq[:512])
        with pytest.raises(MemoryError):
            s.kmer_threshold()
        with pytest.raises(MemoryError):   # the status word says why
            s.sync()


@pytest.mark.gpu
def test_gpu_count_present_stops_on_a_table_without_empty_slot():
    """Pass B on a table with no empty slot: a probe for an absent key raises KBBQ_FLAG_KMER_FULL (instead of walking
    the whole table for every such window) and nothing is added to the keys that are there."""
    import torch
    from kbbq import _native
    seq, _, _, n = batch(23, 100)
    d = DevSieve(seq, 100, 23)
    cap = 64
    table = d.buf(2 * cap)
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    windows = torch.zeros(1, dtype=torch.int64, device="cuda")
    d.ok(d.lib.kbbq_kmer_clear(d.p(table), cap, d.stream))
    d.ok(d.lib.kbbq_kmer_count(d.p(d.seq), 4, 100, 23, d.p(table), cap, d.p(status), d.stream))   # fills every slot
    before = d.entries(table)
    assert before.shape[0] == cap
    status.zero_()
    d.ok(d.lib.kbbq_kmer_count_present(d.p(d.seq, 1000 * 100), n - 1000, 100, 23, d.p(table), cap, d.p(windows),
                                       d.p(status), d.stream))
    assert int(status.cpu()[0]) & _native.FLAG_KMER_FULL


@pytest.mark.gpu
def test_gpu_session_calls_out_of_order():
    from kbbq import _native
    L_ = _native.lib()
    seq, qual, second, n = batch(23, 100, lower=0.0)
    seq, qual, second = seq[:64], qual[:64], second[:64]
    p = _native.ptr
    with _native.Session(100, 1, 6, chunk_reads=64, resident_reads=64) as res:   # chunks kept resident: not this path
        assert L_.kbbq_session_kmer_begin(res.h, 23, 64 * 78, 0, 0) == E_ARG
    with _native.Session(100, 1, 6, chunk_reads=64, resident_reads=0) as s:
        h = s.h
        assert L_.kbbq_session_kmer_sieve(h, p(seq), 64) == E_ARG                  # before begin
        assert L_.kbbq_session_kmer_count(h, p(seq), 64) == E_ARG
        assert L_.kbbq_session_kmer_threshold(h, 0, None, None) == E_ARG
        assert L_.kbbq_session_build_chunk_kmer(h, p(seq), p(qual), None, p(second), 64) == E_ARG
        assert L_.kbbq_session_kmer_begin(h, 23, 64 * 78, 1000, 1024) == E_ARG    # not a power of two
        assert L_.kbbq_session_kmer_begin(h, 23, 64 * 78, 1024, 0) == E_ARG       # one size without the other
        assert L_.kbbq_session_kmer_begin(h, 0, 64 * 78, 0, 0) == E_ARG
        s.kmer_begin(23, 64 * 78)
        assert L_.kbbq_session_kmer_begin(h, 23, 64 * 78, 0, 0) == E_ARG          # twice
        # the plain passes do not mix with the k-mer passes before the threshold
        assert L_.kbbq_session_build_chunk(h, p(seq), p(qual), p(seq), None, p(second), 64, 0) == E_ARG
        assert L_.kbbq_session_build_range(h, p(seq), p(qual), p(seq), None, p(second), 64) == E_ARG
        out = np.zeros((64, 100), np.uint8)
        assert L_.kbbq_session_apply_chunk(h, p(seq), p(qual), None, p(second), 64, p(out)) == E_ARG
        assert L_.kbbq_session_kmer_sieve(h, p(seq), 65) == E_ARG                 # more than a chunk
        assert L_.kbbq_session_kmer_threshold(h, 0, None, None) == E_ARG          # before pass B
        s.kmer_sieve(seq)
        assert L_.kbbq_session_build_chunk_kmer(h, p(seq), p(qual), None, p(second), 64) == E_ARG
        s.kmer_count(seq)
        assert L_.kbbq_session_kmer_sieve(h, p(seq), 64) == E_ARG                 # sieving after counting
        assert L_.kbbq_session_build_chunk_kmer(h, p(seq), p(qual), None, p(second), 64) == E_ARG
        t, _ = s.kmer_threshold()
        assert L_.kbbq_session_kmer_threshold(h, 0, None, None) == E_ARG          # twice
        assert L_.kbbq_session_kmer_count(h, p(seq), 64) == E_ARG                 # counting after the threshold
        s.build_chunk_kmer(seq, qual, None, second)
        s.model()
        s.sync()
        s.reset()   # releases the k-mer buffers: a new run may begin
        s.kmer_begin(23, 64 * 78)
        assert s.kmer_sizes()[1] >= 1


# ---- GPU: the CLI ---------------------------------------------------------------------------------------------------

def _main(monkeypatch, argv):
    import kbbq.main
    with monkeypatch.context() as m:
        m.setattr(sys, "argv", [sys.argv[0], "recalibrate"] + argv)
        kbbq.main.main()


@pytest.mark.gpu
@pytest.mark.parametrize("infer_rg", [False, True])
def test_gpu_cli_streamed_equals_single_batch(tmp_path, monkeypatch, capfd, infer_rg):
    """`kbbq recalibrate -r` prints the same bytes whether the file goes through as one batch or streams in batches
    of a size that does not divide it, on a file of three read groups."""
    from kbbq import synth
    L, G = 150, 20_000
    n = 30 * G // L
    seq, qual, _, second = synth.genome_reads(23, G, n, L, 0.01, 0.002)
    rg = (np.arange(n) // 2 % 3).astype(np.uint16)
    reads = str(tmp_path / "reads.fq")
    synth.write_fastq(reads, str(tmp_path / "unused.fq"), seq, qual, seq, rg, second, infer_rg=True)
    argv = ["-r", reads] + (["--infer-rg"] if infer_rg else [])
    monkeypatch.delenv("KBBQ_BATCH_READS", raising=False)
    capfd.readouterr()
    _main(monkeypatch, argv)
    want = capfd.readouterr().out
    assert n % 997 and want.count("\n") == 4 * n
    monkeypatch.setenv("KBBQ_BATCH_READS", "997")
    _main(monkeypatch, argv)
    got = capfd.readouterr().out
    assert got == want
