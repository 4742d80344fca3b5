"""`kbbq recalibrate -r` streamed with its sieved k-mer table split by key across GPUs (DESIGN.md §10, "Several GPUs"):
the partition entry points (kbbq_kmer_sieve_part / _count_present_part / _flag_parts / _correct_parts), the session
(kbbq_session_kmer_begin_parts) and the driver.  Every GPU comparison is bit for bit, against the C oracles, an exact
table of the same reads and the single-batch path.  One GPU listed several times runs every partition path; the tests
that need two GPUs are skipped below that."""
import ctypes as C
import importlib.util
import os
import sys

import numpy as np
import pytest

E_ARG, E_PEER = -1, -11
HERE = os.path.dirname(os.path.abspath(__file__))
EMPTY = np.uint64(2 ** 64 - 1)


def _load(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(HERE, name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="module")
def kmer_oracle():
    return _load("kmer_oracle")


@pytest.fixture(scope="module")
def walk_oracle():
    return _load("kmer_correct_oracle")


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


def owner(keys, n):
    """The partition of each key: ((splitmix64(key) >> 32) * n) >> 32, restated in numpy."""
    x = np.asarray(keys, np.uint64).copy()
    with np.errstate(over="ignore"):
        x ^= x >> np.uint64(30)
        x *= np.uint64(0xBF58476D1CE4E5B9)
        x ^= x >> np.uint64(27)
        x *= np.uint64(0x94D049BB133111EB)
        x ^= x >> np.uint64(31)
    return ((x >> np.uint64(32)) * np.uint64(n)) >> np.uint64(32)


# ---- CPU: the rule and the argument checks that need no device ------------------------------------------------------

def test_owner_rule_spreads_keys():
    keys = np.random.default_rng(0).integers(0, 1 << 46, 1 << 16, dtype=np.uint64)
    assert (owner(keys, 1) == 0).all()
    for n in (2, 3, 8, 16):
        share = np.bincount(owner(keys, n).astype(np.int64), minlength=n) / keys.size
        assert share.size == n and abs(share - 1 / n).max() < 0.01


def test_device_entry_points_check_arguments():
    from kbbq import _native
    L = _native.lib()
    p = C.c_void_p(1 << 20)   # never dereferenced: every call below returns before touching the device
    z = C.c_void_p(None)
    big = (1 << 32) * 2
    for part, n in ((0, 0), (0, 17), (-1, 2), (2, 2)):
        assert L.kbbq_kmer_sieve_part(p, 4, 50, 23, part, n, p, 1024, p, 1024, p, z) == E_ARG
        assert L.kbbq_kmer_count_present_part(p, 4, 50, 23, part, n, p, 1024, p, p, z) == E_ARG
    assert L.kbbq_kmer_sieve_part(p, 4, 50, 23, 1, 2, p, 1024, p, big, p, z) == E_ARG       # slots past 2^32
    assert L.kbbq_kmer_count_present_part(p, 4, 50, 23, 1, 2, p, big, p, p, z) == E_ARG
    assert L.kbbq_kmer_sieve_part(p, 4, 50, 23, 1, 2, p, 1024, z, 1024, p, z) == E_ARG      # no table
    assert L.kbbq_kmer_sieve_part(p, 4, 50, 23, 1, 2, p, 1000, p, 1024, p, z) == E_ARG      # as kbbq_kmer_sieve
    assert L.kbbq_kmer_count_present_part(p, 4, 50, 23, 1, 2, p, 1024, z, p, z) == E_ARG    # no window counter
    assert L.kbbq_kmer_sieve_part(z, 0, 50, 23, 1, 2, p, 1024, p, 1024, p, z) == 0          # nothing to do
    assert L.kbbq_kmer_count_present_part(z, 4, 20, 23, 1, 2, p, 1024, p, p, z) == 0        # L < k
    two = (C.c_void_p * 2)(p, p)
    one_null = (C.c_void_p * 2)(p, None)
    for fn in (L.kbbq_kmer_flag_parts, L.kbbq_kmer_correct_parts):
        assert fn(p, 4, 50, 23, z, 2, 1024, 3, p, p, z) == E_ARG                           # no table set
        assert fn(p, 4, 50, 23, one_null, 2, 1024, 3, p, p, z) == E_ARG                    # a NULL table
        assert fn(p, 4, 50, 23, two, 0, 1024, 3, p, p, z) == E_ARG
        assert fn(p, 4, 50, 23, two, 17, 1024, 3, p, p, z) == E_ARG
        assert fn(p, 4, 50, 23, two, 2, big, 3, p, p, z) == E_ARG
        assert fn(p, 4, 50, 23, two, 2, 1000, 3, p, p, z) == E_ARG                         # not a power of two
        assert fn(p, 4, 50, 23, two, 2, 1024, 0, p, p, z) == E_ARG                         # t = 0
        assert fn(p, 4, 50, 23, two, 2, 1024, 3, p, z, z) == E_ARG                         # no status
        assert fn(z, 0, 50, 23, two, 2, 1024, 3, p, p, z) == 0


def test_session_begin_parts_checks_arguments():
    from kbbq import _native
    L = _native.lib()
    z = C.c_void_p(None)
    devs = (C.c_int * 2)(0, 0)
    assert L.kbbq_session_kmer_begin_parts(z, 23, 100, 0, 0, devs, 2) == E_ARG


# ---- CPU: the driver ------------------------------------------------------------------------------------------------

@pytest.fixture
def small_fastq(tmp_path):
    from kbbq import synth
    seq, qual, _, second = synth.genome_reads(4, 2000, 40, 60, 0.01)
    path = str(tmp_path / "reads.fq")
    synth.write_reads_fastq(path, seq, qual, second)
    return path


def test_driver_passes_devices_to_the_streamed_path(monkeypatch, small_fastq):
    from kbbq import _native, recalibrate
    seen = []
    monkeypatch.setattr(recalibrate, "_recalibrate_reads_streamed",
                        lambda reads, infer_rg, k, min_count, batch_reads, device, **kw:
                        seen.append(dict(batch_reads=batch_reads, device=device, **kw)))
    monkeypatch.setattr(_native, "recalibrate_kmer_host", lambda *a, **kw: pytest.fail("single batch taken"))
    monkeypatch.setenv("KBBQ_BATCH_READS", "7")
    recalibrate.recalibrate_reads(small_fastq, devices=[2, 0, 2])
    recalibrate.recalibrate_reads(small_fastq, devices=[1], correct=True)
    monkeypatch.setenv("KBBQ_DEVICES", "3,1")
    recalibrate.recalibrate_reads(small_fastq)
    assert seen == [dict(batch_reads=7, device=2, devices=[2, 0, 2]), dict(batch_reads=7, device=1, correct=True),
                    dict(batch_reads=7, device=3, devices=[3, 1])]


def test_driver_single_batch_stays_on_the_first_device(monkeypatch, small_fastq, capfd):
    from kbbq import _native, recalibrate
    monkeypatch.setattr(recalibrate, "_recalibrate_reads_streamed", lambda *a, **kw: pytest.fail("streamed"))
    calls = []

    def single(seq, qual, rg, second, L, R, minscore, k, min_count, device=None):
        calls.append(device)
        return np.full(seq.shape, 30, np.uint8), 4
    monkeypatch.setattr(_native, "recalibrate_kmer_host", single)
    monkeypatch.delenv("KBBQ_BATCH_READS", raising=False)
    recalibrate.recalibrate_reads(small_fastq, devices=[1, 0, 1])
    assert calls == [1]
    assert capfd.readouterr().out.count("\n") == 160


class FakeSession:
    """Records what the streamed driver asks of a Session; kmer_begin over several devices raises PeerUnreachable."""

    def __init__(self, log, *a, **kw):
        self.log = log
        log.append(("session", kw.get("device")))

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        pass

    def kmer_begin(self, k, windows, devices=None):
        from kbbq import _native
        self.log.append(("begin", devices))
        if devices is not None:
            raise _native.PeerUnreachable("no peer")

    def __getattr__(self, name):
        return lambda *a, **kw: self.log.append((name,))


def test_driver_falls_back_to_one_partition(monkeypatch, small_fastq):
    from kbbq import _native, fastx, recalibrate
    log = []
    monkeypatch.setattr(_native, "Session", lambda *a, **kw: FakeSession(log, *a, **kw))
    monkeypatch.setattr(recalibrate, "_apply_pass", lambda *a: log.append(("apply",)))
    reads = fastx.NativeFastq(small_fastq)
    try:
        recalibrate._recalibrate_reads_streamed(reads, False, 15, 0, 16, 2, devices=[2, 2, 5])
    finally:
        reads.close()
    assert log[:3] == [("session", 2), ("begin", [2, 2, 5]), ("begin", None)]
    assert ("kmer_threshold",) in log and log[-1] == ("apply",)


# ---- GPU: the partition entry points on torch buffers ---------------------------------------------------------------

class DevParts:
    """A batch on the device, the exact table of its reads (kbbq_kmer_count), and runs of the partition passes."""

    def __init__(self, seq, L, k):
        import torch
        from kbbq import _native
        self.torch, self.lib, self.native = torch, _native.lib(), _native
        self.N, self.L, self.k = seq.shape[0], L, k
        self.seq = torch.from_numpy(np.ascontiguousarray(seq).ravel()).cuda()
        self.stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        self.exact_cap = _native.kmer_table_bytes(self.N, L, k)[0]
        table = self.buf(2 * self.exact_cap)
        status = self.zeros(1, torch.int32)
        self.ok(self.lib.kbbq_kmer_clear(self.p(table), self.exact_cap, self.stream))
        self.ok(self.lib.kbbq_kmer_count(self.p(self.seq), self.N, L, k, self.p(table), self.exact_cap, self.p(status),
                                         self.stream))
        assert int(status.cpu()[0]) == 0
        self.exact = self.entries(table)

    def buf(self, n):
        return self.torch.empty(n, dtype=self.torch.int64, device="cuda")

    def zeros(self, n, dtype=None):
        return self.torch.zeros(n, dtype=dtype or self.torch.int64, device="cuda")

    def p(self, t, off=0):
        return C.c_void_p(t.data_ptr() + off)

    def ok(self, rc):
        self.native.check(rc)

    @staticmethod
    def entries(table):
        t = table.cpu().numpy().view(np.uint64).reshape(-1, 2)
        t = t[t[:, 0] != EMPTY]
        return t[np.argsort(t[:, 0])]

    def run(self, n_parts, filter_words, cap, chunks):
        """Passes A and B of every partition over the chunks, and each partition's sieved histogram.
        -> (tables, hists, windows, status)"""
        lib, L, k = self.lib, self.L, self.k
        tables = [self.buf(2 * cap) for _ in range(n_parts)]
        filters = [self.zeros(filter_words) for _ in range(n_parts)]
        windows = [self.zeros(1) for _ in range(n_parts)]
        hists = [self.zeros(256) for _ in range(n_parts)]
        status = self.zeros(n_parts, self.torch.int32)
        for t in tables:
            self.ok(lib.kbbq_kmer_clear(self.p(t), cap, self.stream))
        assert sum(chunks) == self.N
        for count in (False, True):
            r0 = 0
            for n in chunks:
                s = self.p(self.seq, r0 * L)
                for q in range(n_parts):
                    st = self.p(status, 4 * q)
                    if count:
                        self.ok(lib.kbbq_kmer_count_present_part(s, n, L, k, q, n_parts, self.p(tables[q]), cap,
                                                                 self.p(windows[q]), st, self.stream))
                    else:
                        self.ok(lib.kbbq_kmer_sieve_part(s, n, L, k, q, n_parts, self.p(filters[q]), filter_words,
                                                         self.p(tables[q]), cap, st, self.stream))
                r0 += n
        for q in range(n_parts):
            self.ok(lib.kbbq_kmer_histogram_sieved(self.p(tables[q]), cap, self.p(windows[q]), self.p(hists[q]),
                                                   self.stream))
        return (tables, [h.cpu().numpy().astype(np.uint64) for h in hists], [int(w.cpu()[0]) for w in windows],
                status.cpu().numpy())

    def map(self, call):
        """A map call(seq, bits, status) over the whole batch -> (bits, status)"""
        bits = self.torch.full(((self.N * self.L + 31) // 32,), -1, dtype=self.torch.int32, device="cuda")
        status = self.zeros(1, self.torch.int32)
        self.ok(call(self.p(self.seq), self.p(bits), self.p(status)))
        return bits.cpu().numpy().view(np.uint32), int(status.cpu()[0])

    def map_parts(self, fn, tables, cap, t):
        """kbbq_kmer_flag_parts / _correct_parts -> (bits, status)"""
        ptrs = (C.c_void_p * len(tables))(*[x.data_ptr() for x in tables])
        return self.map(lambda s, b, st: fn(s, self.N, self.L, self.k, ptrs, len(tables), cap, t, b, st, self.stream))

    def map_one(self, fn, table, cap, t):
        """kbbq_kmer_flag_sieved / kbbq_kmer_correct on one table -> (bits, status)"""
        return self.map(lambda s, b, st: fn(s, self.N, self.L, self.k, self.p(table), cap, t, b, st, self.stream))


@pytest.mark.gpu
@pytest.mark.parametrize("n_parts", [1, 2, 3, 8])
@pytest.mark.parametrize("k", [15, 23, 31])
@pytest.mark.parametrize("L", [33, 100, 151])
def test_gpu_parts_match_oracle(kmer_oracle, walk_oracle, n_parts, k, L):
    """Every partition holds only its own keys; together they hold every repeated key with its exact count; the sum
    of their histograms is the exact one; the maps equal the oracles' for t in {0, 1, 3}."""
    from kbbq import _native
    seq, _, _, n = batch(k, L)
    d = DevParts(seq, L, k)
    exact_keys, exact_counts = d.exact[:, 0], d.exact[:, 1]
    W = int(exact_counts.sum())
    want = {t: (kmer_oracle.kmer_errors(seq, L, k, t), walk_oracle.kmer_corrections(seq, L, k, t)) for t in (0, 1, 3)}
    planned = _native.kmer_stream_plan(-(-W // n_parts), 2 << 20)
    for filter_words, cap in ((1, d.exact_cap), planned):
        for chunks in ([n], [1, 33, n - 34]):
            where = (n_parts, filter_words, cap, chunks)
            tables, hists, windows, status = d.run(n_parts, filter_words, cap, chunks)
            assert not status.any(), where
            assert sum(windows) == W, where
            ents = [d.entries(t) for t in tables]
            for q, ent in enumerate(ents):
                assert (owner(ent[:, 0], n_parts) == q).all(), where
                i = np.searchsorted(exact_keys, ent[:, 0])
                assert (i < exact_keys.size).all() and np.array_equal(exact_keys[i], ent[:, 0]), where
                assert np.array_equal(ent[:, 1], exact_counts[i]), where
                # W_p: the valid windows whose keys the partition owns
                assert windows[q] == int(exact_counts[owner(exact_keys, n_parts) == q].sum()), where
            repeated = np.concatenate([e[e[:, 1] >= 2] for e in ents])
            repeated = repeated[np.argsort(repeated[:, 0])]
            assert np.array_equal(repeated, d.exact[exact_counts >= 2]), where
            hist = np.sum(hists, axis=0, dtype=np.uint64)
            for t_arg, ((bits_b, want_hist, want_t), (bits_c, _, _)) in want.items():
                assert np.array_equal(hist, want_hist), where
                t = t_arg or _native.kmer_min_count(hist)
                assert t == want_t, where
                got_b, st_b = d.map_parts(d.lib.kbbq_kmer_flag_parts, tables, cap, t)
                got_c, st_c = d.map_parts(d.lib.kbbq_kmer_correct_parts, tables, cap, t)
                assert st_b == st_c == 0, where
                assert np.array_equal(got_b, bits_b), (where, t)
                assert np.array_equal(got_c, bits_c), (where, t)
                if n_parts == 1:   # the single-table calls
                    assert np.array_equal(d.map_one(d.lib.kbbq_kmer_flag_sieved, tables[0], cap, t)[0], got_b), where
                    assert np.array_equal(d.map_one(d.lib.kbbq_kmer_correct, tables[0], cap, t)[0], got_c), where


@pytest.mark.gpu
def test_gpu_part_full_table():
    """A partition too small for its repeated k-mers raises KBBQ_FLAG_KMER_FULL in its status word."""
    from kbbq import _native
    seq, _, _, n = batch(23, 100)
    d = DevParts(seq, 100, 23)
    status = d.run(3, 1 << 10, 64, [n])[3]
    assert (status & _native.FLAG_KMER_FULL).all()


# ---- GPU: sessions --------------------------------------------------------------------------------------------------

def _session_run(seq, qual, rg, second, L, R, k, min_count, chunk, devices, correct=False):
    """The streamed path through a Session with the table over `devices` -> (out, tables, deltas, t, hist, sizes)"""
    from kbbq import _native
    n = seq.shape[0]
    with _native.Session(L, R, 6, chunk_reads=chunk, resident_reads=0, device=devices[0]) as s:
        s.kmer_begin(k, n * max(0, L - k + 1), devices=devices)
        if correct:
            s.kmer_rule(_native.KMER_CORRECT)
        sizes = s.kmer_sizes()
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
    return out, tables, deltas, t, hist, sizes


def _check_session(kmer_oracle, seq, qual, second, n, R, k, L, min_count, chunk, device_lists, correct):
    from kbbq import _native
    rg = (np.arange(n) // 2 % R).astype(np.uint16)
    want_out, want_t, want_tabs, want_deltas = _native.recalibrate_kmer_host(seq, qual, rg, second, L, R, 6, k,
                                                                             min_count, want_tables=True,
                                                                             **({"correct": True} if correct else {}))
    want_hist = kmer_oracle.kmer_errors(seq, L, k, min_count)[1]
    for devices in device_lists:
        out, tables, deltas, t, hist, sizes = _session_run(seq, qual, rg, second, L, R, k, min_count, chunk, devices,
                                                           correct)
        assert t == want_t, devices
        assert np.array_equal(hist, want_hist), devices
        assert np.array_equal(out, want_out), devices
        assert np.array_equal(tables, np.concatenate([a.ravel() for a in want_tabs])), devices
        for a, b in zip(deltas, want_deltas):
            assert np.array_equal(a, b), devices
        assert len(devices) == 1 or sizes[1] <= 1 << 32


@pytest.mark.gpu
@pytest.mark.parametrize("correct", [False, True])
@pytest.mark.parametrize("chunk", [16, 1000, "all"])
@pytest.mark.parametrize("R", [1, 3])
def test_gpu_session_parts_match_single_batch(kmer_oracle, correct, chunk, R):
    """Sessions with the table on [d], [d, d], [d, d, d] and [d] x 8 print what kbbq_recalibrate_kmer_rule_host
    prints, with the same tables, deltas, threshold and histogram."""
    from kbbq import _native
    k, L = 23, 150
    seq, qual, second, n = batch(k, L, seed=9, lower=0.0)   # lowercase is a bad base to the build
    chunk = n if chunk == "all" else chunk
    d = _native.DEVICE
    _check_session(kmer_oracle, seq, qual, second, n, R, k, L, 0, chunk, [[d], [d, d], [d, d, d], [d] * 8], correct)


@pytest.mark.gpu
def test_gpu_session_part_full_table_raises_memory_error():
    from kbbq import _native
    seq, _, _, n = batch(23, 100)
    d = _native.DEVICE
    with _native.Session(100, 1, 6, chunk_reads=512, resident_reads=0, device=d) as s:
        s.kmer_begin(23, n * 78, filter_words=1024, capacity=64, devices=[d, d, d])
        assert s.kmer_sizes() == (1024, 64)
        for lo in range(0, n, 512):
            s.kmer_sieve(seq[lo:lo + 512])
        with pytest.raises(MemoryError, match="3 partitions of 64 slots"):
            s.kmer_count(seq[:512])
        with pytest.raises(MemoryError):
            s.kmer_threshold()
        with pytest.raises(MemoryError):
            s.sync()


@pytest.mark.gpu
def test_gpu_session_begin_parts_refuses(monkeypatch):
    import torch
    from kbbq import _native
    L_ = _native.lib()
    d = _native.DEVICE
    devs = lambda *x: (C.c_int * len(x))(*x)
    with _native.Session(100, 1, 6, chunk_reads=64, resident_reads=64, device=d) as res:   # chunks kept resident
        assert L_.kbbq_session_kmer_begin_parts(res.h, 23, 64 * 78, 0, 0, devs(d, d), 2) == E_ARG
    with _native.Session(100, 1, 6, chunk_reads=64, resident_reads=0, device=d) as s:
        other = torch.cuda.device_count()   # not a device of this box
        assert L_.kbbq_session_kmer_begin_parts(s.h, 23, 64 * 78, 0, 0, devs(other, d), 2) == E_ARG   # not devices[0]
        assert L_.kbbq_session_kmer_begin_parts(s.h, 23, 64 * 78, 0, 0, devs(d, other), 2) == E_ARG
        assert L_.kbbq_session_kmer_begin_parts(s.h, 23, 64 * 78, 0, 0, devs(d), 0) == E_ARG
        assert L_.kbbq_session_kmer_begin_parts(s.h, 23, 64 * 78, 0, 0, devs(*[d] * 17), 17) == E_ARG
        assert L_.kbbq_session_kmer_begin_parts(s.h, 23, 64 * 78, 0, 0, None, 2) == E_ARG
        assert L_.kbbq_session_kmer_begin_parts(s.h, 23, 64 * 78, 1024, 1 << 33, devs(d, d), 2) == E_ARG
        monkeypatch.setenv("KBBQ_MULTI_NO_P2P", "1")
        assert L_.kbbq_session_kmer_begin_parts(s.h, 23, 64 * 78, 0, 0, devs(d, d), 2) == E_PEER
        with pytest.raises(_native.PeerUnreachable):
            s.kmer_begin(23, 64 * 78, devices=[d, d])
        assert s.kmer_sizes() == (0, 0)   # nothing allocated
        s.kmer_begin(23, 64 * 78, devices=[d])   # one partition needs no peer
        assert L_.kbbq_session_kmer_begin_parts(s.h, 23, 64 * 78, 0, 0, devs(d, d), 2) == E_ARG   # twice
        s.reset()
        monkeypatch.delenv("KBBQ_MULTI_NO_P2P")
        s.kmer_begin(23, 64 * 78, devices=[d, d])
        f, cap = s.kmer_sizes()
        assert f >= 1 and 1 <= cap <= 1 << 32
        s.reset()   # releases every partition: a new run may begin
        s.kmer_begin(23, 64 * 78, devices=[d] * 4)


@pytest.mark.gpu
def test_gpu_session_sizes_split_the_windows():
    """filter_words = capacity = 0: each of n partitions is planned for ceil(windows / n) windows."""
    from kbbq import _native
    d = _native.DEVICE
    W = 10_000_000
    with _native.Session(150, 1, 6, chunk_reads=1 << 16, resident_reads=0, device=d) as s:
        s.kmer_begin(23, W)
        one = s.kmer_sizes()
        s.reset()
        s.kmer_begin(23, W, devices=[d, d])
        two = s.kmer_sizes()
    assert one == (1 << 20, 1 << 24)   # the filter: 8 F <= W bytes; the table: the exact capacity
    assert two == (1 << 19, 1 << 23)


# ---- GPU: the CLI ---------------------------------------------------------------------------------------------------

def _main(monkeypatch, argv):
    import kbbq.main
    with monkeypatch.context() as m:
        m.setattr(sys, "argv", [sys.argv[0], "recalibrate"] + argv)
        kbbq.main.main()


@pytest.mark.gpu
@pytest.mark.parametrize("correct", [False, True])
def test_gpu_cli_parts_same_bytes(tmp_path, monkeypatch, capfd, correct):
    """`kbbq recalibrate -r` streamed with KBBQ_DEVICES=d,d,d prints what KBBQ_DEVICES=d prints, with peer access and
    without it (one partition then)."""
    from kbbq import _native, synth
    L, G = 150, 20_000
    n = 30 * G // L
    seq, qual, _, second = synth.genome_reads(23, G, n, L, 0.01, 0.002)
    rg = (np.arange(n) // 2 % 3).astype(np.uint16)
    reads = str(tmp_path / "reads.fq")
    synth.write_fastq(reads, str(tmp_path / "unused.fq"), seq, qual, seq, rg, second, infer_rg=True)
    argv = ["-r", reads, "--infer-rg"] + (["--correct"] if correct else [])
    d = str(_native.DEVICE)
    monkeypatch.setenv("KBBQ_BATCH_READS", "997")
    monkeypatch.setenv("KBBQ_DEVICES", d)
    capfd.readouterr()
    _main(monkeypatch, argv)
    want = capfd.readouterr().out
    assert want.count("\n") == 4 * n
    monkeypatch.setenv("KBBQ_DEVICES", ",".join([d] * 3))
    _main(monkeypatch, argv)
    assert capfd.readouterr().out == want
    monkeypatch.setenv("KBBQ_MULTI_NO_P2P", "1")
    _main(monkeypatch, argv)
    assert capfd.readouterr().out == want


# ---- two or more GPUs -----------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_gpu_two_devices_same_result(kmer_oracle):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    seq, qual, second, n = batch(23, 150, seed=9, lower=0.0)
    for correct in (False, True):
        _check_session(kmer_oracle, seq, qual, second, n, 3, 23, 150, 0, 1000, [[0, 1], [1, 0], [0, 1, 0]], correct)
