"""The correcting walk (kbbq_kmer_correct, `kbbq recalibrate -r --correct`, DESIGN.md §10 "The correcting walk"): its C
oracle (tests/kmer_correct_oracle.c) against a plain Python restatement of the rule, hand-made reads, detection quality, the CLI and the argument
checks on the CPU; on the GPU the kernel bit for bit against the oracle on exact and sieved tables, and the whole path
against the corrected-file path fed the oracle's map."""
import ctypes as C
import importlib.util
import os
import sys
from collections import Counter

import numpy as np
import pytest

E_ARG = -1
CORRECT = 1

CODE = {ord("A"): 0, ord("C"): 1, ord("G"): 2, ord("T"): 3}
SWAP = np.arange(256, dtype=np.uint8)   # A<->C, G<->T: a corrected base that differs from the read's
for _a, _b in (("A", "C"), ("G", "T")):
    SWAP[ord(_a)], SWAP[ord(_b)] = ord(_b), ord(_a)


def _load(name):
    """tests/<name>.py, loaded by path (it compiles its C file into a temporary directory)."""
    spec = importlib.util.spec_from_file_location(name, os.path.join(os.path.dirname(os.path.abspath(__file__)),
                                                                     name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="module")
def kmer_oracle():
    """The boundary rule's oracle (tests/kmer_oracle.c)."""
    return _load("kmer_oracle")


@pytest.fixture(scope="module")
def walk_oracle():
    """The correcting walk's oracle (tests/kmer_correct_oracle.c)."""
    return _load("kmer_correct_oracle")


def key(w):
    if any(b not in CODE for b in w):
        return None
    f = r = 0
    for b in w:
        f = 4 * f + CODE[b]
    for b in reversed(w):
        r = 4 * r + 3 - CODE[b]
    return min(f, r)


def py_kmer_corrections(seq, k, min_count):
    """The correcting walk with a dict, on a bytearray copy of each read: -> (errors bool[N, L], hist[256], t)."""
    N, L = seq.shape
    nw = L - k + 1
    counts = Counter(x for row in seq for j in range(max(0, nw)) for x in [key(bytes(row[j:j + k]))] if x is not None)
    hist = [0] * 256
    for c in counts.values():
        hist[min(c, 255)] += 1
    t = min_count if min_count > 0 else next((c for c in range(2, 255) if hist[c] <= hist[c + 1]), 255)
    err = np.zeros((N, L), bool)
    for r in range(N):
        w = bytearray(seq[r].tobytes())

        def solid(j):
            x = key(bytes(w[j:j + k]))
            return x is not None and counts.get(x, 0) >= t

        sol = [solid(j) for j in range(max(0, nw))]
        best, a0, j = 0, None, 0
        while j < len(sol):   # the anchor: the longest run of solid windows, the leftmost of equal ones
            if not sol[j]:
                j += 1
                continue
            b = j
            while b < len(sol) and sol[b]:
                b += 1
            if b - j > best:
                best, a0 = b - j, j
            j = b
        if not best:
            continue
        for j, step in ((a0 + best, 1), (a0 - 1, -1)):
            while 0 <= j < nw:
                if solid(j):
                    j += step
                    continue
                e = j + k - 1 if step > 0 else j
                if w[e] not in CODE:
                    break
                m = min(k, nw - j if step > 0 else j + 1)
                scores = {}
                orig = w[e]
                for c in b"ACGT":
                    if c == orig:
                        continue
                    w[e] = c
                    n = 0
                    while n < m and solid(j + step * n):
                        n += 1
                    scores[c] = n
                w[e] = orig
                err[r, e] = True
                top = max(scores.values())
                winners = [c for c, n in scores.items() if n == top]
                if top < 1 or len(winners) != 1:
                    break
                w[e] = winners[0]
                j += step
    return err, np.array(hist, np.uint64), t


def bits_mask(bits, N, L):
    from kbbq.kmer import bits_to_mask
    return bits_to_mask(bits, N, L)


def small_batch(seed, L, n_reads=120, genome_len=600, lower=0.002, n_rate=0.004):
    """Reads of a small genome (repeated k-mers), with N bases and a few lowercase bytes -> seq, qual, second."""
    from kbbq import synth
    seq, qual, _, second = synth.genome_reads(seed, max(genome_len, 2 * L), n_reads, L, 0.01, n_rate)
    rng = np.random.default_rng(seed + 1)
    low = rng.random(seq.shape) < lower
    seq[low] = seq[low] | 0x20
    return seq, qual, second


# ---- CPU: the oracle against the Python restatement -----------------------------------------------------------------

@pytest.mark.parametrize("k", [1, 2, 15, 23, 31])
@pytest.mark.parametrize("L", ["short", "k", 151])
@pytest.mark.parametrize("min_count", [0, 1, 3])
def test_oracle_matches_python_rule(walk_oracle, k, L, min_count):
    L = {"short": max(1, k - 1), "k": k}.get(L, L)
    seq = small_batch(1000 * k + L + 7, L, n_reads=60 if L == 151 else 200, genome_len=400)[0]
    want, want_h, want_t = py_kmer_corrections(seq, k, min_count)
    bits, hist, t = walk_oracle.kmer_corrections(seq, L, k, min_count)
    assert t == want_t
    assert np.array_equal(hist, want_h)
    assert np.array_equal(bits_mask(bits, *seq.shape), want)
    # every flagged base is A/C/G/T
    assert np.isin(seq[want], list(CODE)).all()
    if L < k or min_count == 1:
        assert not want.any()
    if L == 151 and min_count != 1 and k >= 15:
        assert want.any()


# ---- CPU: hand-made reads -------------------------------------------------------------------------------------------

K, LH = 11, 60


def tiling(genome):
    """Every read of length LH of the circular genome: each k-mer LH - K + 1 = 50 times."""
    g = np.frombuffer(genome + genome[:LH - 1], np.uint8)
    return np.stack([g[i:i + LH] for i in range(len(genome))])


def other(b, *avoid):
    return next(c for c in b"ACGT" if c != b and c not in avoid)


@pytest.fixture(scope="module")
def genome():
    rng = np.random.default_rng(17)
    return bytes(np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 300)])


def run_hand(kmer_oracle, walk_oracle, genome, reads, min_count=3, extra=()):
    """The reads after the genome's tiling (and `extra` reads): -> (walk flags, boundary flags) of the hand-made reads,
    the walk checked against the Python restatement."""
    reads = np.stack(reads)
    seq = np.concatenate([tiling(genome)] + [tiling(x) for x in extra] + [reads])
    n, h = seq.shape[0], reads.shape[0]
    bits, _, t = walk_oracle.kmer_corrections(seq, LH, K, min_count)
    got = bits_mask(bits, n, LH)
    assert t == min_count
    assert np.array_equal(got, py_kmer_corrections(seq, K, min_count)[0])
    assert not got[:-h].any()   # error-free reads: nothing
    boundary = bits_mask(kmer_oracle.kmer_errors(seq, LH, K, min_count)[0], n, LH)
    return got[-h:], boundary[-h:]


def read_at(genome, o, subs=()):
    r = np.frombuffer(genome[o:o + LH], np.uint8).copy()
    for p, b in subs:
        r[p] = b
    return r


def flagged(mask):
    return [list(np.flatnonzero(row)) for row in mask]


def test_hand_one_error_and_read_ends(kmer_oracle, walk_oracle, genome):
    g = genome
    reads = [read_at(g, 10, [(30, other(g[40]))]),
             read_at(g, 50, [(0, other(g[50]))]),
             read_at(g, 90, [(LH - 1, other(g[90 + LH - 1]))]),
             read_at(g, 130, [(0, other(g[130])), (LH - 1, other(g[130 + LH - 1]))]),
             # two errors within k of the read end: the boundary rule flags only the inner one
             read_at(g, 170, [(LH - 4, other(g[170 + LH - 4])), (LH - 1, other(g[170 + LH - 1]))])]
    got, boundary = run_hand(kmer_oracle, walk_oracle, g, reads)
    assert flagged(got) == [[30], [0], [LH - 1], [0, LH - 1], [LH - 4, LH - 1]]
    assert flagged(boundary)[4] == [LH - 4]


def test_hand_cluster_of_three(kmer_oracle, walk_oracle, genome):
    """Three errors within k: all three flagged; the boundary rule flags the ends of the run and misses the middle."""
    g = genome
    pos = [25, 29, 33]
    reads = [read_at(g, 40, [(p, other(g[40 + p])) for p in pos]),
             read_at(g, 120, [(p, other(g[120 + p])) for p in (8, 12, 16)]),   # anchor to the right of the cluster
             read_at(g, 200, [(p, other(g[200 + p])) for p in (43, 47, 51)])]  # anchor to the left
    got, boundary = run_hand(kmer_oracle, walk_oracle, g, reads)
    assert flagged(got) == [pos, [8, 12, 16], [43, 47, 51]]
    assert flagged(boundary)[0] == [25, 33]
    assert not boundary[0, 29]


def test_hand_tie_stops_the_walk(kmer_oracle, walk_oracle, genome):
    """Two alleles of the genome at one base: a third base there ties their scores, so that base is flagged and
    nothing beyond it, not even a plain error."""
    g = genome
    o, p = 20, 40
    g2 = bytearray(g)
    g2[o + p] = other(g[o + p])
    third = other(g[o + p], g2[o + p])
    read = read_at(g, o, [(p, third), (55, other(g[o + 55]))])
    got, boundary = run_hand(kmer_oracle, walk_oracle, g, [read], extra=[bytes(g2)])
    assert flagged(got) == [[p]]
    assert boundary[0, 55]


def test_hand_no_solid_window_n_and_t1(kmer_oracle, walk_oracle, genome):
    g = genome
    rng = np.random.default_rng(3)
    alien = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, LH)].copy()
    n_stop = read_at(g, 30, [(45, other(g[75])), (50, ord("N")), (55, other(g[85]))])
    reads = [alien, n_stop, read_at(g, 60, [(30, other(g[90]))])]
    got, _ = run_hand(kmer_oracle, walk_oracle, g, reads)
    # no solid window: nothing; the N stops the walk after 45 was corrected, so 55 is never reached
    assert flagged(got) == [[], [45], [30]]
    seq = np.concatenate([tiling(g), np.stack(reads)])
    bits, _, t = walk_oracle.kmer_corrections(seq, LH, K, 1)
    assert t == 1 and not bits.any()


# ---- CPU: detection quality -----------------------------------------------------------------------------------------

def test_detection_quality(kmer_oracle, walk_oracle):
    """The reads of test_kmer.py::test_detection_quality (30x of a 200 kb genome, L = 150, 1 % substitutions) at
    k = 23: the walk finds >= 99 % of the errors, more than the boundary rule, and flags almost nothing else."""
    from kbbq import synth
    G, L = 200_000, 150
    n = 30 * G // L
    seq, _, err, _ = synth.genome_reads(11, G, n, L, 0.01)
    got = bits_mask(walk_oracle.kmer_corrections(seq, L, 23)[0], n, L)
    old = bits_mask(kmer_oracle.kmer_errors(seq, L, 23)[0], n, L)
    tp = int((got & err).sum())
    precision, recall = tp / got.sum(), tp / err.sum()
    assert precision >= 0.999 and recall >= 0.99, (precision, recall)
    assert recall > int((old & err).sum()) / err.sum()


# ---- CPU: the CLI, the drivers and the argument checks --------------------------------------------------------------

def _main(monkeypatch, argv):
    import kbbq.main
    with monkeypatch.context() as m:
        m.setattr(sys, "argv", [sys.argv[0], "recalibrate"] + argv)
        kbbq.main.main()


def test_cli_passes_correct(monkeypatch):
    from kbbq import recalibrate
    seen = {}
    monkeypatch.setattr(recalibrate, "recalibrate_reads", lambda path, **kw: seen.update(path=path, **kw))
    _main(monkeypatch, ["-r", "x.fq", "--correct", "-k", "19"])
    assert seen == dict(path="x.fq", infer_rg=False, k=19, min_count=0, devices=None, correct=True)


@pytest.mark.parametrize("argv", [
    ["-f", "a.fq", "b.fq", "--correct"],
    ["-b", "a.bam", "--correct"],
    ["--correct"],
])
def test_cli_refuses_correct_without_reads(monkeypatch, capsys, argv):
    with pytest.raises(SystemExit) as e:
        _main(monkeypatch, argv)
    assert e.value.code == 2


@pytest.fixture
def small_fastq(tmp_path):
    from kbbq import synth
    seq, qual, _, second = synth.genome_reads(4, 2000, 40, 60, 0.01)
    path = str(tmp_path / "reads.fq")
    synth.write_reads_fastq(path, seq, qual, second)
    return path


def test_drivers_receive_correct(monkeypatch, small_fastq, capfd):
    from kbbq import _native, recalibrate
    seen = []
    monkeypatch.setattr(recalibrate, "_recalibrate_reads_streamed",
                        lambda reads, infer_rg, k, min_count, batch_reads, device, correct=False:
                        seen.append(("streamed", batch_reads, correct)))

    def single(seq, qual, rg, second, L, R, minscore, k, min_count, device=None, correct=False):
        seen.append(("single", k, correct))
        return np.full(seq.shape, 30, np.uint8), 4
    monkeypatch.setattr(_native, "recalibrate_kmer_host", single)
    monkeypatch.setenv("KBBQ_BATCH_READS", "7")
    recalibrate.recalibrate_reads(small_fastq, correct=True)
    monkeypatch.delenv("KBBQ_BATCH_READS")
    recalibrate.recalibrate_reads(small_fastq, k=21, correct=True)
    recalibrate.recalibrate(None, None, reads=small_fastq, kmer_correct=True)
    assert seen == [("streamed", 7, True), ("single", 21, True), ("single", 23, True)]
    assert capfd.readouterr().out.count("\n") == 2 * 160


def test_entry_points_check_arguments():
    from kbbq import _native
    L = _native.lib()
    p = C.c_void_p(1 << 20)   # never dereferenced: every call below returns before touching the device
    z = C.c_void_p(None)
    t = C.c_int(0)
    assert L.kbbq_kmer_correct(p, 4, 50, 23, p, 1024, 0, p, p, z) == E_ARG            # t = 0
    assert L.kbbq_kmer_correct(p, 4, 50, 23, p, 1024, 3, p, z, z) == E_ARG            # no status word
    assert L.kbbq_kmer_correct(p, 4, 50, 32, p, 1024, 3, p, p, z) == E_ARG            # k > 31
    assert L.kbbq_kmer_correct(p, 4, 50, 23, p, 1000, 3, p, p, z) == E_ARG            # table not a power of two
    assert L.kbbq_kmer_correct(z, 4, 50, 23, p, 1024, 3, p, p, z) == E_ARG            # no reads
    assert L.kbbq_kmer_correct(z, 0, 50, 23, p, 1024, 3, z, p, z) == 0                # nothing to do
    seq = np.zeros(100, np.uint8)
    bits = np.zeros(4, np.uint32)
    for rule in (-1, 2):
        assert L.kbbq_kmer_errors_rule_host(_native.ptr(seq), 2, 50, 23, 0, rule, _native.ptr(bits), None,
                                            C.byref(t), 0) == E_ARG
        assert L.kbbq_recalibrate_kmer_rule_host(_native.ptr(seq), _native.ptr(seq), None, None, 2, 50, 1, 6, 23, 0,
                                                 rule, _native.ptr(seq), None, None, None, None, 0) == E_ARG
    assert L.kbbq_session_kmer_rule(z, CORRECT) == E_ARG


# ---- GPU: the kernel on exact and sieved tables ---------------------------------------------------------------------

def gpu_batch(k, L, seed=3, lower=0.001):
    """Every k-mer of an 8 kb genome ~25 times, 1 % substitutions, N bases and a few lowercase bytes.
    -> seq, qual, second, N"""
    G = 8000
    n = (25 * G // (L - k + 1)) & ~1
    return small_batch(seed + 31 * k + L, L, n_reads=n, genome_len=G, lower=lower, n_rate=0.003) + (n,)


class Dev:
    """A batch on the device and the entry points on torch buffers."""

    def __init__(self, seq, L, k):
        import torch
        from kbbq import _native
        self.torch, self.lib, self.native = torch, _native.lib(), _native
        self.N, self.L, self.k = seq.shape[0], L, k
        self.seq = torch.from_numpy(np.ascontiguousarray(seq).ravel()).cuda()
        self.stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        self.exact_cap = _native.kmer_table_bytes(self.N, L, k)[0]

    def buf(self, n, fill=None, dtype=None):
        t = self.torch
        return t.zeros(n, dtype=dtype or t.int64, device="cuda") if fill is None else \
            t.full((n,), fill, dtype=dtype or t.int64, device="cuda")

    def p(self, t, off=0):
        return C.c_void_p(t.data_ptr() + off)

    def ok(self, rc):
        self.native.check(rc)

    def exact(self, cap=None):
        """An exact table of the batch -> (table, cap, status)"""
        cap = cap or self.exact_cap
        table, status = self.buf(2 * cap), self.buf(1, dtype=self.torch.int32)
        self.ok(self.lib.kbbq_kmer_clear(self.p(table), cap, self.stream))
        self.ok(self.lib.kbbq_kmer_count(self.p(self.seq), self.N, self.L, self.k, self.p(table), cap, self.p(status),
                                         self.stream))
        return table, cap, status

    def sieved(self, filter_words, cap, chunks):
        """A sieved table filled over the chunks (read counts) -> (table, cap, status, hist)"""
        lib, L, k = self.lib, self.L, self.k
        filt, table = self.buf(filter_words), self.buf(2 * cap)
        status, windows, hist = self.buf(1, dtype=self.torch.int32), self.buf(1), self.buf(256)
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
        return table, cap, status, hist.cpu().numpy().astype(np.uint64)

    def correct(self, table, cap, t, status):
        bits = self.buf((self.N * self.L + 31) // 32, fill=-1, dtype=self.torch.int32)   # every word is written
        self.ok(self.lib.kbbq_kmer_correct(self.p(self.seq), self.N, self.L, self.k, self.p(table), cap, t,
                                           self.p(bits), self.p(status), self.stream))
        return bits.cpu().numpy().view(np.uint32)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [15, 23, 31])
@pytest.mark.parametrize("L", [33, 100, 150, 151])
@pytest.mark.parametrize("min_count", [0, 1, 3])
def test_gpu_correct_matches_oracle(walk_oracle, k, L, min_count):
    from kbbq import _native, kmer
    seq, _, _, n = gpu_batch(k, L)
    want_bits, want_hist, want_t = walk_oracle.kmer_corrections(seq, L, k, min_count)
    assert want_bits.any() or min_count == 1
    # the host-buffer entry point and kbbq.kmer
    bits, hist, t = _native.kmer_errors_host(seq, L, k, min_count, rule=_native.KMER_CORRECT)
    assert t == want_t and np.array_equal(hist, want_hist)
    assert np.array_equal(bits, want_bits)
    err, t, _ = kmer.find_errors(seq, L, k, min_count, correct=True)
    assert t == want_t and np.array_equal(err, bits_mask(want_bits, n, L))
    # the device entry point on an exact table
    d = Dev(seq, L, k)
    table, cap, status = d.exact()
    assert np.array_equal(d.correct(table, cap, want_t, status), want_bits)
    assert int(status.cpu()[0]) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("k", [15, 23, 31])
@pytest.mark.parametrize("L", [33, 100, 151])
@pytest.mark.parametrize("min_count", [0, 1, 3])
def test_gpu_correct_sieved_matches_oracle(walk_oracle, k, L, min_count):
    """On a sieved table (t >= 2: an absent key has count <= 1 < t) the walk gives the exact table's bits, including
    for candidate k-mers that occur nowhere in the reads."""
    from kbbq import _native
    seq, _, _, n = gpu_batch(k, L)
    want_bits, want_hist, want_t = walk_oracle.kmer_corrections(seq, L, k, min_count)
    d = Dev(seq, L, k)
    W = n * (L - k + 1)
    planned = _native.kmer_stream_plan(W, 2 << 20)
    for filter_words, cap in ((1, d.exact_cap), (1 << 10, d.exact_cap), planned):
        for chunks in ([n], [1, 33, n - 34]):
            where = (filter_words, cap, chunks)
            table, cap, status, hist = d.sieved(filter_words, cap, chunks)
            assert np.array_equal(hist, want_hist), where
            t = min_count or _native.kmer_min_count(hist)
            assert t == want_t, where
            assert np.array_equal(d.correct(table, cap, t, status), want_bits), where
            assert int(status.cpu()[0]) == 0, where


@pytest.mark.gpu
def test_gpu_correct_full_table():
    """A table too small for the batch raises KBBQ_FLAG_KMER_FULL in the walk's lookups."""
    from kbbq import _native
    seq, _, _, n = gpu_batch(23, 100)
    d = Dev(seq, 100, 23)
    table, cap, status = d.exact(64)
    status.zero_()
    d.correct(table, cap, 3, status)
    assert int(status.cpu()[0]) & _native.FLAG_KMER_FULL


# ---- GPU: the whole path --------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("k,L", [(15, 100), (23, 150), (31, 151)])
@pytest.mark.parametrize("R", [1, 3])
def test_gpu_recalibrate_correct_matches_corrected(walk_oracle, k, L, R):
    """kbbq_recalibrate_kmer_rule_host(KBBQ_KMER_CORRECT) = kbbq_recalibrate_host fed corrected reads that differ where
    the oracle's walk flags."""
    from kbbq import _native
    seq, qual, second, n = gpu_batch(k, L, seed=9, lower=0.0)   # lowercase is a bad base to the build
    rg = (np.arange(n) // 2 % R).astype(np.uint16)
    min_count = 0 if k != 31 else 3
    bits, _, want_t = walk_oracle.kmer_corrections(seq, L, k, min_count)
    corr = np.where(bits_mask(bits, n, L), SWAP[seq], seq)
    want_out, want_tabs, want_deltas = _native.recalibrate_host(seq, qual, corr, rg, second, L, R, 6, want_tables=True)
    out, t, tabs, deltas = _native.recalibrate_kmer_host(seq, qual, rg, second, L, R, 6, k, min_count,
                                                         want_tables=True, correct=True)
    assert t == want_t
    assert np.array_equal(out, want_out)
    for a, b in zip(tabs, want_tabs):
        assert np.array_equal(a, b)
    for a, b in zip(deltas, want_deltas):
        assert np.array_equal(a, b)
    # a session in chunks of a size that does not divide the batch gives the same
    with _native.Session(L, R, 6, chunk_reads=1000, resident_reads=0) as s:
        s.kmer_begin(k, n * (L - k + 1))
        s.kmer_rule(_native.KMER_CORRECT)
        spans = [(lo, min(1000, n - lo)) for lo in range(0, n, 1000)]
        for lo, m in spans:
            s.kmer_sieve(seq[lo:lo + m])
        for lo, m in spans:
            s.kmer_count(seq[lo:lo + m])
        assert s.kmer_threshold(min_count)[0] == want_t
        for lo, m in spans:
            s.build_chunk_kmer(seq[lo:lo + m], qual[lo:lo + m], rg[lo:lo + m], second[lo:lo + m])
        got_deltas = s.model(want_deltas=True)
        got_tables = s.tables()
        got = np.zeros((n, L), np.uint8)
        for lo, m in spans:
            s.apply_chunk(seq[lo:lo + m], qual[lo:lo + m], rg[lo:lo + m], second[lo:lo + m], got[lo:lo + m])
        s.sync()
    assert np.array_equal(got, want_out)
    assert np.array_equal(got_tables, np.concatenate([a.ravel() for a in want_tabs]))
    for a, b in zip(got_deltas, want_deltas):
        assert np.array_equal(a, b)


@pytest.mark.gpu
def test_gpu_session_rule_out_of_order():
    from kbbq import _native
    L_ = _native.lib()
    seq, qual, second, n = gpu_batch(23, 100, lower=0.0)
    seq, qual, second = seq[:64], qual[:64], second[:64]
    with _native.Session(100, 1, 6, chunk_reads=64, resident_reads=0) as s:
        assert L_.kbbq_session_kmer_rule(s.h, CORRECT) == E_ARG   # before kmer_begin
        s.kmer_begin(23, 64 * 78)
        assert L_.kbbq_session_kmer_rule(s.h, 2) == E_ARG         # unknown rule
        assert L_.kbbq_session_kmer_rule(s.h, -1) == E_ARG
        s.kmer_rule(_native.KMER_CORRECT)
        s.kmer_sieve(seq)
        s.kmer_rule(_native.KMER_BOUNDARIES)                      # any time before the first flagged chunk
        s.kmer_count(seq)
        s.kmer_threshold()
        s.kmer_rule(_native.KMER_CORRECT)
        s.build_chunk_kmer(seq, qual, None, second)
        assert L_.kbbq_session_kmer_rule(s.h, CORRECT) == E_ARG   # after a chunk has been flagged
        s.model()
        s.sync()
        s.reset()                                                  # a new run starts with the boundary rule
        assert L_.kbbq_session_kmer_rule(s.h, CORRECT) == E_ARG
        s.kmer_begin(23, 64 * 78)
        s.kmer_rule(_native.KMER_CORRECT)


@pytest.mark.gpu
@pytest.mark.parametrize("batch_reads", [None, "997"])
def test_gpu_cli_correct_equals_corrected_file(kmer_oracle, walk_oracle, tmp_path, monkeypatch, capfd, batch_reads):
    """`kbbq recalibrate -r reads.fq --correct` prints what `-f reads.fq corr.fq` prints when corr.fq differs at the
    bases the walk flags, in one batch and streamed in batches of a size that does not divide the file."""
    from kbbq import synth
    L, G = 150, 20_000
    n = 30 * G // L
    seq, qual, _, second = synth.genome_reads(21, G, n, L, 0.01, 0.002)
    bits, _, _ = walk_oracle.kmer_corrections(seq, L, 23)
    corr = np.where(bits_mask(bits, n, L), SWAP[seq], seq)
    reads, fixed = str(tmp_path / "reads.fq"), str(tmp_path / "corr.fq")
    synth.write_reads_fastq(reads, seq, qual, second)
    synth.write_reads_fastq(fixed, corr, qual, second)
    monkeypatch.delenv("KBBQ_BATCH_READS", raising=False)
    capfd.readouterr()
    _main(monkeypatch, ["-f", reads, fixed])
    want = capfd.readouterr().out
    if batch_reads:
        assert n % int(batch_reads)
        monkeypatch.setenv("KBBQ_BATCH_READS", batch_reads)
    _main(monkeypatch, ["-r", reads, "--correct"])
    got = capfd.readouterr().out
    assert got.count("\n") == 4 * n
    assert got == want
    # and the walk is not the boundary rule on these reads
    old = bits_mask(kmer_oracle.kmer_errors(seq, L, 23)[0], n, L)
    assert (old != bits_mask(bits, n, L)).any()
