"""Errors from k-mer counts (kbbq.kmer, kbbq_kmer_*): the C oracle against a plain Python restatement of the rule,
the threshold, the CLI, detection quality on simulated reads, and the GPU bit for bit against the oracle."""
import ctypes as C
import importlib.util
import os
import sys
from collections import Counter

import numpy as np
import pytest


@pytest.fixture(scope="module")
def kmer_oracle():
    """tests/kmer_oracle.py, loaded by path (it compiles tests/kmer_oracle.c into a temporary directory)."""
    spec = importlib.util.spec_from_file_location(
        "kmer_oracle", os.path.join(os.path.dirname(os.path.abspath(__file__)), "kmer_oracle.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


CODE = {ord("A"): 0, ord("C"): 1, ord("G"): 2, ord("T"): 3}
SWAP = np.arange(256, dtype=np.uint8)   # A<->C, G<->T: a corrected base that differs from the read's
for a, b in (("A", "C"), ("G", "T")):
    SWAP[ord(a)], SWAP[ord(b)] = ord(b), ord(a)


def py_kmer_errors(seq, k, min_count):
    """The rule of DESIGN.md, "Errors from k-mer counts", with a dict: -> (errors bool[N, L], hist[256], t)."""
    N, L = seq.shape

    def key(w):
        if any(b not in CODE for b in w):
            return None
        f = r = 0
        for b in w:
            f = 4 * f + CODE[b]
        for b in reversed(w):
            r = 4 * r + 3 - CODE[b]
        return min(f, r)

    keys = [[key(bytes(row[j:j + k])) for j in range(L - k + 1)] for row in seq]
    counts = Counter(x for row in keys for x in row if x is not None)
    hist = [0] * 256
    for c in counts.values():
        hist[min(c, 255)] += 1
    t = min_count if min_count > 0 else next((c for c in range(2, 255) if hist[c] <= hist[c + 1]), 255)
    err = np.zeros((N, L), bool)
    for r, row in enumerate(keys):
        solid = [x is not None and counts[x] >= t for x in row]
        if not any(solid):
            continue
        covered = [any(solid[j] for j in range(max(0, i - k + 1), min(i, len(solid) - 1) + 1)) for i in range(L)]
        i = 0
        while i < L:
            if covered[i]:
                i += 1
                continue
            a = i
            while i < L and not covered[i]:
                i += 1
            b = i - 1
            ends = (a, b) if a > 0 and b < L - 1 else (b,) if a == 0 else (a,)
            for e in ends:
                if seq[r, e] in CODE:
                    err[r, e] = True
    return err, np.array(hist, np.uint64), t


def bits_mask(bits, N, L):
    from kbbq.kmer import bits_to_mask
    return bits_to_mask(bits, N, L)


def revcomp(seq):
    comp = np.arange(256, dtype=np.uint8)
    for a, b in (("A", "T"), ("C", "G")):
        comp[ord(a)], comp[ord(b)] = ord(b), ord(a)
    return comp[seq[:, ::-1]]


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
@pytest.mark.parametrize("min_count", [0, 3])
def test_oracle_matches_python_rule(kmer_oracle, k, L, min_count):
    L = {"short": max(1, k - 1), "k": k}.get(L, L)
    seq = small_batch(1000 * k + L, L, n_reads=60 if L == 151 else 200, genome_len=400)[0]
    want, want_h, want_t = py_kmer_errors(seq, k, min_count)
    bits, hist, t = kmer_oracle.kmer_errors(seq, L, k, min_count)
    assert t == want_t
    assert np.array_equal(hist, want_h)
    assert np.array_equal(bits_mask(bits, *seq.shape), want)
    if L < k:
        assert not want.any() and not hist.any()


def test_oracle_runs_at_read_ends(kmer_oracle):
    """A substitution within k of a read end makes an uncovered run out to that end: only its inner end is flagged."""
    from kbbq import synth
    L, k = 60, 11
    seq, _, _, _ = synth.genome_reads(5, 300, 400, L, 0.0)
    bad = seq.copy()
    for r, pos in ((0, 2), (1, L - 3), (2, 30), (3, 0), (4, L - 1)):
        bad[r, pos] = SWAP[bad[r, pos]]
    bits, _, t = kmer_oracle.kmer_errors(bad, L, k, 3)
    got = bits_mask(bits, *bad.shape)
    want = np.zeros_like(got)
    for r, pos in ((0, 2), (1, L - 3), (2, 30), (3, 0), (4, L - 1)):
        want[r, pos] = True
    assert np.array_equal(got[:5], want[:5])
    assert np.array_equal(got, py_kmer_errors(bad, k, 3)[0])


def test_oracle_strand_symmetry(kmer_oracle):
    """A read and its reverse complement count on one key: the reverse-complemented batch has the same spectrum and
    the mirrored flags."""
    seq = small_batch(7, 90, n_reads=300, lower=0.0)[0]
    for k in (5, 23):
        b1, h1, t1 = kmer_oracle.kmer_errors(seq, 90, k)
        b2, h2, t2 = kmer_oracle.kmer_errors(revcomp(seq), 90, k)
        assert t1 == t2 and np.array_equal(h1, h2)
        assert np.array_equal(bits_mask(b2, 300, 90), bits_mask(b1, 300, 90)[:, ::-1])


# ---- CPU: the threshold ---------------------------------------------------------------------------------------------

def _hist(pairs):
    h = np.zeros(256, np.uint64)
    for c, v in pairs:
        h[c] = v
    return h


@pytest.mark.parametrize("hist,want", [
    (_hist([(1, 1000), (2, 50), (3, 20), (4, 25), (5, 40), (6, 10)]), 3),           # a valley
    (_hist([(1, 1000), (2, 50), (3, 50)]), 2),                                        # a tie is a valley
    (_hist([(c, 1000 - c) for c in range(1, 256)]), 255),                             # monotone: none
    (np.zeros(256, np.uint64), 2),                                                    # all zero
    (_hist([(c, 1000 - c) for c in range(1, 255)] + [(255, 1000)]), 254),            # the valley at 254
])
def test_min_count_rule(hist, want):
    from kbbq import _native
    assert _native.kmer_min_count(hist) == want


def test_min_count_null():
    from kbbq import _native
    assert _native.lib().kbbq_kmer_min_count(None) == -1


def test_table_bytes():
    from kbbq import _native
    assert _native.kmer_table_bytes(10_000_000, 150, 23) == (1 << 31, 16 << 31)
    assert _native.kmer_table_bytes(2, 10, 5)[0] == 32    # 12 windows, 1.5 x = 18
    assert _native.kmer_table_bytes(2, 7, 5)[0] == 16     # 6 windows, 1.5 x = 9
    assert _native.kmer_table_bytes(0, 10, 5)[0] == 1
    assert _native.kmer_table_bytes(4, 10, 11)[0] == 1    # L < k: no windows


# ---- CPU: the CLI ---------------------------------------------------------------------------------------------------

def _main(monkeypatch, argv):
    import kbbq.main
    with monkeypatch.context() as m:
        m.setattr(sys, "argv", [sys.argv[0], "recalibrate"] + argv)
        kbbq.main.main()


@pytest.mark.parametrize("argv", [
    ["-r", "a.fq", "-f", "a.fq", "b.fq"],
    ["-r", "a.fq", "-b", "a.bam"],
    ["-r", "a.fq", "-k", "0"],
    ["-r", "a.fq", "-k", "32"],
    ["-r", "a.fq", "--min-count", "-1"],
    [],
])
def test_cli_refuses(monkeypatch, capsys, argv):
    with pytest.raises(SystemExit) as e:
        _main(monkeypatch, argv)
    assert e.value.code == 2


def test_cli_gatkreport_with_reads(monkeypatch):
    with pytest.raises(NotImplementedError):
        _main(monkeypatch, ["-r", "a.fq", "-g", "report.txt"])


def test_cli_passes_kmer_options(monkeypatch):
    from kbbq import recalibrate
    seen = {}
    monkeypatch.setattr(recalibrate, "recalibrate_reads", lambda path, **kw: seen.update(path=path, **kw))
    _main(monkeypatch, ["-r", "x.fq", "-k", "31", "--min-count", "4", "--infer-rg"])
    assert seen == dict(path="x.fq", infer_rg=True, k=31, min_count=4, devices=None)
    _main(monkeypatch, ["-r", "y.fq"])
    assert seen["k"] == 23 and seen["min_count"] == 0


# ---- CPU: detection quality -----------------------------------------------------------------------------------------

def test_detection_quality(kmer_oracle):
    """30x of a 200 kb genome, L = 150, 1 % substitutions, k = 23: the rule finds >= 88 % of the errors and flags
    almost nothing else."""
    from kbbq import synth
    G, L = 200_000, 150
    n = 30 * G // L
    seq, _, err, _ = synth.genome_reads(11, G, n, L, 0.01)
    bits, _, t = kmer_oracle.kmer_errors(seq, L, 23)
    got = bits_mask(bits, n, L)
    tp = int((got & err).sum())
    precision, recall = tp / got.sum(), tp / err.sum()
    assert 3 <= t <= 8
    assert precision >= 0.999 and recall >= 0.88, (t, precision, recall)


# ---- GPU ------------------------------------------------------------------------------------------------------------

def gpu_batch(k, L, seed=3, lower=0.001):
    """Every k-mer of a genome ~25 times, with N bases (and lowercase bytes): repeated k-mers, reads without a solid
    window, runs at both read ends.  -> seq, qual, second, N"""
    G = 8000
    n = (25 * G // (L - k + 1)) & ~1
    return small_batch(seed + 31 * k + L, L, n_reads=n, genome_len=G, lower=lower, n_rate=0.003) + (n,)


class DevKmer:
    """The device entry points on torch buffers."""

    def __init__(self, seq, L, k, capacity=None):
        import torch
        from kbbq import _native
        self.torch, self.lib = torch, _native.lib()
        self.N, self.L, self.k = seq.shape[0], L, k
        self.cap = capacity or _native.kmer_table_bytes(self.N, L, k)[0]
        self.seq = torch.from_numpy(np.ascontiguousarray(seq).ravel()).cuda()
        self.table = torch.empty(2 * self.cap, dtype=torch.int64, device="cuda")
        self.status = torch.zeros(1, dtype=torch.int32, device="cuda")
        self.hist = torch.zeros(256, dtype=torch.int64, device="cuda")
        self.bits = torch.empty((self.N * L + 31) // 32, dtype=torch.int32, device="cuda")
        self.stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def p(self, t, off=0):
        return C.c_void_p(t.data_ptr() + off)

    def ok(self, rc):
        from kbbq import _native
        _native.check(rc)

    def clear(self):
        self.ok(self.lib.kbbq_kmer_clear(self.p(self.table), self.cap, self.stream))

    def count(self, r0=0, n=None):
        n = self.N - r0 if n is None else n
        self.ok(self.lib.kbbq_kmer_count(self.p(self.seq, r0 * self.L), n, self.L, self.k, self.p(self.table),
                                         self.cap, self.p(self.status), self.stream))

    def histogram(self):
        self.ok(self.lib.kbbq_kmer_histogram(self.p(self.table), self.cap, self.p(self.hist), self.stream))
        return self.hist.cpu().numpy().astype(np.uint64)

    def flag(self, t):
        self.ok(self.lib.kbbq_kmer_flag(self.p(self.seq), self.N, self.L, self.k, self.p(self.table), self.cap, t,
                                        self.p(self.bits), self.p(self.status), self.stream))
        return self.bits.cpu().numpy().view(np.uint32)

    def entries(self):
        t = self.table.cpu().numpy().view(np.uint64).reshape(-1, 2)
        t = t[t[:, 0] != np.uint64(2 ** 64 - 1)]
        return t[np.argsort(t[:, 0])]

    def status_word(self):
        return int(self.status.cpu()[0])


@pytest.mark.gpu
@pytest.mark.parametrize("k", [15, 23, 31])
@pytest.mark.parametrize("L", [33, 100, 150, 151])
@pytest.mark.parametrize("min_count", [0, 3])
def test_gpu_errors_match_oracle(kmer_oracle, k, L, min_count):
    from kbbq import _native
    seq, _, _, n = gpu_batch(k, L)
    want_bits, want_hist, want_t = kmer_oracle.kmer_errors(seq, L, k, min_count)
    assert want_bits.any()
    bits, hist, t = _native.kmer_errors_host(seq, L, k, min_count)
    assert t == want_t
    assert np.array_equal(hist, want_hist)
    assert np.array_equal(bits, want_bits)
    # the device entry points, the threshold resolved on the host
    d = DevKmer(seq, L, k)
    d.clear()
    d.count()
    h = d.histogram()
    assert np.array_equal(h, want_hist)
    t = min_count or _native.kmer_min_count(h)
    assert t == want_t
    assert np.array_equal(d.flag(t), want_bits)
    assert d.status_word() == 0


@pytest.mark.gpu
def test_gpu_find_errors(kmer_oracle):
    from kbbq import kmer
    seq, _, _, n = gpu_batch(23, 150)
    err, t, hist = kmer.find_errors(seq, 150)
    bits, want_hist, want_t = kmer_oracle.kmer_errors(seq, 150, 23)
    assert t == want_t and np.array_equal(hist, want_hist)
    assert np.array_equal(err, bits_mask(bits, n, 150))


@pytest.mark.gpu
def test_gpu_count_in_chunks():
    """Counts accumulate: two chunks give the table of one call (the same keys with the same counts)."""
    seq, _, _, n = gpu_batch(23, 100)
    one = DevKmer(seq, 100, 23)
    one.clear()
    one.count()
    two = DevKmer(seq, 100, 23)
    two.clear()
    two.count(0, n // 3)
    two.count(n // 3)
    a, b = one.entries(), two.entries()
    assert a.shape[0] > 1000
    assert np.array_equal(a, b)
    assert np.array_equal(one.histogram(), two.histogram())


@pytest.mark.gpu
def test_gpu_full_table():
    """A table too small for the batch raises KBBQ_FLAG_KMER_FULL and the calls return."""
    from kbbq import _native
    seq, _, _, n = gpu_batch(23, 100)
    d = DevKmer(seq, 100, 23, capacity=64)
    d.clear()
    d.count()
    assert d.status_word() & _native.FLAG_KMER_FULL
    assert d.histogram().sum() == 64
    d.status.zero_()
    d.flag(3)
    assert d.status_word() & _native.FLAG_KMER_FULL


@pytest.mark.gpu
@pytest.mark.parametrize("k", [15, 23, 31])
@pytest.mark.parametrize("L", [33, 100, 150, 151])
@pytest.mark.parametrize("R", [1, 3])
def test_gpu_recalibrate_kmer_matches_corrected(kmer_oracle, k, L, R):
    """kbbq_recalibrate_kmer_host = kbbq_recalibrate_host fed corrected reads that differ where the oracle flags."""
    from kbbq import _native
    seq, qual, second, n = gpu_batch(k, L, seed=9, lower=0.0)   # lowercase is a bad base to the build
    rg = (np.arange(n) // 2 % R).astype(np.uint16)
    min_count = 0 if k != 31 else 3
    bits, _, want_t = kmer_oracle.kmer_errors(seq, L, k, min_count)
    mask = bits_mask(bits, n, L)
    corr = np.where(mask, SWAP[seq], seq)
    want_out, want_tabs, want_deltas = _native.recalibrate_host(seq, qual, corr, rg, second, L, R, 6, want_tables=True)
    out, t, tabs, deltas = _native.recalibrate_kmer_host(seq, qual, rg, second, L, R, 6, k, min_count, want_tables=True)
    assert t == want_t
    assert np.array_equal(out, want_out)
    for a, b in zip(tabs, want_tabs):
        assert np.array_equal(a, b)
    for a, b in zip(deltas, want_deltas):
        assert np.array_equal(a, b)


@pytest.mark.gpu
def test_gpu_cli_reads_equals_corrected_file(kmer_oracle, tmp_path, monkeypatch, capfd):
    """`kbbq recalibrate -r reads.fq` prints what `-f reads.fq corr.fq` prints when corr.fq differs at the flagged
    bases."""
    from kbbq import synth
    L, G = 150, 20_000
    n = 30 * G // L
    seq, qual, _, second = synth.genome_reads(21, G, n, L, 0.01, 0.002)
    bits, _, _ = kmer_oracle.kmer_errors(seq, L, 23)
    corr = np.where(bits_mask(bits, n, L), SWAP[seq], seq)
    reads, fixed = str(tmp_path / "reads.fq"), str(tmp_path / "corr.fq")
    synth.write_reads_fastq(reads, seq, qual, second)
    synth.write_reads_fastq(fixed, corr, qual, second)
    capfd.readouterr()
    _main(monkeypatch, ["-r", reads])
    got = capfd.readouterr().out
    _main(monkeypatch, ["-f", reads, fixed])
    want = capfd.readouterr().out
    assert got.count("\n") == 4 * n
    assert got == want


def test_reads_of_unequal_length(tmp_path):
    from kbbq import recalibrate
    path = tmp_path / "ragged.fq"
    path.write_text("@a/1\nACGTACGT\n+\nIIIIIIII\n@a/2\nACGTAC\n+\nIIIIII\n")
    with pytest.raises(ValueError):
        recalibrate.recalibrate_reads(str(path))
