"""numpy twin of the device generator kbbq-py_b200/csrc/synth.cuh (identical bytes for the same
(seed, read index, cycle)).  Bench / test input only; see synth.cuh for the distribution."""
import numpy as np

_M1, _M2 = np.uint64(0xBF58476D1CE4E5B9), np.uint64(0x94D049BB133111EB)
_GOLD, _STEP = np.uint64(0x9E3779B97F4A7C15), np.uint64(0xD6E8FEB86659FD93)


def _mix64(x):
    x = x.astype(np.uint64, copy=True)
    x ^= x >> np.uint64(30)
    x *= _M1
    x ^= x >> np.uint64(27)
    x *= _M2
    x ^= x >> np.uint64(31)
    return x


def synth_reads(seed, first_read, n, L, R, block=65536):
    """-> seq, qual, corr u8[n, L], rg u16[n], second u8[n] for reads [first_read, first_read + n).
    Generated in blocks of `block` reads to bound the int64 temporaries."""
    if n > block:
        parts = [_synth_block(seed, first_read + lo, min(block, n - lo), L, R) for lo in range(0, n, block)]
        return tuple(np.concatenate([p[k] for p in parts]) for k in range(5))
    return _synth_block(seed, first_read, n, L, R)


def _synth_block(seed, first_read, n, L, R):
    with np.errstate(over="ignore"):
        key = np.uint64(seed) * _GOLD
        r = np.arange(first_read, first_read + n, dtype=np.uint64)
        hr = _mix64(key + r * np.uint64(2) + np.uint64(1))
        hp = _mix64(key + (r >> np.uint64(1)) * np.uint64(2))
        sec = (r & np.uint64(1)).astype(np.int64)
        rg = ((hp >> np.uint64(8)) % np.uint64(R)).astype(np.uint16)
        mu = 36 + np.bitwise_count(hr & np.uint64(0xFFFFFF)).astype(np.int64) - 12 - 2 * sec
        l4 = max(L // 4, 1)
        has_tail = ((hr >> np.uint64(24)) & np.uint64(0xFF)) < np.uint64(13)
        tail = np.where(has_tail, 1 + (((hr >> np.uint64(32)) & np.uint64(0xFFFF)) % np.uint64(l4)).astype(np.int64), 0)
        i = np.arange(L, dtype=np.int64)
        h = _mix64(hr[:, None] + (i[None, :] + 1).astype(np.uint64) * _STEP)
    b = (h & np.uint64(3)).astype(np.int64)
    isn = ((h >> np.uint64(2)) & np.uint64(0x3FF)) == 0
    noise = np.bitwise_count((h >> np.uint64(12)) & np.uint64(0xFFFF)).astype(np.int64) - 8
    iserr = ((h >> np.uint64(28)) & np.uint64(0xFFFF)) < np.uint64(655)
    sh = 1 + (((h >> np.uint64(44)) & np.uint64(0xFFFF)) % np.uint64(3)).astype(np.int64)
    decay = (8 * i * i + (L * L) // 2) // (L * L)
    q = np.clip(mu[:, None] - decay[None, :] + noise, 2, 41)
    q = np.where((i[None, :] >= (L - tail)[:, None]) | isn, 2, q)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    seq = np.where(isn, np.uint8(ord("N")), acgt[b]).astype(np.uint8)
    corr = np.where(iserr, acgt[(b + sh) & 3], seq).astype(np.uint8)
    return seq, q.astype(np.uint8), corr, rg, sec.astype(np.uint8)


def genome_reads(seed, genome_len, n_reads, L, sub_rate=0.01, n_rate=0.0, block=1 << 20):
    """Reads sampled from a random genome, for the k-mer error path (kbbq.kmer): unlike synth_reads, whose bases are
    iid, these repeat each other's k-mers as real reads do.

    A seeded numpy stream draws a uniform random genome of `genome_len` bases.  Reads come in pairs (read 2i named
    r<i>/1, read 2i + 1 r<i>/2): a fragment of L to 2L bases at a uniform position, read 1 its first L bases, read 2
    the reverse complement of its last L.  Every base is then replaced by one of the three other bases with
    probability `sub_rate` (a sequencing error) or by N with probability `n_rate`.  Qualities: 25..40 on correct
    bases, 2..20 on errors, 2 on N.
    -> seq u8[n, L], qual u8[n, L], errors bool[n, L] (the substitutions), second u8[n]."""
    if n_reads and genome_len < 2 * L:
        raise ValueError("genome_len must be at least 2 L")
    rng = np.random.default_rng(seed)
    genome = rng.integers(0, 4, genome_len, dtype=np.uint8)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    seq = np.empty((n_reads, L), np.uint8)
    qual = np.empty((n_reads, L), np.uint8)
    err = np.empty((n_reads, L), bool)
    second = (np.arange(n_reads) & 1).astype(np.uint8)
    cols = np.arange(L)
    block += block & 1   # the two reads of a pair share a block
    for lo in range(0, n_reads, block):
        hi = min(n_reads, lo + block)
        n = hi - lo
        pair = (np.arange(lo, hi) >> 1)
        npairs = int(pair[-1] - pair[0] + 1)
        frag = rng.integers(L, 2 * L + 1, npairs)
        start = rng.integers(0, genome_len - frag + 1)
        frag, start = frag[pair - pair[0]], start[pair - pair[0]]
        is2 = second[lo:hi].astype(bool)
        first = np.where(is2, start + frag - L, start)
        codes = genome[first[:, None] + cols[None, :]]
        codes[is2] = 3 - codes[is2][:, ::-1]   # read 2: the reverse complement of the fragment's end
        e = rng.random((n, L)) < sub_rate
        shift = rng.integers(1, 4, (n, L), dtype=np.uint8)
        codes = np.where(e, (codes + shift) & 3, codes)
        isn = rng.random((n, L)) < n_rate
        seq[lo:hi] = np.where(isn, np.uint8(ord("N")), acgt[codes])
        q = np.where(e, rng.integers(2, 21, (n, L)), rng.integers(25, 41, (n, L)))
        qual[lo:hi] = np.where(isn, 2, q)
        err[lo:hi] = e & ~isn
    return seq, qual, err, second


def write_reads_fastq(path, seq, qual, second):
    """One FASTQ file of genome_reads' pairs, named r<i>/1 and r<i>/2."""
    n, L = seq.shape
    with open(path, "wb") as f:
        for i in range(n):
            f.write(b"@r%d/%d\n%s\n+\n%s\n" % (i // 2, int(second[i]) + 1, seq[i].tobytes(),
                                               (qual[i] + 33).astype(np.uint8).tobytes()))


def write_fastq(path_uncorr, path_corr, seq, qual, corr, rg, second, infer_rg=True):
    """Write the packed reads as the two FASTQ files `kbbq recalibrate -f` takes, named per
    docs/cli/fastq_input.rst of the reference (name/1_RG:Z:<rg>)."""
    names = []
    with open(path_uncorr, "w") as fu, open(path_corr, "w") as fc:
        for i in range(seq.shape[0]):
            name = "r%d/%d" % (i // 2, int(second[i]) + 1)
            if infer_rg:
                name += "_RG:Z:g%d" % int(rg[i])
            names.append(name)
            q = (qual[i] + 33).astype(np.uint8).tobytes().decode()
            fu.write("@%s\n%s\n+\n%s\n" % (name, seq[i].tobytes().decode(), q))
            fc.write("@%s\n%s\n+\n%s\n" % (name, corr[i].tobytes().decode(), q))
    return names


def write_fastq_fast(path_uncorr, path_corr, seq, qual, corr, rg, second, infer_rg=True):
    """write_fastq for millions of reads: fixed-width names (r0000123/1[_RG:Z:g07]) so that every record has
    the same byte length and the two files are written as one uint8 matrix each.  Same naming scheme as
    write_fastq (docs/cli/fastq_input.rst of the reference), zero-padded."""
    n, L = seq.shape
    idw = max(1, len(str(max(n // 2, 1))))
    rgw = max(1, len(str(int(rg.max()) if n else 0)))

    def digits(v, width):
        v = v.astype(np.int64)
        out = np.empty((v.size, width), np.uint8)
        for k in range(width):
            out[:, width - 1 - k] = 48 + (v // 10 ** k) % 10
        return out

    parts = [np.full((n, 1), ord("@"), np.uint8), np.full((n, 1), ord("r"), np.uint8), digits(np.arange(n) // 2, idw),
             np.full((n, 1), ord("/"), np.uint8), (49 + second.astype(np.uint8)).reshape(n, 1)]
    if infer_rg:
        parts += [np.tile(np.frombuffer(b"_RG:Z:g", np.uint8), (n, 1)), digits(rg, rgw)]
    nl = np.full((n, 1), 10, np.uint8)
    plus = np.tile(np.frombuffer(b"\n+\n", np.uint8), (n, 1))
    q = (qual + 33).astype(np.uint8)
    head = np.concatenate(parts, axis=1)
    np.concatenate([head, nl, seq, plus, q, nl], axis=1).tofile(path_uncorr)
    np.concatenate([head, nl, corr, plus, q, nl], axis=1).tofile(path_corr)
    return head.shape[1] - 1   # name length
