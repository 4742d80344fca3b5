"""Sequencing errors from the reads' own k-mer spectrum, on the GPU (kbbq_kmer_*, include/kbbq_b200.h).

The rule is in DESIGN.md ("Errors from k-mer counts"): exact counts of the canonical k-mers of the batch, a threshold
t (the first valley of the count histogram unless given), and the boundaries of every run of bases that no k-mer with
count >= t covers -- or, with correct=True, every base the correcting walk changes when it corrects the read against
its trusted k-mers (DESIGN.md §10, "The correcting walk").  The result stands in for what a separate error
corrector's output gives `kbbq recalibrate -f`: the bases where the corrected read would differ.  Only the map is
returned, not the corrected reads.
"""
import numpy as np

from . import _native

DEFAULT_K = 23


def bits_to_mask(bits, N, L):
    """The 1-bit map of kbbq_host_mismatch_bits (bit i in word i // 32, LSB first) -> bool [N, L]."""
    b = np.ascontiguousarray(bits, dtype="<u4").view(np.uint8)
    return np.unpackbits(b, bitorder="little")[:N * L].astype(bool).reshape(N, L)


def find_errors(seq, L, k=DEFAULT_K, min_count=0, device=None, correct=False):
    """seq u8 [N, L] (or flat) -> (errors bool [N, L], min_count_used, histogram u64[256]).

    min_count = 0 picks the threshold from the histogram.  correct: find the errors by the correcting walk instead of
    the boundary rule.  Raises MemoryError when the k-mer table fills and
    ValueError when the reads and the table do not fit the GPU."""
    if not 1 <= k <= 31:
        raise ValueError("k must be in 1..31, got %d" % k)
    if min_count < 0:
        raise ValueError("min_count must be >= 0, got %d" % min_count)
    seq = np.ascontiguousarray(seq, dtype=np.uint8).ravel()
    N = seq.size // L
    rule = _native.KMER_CORRECT if correct else _native.KMER_BOUNDARIES
    bits, hist, t = _native.kmer_errors_host(seq, L, k, min_count, device, rule)
    return bits_to_mask(bits, N, L), t, hist
