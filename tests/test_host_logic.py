"""Host-side logic that needs no GPU: the C-ABI library loads and exports every declared symbol,
FASTQ batching, name inference, the synthetic-read twin, shard ranges."""
import os
import re

import numpy as np
import pytest

from conftest import ROOT, load_case


def test_library_exports_every_declared_symbol():
    from kbbq import _native
    header = open(os.path.join(ROOT, "include", "kbbq_b200.h")).read()
    declared = set(re.findall(r"\b(kbbq_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(_native.SIGNATURES), declared ^ set(_native.SIGNATURES)
    lib = _native.lib()  # raises if the .so is missing: there is no fallback
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.kbbq_abi_version() == 1
    assert lib.kbbq_strerror(-1) == b"bad argument"
    assert lib.kbbq_pos_table_elems(150, 2) == 2 * 43 * 300
    assert lib.kbbq_din_table_elems(3) == 3 * 43 * 16


def test_workspace_query_and_argument_checks():
    import ctypes as C
    from kbbq import _native
    lib = _native.lib()
    nbytes = C.c_size_t(0)
    assert lib.kbbq_workspace_bytes(1000, 150, 1, C.byref(nbytes)) == 0 and nbytes.value > 0
    assert lib.kbbq_workspace_bytes(-1, 150, 1, C.byref(nbytes)) == -1
    assert lib.kbbq_workspace_bytes(10, 150, 0, C.byref(nbytes)) == -1


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from kbbq import _native
    monkeypatch.setattr(_native, "_lib", None)
    monkeypatch.setattr(_native, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_native.KbbqNativeError):
        _native.lib()


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "kbbq-py_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.lower(), (dirpath, f)


def test_fastx_and_batch(tmp_path):
    from kbbq import fastx
    from kbbq.batch import ReadBatch, infer_rg, infer_second
    g = load_case("tiny_r2")
    fu, fc = tmp_path / "u.fq", tmp_path / "c.fq"
    fu.write_text(str(g["fastq_in"]))
    fc.write_text(str(g["fastq_corr"]))
    b = ReadBatch.from_fastq((str(fu), str(fc)), True)
    assert np.array_equal(b.seq, g["seq"]) and np.array_equal(b.qual, g["qual"]) and np.array_equal(b.corr, g["corr"])
    assert np.array_equal(b.rg, g["rg"]) and np.array_equal(b.second, g["second"]) and b.R == int(g["R"])
    assert b.names == str(g["names"]).split("\n")
    recs = list(fastx.FastxFile(str(fc)))
    assert recs[0].comment == "corrected by lighter" and recs[0].name == b.names[0]
    assert str(fastx.FastxRecord("foo", "ATG", "((#")) == "@foo\nATG\n+\n((#"
    # no --infer-rg: a single group
    b1 = ReadBatch.from_fastq((str(fu), str(fc)), False)
    assert b1.R == 1 and not b1.rg.any()
    # reference behaviours: kbbq/compare_reads.py:304-318
    assert infer_second(["a/1", "a/2", "b/2_RG:Z:x", "c"]).tolist() == [0, 1, 1, 0]
    rg, keys = infer_rg(["a/1_RG:Z:foo", "a/2_RG:Z:bar", "b/1_RG:Z:foo"], True)
    assert rg.tolist() == [0, 1, 0] and keys == ["foo", "bar"]
    with pytest.raises(AssertionError):
        infer_rg(["a/1_XX:Z:foo"], True)
    with pytest.raises(IndexError):
        infer_rg(["a/1"], True)


def test_batch_name_mismatch_and_ragged(tmp_path):
    from kbbq.batch import ReadBatch
    fu, fc = tmp_path / "u.fq", tmp_path / "c.fq"
    fu.write_text("@r1\nACGT\n+\nIIII\n")
    fc.write_text("@x1\nACGT\n+\nIIII\n")
    with pytest.raises(AssertionError):  # find_corrected_sites, kbbq/recalibrate.py:17
        ReadBatch.from_fastq((str(fu), str(fc)))
    fu.write_text("@r1\nACGT\n+\nIIII\n@r2\nACG\n+\nIII\n")
    with pytest.raises(ValueError):
        ReadBatch.from_fastq((str(fu), str(fu)))
    fu.write_text("")
    fc.write_text("")
    assert ReadBatch.from_fastq((str(fu), str(fc))).N == 0


def test_host_helpers_match_reference_kats():
    from kbbq import compare_reads as cr
    # tests/test_compare_reads.py:124-139,153-189 of the reference
    assert cr.RescaledNormal.prior(0) == np.log(.9)
    assert np.all(cr.RescaledNormal.prior_dist < 0)
    s = load_case("scalars")
    assert np.array_equal(np.asarray(cr.RescaledNormal.prior_dist, dtype=np.float64), s["prior_dist"])
    assert cr.Dinucleotide.dinucs == ['AA', 'AT', 'AG', 'AC', 'TA', 'TT', 'TG', 'TC', 'GA', 'GT', 'GG', 'GC',
                                      'CA', 'CT', 'CG', 'CC']
    assert np.array_equal(cr.Dinucleotide.vecget(np.array(cr.Dinucleotide.dinucs)), np.arange(16))
    assert np.array_equal(cr.p_to_q(np.array([.2, .3, .4, .1, .01, .001])), [6, 5, 3, 10, 20, 30])
    assert np.array_equal(cr.p_to_q(cr.q_to_p(np.arange(43))), s["p_to_q_roundtrip"])
    assert np.allclose(cr.q_to_p(np.array([6, 10, 20, 30])).astype(float), [.251188643, .1, .01, .001])
    assert np.array_equal(cr.generic_cycle_covariate(17), np.arange(17))
    assert np.array_equal(cr.generic_cycle_covariate(17, True), -(np.arange(17) + 1))
    seq = np.array(list('ATGCATGC'))
    q = np.array([10] * 8)
    correct = np.concatenate([[-1], cr.Dinucleotide.vecget(np.array(['AT', 'TG', 'GC', 'CA', 'AT', 'TG', 'GC']))])
    assert np.array_equal(cr.generic_dinuc_covariate(seq, q), correct)
    seq[1] = 'N'
    correct[1] = correct[2] = -1
    assert np.array_equal(cr.generic_dinuc_covariate(seq, q), correct)
    q[6] = 2
    correct[6] = -1
    assert np.array_equal(cr.generic_dinuc_covariate(seq, q), correct)
    with pytest.raises(TypeError):
        cr.generic_dinuc_covariate(np.array(list('AXGC')), np.array([10] * 4))


def test_synth_twin_is_deterministic_and_shaped():
    from kbbq import synth
    a = synth.synth_reads(1002, 0, 512, 150, 4)
    b = synth.synth_reads(1002, 256, 256, 150, 4)
    for x, y in zip(a, b):
        assert np.array_equal(x[256:], y)  # any read range can be regenerated independently
    seq, qual, corr, rg, second = a
    assert set(np.unique(seq)) <= set(b"ACGTN") and qual.min() >= 2 and qual.max() <= 41
    assert np.all(qual[seq == ord("N")] == 2)
    assert second.tolist() == [0, 1] * 256 and np.array_equal(rg[0::2], rg[1::2]) and rg.max() < 4
    assert 0.005 < (seq != corr).mean() < 0.015
    assert not np.array_equal(seq, synth.synth_reads(1003, 0, 512, 150, 4)[0])


def test_shard_ranges_cover_and_align():
    from kbbq.parallel import shard_range
    for n in (0, 1, 15, 16, 17, 1000, 10_000_001):
        for world in (1, 2, 3, 8):
            spans = [shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            for (a, b), (c, d) in zip(spans, spans[1:]):
                assert b == c and a <= b
            assert all(lo % 16 == 0 for lo, _ in spans if lo < n)


def test_host_mismatch_bits_matches_numpy():
    """kbbq_host_mismatch_bits (csrc/host_pack.cpp): bit i = seq[i] != corr[i], little-endian in u32 words."""
    from kbbq import _native
    lib = _native.lib()
    rng = np.random.default_rng(3)
    for n in (0, 1, 31, 32, 33, 4096 * 32 * 3 + 17, 1_000_003):
        seq = rng.integers(65, 85, size=n, dtype=np.uint8)
        corr = seq.copy()
        flip = rng.random(n) < 0.05
        corr[flip] ^= rng.integers(1, 64, size=int(flip.sum()), dtype=np.uint8)
        bits = np.full((n + 31) // 32 + 1, 0xDEADBEEF, np.uint32)
        for threads in (1, 0):
            assert lib.kbbq_host_mismatch_bits(_native.ptr(seq), _native.ptr(corr), n, _native.ptr(bits), threads) == 0
            want = np.packbits(seq != corr, bitorder="little")
            got = bits[:(n + 31) // 32].view(np.uint8)[:want.size]
            assert np.array_equal(got, want), (n, threads)
            assert bits[(n + 31) // 32] == 0xDEADBEEF  # nothing written past the map


def test_host_pack_nibbles_matches_numpy():
    """kbbq_host_pack_nibbles (csrc/host_pack.cpp): 4 bits per base = (base >> 1) & 7 | mismatch << 3, two bases
    per byte (even base in the low nibble); a byte outside ACGTN is reported, as the reference's TypeError is."""
    import ctypes as C
    from kbbq import _native
    lib = _native.lib()
    rng = np.random.default_rng(4)
    alphabet = np.frombuffer(b"ACGTN", np.uint8)
    for n in (0, 1, 2, 63, 64, 65, 2048 * 64 * 3 + 21, 1_000_003):
        seq = alphabet[rng.integers(0, 5, size=n)]
        corr = seq.copy()
        flip = rng.random(n) < 0.05
        corr[flip] = alphabet[rng.integers(0, 5, size=int(flip.sum()))]   # some of them equal again
        for offset in (0, 1):   # destination 32-byte aligned (streaming stores) or not
            buf = np.full((n + 1) // 2 + 33, 0xAB, np.uint8)
            start = (-buf.ctypes.data) % 32 + offset
            packed = buf[start:start + (n + 1) // 2 + 1]
            for threads in (1, 0):
                bad = C.c_int(-1)
                assert lib.kbbq_host_pack_nibbles(_native.ptr(seq), _native.ptr(corr), n, _native.ptr(packed), threads, C.byref(bad)) == 0
                assert bad.value == 0
                nib = ((seq >> 1) & 7) | ((seq != corr).astype(np.uint8) << 3)
                if n & 1:
                    nib = np.append(nib, np.uint8(0))
                want = nib[0::2] | (nib[1::2] << 4)
                assert np.array_equal(packed[:(n + 1) // 2], want), (n, threads, offset)
                assert packed[(n + 1) // 2] == 0xAB  # nothing written past the packed bases
    # every byte value that is not one of ACGTN is reported, wherever it sits
    n = 2048 * 64 * 2 + 5
    seq = alphabet[rng.integers(0, 5, size=n)]
    packed = np.zeros((n + 1) // 2, np.uint8)
    for value in list(range(0, 256, 7)) + [ord("a"), ord("c"), ord("B"), ord("O"), ord("U"), 0x4F, 0xC1]:
        if value in b"ACGTN":
            continue
        for pos in (0, 70, n // 2, n - 1):
            s2 = seq.copy()
            s2[pos] = value
            bad = C.c_int(0)
            assert lib.kbbq_host_pack_nibbles(_native.ptr(s2), _native.ptr(seq), n, _native.ptr(packed), 0, C.byref(bad)) == 0
            assert bad.value == 1, (value, pos)


def test_shared_memory_plans_fit_for_every_read_length():
    """kbbq_plan_info (host only): every read length the shared-memory kernels claim (4 .. 288) gets a plan that
    fits the 227 KB of a B200 SM, whole warps of consumers + producer warps within 1024 threads, a ring of at least
    two stages -- for one and for several read groups, build (3 arrays staged) and apply (2), in read order and for
    a segmented batch (arrays | 0x100, KBBQ_PLAN_SEGMENTED)."""
    import ctypes as C
    from kbbq import _native
    lib = _native.lib()
    out = (C.c_int * 10)()
    planned = 0
    for L in range(4, 300):
        for R in (1, 8):
            for arrays in (3, 2, 3 | 0x100, 2 | 0x100):
                rc = lib.kbbq_plan_info(L, R, 6, arrays, 0, out)
                if L > 288:
                    assert rc != 0, (L, R, arrays)     # longer reads take the generic kernels
                    continue
                assert rc == 0, (L, R, arrays)
                G, lanes, ng, threads, nprod, kps, stages, drep, total, table_bytes = list(out)
                planned += 1
                assert total <= 232448 and table_bytes < total, (L, R, arrays, total)
                assert threads % 32 == 0 and threads + 32 * nprod <= 1024 and ng * lanes <= threads, (L, R, arrays)
                assert (G * L) % 4 == 0 and 1 <= kps <= 8 and stages >= 2 and drep in (8, 16, 32), (L, R, arrays)
                # two cycle tables of 44 - minscore rows each (row stride a multiple of 128 B covering L cycles)
                rows, rs = 44 - 6, (4 * ((L + 3) // 4) * 4 + 127) // 128 * 128
                assert table_bytes >= 2 * rows * rs + rows * 16 * drep * 4, (L, R, arrays)
    assert planned == 285 * 8
