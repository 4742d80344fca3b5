"""Native FASTQ ingest / egress (csrc/fastq_io.cpp, SURVEY.md section 8 row f1) against the Python tokenizer
that mirrors pysam.FastxFile (kbbq/fastx.py) and against the reference's naming rules
(kbbq/compare_reads.py:304-318, kbbq/recalibrate.py:17,59-64,152-156).  Host only: no GPU needed."""
import gzip
import os

import numpy as np
import pytest

from kbbq import fastx


def _write(path, records, eol="\n", final_newline=True):
    text = eol.join("@%s%s\n%s\n+\n%s".replace("\n", eol) % (n, (" " + c) if c else "", s, q) for n, c, s, q in records)
    if final_newline:
        text += eol
    opener = gzip.open if str(path).endswith(".gz") else open
    with opener(path, "wt", newline="") as fh:
        fh.write(text)


def _random_records(rng, n, L, n_rg=5, comments=True):
    recs = []
    for i in range(n):
        pair = i // 2
        name = "r%d/%d_RG:Z:g%d" % (pair, 1 + (i & 1), rng.integers(0, n_rg))
        seq = "".join(rng.choice(list("ACGTN"), size=L))
        qual = "".join(chr(33 + int(q)) for q in rng.integers(2, 42, size=L))
        recs.append((name, "comment %d" % i if comments and i % 3 == 0 else "", seq, qual))
    return recs


@pytest.mark.parametrize("eol,final,suffix", [("\n", True, ".fq"), ("\r\n", True, ".fq"), ("\n", False, ".fq"),
                                              ("\n", True, ".fq.gz")])
def test_pack_matches_python_tokenizer(tmp_path, eol, final, suffix):
    rng = np.random.default_rng(3)
    recs = _random_records(rng, 1237, 41)
    path = tmp_path / ("x" + suffix)
    _write(path, recs, eol, final)
    f = fastx.NativeFastq(path, threads=5)
    assert f.N == len(recs) and f.L == 41
    seq, qual = f.pack()
    for i, rec in enumerate(fastx.FastxFile(str(path))):
        assert rec.name == recs[i][0] == f.name(i)
        assert seq[i].tobytes().decode() == rec.sequence == recs[i][2]
        assert list(qual[i]) == rec.get_quality_array()
    part_s, part_q = f.pack(100, 50)
    assert np.array_equal(part_s, seq[100:150]) and np.array_equal(part_q, qual[100:150])
    f.close()


@pytest.mark.parametrize("threads", [1, 3, 8])
def test_infer_rg_first_seen_order_and_second(tmp_path, threads):
    rng = np.random.default_rng(4)
    recs = _random_records(rng, 5000, 8, n_rg=7)
    path = tmp_path / "x.fq"
    _write(path, recs)
    f = fastx.NativeFastq(path, threads=threads)
    rg, second, keys = f.infer(True)
    seen = {}
    for i, (name, _, _, _) in enumerate(recs):  # kbbq/recalibrate.py:59-64 with fastq_infer_rg
        key = name.split("_")[1].split(":")[-1]
        assert rg[i] == seen.setdefault(key, len(seen))
        assert second[i] == (name.split("_")[0][-2:] == "/2")
    assert keys == list(seen)
    rg0, second0, keys0 = f.infer(False)
    assert not rg0.any() and keys0 == [0] and np.array_equal(second0, second)


def test_name_rules_raise_like_the_reference(tmp_path):
    a, b = tmp_path / "a.fq", tmp_path / "b.fq"
    _write(a, [("foo/1", "", "ACG", "III"), ("bar/2_XX:Z:g", "", "ACG", "III")])
    f = fastx.NativeFastq(a)
    with pytest.raises(IndexError):       # no second '_' field
        f.infer(True)
    _write(a, [("bar/2_XX:Z:g", "", "ACG", "III")])
    with pytest.raises(AssertionError):   # second field does not start with RG
        fastx.NativeFastq(a).infer(True)
    _write(a, [("foo/1", "", "ACG", "III"), ("bar/2", "", "ACG", "III")])
    _write(b, [("foo/1", "corrected", "ACG", "III"), ("baz/2", "", "ACG", "III")])
    with pytest.raises(AssertionError):   # find_corrected_sites name check
        fastx.NativeFastq(a).check_names(fastx.NativeFastq(b), 2)
    fastx.NativeFastq(a).check_names(fastx.NativeFastq(b), 1)


def test_malformed_and_ragged_inputs(tmp_path):
    p = tmp_path / "x.fq"
    p.write_text("@a\nACG\n+\nIII\n@b\nAC\n")
    with pytest.raises(ValueError):
        fastx.NativeFastq(p)
    p.write_text("@a\nACG\n+\nII\n")
    with pytest.raises(ValueError):
        fastx.NativeFastq(p)
    p.write_text("@a\nACG\n+\nIII\n@b\nAC\n+\nII\n")
    f = fastx.NativeFastq(p)
    assert f.N == 2 and f.L == -1
    with pytest.raises(ValueError):
        f.pack()
    p.write_text("")
    f = fastx.NativeFastq(p)
    assert f.N == 0
    names, seq, qual = fastx.read_packed(p)
    assert names == [] and seq.size == 0
    with pytest.raises(OSError):
        fastx.NativeFastq(tmp_path / "missing.fq")


def test_write_round_trip(tmp_path):
    rng = np.random.default_rng(6)
    recs = _random_records(rng, 70_001, 23)
    src, dst = tmp_path / "in.fq", tmp_path / "out.fq"
    _write(src, recs)
    f = fastx.NativeFastq(src, threads=4)
    newq = rng.integers(0, 60, size=(f.N, f.L)).astype(np.uint8)
    fd = os.open(dst, os.O_WRONLY | os.O_CREAT | os.O_TRUNC)
    f.write(fd, newq)
    os.close(fd)
    g = fastx.NativeFastq(dst)
    seq, qual = g.pack()
    seq0, _ = f.pack()
    assert np.array_equal(seq, seq0) and np.array_equal(qual, newq)
    with open(dst) as fh:  # header without the comment, '+' line bare (kbbq/recalibrate.py:152-156)
        head = [fh.readline() for _ in range(4)]
    assert head[0] == "@" + recs[0][0] + "\n" and head[2] == "+\n"


def test_write_to_pipe_append_and_offset_agree(tmp_path):
    """The formatter writes at per-thread offsets into seekable files and serially into pipes and
    O_APPEND files; the bytes must be the same, and a seekable descriptor continues where it stood."""
    import threading
    rng = np.random.default_rng(9)
    recs = _random_records(rng, 20_003, 31)
    src = tmp_path / "in.fq"
    _write(src, recs)
    f = fastx.NativeFastq(src, threads=4)
    newq = rng.integers(0, 60, size=(f.N, f.L)).astype(np.uint8)
    plain = tmp_path / "plain.fq"
    fd = os.open(plain, os.O_WRONLY | os.O_CREAT | os.O_TRUNC)
    os.write(fd, b"# kept\n")          # the descriptor does not start at 0
    f.write(fd, newq)
    os.write(fd, b"# after\n")         # ... and is left behind the records
    os.close(fd)
    want = plain.read_bytes()
    assert want.startswith(b"# kept\n@") and want.endswith(b"\n# after\n")
    body = want[len(b"# kept\n"):-len(b"# after\n")]
    app = tmp_path / "append.fq"
    fd = os.open(app, os.O_WRONLY | os.O_CREAT | os.O_APPEND)
    f.write(fd, newq)
    os.close(fd)
    assert app.read_bytes() == body
    r, w = os.pipe()
    got = []
    t = threading.Thread(target=lambda: got.append(b"".join(iter(lambda: os.read(r, 1 << 20), b""))))
    t.start()
    f.write(w, newq)
    os.close(w)
    t.join()
    os.close(r)
    assert got[0] == body


def test_open_is_tolerant_like_pysam(tmp_path):
    """Blank lines at the end of the file, gzip without the .gz suffix, a named pipe instead of a file."""
    import shutil
    import threading
    rng = np.random.default_rng(7)
    recs = _random_records(rng, 301, 25)
    plain = tmp_path / "x.fq"
    _write(plain, recs)
    want = fastx.NativeFastq(plain, threads=3)
    ws, wq = want.pack()
    with open(plain, "rb") as fh:
        body = fh.read()
    for tail in (b"\n", b"\n\n\n", b"\r\n"):
        p = tmp_path / "blank.fq"
        p.write_bytes(body + tail)
        f = fastx.NativeFastq(p, threads=3)
        assert f.N == want.N and f.L == want.L
        s, q = f.pack()
        assert np.array_equal(s, ws) and np.array_equal(q, wq) and f.name(f.N - 1) == want.name(want.N - 1)
        f.close()
    gz = tmp_path / "x.fq.gz"
    _write(gz, recs)
    shutil.copy(gz, tmp_path / "disguised.fastq")   # gzip bytes, no .gz suffix
    f = fastx.NativeFastq(tmp_path / "disguised.fastq", threads=2)
    s, q = f.pack()
    assert np.array_equal(s, ws) and np.array_equal(q, wq)
    f.close()
    fifo = tmp_path / "pipe.fq"
    os.mkfifo(fifo)
    feeder = threading.Thread(target=lambda: open(fifo, "wb").write(body))
    feeder.start()
    f = fastx.NativeFastq(fifo, threads=2)
    feeder.join()
    s, q = f.pack()
    assert f.N == want.N and np.array_equal(s, ws) and np.array_equal(q, wq)
    f.close()
    want.close()


@pytest.mark.parametrize("flags", [os.O_WRONLY, os.O_RDWR])
def test_writer_mapped_equals_plain(tmp_path, monkeypatch, flags):
    """The writer maps the output file (reopened read-write through /proc when the descriptor is write-only, as a
    shell redirection is) and must produce the bytes of the pwrite path; text already in the file is kept."""
    rng = np.random.default_rng(8)
    recs = _random_records(rng, 20_011, 31)
    path = tmp_path / "x.fq"
    _write(path, recs)
    f = fastx.NativeFastq(path, threads=6)
    out = rng.integers(0, 60, size=(f.N, f.L)).astype(np.uint8)
    texts = []
    for no_mmap in ("", "1"):
        if no_mmap:
            monkeypatch.setenv("KBBQ_FASTQ_NO_MMAP", "1")
        p = tmp_path / ("out%s.fq" % no_mmap)
        fd = os.open(p, flags | os.O_CREAT | os.O_TRUNC, 0o600)
        os.write(fd, b"# header line\n")
        f.write(fd, out[:5000], 0, 5000)
        f.write(fd, out[5000:], 5000, f.N - 5000)   # appends where the first call stopped
        os.close(fd)
        texts.append(p.read_bytes())
    assert texts[0] == texts[1] and texts[0].startswith(b"# header line\n@r0/1")
    lines = texts[0].decode().split("\n")
    assert len(lines) == 1 + 4 * f.N + 1
    assert lines[1 + 4 * 7 + 3] == "".join(chr(33 + int(v)) for v in out[7])
    # the in-memory formatter is the same text
    import ctypes as C
    from kbbq import _native
    nbytes = C.c_int64(0)
    assert _native.lib().kbbq_fastq_format_size(f._h, 0, f.N, 4, C.byref(nbytes)) == 0
    buf = np.empty(nbytes.value, np.uint8)
    assert _native.lib().kbbq_fastq_format(f._h, 0, f.N, _native.ptr(out), _native.ptr(buf), nbytes.value, 4) == 0
    assert buf.tobytes() == texts[0][len(b"# header line\n"):]
    # a descriptor opened without O_TRUNC over a longer file (`1<>file`): the records overwrite their share of it and
    # the bytes behind them stay, mapped as written
    body = texts[0][len(b"# header line\n"):]
    old = b"# header line\n" + bytes(range(1, 251)) * (len(body) // 250 + 40)
    longer = []
    for no_mmap in ("", "1"):
        monkeypatch.delenv("KBBQ_FASTQ_NO_MMAP", raising=False)
        if no_mmap:
            monkeypatch.setenv("KBBQ_FASTQ_NO_MMAP", "1")
        p = tmp_path / ("longer%s.fq" % no_mmap)
        p.write_bytes(old)
        fd = os.open(p, flags)
        os.lseek(fd, len(b"# header line\n"), os.SEEK_SET)
        f.write(fd, out[:5000], 0, 5000)
        f.write(fd, out[5000:], 5000, f.N - 5000)
        assert os.lseek(fd, 0, os.SEEK_CUR) == len(b"# header line\n") + len(body)
        os.close(fd)
        longer.append(p.read_bytes())
    assert longer[0] == longer[1] == b"# header line\n" + body + old[len(b"# header line\n") + len(body):]
    f.close()


@pytest.mark.parametrize("final", [True, False])
def test_uniform_record_index_equals_general_scan(tmp_path, monkeypatch, final):
    """The header-only index of uniform files (every thread finds the first record of its share of the bytes and
    the walks have to meet) against the general newline scan, on a file built to mislead the search for a record
    start: most quality lines begin with '@', and headers are exactly as long as a read, so that a quality line
    taken for a header finds a line end where it expects one."""
    rng = np.random.default_rng(17)
    L, n = 23, 120_000   # ~6 MB: several threads take part
    bases = np.frombuffer(b"ACGTN", np.uint8)[rng.integers(0, 5, (n, L))]
    quals = rng.integers(35, 74, (n, L)).astype(np.uint8)
    quals[rng.random(n) < 0.8, 0] = ord("@")
    quals[rng.random(n) < 0.3, :] = ord("@")
    lines = []
    for i in range(n):
        name = ("r%d/%d" % (i // 2, 1 + (i & 1))).ljust(L - 1, "x") if i % 3 else "r%d/%d" % (i // 2, 1 + (i & 1))
        lines.append(b"@" + name.encode() + b"\n" + bases[i].tobytes() + b"\n+\n" + quals[i].tobytes())
    text = b"\n".join(lines) + (b"\n" if final else b"")
    p = tmp_path / "tricky.fq"
    p.write_bytes(text)
    got = {}
    for general in ("", "1"):
        if general:
            monkeypatch.setenv("KBBQ_FASTQ_GENERAL_INDEX", "1")
        for threads in (1, 7):
            f = fastx.NativeFastq(p, threads=threads)
            assert f.N == n and f.L == L
            seq, qual = f.pack()
            got[(general, threads)] = (seq, qual, [f.name(i) for i in (0, 1, n // 2, n - 2, n - 1)])
            f.close()
    ref = got[("1", 1)]
    assert np.array_equal(ref[0], bases) and np.array_equal(ref[1], quals - 33)
    for key, (seq, qual, names) in got.items():
        assert np.array_equal(seq, ref[0]) and np.array_equal(qual, ref[1]) and names == ref[2], key
    # one record in the middle a base short: both paths agree that the reads differ in length
    bad = lines[:]
    bad[n // 2] = bad[n // 2].replace(b"\n+\n", b"\n+\n", 1)[:len(bad[n // 2]) - 1]
    seq_line = bad[n // 2].split(b"\n")
    seq_line[1] = seq_line[1][:-1]
    bad[n // 2] = b"\n".join(seq_line)
    p.write_bytes(b"\n".join(bad) + b"\n")
    monkeypatch.delenv("KBBQ_FASTQ_GENERAL_INDEX")
    f = fastx.NativeFastq(p, threads=7)
    assert f.N == n and f.L == -1
    f.close()


@pytest.mark.parametrize("pool", ["1", "0"])
def test_parallel_loops_from_several_callers(tmp_path, monkeypatch, pool):
    """The native loops share one pool of worker threads; several callers may be inside it at once (both FASTQ
    files of a run are indexed at the same time).  Same results as a thread per index (KBBQ_FASTQ_NO_POOL)."""
    import threading
    if pool == "0":
        monkeypatch.setenv("KBBQ_FASTQ_NO_POOL", "1")
    rng = np.random.default_rng(23)
    recs = _random_records(rng, 30_000, 60)
    p = tmp_path / "x.fq"
    _write(p, recs)
    want_seq = np.array([list(r[2].encode()) for r in recs], np.uint8)
    errors = []

    def work(k):
        try:
            for rep in range(3):
                f = fastx.NativeFastq(p, threads=2 + (k + rep) % 7)
                assert f.N == len(recs) and f.L == 60
                rg, second, keys = f.infer(True)
                seq, qual = f.pack()
                assert np.array_equal(seq, want_seq)
                assert len(keys) == 5 and int(second.sum()) == len(recs) // 2
                f.close()
        except Exception as e:   # noqa: BLE001 -- reported by the main thread
            errors.append(repr(e))

    callers = [threading.Thread(target=work, args=(k,)) for k in range(6)]
    for c in callers:
        c.start()
    for c in callers:
        c.join(timeout=120)
    assert not any(c.is_alive() for c in callers), "a caller is stuck in the worker pool"
    assert errors == []
