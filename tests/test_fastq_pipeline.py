"""The native FASTQ pipeline of `kbbq recalibrate -f` (kbbq_recalibrate_fastq, csrc/host_api.cu) byte for byte against
the CPU oracle and a formatter written here.

It covers many chunks and a partial last chunk, read groups first seen in a later chunk, every transport of pass 1,
output descriptors of every kind, bad input found in the last read of the last chunk, and the sessions and pinned
slots kept between calls.  The checks made before the GPU is touched (arguments, files, names) run without a GPU; the
rest is marked gpu."""
import contextlib
import ctypes as C
import gzip
import os
import sys
import threading

import numpy as np
import pytest

from kbbq import _native, synth

E_ARG, E_DATA, E_IO, E_FORMAT, E_RAGGED = -1, -4, -5, -6, -7
E_NAME_FIELD, E_NAME_RG, E_NAME_MISMATCH, E_UNSUPPORTED = -8, -9, -10, -12
AFTER = b"# after\n"

# pass-1 transports (host_api.cu: pack_mode); the FASTQ pipeline sends the reads as they are unless KBBQ_FASTQ_PACK
TRANSPORTS = {
    "default": {},
    "nibbles": {"KBBQ_FASTQ_PACK": "1", "KBBQ_HOST_BITMAP": "1"},
    "bitmap": {"KBBQ_FASTQ_PACK": "1", "KBBQ_HOST_BITMAP": "1", "KBBQ_HOST_NO_NIBBLES": "1"},
    "plain": {"KBBQ_FASTQ_PACK": "1", "KBBQ_HOST_NO_BITMAP": "1"},
}
HOOKS = ("KBBQ_FASTQ_CHUNK_READS", "KBBQ_FASTQ_PACK", "KBBQ_HOST_BITMAP", "KBBQ_HOST_NO_NIBBLES", "KBBQ_HOST_NO_BITMAP",
         "KBBQ_FASTQ_NO_MMAP", "KBBQ_FASTQ_NO_FALLOCATE", "KBBQ_HOST_FORCE_STREAMING", "KBBQ_BATCH_READS")


@pytest.fixture(autouse=True)
def _clean_hooks(monkeypatch):
    """Every test starts without the pipeline's environment hooks."""
    for k in HOOKS:
        monkeypatch.delenv(k, raising=False)


def _same(got, want):
    """-> '' when the two byte strings are equal, else where they first differ (no diff of megabytes)."""
    if got == want:
        return ""
    n = min(len(got), len(want))
    i = next((j for j in range(0, n, 4096) if got[j:j + 4096] != want[j:j + 4096]), n)
    i = next((j for j in range(i, min(n, i + 4096)) if got[j] != want[j]), n)
    return "%d vs %d bytes, first difference at %d: %r vs %r" % (len(got), len(want), i, got[max(0, i - 40):i + 40],
                                                                  want[max(0, i - 40):i + 40])


def _comment_headers(path):
    """Give every header of the corrected file a comment, which the output must not carry."""
    with open(path, "rb") as fh:
        lines = fh.read().split(b"\n")
    lines[:-1:4] = [h + b" corrected" for h in lines[:-1:4]]
    with open(path, "wb") as fh:
        fh.write(b"\n".join(lines))


def _fast_names(rg, second, infer_rg):
    """The names synth.write_fastq_fast writes (fixed width, zero-padded)."""
    n = second.size
    idw = max(1, len(str(max(n // 2, 1))))
    rgw = max(1, len(str(int(rg.max()) if n else 0)))
    return ["r%0*d/%d" % (idw, i // 2, int(second[i]) + 1) + ("_RG:Z:g%0*d" % (rgw, int(rg[i])) if infer_rg else "")
            for i in range(n)]


def _first_seen(rgk):
    """Read-group numbers in first-seen order, as kbbq_fastq_infer (kbbq/recalibrate.py:59-64) gives them."""
    keys, first = np.unique(rgk, return_index=True)
    remap = np.zeros(int(keys.max()) + 1, np.uint16)
    remap[keys[np.argsort(first)]] = np.arange(keys.size, dtype=np.uint16)
    return remap[rgk], int(keys.size)


def _format(names, seq, outq):
    """The expected text: '@name / bases / + / chr(q + 33)' per read, written here, not by the library."""
    L = seq.shape[1]
    sb = seq.tobytes()
    qb = (outq.astype(np.int64) + 33).astype(np.uint8).tobytes()
    return b"".join(b"@%s\n%s\n+\n%s\n" % (nm.encode(), sb[i * L:(i + 1) * L], qb[i * L:(i + 1) * L])
                    for i, nm in enumerate(names))


class Case:
    """Two FASTQ files written from kbbq.synth reads (plus edits), and the oracle's answer for them."""

    def __init__(self, d, N, L, R_synth, seed, fast=False, edit=None):
        import oracle
        self.oracle = oracle
        seq, qual, corr, rgk, second = synth.synth_reads(seed, 0, N, L, R_synth)
        if edit is not None:
            edit(seq, qual, corr, rgk, second)
        os.makedirs(d, exist_ok=True)
        self.fu, self.fc = os.path.join(d, "reads.fq"), os.path.join(d, "corrected.fq")
        if fast:
            synth.write_fastq_fast(self.fu, self.fc, seq, qual, corr, rgk, second, infer_rg=True)
            self.names = _fast_names(rgk, second, True)
        else:
            self.names = synth.write_fastq(self.fu, self.fc, seq, qual, corr, rgk, second, infer_rg=True)
        _comment_headers(self.fc)
        self.N, self.L = N, L
        self.seq, self.qual, self.corr, self.rgk, self.second = seq, qual, corr, rgk, second
        self._want = {}

    def expected(self, infer_rg=True, minscore=6):
        """-> (text, R, outq) of the reference for these files."""
        key = (infer_rg, minscore)
        if key not in self._want:
            o = self.oracle
            rg, R = _first_seen(self.rgk) if infer_rg else (np.zeros(self.N, np.uint16), 1)
            pe, pt, de, dt = o.build_tables(self.seq, self.qual, self.corr, rg, self.second, self.L, R, minscore,
                                            threads=os.cpu_count() or 1)
            tabs = o.marginals(pe, pt) + (pe, pt, de, dt)
            outq = o.apply(self.seq, self.qual, rg, self.second, self.L, R, tabs[0], *o.get_delta_qs(*tabs),
                           minscore=minscore)
            self._want[key] = (_format(self.names, self.seq, outq), R, outq)
        return self._want[key]


def _abi(fu, fc, fd, infer_rg=True, minscore=6, threads=4, device=None):
    """kbbq_recalibrate_fastq -> (rc, n_reads_out, n_rg_out, status_out)."""
    n, nrg, st = C.c_int64(-1), C.c_int(-1), C.c_int(-1)
    rc = _native.lib().kbbq_recalibrate_fastq(str(fu).encode(), str(fc).encode(), 1 if infer_rg else 0, minscore, fd,
                                              _native.DEVICE if device is None else device, threads, C.byref(n),
                                              C.byref(nrg), C.byref(st))
    return rc, n.value, nrg.value, st.value


def _run_file(case, path, infer_rg=True, minscore=6, threads=4):
    """One call into a new file; the descriptor must stand right behind the text. -> the file's bytes."""
    fd = os.open(path, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o600)
    try:
        res = _abi(case.fu, case.fc, fd, infer_rg, minscore, threads)
        end = os.lseek(fd, 0, os.SEEK_CUR)
        os.write(fd, AFTER)
    finally:
        os.close(fd)
    with open(path, "rb") as fh:
        got = fh.read()
    return res, end, got


def _check_run(case, path, infer_rg=True, minscore=6, threads=4, what=""):
    want, R, _ = case.expected(infer_rg, minscore)
    (rc, n, nrg, st), end, got = _run_file(case, path, infer_rg, minscore, threads)
    assert (rc, n, nrg, st) == (0, case.N, R, 0), what
    assert end == len(want), what
    msg = _same(got, want + AFTER)
    assert not msg, "%s: %s" % (what, msg)


def _set_env(monkeypatch, env=None, chunk=None):
    for k in HOOKS:
        monkeypatch.delenv(k, raising=False)
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    if chunk is not None:
        monkeypatch.setenv("KBBQ_FASTQ_CHUNK_READS", str(chunk))


@contextlib.contextmanager
def _stdout_on(fd):
    """fd 1 duplicated onto `fd`, as a shell redirection leaves it, with sys.stdout writing to fd 1 (the test runner
    replaces sys.stdout with its own capture)."""
    sys.stdout.flush()
    saved_fd, saved_obj = os.dup(1), sys.stdout
    os.dup2(fd, 1)
    sys.stdout = open(1, "w", closefd=False)
    try:
        yield
    finally:
        sys.stdout.flush()
        sys.stdout = saved_obj
        os.dup2(saved_fd, 1)
        os.close(saved_fd)


def _run_python(files, path, infer_rg=True):
    """kbbq.recalibrate.recalibrate_fastq with stdout on a new file -> the file's bytes."""
    from kbbq import recalibrate
    fd = os.open(path, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o600)
    try:
        with _stdout_on(fd):
            recalibrate.recalibrate_fastq(files, infer_rg=infer_rg)
    finally:
        os.close(fd)
    with open(path, "rb") as fh:
        return fh.read()


def _drain(r):
    """A reader thread for a pipe; -> (thread, list that receives everything read)."""
    got = []
    t = threading.Thread(target=lambda: got.append(b"".join(iter(lambda: os.read(r, 1 << 20), b""))))
    t.start()
    return t, got


# ---- datasets (module scope: the oracle runs once per dataset and setting) ------------------------------------------

def _late_group(seq, qual, corr, rgk, second):
    """A read group (7) that first appears after read 50 000: every third read from there on."""
    rgk[50_001::3] = 7


@pytest.fixture(scope="module")
def ds1(tmp_path_factory, oracle_mod):
    """70 003 reads of 151 bp, one read group, names of varying width."""
    return Case(str(tmp_path_factory.mktemp("ds1")), 70_003, 151, 1, 11)


@pytest.fixture(scope="module")
def ds2(tmp_path_factory, oracle_mod):
    """600 000 reads of 100 bp, 4 read groups, fixed-width names: three default chunks, > 64 MB of output."""
    return Case(str(tmp_path_factory.mktemp("ds2")), 600_000, 100, 4, 12, fast=True)


@pytest.fixture(scope="module")
def ds3(tmp_path_factory, oracle_mod):
    """60 001 reads of 100 bp, 8 read groups, one of them first seen after read 50 000."""
    return Case(str(tmp_path_factory.mktemp("ds3")), 60_001, 100, 7, 13, edit=_late_group)


@pytest.fixture(scope="module")
def ds3g(tmp_path_factory, oracle_mod):
    """20 011 reads of 300 bp, 3 read groups: the generic kernels' range."""
    return Case(str(tmp_path_factory.mktemp("ds3g")), 20_011, 300, 3, 14)


# ---- GPU: chunking --------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [16, 4000, 35_008, 70_003, 1 << 20])
def test_chunks_give_the_reference_bytes(ds1, tmp_path, monkeypatch, chunk):
    """16 reads a chunk (4376 chunks), 4000 (a partial last chunk of 3), 35 008 (two, the second partial) and one."""
    _set_env(monkeypatch, chunk=chunk)
    _check_run(ds1, tmp_path / "out.fq", what="C = %d" % chunk)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [5, 37])
@pytest.mark.parametrize("N", [1, 15, 17, 33])
def test_tiny_files(tmp_path, monkeypatch, oracle_mod, N, L):
    case = Case(str(tmp_path), N, L, 2, 100 + N + L)
    _set_env(monkeypatch, chunk=16)
    _check_run(case, tmp_path / "out.fq", what="N = %d, L = %d" % (N, L))


@pytest.mark.gpu
def test_default_chunk_size_and_gzip(ds2, tmp_path):
    """No hook: 262 144 / 262 144 / 75 712 reads, an output the allocation thread covers in several slices; then the
    same reads from a gzip file."""
    _check_run(ds2, tmp_path / "out.fq", what="default chunks")
    want, R, _ = ds2.expected()
    gz = tmp_path / "reads.fq.gz"
    with open(ds2.fu, "rb") as src, gzip.open(gz, "wb", compresslevel=1) as dst:
        dst.write(src.read())
    fd = os.open(tmp_path / "out_gz.fq", os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o600)
    try:
        res = _abi(gz, ds2.fc, fd)
    finally:
        os.close(fd)
    assert res == (0, ds2.N, R, 0)
    msg = _same((tmp_path / "out_gz.fq").read_bytes(), want)
    assert not msg, msg


# ---- GPU: read groups -----------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("infer_rg", [True, False])
@pytest.mark.parametrize("chunk", [1024, 2048, 9008])
def test_read_groups_across_chunks(ds3, tmp_path, monkeypatch, chunk, infer_rg):
    """R = 8: below (read order, resident) and at the segmented layout's chunk bound (32 R 8 reads), and well above
    it; a group first seen in the last chunks.  Without --infer-rg the same files are one read group."""
    _set_env(monkeypatch, chunk=chunk)
    assert ds3.expected(infer_rg)[1] == (8 if infer_rg else 1)
    _check_run(ds3, tmp_path / "out.fq", infer_rg=infer_rg, what="C = %d, infer_rg = %s" % (chunk, infer_rg))


@pytest.mark.gpu
def test_read_groups_generic_kernels(ds3g, tmp_path, monkeypatch):
    _set_env(monkeypatch, chunk=3008)
    _check_run(ds3g, tmp_path / "out.fq", what="L = 300, R = 3")


# ---- GPU: data edges ------------------------------------------------------------------------------------------------

def _edges(seq, qual, corr, rgk, second):
    """N bases in the reads and in the corrected reads, qualities 0, 5, 6 and 42, all-N reads, all-42 reads."""
    rng = np.random.default_rng(21)
    N, L = seq.shape
    m = rng.random((N, L)) < 0.25
    qual[m] = rng.choice(np.array([0, 5, 6, 42], np.uint8), int(m.sum()))
    n_read = rng.random((N, L)) < 0.03
    seq[n_read] = ord("N")
    corr[n_read] = ord("N")
    n_corr = rng.random((N, L)) < 0.03
    corr[n_corr] = ord("N")
    seq[7] = corr[7] = ord("N")
    seq[8] = ord("N")
    qual[9] = 42
    qual[10] = 0
    qual[11] = 6
    qual[12] = 5


@pytest.mark.gpu
@pytest.mark.parametrize("transport", ["default", "nibbles", "bitmap"])
@pytest.mark.parametrize("chunk", [4000, None])
def test_data_edges(tmp_path, monkeypatch, oracle_mod, chunk, transport):
    case = Case(str(tmp_path), 20_011, 61, 2, 22, edit=_edges)
    assert case.second.any() and not case.second.all()
    _set_env(monkeypatch, TRANSPORTS[transport], chunk)
    _check_run(case, tmp_path / "out.fq", what="C = %s, %s" % (chunk, transport))


# ---- GPU: minscore and threads through the ABI ----------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("minscore", [1, 6, 20])
def test_minscore_and_threads(ds3, tmp_path, monkeypatch, minscore):
    _set_env(monkeypatch, chunk=2048)
    for threads in (1, 2, 0):
        _check_run(ds3, tmp_path / "out.fq", minscore=minscore, threads=threads,
                   what="minscore = %d, threads = %d" % (minscore, threads))


# ---- GPU: transports ------------------------------------------------------------------------------------------------

def _h2d_bytes(n, L, R, chunk, transport):
    """Bytes pass 1 sends to the device: qual, seq unless nibbles, rg when R > 1, mate flags, then the corrected
    reads as they are, as nibbles or as a bit map."""
    C16 = min((chunk + 15) // 16 * 16, (n + 15) // 16 * 16)
    total = 0
    for r0 in range(0, n, C16):
        m = min(C16, n - r0)
        nb = m * L
        total += nb + (0 if transport == "nibbles" else nb) + (2 * m if R > 1 else 0) + m
        total += {"nibbles": (nb + 1) // 2, "bitmap": (nb + 31) // 32 * 4}.get(transport, nb)
    return total


@pytest.mark.gpu
@pytest.mark.parametrize("transport", ["nibbles", "bitmap", "plain"])
def test_transports(ds1, ds3, tmp_path, monkeypatch, transport):
    """Every transport of pass 1 on one and on eight read groups at several chunk sizes; the bytes sent up show that
    the transport asked for is the one taken."""
    for case, chunks in ((ds1, (4000, 35_008)), (ds3, (1024, 2048, 9008))):
        for chunk in chunks:
            _set_env(monkeypatch, TRANSPORTS[transport], chunk)
            _check_run(case, tmp_path / "out.fq", what="%s, C = %d" % (transport, chunk))
            up, down = C.c_int64(0), C.c_int64(0)
            assert _native.lib().kbbq_host_last_traffic(_native.DEVICE, C.byref(up), C.byref(down)) == 0
            R = case.expected()[1]
            assert up.value == _h2d_bytes(case.N, case.L, R, chunk, transport), (transport, chunk)
            assert down.value == case.N * case.L


# ---- GPU: output descriptors ----------------------------------------------------------------------------------------

PREFIX = (b"# text already in the file\n" * 200)


@pytest.mark.gpu
@pytest.mark.parametrize("mode,prefix,flags,env", [
    ("new", 0, os.O_WRONLY, {}),
    ("new", 7, os.O_WRONLY, {}),
    ("new", 4101, os.O_WRONLY, {}),
    ("new", 4101, os.O_RDWR, {}),
    ("new", 7, os.O_WRONLY, {"KBBQ_FASTQ_NO_FALLOCATE": "1"}),
    ("new", 7, os.O_WRONLY, {"KBBQ_FASTQ_NO_MMAP": "1"}),
    ("append", 7, os.O_WRONLY | os.O_APPEND, {}),
    ("longer", 4101, os.O_RDWR, {}),
    ("longer", 7, os.O_WRONLY, {}),
    ("longer", 4101, os.O_RDWR, {"KBBQ_FASTQ_NO_MMAP": "1"}),
], ids=["wronly-0", "wronly-7", "wronly-4101", "rdwr-4101", "no-fallocate", "no-mmap", "append", "longer-rdwr",
        "longer-wronly", "longer-no-mmap"])
def test_output_descriptors(ds1, tmp_path, monkeypatch, mode, prefix, flags, env):
    """The text lands at the descriptor's offset (not page-aligned), the bytes before it and behind it stay as write()
    leaves them, and the descriptor stands right behind the text."""
    want, R, _ = ds1.expected()
    _set_env(monkeypatch, env, 4000)
    head = PREFIX[:prefix]
    tail = bytes(range(1, 251)) * ((len(want) + 9000) // 250) if mode == "longer" else b""
    p = tmp_path / "out.fq"
    p.write_bytes(head + tail)
    fd = os.open(p, flags | (os.O_TRUNC if mode == "new" else 0))
    try:
        if mode == "new":
            os.write(fd, head)
        else:
            os.lseek(fd, len(head), os.SEEK_SET)
        res = _abi(ds1.fu, ds1.fc, fd)
        end = os.lseek(fd, 0, os.SEEK_CUR)
        os.write(fd, AFTER)
    finally:
        os.close(fd)
    assert res == (0, ds1.N, R, 0)
    assert end == len(head) + len(want)
    expect = head + want + AFTER + tail[len(want) + len(AFTER):]
    msg = _same(p.read_bytes(), expect)
    assert not msg, msg


@pytest.mark.gpu
def test_output_into_a_pipe(ds1, tmp_path, monkeypatch):
    want, R, _ = ds1.expected()
    _set_env(monkeypatch, chunk=4000)
    r, w = os.pipe()
    t, got = _drain(r)
    try:
        res = _abi(ds1.fu, ds1.fc, w)
        os.write(w, AFTER)
    finally:
        os.close(w)
        t.join()
        os.close(r)
    assert res == (0, ds1.N, R, 0)
    msg = _same(got[0], want + AFTER)
    assert not msg, msg


# ---- GPU: bad input in the last read of the last chunk --------------------------------------------------------------

def _spoil_last_read(case, d, kind):
    """Copies of the case's files with the last read spoilt at its middle base. -> (reads, corrected)."""
    L = case.L
    fu, fc = os.path.join(d, "bad_reads.fq"), os.path.join(d, "bad_corrected.fq")
    u, c = bytearray(open(case.fu, "rb").read()), bytearray(open(case.fc, "rb").read())
    j = L // 2
    q_at = len(u) - 1 - L + j                     # the last line is the last read's qualities
    s_at = len(u) - 1 - L - 3 - L + j             # its bases: '\n+\n' before the qualities
    cs_at = len(c) - 1 - L - 3 - L + j
    if kind == "quality43":
        u[q_at] = ord("L")
    elif kind == "base":
        u[s_at] = c[cs_at] = ord("X")
        u[q_at] = ord("I")                        # a usable site
    elif kind == "quality_char":
        u[q_at] = ord(" ")                        # below '!': the tokeniser's KBBQ_E_FORMAT, in the middle of pass 1
    open(fu, "wb").write(bytes(u))
    open(fc, "wb").write(bytes(c))
    return fu, fc


BAD = {"quality43": (E_DATA, _native.FLAG_QUAL_RANGE, IndexError),
       "base": (E_DATA, _native.FLAG_BAD_BASE, TypeError),
       "quality_char": (E_FORMAT, 0, ValueError)}


@pytest.fixture(scope="module")
def ds_err(tmp_path_factory, oracle_mod):
    """9 001 reads of 151 bp, two read groups: at 4000 reads a chunk the last chunk holds one read."""
    return Case(str(tmp_path_factory.mktemp("ds_err")), 9_001, 151, 2, 31)


@pytest.mark.gpu
@pytest.mark.parametrize("transport", ["default", "nibbles"])
@pytest.mark.parametrize("kind", sorted(BAD))
def test_bad_input_in_the_last_chunk_writes_nothing(ds_err, tmp_path, monkeypatch, kind, transport):
    """The call reports the error and writes nothing: a regular file keeps its bytes, size and offset (one the call
    would have grown and one longer than the text), a pipe receives no byte, and the Python driver raises the
    reference's exception.  The next call, on good files, gives the right bytes."""
    rc_want, flag, exc = BAD[kind]
    _set_env(monkeypatch, TRANSPORTS[transport], 4000)
    fu, fc = _spoil_last_read(ds_err, str(tmp_path), kind)
    want, R, _ = ds_err.expected()
    for longer in (False, True):
        p = tmp_path / "out.fq"
        before = PREFIX[:4101] + (bytes(range(1, 251)) * 16_000 if longer else b"")
        p.write_bytes(before)
        fd = os.open(p, os.O_WRONLY)
        try:
            os.lseek(fd, 4101, os.SEEK_SET)
            rc, n, nrg, st = _abi(fu, fc, fd)
            assert os.lseek(fd, 0, os.SEEK_CUR) == 4101
        finally:
            os.close(fd)
        assert rc == rc_want and (st & flag) == flag, (rc, st)
        assert n == ds_err.N and nrg == R
        assert os.path.getsize(p) == len(before)
        assert p.read_bytes() == before
    r, w = os.pipe()
    t, got = _drain(r)
    try:
        rc = _abi(fu, fc, w)[0]
    finally:
        os.close(w)
        t.join()
        os.close(r)
    assert rc == rc_want and got[0] == b""
    with pytest.raises(exc):
        _run_python((fu, fc), tmp_path / "py.fq")
    assert os.path.getsize(tmp_path / "py.fq") == 0
    _check_run(ds_err, tmp_path / "good.fq", what="after the error")


# ---- GPU: cached sessions and pinned slots --------------------------------------------------------------------------

@pytest.mark.gpu
def test_cached_sessions_and_pinned_slots(ds1, ds2, ds3, ds3g, tmp_path, monkeypatch):
    """Calls of other shapes one after another reuse or replace the cached session and the pinned slots; each result
    is checked byte for byte."""
    out = tmp_path / "out.fq"

    def run(case, chunk, what):
        _set_env(monkeypatch, chunk=chunk)
        _check_run(case, out, what=what)

    run(ds1, 4000, "ds1, C = 4000")
    run(ds1, None, "ds1, default C")
    run(ds3, 2048, "ds3")
    _set_env(monkeypatch)
    rg, R = _first_seen(ds3g.rgk)
    got = _native.recalibrate_host(ds3g.seq, ds3g.qual, ds3g.corr, rg, ds3g.second, ds3g.L, R, 6)
    assert np.array_equal(got.astype(np.int16), ds3g.expected()[2]), "host-buffer call on the shared session slot"
    run(ds1, 4000, "ds1, C = 4000 again")
    assert _native.lib().kbbq_host_release(_native.DEVICE) == 0
    run(ds1, 4000, "ds1 after kbbq_host_release")
    run(ds1, 512, "small C")
    run(ds2, None, "large C: larger pinned slots")
    run(ds1, 512, "small C again")


# ---- GPU: the fallbacks give the same bytes -------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"KBBQ_HOST_FORCE_STREAMING": "1"}, {"KBBQ_BATCH_READS": "50000"}],
                         ids=["force-streaming", "batch-reads"])
def test_fallback_paths_give_the_same_bytes(ds2, ds3, tmp_path, monkeypatch, env):
    """KBBQ_HOST_FORCE_STREAMING: the native call returns KBBQ_E_UNSUPPORTED and recalibrate_fastq takes the ReadBatch
    path; KBBQ_BATCH_READS: the streamed session driver.  Both print the pipeline's bytes."""
    if "KBBQ_HOST_FORCE_STREAMING" in env:
        _set_env(monkeypatch, env)
        fd = os.open(tmp_path / "none.fq", os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o600)
        try:
            assert _abi(ds3.fu, ds3.fc, fd)[0] == E_UNSUPPORTED
        finally:
            os.close(fd)
        assert os.path.getsize(tmp_path / "none.fq") == 0
    for case in (ds2, ds3):
        _set_env(monkeypatch, env)
        got = _run_python((case.fu, case.fc), tmp_path / "out.fq")
        msg = _same(got, case.expected()[0])
        assert not msg, msg
    _set_env(monkeypatch)
    got = _run_python((ds3.fu, ds3.fc), tmp_path / "out.fq")
    assert not _same(got, ds3.expected()[0]), "the pipeline through recalibrate_fastq"


# ---- CPU: everything before the device is touched -------------------------------------------------------------------

def _write_pair(d, names, L, corr_names=None, n_corr=None, L_corr=None):
    """Two small FASTQ files: reads named `names`, the corrected ones `corr_names` (default: the same, commented)."""
    rng = np.random.default_rng(len(names) + L)
    fu, fc = os.path.join(d, "u.fq"), os.path.join(d, "c.fq")
    corr_names = names if corr_names is None else corr_names
    n_corr = len(corr_names) if n_corr is None else n_corr
    L_corr = L if L_corr is None else L_corr
    with open(fu, "w") as hu:
        for nm in names:
            hu.write("@%s\n%s\n+\n%s\n" % (nm, "".join(rng.choice(list("ACGT"), L)), "I" * L))
    with open(fc, "w") as hc:
        for nm in corr_names[:n_corr]:
            hc.write("@%s corrected\n%s\n+\n%s\n" % (nm, "".join(rng.choice(list("ACGT"), L_corr)), "I" * L_corr))
    return fu, fc


def _names(n, rg=True):
    return ["r%d/%d" % (i // 2, 1 + (i & 1)) + ("_RG:Z:g%d" % (i % 3) if rg else "") for i in range(n)]


@pytest.mark.parametrize("longer", [False, True], ids=["grown", "longer"])
def test_errors_before_the_device_leave_the_output_as_it_was(tmp_path, longer):
    """Every error found before the GPU is touched.  Those found after the output was sized and mapped (the name
    check, the read-group inference) must leave the file's bytes, size and offset exactly as they were: both when the
    call grew the file and when the file is longer than the text would have been."""
    d = str(tmp_path)
    lib = _native.lib()
    n = C.c_int64(0)
    nrg, st = C.c_int(0), C.c_int(0)
    good_u, good_c = _write_pair(d, _names(301), 40)
    assert lib.kbbq_recalibrate_fastq(None, good_c.encode(), 1, 6, 1, 0, 2, C.byref(n), C.byref(nrg), C.byref(st)) == E_ARG
    assert lib.kbbq_recalibrate_fastq(good_u.encode(), None, 1, 6, 1, 0, 2, C.byref(n), C.byref(nrg), C.byref(st)) == E_ARG
    cases = []

    def add(what, rc, mk, infer_rg=True):
        sub = os.path.join(d, what)
        os.makedirs(sub)
        cases.append((what, rc, mk(sub), infer_rg))

    add("bad fd", E_ARG, lambda s: (good_u, good_c))
    add("bad device", E_ARG, lambda s: (good_u, good_c))
    add("missing", E_IO, lambda s: (os.path.join(s, "missing.fq"), _write_pair(s, _names(5), 40)[1]))
    add("counts", E_UNSUPPORTED, lambda s: _write_pair(s, _names(301), 40, n_corr=300))
    add("lengths", E_RAGGED, lambda s: _write_pair(s, _names(301), 40, L_corr=41))
    add("name mismatch", E_NAME_MISMATCH, lambda s: _write_pair(s, _names(301), 40, _names(300) + ["x150/1_RG:Z:g1"]))
    add("no rg field", E_NAME_FIELD, lambda s: _write_pair(s, _names(300) + ["r150/1"], 40))
    add("not rg", E_NAME_RG, lambda s: _write_pair(s, _names(300) + ["r150/1_XX:Z:g1"], 40))
    add("empty", 0, lambda s: _write_pair(s, [], 40))
    for what, rc_want, (fu, fc), infer_rg in cases:
        p = tmp_path / (what.replace(" ", "_") + ".out")
        before = PREFIX[:4101] + (bytes(range(1, 251)) * 400 if longer else b"")
        p.write_bytes(before)
        fd = os.open(p, os.O_WRONLY)
        try:
            os.lseek(fd, 4101, os.SEEK_SET)
            out_fd = -1 if what == "bad fd" else fd
            device = -1 if what == "bad device" else 0
            rc = lib.kbbq_recalibrate_fastq(fu.encode(), fc.encode(), 1 if infer_rg else 0, 6, out_fd, device, 2,
                                            C.byref(n), C.byref(nrg), C.byref(st))
            assert rc == rc_want, (what, rc)
            assert os.lseek(fd, 0, os.SEEK_CUR) == 4101, what
        finally:
            os.close(fd)
        assert os.path.getsize(p) == len(before), what
        assert p.read_bytes() == before, what
        if what == "empty":
            assert (n.value, nrg.value, st.value) == (0, 1, 0)
