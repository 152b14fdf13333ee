"""FASTQ input (utb_searcher_set_input, utb_frame_fastq_records): the host framer against a Python restatement of
the 4-line rules, and on the GPU the search of a FASTQ file against the search of the FASTA made of its headers and
sequence lines (fq2fa), with and without quality masking."""
import os
import threading

import numpy as np
import pytest

import conftest  # noqa: F401  (puts the repo root on sys.path)
from oracle import oracle_api
from conftest import CASES, GOLD, gold

LINELEN = 1 << 24
FQ_NOHEADER, FQ_NOSEPARATOR, FQ_QUALLEN, FQ_TOOLONG, FQ_TRUNCATED = 1, 2, 3, 4, 5


# ---- building FASTQ from FASTA ---------------------------------------------------------------------------------
def _fasta_lines(data):
    """[(header line, sequence line)] of a linearised FASTA, line ends kept except a missing last one."""
    lines = data.split(b"\n")
    if data.endswith(b"\n"):
        lines = lines[:-1]
    assert len(lines) % 2 == 0
    return list(zip(lines[0::2], lines[1::2]))


def to_fastq(data, seed, final_newline=None):
    """FASTQ whose fq2fa is `data` (a well-formed FASTA): seeded qualities in '!'..'J'; every third record repeats
    its name on the '+' line; about a third of the quality lines begin with '@' and some with '+'.  A sequence line
    ending in '\\r' gets a quality line ending in '\\r'."""
    rng = np.random.default_rng(seed)
    out = []
    for i, (h, s) in enumerate(_fasta_lines(data)):
        cr = s.endswith(b"\r")
        n = len(s) - cr
        q = rng.integers(33, 75, n, dtype=np.uint8)
        if n and i % 3 == 1:
            q[0] = ord("@")
        elif n and i % 7 == 2:
            q[0] = ord("+")
        sep = b"+" + h[1:].split(b" ")[0].rstrip(b"\r") if i % 3 == 0 else b"+"
        out.append(b"@" + h[1:] + b"\n" + s + b"\n" + sep + (b"\r" if cr else b"") + b"\n" + q.tobytes() + (b"\r" if cr else b"") + b"\n")
    fq = b"".join(out)
    if final_newline is False or (final_newline is None and not data.endswith(b"\n")):
        fq = fq[:-1]
    return fq


def fq2fa(fq, min_qual=0):
    """The FASTA the FASTQ search must equal: '@' -> '>', lines 3 and 4 dropped; with min_qual, bases whose quality
    byte is below 33 + min_qual replaced by 'N'."""
    lines = fq.split(b"\n")
    if fq.endswith(b"\n"):
        lines = lines[:-1]
    out = []
    for r in range(len(lines) // 4):
        h, s, q = lines[4 * r], lines[4 * r + 1], lines[4 * r + 3]
        if min_qual:
            cr = s.endswith(b"\r")
            b = np.frombuffer(s[:len(s) - cr], dtype=np.uint8).copy()
            qa = np.frombuffer(q[:len(b)], dtype=np.uint8)
            b[qa < 33 + min_qual] = ord("N")
            s = b.tobytes() + (b"\r" if cr else b"")
        out.append(b">" + h[1:] + b"\n" + s + b"\n")
    return b"".join(out)


def py_frame_fastq(data):
    """The 4-line rules restated: ([(name, seq, qual)], (1-based bad record, code) or (0, 0))."""
    if not data:
        return [], (0, 0)
    lines = data.split(b"\n")
    ends = [1] * len(lines)
    if data.endswith(b"\n"):
        lines = lines[:-1]
        ends = ends[:-1]
    else:
        ends[-1] = 0
    recs = []
    for r in range(len(lines) // 4):
        ln = lines[4 * r:4 * r + 4]
        span = [len(x) + e for x, e in zip(ln, ends[4 * r:4 * r + 4])]
        h, s, p, q = ln
        s = s[:-1] if s.endswith(b"\r") else s
        q = q[:-1] if q.endswith(b"\r") else q
        if max(span) >= LINELEN:
            return recs, (r + 1, FQ_TOOLONG)
        if h[:1] != b"@":
            return recs, (r + 1, FQ_NOHEADER)
        if p[:1] != b"+":
            return recs, (r + 1, FQ_NOSEPARATOR)
        if len(q) != len(s):
            return recs, (r + 1, FQ_QUALLEN)
        recs.append((h[1:].split(b" ")[0], s, q))
    if len(lines) % 4:
        return recs, (len(recs) + 1, FQ_TRUNCATED)
    return recs, (0, 0)


def _odd_inputs():
    rng = np.random.default_rng(7)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    recs = []
    for n in range(0, 97):                                          # every length residue mod 32, three times
        s = acgt[rng.integers(0, 4, n)].tobytes()
        q = rng.integers(33, 75, n, dtype=np.uint8).tobytes()
        recs.append(b"@len%d some description\n%s\n+\n%s\n" % (n, s, q))
    body = b"".join(recs)
    return {
        "residues": body,
        "residues_no_final_newline": body[:-1],
        "crlf": body.replace(b"\n", b"\r\n"),
        "crlf_no_final_newline": body.replace(b"\n", b"\r\n")[:-1],
        "empty_reads": b"@e1\n\n+\n\n@e2 x\n\n+e2\n\n@x\nACGT\n+\nIIII\n@e3\n\n+\n\n",
        "names": b"@a b\tc\nAC\n+\nII\n@tab\there x\nGT\n+\n@@\n@\nA\n+\n+\n@ lead\nC\n+@\nI\n@a\rb c\r\nG\r\n+\r\nI\r\n",
        "qual_starts_at_and_plus": b"@r1\nACGT\n+\n@III\n@r2\n+CGT\n+\n+III\n@r3\nA\n+\n@\n",
        "single_no_newline": b"@r\nACGT\n+\nIIII",
        "nul_is_an_ordinary_byte": b"@n\0ame x\nAC\0GT\n+\nII\0II\n@\0\n\0\n+\n\0\n",
        "golden_toyA": to_fastq(open(gold("toyA_reads.fa"), "rb").read(), 1),
        "golden_edge": to_fastq(open(gold("edge_reads.fa"), "rb").read(), 2),
    }


def _malformed(good):
    """Each malformed case as (name, bytes, (record, code)) placed after the records of `good`."""
    n = good.count(b"\n") // 4
    return [
        ("noheader", good + b"r\nACGT\n+\nIIII\n@ok\nA\n+\nI\n", (n + 1, FQ_NOHEADER)),
        ("noseparator", good + b"@r\nACGT\n-\nIIII\n", (n + 1, FQ_NOSEPARATOR)),
        ("quallen", good + b"@r\nACGT\n+\nIII\n@ok\nA\n+\nI\n", (n + 1, FQ_QUALLEN)),
        ("quallen_two_cr", good + b"@r\r\nACGT\r\n+\r\nIIII\r\r\n@ok\nA\n+\nI\n", (n + 1, FQ_QUALLEN)),
        ("wrapped", good + b"@r\nACGT\nACGT\n+\nIIII\nIIII\n", (n + 1, FQ_NOSEPARATOR)),
        ("toolong", good + b"@r\n" + b"A" * LINELEN + b"\n+\n" + b"I" * LINELEN + b"\n", (n + 1, FQ_TOOLONG)),
        ("truncated", good + b"@r\nACGT\n+\n", (n + 1, FQ_TRUNCATED)),
        ("truncated_header_only", good + b"@r", (n + 1, FQ_TRUNCATED)),
        # a long read whose quality line is empty, then a small record that ends the input: the chunk ends shortly
        # after the flagged record, whose quality line is 10 MB shorter than its sequence
        ("long_read_short_quality", good + b"@long\n" + b"A" * 10_000_000 + b"\n+\n\n@s\nA\n+\nI\n", (n + 1, FQ_QUALLEN)),
    ]


# ---- CPU: the host framer -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("threads", [1, 4, 16])
def test_fastq_framer_matches_python_rules(built, threads):
    from utree_b200 import capi
    for name, data in _odd_inputs().items():
        want, err = py_frame_fastq(data)
        assert err == (0, 0), name
        rc, used, recs, e = capi.frame_fastq_records(data, eof=True, threads=threads)
        assert (rc, e) == (0, (0, 0)), (name, capi.lib().utb_last_error())
        assert recs == want, name
        assert used == len(data), name


@pytest.mark.parametrize("threads", [1, 4, 16])
def test_fastq_framer_reports_the_first_bad_record(built, threads):
    from utree_b200 import capi
    good = _odd_inputs()["golden_toyA"]
    for name, data, where in _malformed(good):
        want, err = py_frame_fastq(data)
        assert err == where, name
        rc, used, recs, e = capi.frame_fastq_records(data, eof=True, threads=threads)
        assert rc == 3 and e == where, (name, e)
        assert recs == want, name
        assert f"[record {where[0]}]".encode() in capi.lib().utb_last_error(), name
    # two bad records: the first one decides, whichever worker finds it
    data = b"@a\nA\n+\nI\n" * 5000 + b"@b\nAC\n+\nI\n" + b"@a\nA\n+\nI\n" * 5000 + b"x\nA\n+\nI\n"
    rc, used, recs, e = capi.frame_fastq_records(data, eof=True, threads=threads)
    assert (rc, e, len(recs)) == (3, (5001, FQ_QUALLEN), 5000)


def test_fastq_framer_carries_an_incomplete_record(built):
    """Without EOF an incomplete last record is left for the next buffer, not reported as truncated."""
    from utree_b200 import capi
    data = b"@a\nACGT\n+\nIIII\n@b\nGG\n+\nII\n@c\nAC\n+"
    rc, used, recs, e = capi.frame_fastq_records(data, eof=False, threads=3)
    assert (rc, e) == (0, (0, 0)) and [r[0] for r in recs] == [b"a", b"b"] and data[used:] == b"@c\nAC\n+"
    rc, used, recs, e = capi.frame_fastq_records(data, eof=False, threads=2, max_reads=1)
    assert rc == 0 and [r[0] for r in recs] == [b"a"] and data[used:].startswith(b"@b\n")


def test_fastq_input_arguments_are_checked(built):
    from utree_b200 import capi
    import ctypes as C
    L = capi.lib()
    L.utb_searcher_set_input.argtypes = [C.c_void_p, C.c_int, C.c_uint32]
    assert L.utb_searcher_set_input(None, capi.INPUT_FASTQ, 0) == 1


# ---- GPU ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu(built, ctrs):
    from utree_b200 import capi
    assert capi.device_count() >= 1
    state = {}
    for name, path in ctrs.items():
        ctr = capi.Ctr(path)
        state[name] = (ctr, oracle_api.OracleDb(path))
    yield state
    for ctr, orc in state.values():
        orc.free(); ctr.close()


def _searcher(ctr, env=None, devices=(0,), threads=4, shallow=False, fastq=True, min_qual=0):
    from utree_b200 import capi
    env = env or {}
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        s = capi.Searcher(ctr, devices=devices, host_threads=threads)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    if shallow:
        s.set_shallow(True)
    if fastq:
        s.set_input(True, min_qual)
    return s


FRAMING = [{}, {"UTB_HOST_FRAME": "1"}]


@pytest.mark.gpu
@pytest.mark.parametrize("env", FRAMING, ids=["device", "host"])
def test_fastq_search_gives_the_golden_outputs(gpu, tmp_path, env):
    """Every golden read set as FASTQ: the reference's output on the FASTA, through a file and through memory, on
    two virtual devices (batches dealt over both)."""
    for i, (db, reads, out, rc) in enumerate(CASES):
        fa = open(gold(reads), "rb").read()
        fq = to_fastq(fa, i)
        p = str(tmp_path / (reads + ".fq"))
        open(p, "wb").write(fq)
        want = open(gold(out), "rb").read()
        s = _searcher(gpu[db][0], env, devices=(0, 0))
        try:
            o = str(tmp_path / "o.out")
            r, ex, st = s.search_file(p, o, do_rc=bool(rc))
            assert (r, ex) == (0, 0) and open(o, "rb").read() == want, (reads, out)
            r, ex, text, st2 = s.search_mem(fq, do_rc=bool(rc))
            assert (r, ex) == (0, 0) and text == want, (reads, out)
            assert st["reads"] == st2["reads"] == len(_fasta_lines(fa)) and st["good_finds"] == st2["good_finds"]
        finally:
            s.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("env", FRAMING, ids=["device", "host"])
def test_fastq_shallow_search_gives_the_golden_outputs(gpu, tmp_path, env):
    import json
    for name, m in sorted(json.load(open(os.path.join(GOLD, "meta_shallow.json"))).items()):
        fq = to_fastq(open(gold(m["reads"]), "rb").read(), 5)
        s = _searcher(gpu[m["db"]][0], env, shallow=True)
        try:
            r, ex, text, st = s.search_mem(fq, do_rc=bool(m["rc"]))
            assert (r, ex) == (0, 0) and text == open(gold(name), "rb").read(), name
            assert [f"Good finds: {st['good_finds']}", f"Searched {st['reads']} queries"] == m["stdout_tail"], name
        finally:
            s.destroy()


def _big_fastq():
    """About 240 MB of FASTQ, a third of whose quality lines begin with '@': several device chunks."""
    one = open(gold("toyA_reads.fa"), "rb").read() + open(gold("toyB_reads.fa"), "rb").read()
    unit = to_fastq(one, 11)
    return unit * (240_000_000 // len(unit) + 1), fq2fa(unit) * (240_000_000 // len(unit) + 1)


@pytest.mark.gpu
def test_fastq_chunk_cuts_over_many_chunks(gpu, tmp_path):
    """Zero copy from a page-locked buffer, an ordinary buffer, a file and a pipe (host framer): the FASTA search of
    fq2fa of the same input."""
    import torch
    fq, fa = _big_fastq()
    ctr = gpu["toyB_u32"][0]
    s = _searcher(ctr, devices=(0, 0), threads=8, fastq=False)
    try:
        r, ex, want, st_fa = s.search_mem(fa, do_rc=True)
        assert r == 0 and len(want) > 0
        s.set_input(True)
        pinned = torch.empty(len(fq), dtype=torch.uint8, pin_memory=True)
        pinned.numpy()[:] = np.frombuffer(fq, dtype=np.uint8)
        r, ex, text, st = s.search_mem(None, do_rc=True, ptr=pinned.data_ptr(), n=len(fq))
        assert r == 0 and text == want and st["batches"] >= 3 and st["reads"] == st_fa["reads"]
        del pinned
        r, ex, text, st = s.search_mem(fq, do_rc=True)
        assert r == 0 and text == want
        p, o = str(tmp_path / "big.fq"), str(tmp_path / "big.out")
        open(p, "wb").write(fq)
        r, ex, st = s.search_file(p, o, do_rc=True)
        assert r == 0 and open(o, "rb").read() == want
        os.unlink(o)
        fifo = str(tmp_path / "fifo")
        os.mkfifo(fifo)
        def feed():
            with open(fifo, "wb") as f:
                f.write(fq)
        w = threading.Thread(target=feed)
        w.start()
        r, ex, st = s.search_file(fifo, o, do_rc=True)
        w.join()
        assert r == 0 and open(o, "rb").read() == want
    finally:
        s.destroy()


@pytest.mark.gpu
def test_fastq_long_reads_are_masked(gpu, tmp_path):
    """The long reads and reads of up to 16 Mb, masked at min_qual 20: a read is spread over as many mask threads as
    it has 32-base groups.  The checker searches the masked fq2fa FASTA.  The searcher's 33 MiB batches cannot hold a
    FASTQ record of four maximal lines, so switching to FASTQ gives it larger ones."""
    ctr, orc = gpu["toyA"]
    long_fa = open(gold("long_reads.fa"), "rb").read()
    seqs = b"".join(s for _, s in _fasta_lines(long_fa))
    huge = seqs * (16_777_221 // len(seqs) + 1)
    fa = long_fa + b">huge1 16 Mb\n" + huge[:16_000_000] + b"\n>huge2\n" + huge[7:7 + 16_777_214] + b"\n" + long_fa
    fq = to_fastq(fa, 3)
    for q in (0, 20):
        p, o = str(tmp_path / "m.fa"), str(tmp_path / "m.out")
        open(p, "wb").write(fq2fa(fq, q))
        orc.search_file(p, o, do_rc=True)
        want = open(o, "rb").read()
        for env in FRAMING:
            s = _searcher(ctr, dict(env, UTB_BATCH_MB="33"), min_qual=q)
            try:
                r, ex, text, st = s.search_mem(fq, do_rc=True)
                assert (r, ex) == (0, 0) and text == want, (q, env)
            finally:
                s.destroy()
        if q == 0:
            assert want.startswith(open(gold("long_rc.out"), "rb").read())


@pytest.mark.gpu
@pytest.mark.parametrize("min_qual", [0, 20])
def test_fastq_malformed_input_in_a_late_chunk(gpu, min_qual):
    """Each malformed case after more than one chunk of good records: the same partial output, return code, exit
    code and message whether the device or the host framed the input, with and without masking (the mask kernel
    runs on a device chunk before its verdict is known)."""
    from utree_b200 import capi
    ctr = gpu["toyA"][0]
    unit = to_fastq(open(gold("toyA_reads.fa"), "rb").read(), 4)
    good = unit * (150_000_000 // len(unit))
    sd, sh = _searcher(ctr, {}, min_qual=min_qual), _searcher(ctr, {"UTB_HOST_FRAME": "1"}, min_qual=min_qual)
    try:
        r, ex, want, st = sd.search_mem(good, do_rc=True)
        assert r == 0 and st["batches"] >= 2
        for name, data, (rec, code) in _malformed(good):
            got = []
            for s in (sd, sh):
                r, ex, text, st = s.search_mem(data, do_rc=True)
                got.append((r, ex, text, capi.lib().utb_last_error()))
            assert got[0] == got[1], name
            assert got[0][:3] == (3, 2, want), name
            assert f"[record {rec}]".encode() in got[0][3], (name, got[0][3])
        r, ex, text, st = sd.search_mem(good, do_rc=True)                  # the searcher is reusable afterwards
        assert r == 0 and text == want
    finally:
        sd.destroy(); sh.destroy()


FIRST_CHUNK = 4 * LINELEN + 4096        # a FASTQ searcher's first chunk of a large input: the batch floor, one record
                                        # of four maximal lines (pipeline.c, MAX_RECORD)


def _wrong_cut_input():
    """Well-formed FASTQ in which the reader's cut of the first chunk is wrong: the line holding byte FIRST_CHUNK is a
    sequence line that begins with '+', and the line before its header is a quality line that begins with '@'.  So
    the last line of the chunk that begins with '@' and whose line L+2 begins with '+' is that quality line, the chunk
    ends three lines into a record, and the device must reject it for the host framer to take over."""
    unit = to_fastq(open(gold("toyA_reads.fa"), "rb").read(), 6)
    k = (FIRST_CHUNK - 100_000) // len(unit)
    m = (FIRST_CHUNK - k * len(unit) - 7 - 500) // 2                  # the trap's sequence line then holds FIRST_CHUNK
    pad = b"@p\n" + b"A" * m + b"\n+\n" + b"@" + b"I" * (m - 1) + b"\n"
    trap = b"@t\n+" + b"A" * 999 + b"\n+\n" + b"I" * 1000 + b"\n"
    data = unit * k + pad + trap + unit * (40_000_000 // len(unit))
    start = data.rfind(b"\n", 0, FIRST_CHUNK) + 1                     # the line that holds byte FIRST_CHUNK
    assert data[start:start + 1] == b"+" and data[start - 3:start] == b"@t\n"
    assert data.find(b"\n", FIRST_CHUNK) > FIRST_CHUNK and data[data.rfind(b"\n", 0, start - 4) + 1] == ord("@")
    return data


@pytest.mark.gpu
def test_fastq_wrong_chunk_cut_is_rejected_and_reframed(gpu, tmp_path):
    """The cut rule guesses wrong on this input; the device's line-count check rejects the chunk and the host framer
    frames it: memory and file input give the FASTA search of fq2fa, with device and host framing alike."""
    data = _wrong_cut_input()
    ctr = gpu["toyA"][0]
    p, o = str(tmp_path / "w.fq"), str(tmp_path / "w.out")
    open(p, "wb").write(data)
    for env in FRAMING:
        s = _searcher(ctr, env, fastq=False)
        try:
            r, ex, want, st = s.search_mem(fq2fa(data), do_rc=True)
            assert r == 0 and len(want) > 0
            s.set_input(True)
            r, ex, text, st = s.search_mem(data, do_rc=True)
            assert (r, ex) == (0, 0) and text == want, env
            r, ex, st = s.search_file(p, o, do_rc=True)
            assert (r, ex) == (0, 0) and open(o, "rb").read() == want, env
        finally:
            s.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("db,reads", [("toyA", "toyA_reads.fa"), ("dense", "dense_reads.fa")])
def test_fastq_quality_masking(gpu, tmp_path, db, reads):
    """min_qual 0, 20 and 94 against the checker's search of the masked fq2fa FASTA; at 94 every base is masked, so
    there is no line.  The caller's page-locked buffer is left as it was."""
    import torch
    ctr, orc = gpu[db]
    fq = to_fastq(open(gold(reads), "rb").read(), 9)
    pinned = torch.empty(len(fq), dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[:] = np.frombuffer(fq, dtype=np.uint8)
    for q in (0, 20, 94):
        p, o = str(tmp_path / "m.fa"), str(tmp_path / "m.out")
        open(p, "wb").write(fq2fa(fq, q))
        orc.search_file(p, o, do_rc=True)
        want = open(o, "rb").read()
        if q == 94:
            assert want == b""
        for env in FRAMING:
            s = _searcher(ctr, env, min_qual=q)
            try:
                r, ex, text, st = s.search_mem(None, do_rc=True, ptr=pinned.data_ptr(), n=len(fq))
                assert (r, ex) == (0, 0) and text == want, (q, env)
                assert pinned.numpy().tobytes() == fq
            finally:
                s.destroy()


@pytest.mark.gpu
def test_fasta_search_after_fastq_on_the_same_searcher(gpu):
    from utree_b200 import capi
    s = _searcher(gpu["toyA"][0], min_qual=30)
    try:
        fa = open(gold("toyA_reads.fa"), "rb").read()
        r, ex, text, st = s.search_mem(to_fastq(fa, 1), do_rc=True)
        assert r == 0
        with pytest.raises(capi.UtbError):
            s.set_input(False, 30)                                          # masking needs qualities
        s.set_input(False)
        r, ex, text, st = s.search_mem(fa, do_rc=True)
        assert (r, ex) == (0, 0) and text == open(gold("toyA_rc.out"), "rb").read()
    finally:
        s.destroy()
