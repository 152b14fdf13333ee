"""Wrapped (multi-line) FASTA input (utb_searcher_set_input with UTB_INPUT_FASTA_WRAPPED, utb_frame_wrapped_records):
the host framer against a Python restatement of the rules, and on the GPU the search of wrapped input against the
search of lin(input), the linearised FASTA, which the project already pins against the reference."""
import json
import os
import threading

import numpy as np
import pytest

import conftest  # noqa: F401  (puts the repo root on sys.path)
from oracle import oracle_api
from conftest import BAD_CASES, CASES, GOLD, gold

LINELEN = 1 << 24
MAXSEQ = LINELEN - 2
FW_NOHEADER, FW_TOOLONG = 1, 4
READ_SETS = ["toyA_reads.fa", "toyB_reads.fa", "quirk_reads.fa", "dense_reads.fa", "long_reads.fa", "edge_reads.fa",
             "shallow_reads.fa"]


# ---- building wrapped FASTA ---------------------------------------------------------------------------------------
def _fasta_lines(data):
    """[(header line, sequence line)] of a linearised FASTA, line ends kept except a missing last one."""
    lines = data.split(b"\n")
    if data.endswith(b"\n"):
        lines = lines[:-1]
    assert len(lines) % 2 == 0
    return list(zip(lines[0::2], lines[1::2]))


def rewrap(linear_fasta, widths, crlf=False, blank_lines=0, final_newline=True):
    """The records of a linearised FASTA with each sequence cut into lines: `widths` is a width, or a list of widths
    used in turn (ragged).  crlf: every sequence line ends in '\\r\\n'; blank_lines: that many empty lines after every
    5th sequence line and between records; final_newline=False drops the last '\\n'.  A sequence's trailing '\\r'
    (which the FASTA reader trims) is dropped first."""
    ws = [widths] if isinstance(widths, int) else list(widths)
    eol = b"\r\n" if crlf else b"\n"
    out, k = [], 0
    for h, s in _fasta_lines(linear_fasta):
        s = s[:-1] if s.endswith(b"\r") else s
        out.append(h + b"\n")
        i, j = 0, 0
        while i < len(s):
            w = ws[k % len(ws)]
            k += 1
            out.append(s[i:i + w] + eol)
            i += w
            j += 1
            if blank_lines and j % 5 == 0:
                out.append(eol * blank_lines)
        if blank_lines:
            out.append(b"\n" * blank_lines)
    data = b"".join(out)
    return data if final_newline else data[:-1]


def ragged(seed, n=64):
    return [int(w) for w in np.random.default_rng(seed).integers(1, 200, n)]


def _lines(data):
    """[(line without its end, its length counting the '\\n')]."""
    parts = data.split(b"\n")
    out = [(p, len(p) + 1) for p in parts[:-1]]
    if parts[-1]:
        out.append((parts[-1], len(parts[-1])))
    return out


def py_frame_wrapped(data):
    """The wrapped-FASTA rules restated: ([(name, joined sequence)], (1-based bad record, code) or (0, 0))."""
    if not data:
        return [], (0, 0)
    if data[:1] != b">":
        return [], (1, FW_NOHEADER)
    recs, cur = [], None

    def close(cur):
        name, seq, bad = cur
        if bad or len(seq) > MAXSEQ:
            return False
        recs.append((name, seq))
        return True
    for line, span in _lines(data):
        if line[:1] == b">":
            if cur is not None and not close(cur):
                return recs, (len(recs) + 1, FW_TOOLONG)
            cur = [line[1:].split(b" ")[0], b"", span >= LINELEN]
        else:
            cur[1] += line[:-1] if line.endswith(b"\r") else line
            cur[2] = cur[2] or span >= LINELEN
    if not close(cur):
        return recs, (len(recs) + 1, FW_TOOLONG)
    return recs, (0, 0)


def lin(data):
    """Each record's header line unchanged, then its joined sequence, then '\\n'."""
    out, seq = [], None
    for line, _ in _lines(data):
        if line[:1] == b">":
            if seq is not None:
                out.append(b"".join(seq) + b"\n")
            out.append(line + b"\n")
            seq = []
        else:
            seq.append(line[:-1] if line.endswith(b"\r") else line)
    if seq is not None:
        out.append(b"".join(seq) + b"\n")
    return b"".join(out)


def _odd_inputs():
    inputs = {}
    for name in READ_SETS:
        fa = open(gold(name), "rb").read()
        for w in (1, 31, 32, 33, 60, 80):
            inputs[f"{name}_w{w}"] = rewrap(fa, w)
        inputs[f"{name}_ragged"] = rewrap(fa, ragged(len(name)))
    fa = open(gold("toyA_reads.fa"), "rb").read()
    inputs["crlf"] = rewrap(fa, 60, crlf=True)
    inputs["crlf_no_final_newline"] = rewrap(fa, 60, crlf=True, final_newline=False)
    inputs["final_cr"] = rewrap(fa, 70)[:-1] + b"\r"
    inputs["no_final_newline"] = rewrap(fa, 80, final_newline=False)
    inputs["blank_lines"] = rewrap(fa, ragged(3), blank_lines=2)
    inputs["blank_crlf_lines"] = rewrap(fa, 33, crlf=True, blank_lines=1)
    inputs["header_only"] = b">h1\n>a x\nAC\nGT\n>h2\n>h3 y\n\n>b\nA\n>end"
    inputs["header_only_at_eof"] = b">a\nACGT\n>b\n"
    inputs["gt_and_semicolon_inside"] = b">a\nAC>GT\n;comment\nA>\n>b\tc d\nG\n> lead\nC\n>\n"
    inputs["names"] = b">a b\tc\nAC\n>tab\there x\nGT\n>\nA\n>a\rb c\r\nG\r\n>cr\r\nA\r\r\n"
    inputs["nul_is_an_ordinary_byte"] = b">n\0ame x\nAC\0GT\n\0\n>\0\n\0\n"
    # one record over every worker's segment, between small ones
    inputs["spanning"] = b">s1\nACGT\n>big\n" + b"ACGTTGCA" * 20000 + b"\n" + rewrap(b">x\n" + b"A" * 300000 + b"\n", 61) + b">s2\nA\n"
    return inputs


def _malformed(good):
    """Each malformed case as (name, bytes, (record, code)) placed after the records of `good`."""
    n = good.count(b"\n>") + 1
    return [
        ("header_line_toolong", good + b">" + b"h" * (LINELEN - 2) + b"\nACGT\n>ok\nA\n", (n + 1, FW_TOOLONG)),
        ("sequence_line_toolong", good + b">r\nAC\n" + b"A" * (LINELEN - 1) + b"\n>ok\nA\n", (n + 1, FW_TOOLONG)),
        ("sequence_toolong", good + b">r\n" + rewrap(b">x\n" + b"C" * (MAXSEQ + 1) + b"\n", 997)[3:] + b">ok\nA\n",
         (n + 1, FW_TOOLONG)),
    ]


# ---- CPU: the host framer -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("threads", [1, 4, 16])
def test_wrapped_framer_matches_python_rules(built, threads):
    from utree_b200 import capi
    for name, data in _odd_inputs().items():
        want, err = py_frame_wrapped(data)
        assert err == (0, 0), name
        rc, used, recs, e = capi.frame_wrapped_records(data, eof=True, threads=threads)
        assert (rc, e) == (0, (0, 0)), (name, capi.lib().utb_last_error())
        assert recs == want, name
        assert used == len(data), name


def test_rewrap_is_undone_by_lin():
    for name in READ_SETS:
        fa = open(gold(name), "rb").read()
        want = [(h, s[:-1] if s.endswith(b"\r") else s) for h, s in _fasta_lines(fa)]
        for w in (1, 60, ragged(1)):
            got = _fasta_lines(lin(rewrap(fa, w, crlf=w == 60, blank_lines=1 if w == 1 else 0)))
            assert got == want, name


@pytest.mark.parametrize("threads", [1, 4, 16])
def test_wrapped_framer_reports_the_first_bad_record(built, threads):
    from utree_b200 import capi
    good = rewrap(open(gold("toyA_reads.fa"), "rb").read(), 60)
    for name, data, where in _malformed(good):
        want, err = py_frame_wrapped(data)
        assert err == where, name
        rc, used, recs, e = capi.frame_wrapped_records(data, eof=True, threads=threads)
        assert rc == 3 and e == where, (name, e)
        assert recs == want, name
        assert f"[record {where[0]}]".encode() in capi.lib().utb_last_error(), name
    for data in (b"x\n>a\nACGT\n", b"\n>a\nACGT\n", b";c\n>a\nA\n"):               # leading text or a blank line
        assert py_frame_wrapped(data) == ([], (1, FW_NOHEADER))
        rc, used, recs, e = capi.frame_wrapped_records(data, eof=True, threads=threads)
        assert (rc, recs, e) == (3, [], (1, FW_NOHEADER))
        assert b"[record 1]" in capi.lib().utb_last_error()
    # the base limit: exactly 16777214 bases over short lines pass, one more fails
    seq = b"ACGTTGCAAC" * (MAXSEQ // 10 + 1)
    ok = b">a\nAC\n>lim\n" + rewrap(b">x\n" + seq[:MAXSEQ] + b"\n", 101)[3:] + b">z\nA\n"
    rc, used, recs, e = capi.frame_wrapped_records(ok, eof=True, threads=threads)
    assert (rc, e, [len(s) for _, s in recs]) == (0, (0, 0), [2, MAXSEQ, 1])
    bad = b">a\nAC\n>lim\n" + rewrap(b">x\n" + seq[:MAXSEQ + 1] + b"\n", 101)[3:] + b">z\nA\n"
    rc, used, recs, e = capi.frame_wrapped_records(bad, eof=True, threads=threads)
    assert (rc, e, len(recs)) == (3, (2, FW_TOOLONG), 1)
    # two bad records: the first one decides, whichever worker finds it
    data = b">a\nA\nC\n" * 5000 + b">b\n" + b"A" * LINELEN + b"\n" + b">a\nA\n" * 5000 + b">c\n" + b"T" * LINELEN + b"\n"
    rc, used, recs, e = capi.frame_wrapped_records(data, eof=True, threads=threads)
    assert (rc, e, len(recs)) == (3, (5001, FW_TOOLONG), 5000)


def test_wrapped_framer_carries_the_last_record(built):
    """Without EOF the record after the last header is left for the next buffer; max_reads cuts before a header."""
    from utree_b200 import capi
    data = b">a\nAC\nGT\n>b\nGG\n\n>c\nAC\nG"
    rc, used, recs, e = capi.frame_wrapped_records(data, eof=False, threads=3)
    assert (rc, e) == (0, (0, 0)) and recs == [(b"a", b"ACGT"), (b"b", b"GG")] and data[used:] == b">c\nAC\nG"
    rc, used, recs, e = capi.frame_wrapped_records(data, eof=False, threads=2, max_reads=1)
    assert rc == 0 and recs == [(b"a", b"ACGT")] and data[used:].startswith(b">b\n")
    rc, used, recs, e = capi.frame_wrapped_records(b">only\nACGT\nAC", eof=False, threads=2)
    assert (rc, used, recs) == (0, 0, [])
    rc, used, recs, e = capi.frame_wrapped_records(data, eof=True, threads=5, max_reads=2)
    assert rc == 0 and len(recs) == 2 and data[used:] == b">c\nAC\nG"


def test_wrapped_input_arguments_are_checked(built):
    from utree_b200 import capi
    import ctypes as C
    L = capi.lib()
    L.utb_searcher_set_input.argtypes = [C.c_void_p, C.c_int, C.c_uint32]
    assert L.utb_searcher_set_input(None, capi.INPUT_FASTA_WRAPPED, 0) == 1
    with pytest.raises(ValueError):
        capi.Searcher.set_input(object(), True, 0, True)                 # FASTQ cannot be wrapped


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


def _searcher(ctr, env=None, devices=(0,), threads=4, shallow=False, wrapped=True):
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
    if wrapped:
        s.set_input(False, 0, wrapped=True)
    return s


FRAMING = [{}, {"UTB_HOST_FRAME": "1"}]
WIDTHS = [60, 80, 1, 33, "ragged"]


def _wrap_case(fa, i):
    w = WIDTHS[i % len(WIDTHS)]
    return rewrap(fa, ragged(i) if w == "ragged" else w, crlf=i % 3 == 1, blank_lines=i % 4 == 2)


@pytest.mark.gpu
@pytest.mark.parametrize("env", FRAMING, ids=["device", "host"])
def test_wrapped_search_gives_the_golden_outputs(gpu, tmp_path, env):
    """Every golden read set rewrapped: the reference's output on the linear FASTA, through a file and through
    memory, on two virtual devices (batches dealt over both)."""
    for i, (db, reads, out, rc) in enumerate(CASES):
        fa = open(gold(reads), "rb").read()
        wr = _wrap_case(fa, i)
        p = str(tmp_path / (reads + ".wrapped.fa"))
        open(p, "wb").write(wr)
        want = open(gold(out), "rb").read()
        s = _searcher(gpu[db][0], env, devices=(0, 0))
        try:
            o = str(tmp_path / "o.out")
            r, ex, st = s.search_file(p, o, do_rc=bool(rc))
            assert (r, ex) == (0, 0) and open(o, "rb").read() == want, (reads, out)
            r, ex, text, st2 = s.search_mem(wr, do_rc=bool(rc))
            assert (r, ex) == (0, 0) and text == want, (reads, out)
            assert st["reads"] == st2["reads"] == len(_fasta_lines(fa)) and st["good_finds"] == st2["good_finds"]
        finally:
            s.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("env", FRAMING, ids=["device", "host"])
def test_wrapped_shallow_search_gives_the_golden_outputs(gpu, env):
    for i, (name, m) in enumerate(sorted(json.load(open(os.path.join(GOLD, "meta_shallow.json"))).items())):
        wr = _wrap_case(open(gold(m["reads"]), "rb").read(), i)
        s = _searcher(gpu[m["db"]][0], env, shallow=True, devices=(0, 0))
        try:
            r, ex, text, st = s.search_mem(wr, do_rc=bool(m["rc"]))
            assert (r, ex) == (0, 0) and text == open(gold(name), "rb").read(), name
            assert [f"Good finds: {st['good_finds']}", f"Searched {st['reads']} queries"] == m["stdout_tail"], name
        finally:
            s.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("env", FRAMING, ids=["device", "host"])
def test_wrapped_verdicts_on_the_bad_inputs(gpu, env):
    """bad_noheader.fa is UTB_FW_NOHEADER at record 1; in the other two the trailing headers are reads without
    windows, so the output is the reference's output for the records before them and the search succeeds."""
    from utree_b200 import capi
    s = _searcher(gpu["toyA"][0], env)
    try:
        for name in BAD_CASES:
            data = open(gold(name), "rb").read()
            r, ex, text, st = s.search_mem(data, do_rc=True)
            if name == "bad_noheader.fa":
                assert (r, ex, text) == (3, 2, b"") and b"[record 1]" in capi.lib().utb_last_error()
            else:
                assert (r, ex) == (0, 0) and text == open(gold(name + ".out"), "rb").read(), name
                assert st["reads"] == data.count(b">"), name
    finally:
        s.destroy()


def _big_linear():
    one = open(gold("toyA_reads.fa"), "rb").read() + open(gold("toyB_reads.fa"), "rb").read()
    return one, 200_000_000 // len(one) + 1


@pytest.mark.gpu
@pytest.mark.parametrize("width", [60, "ragged"])
def test_wrapped_search_over_many_chunks(gpu, tmp_path, width):
    """About 200 MB rewrapped: zero copy from a page-locked buffer, an ordinary buffer, a file and a pipe (host
    framer) give the linear FASTA search of the same reads."""
    import torch
    one, k = _big_linear()
    wr = rewrap(one, 60 if width == 60 else ragged(5)) * k
    ctr = gpu["toyB_u32"][0]
    s = _searcher(ctr, devices=(0, 0), threads=8, wrapped=False)
    try:
        r, ex, want, st_fa = s.search_mem(one * k, do_rc=True)
        assert r == 0 and len(want) > 0
        s.set_input(False, wrapped=True)
        pinned = torch.empty(len(wr), dtype=torch.uint8, pin_memory=True)
        pinned.numpy()[:] = np.frombuffer(wr, dtype=np.uint8)
        r, ex, text, st = s.search_mem(None, do_rc=True, ptr=pinned.data_ptr(), n=len(wr))
        assert r == 0 and text == want and st["batches"] >= 3 and st["reads"] == st_fa["reads"]
        assert pinned.numpy().tobytes() == wr                             # the caller's buffer is never written
        del pinned
        r, ex, text, st = s.search_mem(wr, do_rc=True)
        assert r == 0 and text == want and st["batches"] >= 3
        p, o = str(tmp_path / "big.fa"), str(tmp_path / "big.out")
        open(p, "wb").write(wr)
        r, ex, st = s.search_file(p, o, do_rc=True)
        assert r == 0 and open(o, "rb").read() == want
        os.unlink(o)
        fifo = str(tmp_path / "fifo")
        os.mkfifo(fifo)

        def feed():
            with open(fifo, "wb") as f:
                f.write(wr)
        w = threading.Thread(target=feed)
        w.start()
        r, ex, st = s.search_file(fifo, o, do_rc=True)
        w.join()
        assert r == 0 and open(o, "rb").read() == want
    finally:
        s.destroy()


@pytest.mark.gpu
def test_wrapped_genome_sized_records(gpu, tmp_path):
    """Records of 16 000 000 and 16 777 214 bases at widths 60, 80 and 1 (CRLF) against the checker's search of
    lin(input).  The searcher's 33 MiB batches are grown when wrapped input is selected.  One base more than the
    limit gives the output of the records before it and names the record."""
    from utree_b200 import capi
    ctr, orc = gpu["toyA"]
    long_fa = open(gold("long_reads.fa"), "rb").read()
    seqs = b"".join(s for _, s in _fasta_lines(long_fa))
    huge = seqs * (16_777_221 // len(seqs) + 1)
    fa = long_fa + b">huge1 16 Mb\n" + huge[:16_000_000] + b"\n>huge2\n" + huge[7:7 + MAXSEQ] + b"\n" + long_fa
    for w, crlf in ((60, False), (80, False), (1, True)):
        wr = rewrap(fa, w, crlf=crlf)
        p, o = str(tmp_path / "l.fa"), str(tmp_path / "l.out")
        open(p, "wb").write(lin(wr))
        orc.search_file(p, o, do_rc=True)
        want = open(o, "rb").read()
        assert want.startswith(open(gold("long_rc.out"), "rb").read())
        for env in FRAMING:
            s = _searcher(ctr, dict(env, UTB_BATCH_MB="33"))
            try:
                r, ex, text, st = s.search_mem(wr, do_rc=True)
                assert (r, ex) == (0, 0) and text == want, (w, env)
            finally:
                s.destroy()
    n_before = len(_fasta_lines(long_fa)) + 1
    bad = rewrap(long_fa + b">huge1\n" + huge[:16_000_000] + b"\n>over\n" + huge[:MAXSEQ + 1] + b"\n" + long_fa, 60)
    good = lin(bad[:bad.index(b">over\n")])
    p, o = str(tmp_path / "g.fa"), str(tmp_path / "g.out")
    open(p, "wb").write(good)
    orc.search_file(p, o, do_rc=True)
    want = open(o, "rb").read()
    for env in FRAMING:
        s = _searcher(ctr, dict(env, UTB_BATCH_MB="33"))
        try:
            r, ex, text, st = s.search_mem(bad, do_rc=True)
            assert (r, ex, text) == (3, 2, want), env
            assert f"[record {n_before + 1}]".encode() in capi.lib().utb_last_error()
        finally:
            s.destroy()


@pytest.mark.gpu
def test_wrapped_malformed_input_in_a_late_chunk(gpu):
    """Each malformed case after more than one chunk of good records: the same partial output, return code, exit
    code and message whether the device or the host framed the input."""
    from utree_b200 import capi
    ctr = gpu["toyA"][0]
    unit = rewrap(open(gold("toyA_reads.fa"), "rb").read(), 60)
    good = unit * (150_000_000 // len(unit))
    sd, sh = _searcher(ctr, {}), _searcher(ctr, {"UTB_HOST_FRAME": "1"})
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


@pytest.mark.gpu
def test_wrapped_chunk_with_more_records_than_the_batch_holds(gpu):
    """Tiny records: the first device chunk holds more headers than the batch has reads, is flagged, and is framed
    again by the host; the output is the linear search's."""
    ctr = gpu["toyA"][0]
    body = open(gold("toyA_reads.fa"), "rb").read()
    tiny = b"".join(b">t%d\nAC\nG\n" % i for i in range(3_000_000))
    wr = rewrap(body, 60) + tiny + rewrap(body, 61)
    s = _searcher(ctr, wrapped=False)
    try:
        r, ex, want, st_fa = s.search_mem(lin(wr), do_rc=True)
        assert r == 0 and len(want) > 0
        s.set_input(False, wrapped=True)
        r, ex, text, st = s.search_mem(wr, do_rc=True)
        assert (r, ex) == (0, 0) and text == want and st["reads"] == st_fa["reads"]
    finally:
        s.destroy()


@pytest.mark.gpu
def test_linear_inputs_after_wrapped_on_the_same_searcher(gpu):
    """The same searcher then gives the unchanged FASTA and FASTQ outputs; a quality threshold is refused for wrapped
    input, and so is an unknown format."""
    from utree_b200 import capi
    import ctypes as C
    from test_fastq import to_fastq
    s = _searcher(gpu["toyA"][0])
    try:
        fa = open(gold("toyA_reads.fa"), "rb").read()
        want = open(gold("toyA_rc.out"), "rb").read()
        r, ex, text, st = s.search_mem(rewrap(fa, 70), do_rc=True)
        assert (r, ex) == (0, 0) and text == want
        L = capi.lib()
        L.utb_searcher_set_input.argtypes = [C.c_void_p, C.c_int, C.c_uint32]
        assert L.utb_searcher_set_input(s.h, capi.INPUT_FASTA_WRAPPED, 20) == 1
        assert L.utb_searcher_set_input(s.h, 3, 0) == 1
        s.set_input(False)
        r, ex, text, st = s.search_mem(fa, do_rc=True)
        assert (r, ex) == (0, 0) and text == want
        s.set_input(True)
        r, ex, text, st = s.search_mem(to_fastq(fa, 1), do_rc=True)
        assert (r, ex) == (0, 0) and text == want
        s.set_input(False, wrapped=True)
        r, ex, text, st = s.search_mem(rewrap(fa, ragged(9), crlf=True), do_rc=True)
        assert (r, ex) == (0, 0) and text == want
    finally:
        s.destroy()
