"""File formats (python compress == reference compress), the host CTR loader
against the oracle's, and the C-ABI surface.  CPU only: no compute calls."""
import ctypes
import hashlib
import os
import re
import subprocess

import numpy as np
import pytest

import conftest  # noqa: F401  (puts the repo root on sys.path)
from oracle import oracle_api
from conftest import GOLD, REFDIR, ROOT, gold


def _sha(p):
    return hashlib.sha256(open(p, "rb").read()).hexdigest()


@pytest.mark.parametrize("name", ["toyA", "toyB_u32", "quirk", "dense"])
def test_python_compress_equals_reference_compress(ctrs, meta, name):
    assert _sha(ctrs[name]) == meta[name]["ctr_sha256"]


def test_reference_compress_live(tmp_path, ctrs, meta):
    """The reference's utree-compress of quirk.ubt: its sha256 as recorded in meta.json, and live when oracle/_ref
    is built."""
    want = meta["quirk"]["ctr_sha256"]
    exe = os.path.join(REFDIR, "utree-compress")
    if os.path.exists(exe):
        out = str(tmp_path / "q.ctr")
        subprocess.run([exe, gold("quirk.ubt"), out], check=True, stdout=subprocess.DEVNULL)
        assert _sha(out) == want
    assert _sha(ctrs["quirk"]) == want


def test_library_exports_every_declared_symbol(built):
    from utree_b200 import capi
    hdr = open(os.path.join(ROOT, "include", "utree_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(utb_[a-z0-9_]+)\s*\(", hdr)))
    assert declared == sorted(capi.EXPORTS)
    L = ctypes.CDLL(capi.LIB_PATH)
    for sym in declared:
        assert hasattr(L, sym), sym


def test_product_does_not_reference_oracle():
    """The oracle is test infrastructure: nothing under utree_b200/csrc or include/ may name it."""
    for d in ("utree_b200/csrc", "include", "utree_b200"):
        for f in os.listdir(os.path.join(ROOT, d)):
            if f.endswith((".c", ".cu", ".h", ".py")):
                txt = open(os.path.join(ROOT, d, f)).read()
                assert "oracle" not in txt.lower(), f
    so = open(os.path.join(ROOT, "utree_b200", "csrc", "libutree_b200.so"), "rb").read()
    assert b"orc_" not in so and b"liboracle" not in so


@pytest.mark.parametrize("name", ["toyA", "toyB_u32", "quirk", "dense"])
def test_ctr_loader_matches_oracle_loader(built, ctrs, name):
    from utree_b200 import capi
    ctr, orc = capi.Ctr(ctrs[name]), oracle_api.OracleDb(ctrs[name])
    O = oracle_api.oracle()
    try:
        assert ctr.num_nodes == O.orc_db_num_nodes(orc.h)
        assert ctr.ix_bytes == O.orc_db_ix_bytes(orc.h) and ctr.binix_bytes == O.orc_db_binix_bytes(orc.h)
        assert ctr.max_ix == orc.max_ix and ctr.last_bin == ctr.num_nodes
        labels = [ctr.label(i) for i in range(ctr.max_ix)]
        assert labels == [orc.label(i) for i in range(orc.max_ix)]
        order = sorted(range(ctr.max_ix), key=lambda i: labels[i])       # bytes compare == strcmp
        assert [ctr.rank(i) for i in order] == list(range(ctr.max_ix))
    finally:
        ctr.close(); orc.free()


def test_ctr_loader_dedups_repeated_labels(built, tmp_path):
    """A label string seen twice keeps its first id (addSampleUdX, itree.c:219-220)."""
    from utree_b200 import capi
    from tools import synth
    words = np.array([5 << 40 | 7, 5 << 40 | 9, 6 << 40 | 1], dtype=np.uint64)
    tail = b"k__A;p__B\t1\nk__A;p__C\t1\nk__A;p__B\t1\nk__A;p__D\t0\n"
    p = str(tmp_path / "d.ctr")
    synth.ctr_write(p, words, np.array([0, 1, 2]), tail, 2)
    ctr, orc = capi.Ctr(p), oracle_api.OracleDb(p)
    try:
        assert ctr.max_ix == orc.max_ix == 3
        assert [ctr.label(i) for i in range(3)] == [b"k__A;p__B", b"k__A;p__C", b"k__A;p__D"]
    finally:
        ctr.close(); orc.free()


def test_ctr_loader_rejects_bad_files(built, tmp_path):
    from utree_b200 import capi
    with pytest.raises(capi.UtbError, match="Invalid DB file"):
        capi.Ctr(str(tmp_path / "missing.ctr"))
    p = str(tmp_path / "zero.ctr")
    open(p, "wb").write(np.array([8, 0, 2, 0], dtype="<u8").tobytes() + b"\0" * 64)
    with pytest.raises(capi.UtbError, match="Tree malformatted"):
        capi.Ctr(p)
    open(p, "wb").write(np.array([4, 0, 2, 5], dtype="<u8").tobytes() + b"\0" * 64)
    with pytest.raises(capi.UtbError, match="PACKSIZE"):
        capi.Ctr(p)
    open(p, "wb").write(np.array([8, 0, 2, 5], dtype="<u8").tobytes() + b"\0" * 64)
    with pytest.raises(capi.UtbError, match="Error in reading tree"):
        capi.Ctr(p)


def test_read_slots_geometry(built):
    from utree_b200 import capi
    L = capi.lib()
    assert [L.utb_read_slots(n) for n in (0, 1, 31, 32, 150, 159, 160)] == [1, 1, 1, 2, 5, 5, 6]


def test_no_gpu_is_a_loud_error_not_a_fallback(built):
    """Without a device every device entry point fails with UTB_ERR_CUDA."""
    import torch
    from utree_b200 import capi
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(capi.UtbError) as e:
        capi.device_count()
    assert e.value.code == 5 and "no CPU fallback" in str(e.value)


def test_cli_usage_and_db_errors(built, tmp_path):
    exe = os.path.join(ROOT, "bin", "utree-search_gg")
    p = subprocess.run([exe], capture_output=True, text=True)
    assert p.returncode == 1 and "usage: xtree-searchGG" in p.stdout          # itree.c:1358-1360
    p = subprocess.run([exe, str(tmp_path / "nope.ctr"), "a.fa", "o.txt", "1", "RC"], capture_output=True, text=True)
    assert p.returncode == 0                                                    # itree.c:735: exit(0)
    out = p.stdout.splitlines()
    assert out[:5] == ["This is UTree [v2.0RF SigNature Edition]", "Reverse complement consideration is enabled.",
                       "Searching at speed 0.", "Using up to 1 threads.", "Invalid DB file"]


@pytest.mark.parametrize("keep", ["records", "index"])
def test_cli_truncated_tree_prints_the_banner_and_exits_3(built, ctrs, tmp_path, keep):
    """A CTR cut inside its records / inside its prefix index: XT_read32 prints what it has read so far, then
    "Error in reading tree." and exits 3 (itree.c:754-768).  Live against oracle/_ref when it is built."""
    full = open(ctrs["toyA"], "rb").read()
    n = int.from_bytes(full[24:32], "little")
    cut = 32 + (2 ** 24 + 1) * 4 + (n // 2) * 7 + 3 if keep == "records" else 32 + 1_000_003
    bad = str(tmp_path / "cut.ctr")
    open(bad, "wb").write(full[:cut])
    args = [bad, os.path.join(GOLD, "toyA_reads.fa"), str(tmp_path / "o.txt"), "1", "RC"]
    p = subprocess.run([os.path.join(ROOT, "bin", "utree-search_gg")] + args, capture_output=True, text=True)
    got_index = (cut - 32) // 4 if keep == "index" else 2 ** 24 + 1
    assert p.returncode == 3
    assert p.stdout.splitlines()[4:] == ["Using 32-bit counters", f"{got_index} elements read.",
                                         f"Nodes in input tree: {n} (PACKSIZE=32, CNTTYPE=NA, IXTYPE=uint16_t, SZ=7)",
                                         "Error in reading tree."]
    ref = os.path.join(REFDIR, "utree-search_gg")
    if os.path.exists(ref):
        q = subprocess.run([ref] + args, capture_output=True, text=True)
        assert (q.returncode, q.stdout) == (p.returncode, p.stdout)


# ---- host logic: framer and formatter (no GPU) --------------------------------
def _py_frame(data):
    """Reference reader restated in Python (itree.c:866-890); returns (records, error?)."""
    if not data:
        return [], False
    lines = data.split(b"\n")
    if data.endswith(b"\n"):
        lines = lines[:-1]
        ends = [b"\n"] * len(lines)
    else:
        ends = [b"\n"] * (len(lines) - 1) + [b""]
    recs = []
    for i in range(0, len(lines), 2):
        if i + 1 >= len(lines):
            return recs, True                       # can't read sequence
        h, s = lines[i] + ends[i], lines[i + 1] + ends[i + 1]
        if h[:1] != b">" or s[:1] == b">":
            return recs, True
        s = s.split(b"\0")[0]
        if not s:
            return recs, True
        if s.endswith(b"\n"):
            s = s[:-1]
        if s.endswith(b"\r"):
            s = s[:-1]
        name = h[1:]
        for stop in (b"\0", b" ", b"\n"):
            name = name.split(stop)[0]
        recs.append((name, s))
    return recs, False


@pytest.mark.parametrize("fasta", ["toyA_reads.fa", "toyB_reads.fa", "edge_reads.fa", "long_reads.fa", "quirk_reads.fa",
                                   "bad_noheader.fa", "bad_seq_is_header.fa", "bad_truncated.fa"])
@pytest.mark.parametrize("threads", [1, 2, 5, 16])
def test_framer_matches_reference_reader(built, fasta, threads):
    from utree_b200 import capi
    data = open(gold(fasta), "rb").read()
    want, bad = _py_frame(data)
    rc, ex, used, recs, _ = capi.frame_records(data, eof=True, threads=threads)
    assert recs == want
    assert (rc, ex) == ((3, 2) if bad else (0, 0))
    if not bad:
        assert used == len(data)


def test_framer_odd_inputs(built):
    from utree_b200 import capi
    cases = [b"", b">a\nACGT", b">a\nACGT\n", b">a\r\nACGT\r\n", b">a b c\nAC\0GT\n", b">\nA\n", b">x\n\n>y\nAC\n",
             b">a\nACGT\n\n", b"\n", b">a\n", b">a", b">n\0ame z\nACGT\n>b\n\0\n", b">a\nAC\n>b\nGT\n>c\n>d\n"]
    for data in cases:
        want, bad = _py_frame(data)
        for t in (1, 3, 8):
            rc, ex, used, recs, _ = capi.frame_records(data, eof=True, threads=t)
            assert recs == want, (data, t)
            assert (rc != 0) == bad, (data, t)


def test_framer_partial_buffer_carries_the_tail(built):
    """Without EOF an incomplete last record is left for the next buffer."""
    from utree_b200 import capi
    data = b">a\nACGT\n>b\nGGTT\n>c\nAC"
    rc, ex, used, recs, _ = capi.frame_records(data, eof=False, threads=4)
    assert rc == 0 and recs == [(b"a", b"ACGT"), (b"b", b"GGTT")] and data[used:] == b">c\nAC"
    rc, ex, used, recs, _ = capi.frame_records(data + b"\n", eof=False, threads=4)
    assert [r[0] for r in recs] == [b"a", b"b", b"c"] and used == len(data) + 1
    rc, ex, used, recs, _ = capi.frame_records(data, eof=False, threads=2, max_reads=1)
    assert recs == [(b"a", b"ACGT")] and data[used:].startswith(b">b\n")


def test_formatter_matches_oracle_lines(built, ctrs):
    """utb_format_results on oracle votes == the golden output of the reference."""
    from utree_b200 import capi
    ctr, orc = capi.Ctr(ctrs["toyA"]), oracle_api.OracleDb(ctrs["toyA"])
    try:
        data = open(gold("toyA_reads.fa"), "rb").read()
        rc, ex, used, recs, (name_off, name_len) = capi.frame_records(data, threads=3)
        res = np.zeros(len(recs), dtype=capi.RESULT_DTYPE)
        for i, (_, seq) in enumerate(recs):
            hits, _ = orc.slide(seq, do_rc=True)
            v = orc.vote(hits)
            res[i] = (v.kind, v.label, v.cut, v.found, v.uix, v.sl, v.ol, 0)
        text = capi.format_results(ctr, data, name_off, name_len, res)
        assert text == open(gold("toyA_rc.out"), "rb").read()
    finally:
        ctr.close(); orc.free()


# ---- utree-compress equivalent (SURVEY 8f-2) ----------------------------------------
@pytest.mark.parametrize("name", ["toyA", "toyB_u32", "quirk", "dense"])
def test_compress_equals_reference_compressor(built, tmp_path, meta, name):
    """utb_compress_ubt == utree-compress, byte for byte (sha256 recorded from the reference binary),
    including the first-bin quirk (`quirk`, `dense`)."""
    from utree_b200 import capi
    out = str(tmp_path / "c.ctr")
    n, nl = capi.compress_ubt(gold(name + ".ubt"), out)
    assert _sha(out) == meta[name]["ctr_sha256"]
    ctr = capi.Ctr(out)
    try:
        assert (ctr.num_nodes, ctr.max_ix) == (n, nl)
    finally:
        ctr.close()


def test_compress_cli_contract(built, tmp_path, meta):
    exe = os.path.join(ROOT, "bin", "utree-compress")
    p = subprocess.run([exe], capture_output=True, text=True)
    assert p.returncode == 1 and "usage: xtree-compress" in p.stdout                      # itree.c:1353
    out = str(tmp_path / "q.ctr")
    p = subprocess.run([exe, gold("quirk.ubt"), out], capture_output=True, text=True)
    assert p.returncode == 0 and _sha(out) == meta["quirk"]["ctr_sha256"]
    lines = p.stdout.splitlines()
    assert lines[0].startswith("Nodes in input tree: 50 (PACKSIZE=32, CNTTYPE=NA, IXTYPE=uint16_t, el=10)")
    assert lines[1] == "Using 32-bit counters" and lines[-1].startswith("Total nodes in tree: 50 [")
    ref = os.path.join(REFDIR, "utree-compress")
    if os.path.exists(ref):                                                                # live: same stdout, same bytes
        out2 = str(tmp_path / "r.ctr")
        q = subprocess.run([ref, gold("quirk.ubt"), out2], capture_output=True, text=True)
        assert q.stdout == p.stdout and _sha(out2) == _sha(out)
    p = subprocess.run([exe, str(tmp_path / "missing.ubt"), out], capture_output=True, text=True)
    assert p.returncode == 0 and "Invalid input filename" in p.stdout                      # itree.c:1236: exit(0)
