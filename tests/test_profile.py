"""Sample profiles (utb_searcher_set_profile / utb_searcher_profile, bin/utree-profile): reads per taxonomy string,
counted on the GPU.  The oracle is the per-read output the project already produces: Counter(column 2 of the lines),
sorted by bytes.  Trees with chosen labels are checked read by read against the CPU vote, which also names the
smallest label id that prints each string."""
import collections
import contextlib
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import conftest  # noqa: F401  (puts the repo root on sys.path)
from oracle import oracle_api
from conftest import BAD_CASES, CASES, ROOT, gold

EXE = os.path.join(ROOT, "bin", "utree-profile")
UTB_CUT_EMPTY, UTB_CUT_FULL = 0xFFFFFFFF, 0xFFFFFFFE


def oracle_profile(text):
    """[(taxonomy, reads)] of output text, in row order (bytes order puts a prefix first).  Column 2 is the fourth field
    from the end: a read name may hold a tab or a '\r', a label neither."""
    lines = text.split(b"\n")[:-1]
    return sorted(collections.Counter(line.split(b"\t")[-4] for line in lines).items())


def rows_only(profile):
    rows, uncl = profile
    return [(t, n) for t, n, _ in rows]


def expected_table(samples, outputs, reads):
    """The TSV utree-profile writes for samples (paths as given) whose output texts and read counts are given."""
    per = [dict(oracle_profile(o)) for o in outputs]
    keys = sorted(set().union(*per))
    lines = [b"#taxonomy\t" + b"\t".join(os.fsencode(p) for p in samples),
             b"#unclassified\t" + b"\t".join(b"%d" % (n - sum(d.values())) for n, d in zip(reads, per))]
    lines += [k + b"".join(b"\t%d" % d.get(k, 0) for d in per) for k in keys]
    return b"\n".join(lines) + b"\n"


@contextlib.contextmanager
def _env(env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _searcher(ctr, env=None, devices=(0,), threads=4):
    from utree_b200 import capi
    with _env(env or {}):
        s = capi.Searcher(ctr, devices=devices, host_threads=threads)
    s.set_profile(True)
    return s


# ---- CPU ----------------------------------------------------------------------------------------------------------
def test_expected_table_helper():
    outs = [b"r1\tk__A;p__B\t3\t1\t*\nr2\t\t2\t2\t0;1\nr3\tk__A\t5\t1\t1;0\nr4\tk__A;p__B\t1\t1\t*\n",
            b"q1\tk__A\t1\t1\t*\nq2\tk__Z\t4\t1\t*\n"]
    want = (b"#taxonomy\ta.fa\tdir/b.fq\n"
            b"#unclassified\t1\t3\n"
            b"\t1\t0\n"
            b"k__A\t1\t1\n"
            b"k__A;p__B\t2\t0\n"
            b"k__Z\t0\t1\n")
    assert expected_table(["a.fa", "dir/b.fq"], outs, [5, 5]) == want


def test_cli_usage_and_input_errors(built, ctrs, tmp_path):
    fa, t = gold("toyA_reads.fa"), str(tmp_path / "t.tsv")
    run = lambda *a: subprocess.run([EXE] + list(a), capture_output=True, text=True)
    for args in ([], [ctrs["toyA"], t], ["-f", "fasta2", ctrs["toyA"], t, fa], ["-q", "20", ctrs["toyA"], t, fa],
                 ["-t", "0", ctrs["toyA"], t, fa], ["-x", ctrs["toyA"], t, fa], ["-t"]):
        p = run(*args)
        assert p.returncode == 1 and "usage: utree-profile" in p.stderr, args
    p = run(str(tmp_path / "nope.ctr"), t, fa)
    assert p.returncode == 1 and "nope.ctr" in p.stderr
    p = run("-r", ctrs["toyA"], t, fa, str(tmp_path / "missing.fa"))
    assert p.returncode == 1 and "missing.fa" in p.stderr
    full = open(ctrs["toyA"], "rb").read()
    cut = str(tmp_path / "cut.ctr")
    open(cut, "wb").write(full[:32 + 1_000_003])
    assert run(cut, t, fa).returncode == 3
    assert not os.path.exists(t)


def test_cli_without_a_device_exits_4(built, ctrs, tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    t = str(tmp_path / "t.tsv")
    p = subprocess.run([EXE, ctrs["toyA"], t, gold("toyA_reads.fa")], capture_output=True, text=True)
    assert p.returncode == 4 and not os.path.exists(t)


# ---- a tree whose labels share prefixes ---------------------------------------------------------------------------
PREFIX_LABELS = [b"k__A;p__B;c__Cat;o__D", b"k__A;p__B", b"k__A;p__B;c__Cab;o__E", b"k__A;p__B;c__Cat", b"k__A;p__G",
                 b"k__Z;p__Y", b"k__A;p__B;c__Cat;o__F", b"k__Q", b"k__A;p__Bx", b"k__A;p__B;c__F;o__G;f__H",
                 b"k__A;p__B;c__F;o__G", b"k__Z;p__Yz;c__W", b"k__A", b"k__A;p__B;c__Cab", b"k__Q;p__R;c__S"]


@pytest.fixture(scope="module")
def prefix_tree(built, tmp_path_factory):
    """PREFIX_LABELS, and 4000 reads whose forward windows carry 1 to 4 labels neighbouring in byte order.  Per read the
    CPU vote gives its kind, label and cut, so the expected rows and the smallest label of each are known."""
    from test_vote_limits import build_search_tree, search_reads
    d = tmp_path_factory.mktemp("prefix")
    rng = np.random.default_rng(5)
    labels = PREFIX_LABELS
    by_rank = sorted(range(len(labels)), key=lambda i: labels[i])
    spec = [(b"p%d" % i, int(rng.integers(20, 90)), int(rng.integers(1, 5))) for i in range(4000)]
    reads = search_reads(rng, by_rank, len(labels), spec)
    path = str(d / "prefix.ctr")
    build_search_tree(path, labels, reads, 2, rng)
    fa = b"".join(b">" + n + b"\n" + np.frombuffer(b"ACGT", dtype=np.uint8)[c].tobytes() + b"\n" for n, c, _ in reads)
    fa_path = str(d / "prefix.fa")
    open(fa_path, "wb").write(fa)
    orc = oracle_api.OracleDb(path)
    printed = collections.defaultdict(lambda: [0, set()])
    cuts = collections.Counter()
    for _, codes, _ in reads:
        hits, _ = orc.slide(np.frombuffer(b"ACGT", dtype=np.uint8)[codes].tobytes(), do_rc=False)
        v = orc.vote(hits)
        if v.kind == 0:
            continue
        lab = labels[v.label]
        t = lab
        if v.kind == 2 and v.cut == UTB_CUT_EMPTY:
            t, what = b"", "empty"
        elif v.kind == 2 and v.cut != UTB_CUT_FULL and v.cut < len(lab):
            t = lab[:v.cut]
            what = "token" if lab[v.cut:v.cut + 1] == b";" else "mid"
        else:
            what = "full_prefix" if any(o != lab and o.startswith(lab) for o in labels) else "full"
        cuts[what] += 1
        printed[t][0] += 1
        printed[t][1].add(v.label)
    out = str(d / "prefix.out")
    orc.search_file(fa_path, out, do_rc=False)
    yield {"path": path, "fa": fa_path, "text": open(out, "rb").read(), "cuts": cuts,
           "rows": sorted((t, n, min(ls)) for t, (n, ls) in printed.items()),
           "merged": [t for t, (n, ls) in printed.items() if len(ls) > 1], "reads": len(reads)}
    orc.free()


def test_prefix_tree_has_the_cases_that_merge(prefix_tree):
    """The reads end on a token cut, the empty cut and a full label that prefixes another; several label ids print
    one string; and the CPU vote's strings are the checker's column 2."""
    c = prefix_tree["cuts"]
    assert c["empty"] and c["full_prefix"] and c["token"], c
    assert len(prefix_tree["merged"]) >= 3, prefix_tree["merged"]
    assert [(t, n) for t, n, _ in prefix_tree["rows"]] == oracle_profile(prefix_tree["text"])


# ---- GPU ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu(built, ctrs):
    from utree_b200 import capi
    assert capi.device_count() >= 1
    state = {name: capi.Ctr(path) for name, path in ctrs.items()}
    yield state
    for ctr in state.values():
        ctr.close()


def _pinned(data):
    import torch
    p = torch.empty(len(data), dtype=torch.uint8, pin_memory=True)
    p.numpy()[:] = np.frombuffer(data, dtype=np.uint8)
    return p


@pytest.mark.gpu
def test_profile_of_every_golden_case(gpu, tmp_path):
    """With text, the profile is the oracle on the golden output; without text (no file, NULL outputs from a
    page-locked and an ordinary buffer) it is the same, with no output bytes and no file."""
    for db, reads, out, rc in CASES:
        want_text = open(gold(out), "rb").read()
        want = oracle_profile(want_text)
        s = _searcher(gpu[db])
        try:
            o = str(tmp_path / "o.out")
            r, ex, st = s.search_file(gold(reads), o, do_rc=bool(rc))
            assert (r, ex) == (0, 0) and open(o, "rb").read() == want_text, out
            prof = s.profile()
            assert rows_only(prof) == want and prof[1] == st["reads"] - st["good_finds"], out
            assert sum(n for _, n, _ in prof[0]) == st["good_finds"]
            for t, _, lab in prof[0]:
                assert gpu[db].label(lab)[:len(t)] == t, (out, t, lab)
            os.unlink(o)
            r, ex, st2 = s.search_file(gold(reads), None, do_rc=bool(rc))
            assert (r, ex) == (0, 0) and st2["out_bytes"] == 0 and not os.path.exists(o)
            assert s.profile() == prof and st2["good_finds"] == st["good_finds"], out
            data = open(gold(reads), "rb").read()
            r, ex, text, st3 = s.search_mem(data, do_rc=bool(rc), text=False)
            assert (r, ex, text, st3["out_bytes"]) == (0, 0, None, 0) and s.profile() == prof, out
            if data:
                p = _pinned(data)
                r, ex, text, st4 = s.search_mem(None, do_rc=bool(rc), ptr=p.data_ptr(), n=len(data), text=False)
                assert (r, ex, st4["out_bytes"]) == (0, 0, 0) and s.profile() == prof, out
                r, ex, text, st5 = s.search_mem(None, do_rc=bool(rc), ptr=p.data_ptr(), n=len(data))
                assert (r, ex, text) == (0, 0, want_text) and s.profile() == prof, out
                del p
        finally:
            s.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{}, {"UTB_HOST_FRAME": "1"}], ids=["device", "host"])
def test_profile_rows_merge_equal_strings_under_the_smallest_label(gpu, prefix_tree, env):
    from utree_b200 import capi
    ctr = capi.Ctr(prefix_tree["path"])
    s = _searcher(ctr, env, devices=(0, 0))
    try:
        r, ex, text, st = s.search_mem(open(prefix_tree["fa"], "rb").read(), do_rc=False)
        assert (r, ex) == (0, 0) and text == prefix_tree["text"]
        rows, uncl = s.profile()
        assert [(t, n, lab) for t, n, lab in rows] == prefix_tree["rows"]
        assert uncl == prefix_tree["reads"] - st["good_finds"]
        assert rows[0][0] == b""                                           # the empty string sorts first
    finally:
        s.destroy(); ctr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["fastq0", "fastq20", "wrapped"])
def test_profile_of_fastq_and_wrapped_input(gpu, fmt):
    from test_fastq import to_fastq
    from test_wrapped_fasta import rewrap, ragged
    for db, reads, out, rc in CASES[:3] + CASES[5:]:
        fa = open(gold(reads), "rb").read()
        s = _searcher(gpu[db])
        try:
            if fmt == "wrapped":
                s.set_input(False, 0, wrapped=True)
                data = rewrap(fa, ragged(3))
            else:
                s.set_input(True, 0 if fmt == "fastq0" else 20)
                data = to_fastq(fa, 4)
            r, ex, text, st = s.search_mem(data, do_rc=bool(rc))
            assert (r, ex) == (0, 0), reads
            prof = s.profile()
            assert rows_only(prof) == oracle_profile(text) and prof[1] == st["reads"] - st["good_finds"], reads
            r, ex, none, st2 = s.search_mem(data, do_rc=bool(rc), text=False)
            assert r == 0 and s.profile() == prof
        finally:
            s.destroy()


def _big_input():
    one = open(gold("toyA_reads.fa"), "rb").read() + open(gold("toyB_reads.fa"), "rb").read()
    return one * (200_000_000 // len(one) + 1)


@pytest.mark.gpu
def test_profile_over_many_batches_framings_and_devices(gpu):
    """About 200 MB: ramp and full batches, device and host framing, 1, 2 and 4 virtual devices and (when present)
    two GPUs give one profile, the oracle on the text."""
    import torch
    data = _big_input()
    ctr = gpu["toyB_u32"]
    s = _searcher(ctr, devices=(0,), threads=8)
    try:
        r, ex, text, st = s.search_mem(data, do_rc=True)
        assert r == 0 and st["batches"] >= 4
        want = s.profile()
        assert rows_only(want) == oracle_profile(text) and want[1] == st["reads"] - st["good_finds"]
        del text
    finally:
        s.destroy()
    devsets = [(0,), (0, 0), (0, 0, 0, 0)] + ([(0, 1)] if torch.cuda.device_count() >= 2 else [])
    p = _pinned(data)
    for env in ({}, {"UTB_HOST_FRAME": "1"}):
        for devs in devsets:
            s = _searcher(ctr, env, devices=devs, threads=8)
            try:
                r, ex, none, st = s.search_mem(None, do_rc=True, ptr=p.data_ptr(), n=len(data), text=False)
                assert r == 0 and st["out_bytes"] == 0 and st["batches"] >= 4, (env, devs)
                assert s.profile() == want, (env, devs)
            finally:
                s.destroy()
    del p


@pytest.mark.gpu
def test_profile_after_malformed_input(gpu, tmp_path):
    """The reads whose lines were written before the bad record, and nothing of the batches dropped on the way: each
    bad golden case, and a bad record in a late device-framed chunk (device and host framing)."""
    s = _searcher(gpu["toyA"])
    try:
        for name in BAD_CASES:
            o = str(tmp_path / "o.out")
            r, ex, st = s.search_file(gold(name), o, do_rc=True)
            assert (r, ex) == (3, 2), name
            text = open(o, "rb").read()
            prof = s.profile()
            assert rows_only(prof) == oracle_profile(text) and prof[1] == st["reads"] - st["good_finds"], name
            r, ex, st = s.search_file(gold(name), None, do_rc=True)
            assert (r, ex) == (3, 2) and s.profile() == prof, name
    finally:
        s.destroy()
    unit = open(gold("toyA_reads.fa"), "rb").read()
    good = unit * (150_000_000 // len(unit))
    bad = good + b"r\nACGT\n" + unit
    profs = []
    for env in ({}, {"UTB_HOST_FRAME": "1"}):
        s = _searcher(gpu["toyA"], env)
        try:
            r, ex, text, st = s.search_mem(bad, do_rc=True)
            assert (r, ex) == (3, 2) and st["batches"] >= 2, env
            prof = s.profile()
            assert rows_only(prof) == oracle_profile(text), env
            r, ex, none, st2 = s.search_mem(bad, do_rc=True, text=False)
            assert (r, ex) == (3, 2) and s.profile() == prof, env
            profs.append(prof)
        finally:
            s.destroy()
    assert profs[0] == profs[1]


def _tree_one_word_per_label(path, n_labels, rng):
    """A uint32 tree of n_labels labels; label i owns one word, the forward window of read i (32 bases).  Word 0
    (label 0 as well) is the lowest bin's only record, which the compressor folds away."""
    from test_vote_limits import write_tree
    words = np.unique(rng.integers(1, 2 ** 63, int(n_labels * 1.1), dtype=np.int64).astype(np.uint64) * np.uint64(2) + np.uint64(1))
    words = rng.permutation(words)[:n_labels]
    assert words.size == n_labels
    labels = [b"k__T;s__%06d" % i for i in range(n_labels)]
    write_tree(path, labels, np.concatenate([[np.uint64(0)], words]), np.arange(-1, n_labels).clip(0).astype(np.uint64), 4)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    codes = ((words[:, None] >> (np.uint64(2) * np.arange(31, -1, -1, dtype=np.uint64))) & np.uint64(3)).astype(np.uint8)
    return labels, acgt[codes]


@pytest.mark.gpu
def test_profile_hot_key_and_many_keys(gpu, tmp_path):
    """Every read of a full batch printing one string (warp aggregation on one slot), and 200 000 reads each hitting
    its own label of a uint32 tree (more distinct keys per batch than a CTA's shared table holds)."""
    from utree_b200 import capi
    rng = np.random.default_rng(3)
    path = str(tmp_path / "keys.ctr")
    n = 200_000
    labels, seqs = _tree_one_word_per_label(path, n, rng)
    fa = b"".join(b">m%d\n%s\n" % (i, seqs[i].tobytes()) for i in range(n))
    ctr = capi.Ctr(path)
    try:
        s = _searcher(ctr)
        try:
            r, ex, text, st = s.search_mem(fa, do_rc=False)
            assert r == 0 and st["batches"] == 1 and st["good_finds"] == n
            prof = s.profile()
            assert rows_only(prof) == oracle_profile(text) and len(prof[0]) == n and prof[1] == 0
            hot = b"".join(b">h%07d\n%s\n" % (i, seqs[7].tobytes()) for i in range(2_600_000))
            r, ex, text, st = s.search_mem(hot, do_rc=False)
            assert r == 0 and st["good_finds"] == 2_600_000
            rows, uncl = s.profile()
            assert rows_only((rows, uncl)) == oracle_profile(text) == [(labels[7], 2_600_000)] and rows[0][2] == 7
            del text
        finally:
            s.destroy()
    finally:
        ctr.close()


@pytest.mark.gpu
def test_profile_modes(gpu):
    """The profile and the non-GG search exclude each other; with the profile off NULL outputs stay an argument
    error; a profile search does not change the next plain search; no profile after a failed search."""
    from utree_b200 import capi
    L = capi.lib()
    L.utb_search_file.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_int, C.c_void_p, C.c_void_p]
    ctr = gpu["toyA"]
    s = capi.Searcher(ctr, devices=(0,), host_threads=2)
    try:
        s.set_shallow(True)
        with pytest.raises(capi.UtbError) as e:
            s.set_profile(True)
        assert e.value.code == 1
        s.set_shallow(False)
        r, ex, text, st = s.search_mem(b">a\nACGT\n", text=False)
        assert r == 1
        assert L.utb_search_file(s.h, os.fsencode(gold("toyA_reads.fa")), None, 1, None, None) == 1
        s.set_profile(True)
        with pytest.raises(capi.UtbError) as e:
            s.set_shallow(True)
        assert e.value.code == 1
        with pytest.raises(capi.UtbError):
            s.profile()                                                    # no search yet
        data = open(gold("toyA_reads.fa"), "rb").read()
        want = open(gold("toyA_rc.out"), "rb").read()
        r, ex, none, st = s.search_mem(data, text=False)
        assert r == 0 and rows_only(s.profile()) == oracle_profile(want)
        r, ex, st = s.search_file(gold("nope.fa"), None)
        assert r == 2
        with pytest.raises(capi.UtbError):
            s.profile()
        s.set_profile(False)
        r, ex, text, st = s.search_mem(data)
        assert r == 0 and text == want
        with pytest.raises(capi.UtbError):
            s.profile()
    finally:
        s.destroy()


@pytest.mark.gpu
def test_cli_profiles_samples(gpu, ctrs, tmp_path):
    """A FASTA, a FASTQ (-q 20) and a wrapped FASTA sample each give the table of their searched text; several
    samples in one run share the rows; a malformed second sample exits 2 and writes no table."""
    from test_fastq import to_fastq
    from test_wrapped_fasta import rewrap
    fa = open(gold("toyA_reads.fa"), "rb").read()
    edge = open(gold("edge_reads.fa"), "rb").read()
    fq, wr = to_fastq(edge, 2), rewrap(fa + edge, 60)
    paths = [str(tmp_path / n) for n in ("a.fa", "b.fq", "c.fa")]
    fmts = [["-f", "fasta"], ["-f", "fastq", "-q", "20"], ["-f", "wrapped"]]
    outs, reads = [], []
    s = _searcher(gpu["toyA"])
    try:
        for p, d, setup in zip(paths, (fa, fq, wr), (lambda: s.set_input(False), lambda: s.set_input(True, 20),
                                                     lambda: s.set_input(False, 0, wrapped=True))):
            open(p, "wb").write(d)
            setup()
            r, ex, text, st = s.search_mem(d, do_rc=True)
            assert r == 0
            outs.append(text); reads.append(st["reads"])
    finally:
        s.destroy()
    t = str(tmp_path / "t.tsv")
    run = lambda *a: subprocess.run([EXE, "-r", "-t", "4"] + list(a), capture_output=True, text=True)
    for i, p in enumerate(paths):
        q = run(*fmts[i], ctrs["toyA"], t, p)
        assert q.returncode == 0, q.stderr
        assert open(t, "rb").read() == expected_table([p], [outs[i]], [reads[i]]), p
        assert q.stdout.splitlines() == [f"Searched {reads[i]} queries", f"Good finds: {outs[i].count(b'\n')}"]
    many = [paths[2], paths[0], paths[2]]                                 # linear FASTA is wrapped FASTA too
    q = run("-f", "wrapped", ctrs["toyA"], t, *many)
    assert q.returncode == 0 and open(t, "rb").read() == expected_table(many, [outs[2], outs[0], outs[2]],
                                                                        [reads[2], reads[0], reads[2]])
    os.unlink(t)
    bad = str(tmp_path / "bad.fa")
    open(bad, "wb").write(fa + b"r\nACGT\n")
    q = run(ctrs["toyA"], t, paths[0], bad, paths[0])
    assert q.returncode == 2 and "bad.fa" in q.stderr and not os.path.exists(t)
