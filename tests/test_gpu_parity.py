"""Parity of the CUDA path (through the C ABI) against the oracle and the
golden outputs of the reference binary.  Integer/byte work: bit-exact."""
import os
import subprocess

import numpy as np
import pytest

import conftest  # noqa: F401  (puts the repo root on sys.path)
from oracle import oracle_api
from conftest import BAD_CASES, CASES, ROOT, check_reference_run, gold, read_fasta

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu(built, ctrs):
    from utree_b200 import capi
    assert capi.device_count() >= 1
    state = {}
    for name, path in ctrs.items():
        ctr = capi.Ctr(path)
        state[name] = (ctr, capi.Db(ctr, 0), oracle_api.OracleDb(path))
    yield state
    for ctr, db, orc in state.values():
        db.free(); ctr.close(); orc.free()


def _rand_words_for(orc_path_words, rng, n_extra):
    return orc_path_words


@pytest.mark.parametrize("name", ["toyA", "toyB_u32", "quirk", "dense"])
def test_lookup_words_match_oracle(gpu, name):
    """XT_getIX32 on members, near-members, same-prefix strangers and random words."""
    from tools import synth
    ctr, db, orc = gpu[name]
    words, ixs, _, _ = synth.ubt_read(gold(name + ".ubt"))
    rng = np.random.default_rng(5)
    w = [words, words + np.uint64(1), words - np.uint64(1),
         (words & ~np.uint64(0xFFFFFFFFFF)) | rng.integers(0, 1 << 40, words.size, dtype=np.uint64),
         rng.integers(0, np.iinfo(np.uint64).max, 20000, dtype=np.uint64),
         np.array([0, np.iinfo(np.uint64).max, 0xFFFFFFFFFF, 1 << 40], dtype=np.uint64)]
    w = np.concatenate(w)
    if w.size > 120000:
        w = w[rng.permutation(w.size)[:120000]]
    got = db.lookup_words(w)
    want = orc.lookup_many(w)
    assert np.array_equal(got, want)
    assert (got != 0xFFFFFFFF).sum() > 0


def test_pack_matches_oracle_words(gpu):
    """2-bit pack + RC: every looked-up word of the oracle's slide appears, in order."""
    ctr, db, orc = gpu["toyA"]
    recs = read_fasta(gold("edge_reads.fa")) + read_fasta(gold("toyA_reads.fa"))[:60] + read_fasta(gold("toyB_reads.fa"))[:20]
    for name, seq in recs:
        if not seq:
            continue
        fwd, rc, valid = db.pack_sequence(seq)
        _, owords = orc.slide(seq, do_rc=False, want_words=True)
        assert np.array_equal(fwd[valid == 1], owords), name
        _, owords_rc = orc.slide(seq, do_rc=True, want_words=True)
        # oracle order: forward windows, then windows of the RC text = rc words in reverse order
        assert np.array_equal(np.concatenate([fwd[valid == 1], rc[valid == 1][::-1]]), owords_rc), name


@pytest.mark.parametrize("env", [{}, {"UTB_VOTE_SPLIT_SLOTS": "256"}, {"UTB_VOTE_SORT_MAX": "3"},
                                 {"UTB_VOTE_SPLIT_SLOTS": "256", "UTB_VOTE_SORT_MAX": "3"}])
@pytest.mark.parametrize("sparse", [False, True])
@pytest.mark.parametrize("dbname", ["toyA", "toyB_u32"])
def test_vote_matches_oracle(gpu, dbname, sparse, env):
    """Vote on real hit lists, on permuted hit lists (SURVEY 0 #6) and on synthetic multisets; dense
    (warp/block kernels) and through the pipeline's sparse hit map (thread kernel first).  With a tiny
    split threshold every read the warp kernel defers is split across the grid and merged; with a tiny
    sort limit the touched-label list gives way to the sweep over all labels in rank order."""
    ctr, db, orc = gpu[dbname]
    os.environ.update(env)
    rng = np.random.default_rng(9)
    lists = []
    reads = read_fasta(gold("toyA_reads.fa"))[:300] + read_fasta(gold("long_reads.fa")) if dbname == "toyA" \
        else read_fasta(gold("toyB_reads.fa"))[:600]
    for name, seq in reads:
        h, _ = orc.slide(seq, do_rc=True)
        lists.append(h)
        if h.size > 2:
            lists.append(rng.permutation(h))
    for k in range(400):      # random multisets over few and many labels (forces the warp and block paths too)
        nl = int(rng.integers(1, min(ctr.max_ix, (700 if k % 10 == 1 else 90) if k % 2 else 8)))   # > 64: block kernel; > 32: several chunks of its walk; > 512: unstaged walk
        labs = rng.choice(ctr.max_ix, nl, replace=False)
        cnt = rng.integers(1, 40, nl)
        h = np.repeat(labs, cnt).astype(np.uint32)
        lists.append(rng.permutation(h))
    lists.append(np.zeros(0, dtype=np.uint32))
    off = np.zeros(len(lists) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([l.size for l in lists])
    # sprinkle misses between the hits: they must be ignored
    try:
        res = db.vote_hits(np.concatenate(lists), off, sparse=sparse)
    finally:
        for k in env:
            del os.environ[k]
    for i, h in enumerate(lists):
        v = orc.vote(h)
        r = res[i]
        assert r["kind"] == v.kind, i
        if v.kind == 0:
            continue
        assert (r["label"], r["found"], r["uix"]) == (v.label, v.found, v.uix), i
        if v.kind == 2:
            assert (r["cut"], r["sl"], r["ol"]) == (v.cut, v.sl, v.ol), i


def _taxonomy_labels(rng, n_target):
    """A quirky taxonomy with ~n_target distinct labels: shared prefixes, labels that stop at every rank, empty
    ranks, tokens that are prefixes of other tokens, names with underscores -- every branch of itree.c:1052-1069."""
    ranks = [b"k__", b"p__", b"c__", b"o__", b"f__", b"g__", b"s__", b"t__"]
    labels = set()
    names = [b"A", b"Ab", b"Ab_c", b"B", b"Ba", b"C_", b"", b"Zeta", b"Zet", b"Q_1", b"Q_12", b"m"]
    while len(labels) < n_target:
        depth = int(rng.integers(1, 9))
        toks = []
        for d in range(depth):
            pool = 2 if d < 2 else 4 if d < 4 else len(names)
            toks.append(ranks[d] + names[int(rng.integers(0, pool))] + (b"%d" % rng.integers(0, 3) if d >= 5 and rng.random() < 0.5 else b""))
            labels.add(b";".join(toks))
    return sorted(labels, key=lambda _: rng.random())


def test_vote_with_hundreds_of_labels_per_read(built, tmp_path):
    """Long queries touch hundreds of labels: the block kernels' walk over a staged copy of the label strings (32
    neighbour pairs per step, several steps per level), the unstaged walk beyond 512 labels, and the split path."""
    from tools import synth
    from utree_b200 import capi
    rng = np.random.default_rng(77)
    labels = _taxonomy_labels(rng, 900)
    words = np.sort(rng.choice(2 ** 62, len(labels) * 3, replace=False).astype(np.uint64))
    ixs = np.arange(words.size) % len(labels)
    path = str(tmp_path / "many.ctr")
    synth.ctr_write(path, words, ixs, synth._label_tail(labels, np.bincount(ixs, minlength=len(labels))), ix_bytes=2)
    ctr = capi.Ctr(path)
    assert ctr.max_ix == len(labels)
    orc = oracle_api.OracleDb(path)
    by_str = sorted(range(len(labels)), key=lambda i: labels[i])
    lists = []
    for k in range(300):
        nl = int(rng.integers(2, [40, 120, 500, 880][k % 4]))
        # a lineage (a stretch of neighbours in string order) that holds most of the hits, plus strays
        a = int(rng.integers(0, len(labels) - 1))
        width = int(rng.integers(1, max(2, nl // 2)))
        core = [by_str[(a + j) % len(labels)] for j in range(width)]
        stray = rng.choice(len(labels), max(1, nl - width), replace=False)
        heavy = int(rng.integers(1, 2000))
        h = np.concatenate([np.repeat(core, rng.integers(1, heavy + 1, len(core))), np.repeat(stray, rng.integers(1, 4, stray.size))])
        lists.append(rng.permutation(h).astype(np.uint32))
    off = np.zeros(len(lists) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([l.size for l in lists])
    flat = np.concatenate(lists)
    kinds = set()
    try:
        for env in ({}, {"UTB_VOTE_SPLIT_SLOTS": "64"}):
            os.environ.update(env)
            try:
                db = capi.Db(ctr, 0)
                try:
                    for sparse in (False, True):
                        res = db.vote_hits(flat, off, sparse=sparse)
                        for i, h in enumerate(lists):
                            v = orc.vote(h)
                            r = res[i]
                            kinds.add((v.kind, v.cut == 0xFFFFFFFE))
                            assert (r["kind"], r["label"], r["found"], r["uix"]) == (v.kind, v.label, v.found, v.uix), (env, sparse, i)
                            if v.kind == 2:
                                assert (r["cut"], r["sl"], r["ol"]) == (v.cut, v.sl, v.ol), (env, sparse, i)
                finally:
                    db.free()
            finally:
                for k in env:
                    del os.environ[k]
    finally:
        orc.free(); ctr.close()
    assert len(kinds) >= 2


@pytest.mark.parametrize("db_name,reads,out,rc", CASES)
def test_search_file_matches_reference(gpu, tmp_path, db_name, reads, out, rc):
    from utree_b200 import capi
    ctr = gpu[db_name][0]
    s = capi.Searcher(ctr, devices=(0,), host_threads=2)
    try:
        o = str(tmp_path / "out.txt")
        code, ref_exit, st = s.search_file(gold(reads), o, do_rc=bool(rc))
        assert code == 0 and ref_exit == 0
        assert open(o, "rb").read() == open(gold(out), "rb").read()
        assert st["kernel_launches"] >= 3
        data = open(gold(reads), "rb").read()
        code, ref_exit, text, st2 = s.search_mem(data, do_rc=bool(rc))
        assert code == 0 and text == open(gold(out), "rb").read()
        assert st2["lookups"] == st["lookups"] and st2["good_finds"] == st["good_finds"]
    finally:
        s.destroy()


def test_file_sinks_mapping_pwrite_and_fifo_agree(gpu, tmp_path, monkeypatch):
    """The three ways a file sink is written (shared mapping on a memory file system, parallel pwrite,
    sequential write into something that cannot seek) produce the same bytes, over several batches."""
    import threading
    from utree_b200 import capi
    ctr = gpu["toyA"][0]
    one = open(gold("toyA_reads.fa"), "rb").read()
    reads = one * (72_000_000 // len(one) + 1)                      # the smallest batch holds one maximal record (2 x 16 MiB)
    fa = tmp_path / "in.fa"
    fa.write_bytes(reads)
    shm = "/dev/shm/utb_test_%d.out" % os.getpid()
    monkeypatch.setenv("UTB_BATCH_MB", "1")
    s = capi.Searcher(ctr, devices=(0,), host_threads=3)
    try:
        code, _, want, st0 = s.search_mem(reads, do_rc=True)
        assert code == 0 and st0["batches"] >= 2 and want.count(b"\n") > 1000
        for mode, target in (("1", shm), ("0", shm), (None, str(tmp_path / "o.txt"))):
            if mode is None:
                monkeypatch.delenv("UTB_OUT_MMAP", raising=False)
            else:
                monkeypatch.setenv("UTB_OUT_MMAP", mode)
            open(target, "wb").write(b"stale" * 1000)               # an existing longer file must end up truncated
            code, ref_exit, st = s.search_file(str(fa), target, do_rc=True)
            assert code == 0 and ref_exit == 0
            assert open(target, "rb").read() == want, (mode, target)
        fifo = str(tmp_path / "pipe")
        os.mkfifo(fifo)
        got = []
        t = threading.Thread(target=lambda: got.append(open(fifo, "rb").read()))
        t.start()
        code, ref_exit, st = s.search_file(str(fa), fifo, do_rc=True)
        t.join(60)
        assert code == 0 and got and got[0] == want
    finally:
        s.destroy()
        if os.path.exists(shm):
            os.remove(shm)


def test_search_counts_match_oracle(gpu, tmp_path):
    from utree_b200 import capi
    ctr, db, orc = gpu["toyA"]
    s = capi.Searcher(ctr, devices=(0,), host_threads=1)
    try:
        o = str(tmp_path / "o.txt")
        _, _, st = s.search_file(gold("toyA_reads.fa"), o, do_rc=True)
        _, ost, _ = orc.search_file(gold("toyA_reads.fa"), str(tmp_path / "o2.txt"), do_rc=True)
        assert st["lookups"] == ost["lookups"] and st["hits"] == ost["hits"]
        assert st["good_finds"] == ost["good_finds"] and st["reads"] == ost["reads"]
    finally:
        s.destroy()


def test_virtual_devices_same_output(gpu, tmp_path):
    """Shard logic: N device slots mapped onto one GPU give the identical ordered output."""
    from utree_b200 import capi
    ctr = gpu["toyA"][0]
    want = open(gold("toyA_rc.out"), "rb").read()
    os.environ["UTB_BATCH_MB"] = "33"      # small batches -> several per device
    try:
        for devs in ((0, 0), (0, 0, 0, 0)):
            s = capi.Searcher(ctr, devices=devs, host_threads=2)
            try:
                code, _, text, st = s.search_mem(open(gold("toyA_reads.fa"), "rb").read() * 1, do_rc=True)
                assert code == 0 and text == want
            finally:
                s.destroy()
    finally:
        del os.environ["UTB_BATCH_MB"]


@pytest.mark.parametrize("bad", BAD_CASES)
def test_malformed_fasta_exit_codes(gpu, tmp_path, meta, bad):
    from utree_b200 import capi
    ctr = gpu["toyA"][0]
    s = capi.Searcher(ctr, devices=(0,), host_threads=1)
    try:
        o = str(tmp_path / "o.txt")
        code, ref_exit, st = s.search_file(gold(bad), o, do_rc=True)
        assert code == 3 and ref_exit == meta[bad]["exit"] == 2
        assert open(o, "rb").read() == open(gold(bad + ".out"), "rb").read()
    finally:
        s.destroy()


@pytest.mark.parametrize("db_name,reads,out,rc", [CASES[0], CASES[2], CASES[8]])
def test_cli_binary_matches_reference(ctrs, tmp_path, db_name, reads, out, rc):
    exe = os.path.join(ROOT, "bin", "utree-search_gg")
    o = str(tmp_path / "cli.out")
    args = [exe, ctrs[db_name], gold(reads), o, "2"] + (["RC"] if rc else [])
    p = subprocess.run(args, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr
    assert open(o, "rb").read() == open(gold(out), "rb").read()
    lines = p.stdout.splitlines()
    assert lines[0] == "This is UTree [v2.0RF SigNature Edition]"
    assert lines[-1].startswith("Searched ") and lines[-2].startswith("Good finds: ")
    n_out = sum(1 for _ in open(gold(out), "rb"))
    assert lines[-2] == f"Good finds: {n_out}"


@pytest.mark.parametrize("reads,out,rc", [c[1:] for c in (CASES[0], CASES[1], CASES[7], CASES[8])])
def test_cli_with_sieve_forced_on_matches_reference(ctrs, tmp_path, reads, out, rc):
    """The CLI with the sieve kernel forced on writes the golden bytes: reads of 150 bp (both strands and forward
    only), the edge cases, and the 64 kb queries, whose tiles run into the guard groups."""
    exe = os.path.join(ROOT, "bin", "utree-search_gg")
    o = str(tmp_path / "cli.out")
    p = subprocess.run([exe, ctrs["toyA"], gold(reads), o, "2"] + (["RC"] if rc else []), capture_output=True, text=True,
                       timeout=600, env=dict(os.environ, UTB_SIEVE="1"))
    assert p.returncode == 0, p.stderr
    assert open(o, "rb").read() == open(gold(out), "rb").read()


@pytest.mark.parametrize("complevel", [0, 2])
def test_synthetic_ctr_equals_reference_built_tree(built, tmp_path, complevel):
    """The GPU CTR synthesiser (bench input generator) against the REAL builder:
    same universe through utree-build_gg + utree-compress and through
    uts_build_ctr must classify identically, and the product must write on the
    synthesised tree what the reference search wrote (reference_runs.json; live
    when oracle/_ref is built).  The built tree comes from the product's builder
    and compressor, byte-identical to the reference's, and from the reference
    binaries too when they are there."""
    from utree_b200 import build, capi
    from tools import synthgpu
    build.build_synth()
    ref = os.path.join(ROOT, "oracle", "_ref")
    uni = synthgpu.Universe(seed=99, n_phyla=2, n_genera=2, n_species=2, n_strains=3, genome_len=30000)
    fa, mp = str(tmp_path / "g.fa"), str(tmp_path / "g.map")
    with open(fa, "wb") as f, open(mp, "wb") as m:
        for g in range(uni.n_genomes):
            f.write(b">gen%d\n" % g + uni.genome_ascii(g) + b"\n")
            m.write(b"gen%d\t" % g + uni.genome_tax(g) + b"\n")
    ubt, ctr_built, ctr_syn = str(tmp_path / "t.ubt"), str(tmp_path / "built.ctr"), str(tmp_path / "syn.ctr")
    rc, _, _ = capi.build_ubt(fa, mp, ubt, complevel=complevel, gg=True, ix_bytes=2)
    assert rc == 0, capi.lib().utb_last_error()
    capi.compress_ubt(ubt, ctr_built)
    trees = [ctr_built]
    if os.path.exists(os.path.join(ref, "utree-build_gg")):
        ctr_ref, ubt_ref = str(tmp_path / "ref.ctr"), str(tmp_path / "ref.ubt")
        subprocess.run([os.path.join(ref, "utree-build_gg"), fa, mp, ubt_ref, "1", str(complevel)], check=True, stdout=subprocess.DEVNULL)
        subprocess.run([os.path.join(ref, "utree-compress"), ubt_ref, ctr_ref], check=True, stdout=subprocess.DEVNULL)
        assert open(ctr_ref, "rb").read() == open(ctr_built, "rb").read()
        trees.append(ctr_ref)
    n, nl = uni.build_ctr(ctr_syn, complevel=complevel)
    assert n == np.frombuffer(open(ctr_built, "rb").read(32), dtype="<u8")[3]
    reads = str(tmp_path / "r.fa")
    uni.make_reads(20000, read_len=150).tofile(reads)
    outs = []
    for c in trees + [ctr_syn]:
        ctr = capi.Ctr(c)
        s = capi.Searcher(ctr, devices=(0,), host_threads=2)
        try:
            code, _, text, st = s.search_mem(open(reads, "rb").read(), do_rc=True)
            assert code == 0
            outs.append(text)
        finally:
            s.destroy(); ctr.close()
        if c != ctr_syn and os.path.exists(os.path.join(ref, "utree-search_gg")):
            o = c + ".out"
            subprocess.run([os.path.join(ref, "utree-search_gg"), c, reads, o, "1", "RC"], check=True, stdout=subprocess.DEVNULL)
            outs.append(open(o, "rb").read())
    assert all(o == outs[-1] for o in outs) and outs[-1].count(b"\n") > 15000
    check_reference_run(f"synthetic_ctr_complevel{complevel}", outs[-1])


def _lookup_probe_words(words, rng):
    w = np.concatenate([words, words + np.uint64(1), words - np.uint64(1),
                        (words & ~np.uint64(0xFFFFFFFFFF)) | rng.integers(0, 1 << 40, words.size, dtype=np.uint64),
                        (words & ~np.uint64(0xFFFFFFFFFF)), (words | np.uint64(0xFFFFFFFFFF)),
                        rng.integers(0, np.iinfo(np.uint64).max, 5000, dtype=np.uint64)])
    return w[rng.permutation(w.size)[:60000]]


@pytest.mark.parametrize("name", ["toyA", "toyB_u32", "quirk", "dense"])
def test_both_lookup_variants_match_oracle(built, ctrs, name):
    """Interpolation-start search (regular CTRs) and the exact-probe kernel give XT_getIX32's answer."""
    from utree_b200 import capi
    from tools import synth
    words, _, _, _ = synth.ubt_read(gold(name + ".ubt"))
    w = _lookup_probe_words(words, np.random.default_rng(17))
    orc = oracle_api.OracleDb(ctrs[name])
    want = orc.lookup_many(w)
    orc.free()
    ctr = capi.Ctr(ctrs[name])
    try:
        for env, mode in ((None, 1), ("exact", 0)):
            if env:
                os.environ["UTB_LOOKUP"] = env
            try:
                db = capi.Db(ctr, 0)
            finally:
                os.environ.pop("UTB_LOOKUP", None)
            assert db.lookup_mode() == mode          # every reference-compressed tree is regular
            assert np.array_equal(db.lookup_words(w), want), (name, env)
            db.free()
    finally:
        ctr.close()


def test_irregular_ctr_takes_the_exact_probe_path(built, tmp_path):
    """A CTR with an unsorted bucket (never produced by utree-compress): the loader detects it
    and the device emulates xtSuffixBS's probe sequence, matching the oracle hit for hit."""
    from utree_b200 import capi
    from tools import synth
    rng = np.random.default_rng(23)
    words, ixs, tail, _ = synth.ubt_read(gold("dense.ubt"))
    binix = synth.binix_like_reference(words)
    shuffled = words.copy()
    pre = words >> np.uint64(40)
    for p in np.unique(pre)[3::4]:                      # shuffle every 4th bucket in place
        idx = np.flatnonzero(pre == p)
        shuffled[idx] = shuffled[rng.permutation(idx)]
    path = str(tmp_path / "irregular.ctr")
    synth.ctr_write(path, shuffled, ixs, tail, 2, binix=binix)
    ctr, orc = capi.Ctr(path), oracle_api.OracleDb(path)
    db = capi.Db(ctr, 0)
    try:
        assert db.lookup_mode() == 0
        w = _lookup_probe_words(words, rng)
        assert np.array_equal(db.lookup_words(w), orc.lookup_many(w))
        s = capi.Searcher(ctr, devices=(0,), host_threads=2)
        o1, o2 = str(tmp_path / "a.out"), str(tmp_path / "b.out")
        code, _, _ = s.search_file(gold("dense_reads.fa"), o1, do_rc=True)
        orc.search_file(gold("dense_reads.fa"), o2, do_rc=True)
        assert code == 0 and open(o1, "rb").read() == open(o2, "rb").read()
        s.destroy()
    finally:
        db.free(); ctr.close(); orc.free()


@pytest.mark.parametrize("db_name,reads,out,rc", [CASES[0], CASES[2], CASES[7], CASES[8]])
def test_host_formatter_path_matches_reference(gpu, db_name, reads, out, rc):
    """utb_batch_submit hands back one result record per read and utb_format_results writes the lines on the host
    (the search pipeline builds them on the device): the reference's output."""
    from utree_b200 import capi
    ctr, db, _ = gpu[db_name]
    data = open(gold(reads), "rb").read()
    code, _, used, recs, (name_off, name_len) = capi.frame_records(data, threads=2)
    assert code == 0 and used == len(data)
    lens = np.array([len(seq) for _, seq in recs], dtype=np.uint32)
    n, total = len(recs), int(lens.sum())
    b = capi.Batch(db, total + 64, n)
    try:
        b.bytes[:total] = np.frombuffer(b"".join(seq for _, seq in recs), dtype=np.uint8)
        b.seq_off[0] = 0
        b.seq_off[1:n] = np.cumsum(lens[:-1], dtype=np.uint64)
        b.seq_len[:n] = lens
        b.submit(total, n, rc)
        text = capi.format_results(ctr, data, name_off, name_len, b.wait())
    finally:
        b.destroy()
    assert text == open(gold(out), "rb").read()


@pytest.mark.parametrize("host_frame", [0, 1])
def test_zero_copy_from_pinned_caller_buffer(gpu, host_frame):
    """utb_search_mem on a page-locked caller buffer: framed in place (on the device, or by the host framer with
    UTB_HOST_FRAME=1), copied to the device from where it lies."""
    import torch
    from utree_b200 import capi
    data = open(gold("toyB_reads.fa"), "rb").read() + open(gold("edge_reads.fa"), "rb").read()
    want_b = open(gold("toyB_u32_rc.out"), "rb").read()
    pinned = torch.empty(len(data), dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[:] = np.frombuffer(data, dtype=np.uint8)
    if host_frame:
        os.environ["UTB_HOST_FRAME"] = "1"
    os.environ["UTB_BATCH_MB"] = "33"
    try:
        s = capi.Searcher(gpu["toyB_u32"][0], devices=(0, 0), host_threads=6)
    finally:
        os.environ.pop("UTB_HOST_FRAME", None); os.environ.pop("UTB_BATCH_MB", None)
    try:
        rc, ex, text, st = s.search_mem(None, do_rc=True, ptr=pinned.data_ptr(), n=len(data))
        rc2, ex2, text2, st2 = s.search_mem(data, do_rc=True)            # pageable copy of the same bytes
        assert rc == 0 and rc2 == 0 and text == text2
        assert text.startswith(want_b) and st["reads"] == st2["reads"]
    finally:
        s.destroy()


def test_tree_with_a_long_label_is_searched_in_smaller_batches(built, tmp_path):
    """A batch's output lines are built on the device in a buffer sized for every read printing the longest label,
    addressed with 32 bits.  toyA with one label 32 KB longer would need far more than that at the default
    reads per batch, so the searcher takes fewer reads per batch (about 130 thousand here).  Its reads, twice,
    around 200 thousand random 40-mers that hit nothing: two batches at least, with lines in the first and
    the last, 132 of them ending in the long label.  The output equals the checker's."""
    import collections
    from tools import synth
    from utree_b200 import capi
    words, ixs, tail, ix_bytes = synth.ubt_read(gold("toyA.ubt"))
    labels = [l.rsplit(b"\t", 1)[0] for l in tail.split(b"\n") if l]
    printed = collections.Counter(l.split(b"\t")[1] for l in open(gold("toyA_rc.out"), "rb").read().splitlines())
    longest = max(range(len(labels)), key=lambda i: printed[labels[i]])
    labels[longest] += b"x" * 32768
    path = str(tmp_path / "long.ctr")
    synth.ctr_write(path, words, ixs, synth._label_tail(labels, np.bincount(ixs.astype(np.int64), minlength=len(labels))),
                    ix_bytes=ix_bytes)
    rng = np.random.default_rng(3)
    pad = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, (200_000, 40))]
    toy = open(gold("toyA_reads.fa"), "rb").read()
    fa = str(tmp_path / "reads.fa")
    open(fa, "wb").write(toy + b"".join(b">p%d\n%s\n" % (k, pad[k].tobytes()) for k in range(len(pad))) + toy)
    orc = oracle_api.OracleDb(path)
    want = str(tmp_path / "want.out")
    code, ost, err = orc.search_file(fa, want, do_rc=True)
    orc.free()
    assert code == 0, err
    want = open(want, "rb").read()
    assert sum(1 for l in want.splitlines() if l.split(b"\t")[1] == labels[longest]) == 132
    ctr = capi.Ctr(path)
    s = capi.Searcher(ctr, devices=(0,), host_threads=4)
    try:
        o = str(tmp_path / "out.txt")
        code, _, st = s.search_file(fa, o, do_rc=True)
        assert code == 0 and open(o, "rb").read() == want
        code, _, text, st2 = s.search_mem(open(fa, "rb").read(), do_rc=True)
        assert code == 0 and text == want
        for x in (st, st2):
            assert x["batches"] >= 2 and (x["reads"], x["good_finds"]) == (ost["reads"], ost["good_finds"])
    finally:
        s.destroy(); ctr.close()


@pytest.mark.parametrize("env", [{"UTB_SIEVE": "0"}, {"UTB_SIEVE": "1"}, {"UTB_LOOKUP": "exact"}])
@pytest.mark.parametrize("db_name,reads,out,rc", [CASES[0], CASES[2], CASES[5], CASES[7]])
def test_every_lookup_variant_gives_the_reference_output(ctrs, tmp_path, env, db_name, reads, out, rc):
    """Whole search with the sieve forced off (one table lookup per window), forced on (two-phase),
    and with the reference probe sequence: identical bytes."""
    from utree_b200 import capi
    os.environ.update(env)
    try:
        ctr = capi.Ctr(ctrs[db_name])
        s = capi.Searcher(ctr, devices=(0,), host_threads=3)
    finally:
        for k in env:
            del os.environ[k]
    try:
        code, ref_exit, text, st = s.search_mem(open(gold(reads), "rb").read(), do_rc=bool(rc))
        assert code == 0 and text == open(gold(out), "rb").read()
    finally:
        s.destroy(); ctr.close()


def test_long_queries_split_across_ctas_and_merged(ctrs, tmp_path):
    """64 kb queries with the split threshold lowered to 8192 lookup slots: every one of them is voted by
    the whole grid (per-read histogram, touched-label list, one merge + walk): identical bytes."""
    from utree_b200 import capi
    os.environ["UTB_VOTE_SPLIT_SLOTS"] = "8192"
    try:
        ctr = capi.Ctr(ctrs["toyA"])
        s = capi.Searcher(ctr, devices=(0,), host_threads=3)
    finally:
        del os.environ["UTB_VOTE_SPLIT_SLOTS"]
    try:
        data = open(gold("long_reads.fa"), "rb").read() + open(gold("toyA_reads.fa"), "rb").read()
        want = open(gold("long_rc.out"), "rb").read() + open(gold("toyA_rc.out"), "rb").read()
        code, ref_exit, text, st = s.search_mem(data * 3, do_rc=True)
        assert code == 0 and text == want * 3
    finally:
        s.destroy(); ctr.close()


@pytest.mark.parametrize("qcap", ["128", "1024"])
@pytest.mark.parametrize("db_name,reads,out,rc", [CASES[0], CASES[1], CASES[2], CASES[5], CASES[7]])
def test_survivor_queue_overflow_resolves_inline(ctrs, tmp_path, db_name, reads, out, rc, qcap):
    """UTB_QCAP shrinks the survivor queue to one / eight chunks, so almost every sieve survivor takes the
    overflow path (exact lookup inside the sieve kernel) and the consumer sees a full queue whose capacity
    is a whole number of chunks: identical bytes, no entry read that was never written.  The input is
    repeated so that every persistent warp walks several tiles."""
    from utree_b200 import capi
    os.environ["UTB_QCAP"] = qcap
    os.environ["UTB_SIEVE"] = "1"
    try:
        ctr = capi.Ctr(ctrs[db_name])
        s = capi.Searcher(ctr, devices=(0,), host_threads=3)
    finally:
        del os.environ["UTB_QCAP"], os.environ["UTB_SIEVE"]
    try:
        reps = 24 if reads != "long_reads.fa" else 2
        data = open(gold(reads), "rb").read()
        code, ref_exit, text, st = s.search_mem(data * reps, do_rc=bool(rc))
        assert code == 0 and text == open(gold(out), "rb").read() * reps
    finally:
        s.destroy(); ctr.close()


@pytest.mark.parametrize("mode", ["device", "host_frame"])
def test_device_framing_across_batches_and_restart_on_a_bad_record(gpu, mode):
    """Records framed on the GPU (the host only cuts chunks before a line that begins with '>' and never waits
    for the device): several batches with a carried tail, CRLF / tab-in-header / empty-line records, and
    malformed input deep in the stream -- the device flags the chunk or the record, the reader rewinds to
    that batch and the host framer reproduces the reference's partial output and exit code.
    UTB_HOST_FRAME=1 (host framer throughout) must give the same bytes."""
    from utree_b200 import capi
    one = open(gold("toyA_reads.fa"), "rb").read()
    want = open(gold("toyA_rc.out"), "rb").read()
    reps = 180                                                      # 35.6 MB: two 33.5 MB batches
    edge = open(gold("edge_reads.fa"), "rb").read()
    if not edge.endswith(b"\n"):
        edge += b"\n"
    os.environ["UTB_BATCH_MB"] = "33"
    if mode == "host_frame":
        os.environ["UTB_HOST_FRAME"] = "1"
    try:
        s = capi.Searcher(gpu["toyA"][0], devices=(0, 0), host_threads=5)
    finally:
        os.environ.pop("UTB_BATCH_MB", None); os.environ.pop("UTB_HOST_FRAME", None)
    try:
        rc, ex, text, st = s.search_mem(one * reps, do_rc=True)
        assert rc == 0 and st["batches"] >= 2 and st["reads"] == reps * one.count(b">")
        assert text == want * reps
        rc, ex, text, st = s.search_mem(edge, do_rc=True)
        assert rc == 0 and text == open(gold("edge_rc.out"), "rb").read()
        # no header '>' on a record of the second batch
        rc, ex, text, st = s.search_mem(one * reps + b"ACGT\nACGT\n" + one, do_rc=True)
        assert (rc, ex) == (3, 2) and text == want * reps
        # sequence line begins '>' inside the first batch
        rc, ex, text, st = s.search_mem(one + b">x\n>y\n" + one * reps, do_rc=True)
        assert (rc, ex) == (3, 2) and text == want
        # an EARLIER malformed record decides, also when the reader itself stops on a later error (dangling header
        # without newline in the final, host-framed chunk)
        rc, ex, text, st = s.search_mem(one * reps + b"ACGT\nACGT\n" + one * reps + b">dangling", do_rc=True)
        assert (rc, ex) == (3, 2) and text == want * reps
        assert b"no header" in capi.lib().utb_last_error()
        # a stray empty line shifts the pairing (the line count of the chunk before the next '>' is odd): header
        # "" of the next pair has no '>' (itree.c:880)
        rc, ex, text, st = s.search_mem(one + b"\n" + one * reps, do_rc=True)
        assert (rc, ex) == (3, 2) and text == want
        # two anomalies that keep the line count even: ">x" takes ">y" as its sequence
        rc, ex, text, st = s.search_mem(one * 3 + b">x\n>y\nACGT\n>z\n" + one * reps, do_rc=True)
        assert (rc, ex) == (3, 2) and text == want * 3
        # a NUL byte in the chunk: the count flags it and the exact host reader takes the batch
        # (strlen() semantics, itree.c:887: the sequence ends at the NUL)
        first = one.split(b"\n", 2)
        cut = first[0] + b"\n" + first[1][:60] + b"\0" + first[1][60:] + b"\n" + first[2]
        rc, ex, text, st = s.search_mem(cut, do_rc=True)
        orc = gpu["toyA"][2]
        import tempfile
        with tempfile.TemporaryDirectory() as d:
            fa, out = os.path.join(d, "n.fa"), os.path.join(d, "n.out")
            open(fa, "wb").write(cut)
            orc.search_file(fa, out, do_rc=True)
            assert rc == 0 and text == open(out, "rb").read()
        # and the searcher is reusable afterwards
        rc, ex, text, st = s.search_mem(one * 2, do_rc=True)
        assert rc == 0 and text == want * 2
    finally:
        s.destroy()


def test_empty_and_hitless_inputs(gpu, tmp_path):
    """Empty FASTA, reads shorter than k, reads of only N: no output line, exit 0 (itree.c:1028)."""
    from utree_b200 import capi
    s = capi.Searcher(gpu["toyA"][0], devices=(0,), host_threads=2)
    try:
        for name, data, n_reads in (("empty", b"", 0), ("short", b">a\nACGT\n>b\n" + b"A" * 31 + b"\n", 2),
                                    ("allN", b">n1\n" + b"N" * 200 + b"\n>n2\n\n", 2)):
            p = str(tmp_path / (name + ".fa"))
            open(p, "wb").write(data)
            o = str(tmp_path / (name + ".out"))
            rc, ex, st = s.search_file(p, o, do_rc=True)
            assert (rc, ex) == (0, 0) and open(o, "rb").read() == b"" and st["reads"] == n_reads and st["good_finds"] == 0
            rc, ex, text, st = s.search_mem(data, do_rc=True)
            assert (rc, ex, text) == (0, 0, b"")
    finally:
        s.destroy()


def test_cli_reads_fasta_from_a_pipe(ctrs, tmp_path):
    """Non-seekable input (serial read path) gives the same bytes."""
    exe = os.path.join(ROOT, "bin", "utree-search_gg")
    o = str(tmp_path / "pipe.out")
    with open(gold("toyA_reads.fa"), "rb") as f:
        p = subprocess.run([exe, ctrs["toyA"], "/dev/stdin", o, "4", "RC"], stdin=f, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr
    assert open(o, "rb").read() == open(gold("toyA_rc.out"), "rb").read()
    # through a real pipe as well
    q = subprocess.run(f"cat {gold('toyB_reads.fa')} | {exe} {ctrs['toyB_u32']} /dev/stdin {o} 3 RC", shell=True,
                       capture_output=True, text=True, timeout=600)
    assert q.returncode == 0, q.stderr
    assert open(o, "rb").read() == open(gold("toyB_u32_rc.out"), "rb").read()


# ---- the non-GG binary (utree-search, -D SEARCH): SPARSITY-skip slide + shallow vote (SURVEY 8f-3) --------------
import json as _json
SHALLOW = _json.load(open(os.path.join(conftest.GOLD, "meta_shallow.json")))


@pytest.mark.parametrize("name", sorted(SHALLOW))
def test_shallow_search_matches_the_reference_binary(ctrs, tmp_path, name):
    """utb_searcher_set_shallow: the bytes oracle/_ref/utree-search wrote for the same tree and reads (golden files made
    by scripts/make_golden_shallow.py), "Good finds" and "Searched" included.  The vote of a read depends on the reads
    before it (itree.c:982), so equality here also pins the input order through the batches."""
    from utree_b200 import capi
    m = SHALLOW[name]
    ctr = capi.Ctr(ctrs[m["db"]])
    s = capi.Searcher(ctr, devices=(0,), host_threads=3)
    try:
        s.set_shallow(True)
        out = str(tmp_path / "o.out")
        rc, ex, st = s.search_file(gold(m["reads"]), out, do_rc=bool(m["rc"]))
        assert rc == 0 and open(out, "rb").read() == open(gold(name), "rb").read()
        assert [f"Good finds: {st['good_finds']}", f"Searched {st['reads']} queries"] == m["stdout_tail"]
        # memory API, twice: every search starts from a clean AllTheKingsHorses, like a fresh process
        for _ in range(2):
            rc, ex, text, st = s.search_mem(open(gold(m["reads"]), "rb").read(), do_rc=bool(m["rc"]))
            assert rc == 0 and text == open(gold(name), "rb").read()
    finally:
        s.destroy(); ctr.close()


@pytest.mark.parametrize("env", [{}, {"UTB_HOST_FRAME": "1"}, {"UTB_SIEVE": "0"}, {"UTB_LOOKUP": "exact"}])
def test_shallow_search_across_batches_and_lookup_variants(gpu, tmp_path, env):
    """Several batches (the stale entry of itree.c:982 crosses batch boundaries), device- and host-framed, with the
    sieve off (dense hit slots instead of the hit map) and with the reference probe sequence: the CPU checker's
    restatement of the non-GG binary (itself pinned by the golden files) gives the expected bytes."""
    from utree_b200 import capi
    ctr, db, orc = gpu["toyA"]
    data = (open(gold("shallow_reads.fa"), "rb").read() + open(gold("toyA_reads.fa"), "rb").read() + open(gold("long_reads.fa"), "rb").read()) * 110   # 42 MB
    fa, want = str(tmp_path / "in.fa"), str(tmp_path / "want.out")
    open(fa, "wb").write(data)
    rc, st, err = orc.search_file_shallow(fa, want, do_rc=True)
    assert rc == 0, err
    os.environ.update(env)
    os.environ["UTB_BATCH_MB"] = "33"
    try:
        s = capi.Searcher(ctr, devices=(0, 0), host_threads=4)
        s.set_shallow(True)
    finally:
        for k in list(env) + ["UTB_BATCH_MB"]:
            del os.environ[k]
    try:
        rc, ex, text, st2 = s.search_mem(data, do_rc=True)
        assert rc == 0 and st2["batches"] >= 2 and text == open(want, "rb").read()
        assert (st2["good_finds"], st2["reads"]) == (st["good_finds"], st["reads"])
    finally:
        s.destroy()


def test_shallow_cli_binary(ctrs, tmp_path):
    """bin/utree-search: argv, banner and output of the reference's non-GG binary."""
    exe = os.path.join(ROOT, "bin", "utree-search")
    p = subprocess.run([exe], capture_output=True, text=True)
    assert p.returncode == 1 and "usage: xtree-search compTree.ctr" in p.stdout
    out = str(tmp_path / "o.out")
    p = subprocess.run([exe, ctrs["toyA"], gold("toyA_reads.fa"), out, "2", "RC"], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    assert open(out, "rb").read() == open(gold("shallow_toyA_toyA_rc.out"), "rb").read()
    assert p.stdout.splitlines()[-2:] == SHALLOW["shallow_toyA_toyA_rc.out"]["stdout_tail"]
    ref = os.path.join(ROOT, "oracle", "_ref", "utree-search")
    if os.path.exists(ref):
        q = subprocess.run([ref, ctrs["toyA"], gold("toyA_reads.fa"), out + ".ref", "2", "RC"], capture_output=True, text=True)
        assert q.stdout == p.stdout


# ---- utree-build_gg on the GPU (SURVEY 8f-4) ---------------------------------------------------------------------
BUILD_CASES = [
    # name, make_genomes kwargs, complevel, ix_bytes, golden .ubt made by the reference builder (scripts/make_golden.py);
    # None: compared with the digests of the reference's output in reference_runs.json
    ("toyA", dict(seed=11, n_phyla=2, n_genera=2, n_species=2, n_strains=2, length=4000), 0, 2, "toyA.ubt"),
    ("toyB", dict(seed=21, n_phyla=3, n_genera=2, n_species=2, n_strains=2, length=6000, quirky_tax=True), 1, 4, "toyB_u32.ubt"),
    ("mid2", dict(seed=5, n_phyla=3, n_genera=3, n_species=3, n_strains=2, length=30000), 2, 2, None),
    ("mid4", dict(seed=6, n_phyla=2, n_genera=3, n_species=2, n_strains=3, length=60000, quirky_tax=True), 4, 2, None),
]


@pytest.mark.parametrize("name,kw,complevel,ix_bytes,golden", BUILD_CASES)
def test_gpu_builder_is_byte_identical_to_the_reference_builder(built, tmp_path, name, kw, complevel, ix_bytes, golden):
    """FASTA + map -> .ubt on the GPU: the bytes the reference's serial builder writes (words, label ids in its
    order of registration incl. superseded derived labels, counts, .gg.log), against the committed .ubt fixtures
    or the digests of the reference's files and stdout, and, where oracle/_ref is present, against the reference
    builder run live on the same input."""
    from tools import synth
    from utree_b200 import capi
    genomes = synth.make_genomes(**kw)
    fa, mp, out = str(tmp_path / "g.fa"), str(tmp_path / "g.map"), str(tmp_path / "ours.ubt")
    synth.write_fasta_and_map(genomes, fa, mp)
    rc, ex, st = capi.build_ubt(fa, mp, out, complevel=complevel, gg=True, ix_bytes=ix_bytes)
    assert rc == 0, capi.lib().utb_last_error()
    got = open(out, "rb").read()
    assert st["records"] == int.from_bytes(got[24:32], "little") > 0
    if golden:
        assert got == open(gold(golden), "rb").read()
    else:
        check_reference_run(f"build_{name}.ubt", got, text=False)
        check_reference_run(f"build_{name}.ubt.gg.log", open(out + ".gg.log", "rb").read())
        p = subprocess.run([os.path.join(ROOT, "bin", "utree-build_gg"), fa, mp, out + "2", "1", str(complevel)], capture_output=True)
        assert p.returncode == 0 and open(out + "2", "rb").read() == got
        check_reference_run(f"build_{name}.stdout", p.stdout)
    ref = os.path.join(ROOT, "oracle", "_ref", "utree-build_gg" + ("_u32" if ix_bytes == 4 else ""))
    if os.path.exists(ref):
        rout = str(tmp_path / "ref.ubt")
        q = subprocess.run([ref, fa, mp, rout, "1", str(complevel)], capture_output=True, text=True)
        assert q.returncode == 0
        assert got == open(rout, "rb").read()
        assert open(out + ".gg.log", "rb").read() == open(rout + ".gg.log", "rb").read()
        if ix_bytes == 2:                                           # the CLI: same stdout lines
            env = dict(os.environ)
            p = subprocess.run([os.path.join(ROOT, "bin", "utree-build_gg"), fa, mp, out + "2", "1", str(complevel)], capture_output=True, text=True, env=env)
            assert p.returncode == 0 and open(out + "2", "rb").read() == got
            assert p.stdout == q.stdout
