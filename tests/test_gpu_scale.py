"""Parity at the scales BASELINE.json names, against the UNMODIFIED reference
binary (threads=1 = input order): the L2-scale CTR, the L4 CTR, a uint32_t-label
CTR with > 65,536 labels at complevel 0, and long / whole-genome queries up to the
16,777,214-base limit.  Inputs come from the seeded GPU synthesiser (itself checked
against the real builder in test_gpu_parity.py); what the reference wrote for them
is kept in tests/golden/reference_runs.json, and the reference also runs live when
oracle/_ref is built."""
import os
import subprocess
import sys
import time

import numpy as np
import pytest

from conftest import ROOT, check_reference_run

pytestmark = pytest.mark.gpu
REF = os.path.join(ROOT, "oracle", "_ref")


def _ref_search(ctr, fasta, out, u32=False):
    """The reference binary's output, or None when oracle/_ref is not built."""
    exe = os.path.join(REF, "utree-search_gg" + ("_u32" if u32 else ""))
    if not os.path.exists(exe):
        return None
    p = subprocess.run([exe, ctr, fasta, out, "1", "RC"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert p.returncode == 0, p.stderr[-500:]
    return open(out, "rb").read()


def _ours(ctr_path, fasta_bytes):
    from utree_b200 import capi
    ctr = capi.Ctr(ctr_path)
    s = capi.Searcher(ctr, devices=(0,), host_threads=8)
    try:
        rc, ex, text, st = s.search_mem(fasta_bytes, do_rc=True)
        assert rc == 0 and ex == 0
        return text, st
    finally:
        s.destroy(); ctr.close()


@pytest.fixture(scope="module")
def bench_mod(built):
    sys.path.insert(0, ROOT)
    import bench
    from utree_b200 import build
    build.build_synth()
    return bench


@pytest.mark.parametrize("config,n_reads", [("l2s", 150_000), ("l4", 300_000)])
def test_l2_scale_and_l4_match_reference(bench_mod, tmp_path, config, n_reads):
    cfg = dict(bench_mod.CONFIGS[config])
    ctr_path, meta = bench_mod.ensure_ctr(config, cfg, 0)
    assert meta["records"] > (900_000_000 if config == "l2s" else 40_000_000)
    reads, _ = bench_mod.make_reads(cfg, 60_000_000, n_reads, 0)          # a window of the read stream the bench never uses
    fa = str(tmp_path / "r.fa")
    reads.tofile(fa)
    got, st = _ours(ctr_path, reads.tobytes())
    check_reference_run(f"scale_{config}_{n_reads}", got)
    want = _ref_search(ctr_path, fa, str(tmp_path / "ref.out"))
    assert want is None or got == want
    assert got.count(b"\n") > 0.9 * n_reads * (0.5 if config == "l4" else 1) * 0.5
    assert st["lookups"] > 200 * n_reads


def test_l2_scale_two_million_reads_every_batch_size(bench_mod, tmp_path):
    """2 M reads against the L2-scale tree: full-size 128 MiB batches (the shape the bench's e2e leg runs) and the
    ramp batches at both ends.  The reference runs with all host threads, so its lines come in any order
    (SURVEY 0 #3): the two outputs must hold the same lines, ours in input order.  The recorded output is those
    lines in input order."""
    cfg = dict(bench_mod.CONFIGS["l2s"])
    ctr_path, _ = bench_mod.ensure_ctr("l2s", cfg, 0)
    n_reads = 2_000_000
    reads, _ = bench_mod.make_reads(cfg, 70_000_000, n_reads, 0)
    fa = str(tmp_path / "r.fa")
    got, st = _ours(ctr_path, reads.tobytes())
    assert st["batches"] >= 4 and st["reads"] == n_reads
    check_reference_run("scale_l2s_2M_every_batch_size", got)
    lines = got.split(b"\n")
    exe = os.path.join(REF, "utree-search_gg")
    if os.path.exists(exe):
        reads.tofile(fa)
        p = subprocess.run([exe, ctr_path, fa, str(tmp_path / "ref.out"), str(os.cpu_count() or 4), "RC"],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        assert p.returncode == 0, p.stderr[-500:]
        want = open(str(tmp_path / "ref.out"), "rb").read().split(b"\n")
        assert sorted(lines) == sorted(want)
    names = [ln.split(b"\t", 1)[0] for ln in lines if ln]
    assert names == sorted(names) and len(names) > 0.9 * n_reads      # names are r%09u: input order = sorted


def test_two_physical_gpus_one_searcher(bench_mod, tmp_path):
    """ONE searcher over two physical devices (tables uploaded to the first, cloned to the second over NVLink,
    batches dealt round-robin, ordered merge) gives the bytes of a single-device search."""
    from utree_b200 import capi
    if capi.device_count() < 2:
        pytest.skip("one GPU visible")
    cfg = dict(bench_mod.CONFIGS["small"])
    ctr_path, _ = bench_mod.ensure_ctr("small", cfg, 0)
    reads, _ = bench_mod.make_reads(cfg, 0, 1_500_000, 0)
    data = reads.tobytes()
    one, st1 = _ours(ctr_path, data)
    ctr = capi.Ctr(ctr_path)
    s = capi.Searcher(ctr, devices=(0, 1), host_threads=8)
    try:
        rc, ex, two, st2 = s.search_mem(data, do_rc=True)
        assert rc == 0 and two == one and st2["reads"] == st1["reads"] and st2["batches"] >= 4
    finally:
        s.destroy(); ctr.close()


def test_uint32_labels_over_64k_match_reference(bench_mod, tmp_path):
    """IXTYPE=uint32_t (SZ=9), complevel 0, 73,260 labels, 250 bp reads."""
    from tools import synthgpu
    uni = synthgpu.Universe(77, 60, 11, 10, 10, 6000)                 # 66,000 genomes
    ctr_path = os.path.join(bench_mod.work_dir(), "u32_test.ctr")
    n, nl = uni.build_ctr(ctr_path, complevel=0, ix_bytes=4)
    try:
        assert nl > 65536 and n > 50_000_000
        reads = uni.make_reads(100_000, read_len=250, read_seed=5)
        fa = str(tmp_path / "r.fa")
        reads.tofile(fa)
        got, st = _ours(ctr_path, reads.tobytes())
        check_reference_run("scale_u32_100k", got)
        want = _ref_search(ctr_path, fa, str(tmp_path / "ref.out"), u32=True)
        assert want is None or got == want
        assert st["hits"] > 10 * 100_000                              # dense tree: most k-mers of a read hit
    finally:
        os.remove(ctr_path)


def test_long_and_whole_genome_queries_match_reference(bench_mod, tmp_path):
    """10 kb - 1 Mb reads, whole genomes, and one query at the 16,777,214-base limit vs the L2-scale CTR."""
    from tools import synthgpu
    cfg = dict(bench_mod.CONFIGS["l2s"])
    ctr_path, _ = bench_mod.ensure_ctr("l2s", cfg, 0)
    uni = synthgpu.Universe(bench_mod.SEED, *cfg["universe"])
    rng = np.random.default_rng(4)
    g = [uni.genome_ascii(i) for i in (0, 1, 2, 77, 4999)]            # 4 Mb each
    comp = bytes.maketrans(b"ACGT", b"TGCA")
    recs = [(b"whole_genome_0", g[0]), (b"whole_genome_rc", g[3].translate(comp)[::-1]),
            (b"max_length", (g[0] + g[1] + g[2] + g[4] + g[3])[:16_777_214])]
    for i in range(40):
        L = int(10 ** rng.uniform(4, 6))
        src = g[int(rng.integers(len(g)))]
        st = int(rng.integers(0, len(src) - L))
        seq = bytearray(src[st:st + L])
        for p in rng.integers(0, L, L // 100):                         # 1 % substitutions
            seq[p] = b"ACGT"[(b"ACGT".index(seq[p]) + 1) % 4]
        if i % 5 == 0:
            seq[L // 2:L // 2 + 3] = b"NNN"
        recs.append((b"long%d" % i, bytes(seq)))
    recs.append((b"short_after_long", g[1][1000:1150]))
    fasta = b"".join(b">" + n + b"\n" + s + b"\n" for n, s in recs)
    fa = str(tmp_path / "long.fa")
    open(fa, "wb").write(fasta)
    got, st = _ours(ctr_path, fasta)
    check_reference_run("scale_long_queries", got)
    assert got.count(b"\n") == len(recs)
    t = time.time()
    want = _ref_search(ctr_path, fa, str(tmp_path / "ref.out"))
    assert want is None or got == want
    if want is not None:
        print(f"long queries: {sum(len(s) for _, s in recs) / 1e6:.1f} Mb, reference {time.time() - t:.1f} s (incl. load), "
              f"ours {st['seconds_total']:.2f} s")


def test_tree_with_more_than_2_32_records(bench_mod):
    """4,295,000,000 records: the CTR carries 8-byte prefix-index entries (itree.c:757, 1303) and record indices
    beyond 32 bits.  Content is closed-form (tools/synth.cu big_word), so members, their labels and non-members
    are known by arithmetic; both device paths -- the sector hash table (+ sieve) built from the index, and the
    reference probe sequence on the on-disk image -- must agree with it."""
    import shutil
    from tools import synthgpu
    from utree_b200 import capi
    wd = bench_mod.work_dir()
    n, n_labels = 4_295_000_000, 1000
    if shutil.disk_usage(wd).free < 40 * 10 ** 9:
        pytest.skip("not enough room in " + wd)
    path = os.path.join(wd, "big64.ctr")
    try:
        synthgpu.build_big_ctr(path, n, n_labels)
        ctr = capi.Ctr(path)
        assert ctr.binix_bytes == 8 and ctr.num_nodes == n and ctr.max_ix == n_labels
        rng = np.random.default_rng(3)
        idx = np.concatenate([np.array([0, 1, 2, 2 ** 32 - 2, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 1, n - 2, n - 1], dtype=np.uint64),
                              rng.integers(0, n, 300_000, dtype=np.uint64), rng.integers(2 ** 32, n, 50_000, dtype=np.uint64)])
        words, labels = synthgpu.big_ctr_word_label(idx, n, n_labels)
        nxt, _ = synthgpu.big_ctr_word_label(np.minimum(idx + np.uint64(1), np.uint64(n - 1)), n, n_labels)
        strangers = words + np.uint64(1)
        ok = strangers != nxt                                       # word + 1 is a member only if it is the next record
        q = np.concatenate([words, strangers[ok]])
        want = np.concatenate([labels, np.full(int(ok.sum()), 0xFFFFFFFF, dtype=np.uint32)])
        for env in ({}, {"UTB_LOOKUP": "exact"}):
            os.environ.update(env)
            try:
                db = capi.Db(ctr, 0)
            finally:
                for k in env:
                    del os.environ[k]
            try:
                assert db.lookup_mode() == (0 if env else 1)
                got = db.lookup_words(q)
                assert np.array_equal(got, want), (env, int((got != want).sum()))
            finally:
                db.free()
        ctr.close()
    finally:
        if os.path.exists(path):
            os.remove(path)
