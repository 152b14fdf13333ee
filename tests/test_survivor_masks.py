"""The sieve survivors travel from phase A (sieve_kernel) to phase B (queue_lookup_kernel) as one 64-bit mask per
32-position step: bits 0-31 the forward windows of the step's 32 positions, bits 32-63 their reverse complements.
Phase B expands the masks of 32 steps at a time into a list.  These searches run with the sieve on and compare bytes
and lookup / hit / good-find counts with the checker's, on inputs made to reach the corners of that hand-over:

- full masks: a tree that holds every 32-mer of its reads on both strands, so every bit of most steps is set and a
  round of 32 steps carries 2,048 survivors;
- batch ends: one read of G groups for every G from 2 to 65, i.e. every residue of the group count mod 32 and mod
  the sieve kernel's steps per tile, the batch's last step with windows full of survivors;
- stale masks: a shorter batch after a hit-dense one in the same stream slot, whose masks past the new last step
  are left over and must not be decoded;
- padding: a tree that holds the all-A 32-mer, which is what the padding behind every read packs to, so a mask
  written for a step without windows would turn into a wrong hit."""
import contextlib
import os

import numpy as np
import pytest

import conftest  # noqa: F401  (puts the repo root on sys.path)

_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
LABELS = [b"k__B", b"k__B;p__A", b"k__B;p__Ab;c__C", b"k__Z", b"k__Z;p__Q_1", b"k__Z;p__Q_12;c__m"]
FRAMING = {"device": {}, "host": {"UTB_HOST_FRAME": "1"}}


def revcomp(seq):
    return seq.translate(bytes.maketrans(b"ACGT", b"TGCA"))[::-1]


def kmers(seq):
    """The 2-bit words of every 32-mer of seq (first base most significant)."""
    c = np.frombuffer(seq, dtype=np.uint8)
    code = ((c >> 1) ^ (c >> 2)) & 3                               # A 0, C 1, G 2, T 3
    n = len(seq) - 31
    w = np.zeros(n, dtype=np.uint64)
    for j in range(32):
        w |= code[j:j + n].astype(np.uint64) << np.uint64(62 - 2 * j)
    return w


def fasta(seqs):
    return b"".join(b">r%d\n%s\n" % (i, s) for i, s in enumerate(seqs))


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


def _tree(path, words, rng):
    from tools import synth
    words = np.unique(np.asarray(words, dtype=np.uint64))
    ixs = rng.integers(0, len(LABELS), words.size).astype(np.uint64)
    synth.ctr_write(path, words, ixs, synth._label_tail(LABELS, np.bincount(ixs.astype(np.int64), minlength=len(LABELS))),
                    ix_bytes=2)


@pytest.fixture(scope="module")
def full(built, tmp_path_factory):
    """Reads of 69 and 70 groups, half of them made of reverse-complement palindromes (X + revcomp(X) per 32
    bases), and a tree of all their 32-mers and of the reverse complements of those."""
    from oracle import oracle_api
    from utree_b200 import capi
    assert capi.device_count() >= 1
    rng = np.random.default_rng(61)
    seqs = []
    for i in range(12):
        if i % 2:
            halves = [bytes(_ACGT[rng.integers(0, 4, 16)]) for _ in range(70)]
            seqs.append(b"".join(h + revcomp(h) for h in halves)[:32 * 70 - 1])
        else:
            seqs.append(bytes(_ACGT[rng.integers(0, 4, 32 * 69 - 1 + i)]))
    src = bytes(_ACGT[rng.integers(0, 4, 32 * 66)])                # the batch-end reads are prefixes of it
    words = np.concatenate([kmers(s) for s in seqs + [src]] + [kmers(revcomp(s)) for s in seqs + [src]])
    path = str(tmp_path_factory.mktemp("survivor_masks") / "full.ctr")
    _tree(path, words, rng)
    ctr, orc = capi.Ctr(path), oracle_api.OracleDb(path)
    yield {"ctr": ctr, "orc": orc, "seqs": seqs, "src": src}
    ctr.close(); orc.free()


def _expect(orc, data, tmp_path, do_rc, shallow=False):
    fa, out = str(tmp_path / "q.fa"), str(tmp_path / "want.out")
    with open(fa, "wb") as f:
        f.write(data)
    rc, ost, err = (orc.search_file_shallow if shallow else orc.search_file)(fa, out, do_rc=do_rc)
    assert rc == 0, err
    return open(out, "rb").read(), ost


def _searcher(ctr, env):
    from utree_b200 import capi
    with _env(dict(env, UTB_SIEVE="1")):
        return capi.Searcher(ctr, devices=(0,), host_threads=3)


def _check(s, orc, data, tmp_path, do_rc, what):
    want, ost = _expect(orc, data, tmp_path, do_rc)
    code, _, text, st = s.search_mem(data, do_rc=do_rc)
    assert code == 0, what
    assert (st["lookups"], st["hits"], st["good_finds"]) == (ost["lookups"], ost["hits"], ost["good_finds"]), what
    assert text == want, what
    return ost


@pytest.mark.gpu
@pytest.mark.parametrize("framing", sorted(FRAMING))
def test_full_masks(full, tmp_path, framing):
    """Every window of every read is a member on both strands (but the one record the reference's index loses):
    2,048 survivors in each full round of 32 steps."""
    s = _searcher(full["ctr"], FRAMING[framing])
    try:
        for do_rc in (True, False):
            ost = _check(s, full["orc"], fasta(full["seqs"]), tmp_path, do_rc, do_rc)
            assert ost["lookups"] > 12 * 64 * 32 * (2 if do_rc else 1) and ost["hits"] >= ost["lookups"] - 4
    finally:
        s.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("framing", sorted(FRAMING))
def test_batch_ends(full, tmp_path, framing):
    """One read of 32 G - 1 bases (G groups; its last step with windows, G - 2, is full of survivors) per batch,
    G = 2 .. 65: every residue of G mod 32 and mod 6 (the sieve kernel's steps per tile)."""
    s = _searcher(full["ctr"], FRAMING[framing])
    try:
        for g in range(2, 66):
            for do_rc in (True, False):
                ost = _check(s, full["orc"], fasta([full["src"][:32 * g - 1]]), tmp_path, do_rc, (g, do_rc))
                assert ost["lookups"] == (g - 1) * 32 * (2 if do_rc else 1) and ost["hits"] >= ost["lookups"] - 4, (g, do_rc)
    finally:
        s.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("framing", sorted(FRAMING))
def test_shorter_batch_after_a_dense_one(full, tmp_path, framing):
    """Every search starts in the same stream slot: the batches after the first, hit-dense one have fewer steps,
    and the masks behind their last step are the dense batch's."""
    s = _searcher(full["ctr"], FRAMING[framing])
    try:
        dense = fasta(full["seqs"] * 4)
        for do_rc in (True, False):
            _check(s, full["orc"], dense, tmp_path, do_rc, ("dense", do_rc))
            for g in (3, 33, 40, 64):
                _check(s, full["orc"], fasta([full["src"][:32 * g - 1]]), tmp_path, do_rc, (g, do_rc))
            _check(s, full["orc"], fasta(full["seqs"][:3]), tmp_path, do_rc, ("three reads", do_rc))
    finally:
        s.destroy()


@pytest.mark.gpu
def test_full_masks_non_gg(full, tmp_path):
    """The non-GG search (bin/utree-search): phase B files the hits by slot and marks them in the hit map."""
    data = fasta(full["seqs"])
    s = _searcher(full["ctr"], {})
    try:
        s.set_shallow(True)
        for do_rc in (True, False):
            want, ost = _expect(full["orc"], data, tmp_path, do_rc, shallow=True)
            code, _, text, st = s.search_mem(data, do_rc=do_rc)
            assert code == 0 and text == want, do_rc
            assert (st["good_finds"], st["reads"]) == (ost["good_finds"], ost["reads"]), do_rc
    finally:
        s.destroy()


@pytest.mark.gpu
def test_full_masks_across_batches(full, tmp_path):
    """Batches of 33 MB: one search of several hit-dense batches, the last one shorter than the others."""
    one = fasta(full["seqs"])
    reps = 80 * 1024 * 1024 // len(one) + 1
    want, ost = _expect(full["orc"], one, tmp_path, True)
    s = _searcher(full["ctr"], {"UTB_BATCH_MB": "33"})
    try:
        code, _, text, st = s.search_mem(one * reps, do_rc=True)
        assert code == 0 and st["batches"] >= 3
        assert (st["lookups"], st["hits"], st["good_finds"]) == (ost["lookups"] * reps, ost["hits"] * reps,
                                                                 ost["good_finds"] * reps)
        assert text == want * reps
    finally:
        s.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("do_rc", [True, False])
def test_padding_packs_to_a_member(built, tmp_path, do_rc):
    """All-A reads of many lengths between random ones, in a tree that holds the all-A and the all-T 32-mer (and a
    second word of the all-A prefix bin, so that the reference's index keeps the bin): the last step of every read has no window, and
    padding packs to A, so any mask left in such a step would add hits of the all-A word.  The sieve kernel's warps
    walk several tiles each, so a step without windows follows one with survivors in the same warp's registers."""
    from oracle import oracle_api
    from utree_b200 import capi
    rng = np.random.default_rng(62)
    seqs = []
    for i in range(12000):                                         # several tiles of the sieve kernel per warp
        seqs.append(b"A" * int(rng.integers(32, 400)) if i % 3 else bytes(_ACGT[rng.integers(0, 4, int(rng.integers(32, 400)))]))
    rand = [s for s in seqs if s.count(b"A") != len(s)]
    words = np.concatenate([np.array([0, 1, (1 << 64) - 1], dtype=np.uint64)] + [kmers(s) for s in rand[::2]] + [kmers(revcomp(s)) for s in rand[1::2]])
    path = str(tmp_path / "a.ctr")
    _tree(path, words, rng)
    ctr, orc = capi.Ctr(path), oracle_api.OracleDb(path)
    try:
        for framing in sorted(FRAMING):
            s = _searcher(ctr, FRAMING[framing])
            try:
                ost = _check(s, orc, fasta(seqs), tmp_path, do_rc, framing)
                assert ost["hits"] > 0.6 * ost["lookups"]
            finally:
                s.destroy()
    finally:
        ctr.close(); orc.free()
