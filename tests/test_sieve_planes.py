"""The sieve works on the bit planes of a 32-mer (code bit 1 of every base in one u32, code bit 0 in another, base 0
the most significant bit), the exact lookup on the 2-bit word.  These tests cover what a change of that encoding can
break: strand symmetry of the 16-mer keys (palindromes, ties in the canonical minimum, all-A / all-T), the first and
the last 16-mer of a window as its minimizer (lane 0 and the funnel-shift edge of the sieve kernel), the plane <-> word
conversions on the survivor path, and the 2-bit packing that the other consumers still read."""
import contextlib
import os

import numpy as np
import pytest

import conftest  # noqa: F401  (puts the repo root on sys.path)

M32 = 0xFFFFFFFF
MISS = 0xFFFFFFFF
_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
LABELS = [b"k__B", b"k__B;p__A", b"k__B;p__Ab;c__C", b"k__Z", b"k__Z;p__Q_1", b"k__Z;p__Q_12;c__m"]


# ---- a model of the sieve's 16-mer keys (kernels.cu sv_kmer16 / sv_rc16 / sv_mhash) --------------------------------
def seq_word(s):
    w = 0
    for c in s:
        w = (w << 2) | b"ACGT".index(c)
    return w


def word_seq(w):
    return bytes(_ACGT[[(w >> (62 - 2 * i)) & 3 for i in range(32)]])


def revcomp(seq):
    return seq.translate(bytes.maketrans(b"ACGTacgtN", b"TGCAtgcaN"))[::-1]


def planes(w):
    x1 = x0 = 0
    for i in range(32):
        c = (w >> (62 - 2 * i)) & 3
        x1, x0 = (x1 << 1) | (c >> 1), (x0 << 1) | (c & 1)
    return x1, x0


def brev32(x):
    return int(f"{x:032b}"[::-1], 2)


def key16(x1, x0, j):
    """Key of the 16-mer at offset j: its planes a1, a0 laid out as a1[15:8] | a0 | a1[7:0]."""
    a1, a0 = (x1 >> (16 - j)) & 0xFFFF, (x0 >> (16 - j)) & 0xFFFF
    return ((a1 >> 8) << 24) | (a0 << 8) | (a1 & 0xFF)


def rc16(m):
    return ~brev32(m) & M32


def mhash(m):
    a = min(m, rc16(m))
    a = a * 0x9E3779B1 & M32
    a ^= a >> 15
    return a * 0x85EBCA77 & M32


def order_keys(w):
    x1, x0 = planes(w)
    return [mhash(key16(x1, x0, j)) for j in range(17)]


def rc_word(w):
    return seq_word(revcomp(word_seq(w)))


# ---- the words the sieve must not lose -----------------------------------------------------------------------------
def sieve_words(seed=7):
    """name -> member words."""
    rng = np.random.default_rng(seed)

    def rand(n):
        return bytes(_ACGT[rng.integers(0, 4, n)])
    out = {"homopolymers": [seq_word(b * 32) for b in (b"A", b"C", b"G", b"T")],
           "palindromes": [], "first": [], "last": []}
    for k in range(64):                          # a 16-mer that is its own reverse complement, at every offset 0..16
        h = rand(8)
        pal = h + revcomp(h)
        o = k % 17
        out["palindromes"].append(seq_word(rand(o) + pal + rand(16 - o)))
    for k in range(16):                          # a 32-mer that is its own reverse complement: every key ties twice
        h = rand(16)
        out["palindromes"].append(seq_word(h + revcomp(h)))
    out["palindromes"].append(seq_word(b"ACGT" * 8))
    while len(out["first"]) < 64 or len(out["last"]) < 64:
        w = int(rng.integers(0, 1 << 63, dtype=np.uint64)) * 2 + int(rng.integers(0, 2))
        h = order_keys(w)
        j = h.index(min(h))
        if h.count(min(h)) == 1 and j in (0, 16):
            lst = out["first" if j == 0 else "last"]
            if len(lst) < 64:
                lst.append(w)
    return out


def test_keys_are_strand_symmetric():
    """The reverse complement of a word has the same 17 keys in reverse order: same minimizer, and the first and the
    last key (the block) swap."""
    ws = sieve_words()
    for name, lst in ws.items():
        for w in lst:
            assert order_keys(rc_word(w)) == order_keys(w)[::-1], (name, hex(w))


def test_constructed_minimizer_positions():
    ws = sieve_words()
    for name, j in (("first", 0), ("last", 16)):
        for w in ws[name]:
            h = order_keys(w)
            assert h.index(min(h)) == j and h.count(min(h)) == 1
    # the reverse complement of a "first" word has its minimizer last, and the other way round
    for w in ws["first"]:
        h = order_keys(rc_word(w))
        assert h.index(min(h)) == 16
    # palindromic 16-mers: their key is their own reverse complement's
    pal = ws["palindromes"][0]
    assert any(key16(*planes(pal), j) == rc16(key16(*planes(pal), j)) for j in range(17))


# ---- GPU -----------------------------------------------------------------------------------------------------------
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


@pytest.fixture(scope="module")
def sieve_tree(built, tmp_path_factory):
    """A tree of the sieve words and random controls; the reverse complements of the words that are not
    palindromes stay absent, so the sieve has to tell the strands apart."""
    from tools import synth
    from utree_b200 import capi
    assert capi.device_count() >= 1
    rng = np.random.default_rng(8)
    ws = sieve_words()
    members = set(w for lst in ws.values() for w in lst)
    members |= set(int(x) * 2 + 1 for x in rng.integers(0, 1 << 63, 4000, dtype=np.uint64))
    words = np.array(sorted(members), dtype=np.uint64)
    ixs = rng.integers(0, len(LABELS), words.size).astype(np.uint64)
    path = str(tmp_path_factory.mktemp("sieve_planes") / "t.ctr")
    synth.ctr_write(path, words, ixs, synth._label_tail(LABELS, np.bincount(ixs.astype(np.int64), minlength=len(LABELS))),
                    ix_bytes=2)
    absent = [rc_word(w) for lst in ws.values() for w in lst]
    absent += [int(x) * 2 for x in rng.integers(0, 1 << 63, 4000, dtype=np.uint64)]
    absent = [w for w in absent if w not in members]
    return path, ws, words, np.array(absent, dtype=np.uint64)


@pytest.mark.gpu
def test_lookup_words_with_the_sieve_misses_no_member(sieve_tree):
    from oracle import oracle_api
    from utree_b200 import capi
    path, ws, words, absent = sieve_tree
    ctr, orc = capi.Ctr(path), oracle_api.OracleDb(path)
    try:
        probe = np.concatenate([words, absent])
        want = orc.lookup_many(probe)
        want = np.where(want < orc.max_ix, want, MISS).astype(np.uint32)
        assert np.count_nonzero(want[:words.size] == MISS) <= 1     # the first bucket's folded record 0 (all-A here)
        for env in ({"UTB_SIEVE": "1"}, {"UTB_SIEVE": "0"}):
            with _env(env):
                db = capi.Db(ctr, 0)
            try:
                assert db.lookup_mode() == 1
                got = db.lookup_words(probe)
                bad = np.flatnonzero(got != want)
                assert bad.size == 0, (env, [(hex(int(probe[i])), int(got[i]), int(want[i])) for i in bad[:8]])
            finally:
                db.free()
    finally:
        ctr.close(); orc.free()


@pytest.mark.gpu
@pytest.mark.parametrize("do_rc", [True, False])
def test_search_with_the_sieve_misses_no_member(sieve_tree, tmp_path, do_rc):
    """The sieve kernel builds every window from planes: reads that put each word at lane 0 of a group and at every
    other offset (so that its last 16-mer comes from the next group), forward and reverse complement.  Bytes and
    lookup / hit / good-find counts equal the checker's, with the survivor queue and with its overflow path."""
    from oracle import oracle_api
    from utree_b200 import capi
    path, ws, words, absent = sieve_tree
    rng = np.random.default_rng(9)
    special = [word_seq(w) for lst in ws.values() for w in lst]
    seqs = list(special)
    for i, s in enumerate(special):
        pad = bytes(_ACGT[rng.integers(0, 4, i % 32)])
        seqs.append(pad + s + bytes(_ACGT[rng.integers(0, 4, 7)]))
    seqs += [revcomp(s) for s in seqs]
    data = b"".join(b">r%d\n%s\n" % (i, s) for i, s in enumerate(seqs))
    fa, out = str(tmp_path / "q.fa"), str(tmp_path / "want.out")
    open(fa, "wb").write(data)
    orc = oracle_api.OracleDb(path)
    ctr = capi.Ctr(path)
    try:
        rc, ost, err = orc.search_file(fa, out, do_rc=do_rc)
        assert rc == 0, err
        assert ost["hits"] >= len(special)
        want = open(out, "rb").read()
        for env in ({"UTB_SIEVE": "1"}, {"UTB_SIEVE": "1", "UTB_QCAP": "128"}, {"UTB_SIEVE": "0"}):
            with _env(env):
                s = capi.Searcher(ctr, devices=(0,), host_threads=2)
            try:
                code, _, text, st = s.search_mem(data, do_rc=do_rc)
            finally:
                s.destroy()
            assert code == 0 and text == want, env
            assert (st["lookups"], st["hits"], st["good_finds"]) == (ost["lookups"], ost["hits"], ost["good_finds"]), env
    finally:
        ctr.close(); orc.free()


@pytest.mark.gpu
def test_pack_sequence_every_length_residue(built, tmp_path):
    """utb_pack_sequence (the 2-bit packing, unchanged) against a model, for lengths of every residue mod 32, with N
    and lower case."""
    from utree_b200 import capi
    from tools import synth
    assert capi.device_count() >= 1
    rng = np.random.default_rng(10)
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    path = str(tmp_path / "toyA.ctr")
    synth.compress(os.path.join(gold, "toyA.ubt"), path)
    ctr = capi.Ctr(path)
    db = capi.Db(ctr, 0)
    try:
        for n in range(1, 130):
            s = bytearray(_ACGT[rng.integers(0, 4, n)].tobytes())
            if n % 3 == 0:
                s[int(rng.integers(0, n))] = ord("N")
            if n % 5 == 0:
                s = bytearray(s.lower())
            s = bytes(s)
            fwd, rcw, valid = db.pack_sequence(s)
            up = s.upper()
            for p in range(n):
                ok = p + 32 <= n and b"N" not in up[p:p + 32]
                assert valid[p] == ok, (n, p)
                if ok:
                    assert int(fwd[p]) == seq_word(up[p:p + 32]), (n, p)
                    assert int(rcw[p]) == seq_word(revcomp(up[p:p + 32])), (n, p)
                else:
                    assert fwd[p] == 0 and rcw[p] == 0, (n, p)
    finally:
        db.free(); ctr.close()
