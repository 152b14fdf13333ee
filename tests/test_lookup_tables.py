"""The two lookup structures a regular CTR is searched through, on trees built to reach their edges.

The sector hash table (kernels.cu, kt_lookup / ktab_build_kernel) and the minimizer sieve in front of it are
built at load time.  Natural trees never displace an entry by more than a sector or two, never wrap, never
grow the table and put a member word at only a few lane offsets of the sieve kernel, so every tree here is
constructed: mix64 is invertible, so a record with any chosen hash, hence any chosen home sector, is
unmix64(hash).  Every answer is compared with the CPU checker (oracle/), which the golden tests pin to the
reference.  The CPU tests check the construction itself with a model of the table."""
import contextlib
import os

import numpy as np
import pytest

import conftest  # noqa: F401  (puts the repo root on sys.path)

MISS = 0xFFFFFFFF
M64 = (1 << 64) - 1
C1, C2 = 0xFF51AFD7ED558CCD, 0xC4CEB9FE1A85EC53
I1, I2 = pow(C1, -1, 1 << 64), pow(C2, -1, 1 << 64)
KT_MAXD = 63                                    # a record sits at most 63 sectors past its home
KT_MIN_SECTORS = (KT_MAXD + 1) << 16            # 2^22


# ---- the table, restated ----------------------------------------------------------------------------------------
def mix64(x):
    x ^= x >> 33
    x = x * C1 & M64
    x ^= x >> 33
    x = x * C2 & M64
    return x ^ (x >> 33)


def unmix64(h):
    h ^= h >> 33                                # x ^= x >> 33 is its own inverse on 64 bits
    h = h * I2 & M64
    h ^= h >> 33
    h = h * I1 & M64
    return h ^ (h >> 33)


def word_with_hash(h):
    return unmix64(h)


def home(h, S):
    return (h * S) >> 64


def slots(ix_bytes):
    """Entries per 32-byte sector: four (tag, remainder) words, or three with the 32-bit id inside."""
    return 3 if ix_bytes == 4 else 4


def table_sectors(n, ix_bytes):
    """The sizes the loader tries for n records: load <= 0.5, at least 2^22 sectors, then x1.5 three times."""
    s = n // 3 * 2 + 1 if ix_bytes == 4 else n // 2 + 1
    sizes = [max(s, KT_MIN_SECTORS)]
    for _ in range(3):
        sizes.append(sizes[-1] + sizes[-1] // 2)
    return sizes


def hash_in_sector(j, S, rng):
    """A hash whose home at S is sector j."""
    lo, hi = -(-(j << 64) // S), -(-((j + 1) << 64) // S)
    h = lo + int(rng.integers(0, hi - lo))
    assert home(h, S) == j
    return h


class Occupancy:
    """Linear probing over sectors of E entries.  Which entry ends where depends on the insertion order, how many
    entries each sector holds does not (as long as nothing overflows), so the sectors a MISS touches are exact."""

    def __init__(self, hashes, S, E):
        self.S, self.E, self.count, self.overflow = S, E, {}, 0
        for h in hashes:
            s = home(h, S)
            for _ in range(KT_MAXD + 1):
                if self.count.get(s, 0) < E:
                    self.count[s] = self.count.get(s, 0) + 1
                    break
                s = (s + 1) % S
            else:
                self.overflow += 1

    def full(self, s):
        return self.count.get(s % self.S, 0) == self.E

    def miss_sectors(self, h):
        """Sectors kt_lookup reads before it gives up on an absent word: up to the first one with a free slot."""
        s = home(h, self.S)
        for d in range(KT_MAXD + 1):
            if not self.full(s):
                return d + 1
            s = (s + 1) % self.S
        return KT_MAXD + 1


def reachable_slots(hashes, S, E):
    """Slots any record can take: those of the sectors within KT_MAXD of some record's home."""
    secs = set()
    for h in hashes:
        s = home(h, S)
        secs.update((s + d) % S for d in range(KT_MAXD + 1))
    return len(secs) * E


def max_homes_per_sector(hashes, S):
    c = {}
    for h in hashes:
        c[home(h, S)] = c.get(home(h, S), 0) + 1
    return max(c.values())


# ---- 2-bit words and FASTA ------------------------------------------------------------------------------------
_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def word_seq(w):
    """The 32 bases of a word, first base in the top bits (itree.c:924)."""
    return bytes(_ACGT[[(int(w) >> (62 - 2 * i)) & 3 for i in range(32)]])


def seq_words(seq):
    """Forward 32-mers of a sequence without N (upper or lower case)."""
    codes = np.frombuffer(seq.upper().translate(bytes.maketrans(b"ACGT", b"\0\1\2\3")), dtype=np.uint8)
    from tools import synth
    return synth.kmer_words(codes)


def revcomp(seq):
    return seq.translate(bytes.maketrans(b"ACGTacgtN", b"TGCAtgcaN"))[::-1]


def fasta(seqs, prefix="q"):
    return b"".join(b">%s%d\n%s\n" % (prefix.encode(), i, s) for i, s in enumerate(seqs))


LABELS = [b"k__B", b"k__B;p__A", b"k__B;p__Ab", b"k__B;p__Ab_c;c__", b"k__B;p__Ab;c__C;o__",
          b"k__B;p__Ab;c__C;o__O;f__F;g__G;s__S", b"k__B;p__Ab;c__C;o__O;f__F;g__G;s__S;t__T1",
          b"k__B;p__Ab;c__C;o__O;f__F;g__G;s__S;t__T12", b"k__B;p__Ab;c__C;o__O;f__F;g__Gz", b"k__Z;p__Q_1",
          b"k__Z;p__Q_12;c__m", b"k__Z"]


def write_ctr(path, hashes_ix, ix_bytes, labels=LABELS):
    """CTR file of records {unmix64(h): ix} with the reference compressor's prefix index (first-bin quirk
    included).  Ids >= len(labels) are kept as they are: the reference stores them and filters on lookup."""
    from tools import synth
    words = np.array([word_with_hash(h) for h, _ in hashes_ix], dtype=np.uint64)
    ixs = np.array([ix for _, ix in hashes_ix], dtype=np.uint64)
    order = np.argsort(words)
    words, ixs = words[order], ixs[order]
    assert np.all(words[1:] > words[:-1])
    valid = ixs[ixs < len(labels)].astype(np.int64)
    counts = np.bincount(valid, minlength=len(labels))
    synth.ctr_write(path, words, ixs, synth._label_tail(labels, counts), ix_bytes=ix_bytes)
    return words


# ---- the constructed trees ------------------------------------------------------------------------------------
class Tree:
    """records: [(hash, id)]; probes: name -> [hash]; placed: hashes the table holds (model input)."""

    def __init__(self):
        self.records, self.probes, self.placed, self.extra_words = [], {}, [], []


def _ids(rng, n):
    return [int(i) for i in rng.integers(0, len(LABELS), n)]


def tree_runs(ix_bytes, seed=1):
    """Cases 1-4, 7 and 8 on one table of S = 2^22 sectors (E entries each):
    run1   E*64 records homed at H1: they fill H1..H1+63, the last ones at displacement 63;
    h2     one record homed at H1+64, alone in its sector; h2 - 2^48 has the same low 48 bits and home H1;
    wrap   E*21 homed at S-24, E*23 at S-3, E*20 at sector 0: together S-24..39 full, across the table's end;
           one record at sector 40 (top 16 hash bits 0) whose low 48 bits a hash with top bits 0xFFFF and home
           S-24 shares;
    run7   ids the reference filters out (>= maxIX, the sentinels of 16-bit trees) amid a two-sector run;
    run8   a run holding the one record of the lowest prefix bin, which the reference's compressor folds away."""
    rng = np.random.default_rng(seed)
    E = slots(ix_bytes)
    S = KT_MIN_SECTORS
    H1, H7, H8 = 1_234_567, 2_345_678, 3_456_789
    t = Tree()
    t.S, t.E, t.ix_bytes = S, E, ix_bytes
    rec = t.records
    run1 = [hash_in_sector(H1, S, rng) for _ in range(E * 64)]
    h2 = hash_in_sector(H1 + 64, S, rng)
    rec += list(zip(run1 + [h2], _ids(rng, E * 64 + 1)))
    wrap = [hash_in_sector(S - 24, S, rng) for _ in range(E * 21)] + \
           [hash_in_sector(S - 3, S, rng) for _ in range(E * 23)] + [hash_in_sector(0, S, rng) for _ in range(E * 20)]
    h2w = hash_in_sector(40, S, rng)
    rec += list(zip(wrap + [h2w], _ids(rng, len(wrap) + 1)))
    maxix = len(LABELS)
    bad = [maxix, maxix + 1, 0x1234, 0xFFFD, 0xFFFE, 0xFFFF] if ix_bytes == 2 else \
          [maxix, maxix + 1, 0xFFFF, 0x10000, 0xFFFFFFFE, 0xFFFFFFFF]
    run7 = [hash_in_sector(H7, S, rng) for _ in range(E * 2 + len(bad))] + [hash_in_sector(H7 + 1, S, rng) for _ in range(E)]
    ids7 = _ids(rng, len(run7))
    for k, b in enumerate(bad):                  # spread over the run: before, between and after valid entries
        ids7[2 * k] = b
    rec += list(zip(run7, ids7))
    # run 8: the record of smallest word (alone in the lowest prefix bin) is homed at H8 among E*3 others
    best = min((hash_in_sector(H8, S, rng) for _ in range(60000)), key=word_with_hash)
    run8 = [hash_in_sector(H8, S, rng) for _ in range(E * 3)]
    rec += list(zip(run8 + [best], _ids(rng, E * 3 + 1)))
    t.quirk_hash = best
    words = sorted(word_with_hash(h) for h, _ in rec)
    assert words[0] == word_with_hash(best) and (words[0] >> 40) < (words[1] >> 40), "quirk record not alone in the first bin"
    # the compressor's fold: bin of words[1] starts at record 0, whose 40 suffix bits then read as that bin's
    p1, suf0, suf1 = words[1] >> 40, words[0] & ((1 << 40) - 1), words[1] & ((1 << 40) - 1)
    folded = (p1 << 40) | suf0
    t.extra_words = [words[0], folded]
    t.placed = [h for h, ix in rec if h != best and (ix < 0xFFFE if ix_bytes == 2 else ix < maxix)]
    if suf0 < suf1:                              # bucket still sorted: the table holds record 0 under the folded word
        t.placed.append(mix64(folded))
    # absent probes
    P = t.probes
    P["deep_home"] = [hash_in_sector(H1, S, rng) for _ in range(16)]
    P["deep_inside"] = [hash_in_sector(H1 + k, S, rng) for k in range(1, 64)]
    P["remainder"] = [(h2 - (1 << 48)) & M64, ((0xFFFF << 48) | h2w)]
    P["wrap_end"] = [hash_in_sector(S - 1, S, rng) for _ in range(8)] + [hash_in_sector(S - 24, S, rng) for _ in range(4)]
    P["wrap_inside"] = [hash_in_sector(k, S, rng) for k in (0, 1, 5, 20, 39)] + [hash_in_sector(S - 3, S, rng)]
    P["near7"] = [hash_in_sector(H7 + k, S, rng) for k in (0, 0, 1, 2)]
    P["near8"] = [hash_in_sector(H8 + k, S, rng) for k in (0, 0, 1)]
    t.h2, t.h2w = h2, h2w
    return t


def tree_growth(ix_bytes, seed=2):
    """Case 5: records spread evenly over a stretch of home sectors -- 5 per sector over 300 sectors (4-entry
    sectors) or 4 over 250 (3-entry) -- at fixed fractions of each sector, so that at S they outnumber every slot
    they can reach and at 1.5 S no sector is the home of more than it holds."""
    rng = np.random.default_rng(seed)
    E = slots(ix_bytes)
    per, span = (5, 300) if E == 4 else (4, 250)
    S = table_sectors(per * span, ix_bytes)[0]
    G = 1_111_111
    hashes = []
    for j in range(span):
        base = (G + j) << 42
        for i in range(per):
            hashes.append(base + (2 * i + 1) * (1 << 42) // (2 * per) + int(rng.integers(0, 1 << 30)))
    assert all(home(h, S) >= G for h in hashes)
    t = Tree()
    t.S, t.E, t.ix_bytes = S, E, ix_bytes
    t.records = list(zip(hashes, _ids(rng, len(hashes))))
    t.placed = hashes
    t.probes = {"around": [hash_in_sector(G + k, S, rng) for k in range(0, span + 70, 3)]}
    return t


def tree_unbuildable(ix_bytes, seed=3):
    """Case 6: 300 records whose hashes lie inside one sector of the largest table the loader tries."""
    rng = np.random.default_rng(seed)
    E = slots(ix_bytes)
    n = 300
    sizes = table_sectors(n, ix_bytes)
    j = 9_000_001
    hashes = [hash_in_sector(j, sizes[-1], rng) for _ in range(n)]
    t = Tree()
    t.S, t.E, t.ix_bytes, t.sizes = sizes[0], E, ix_bytes, sizes
    t.records = list(zip(hashes, _ids(rng, n)))
    t.placed = hashes
    t.probes = {"around": [hash_in_sector(home(hashes[0], sizes[0]) + k, sizes[0], rng) for k in range(-2, 70)]}
    return t


def tree_control(n, ix_bytes, seed=4):
    rng = np.random.default_rng(seed)
    t = Tree()
    t.records = [(int(h), ix) for h, ix in zip(rng.integers(0, 1 << 63, n, dtype=np.uint64) * 2 + 1, _ids(rng, n))]
    return t


# ---- CPU: the construction does what the GPU tests rely on -----------------------------------------------------
def test_mix64_inverse_round_trip():
    rng = np.random.default_rng(11)
    for w in [0, 1, M64, 1 << 63] + [int(x) for x in rng.integers(0, 1 << 63, 2000, dtype=np.uint64) * 2 + 1]:
        assert unmix64(mix64(w)) == w and mix64(unmix64(w)) == w
    # the finaliser the kernels use, on known values: mix64(1) from the constants by hand
    x = 1 ^ (1 >> 33)
    x = x * C1 & M64
    x ^= x >> 33
    x = x * C2 & M64
    assert mix64(1) == x ^ (x >> 33)


def test_table_sizes_follow_the_loader():
    assert table_sectors(100, 2) == [1 << 22, 3 << 21, 9 << 20, 27 << 19]
    assert table_sectors(20_000_000, 2)[0] == 10_000_001
    assert table_sectors(20_000_000, 4)[0] == 20_000_000 // 3 * 2 + 1


@pytest.mark.parametrize("ix_bytes", [2, 4])
def test_constructed_homes(ix_bytes):
    rng = np.random.default_rng(12)
    for S in table_sectors(1000, ix_bytes):
        for j in (0, 1, S // 2, S - 1):
            h = hash_in_sector(j, S, rng)
            assert home(h, S) == j and home(mix64(word_with_hash(h)), S) == j


@pytest.mark.parametrize("ix_bytes", [2, 4])
def test_runs_tree_shape(ix_bytes):
    t = tree_runs(ix_bytes)
    S, E = t.S, t.E
    occ = Occupancy(t.placed, S, E)
    assert occ.overflow == 0
    H1 = home(t.probes["deep_home"][0], S)
    assert all(occ.full(H1 + d) for d in range(64)) and occ.count[H1 + 64] == 1    # run 1 + h2 alone
    assert all(occ.full(s) for s in list(range(S - 24, S)) + list(range(40))) and occ.count[40] == 1
    # the remainder pairs: same low 48 bits, homes exactly 64 sectors apart modulo S
    for probe, member in zip(t.probes["remainder"], (t.h2, t.h2w)):
        assert probe & ((1 << 48) - 1) == member & ((1 << 48) - 1)
        assert (home(member, S) - home(probe, S)) % S == 64
        assert occ.miss_sectors(probe) == 64
    assert home(t.probes["remainder"][1], S) == S - 24 and t.probes["remainder"][1] >> 48 == 0xFFFF
    assert [occ.miss_sectors(h) for h in t.probes["deep_inside"]] == [65 - k for k in range(1, 64)]
    assert all(occ.miss_sectors(h) == 42 for h in t.probes["wrap_end"][:8])        # S-1, 0..39, 40
    # h2 is the record the wider reach would find: KT_MAXD + 1 sectors from the probe
    assert {home(t.h2, S), home(t.h2w, S)} == {H1 + 64, 40}


@pytest.mark.parametrize("ix_bytes", [2, 4])
def test_growth_tree_overflows_at_s_and_fits_at_one_and_a_half_s(ix_bytes):
    """Order-independent: at S the records outnumber every slot they can reach (so some record is unplaced
    whatever the order), at 1.5 S no sector is the home of more records than it holds (so none moves)."""
    t = tree_growth(ix_bytes)
    sizes = table_sectors(len(t.records), ix_bytes)
    assert sizes[0] == t.S == KT_MIN_SECTORS
    assert reachable_slots(t.placed, sizes[0], t.E) < len(t.placed)
    assert reachable_slots(t.placed, sizes[0], t.E) == (363 * 4 if ix_bytes == 2 else 313 * 3)
    assert max_homes_per_sector(t.placed, sizes[1]) <= t.E
    assert Occupancy(t.placed, sizes[1], t.E).overflow == 0


@pytest.mark.parametrize("ix_bytes", [2, 4])
def test_unbuildable_tree_overflows_at_every_size(ix_bytes):
    t = tree_unbuildable(ix_bytes)
    for S in t.sizes:
        homes = {home(h, S) for h in t.placed}
        assert len(homes) <= 2 and max(homes) - min(homes) <= 1
        assert reachable_slots(t.placed, S, t.E) <= 65 * t.E < len(t.placed)


# ---- GPU -----------------------------------------------------------------------------------------------------
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


def _want_lookup(orc, words):
    """XT_getIX32 and the ix < maxIX filter after it (itree.c:928-929): what the device lookups return."""
    w = orc.lookup_many(words)
    return np.where(w < orc.max_ix, w, MISS).astype(np.uint32)


def _check_lookups(ctr, orc, words, envs=({}, {"UTB_SIEVE": "0"}), mode=1):
    want = _want_lookup(orc, words)
    from utree_b200 import capi
    for env in envs:
        with _env(env):
            db = capi.Db(ctr, 0)
        try:
            assert db.lookup_mode() == mode, env
            got = db.lookup_words(words)
            bad = np.flatnonzero(got != want)
            assert bad.size == 0, (env, [(hex(int(words[i])), int(got[i]), int(want[i])) for i in bad[:8]])
        finally:
            db.free()
    return want


SEARCH_ENVS = ({"UTB_SIEVE": "0"}, {"UTB_SIEVE": "1"}, {"UTB_SIEVE": "1", "UTB_QCAP": "128"})


def _check_search(ctr_path, orc, data, tmp_path, envs=SEARCH_ENVS, do_rc=True):
    """Search bytes and the lookups / hits / good finds counts equal the CPU checker's."""
    from utree_b200 import capi
    fa, out = str(tmp_path / "q.fa"), str(tmp_path / "want.out")
    open(fa, "wb").write(data)
    rc, ost, err = orc.search_file(fa, out, do_rc=do_rc)
    assert rc == 0, err
    want = open(out, "rb").read()
    ctr = capi.Ctr(ctr_path)
    try:
        for env in envs:
            with _env(env):
                s = capi.Searcher(ctr, devices=(0,), host_threads=2)
            try:
                code, _, text, st = s.search_mem(data, do_rc=do_rc)
            finally:
                s.destroy()
            assert code == 0 and text == want, env
            assert (st["lookups"], st["hits"], st["good_finds"]) == (ost["lookups"], ost["hits"], ost["good_finds"]), env
    finally:
        ctr.close()
    return ost


def _reads_for(t, members, absent):
    """32-bp reads of single words (one window each), concatenations of member words and their reverse
    complements."""
    seqs = [word_seq(w) for w in list(members) + list(absent)]
    m = [word_seq(w) for w in members]
    cat = [b"".join(m[i:i + 5]) for i in range(0, len(m), 5)]
    return fasta(seqs + cat + [revcomp(c) for c in cat])


def _sector_count(ctr, words, expect):
    """Absent probes alone, sieve off, one strand: table sectors the batch read == the model's count."""
    from utree_b200 import capi
    with _env({"UTB_SIEVE": "0"}):
        db = capi.Db(ctr, 0)
    b = capi.Batch(db, 64 * len(words) + 64, len(words))
    try:
        for i, w in enumerate(words):
            b.bytes[33 * i:33 * i + 33] = np.frombuffer(word_seq(w) + b"\n", dtype=np.uint8)
        b.seq_off[:len(words)] = np.arange(len(words), dtype=np.uint64) * 33
        b.seq_len[:len(words)] = 32
        b.submit(33 * len(words), len(words), False)
        b.wait()
        assert b.counts() == (len(words), 0)
        assert b.lookup_detail()[1][1] == expect
    finally:
        b.destroy(); db.free()


@pytest.fixture(scope="module")
def gpu_built(built):
    from utree_b200 import capi
    assert capi.device_count() >= 1
    return True


@pytest.mark.gpu
@pytest.mark.parametrize("ix_bytes", [2, 4])
def test_runs_displacement_wrap_remainder_filtered_ids_and_quirk(gpu_built, tmp_path, ix_bytes):
    """Cases 1-4, 7 and 8 on one constructed tree per id width."""
    from oracle import oracle_api
    from utree_b200 import capi
    t = tree_runs(ix_bytes)
    path = str(tmp_path / "runs.ctr")
    write_ctr(path, t.records, ix_bytes)
    orc = oracle_api.OracleDb(path)
    ctr = capi.Ctr(path)
    try:
        assert orc.max_ix == len(LABELS)
        members = [word_with_hash(h) for h, _ in t.records]
        absent = [word_with_hash(h) for p in t.probes.values() for h in p]
        rng = np.random.default_rng(7)
        rand = [int(x) for x in rng.integers(0, 1 << 63, 2000, dtype=np.uint64)]
        words = np.array(members + absent + t.extra_words + rand, dtype=np.uint64)
        want = _check_lookups(ctr, orc, words)
        n_m = len(members)
        valid = np.array([ix < len(LABELS) and h != t.quirk_hash for h, ix in t.records])
        assert np.all(want[:n_m][valid] != MISS)                     # the members the reference finds...
        assert np.all(want[:n_m][~valid] == MISS)                    # ...and the filtered ids and the folded record
        assert np.all(want[n_m:n_m + len(absent)] == MISS)           # constructed probes are absent
        assert want[n_m + len(absent)] == MISS                       # the folded record, under its own word
        # the table's sectors for absent probes of cases 2-4 follow the model: the chains are 64 sectors long
        occ = Occupancy(t.placed, t.S, t.E)
        deep = [h for k in ("deep_home", "deep_inside", "remainder", "wrap_end", "wrap_inside") for h in t.probes[k]]
        expect = sum(occ.miss_sectors(h) for h in deep)
        assert expect > 30 * len(deep)
        _sector_count(ctr, [word_with_hash(h) for h in deep], expect)
        data = _reads_for(t, members, absent + t.extra_words)
        ost = _check_search(path, orc, data, tmp_path)
        assert ost["hits"] >= int(valid.sum())
    finally:
        ctr.close(); orc.free()


@pytest.mark.gpu
@pytest.mark.parametrize("ix_bytes", [2, 4])
def test_table_grows_when_a_record_cannot_be_placed(gpu_built, tmp_path, ix_bytes):
    """Case 5: placement overflows at S under any insertion order and fits at 1.5 S: the table grew by
    S/2 sectors of 32 bytes over a tree of as many records, and every answer is right."""
    from oracle import oracle_api
    from utree_b200 import capi
    t = tree_growth(ix_bytes)
    path, cpath = str(tmp_path / "grow.ctr"), str(tmp_path / "control.ctr")
    write_ctr(path, t.records, ix_bytes)
    write_ctr(cpath, tree_control(len(t.records), ix_bytes).records, ix_bytes)
    orc = oracle_api.OracleDb(path)
    ctr, cctr = capi.Ctr(path), capi.Ctr(cpath)
    try:
        sizes = []
        for c in (ctr, cctr):
            with _env({"UTB_SIEVE": "0"}):
                db = capi.Db(c, 0)
            assert db.lookup_mode() == 1
            sizes.append(db.hbm_bytes())
            db.free()
        assert sizes[0] - sizes[1] >= (1 << 21) * 32, sizes
        members = [word_with_hash(h) for h, _ in t.records]
        absent = [word_with_hash(h) for h in t.probes["around"]]
        want = _check_lookups(ctr, orc, np.array(members + absent, dtype=np.uint64))
        assert (want[:len(members)] == MISS).sum() <= 1 and np.all(want[len(members):] == MISS)   # <= 1: a folded first bin
        _check_search(path, orc, _reads_for(t, members, absent), tmp_path)
    finally:
        ctr.close(); cctr.close(); orc.free()


@pytest.mark.gpu
@pytest.mark.parametrize("ix_bytes", [2, 4])
def test_tree_whose_table_cannot_be_built_is_searched_on_the_probe_path(gpu_built, tmp_path, ix_bytes):
    """Case 6: a valid, regular CTR whose records no table size the loader tries can hold within KT_MAXD
    sectors.  It loads, on the reference probe sequence, and answers like the reference."""
    from oracle import oracle_api
    from utree_b200 import capi
    t = tree_unbuildable(ix_bytes)
    path = str(tmp_path / "crowded.ctr")
    write_ctr(path, t.records, ix_bytes)
    orc = oracle_api.OracleDb(path)
    ctr = capi.Ctr(path)
    try:
        members = [word_with_hash(h) for h, _ in t.records]
        absent = [word_with_hash(h) for h in t.probes["around"]]
        want = _check_lookups(ctr, orc, np.array(members + absent, dtype=np.uint64), mode=0)
        assert (want[:len(members)] == MISS).sum() <= 1 and np.all(want[len(members):] == MISS)   # <= 1: a folded first bin
        _check_search(path, orc, _reads_for(t, members, absent), tmp_path)
    finally:
        ctr.close(); orc.free()


# ---- the sieve on a tree of which every forward window of the reads is a member --------------------------------
def _dense_labels(rng, n):
    ranks = [b"k__", b"p__", b"c__", b"o__", b"f__", b"g__", b"s__", b"t__"]
    names = [b"A", b"Ab", b"Ab_c", b"B", b"", b"Zet", b"Zeta", b"Q_1", b"Q_12"]
    out = set()
    while len(out) < n:
        depth = int(rng.integers(1, 9))
        out.add(b";".join(ranks[d] + names[int(rng.integers(0, 2 if d < 2 else len(names)))] for d in range(depth)))
    return sorted(out)


def dense_reads(seed=41):
    """(reads, sources): the reads as searched, and the sequences whose forward windows the tree holds.
    Lengths 32..~1200 over every residue mod 32; N runs at every lane offset of a group; lower-case reads;
    palindromes (ACGT repeats, their own reverse complement); reads given only as the reverse complement of
    their source."""
    rng = np.random.default_rng(seed)

    def rand_seq(n):
        return bytes(_ACGT[rng.integers(0, 4, n)])
    reads, sources = [], []
    for r in range(32):
        for k in (0, 1, 4, 9, 17, 36):
            s = rand_seq(32 + r + 32 * k)
            reads.append(s); sources.append(s)
    for off in range(32):                        # an N run covering lane offset `off` of the read's second group
        s = bytearray(rand_seq(200 + 7 * off))
        run = 1 + off % 3
        s[32 + off:32 + off + run] = b"N" * run
        reads.append(bytes(s)); sources.append(bytes(s))
    for k in range(12):
        s = rand_seq(40 + 61 * k)
        reads.append(s.lower()); sources.append(s)
    for k in range(8):
        s = b"ACGT" * (8 + 5 * k) + b"ACGT"[:(k % 2) * 2]
        reads.append(s); sources.append(s)
    for k in range(24):
        s = rand_seq(33 + 47 * k)
        reads.append(revcomp(s)); sources.append(s)
    return reads, sources


def write_dense_tree(path, ix_bytes, seed=42):
    from tools import synth
    rng = np.random.default_rng(seed)
    reads, sources = dense_reads()
    labels = _dense_labels(rng, 40)
    words, ixs = {}, []
    for i, s in enumerate(sources):
        fam = int(rng.integers(0, len(labels)))
        for piece in s.upper().split(b"N"):
            for w in seq_words(piece).tolist():
                if w not in words:
                    words[w] = (fam + int(rng.integers(0, 3))) % len(labels)
    w = np.array(sorted(words), dtype=np.uint64)
    ix = np.array([words[x] for x in w.tolist()], dtype=np.uint64)
    synth.ctr_write(path, w, ix, synth._label_tail(labels, np.bincount(ix.astype(np.int64), minlength=len(labels))),
                    ix_bytes=ix_bytes)
    return reads


DENSE_REPS = 24                                  # > 148 SMs x 3 CTAs x 8 warps x 6 steps x 3 tiles of groups


@pytest.fixture(scope="module", params=[2, 4], ids=["ix2", "ix4"])
def dense(request, gpu_built, tmp_path_factory):
    """The dense tree, its reads once and DENSE_REPS times, and the checker's output and counts for one copy."""
    from oracle import oracle_api
    ix_bytes = request.param
    d = tmp_path_factory.mktemp("dense%d" % ix_bytes)
    path = str(d / "dense.ctr")
    reads = write_dense_tree(path, ix_bytes)
    one = fasta(reads, "d")
    groups = sum((len(r) + 1 + 31) // 32 for r in reads) * DENSE_REPS
    assert groups > 148 * 3 * 8 * 6 * 3
    open(d / "one.fa", "wb").write(one)
    open(d / "all.fa", "wb").write(one * DENSE_REPS)
    orc = oracle_api.OracleDb(path)
    want = {}
    for rc in (1, 0):
        code, st, err = orc.search_file(str(d / "one.fa"), str(d / ("want%d.out" % rc)), do_rc=bool(rc))
        assert code == 0, err
        want[rc] = (open(d / ("want%d.out" % rc), "rb").read(), st)
    yield {"path": path, "dir": d, "one": one, "want": want, "orc": orc, "ix_bytes": ix_bytes}
    orc.free()


def _dense_expect(dense, rc, reps=DENSE_REPS):
    text, st = dense["want"][rc]
    assert st["hits"] > st["lookups"] // (2 if rc else 1) * 8 // 10     # nearly every forward window is a member
    return text * reps, tuple(st[k] * reps for k in ("lookups", "hits", "good_finds"))


@pytest.mark.gpu
@pytest.mark.parametrize("env,reps", [({}, DENSE_REPS), ({"UTB_HOST_FRAME": "1"}, DENSE_REPS), ({}, 1),
                                      ({"UTB_HOST_FRAME": "1"}, 1), ({"UTB_BATCH_MB": "33"}, 0)],
                         ids=["device_frame", "host_frame", "device_frame_one_copy", "host_frame_one_copy", "batches"])
def test_dense_tree_sieve_has_no_false_negatives(dense, env, reps):
    """Sieve forced on.  The sieve kernel's grid follows the batch: persistent warps over several tiles each
    (DENSE_REPS copies of the reads), one tile per warp (one copy), and several batches of 33 MiB (reps 0: over
    100 MiB).  The group count it stops at comes from the device framer, or with UTB_HOST_FRAME=1 from the host.
    Both strands and forward only: the bytes and the lookups, hits and good finds counts equal the checker's."""
    from utree_b200 import capi
    reps = reps or 110 * 1024 * 1024 // len(dense["one"]) + 1
    ctr = capi.Ctr(dense["path"])
    with _env({"UTB_SIEVE": "1", **env}):
        s = capi.Searcher(ctr, devices=(0,), host_threads=3)
    try:
        for rc in (1, 0):
            text, counts = _dense_expect(dense, rc, reps)
            code, _, got, st = s.search_mem(dense["one"] * reps, do_rc=bool(rc))
            assert code == 0 and (st["lookups"], st["hits"], st["good_finds"]) == counts, rc
            assert got == text, rc
            assert st["batches"] >= (3 if "UTB_BATCH_MB" in env else 1)
    finally:
        s.destroy(); ctr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"UTB_SIEVE": "1", "UTB_QCAP": "128"}, {"UTB_SIEVE": "0"}],
                         ids=["qcap128", "sieve_off"])
def test_dense_tree_queue_overflow_and_strands(dense, env):
    from utree_b200 import capi
    ctr = capi.Ctr(dense["path"])
    with _env(env):
        s = capi.Searcher(ctr, devices=(0,), host_threads=3)
    try:
        for rc in (1, 0):
            text, counts = _dense_expect(dense, rc)
            code, _, got, st = s.search_mem(dense["one"] * DENSE_REPS, do_rc=bool(rc))
            assert code == 0 and (st["lookups"], st["hits"], st["good_finds"]) == counts, (env, rc)
            assert got == text, (env, rc)
    finally:
        s.destroy(); ctr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{}, {"UTB_SIEVE": "1"}, {"UTB_SIEVE": "1", "UTB_QCAP": "128"}], ids=["auto", "sieve", "qcap128"])
def test_dense_tree_non_gg_search(dense, tmp_path, env):
    """The non-GG search looks up the 24 corrupted words after each hit; on this tree every window hits."""
    from utree_b200 import capi
    fa, want = str(dense["dir"] / "all.fa"), str(tmp_path / "shallow.out")
    rc, ost, err = dense["orc"].search_file_shallow(fa, want, do_rc=True)
    assert rc == 0, err
    ctr = capi.Ctr(dense["path"])
    with _env(env):
        s = capi.Searcher(ctr, devices=(0,), host_threads=3)
    try:
        s.set_shallow(True)
        code, _, text, st = s.search_mem(open(fa, "rb").read(), do_rc=True)
        assert code == 0 and text == open(want, "rb").read()
        assert (st["good_finds"], st["reads"]) == (ost["good_finds"], ost["reads"])
    finally:
        s.destroy(); ctr.close()


@pytest.mark.gpu
def test_dense_tree_auto_sieve_switch_across_batches(dense):
    """UTB_BATCH_MB=33 and the default (auto) sieve: the hit rate of the first batches turns the sieve off for
    later ones, so one search mixes batches that resolve hits through per-read lists and batches with one slot
    per lookup.  Two stream slots, so that the third batch is submitted after the first one's counts are in.
    The bytes equal the checker's."""
    from utree_b200 import capi
    reps = 110 * 1024 * 1024 // len(dense["one"]) + 1
    text, st = dense["want"][1]
    ctr = capi.Ctr(dense["path"])
    with _env({"UTB_BATCH_MB": "33", "UTB_SLOTS": "2"}):
        s = capi.Searcher(ctr, devices=(0,), host_threads=4)
    try:
        code, _, got, st2 = s.search_mem(dense["one"] * reps, do_rc=True)
        assert code == 0 and st2["batches"] >= 3
        assert got == text * reps
        assert (st2["lookups"], st2["hits"]) == (st["lookups"] * reps, st["hits"] * reps)
    finally:
        s.destroy(); ctr.close()
