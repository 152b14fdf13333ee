"""The vote at its dispatch limits, against the CPU vote (oracle_api.OracleDb.vote, pinned by the reference's goldens).

Which of the five vote kernels votes a read, and how, depends on constants fixed in kernels.cu (mirrored below).  Every
test here sits on both sides of one of them, with real-size limits (no environment variable lowers them unless a test
says so), in the stage API (utb_vote_hits: warp -> block kernels; utb_vote_hits_sparse: thread -> warp -> block) and
through the whole search on trees built so that the pipeline's own hit lists land on the limits.

The walk cases put the byte that decides a neighbour comparison (itree.c:1060-1069) at every offset of an 8-byte word
(scan_token compares eight bytes at a time), in the first, second, fifth and ninth word (walk_warp scans 32 bytes per
ballot).  Two outcomes of the walk are out of reach of labels inside the contract (DESIGN.md 2:
distinct, non-empty, not starting with ';'), so no case claims them: itree.c:1052 (the first string of a pair ends
at the depth of the level) needs a label of the current run to end at dv, but every label of a run shares the token
that ends at dv (or continues past it); for the same reason a numeric cut is always shorter than the winning label.
"""
import contextlib
import os

import numpy as np
import pytest

import conftest  # noqa: F401  (puts the repo root on sys.path)

# ---- the limits (kernels.cu) ------------------------------------------------------------------------------------
VT_K = 6                      # VT_K: distinct labels vote_thread_kernel keeps in registers
VT_MAXHITS = 512              # VT_MAXHITS: entries vote_thread_kernel scans
VW_SLOTS = 64                 # VW_SLOTS: vote_warp_kernel's shared hash table (linear probe, wraps at slot 63)
VW_MAXHITS = 4096             # VW_MAXHITS: entries vote_warp_kernel scans
VL_CACHE = 64                 # VL_CACHE: vote_block_kernel's (label, count) cache; vl_add probes 4 slots, then `hist`
VL_PROBES = 4                 # vl_add's probes before it adds to `hist`
VB_SORT_MAX = 2048            # VB_SORT_MAX: touched labels sorted in shared memory; beyond: sweep in rank order
VL_STAGE_MAX = 512            # VL_STAGE_MAX: labels vl_stage copies to shared memory
VL_STR_BYTES = 24576          # VL_STR_BYTES: their strings; staged while bytes + 32 <= VL_STR_BYTES
SPLIT_SLOTS = 128 << 10       # vs_alloc: entries beyond which a read is split over the grid (vote_big_*)
VBIG_CHUNK = 32 * 2048        # VBIG_CHUNK_WORDS x 32: entries of a split read one CTA accumulates at a time
VBIG_POOL_MAX = 2048          # VBIG_POOL_MAX
HIT_MISS, HIT_NOWIN = 0xFFFFFFFF, 0xFFFFFFFE
CUT_EMPTY, CUT_FULL = 0xFFFFFFFF, 0xFFFFFFFE


def pool(max_ix):
    """Split reads one batch (or one utb_vote_hits call) votes over the grid; vs_alloc: 384 MiB of histograms."""
    return max(1, min(VBIG_POOL_MAX, (384 << 20) // (12 * max_ix)))


def slot(h):
    """Home slot of label h in vote_warp_kernel's table and in VL_CACHE: (h * 2654435761) >> 26 on 32 bits."""
    return ((int(h) * 2654435761) & 0xFFFFFFFF) >> 26


def staged_bytes(label):
    """Bytes vl_stage gives a label: its length with the NUL, rounded up to 8."""
    return (len(label) + 1 + 7) & ~7


def head_mis(start):
    """Entries before the first 16-byte boundary, which vote_warp_read loads one by one."""
    return (4 - (start & 3)) & 3


# ---- the walk, restated with a trace ----------------------------------------------------------------------------
def cutoff_of(x):
    c = x - x // 4
    return c + ((x >> 1) >= c)


def walk(T):
    """itree.c:1041-1098 over T = [(label, count)] sorted by label.  Returns ((winner index, cut, sl, ol), trace): per
    compared pair (branch, td, level, z, st) with branch S (1062), O_prefix / O_under (1063, first / second rule),
    E (1068, the walk stops before z) or D (1069)."""
    n = sum(c for _, c in T)
    S = [l + b"\0" * 1024 for l, _ in T]
    C = [c for _, c in T]
    cutoff, st, ed, dv, orun, level = cutoff_of(n), 0, len(T), CUT_EMPTY, n, 0
    trace = []
    while True:
        run, td = C[st], dv
        z = st + 1
        while z < ed:
            s1, s2 = S[z - 1], S[z]
            if s1[0 if dv == CUT_EMPTY else dv] == 0:                  # itree.c:1052 (out of contract, see above)
                trace.append(("K", dv, level, z, st))
                run, st = C[z], z
                orun -= C[z - 1]
                cutoff = cutoff_of(orun)
                z += 1
                continue
            td = 0 if dv == CUT_EMPTY else dv + 1
            while s1[td] and s1[td] == s2[td] and s1[td] != ord(";"):
                td += 1
            a, b = s1[td], s2[td]
            if a == b:
                trace.append(("S", td, level, z, st))
                run += C[z]
            elif (a == 0 and b == ord(";")) or ((a == ord(";") or a == 0) and td > 0 and s1[td - 1] == ord("_")):
                trace.append(("O_prefix" if a == 0 and b == ord(";") else "O_under", td, level, z, st))
                run, st = C[z], z
                orun -= C[z - 1]
                cutoff = cutoff_of(orun)
            elif run >= cutoff:
                trace.append(("E", td, level, z, st))
                ed = z
                break
            else:
                trace.append(("D", td, level, z, st))
                run, st = C[z], z
            z += 1
        sl, ol = run, orun
        if run < cutoff:
            break
        if st + 1 >= ed:
            if C[ed - 1] >= cutoff:
                dv = CUT_FULL
            break
        orun, dv, cutoff, level = run, td, cutoff_of(run), level + 1
    return (ed - 1, dv, sl, ol), trace


# ---- walk cases ---------------------------------------------------------------------------------------------------
POSITIONS = list(range(0, 16)) + list(range(32, 40)) + list(range(64, 72))   # words 0, 1, 4 and 8 of the label
BRANCHES = ("S", "O_prefix", "O_under", "E", "D")


def _fill(p, alpha=b"mnopqrstuvwxyzabcdefghijkl"):
    return (alpha * (p // len(alpha) + 1))[:p]


def _pair(branch, p):
    """Two labels (sorted) and their counts whose comparison at level 0 decides at byte p by `branch`; None where p is
    too short for it (a label cannot start with ';')."""
    P = _fill(p)
    G = _fill(p - 1) + b"_" if p >= 1 else None
    if branch == "S":
        return ([P + b";a", P + b";b"], [2, 1]) if p >= 1 else None
    if branch == "O_prefix":
        return ([P, P + b";x"], [2, 1]) if p >= 1 else None
    if branch == "O_under":                                      # the '_' rule, with a NUL and with a ';' at p
        return ([G, G + b"x"], [2, 1]) if p >= 1 else None
    if branch == "O_under;":
        return ([G + b";x", G + b"y"], [1, 2]) if p >= 1 else None
    if branch == "E":
        return [P + b"a", P + b"b"], [3, 1]
    if branch == "E0":                                           # E where the first string ends (a == NUL)
        return ([P, P + b"b"], [3, 1]) if p >= 1 else None
    if branch == "E;":                                           # E at a ';' without '_' before it
        return ([P + b";", P + b"b"], [3, 1]) if p >= 1 else None
    if branch == "D":
        return [P + b"a", P + b"b"], [1, 3]
    if branch == "D1":                                           # D, and the run ends below the cutoff: cut EMPTY
        return [P + b"a", P + b"b"], [1, 1]
    raise ValueError(branch)


def walk_cases():
    """[(labels, counts)]: each a read's labels (any order) with their counts.  Per branch and position: the pair at
    level 0, and under a shared first token of 1-7 bytes (level 1, whose scan starts at every offset of a word)."""
    cases = []
    kinds = ("S", "O_prefix", "O_under", "O_under;", "E", "E0", "E;", "D", "D1")
    for P in POSITIONS:
        for br in kinds:
            c = _pair(br, P)
            if c:
                cases.append(c)
            q = 1 + P % 7                                       # level 1: token of q bytes, ';', then the pair
            c = _pair(br, P - q - 1) if P - q - 1 >= 0 else None
            if c:
                H = _fill(q, b"KLMNOPQ") + b";"
                cases.append(([H + l for l in c[0]], c[1]))
    # deeper walks: a lineage with runs that shrink the outer run, labels stopping at every rank
    ranks = [b"k__Ba", b"p__Fi_", b"c__C", b"o__", b"f__Fam_ily", b"g__G", b"s__S_1"]
    lin = [b";".join(ranks[:d]) for d in range(1, len(ranks) + 1)]
    cases.append((lin, [1, 1, 2, 3, 5, 8, 13]))
    cases.append((lin + [lin[3] + b"x", lin[5] + b"2"], [1, 1, 1, 1, 1, 9, 30, 1, 4]))
    cases.append(([lin[-1]], [5]))                              # one label: "*"
    return cases


def _walk_labels():
    out = set()
    for labels, _ in walk_cases():
        out.update(labels)
    return sorted(out)


# ---- label sets of the trees -------------------------------------------------------------------------------------
def x_labels(n=600):
    """Neighbours in rank order that differ inside their only token: every pair between two of them is D or E."""
    return [b"x%04d" % i for i in range(n)]


def xs_labels():
    """x%04d;a / x%04d;b: an S pair before the x labels that follow."""
    return [b"x%04d;%s" % (i, t) for i in (5, 40, 70) for t in (b"a", b"b")]


def w_labels():
    """w;%03d: one token shared by 40 labels, so a run of S pairs crosses the staged walk's first 32-pair step."""
    return [b"w;%03d" % i for i in range(40)]


def staged_labels():
    """m labels of 256 staged bytes each, l labels of 8k staged bytes (k = 1..64)."""
    m = [(b"m%04d" % i + b"z" * 251)[:255] for i in range(100)]
    l = [(b"l%03d" % k + b"y" * 512)[:8 * k - 1] for k in range(1, 65)]
    return m, l


def filler_labels(rng, n):
    ranks = [b"k__", b"p__", b"c__", b"o__", b"f__", b"g__", b"s__", b"t__"]
    names = [b"A", b"Ab", b"Ab_c", b"B", b"", b"Zet", b"Zeta", b"Q_1", b"Q_12", b"Vibrio", b"Pseudomonas_a"]
    out = set()
    while len(out) < n:
        depth = int(rng.integers(1, 9))
        out.add(b";".join(ranks[d] + names[int(rng.integers(0, 2 if d < 2 else len(names)))] +
                          (b"%d" % rng.integers(0, 40) if d >= 3 else b"") for d in range(depth)))
    return sorted(out)


def small_tree_labels(seed=3):
    """About 3000 labels: the walk cases', the x / xs / staged families and taxonomy-like fillers."""
    m, l = staged_labels()
    base = set(_walk_labels()) | set(x_labels()) | set(xs_labels()) | set(w_labels()) | set(m) | set(l)
    rng = np.random.default_rng(seed)
    fill = [f for f in filler_labels(rng, 3000 - len(base) + 200) if f not in base][:max(0, 3000 - len(base))]
    labels = sorted(base | set(fill))
    return [labels[i] for i in rng.permutation(len(labels))]     # ids in no particular rank order


def big_tree_labels(n=200_000):
    return [b"k__B;p__P%d;c__C%d;g__G%d;s__S%06d" % (i % 7, i % 97, i % 1009, i) for i in range(n)]


# ---- hit lists on the limits ---------------------------------------------------------------------------------------
class Lists:
    def __init__(self):
        self.tags, self.lists = [], []

    def add(self, tag, ids, counts=None, rng=None):
        h = np.repeat(np.asarray(ids, dtype=np.uint32), counts) if counts is not None else np.asarray(ids, dtype=np.uint32)
        if rng is not None:
            h = rng.permutation(h)
        self.tags.append(tag)
        self.lists.append(h.astype(np.uint32))

    def total(self):
        return sum(x.size for x in self.lists)

    def offsets(self):
        off = np.zeros(len(self.lists) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([x.size for x in self.lists])
        return off


def _lineage(rng, by_rank, k):
    """k labels next to each other in rank order (a lineage), counts 1-3 and a few heavy ones."""
    a = int(rng.integers(0, len(by_rank) - k + 1))
    ids = by_rank[a:a + k]
    cnt = rng.integers(1, 4, k)
    cnt[rng.integers(0, k, max(1, k // 8))] += rng.integers(2, 12)
    return ids, cnt


def _with_entries(rng, ids, n):
    """n entries over the labels ids, each at least once."""
    ids = np.asarray(ids)
    h = np.concatenate([ids, ids[rng.integers(0, ids.size, n - ids.size)]])
    return rng.permutation(h)


def misses(rng, max_ix, n):
    pool_ = np.array([HIT_MISS, HIT_NOWIN, max_ix, max_ix + 1, 0xFFFF, 0x10000, HIT_NOWIN - 1], dtype=np.uint64)
    v = pool_[rng.integers(0, pool_.size, n)]
    v = v[(v >= max_ix)]
    return v.astype(np.uint32)


def sprinkle(rng, h, max_ix, frac=0.5):
    """h with misses inserted between its hits (HIT_MISS, HIT_NOWIN and ids in [max_ix, HIT_NOWIN))."""
    m = misses(rng, max_ix, max(1, int(h.size * frac)) + 3)
    out = np.concatenate([h, m])
    pos = np.concatenate([np.arange(h.size) * 2 + 1, rng.integers(0, 2 * h.size + 2, m.size)])
    return out[np.argsort(pos, kind="stable")].astype(np.uint32)


def stage_lists(labels, rng, big_split=True):
    """The lists of the stage-level test on a tree with these labels (ids = positions)."""
    M = len(labels)
    by_rank = np.array(sorted(range(M), key=lambda i: labels[i]), dtype=np.uint32)
    idx = {l: i for i, l in enumerate(labels)}
    L = Lists()
    # distinct labels
    for k in (VT_K, VT_K + 1, VW_SLOTS, VW_SLOTS + 1, VL_STAGE_MAX, VL_STAGE_MAX + 1, VB_SORT_MAX, VB_SORT_MAX + 1):
        for rep in range(2):
            ids, cnt = _lineage(rng, by_rank, k)
            if k >= VB_SORT_MAX:
                cnt = np.minimum(cnt, 2 if rep else 1)
            L.add("labels%d" % k, ids, cnt, rng)
            assert np.unique(L.lists[-1]).size == k
    # entries
    for n in (VT_MAXHITS, VT_MAXHITS + 1, VW_MAXHITS, VW_MAXHITS + 1):
        ids, _ = _lineage(rng, by_rank, 3)
        L.add("entries%d" % n, _with_entries(rng, ids, n))
    if big_split:
        for k in (2, 3):
            for n in (VBIG_CHUNK * k - 1, VBIG_CHUNK * k, VBIG_CHUNK * k + 1):
                ids, _ = _lineage(rng, by_rank, 4)
                L.add("entries%d" % n, _with_entries(rng, ids, n))
    # vote_warp_kernel's table: 64 labels homed in the top 8 slots fill it and wrap; 65 overflow it
    top = np.array([i for i in range(M) if slot(i) >= 56], dtype=np.uint32)
    for k in (VW_SLOTS, VW_SLOTS + 1):
        ids = rng.choice(top, k, replace=False)
        L.add("wrap%d" % k, ids, rng.integers(1, 5, k), rng)
    # VL_CACHE: 8 labels of one home slot in every warp's 32 entries (4 probes hold 4 of them), > VW_MAXHITS entries
    s = int(rng.integers(0, 64))
    same = np.array([i for i in range(M) if slot(i) == s][:2 * VL_PROBES], dtype=np.uint32)
    L.add("cache", np.tile(same, 600))
    ids, cnt = _lineage(rng, by_rank, 70)
    L.add("cache+70", np.concatenate([np.tile(same, 300), np.repeat(ids, cnt)]))
    # staged bytes: 24,544 (staged) and 24,552 (walk_warp from global memory)
    if b"m0000" + b"z" * 250 in idx:
        m, l = staged_labels()
        for total in (VL_STR_BYTES - 32, VL_STR_BYTES - 24):
            ids = [idx[x] for x in m[:95]] + [idx[l[(total - 95 * 256) // 8 - 1]]]
            assert sum(staged_bytes(labels[i]) for i in ids) == total
            L.add("staged%d" % total, ids, rng.integers(1, 6, len(ids)), rng)
        # walk_warp_staged ends its run at lane 0, lane 31, the first pair of the second step; with the run exactly
        # at the cutoff (`>=`) and one above; after an S pair (the run's start stays below the breaking lane)
        xs = [idx[x] for x in x_labels()]
        for j in (0, 31, 32):
            for exact in (True, False):
                ids = xs[j * 3:j * 3 + 100]
                cnt = np.ones(100, dtype=np.int64)
                cnt[j] = heavy_for(99, exact)
                L.add("lane%d%s" % (j, "=" if exact else ">"), ids, cnt, rng)
        for i, first in ((5, 6), (40, 41), (70, 71)):
            for exact in (True, False):
                ids = [idx[b"x%04d;a" % i], idx[b"x%04d;b" % i]] + xs[first:first + 85]
                h = heavy_for(85, exact)
                cnt = np.array([h - h // 2, h // 2] + [1] * 85)
                L.add("s_then_e%d%s" % (i, "=" if exact else ">"), ids, cnt, rng)
        # a run of S pairs from the first step into the second, ended there by E with no run start before its lane
        ids = [idx[x] for x in w_labels()] + xs[:40]
        L.add("cross", ids, [5] * 40 + [1] * 40, rng)
        # the walk cases: dense -> walk_warp, sparse -> walk_thread, counts x 1500 -> vote_block_kernel, staged walk
        for labels_, cnt in walk_cases():
            ids = [idx[x] for x in labels_]
            L.add("walk", ids, cnt, rng)
            L.add("walk_x1500", ids, np.array(cnt) * 1500, rng)
    # every read at all four alignments of its first entry, with counts around the warp kernel's 128-entry rounds
    for a in range(4):
        for k in (1, 2, 31):
            for d in (-1, 0, 1):
                pad = (a - L.total()) % 4
                if pad:
                    L.add("pad", np.full(pad, HIT_MISS, np.uint32))
                assert L.total() % 4 == a
                n = 128 * k + head_mis(a) + d
                ids, _ = _lineage(rng, by_rank, 3)
                L.add("align%d_%d" % (a, n), _with_entries(rng, ids, n))
    # misses mixed in, and reads with entries but no hit, in every size class
    for i in range(0, len(L.lists), 3):
        if L.lists[i].size <= 5000 and L.tags[i] != "pad":
            L.add(L.tags[i] + "+misses", sprinkle(rng, L.lists[i], M))
    for n in (1, VT_MAXHITS, VT_MAXHITS + 1, VW_MAXHITS, VW_MAXHITS + 1) + ((SPLIT_SLOTS + 1,) if big_split else ()):
        L.add("nohit%d" % n, np.resize(misses(rng, M, 4096), n))
    L.add("empty", [])
    return L


def heavy_for(rest, exact):
    """The least count C of one label, beside `rest` others of count 1, whose run reaches the cutoff of the whole:
    C == cutoff_of(C + rest) when `exact`, C > cutoff_of(C + rest) otherwise."""
    for c in range(1, 100 * rest):
        if (c == cutoff_of(c + rest)) if exact else (c > cutoff_of(c + rest)):
            return c
    raise AssertionError(rest)


# ---- trees ---------------------------------------------------------------------------------------------------------
def write_tree(path, labels, words, ixs, ix_bytes):
    from tools import synth
    order = np.argsort(words)
    words, ixs = np.asarray(words, dtype=np.uint64)[order], np.asarray(ixs)[order]
    assert np.all(words[1:] > words[:-1])
    counts = np.bincount(ixs.astype(np.int64), minlength=len(labels))
    synth.ctr_write(path, words, ixs, synth._label_tail(labels, counts), ix_bytes=ix_bytes)


_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def read_words(codes):
    from tools import synth
    return synth.kmer_words(codes)


def search_reads(rng, by_rank, M, n_windows_list):
    """[(name, seq, window labels)]: random reads whose forward windows get the given labels."""
    out = []
    for name, nw, k in n_windows_list:
        codes = rng.integers(0, 4, nw + 31).astype(np.uint8)
        a = int(rng.integers(0, M - k + 1))
        lab = np.asarray(by_rank[a:a + k])
        w = np.concatenate([np.arange(k), rng.integers(0, k, nw - k)]) if nw >= k else rng.integers(0, k, nw)
        skew = rng.integers(0, k, max(1, nw // 3))
        w[rng.integers(k if nw > k else 0, nw, skew.size)] = skew[0]             # one label ahead of the others
        out.append((name, codes, lab[rng.permutation(w)]))
    return out


def build_search_tree(path, labels, reads, ix_bytes, rng):
    """The reads' forward windows with their chosen labels, plus one random word for every other label.  Word 0 is
    the lowest bin's only record, which the reference's compressor folds away (synth.binix_like_reference)."""
    words = {0: 0}
    for _, codes, lab in reads:
        for w, l in zip(read_words(codes).tolist(), lab.tolist()):
            words.setdefault(w, l)
    have = set(words.values())
    for i in range(len(labels)):
        if i not in have:
            w = int(rng.integers(0, 2 ** 63)) * 2 + 1
            while w in words:
                w += 2
            words[w] = i
    w = np.fromiter(words.keys(), dtype=np.uint64, count=len(words))
    ix = np.fromiter(words.values(), dtype=np.uint64, count=len(words))
    write_tree(path, labels, w, ix, ix_bytes)


SMALL_READS = [("lab6", 300, 6), ("lab7", 300, 7), ("lab64", 900, 64), ("lab65", 900, 65),
               ("hits256", 256, 3), ("hits257", 257, 3), ("hits512", 512, 3), ("hits513", 513, 3),
               ("hits2048", 2048, 4), ("hits2049", 2049, 4), ("hits4096", 4096, 4), ("hits4097", 4097, 4),
               ("lab2049", 2049 * 2, 2049), ("hits65536", 65536, 5), ("hits65537", 65537, 5),
               ("hits131072", 131072, 5), ("hits131073", 131073, 5)]


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


# ---- CPU: the cases produce what they claim ---------------------------------------------------------------------
@pytest.fixture(scope="module")
def small(built, tmp_path_factory):
    """The ~3000-label uint16 tree: the walk cases' labels among others; its words are the search reads' windows."""
    from oracle import oracle_api
    d = tmp_path_factory.mktemp("small")
    rng = np.random.default_rng(11)
    labels = small_tree_labels()
    by_rank = sorted(range(len(labels)), key=lambda i: labels[i])
    reads = search_reads(rng, by_rank, len(labels), SMALL_READS)
    path = str(d / "small.ctr")
    build_search_tree(path, labels, reads, 2, rng)
    orc = oracle_api.OracleDb(path)
    assert orc.max_ix == len(labels)
    yield {"path": path, "labels": labels, "reads": reads, "orc": orc, "dir": d}
    orc.free()


def test_pool_of_each_tree():
    assert pool(200_000) == 167 and pool(3000) == VBIG_POOL_MAX and pool(73_000) == 459 and pool(900) == VBIG_POOL_MAX
    assert pool(33_000) < VBIG_POOL_MAX


def test_walk_cases_cover_every_branch_offset_and_cut(small):
    """The restated walk equals the CPU vote on every case, and the cases put the deciding byte of every branch at
    every offset of the first, second, fifth and ninth 8-byte word; all kinds and special cuts occur."""
    orc, labels = small["orc"], small["labels"]
    idx = {l: i for i, l in enumerate(labels)}
    seen, kinds, cuts = set(), set(), set()
    rng = np.random.default_rng(1)
    for labs, cnt in walk_cases() + [([labels[0]], [0])]:
        h = np.repeat([idx[x] for x in labs], cnt).astype(np.uint32)
        v = orc.vote(rng.permutation(h))
        kinds.add(v.kind)
        if v.kind != 2:
            continue
        T = sorted(zip(labs, cnt))
        (win, cut, sl, ol), trace = walk(T)
        assert (v.label, v.cut, v.sl, v.ol, v.uix, v.found) == (idx[T[win][0]], cut, sl, ol, len(T), sum(cnt)), labs
        for br, td, level, z, st in trace:
            seen.add((br, td))
            if br == "O_under" and td % 8 == 0:
                seen.add(("_ ends the previous word", td // 8))
        cuts.add("empty" if cut == CUT_EMPTY else "full" if cut == CUT_FULL else "numeric")
        if cut < CUT_FULL:
            assert cut < len(T[win][0])
    for br in BRANCHES:
        for p in POSITIONS:
            if p == 0 and br in ("S", "O_prefix", "O_under"):
                continue                                          # a label cannot start with ';' or be empty
            assert (br, p) in seen, (br, p)
    assert {("_ ends the previous word", w) for w in (1, 4, 8)} <= seen
    assert not any(b == "K" for b, _ in seen)
    assert kinds == {0, 1, 2} and cuts == {"empty", "full", "numeric"}
    assert {len(l) % 8 for l in _walk_labels()} == set(range(8))


def test_stage_lists_sit_on_the_limits(small):
    """What each stage-level list claims: distinct labels, entries, slots, staged bytes, the lane the staged walk
    stops at, the alignment of its first entry."""
    labels = small["labels"]
    L = stage_lists(labels, np.random.default_rng(5))
    off = L.offsets()
    M = len(labels)
    seen = set()
    for tag, h, start in zip(L.tags, L.lists, off[:-1].tolist()):
        hits = h[h < M]
        if tag.endswith("+misses"):
            assert 0 < hits.size < h.size
            seen.add("misses")
        elif tag.startswith("labels"):
            assert np.unique(hits).size == int(tag[6:])
        elif tag.startswith("entries"):
            assert h.size == int(tag[7:]) and hits.size == h.size
        elif tag.startswith("wrap"):
            u = np.unique(hits)
            assert u.size == int(tag[4:]) and all(slot(i) >= 56 for i in u)
        elif tag == "cache":
            assert len({slot(i) for i in hits}) == 1 and np.unique(hits[:32]).size == 8 and h.size > VW_MAXHITS
        elif tag.startswith("staged"):
            u = np.unique(hits)
            assert sum(staged_bytes(labels[i]) for i in u) == int(tag[6:]) and VW_SLOTS < u.size <= VL_STAGE_MAX
        elif tag.startswith("align"):
            a, n = (int(x) for x in tag[5:].split("_"))
            assert start % 4 == a and h.size == n
            seen.add((a, n - head_mis(a)))
        elif tag.startswith("lane") or tag.startswith("s_then_e"):
            u, c = np.unique(hits, return_counts=True)
            T = sorted((labels[i], int(k)) for i, k in zip(u, c))
            assert VW_SLOTS < len(T) <= VL_STAGE_MAX
            _, trace = walk(T)
            e = [t for t in trace if t[0] == "E" and t[2] == 0]
            assert len(e) == 1
            _, _, _, z, st = e[0]
            run = sum(k for _, k in T[st:z])
            cut = cutoff_of(sum(k for _, k in T))
            assert (run == cut) == tag.endswith("=") and run >= cut
            if tag.startswith("lane"):
                j = int(tag[4:-1])
                assert z - 1 == j and ((z - 1) % 32, (z - 1) // 32) == (j % 32, j // 32)
            else:
                assert st == 0 and z == 2                        # the S pair, then E at lane 1
            seen.add(tag)
        elif tag == "cross":
            u, c = np.unique(hits, return_counts=True)
            _, trace = walk(sorted((labels[i], int(k)) for i, k in zip(u, c)))
            e = [t for t in trace if t[0] == "E" and t[2] == 0]
            assert len(e) == 1 and e[0][3:] == (40, 0) and VW_SLOTS < u.size   # pair 39: lane 7 of the second step
            seen.add(tag)
        elif tag.startswith("nohit"):
            assert hits.size == 0 and h.size == int(tag[5:])
    assert {(a, 128 * k + d) for a in range(4) for k in (1, 2, 31) for d in (-1, 0, 1)} <= seen
    assert {"lane%d%s" % (j, e) for j in (0, 31, 32) for e in "=>"} <= seen
    assert "misses" in seen and "cross" in seen


# ---- GPU: stage level ---------------------------------------------------------------------------------------------
def _check(db, orc, L, sparse, what):
    res = db.vote_hits(np.concatenate(L.lists) if L.lists else np.zeros(0, np.uint32), L.offsets(), sparse=sparse)
    M = orc.max_ix
    bad = []
    cache = {}
    for i, (tag, h) in enumerate(zip(L.tags, L.lists)):
        key = id(h)
        if key not in cache:
            cache[key] = orc.vote(h[h < M])
        v = cache[key]
        r = res[i]
        want = (v.kind, v.label, v.found, v.uix) + ((v.cut, v.sl, v.ol) if v.kind == 2 else ())
        got = (int(r["kind"]), int(r["label"]), int(r["found"]), int(r["uix"])) + ((int(r["cut"]), int(r["sl"]), int(r["ol"])) if v.kind == 2 else ())
        if v.kind == 0:
            want, got = want[:1], got[:1]
        if want != got:
            bad.append((what, sparse, i, tag, got, want))
    assert not bad, bad[:10]


@pytest.fixture(scope="module")
def big(built, tmp_path_factory):
    """The uint32 tree of 200,000 labels (pool 167); its words are one read's 131,073 windows and a word per label."""
    from oracle import oracle_api
    d = tmp_path_factory.mktemp("big")
    rng = np.random.default_rng(12)
    labels = big_tree_labels()
    by_rank = sorted(range(len(labels)), key=lambda i: labels[i])
    reads = search_reads(rng, by_rank, len(labels), [("split", SPLIT_SLOTS + 1, 40)])
    path = str(d / "big.ctr")
    build_search_tree(path, labels, reads, 4, rng)
    orc = oracle_api.OracleDb(path)
    assert orc.max_ix == len(labels) and pool(orc.max_ix) == 167
    yield {"path": path, "labels": labels, "reads": reads, "orc": orc, "dir": d, "by_rank": by_rank}
    orc.free()


@pytest.mark.gpu
@pytest.mark.parametrize("tree", ["small", "big"])
def test_stage_limits_match_the_cpu_vote(request, tree):
    """Both stage APIs on every list of stage_lists, at the real limits."""
    from utree_b200 import capi
    t = request.getfixturevalue(tree)
    L = stage_lists(t["labels"], np.random.default_rng(5 if tree == "small" else 6), big_split=True)
    ctr = capi.Ctr(t["path"])
    db = capi.Db(ctr, 0)
    try:
        for sparse in (False, True):
            _check(db, t["orc"], L, sparse, tree)
    finally:
        db.free(); ctr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("split", [None, 300])
def test_split_pool_overflow(big, split):
    """pool - 1, pool, pool + 1 and 2 pool reads over the split threshold in one call, among short reads: those the
    pool holds are voted over the grid, the others by one CTA each.  At the default threshold (131,073 entries each)
    and with UTB_VOTE_SPLIT_SLOTS=300."""
    from utree_b200 import capi
    rng = np.random.default_rng(21)
    by_rank, M = big["by_rank"], len(big["labels"])
    P = pool(M)
    n = (split or SPLIT_SLOTS) + 1
    variants = []
    for k in (3, 40, 70, 600):
        ids, _ = _lineage(rng, by_rank, min(k, n // 2))
        variants.append(_with_entries(rng, ids, n))
    variants.append(np.resize(misses(rng, M, 4096), n))          # qualifies, hits nothing
    short = stage_lists(big["labels"], np.random.default_rng(7), big_split=False)
    ctr = capi.Ctr(big["path"])
    db = capi.Db(ctr, 0)
    try:
        for q in (P - 1, P, P + 1, 2 * P):
            L = Lists()
            for i in range(q):
                L.tags.append("split%d" % (i % len(variants)))
                L.lists.append(variants[i % len(variants)])
                j = int(rng.integers(0, len(short.lists)))
                L.tags.append(short.tags[j]); L.lists.append(short.lists[j])
            with _env({"UTB_VOTE_SPLIT_SLOTS": str(split)} if split else {}):
                for sparse in (False, True):
                    _check(db, big["orc"], L, sparse, "pool%d" % q)
    finally:
        db.free(); ctr.close()


# ---- GPU: through the search --------------------------------------------------------------------------------------
def _fasta(reads, reps=1):
    one = b"".join(b">%s\n%s\n" % (name.encode(), _ACGT[codes].tobytes()) for name, codes, _ in reads)
    return one * reps


def test_search_reads_sit_on_the_limits(small):
    """Per read, the CPU slide's hits and distinct labels (forward strand; the reverse strand hits nothing): the
    sieve path votes over the hits, the sieve-off path over (len - 31) x strands slots."""
    orc = small["orc"]
    for (name, codes, lab), (_, nw, k) in zip(small["reads"], SMALL_READS):
        seq = _ACGT[codes].tobytes()
        h, _ = orc.slide(seq, do_rc=True)
        assert h.size == nw and np.unique(h).size == k, name
    slots = {name: [(nw) * s for s in (1, 2)] for name, nw, _ in SMALL_READS}
    for lim in (VT_MAXHITS, VW_MAXHITS, SPLIT_SLOTS):              # both sides of every entry limit, both strand counts
        for s in (0, 1):
            assert any(v[s] == lim for v in slots.values()) and any(v[s] in (lim + 1, lim + 2) for v in slots.values())


@pytest.mark.gpu
@pytest.mark.parametrize("sieve", ["1", "0"])
@pytest.mark.parametrize("rc", [1, 0])
def test_search_on_the_limits_matches_the_checker(small, sieve, rc):
    from utree_b200 import capi
    d = small["dir"]
    fa, want = str(d / "reads.fa"), str(d / ("want%d.out" % rc))
    open(fa, "wb").write(_fasta(small["reads"]))
    code, ost, err = small["orc"].search_file(fa, want, do_rc=bool(rc), threads=4)
    assert code == 0, err
    ctr = capi.Ctr(small["path"])
    with _env({"UTB_SIEVE": sieve}):
        s = capi.Searcher(ctr, devices=(0,), host_threads=2)
    try:
        code, _, text, st = s.search_mem(open(fa, "rb").read(), do_rc=bool(rc))
        assert code == 0
        assert text == open(want, "rb").read()
        assert (st["good_finds"], st["hits"], st["lookups"]) == (ost["good_finds"], ost["hits"], ost["lookups"])
    finally:
        s.destroy(); ctr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("sieve", ["1", "0"])
@pytest.mark.parametrize("rc", [1, 0])
def test_search_more_split_reads_than_the_pool(big, sieve, rc):
    """One read of 131,073 hits, 2 pool + 3 times, in the 200k-label tree.  A search's first batch is 32 MiB: it holds
    more of them than the pool (the pool's reads split over the grid, the rest voted by one CTA each), the second
    batch fewer.  Identical reads give identical lines."""
    from utree_b200 import capi
    d = big["dir"]
    reps = 2 * pool(big["orc"].max_ix) + 3
    fa, want = str(d / "one.fa"), str(d / ("one%d.out" % rc))
    open(fa, "wb").write(_fasta(big["reads"]))
    code, ost, err = big["orc"].search_file(fa, want, do_rc=bool(rc), threads=2)
    assert code == 0 and ost["good_finds"] == 1, err
    ctr = capi.Ctr(big["path"])
    with _env({"UTB_SIEVE": sieve}):
        s = capi.Searcher(ctr, devices=(0,), host_threads=2)
    try:
        code, _, text, st = s.search_mem(_fasta(big["reads"], reps), do_rc=bool(rc))
        per_batch = (32 << 20) // len(_fasta(big["reads"]))
        assert per_batch > pool(big["orc"].max_ix) > reps - per_batch
        assert code == 0 and st["batches"] == 2
        assert text == open(want, "rb").read() * reps
        assert (st["good_finds"], st["hits"], st["lookups"]) == tuple(ost[k] * reps for k in ("good_finds", "hits", "lookups"))
    finally:
        s.destroy(); ctr.close()
