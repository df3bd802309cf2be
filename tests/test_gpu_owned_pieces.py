"""The owner-restricted count over a sequence in pieces, every rank of a G-GPU box emulated on one device.

Every multi-GPU count ends in count_owned (csrc/dnagpu.cu): each GPU wraps the whole sequence as base-range pieces
(dnagpu_seq_wrap_pieces, its own piece first and the others in ring order) and keeps the k-mers owner_of assigns to
it.  Two kernels collect them: k_collect_owned<WPT, LIN, MASKLO> stages one tile of 256 * WPT words of one piece per
CTA (the pieces are padded to whole tiles in the walk order), and k_collect_owned_any walks the pieces item by item
(the exact fallback, and the only collector under DNAGPU_COUNT_FLAG_EXACT).  Around them, up to three attempts: a
list longer than its guess is collected again with the exact size, a tile whose shared-memory list overflowed drops
keys and the exact kernel takes over with a generous guess, and if that guess is short too it runs once more.

Here the G pieces sit in one device allocation the way ShardRing and count_kmers_multi cut and size them, each
followed by a poison pattern, so that a read past a piece's zero pad word changes the answer.  For each rank d the
pieces are wrapped in d's walk order and counted with owner=(G, d); the union is compared with the CPU oracle (rows up
to ~3 M bases, the order-free digest above), every returned row must belong to d, and the shares must be disjoint.
The collect attempts are asserted from the per-launch profile against a model of the tiles and warps."""
import collections
import functools

import numpy as np
import pytest
import torch

import dnagpu
from dnagpu import Dna, DnaError
from dnagpu.distributed import ring_shards, shard_words
from dnagpu.types import pack_bases, unpack_bases
from oracle import ref_cpu as R

pytestmark = pytest.mark.gpu

EARG = 20
H = 16                      # spectrum bins: counts 1..15 and "16 or more"
ROWS_MAX = 3_000_000        # oracle rows up to this many bases, the digest above
POISON = np.uint64(0xA5C396E1F00D5EED)
N_POISON = 4                # poison words after every piece (keeps the next piece at an even word offset)

# owner_of (csrc/kernels.cuh): the GF(2)-linear form for 2 / 4 / 8 owners, the multiplicative form otherwise
OWNER_MUL = 0x85EBCA6B
OWN_TAU = (0, 3, 6, 9, 13, 16, 19, 22, 26, 29)
OWN_SUB = (0x06E, 0x2D1, 0x1B4)
OWN_TAPS = tuple(sum(1 << OWN_TAU[p] for p in range(len(OWN_TAU)) if sub >> p & 1) for sub in OWN_SUB)
MUL_GS = (3, 5, 6, 7, 9, 16, 17, 31, 32, 33, 63, 64)     # the multiplicative owner counts used below

# k_collect_owned (csrc/partition.cuh): 256 threads, a warp's list of 576 codes, 512 shared overflow slots
OWN_THREADS, OWN_SEG, OWN_OVF = 256, 576, 512


def owner_np(kmers, G):
    """owner_of for an array of k-mers: a function of the k-mer's low 32 bits"""
    x = (np.asarray(kmers, dtype=np.uint64) & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    lin = {2: 1, 4: 2, 8: 3}.get(G, 0)
    if lin:
        r = np.zeros(x.shape, dtype=np.uint32)
        for i in range(lin):
            r |= (np.bitwise_count(x & np.uint32(OWN_TAPS[i])).astype(np.uint32) & np.uint32(1)) << np.uint32(i)
        return r
    h = (x.astype(np.uint64) * np.uint64(OWNER_MUL)) & np.uint64(0xFFFFFFFF)
    return ((h * np.uint64(G)) >> np.uint64(32)).astype(np.uint32)


def wpt_of(G):
    """words per thread of k_collect_owned: a tile is 256 * WPT words = 8192 * WPT starts"""
    return 4 if G >= 8 else 2 if G >= 4 else 1


def boundary_words(rng):
    """One 64-bit word per edge of every owner's hash range of the multiplicative form: its low half hashes to
    ceil(r 2^32 / G) (owned by r) or one less (owned by r - 1).  The k-mer that starts at such a word (k >= 16) sits
    on the edge, where a range computed with floor instead of ceil gives it to the wrong owner."""
    inv = pow(OWNER_MUL, -1, 1 << 32)
    lows = []
    for G in MUL_GS:
        for r in range(1, G):
            h0 = ((r << 32) + G - 1) // G
            lows += [h0 * inv % (1 << 32), (h0 - 1) * inv % (1 << 32)]
    high = rng.integers(0, 1 << 32, size=len(lows), dtype=np.uint64)
    return (high << np.uint64(32)) | np.array(lows, dtype=np.uint64)


@functools.lru_cache(maxsize=None)
def seq_words(seed, n):
    """The synthetic sequence of (seed, n) with edge-of-range k-mers near its start and, at every piece cut that
    ring_shards makes for 2 .. 16 owners, 'G' x 48 (k = 32: the side counter's key) or 'A' x 80 across the cut."""
    words = R.synth_seq(seed, n)
    rng = np.random.default_rng(seed)
    if n >= 64 * 64:
        edge = boundary_words(rng)
        at = 64 + 2 * np.arange(edge.size)
        keep = at < (n - 64) // 32
        words[at[keep]] = edge[keep]
    if n >= 4096:
        codes = unpack_bases(words, n).copy()
        for G in (2, 3, 4, 5, 8, 16):
            for first, _ in ring_shards(n, G)[1:]:
                if 48 <= first < n - 48:
                    if G in (3, 5):
                        codes[first - 40:first + 40] = 0         # A
                    else:
                        codes[first - 24:first + 24] = 3         # G
        words = pack_bases(codes)
    words.flags.writeable = False
    return words


@functools.lru_cache(maxsize=None)
def oracle(seed, n, k):
    return oracle_of(seq_words(seed, n), n, k)


def oracle_of(words, n, k):
    if n <= ROWS_MAX:
        return R.count_query(words, 1, n, words.size, k, faithful=False, threads=8)
    return R.count_query_big(words, 1, n, words.size, k, threads=8)


def ref_hist(counts, h=H):
    counts = np.asarray(counts, dtype=np.uint64)
    return np.bincount(np.minimum(counts, np.uint64(h)).astype(np.int64), minlength=h + 1)[1:].astype(np.uint64)


class Pieces:
    """The base ranges `shards` ([(first_base, n_starts)]) of a packed sequence in ONE device allocation, piece i
    at an even word offset with shard_words words (its bases, the 31-base overlap, zero pad words) followed by
    N_POISON words of POISON."""

    def __init__(self, words, n, shards):
        self.n, self.shards = n, list(shards)
        sizes = [shard_words(n, f, s) for f, s in self.shards]
        self.offs = list(np.cumsum([0] + [s + N_POISON for s in sizes[:-1]]))
        buf = np.full(self.offs[-1] + sizes[-1] + N_POISON, POISON, dtype=np.uint64)
        for (f, s), o, size in zip(self.shards, self.offs, sizes):
            held = (max(0, min(n, f + s + 31) - f) + 31) // 32
            buf[o:o + size] = 0
            buf[o:o + held] = words[f // 32:f // 32 + held]
        assert all(o % 2 == 0 for o in self.offs)
        self.dev = torch.from_numpy(buf.view(np.int64)).cuda()
        torch.cuda.synchronize()

    def wrap(self, gpu, order):
        base = self.dev.data_ptr()
        return gpu.wrap_pieces([base + 8 * int(self.offs[i]) for i in order], [self.shards[i][0] for i in order],
                               [self.shards[i][1] for i in order], self.n, keep=self.dev)

    def ring(self, d):
        """rank d's walk order: its own piece, then the others in ring order (ShardRing.seq)"""
        P = len(self.shards)
        return [(d + i) % P for i in range(P)]


def owned_tables(gpu, seqs, k, G, what, **kw):
    """Count rank d's share of seqs[d] for every d -> [(kmers, counts) sorted] per rank, summed stats.  Every row
    of rank d must be owned by d."""
    tables, stats = [], np.zeros(3, dtype=np.int64)
    for d, seq in enumerate(seqs):
        st, table = gpu.count(seq, k, owner=(G, d), table=True, **kw)
        a, b = table.sorted()
        table.free()
        assert (a.size, int(b.sum()), int((b == 1).sum())) == (st.distinct, st.total, st.unique), (what, d)
        assert np.all(owner_np(a, G) == d), (what, d, "a row of another owner")
        tables.append((a, b))
        stats += (st.total, st.distinct, st.unique)
    return tables, tuple(int(x) for x in stats)


def check_union(gpu, seqs, k, G, want, what, **kw):
    """The shares of seqs against the oracle's result `want`: disjoint, adding up to its stats and rows (digest)."""
    tables, stats = owned_tables(gpu, seqs, k, G, what, **kw)
    kmers = np.concatenate([a for a, _ in tables])
    counts = np.concatenate([b for _, b in tables])
    order = np.argsort(kmers, kind="stable")
    kmers, counts = kmers[order], counts[order]
    assert np.all(kmers[1:] != kmers[:-1]), (what, "the shares overlap")
    assert kmers.size == want.distinct and stats == want.stats, (what, stats, want.stats)
    if want.kmers is not None:
        assert np.array_equal(kmers, want.kmers) and np.array_equal(counts, want.counts), what
    else:
        assert np.array_equal(R.pairs_digest(kmers, counts), want.digest), what
    return tables


def pieced_seqs(gpu, pieces, G, order=None):
    """rank d's view of the pieces for every d (ring order unless order(d) says otherwise)"""
    return [pieces.wrap(gpu, order(d) if order else pieces.ring(d)) for d in range(G)]


def free_all(seqs):
    for s in seqs:
        s.free()


def profiled(gpu, fn):
    """Run fn with per-launch profiling on -> (its result, {launch name: launches})"""
    gpu.profile(True)
    gpu.profile_reset()
    try:
        out = fn()
        names = {name: int(v["launches"]) for name, v in gpu.profile_dump().items()}
    finally:
        gpu.profile(False)
        gpu.profile_reset()
    return out, names


def collects(names):
    return {n: c for n, c in names.items() if n.startswith("collect_owned")}


# ---- the host-side arithmetic the tests rely on -------------------------------------------------------
def test_owner_model_matches_owner_of():
    """owner_np (the numpy owner_of of these tests) against dnagpu_owner_of for every owner count used here,
    on random keys and on the edge-of-range keys."""
    rng = np.random.default_rng(1)
    keys = np.concatenate([rng.integers(0, 2**64, size=300, dtype=np.uint64), boundary_words(rng),
                           np.array([0, 2**64 - 1], dtype=np.uint64)])
    for G in sorted({1, 2, 4, 8, *MUL_GS, 64}):
        sample = keys if G in MUL_GS else keys[:302]
        got = owner_np(sample, G)
        want = [dnagpu.owner_of(int(x), G) for x in sample]
        assert np.array_equal(got, np.array(want, dtype=np.uint32)), G


def test_ring_shards_are_the_shards_of_count_kmers_multi():
    """ring_shards + shard_words (what ShardRing allocates) equal the per / first / starts / w_alloc arithmetic of
    count_kmers_multi (csrc/dnagpu.cu), transcribed here, so that the pieces below are the ones the library cuts."""
    def multi(n, G):
        per, end = ((n + G - 1) // G + 31) // 32 * 32, (n + 31) // 32 * 32
        out = []
        for d in range(G):
            first = min(d * per, end)
            starts = min(per, n - first) if n > first else 0
            held = min(n, first + starts + 31) - min(n, first)
            out.append((first, starts, ((held + 31) // 32 + 3) & ~1))
        return out
    for n in (1, 31, 32, 33, 100, 1290, 65_537, 2_100_180, 40_000_020):
        for G in range(1, 17):
            assert [(f, s, shard_words(n, f, s)) for f, s in ring_shards(n, G)] == multi(n, G), (n, G)
    assert sum(s == 0 for _, s in ring_shards(100, 16)) == 12


# ---- G x k over pieces --------------------------------------------------------------------------------
def matrix_n(k):
    """just past the 2^21 rows of the multi-GPU threshold, not a multiple of 32"""
    return (1 << 21) + k - 1 + 3007


@pytest.mark.parametrize("k", [1, 5, 13, 15, 16, 17, 21, 31, 32])
@pytest.mark.parametrize("G", [2, 3, 4, 5, 8, 16])
def test_pieces_every_owner_count_and_k(gpu, G, k):
    """ring_shards pieces walked in ring order: every (WPT, LIN, MASKLO) instantiation of k_collect_owned, with
    'G' x 32 and poly-A planted across the cuts and k-mers ending in a piece's overlap word, against the oracle."""
    n = matrix_n(k)
    assert n % 32
    pieces = Pieces(seq_words(7, n), n, ring_shards(n, G))
    seqs = pieced_seqs(gpu, pieces, G)
    check_union(gpu, seqs, k, G, oracle(7, n, k), (G, k))
    free_all(seqs)


@pytest.mark.parametrize("k", [13, 31])
@pytest.mark.parametrize("G", [2, 3, 4, 5, 8, 16])
def test_pieces_exact_flag_walks_the_pieces_item_by_item(gpu, G, k):
    """DNAGPU_COUNT_FLAG_EXACT: k_collect_owned_any alone (owned_item's piece walk, every LIN), one launch per rank"""
    n = matrix_n(k)
    pieces = Pieces(seq_words(7, n), n, ring_shards(n, G))
    seqs = pieced_seqs(gpu, pieces, G)
    _, names = profiled(gpu, lambda: check_union(gpu, seqs, k, G, oracle(7, n, k), (G, k, "exact"), exact=True))
    assert collects(names) == {"collect_owned_any": G}, names
    free_all(seqs)


@pytest.mark.parametrize("k", [5, 16, 32])
@pytest.mark.parametrize("G", [2, 3, 5, 8, 16])
def test_pieces_spectrum_adds_up(gpu, G, k):
    """sum over d of count_spectrum(owner=(G, d)) at H = 16 is the oracle's binned counts: what count_kmers_multi
    returns with max_count"""
    n = matrix_n(k)
    want = oracle(7, n, k)
    pieces = Pieces(seq_words(7, n), n, ring_shards(n, G))
    seqs = pieced_seqs(gpu, pieces, G)
    hist, stats = np.zeros(H, dtype=np.uint64), np.zeros(3, dtype=np.int64)
    for d, seq in enumerate(seqs):
        st, h = gpu.count_spectrum(seq, k, max_count=H, owner=(G, d))
        hist += h
        stats += (st.total, st.distinct, st.unique)
    assert tuple(int(x) for x in stats) == want.stats
    assert np.array_equal(hist, ref_hist(want.counts))
    free_all(seqs)


@pytest.mark.parametrize("k", [13, 31])
@pytest.mark.parametrize("G", [3, 8, 16])
def test_walk_order_does_not_change_the_tables(gpu, G, k):
    """ring order, reverse ring order and a seeded random permutation map the pieces to different tiles; every
    rank's table is the same"""
    n = matrix_n(k)
    want = oracle(7, n, k)
    pieces = Pieces(seq_words(7, n), n, ring_shards(n, G))
    rng = np.random.default_rng(G * 100 + k)
    perms = [list(rng.permutation(G)) for _ in range(G)]
    orders = {"ring": None, "reverse": lambda d: [(d - i) % G for i in range(G)], "random": lambda d: perms[d]}
    tables = {}
    for name, order in orders.items():
        seqs = pieced_seqs(gpu, pieces, G, order)
        tables[name] = check_union(gpu, seqs, k, G, want, (G, k, name))
        free_all(seqs)
    for name in ("reverse", "random"):
        for d in range(G):
            a, b = tables[name][d]
            assert np.array_equal(a, tables["ring"][d][0]) and np.array_equal(b, tables["ring"][d][1]), (name, d)


# ---- uneven tilings and short inputs -------------------------------------------------------------------
def tiling(sizes):
    firsts = np.concatenate([[0], np.cumsum(sizes[:-1])]).astype(int)
    return [(int(f), int(s)) for f, s in zip(firsts, sizes)]


def uneven_tilings(n, G):
    """the shards= form of ShardRing: a 32-base piece, pieces of one tile and a tile +- 32 bases, and one piece
    that holds nearly everything"""
    T = 8192 * wpt_of(G)
    head = {3: [32, T], 4: [T - 32, 32, T + 32], 8: [T, 32, T + 32, T - 32, 32 * 7, 64, 32]}[G]
    tiles = head + [n - sum(head)]
    nearly = [32] * G
    nearly[1] = (n - 32 * G) // 32 * 32
    nearly[-1] = n - sum(nearly[:-1])
    return {"tiles": tiling(tiles), "nearly_all": tiling(nearly)}


@pytest.mark.parametrize("k", [13, 32])
@pytest.mark.parametrize("G", [3, 4, 8])
def test_uneven_pieces(gpu, G, k):
    n = 400_001
    want = oracle(11, n, k)
    for name, shards in uneven_tilings(n, G).items():
        assert len(shards) == G and sum(s for _, s in shards) == n
        pieces = Pieces(seq_words(11, n), n, shards)
        for exact in (False, True):
            seqs = pieced_seqs(gpu, pieces, G)
            check_union(gpu, seqs, k, G, want, (G, k, name, exact), exact=exact)
            free_all(seqs)


SHORT = [  # (n, k, G, shards): None = ring_shards(n, G)
    (20, 21, 4, None),                                   # fewer bases than k: no rows
    (21, 21, 4, None),                                   # one row
    (32, 32, 2, None),
    (33, 1, 3, None),
    (100, 1, 16, None), (100, 13, 16, None), (100, 32, 16, None),   # 12 empty pieces
    (1290, 31, 3, [(0, 640), (640, 640), (1280, 10)]),   # the last piece has no row, the one before 620 of 640
    (1290, 5, 3, [(0, 640), (640, 640), (1280, 10)]),    # the last piece has 6 rows of 10 starts
]


@pytest.mark.parametrize("n,k,G,shards", SHORT)
def test_short_inputs_in_pieces(gpu, n, k, G, shards):
    """no rows, one row, empty pieces (ring_shards of a short sequence) and a last piece with fewer rows than
    starts, which owned_view clamps"""
    want = oracle(13, n, k)
    pieces = Pieces(seq_words(13, n), n, shards or ring_shards(n, G))
    for exact in (False, True):
        seqs = pieced_seqs(gpu, pieces, G)
        assert seqs[0].kmer_count(k) == max(0, n - k + 1)
        check_union(gpu, seqs, k, G, want, (n, k, G, exact), exact=exact)
        free_all(seqs)


# ---- single sequences: more owners, a start limit -------------------------------------------------------
@pytest.mark.parametrize("G,k", [(6, 21), (7, 21), (9, 21), (17, 21), (31, 21), (32, 21), (33, 21), (63, 21),
                                 (64, 21), (17, 13), (63, 13)])
def test_single_sequence_up_to_64_owners(gpu, G, k):
    n = 1_000_003
    seq = gpu.upload(Dna.from_words(seq_words(17, n), n))
    check_union(gpu, [seq] * G, k, G, oracle(17, n, k), (G, k))
    seq.free()


def test_owner_count_above_64_is_an_argument_error(gpu):
    seq = gpu.upload(Dna.from_words(seq_words(17, 5000), 5000))
    for owner in ((65, 0), (64, 64), (3, 3)):
        with pytest.raises(DnaError) as e:
            gpu.count(seq, 21, owner=owner)
        assert e.value.code == EARG, owner
    seq.free()


@pytest.mark.parametrize("k", [13, 31])
@pytest.mark.parametrize("G", [3, 8])
def test_start_limit_with_an_owner_restriction(gpu, G, k):
    """dnagpu_seq_set_start_limit (a shard with its overlap) under owner=(G, d): the k-mers starting in the first
    `limit` bases, 0 = no limit"""
    n = 300_001
    rows = n - k + 1
    words = seq_words(19, n)
    seq = gpu.upload(Dna.from_words(words, n))
    tile = 8192 * wpt_of(G)
    for limit in (0, 1, 31, 32, tile, tile + 1, rows + 100):
        m = min(limit, rows) if limit else rows
        want = R.count_query(words, 1, m + k - 1, words.size, k, faithful=False, threads=8)
        seq.set_start_limit(limit)
        assert seq.kmer_count(k) == m
        check_union(gpu, [seq] * G, k, G, want, (G, k, limit))
    seq.free()


# ---- one owner ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [13, 21, 32])
def test_one_owner_of_a_sequence_in_pieces_is_the_plain_count(gpu, k):
    """owner=(1, 0) (ShardRing with world = 1) counts every k-mer of a sequence in pieces, one piece or several,
    and leaves a single sequence's count as it is"""
    n = 500_003
    words = seq_words(23, n)
    want = oracle(23, n, k)
    seq = gpu.upload(Dna.from_words(words, n))
    st, table = gpu.count(seq, k, table=True)
    a, b = table.sorted()
    table.free()
    assert (st.total, st.distinct, st.unique) == want.stats
    assert np.array_equal(a, want.kmers) and np.array_equal(b, want.counts)
    check_union(gpu, [seq], k, 1, want, (k, "single"))
    for shards in (ring_shards(n, 1), ring_shards(n, 3)):
        pieces = Pieces(words, n, shards)
        for exact in (False, True):
            one = pieces.wrap(gpu, pieces.ring(0))
            check_union(gpu, [one], k, 1, want, (k, len(shards), exact), exact=exact)
            st, hist = gpu.count_spectrum(one, k, max_count=H, owner=(1, 0), exact=exact)
            assert (st.total, st.distinct, st.unique) == want.stats
            assert np.array_equal(hist, ref_hist(want.counts))
            with pytest.raises(DnaError) as e:
                gpu.count(one, k, owner=(1, 1))
            assert e.value.code == EARG
            one.free()
    seq.free()


# ---- the collect attempts -------------------------------------------------------------------------------
def collect_model(own, d, walk, G):
    """The launches count_owned makes for rank d, from the owner of every row (`own`) and the pieces in d's walk
    order ([(first, starts)]), with the kernel's constants: a tile of 256 * WPT words per CTA, a warp covers
    1024 * WPT starts and lists 576 of them, the rest go to 512 shared overflow slots; more than that drops keys.
    -> ({launch name: launches}, share of the fullest tile)"""
    rows = own.size
    wpt = wpt_of(G)
    tile, per_warp = 8192 * wpt, 1024 * wpt
    staged, dropped, fullest = 0, False, 0.0
    for first, starts in walk:
        s = min(starts, rows - first) if rows > first else 0
        if s == 0:
            continue
        mine = np.zeros(-(-s // tile) * tile, dtype=bool)
        mine[:s] = own[first:first + s] == d
        cnt = mine.reshape(-1, OWN_THREADS // 32, per_warp).sum(axis=2)
        ovf = np.maximum(cnt - OWN_SEG, 0).sum(axis=1)
        staged += int(np.minimum(cnt, OWN_SEG).sum() + np.minimum(ovf, OWN_OVF).sum())
        dropped |= bool((ovf > OWN_OVF).any())
        fullest = max(fullest, float(cnt.sum(axis=1).max()) / tile)
    n_true = int((own == d).sum())
    expect = rows // G + 1
    cap = expect + expect // 64 + 65536
    launches = ["collect_owned"]
    if not dropped:
        assert staged == n_true
        if n_true > cap:
            launches.append("collect_owned")      # collected again into a list of the exact size
    else:
        cap = max(cap, staged + staged // 2 + 65536)
        launches.append("collect_owned_any")
        if n_true > cap:
            launches.append("collect_owned_any")  # the generous guess was short too: the exact size
    return dict(collections.Counter(launches)), fullest


def periodic_word(k, share=(0.58, 0.62)):
    """a 32-base unit whose 32 phases rank 0 of 2 owns at a share inside `share` (searched over seeds)"""
    for seed in range(1000):
        w = np.random.default_rng(seed).integers(0, 2**64, dtype=np.uint64)
        kmers = R.generate_kmers(np.full(3, w, dtype=np.uint64), 96, k, window=True)[:32]
        s = float((owner_np(kmers, 2) == 0).mean())
        if share[0] < s < share[1]:
            return w, s
    raise AssertionError("no unit found")


@functools.lru_cache(maxsize=None)
def attempt_input(case, k):
    """-> (words, n, G)"""
    if case == "plain":
        n, G = 4_000_000 + k - 1, 2
        return seq_words(29, n), n, G
    if case == "cap_retry":               # rank 0 owns ~0.59 of every warp's starts: above the cap, no drop
        n, G = 4_000_000 + k - 1, 2
        w, _ = periodic_word(k)
        words = np.full((n + 31) // 32, w, dtype=np.uint64)
        words[-1] &= np.uint64((1 << (2 * (n % 32))) - 1)
        return words, n, G
    if case == "drop_fits":               # 1 M x 'A': tiles drop, 1.5 x the staged count covers the rest
        n, G = 4_000_000 + k - 1, 3
        words = R.synth_seq(31, n)
        words[40_000:40_000 + 31_250] = 0
        return words, n, G
    if case == "drop_exact":              # 20 M x 'A' of 40 M: the generous guess is short too
        n, G = 40_000_000 + k - 1, 8
        words = R.synth_seq(37, n)
        words[200_000:200_000 + 625_000] = 0
        return words, n, G
    raise ValueError(case)


@functools.lru_cache(maxsize=None)
def attempt_oracle(case, k):
    words, n, G = attempt_input(case, k)
    own = owner_np(R.generate_kmers(words, n, k, window=True), G)
    return oracle_of(words, n, k), own


ATTEMPTS = {"plain": {"collect_owned": 1}, "cap_retry": {"collect_owned": 2},
            "drop_fits": {"collect_owned": 1, "collect_owned_any": 1},
            "drop_exact": {"collect_owned": 1, "collect_owned_any": 2}}


@pytest.mark.parametrize("layout", ["single", "pieces"])
@pytest.mark.parametrize("case", list(ATTEMPTS))
def test_collect_attempts(gpu, case, layout):
    """The launches of count_owned's three-attempt loop, predicted by collect_model for every rank and asserted
    from the profile: rank 0 of each input takes the attempts named by the case, the other ranks one launch."""
    k = 21
    words, n, G = attempt_input(case, k)
    want, own = attempt_oracle(case, k)
    if layout == "single":
        seq = gpu.upload(Dna.from_words(words, n))
        seqs, walks = [seq] * G, [[(0, n)]] * G
    else:
        pieces = Pieces(words, n, ring_shards(n, G))
        seqs = pieced_seqs(gpu, pieces, G)
        walks = [[pieces.shards[i] for i in pieces.ring(d)] for d in range(G)]
    models = [collect_model(own, d, walks[d], G) for d in range(G)]
    assert models[0][0] == ATTEMPTS[case], (case, layout, models[0])
    if case == "cap_retry":
        assert 0.55 < models[0][1] < 0.625
    for d in range(1, G):
        assert models[d][0] == {"collect_owned": 1}, (case, layout, d, models[d])
    tables = []
    for d, seq in enumerate(seqs):
        (st, table), names = profiled(gpu, lambda: gpu.count(seq, k, owner=(G, d), table=True))
        assert collects(names) == models[d][0], (case, layout, d, names)
        a, b = table.fetch()
        table.free()
        assert (a.size, int(b.sum())) == (st.distinct, st.total) and np.all(owner_np(a, G) == d), (case, d)
        tables.append((a, b, st))
    kmers = np.concatenate([t[0] for t in tables])
    counts = np.concatenate([t[1] for t in tables])
    stats = tuple(sum(getattr(t[2], f) for t in tables) for f in ("total", "distinct", "unique"))
    assert stats == want.stats and np.unique(kmers).size == kmers.size
    if want.kmers is not None:
        order = np.argsort(kmers)
        assert np.array_equal(kmers[order], want.kmers) and np.array_equal(counts[order], want.counts)
    else:
        assert np.array_equal(R.pairs_digest(kmers, counts), want.digest)
    if layout == "single":
        seq.free()
    else:
        free_all(seqs)
