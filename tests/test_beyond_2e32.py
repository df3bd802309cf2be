"""The k-mer paths past 2^32: more than 2^32 rows in one call, and one k-mer with more than 2^32 copies.

Every count, offset and row number of the C ABI is 64-bit, but several kernels keep 32-bit counters that are
safe only by a size argument, and some code exists only for inputs past 2^32 (the 64-bit dense counters, the
64-bit branch of locate_item, the 64-bit extras counter of the bucket count).  A CPU oracle over 4.4 Gbp is
far too slow for a test, so the inputs here are built so that their exact answer follows from the oracle run
on a few million bases:

- periodic:  X = S^r . T with |S| = L a multiple of 32 and L >= k.  Its rows are the L rows of cyc(S) (S
  followed by its first k - 1 bases) r - 1 times, then the rows of S . T; so is its ordered WHERE scan,
  each part filtered by the clause, and count(X) = (r - 1) cyc(S) + lin(S . T).
- homopolymer block:  X = S1 . B^m . S2 with m >= k.  count(X) = count(S1 . B^m0 . S2) + (m - m0) copies of
  the key B^k, for any m0 >= k; with m0 = m (mod 32) the small twin has the same S1 and S2 words.
- read cycle:  n fixed-stride reads, read i equal to read (i mod c).  Every aggregate is floor(n / c) times
  that of the c reads plus that of the first n mod c reads.

The unmarked tests prove each identity against the oracle over the whole constructed input at small sizes;
the GPU tests trust nothing else.  Results too large for the host are compared on the device: ordered rows
period by period, unordered rows by an order-independent digest (row count, sum of x, sum of mix(x), all
mod 2^64).  Memory estimates are the device's total HBM, not its free HBM: the library keeps freed scratch in
the device's memory pool, so the high-water mark of earlier tests stays reserved."""
import ctypes as C
import functools

import numpy as np
import pytest

import dnagpu
from oracle import ref_cpu as R

M64 = (1 << 64) - 1
_X = 0x9E3779B97F4A7C15  # mix(x) = y * y with y = (x ^ _X) * _M, mod 2^64
_M = 0xBF58476D1CE4E5B9
CODE = {"A": 0, "T": 1, "C": 2, "G": 3}  # the 2-bit packing of encode_dna


def _signed(v):
    return v - (1 << 64) if v >= 1 << 63 else v


# ---- packing and the digest ---------------------------------------------------------------------
def pack(codes):
    """2-bit base codes -> packed words (base i at bits 2 (i mod 32) of word i / 32) + one zero pad word."""
    codes = np.asarray(codes, dtype=np.uint64)
    n = codes.size
    full = np.zeros(((n + 31) // 32) * 32, dtype=np.uint64)
    full[:n] = codes
    words = (full.reshape(-1, 32) << (np.arange(32, dtype=np.uint64) * np.uint64(2))).sum(axis=1, dtype=np.uint64)
    return np.concatenate([words, np.zeros(1, dtype=np.uint64)])


def _mix_np(x):
    y = (x ^ np.uint64(_X)) * np.uint64(_M)
    return y * y


def digest_ref(kmers, counts):
    """(rows, sum x, sum mix(x)) mod 2^64 of the multiset where kmers[i] occurs counts[i] times."""
    kmers = np.asarray(kmers, dtype=np.uint64)
    counts = np.asarray(counts, dtype=np.uint64)
    with np.errstate(over="ignore"):
        return (int(counts.sum(dtype=np.uint64)), int((kmers * counts).sum(dtype=np.uint64)),
                int((_mix_np(kmers) * counts).sum(dtype=np.uint64)))


def digest_dev(t, chunk=1 << 28):
    """The same digest of an int64 tensor with torch's wrapping int64 arithmetic, in chunks."""
    s1 = s2 = 0
    for off in range(0, t.numel(), chunk):
        x = t[off:off + chunk]
        s1 += int(x.sum())
        y = (x ^ _signed(_X)) * _signed(_M)
        s2 += int((y * y).sum())
        del x, y
    return (t.numel(), s1 & M64, s2 & M64)


def merge(parts):
    """[(kmers, counts, multiplier), ...] -> (kmers ascending, counts) of the sum."""
    keys = np.unique(np.concatenate([np.asarray(p[0], dtype=np.uint64) for p in parts]))
    cnt = np.zeros(keys.size, dtype=np.uint64)
    for km, c, mult in parts:  # the keys of one part are distinct
        cnt[np.searchsorted(keys, km)] += np.asarray(c, dtype=np.uint64) * np.uint64(mult)
    return keys, cnt


def stats_of(keys, cnt):
    return (int(cnt.sum(dtype=np.uint64)), int(keys.size), int((cnt == 1).sum()))


def clause(k):
    """A selective WHERE clause for k: ^@ 'AC' (or 'A') and a W/S pattern."""
    prefix = "AC" if k >= 2 else "A"
    pattern = "N" * 4 + "SW" + "N" * (k - 6) if k >= 6 else "N" * (k - 1) + "W"
    return prefix, pattern


def _pk(prefix):
    return R.kmer_make(prefix) if prefix else None


def _count(words, n, k, prefix=None, pattern=None, n_seqs=1, stride=None):
    r = R.count_query(words, n_seqs, n, words.size if stride is None else stride, k, prefix=_pk(prefix),
                      pattern=pattern, faithful=False)
    return r.kmers, r.counts


def _rows(words, n, k, prefix=None, pattern=None):
    if prefix is None and pattern is None:
        return R.generate_kmers(words, n, k, window=True)
    return R.filter_kmers(words, n, k, _pk(prefix), pattern)


# ---- references -------------------------------------------------------------------------------
class Periodic:
    """X = S^r . T, |S| = L a multiple of 32."""

    def __init__(self, seed, L, r, nT):
        assert L % 32 == 0
        rng = np.random.default_rng(seed)
        self.S = rng.integers(0, 4, L, dtype=np.uint8)
        self.T = rng.integers(0, 4, nT, dtype=np.uint8)
        self.L, self.r, self.n = L, r, L * r + nT

    def words(self):
        wS = pack(self.S)[:-1]
        return np.concatenate([np.tile(wS, self.r), pack(self.T)])

    def codes(self):
        return np.concatenate([np.tile(self.S, self.r), self.T])

    def _cyc(self, k):
        c = np.concatenate([self.S, self.S[:k - 1]])
        return pack(c), c.size

    def _lin(self):
        c = np.concatenate([self.S, self.T])
        return pack(c), c.size

    def rows(self, k, prefix=None, pattern=None):
        """(rows of one period, rows of S . T): X's rows are the first r - 1 times, then the second."""
        return _rows(*self._cyc(k), k, prefix, pattern), _rows(*self._lin(), k, prefix, pattern)

    def count(self, k, prefix=None, pattern=None):
        return merge([(*_count(*self._cyc(k), k, prefix, pattern), self.r - 1),
                      (*_count(*self._lin(), k, prefix, pattern), 1)])


class Block:
    """X = S1 . B^m . S2 with |S1| not a multiple of 32 and |S1| + m one (S2 starts on a word)."""

    def __init__(self, seed, n1, base, m, n2, k):
        assert n1 % 32 and (n1 + m) % 32 == 0 and m >= k
        rng = np.random.default_rng(seed)
        self.S1 = rng.integers(0, 4, n1, dtype=np.uint8)
        self.S2 = rng.integers(0, 4, n2, dtype=np.uint8)
        self.b, self.m, self.k = CODE[base], m, k
        self.m0 = k + (m - k) % 32  # the twin's block: >= k, same residue mod 32
        self.n = n1 + m + n2
        self.key = sum(self.b << (2 * i) for i in range(k))  # B^k

    def _twin(self):
        c = np.concatenate([self.S1, np.full(self.m0, self.b, dtype=np.uint8), self.S2])
        return pack(c), c.size

    def words(self):
        """X's words: the twin's with (m - m0) / 32 more whole block words."""
        tw, _ = self._twin()
        a = self.S1.size // 32 + 1  # first whole word of the block
        fill = np.uint64(sum(self.b << (2 * i) for i in range(32)))
        return np.concatenate([tw[:a], np.full((self.m - self.m0) // 32, fill, dtype=np.uint64), tw[a:]])

    def codes(self):
        return np.concatenate([self.S1, np.full(self.m, self.b, dtype=np.uint8), self.S2])

    def count(self, prefix=None, pattern=None):
        k = self.k
        parts = [(*_count(*self._twin(), k, prefix, pattern), 1)]
        kw = pack(np.full(k, self.b, dtype=np.uint8))
        if _rows(kw, k, k, prefix, pattern).size:
            parts.append((np.array([self.key], dtype=np.uint64), np.array([self.m - self.m0], dtype=np.uint64), 1))
        return merge(parts)


class ReadCycle:
    """n_reads fixed-stride reads; read i is read (i mod c) of c random reads."""

    def __init__(self, seed, c, bases, stride, n_reads):
        rng = np.random.default_rng(seed)
        self.reads = [rng.integers(0, 4, bases, dtype=np.uint8) for _ in range(c)]
        self.words_c = np.concatenate([np.concatenate([pack(r)[:-1], np.zeros(stride - (bases + 31) // 32,
                                                                              dtype=np.uint64)])
                                       for r in self.reads])
        self.c, self.bases, self.stride, self.n_reads = c, bases, stride, n_reads

    def words(self):
        q, rem = divmod(self.n_reads, self.c)
        return np.concatenate([np.tile(self.words_c, q), self.words_c[:rem * self.stride], np.zeros(1, np.uint64)])

    def count(self, k, prefix=None, pattern=None):
        q, rem = divmod(self.n_reads, self.c)
        parts = [(*_count(self.words_c, self.bases, k, prefix, pattern, self.c, self.stride), q)]
        if rem:
            parts.append((*_count(self.words_c[:rem * self.stride], self.bases, k, prefix, pattern, rem,
                                  self.stride), 1))
        return merge(parts)


# ---- the references against the oracle over the whole input (small sizes, no GPU) -----------------
KS = [1, 5, 21, 31, 32]


def _direct(words, n, k, prefix, pattern, n_seqs=1, stride=None):
    r = R.count_query(words, n_seqs, n, words.size if stride is None else stride, k, prefix=_pk(prefix),
                      pattern=pattern, faithful=True)
    return r


@pytest.mark.parametrize("where", [False, True])
@pytest.mark.parametrize("k", KS)
def test_periodic_reference_matches_oracle(k, where):
    p = Periodic(11, 1024, 7, 1001)
    prefix, pattern = clause(k) if where else (None, None)
    words = p.words()
    assert np.array_equal(words, pack(p.codes()))
    want = _direct(words, p.n, k, prefix, pattern)
    keys, cnt = p.count(k, prefix, pattern)
    assert stats_of(keys, cnt) == want.stats
    assert np.array_equal(keys, want.kmers) and np.array_equal(cnt, want.counts)
    per, tail = p.rows(k, prefix, pattern)
    rows = _rows(words, p.n, k, prefix, pattern)
    assert np.array_equal(np.concatenate([per] * (p.r - 1) + [tail]), rows)
    if not where:
        assert per.size == p.L
    assert digest_ref(keys, cnt) == digest_ref(rows, np.ones(rows.size, np.uint64))


@pytest.mark.parametrize("where", [False, True])
@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("base", ["A", "G"])
@pytest.mark.parametrize("m", [40, 200])
def test_block_reference_matches_oracle(m, base, k, where):
    n1 = 1000 + (-(1000 + m)) % 32  # S2 starts on a word boundary
    n1 = n1 if n1 % 32 else n1 + 32
    b = Block(12, n1, base, m, 517, k)
    prefix, pattern = clause(k) if where else (None, None)
    words = b.words()
    assert np.array_equal(words, pack(b.codes()))
    want = _direct(words, b.n, k, prefix, pattern)
    keys, cnt = b.count(prefix, pattern)
    assert stats_of(keys, cnt) == want.stats
    assert np.array_equal(keys, want.kmers) and np.array_equal(cnt, want.counts)


@pytest.mark.parametrize("where", [False, True])
@pytest.mark.parametrize("k", KS)
def test_read_cycle_reference_matches_oracle(k, where):
    rc = ReadCycle(13, 5, 150, 5, 23)
    prefix, pattern = clause(k) if where else (None, None)
    words = rc.words()
    want = _direct(words, rc.bases, k, prefix, pattern, rc.n_reads, rc.stride)
    keys, cnt = rc.count(k, prefix, pattern)
    assert stats_of(keys, cnt) == want.stats
    assert np.array_equal(keys, want.kmers) and np.array_equal(cnt, want.counts)


def test_device_digest_matches_host_digest():
    """torch's int64 arithmetic wraps like numpy's uint64: the two digests agree (on CPU tensors here)."""
    import torch
    rng = np.random.default_rng(14)
    x = rng.integers(0, 1 << 63, 100_003, dtype=np.uint64) * np.uint64(2) + np.uint64(1)  # top bit set too
    keys, cnt = np.unique(x, return_counts=True)
    assert digest_dev(torch.from_numpy(x.view(np.int64)), chunk=4096) == digest_ref(keys, cnt)


# ---- GPU ----------------------------------------------------------------------------------------
GB = 1 << 30
PER_L, PER_R, PER_T = 1 << 24, 260, 3_000_017  # 4.365e9 bases: the last period and T start past row 2^32
BLOCK_N1, BLOCK_N2 = 1_000_003, 1_000_001


def _need(gpu, gib, what):
    total = gpu.device_info()["hbm_total"]
    if total < gib * GB:
        pytest.skip(f"{what} needs about {gib} GiB of device memory; this device has {total / GB:.0f} GiB")


def _free():
    import gc
    import torch
    gc.collect()
    torch.cuda.empty_cache()


@pytest.fixture(autouse=True)
def _hbm_log(request):
    """Device memory around every GPU test (the pool keeps its high-water mark, so 'free' only falls)."""
    if request.node.get_closest_marker("gpu") is None:
        yield
        return
    gpu = request.getfixturevalue("gpu")
    before = gpu.device_info()["hbm_free"]
    yield
    _free()
    after = gpu.device_info()["hbm_free"]
    print(f"\n[hbm_free] {request.node.name}: {before / GB:.1f} GiB before, {after / GB:.1f} GiB after")


@functools.lru_cache(maxsize=1)
def _periodic():
    return Periodic(21, PER_L, PER_R, PER_T)


@functools.lru_cache(maxsize=1)
def _periodic_words():
    return _periodic().words()


@functools.lru_cache(maxsize=None)
def _periodic_count(k, prefix=None, pattern=None):
    return _periodic().count(k, prefix, pattern)


def _upload_periodic(gpu):
    p = _periodic()
    return gpu.upload(dnagpu.Dna.from_words(_periodic_words(), p.n))


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint64).view(np.int64)).cuda()


def _check_periodic_rows(out, per, tail, r):
    """Ordered rows of X on the device: r - 1 periods, then the tail."""
    import torch
    P = per.size
    assert out.numel() == (r - 1) * P + tail.size
    dper = _dev(per)
    for j in range(r - 1):
        assert torch.equal(out[j * P:(j + 1) * P], dper), f"period {j}"
    assert torch.equal(out[(r - 1) * P:], _dev(tail))


def _check_table(st, table, keys, cnt):
    assert (st.total, st.distinct, st.unique) == stats_of(keys, cnt)
    got_k, got_c = table.sorted()
    assert np.array_equal(got_k, keys) and np.array_equal(got_c, cnt)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [13, 31, 32])
def test_extract_periodic_past_2e32_rows(gpu, k):
    _need(gpu, 64, "a 4.4e9-row extraction")
    p = _periodic()
    per, tail = p.rows(k)
    seq = _upload_periodic(gpu)
    assert seq.kmer_count(k) == p.n - k + 1
    out = gpu.extract(seq, k)
    seq.free()
    _check_periodic_rows(out, per, tail, p.r)
    del out


def _scan_exact(gpu, call, seq, k, prefix, pattern, planes):
    """dnagpu_filter / dnagpu_collect into an exactly sized buffer (the count first)."""
    import torch
    w, _keep = dnagpu._where(prefix, pattern, planes)
    n = C.c_uint64()
    gpu._ok(call(gpu.handle, seq.handle, k, C.byref(w), None, 0, C.byref(n)))
    out = torch.empty(max(int(n.value), 2), dtype=torch.int64, device=f"cuda:{gpu.device}")
    got = C.c_uint64()
    gpu._ok(call(gpu.handle, seq.handle, k, C.byref(w), out.data_ptr(), out.numel(), C.byref(got)))
    gpu.synchronize()
    assert got.value == n.value
    return out[:got.value]


@pytest.mark.gpu
@pytest.mark.parametrize("planes", [False, True])
@pytest.mark.parametrize("which", ["selective", "every_row"])
def test_where_scans_periodic_past_2e32_rows(gpu, which, planes):
    """filter (ordered), collect (unordered) and filter_count; 'N' x k keeps every row (> 2^32 rows out)."""
    import torch
    _need(gpu, 80, "a 4.4e9-row WHERE scan")
    k = 31
    prefix, pattern = clause(k) if which == "selective" else (None, "N" * k)
    p = _periodic()
    per, tail = p.rows(k, prefix, pattern)
    keys, cnt = _periodic_count(k, prefix, pattern)
    seq = _upload_periodic(gpu)
    assert gpu.filter_count(seq, k, prefix, pattern) == int(cnt.sum())
    out = _scan_exact(gpu, gpu.lib.dnagpu_filter, seq, k, prefix, pattern, planes)
    _check_periodic_rows(out, per, tail, p.r)
    del out
    _free()
    col = _scan_exact(gpu, gpu.lib.dnagpu_collect, seq, k, prefix, pattern, planes)
    seq.free()
    assert digest_dev(col) == digest_ref(keys, cnt)
    if which == "selective":
        got = torch.sort(col).values.cpu().numpy()
        assert np.array_equal(got, np.sort(np.repeat(keys, cnt.astype(np.int64)).view(np.int64)))
    del col


GROUP_BY = {  # name: (k, count() keyword arguments)
    "auto_k31": (31, {}),
    "auto_k21": (21, {}),
    "auto_k14": (14, {}),
    "dense_k12": (12, {"method": dnagpu.COUNT_DENSE}),
    "dense_smem_k5": (5, {"method": dnagpu.COUNT_DENSE}),
    "hash_k31": (31, {"method": dnagpu.COUNT_HASH, "expected_keys": 1 << 25}),
    "where_k31": (31, dict(zip(("prefix", "pattern"), clause(31)))),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GROUP_BY))
def test_group_by_periodic_past_2e32_rows(gpu, name):
    _need(gpu, 100, "a 4.4e9-row GROUP BY")
    k, kw = GROUP_BY[name]
    keys, cnt = _periodic_count(k, kw.get("prefix"), kw.get("pattern"))
    seq = _upload_periodic(gpu)
    st, table = gpu.count(seq, k, table=True, **kw)
    seq.free()
    _check_table(st, table, keys, cnt)
    table.free()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [12, 31])
def test_count_keys_of_the_periodic_key_list(gpu, k):
    """count_keys over the extracted 4.4e9-key list (k = 31: partition from keys, k = 12: dense over keys)."""
    _need(gpu, 120, "a GROUP BY of a 4.4e9-key list")
    keys, cnt = _periodic_count(k)
    seq = _upload_periodic(gpu)
    kl = gpu.extract(seq, k)
    seq.free()
    st, table = gpu.count_keys(kl, k, table=True)
    del kl
    _check_table(st, table, keys, cnt)
    table.free()


@pytest.mark.gpu
def test_count_kmers_host_buffer_periodic(gpu):
    """The host-buffer entry (pipelined upload + optimistic level 1) at 4.4e9 rows."""
    _need(gpu, 100, "a 4.4e9-row GROUP BY")
    p = _periodic()
    keys, cnt = _periodic_count(31)
    st, table = gpu.count_kmers(dnagpu.Dna.from_words(_periodic_words(), p.n), 31)
    _check_table(st, table, keys, cnt)
    table.free()


def _owner_shares(gpu, seq, k, G):
    """The G owner shares of a count on one device -> (summed stats, all rows sorted)."""
    tot = [0, 0, 0]
    ks, cs = [], []
    for part in range(G):
        st, table = gpu.count(seq, k, table=True, owner=(G, part))
        tot = [tot[0] + st.total, tot[1] + st.distinct, tot[2] + st.unique]
        a, b = table.fetch()
        table.free()
        ks.append(a)
        cs.append(b)
        _free()
    a, b = np.concatenate(ks), np.concatenate(cs)
    order = np.argsort(a, kind="stable")
    return tuple(tot), a[order], b[order]


@pytest.mark.gpu
@pytest.mark.parametrize("G", [2, 3])
def test_owner_shares_periodic(gpu, G):
    _need(gpu, 100, "the owner shares of a 4.4e9-row count")
    keys, cnt = _periodic_count(31)
    seq = _upload_periodic(gpu)
    tot, a, b = _owner_shares(gpu, seq, 31, G)
    seq.free()
    assert tot == stats_of(keys, cnt)
    assert np.array_equal(a, keys) and np.array_equal(b, cnt)


# ---- one k-mer with more than 2^32 copies ---------------------------------------------------------
def _block(base, k):
    """S1 . B^m . S2 with m - k + 1 ~ 2^32 + 2^20 copies of B^k (and S2 on a word boundary)."""
    m = (1 << 32) + (1 << 20) + k - 1
    m += (-(BLOCK_N1 + m)) % 32
    return Block(31, BLOCK_N1, base, m, BLOCK_N2, k)


def _check_block(st, table, b, keys, cnt):
    key = np.uint64(b.key)  # a Python int would be compared as a float
    i = int(np.searchsorted(keys, key))
    assert keys[i] == key and int(cnt[i]) > (1 << 32) + (1 << 20)
    assert (st.total, st.distinct, st.unique) == stats_of(keys, cnt)
    if table is not None:
        got_k, got_c = table.sorted()
        j = int(np.searchsorted(got_k, key))
        assert j < got_k.size and got_k[j] == key and int(got_c[j]) == int(cnt[i]), \
            f"count of B^k: {int(got_c[j]) if j < got_k.size else None}, want {int(cnt[i])}"
        assert np.array_equal(got_k, keys) and np.array_equal(got_c, cnt)


BLOCK_CASES = {  # name: (base, k, how)
    "A_k31_partition": ("A", 31, "count"),
    "A_k31_host_buffer": ("A", 31, "count_kmers"),
    "A_k31_owner2": ("A", 31, "owner"),
    "A_k8_dense": ("A", 8, "count"),
    "A_k31_hash": ("A", 31, "hash"),
    "G_k31_partition": ("G", 31, "count"),
    "G_k32_side_counter": ("G", 32, "count"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(BLOCK_CASES))
def test_kmer_with_more_than_2e32_copies(gpu, name):
    """B^k occurs ~ 2^32 + 2^20 times: a 32-bit counter would report ~ 2^20 and take the key out of the unique
    set twice."""
    base, k, how = BLOCK_CASES[name]
    _need(gpu, 120 if how == "owner" else 90, "a GROUP BY of a 4.3e9-copy k-mer")
    b = _block(base, k)
    keys, cnt = b.count()
    dna = dnagpu.Dna.from_words(b.words(), b.n)
    if how == "count_kmers":
        st, table = gpu.count_kmers(dna, k)
        _check_block(st, table, b, keys, cnt)
        table.free()
        return
    seq = gpu.upload(dna)
    del dna
    if how == "owner":
        tot, a, c = _owner_shares(gpu, seq, k, 2)
        seq.free()
        assert tot == stats_of(keys, cnt)
        assert np.array_equal(a, keys) and np.array_equal(c, cnt)
        return
    kw = {"method": dnagpu.COUNT_HASH, "expected_keys": 1 << 22} if how == "hash" else {}
    st, _ = gpu.count(seq, k, **kw)  # aggregates only: the counting pass alone
    _check_block(st, None, b, keys, cnt)
    st, table = gpu.count(seq, k, table=True, **kw)  # and the pass that emits the rows
    seq.free()
    _check_block(st, table, b, keys, cnt)
    table.free()


# ---- reads past 2^32 items ------------------------------------------------------------------------
READS_C, READS_BASES, READS_STRIDE, READS_N = 64, 150, 5, (1 << 30) + 5  # 4 n_reads > 2^32 items, 43 GB of words
READS_CLAUSE = ("ACGT", "N" * 4 + "SW" + "N" * 25)  # about 1 row in 1024 at k = 31


@functools.lru_cache(maxsize=1)
def _reads():
    return ReadCycle(41, READS_C, READS_BASES, READS_STRIDE, READS_N)


@functools.lru_cache(maxsize=None)
def _reads_count(k, prefix=None, pattern=None):
    return _reads().count(k, prefix, pattern)


def _wrap_reads(gpu):
    """The batch built on the device by repetition (the host never holds it) and borrowed."""
    import torch
    rc = _reads()
    per = rc.c * rc.stride
    q, rem = divmod(rc.n_reads, rc.c)
    buf = torch.empty(rc.n_reads * rc.stride + 2, dtype=torch.int64, device=f"cuda:{gpu.device}")
    src = _dev(rc.words_c)
    buf[:q * per].view(q, per).copy_(src.unsqueeze(0).expand(q, per))
    buf[q * per:rc.n_reads * rc.stride].copy_(src[:rem * rc.stride])
    buf[rc.n_reads * rc.stride:].zero_()
    return gpu.wrap_reads(buf, rc.n_reads, rc.bases, rc.stride)


@pytest.mark.gpu
@pytest.mark.parametrize("planes", [False, True])
def test_reads_where_scans_past_2e32_items(gpu, planes):
    _need(gpu, 64, "a 43 GB batch of reads")
    k = 31
    prefix, pattern = READS_CLAUSE
    keys, cnt = _reads_count(k, prefix, pattern)
    seq = _wrap_reads(gpu)
    assert gpu.filter_count(seq, k, prefix, pattern) == int(cnt.sum())
    col = _scan_exact(gpu, gpu.lib.dnagpu_collect, seq, k, prefix, pattern, planes)
    seq.free()
    assert digest_dev(col) == digest_ref(keys, cnt)
    del col


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 3, 31])
def test_reads_group_by_past_2e32_items(gpu, k):
    """k = 1 / 3: dense counts of ~ 4e10 / 1e10 per key; k = 31 with the WHERE clause fused into the count."""
    _need(gpu, 64, "a 43 GB batch of reads")
    prefix, pattern = READS_CLAUSE if k == 31 else (None, None)
    keys, cnt = _reads_count(k, prefix, pattern)
    seq = _wrap_reads(gpu)
    st, table = gpu.count(seq, k, prefix=prefix, pattern=pattern, table=True)
    seq.free()
    _check_table(st, table, keys, cnt)
    table.free()


# ---- more than one GPU -----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("which", ["A_block", "periodic"])
def test_two_gpu_context_counts(gpu, which):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    _need(gpu, 100, "a 4.4e9-row GROUP BY")
    if which == "A_block":
        b = _block("A", 31)
        keys, cnt = b.count()
        dna = dnagpu.Dna.from_words(b.words(), b.n)
    else:
        keys, cnt = _periodic_count(31)
        dna = dnagpu.Dna.from_words(_periodic_words(), _periodic().n)
    ctx = dnagpu.Context(devices=[0, 1])
    try:
        st, table = ctx.count_kmers(dna, 31)
        _check_table(st, table, keys, cnt)
        table.free()
    finally:
        ctx.close()
