"""Every GROUP BY dispatch of dnagpu_count and dnagpu_count_keys against the CPU oracle, with the kernels that ran.

A count does not run one kernel per query.  pick_method (csrc/dnagpu.cu) chooses DENSE, HASH or PARTITION from k
and the row count n; count_any then branches on the WHERE clause:

- no clause, or DENSE:         the count kernel over the packed input, the clause fused into it
                               (count_dense_smem for k <= 7, count_dense, count_hash, the partition pipeline);
- a clause, HASH or PARTITION: one predicate scan collects the kept rows (filter_collect) into a buffer of
                               min(n, max(2^20, n / 8)) rows, and a second, exactly sized scan runs when that
                               buffer overflows;
  - nothing kept:              no count kernel at all;
  - n_match <= n / 2, or PARTITION: the collected list is counted, by the method pick_method gives n_match
                               (count_hash_keys, or the partition pipeline from keys);
  - more than n / 2 and HASH:  the fused filtered insert (count_hash), the table sized by n_match.

Key lists (dnagpu_count_keys) run count_dense_keys, count_hash_keys or the partition pipeline from keys.  Every
case here compares stats and the sorted (kmer, count) rows with the oracle and asserts, from the per-launch profile
(dnagpu_profile_dump), which of these kernels ran.  A change of a threshold therefore fails a path assertion even
when the answer stays right; such a change should come with the new expectation here."""
import numpy as np
import pytest
import torch

import dnagpu
from dnagpu import Dna, DnaError
from dnagpu.types import pack_bases
from oracle import ref_cpu as R

pytestmark = pytest.mark.gpu

AUTO, DENSE, HASH, PART = dnagpu.COUNT_AUTO, dnagpu.COUNT_DENSE, dnagpu.COUNT_HASH, dnagpu.COUNT_PARTITION
M64 = (1 << 64) - 1
EARG, EINTERNAL = 20, 25
# the launches that count: one of them is the GROUP BY itself ("count_buckets" is the partition pipeline's
# bucket count, launched again when a level is redone)
COUNT_KERNELS = {"count_dense", "count_dense_smem", "count_dense_keys", "count_hash", "count_hash_keys",
                 "count_buckets"}
KEYS_KERNEL = {DENSE: "count_dense_keys", HASH: "count_hash_keys", PART: "count_buckets"}
METHODS = [("auto", AUTO, False), ("dense", DENSE, False), ("hash", HASH, False), ("partition", PART, False),
           ("partition_exact", PART, True)]
H = 16  # spectrum bins: counts 1..15 and "16 or more", across the 15-copy limit of k_count_buckets_bins


# ---- helpers ----------------------------------------------------------------------------------------
def profiled(gpu, fn, error=False):
    """Run fn with per-launch profiling on -> (its result, {launch name: launches}).  error=True: fn must raise a
    DnaError, which takes the place of the result."""
    gpu.profile(True)
    gpu.profile_reset()
    try:
        try:
            out = fn()
        except DnaError as e:
            if not error:
                raise
            out = e
        else:
            assert not error, "the call was expected to fail"
        names = {name: int(v["launches"]) for name, v in gpu.profile_dump().items()}
    finally:
        gpu.profile(False)
        gpu.profile_reset()
    return out, names


def check_path(got, want, what):
    """want: {"filter_collect": scans, kernel: 1, ...}.  The count kernels that ran must be exactly want's; the
    dense and hash kernels run once, the bucket count at least once."""
    ran = {name for name in got if name in COUNT_KERNELS}
    assert ran == set(want) - {"filter_collect"}, (what, got)
    assert got.get("filter_collect", 0) == want.get("filter_collect", 0), (what, got)
    for name in ran - {"count_buckets"}:
        assert got[name] == 1, (what, got)


def resolve(method, k, n):
    """The method a query of n rows runs: an explicit one (DENSE only up to k = 16), or AUTO's choice."""
    if method == DENSE and k > 16:
        return HASH
    if method != AUTO:
        return method
    if k <= 12 and 4**k <= max(1 << 16, 8 * n):
        return DENSE
    return PART if n >= 1 << 21 else HASH


def expected_path(k, n, method, filtered, n_match, keys=False):
    """The launches count_any makes for a query of n rows (n_match of them kept by the WHERE clause)."""
    m = resolve(method, k, n)
    if n == 0:
        return {}
    if keys:
        return {KEYS_KERNEL[m]: 1}
    if not filtered or m == DENSE:
        return {{DENSE: "count_dense_smem" if k <= 7 else "count_dense", HASH: "count_hash",
                 PART: "count_buckets"}[m]: 1}
    want = {"filter_collect": 1 if n_match <= min(n, max(1 << 20, n // 8)) else 2}
    if n_match == 0:
        return want
    if n_match <= n // 2 or m == PART:
        want[KEYS_KERNEL[resolve(method, k, n_match)]] = 1
    else:
        want["count_hash"] = 1
    return want


def ref_hist(counts, h=H):
    counts = np.asarray(counts, dtype=np.uint64)
    return np.bincount(np.minimum(counts, np.uint64(h)).astype(np.int64), minlength=h + 1)[1:].astype(np.uint64)


def check_rows(st, table, stats, kmers, counts, what):
    assert (st.total, st.distinct, st.unique) == tuple(stats), what
    assert table.rows == len(kmers), what
    kk, cc = table.sorted()
    table.free()
    assert np.array_equal(kk, kmers) and np.array_equal(cc, counts), what


def check_spectrum(gpu, seq, k, want, what, **kw):
    st, hist = gpu.count_spectrum(seq, k, max_count=H, **kw)
    assert (st.total, st.distinct, st.unique) == want.stats, what
    assert np.array_equal(hist, ref_hist(want.counts)), what


def oracle_keys(keys):
    kmers, counts = np.unique(keys, return_counts=True)
    return (keys.size, kmers.size, int((counts == 1).sum())), kmers, counts.astype(np.uint64)


def device(keys):
    return torch.from_numpy(np.ascontiguousarray(keys, dtype=np.uint64).view(np.int64)).cuda()


def rand_words(rng, n):
    words = rng.integers(0, 2**64, size=(n + 31) // 32, dtype=np.uint64)
    if n % 32:
        words[-1] &= np.uint64((1 << (2 * (n % 32))) - 1)
    return words


def distinct_keys(rng, n, k=31):
    """n distinct k-mers in random order ('G' x 32 never among them)"""
    top = 1 << min(2 * k, 63)
    if top <= 4 * n:
        return rng.permutation(top)[:n].astype(np.uint64)
    keys = np.unique(rng.integers(0, top, size=2 * n + 64, dtype=np.uint64))
    rng.shuffle(keys)
    assert keys.size >= n
    return keys[:n]


def with_copies(rng, distinct):
    """1 to 3 copies of every key, shuffled"""
    keys = np.repeat(distinct, rng.integers(1, 4, size=distinct.size))
    rng.shuffle(keys)
    return keys


def ordinary_query_is_right(gpu):
    """After a failed count the context answers the next ordinary query exactly, with and without a table."""
    n, k = 50_001, 21
    words = R.synth_seq(9, n)
    want = R.count_query(words, 1, n, words.size, k, faithful=False)
    seq = gpu.upload(Dna.from_words(words, n))
    st, _ = gpu.count(seq, k)
    assert (st.total, st.distinct, st.unique) == want.stats
    st, table = gpu.count(seq, k, table=True)
    check_rows(st, table, want.stats, want.kmers, want.counts, "after a failed count")
    seq.free()


# ---- the profiling ABI ------------------------------------------------------------------------------
def test_profile_dump_names_every_launch(gpu):
    """dnagpu_profile_*: nothing is recorded with profiling off; with it on every launch is recorded under the name
    passed to launch(), the dump and the prefix query agree, and a reset empties both."""
    seq = gpu.upload(Dna("ACGTTGCAAGGCT" * 100))
    gpu.profile(False)
    gpu.profile_reset()
    gpu.count(seq, 5, method=DENSE)
    assert gpu.profile_dump() == {}
    _, got = profiled(gpu, lambda: gpu.count(seq, 5, method=DENSE))
    assert got["count_dense_smem"] == 1 and got["dense_stats"] == 1, got
    assert "count_dense" not in got and "count_dense_keys" not in got, got
    gpu.profile(True)
    try:
        gpu.count(seq, 5, method=DENSE)
        gpu.count(seq, 9, method=DENSE)
        dump = gpu.profile_dump()
        assert dump["count_dense_smem"]["launches"] == 1 and dump["count_dense"]["launches"] == 1, dump
        ms, n = gpu.profile_query("count_dense")   # a prefix: count_dense and count_dense_smem
        assert n == 2 and ms > 0
        ms, n = gpu.profile_query("")
        assert n == sum(v["launches"] for v in dump.values())
        assert ms == pytest.approx(sum(v["ms"] for v in dump.values()), rel=1e-4, abs=1e-3)
        gpu.profile_reset()
        assert gpu.profile_dump() == {} and gpu.profile_query("") == (0.0, 0)
    finally:
        gpu.profile(False)
        gpu.profile_reset()
    seq.free()


# ---- method x layout x WHERE clause -----------------------------------------------------------------
def _clauses(k):
    """(name, prefix, pattern, planes): ~1/16 (1/4 at k = 1), 3/4, nothing, and the plane test"""
    sel = "AC" if k >= 2 else "A"
    return [("none", None, None, False), ("selective", sel, None, False),
            ("unselective", None, "N" * (k - 1) + "B", False), ("nothing", None, "U" + "N" * (k - 1), False),
            ("planes", sel, None, True)]


def _layout(gpu, layout, k):
    """(device input, oracle(prefix, pattern) -> CountResult)"""
    rng = np.random.default_rng(1000 + k)
    if layout == "single":
        n = 150_001
        words = R.synth_seq(140 + k, n)
        words[100:102] = np.uint64(M64)    # 'G' x 64 and 'A' x 64
        words[200:202] = 0
        return (gpu.upload(Dna.from_words(words, n)),
                lambda pk, pat: R.count_query(words, 1, n, words.size, k, prefix=pk, pattern=pat, faithful=False))
    if layout == "reads":
        n_reads, bpr, stride = 1200, 150, 7   # 5 words of bases per read, 7 apart
        reads = R.synth_reads(k, n_reads, bpr, stride)
        reads[:4] = np.uint64(M64)            # read 0 starts with 'G' x 128
        return (gpu.upload_reads(reads, n_reads, bpr, stride),
                lambda pk, pat: R.count_query(reads, n_reads, bpr, stride, k, prefix=pk, pattern=pat,
                                              faithful=False))
    lens = [1, k - 1, k, k + 1, 31, 32, 33, 3000, 4321] + [int(x) for x in rng.integers(1, 300, size=200)]
    dnas = [Dna.from_words(rand_words(rng, m), m) for m in lens if m > 0] + [Dna("G" * 40 + "ACGT" * 10)]
    return (gpu.upload_ragged(dnas),
            lambda pk, pat: R.count_ragged([(d.words, d.length) for d in dnas], k, prefix=pk, pattern=pat,
                                           faithful=False))


# DENSE at k = 16 counts into 4^16 counters (16 GiB): only these cases of the matrix, one key list and one error
DENSE16 = {("single", "none"), ("single", "selective"), ("reads", "unselective"), ("ragged", "planes")}


@pytest.mark.parametrize("k", [1, 4, 7, 8, 12, 13, 16, 17, 31, 32])
@pytest.mark.parametrize("layout", ["single", "reads", "ragged"])
def test_method_layout_where_matrix(gpu, layout, k):
    """Every branch of count_any for a single sequence, fixed-stride reads and a ragged batch: DENSE with and
    without a clause (count_dense_smem up to k = 7, count_dense from k = 8; DENSE past k = 16 runs count_hash), the
    unfiltered HASH and PARTITION counts (PARTITION with DNAGPU_COUNT_FLAG_EXACT runs its level-1 histogram), and
    with a clause the collect: nothing kept (no count kernel), 1/16 kept (the listed count), 3/4 kept (HASH: the
    fused filtered insert; PARTITION: the listed count).  Rows, stats and the spectrum against the oracle."""
    seq, oracle = _layout(gpu, layout, k)
    n = gpu.count(seq, k)[0].total
    for cname, prefix, pattern, planes in _clauses(k):
        want = oracle(R.kmer_make(prefix) if prefix else None, pattern)
        if cname == "none":
            assert want.total == n > 0
            if k == 32:
                assert np.uint64(M64) in want.kmers   # the 'G' x 32 sentinel is a key of the input
        if cname == "nothing":
            assert want.total == 0
        for mname, method, exact in METHODS:
            if method == DENSE and k == 16 and (layout, cname) not in DENSE16:
                continue
            what = (layout, k, cname, mname)
            kw = dict(prefix=prefix, pattern=pattern, planes=planes, method=method, exact=exact)
            (st, table), got = profiled(gpu, lambda: gpu.count(seq, k, table=True, **kw))
            check_rows(st, table, want.stats, want.kmers, want.counts, what)
            check_path(got, expected_path(k, n, method, prefix is not None or pattern is not None, want.total),
                       what)
            if exact and cname == "none":
                assert "part_hist" in got, (what, got)
            if not (method == DENSE and k == 16):
                check_spectrum(gpu, seq, k, want, what, **kw)
    if k == 1:   # a prefix longer than k is the reference's error, on every path
        for _, method, exact in METHODS:
            with pytest.raises(DnaError, match="Prefix length cannot exceed kmer length") as e:
                gpu.count(seq, 1, prefix="AC", method=method, exact=exact)
            assert e.value.code == 2
    seq.free()


@pytest.mark.parametrize("k", [1, 4, 7, 8, 12, 13, 16, 17, 31, 32])
def test_key_list_every_method(gpu, k):
    """dnagpu_count_keys: count_dense_keys (DENSE up to k = 16, and AUTO for small k), count_hash_keys (HASH, and
    DENSE past k = 16) and the partition pipeline from keys, rows against numpy.unique."""
    rng = np.random.default_rng(k)
    keys = rng.choice(distinct_keys(rng, min(4**k, 50_000), k), size=150_000)
    if k == 32:
        keys[:3] = np.uint64(M64)
    stats, kmers, counts = oracle_keys(keys)
    dev = device(keys)
    for mname, method, _ in METHODS[:4]:
        (st, table), got = profiled(gpu, lambda: gpu.count_keys(dev, k, table=True, method=method))
        check_rows(st, table, stats, kmers, counts, (k, mname))
        check_path(got, expected_path(k, keys.size, method, False, 0, keys=True), (k, mname))


def test_no_rows_launches_nothing(gpu):
    """count_any with n = 0 rows (the sequence is shorter than k): empty result, no kernel, on every path."""
    seq = gpu.upload(Dna("ACGTACG"))
    for _, method, exact in METHODS:
        for prefix in (None, "AC"):
            (st, table), got = profiled(gpu, lambda: gpu.count(seq, 8, prefix=prefix, table=True, method=method,
                                                               exact=exact))
            assert (st.total, st.distinct, st.unique) == (0, 0, 0) and table.rows == 0
            table.free()
            check_path(got, {}, (method, prefix))
    seq.free()


# ---- the n / 2 rule and the collect retry -----------------------------------------------------------
@pytest.mark.parametrize("rows", [100_000, 100_001])
@pytest.mark.parametrize("k", [1, 31])
def test_half_the_rows_is_counted_from_the_list(gpu, k, rows):
    """count_any: a clause that keeps n_match <= n / 2 rows is counted from the collected list (HASH:
    count_hash_keys); one row more and HASH runs the fused filtered insert (count_hash after filter_collect), while
    PARTITION still counts the list.  `^@ 'A'` keeps exactly the rows whose first base is A."""
    rng = np.random.default_rng(rows + k)
    n = rows + k - 1
    for n_match in (rows // 2, rows // 2 + 1):
        codes = rng.integers(1, 4, size=n).astype(np.uint8)           # T, C, G
        codes[rng.choice(rows, size=n_match, replace=False)] = 0      # A at exactly n_match row starts
        words = pack_bases(codes)
        want = R.count_query(words, 1, n, words.size, k, prefix=R.kmer_make("A"), faithful=False)
        assert want.total == n_match
        seq = gpu.upload(Dna.from_words(words, n))
        fused = n_match > rows // 2
        for method in (HASH, AUTO, PART) if k == 31 else (HASH, PART):
            what = (k, rows, n_match, method)
            (st, table), got = profiled(gpu, lambda: gpu.count(seq, k, prefix="A", table=True, method=method))
            check_rows(st, table, want.stats, want.kmers, want.counts, what)
            if method == PART:
                check_path(got, {"filter_collect": 1, "count_buckets": 1}, what)
            else:
                check_path(got, {"filter_collect": 1, "count_hash" if fused else "count_hash_keys": 1}, what)
            check_spectrum(gpu, seq, k, want, what, prefix="A", method=method)
        seq.free()


@pytest.mark.parametrize("layout", ["single", "reads"])
def test_collect_retry_past_the_first_buffer(gpu, layout):
    """count_any's second predicate scan: with n >= 2^23 rows the first collect buffer holds n / 8 rows; a clause
    that keeps more (`^@ 'A'`: ~1/4, `N...NB`: ~3/4) overflows it, and the exactly sized rescan runs
    (filter_collect launched twice).  Then the listed count (AUTO: PARTITION; HASH at ~1/4: count_hash_keys) or the
    fused insert (HASH at ~3/4: count_hash)."""
    k = 31
    if layout == "single":
        n_bases = 9_000_030
        words = R.synth_seq(23, n_bases)
        seq = gpu.upload(Dna.from_words(words, n_bases))
        args = (words, 1, n_bases, words.size)
    else:
        n_reads, bpr, stride = 75_000, 150, 5
        words = R.synth_reads(23, n_reads, bpr, stride)
        seq = gpu.upload_reads(words, n_reads, bpr, stride)
        args = (words, n_reads, bpr, stride)
    n = gpu.count(seq, k)[0].total
    assert n == 9_000_000
    for prefix, pattern in (("A", None), (None, "N" * 30 + "B")):
        want = R.count_query(*args, k, prefix=R.kmer_make(prefix) if prefix else None, pattern=pattern,
                             faithful=False, threads=8)
        assert n // 8 < want.total < n
        for method in (AUTO, HASH):
            what = (layout, prefix, pattern, method)
            (st, table), got = profiled(gpu, lambda: gpu.count(seq, k, prefix=prefix, pattern=pattern, table=True,
                                                               method=method))
            check_rows(st, table, want.stats, want.kmers, want.counts, what)
            check_path(got, expected_path(k, n, method, True, want.total), what)
            assert got["filter_collect"] == 2, (what, got)
        check_spectrum(gpu, seq, k, want, (layout, prefix, pattern), prefix=prefix, pattern=pattern, method=HASH)
    seq.free()


# ---- the HBM hash table at capacity -----------------------------------------------------------------
# cap = max(1024, floor(expected_keys / load) + 1), load clamped to [0.05, 0.95] (0 = the default 0.5)
@pytest.mark.parametrize("expected_keys,load_factor,cap", [(1, 0.0, 1024), (1000, 0.95, 1053), (1000, 2.0, 1053),
                                                           (1000, 0.01, 20001)])
def test_hash_table_exactly_full_and_one_key_too_many(gpu, expected_keys, load_factor, cap):
    """count_hash: cap distinct keys fill the table exactly, so probe runs cross the end of the table and wrap, and
    the rows are exact; cap + 1 distinct keys overflow it (DNAGPU_EINTERNAL), after which the context answers
    correctly.  As a key list (count_hash_keys) and as 32-base reads at k = 32 (count_hash, one k-mer per read)."""
    opts = dict(method=HASH, expected_keys=expected_keys, load_factor=load_factor)
    for seed in range(3):
        rng = np.random.default_rng(seed)
        distinct = distinct_keys(rng, cap + 1, 32)
        for n_distinct in (cap, cap + 1):
            keys = with_copies(rng, distinct[:n_distinct])
            stats, kmers, counts = oracle_keys(keys)
            dev = device(keys)
            reads = gpu.upload_reads(keys, keys.size, 32, 1)
            for what, call in (("keys", lambda: gpu.count_keys(dev, 32, table=True, **opts)),
                               ("reads", lambda: gpu.count(reads, 32, table=True, **opts))):
                what = (what, seed, n_distinct, expected_keys, load_factor)
                out, got = profiled(gpu, call, error=n_distinct > cap)
                check_path(got, {"count_hash_keys" if what[0] == "keys" else "count_hash": 1}, what)
                if n_distinct == cap:
                    check_rows(*out, stats, kmers, counts, what)
                else:
                    assert out.code == EINTERNAL, (what, out)
                    assert f"hash table of {cap} slots overflowed" in str(out), (what, out)
                    ordinary_query_is_right(gpu)
            reads.free()


def test_full_table_with_the_k32_sentinel(gpu):
    """'G' x 32 is the empty-slot marker and is counted on the side counter, not in a slot: 1024 distinct keys plus
    'G' x 32 fit the 1024-slot table (distinct = 1025)."""
    rng = np.random.default_rng(32)
    keys = np.concatenate([with_copies(rng, distinct_keys(rng, 1024, 32)), np.full(5, M64, dtype=np.uint64)])
    rng.shuffle(keys)
    stats, kmers, counts = oracle_keys(keys)
    assert stats[1] == 1025
    dev = device(keys)
    reads = gpu.upload_reads(keys, keys.size, 32, 1)
    for what, call in (("keys", lambda: gpu.count_keys(dev, 32, table=True, method=HASH, expected_keys=1)),
                       ("reads", lambda: gpu.count(reads, 32, table=True, method=HASH, expected_keys=1))):
        (st, table), got = profiled(gpu, call)
        check_rows(st, table, stats, kmers, counts, what)
        check_path(got, {"count_hash_keys" if what == "keys" else "count_hash": 1}, what)
    reads.free()


# ---- AUTO: the boundaries of pick_method ------------------------------------------------------------
# pick_method also had a rule for DENSE at k = 13..16 below 2^21 rows when 4^k <= max(2^16, 8 n).  AUTO could not
# reach it: below 2^21 rows 8 n < 2^24 < 4^13.  It was removed; an explicit DENSE is the only way to those tables.
@pytest.mark.parametrize("k,n,kernel", [
    (7, 1, "count_dense_smem"), (8, 1, "count_dense"),             # 4^k <= 2^16: dense at any size
    (9, 32_767, "count_hash"), (9, 32_768, "count_dense"),         # 4^9 <= 8 n
    (12, (1 << 21) - 1, "count_hash"), (12, 1 << 21, "count_dense"),
    (13, (1 << 21) - 1, "count_hash"), (13, 1 << 21, "count_buckets"),
])
def test_auto_boundaries(gpu, k, n, kernel):
    """pick_method under AUTO at each threshold, one row apart: for a sequence of n rows and a key list of n keys."""
    rng = np.random.default_rng(n + k)
    n_bases = n + k - 1
    words = rand_words(rng, n_bases)
    want = R.count_query(words, 1, n_bases, words.size, k, faithful=False)
    assert want.total == n
    assert expected_path(k, n, AUTO, False, 0) == {kernel: 1}
    seq = gpu.upload(Dna.from_words(words, n_bases))
    (st, table), got = profiled(gpu, lambda: gpu.count(seq, k, table=True))
    check_rows(st, table, want.stats, want.kmers, want.counts, (k, n))
    check_path(got, {kernel: 1}, (k, n))
    keys = R.generate_kmers(words, n_bases, k, window=True)
    keys_kernel = {"count_dense_smem": "count_dense_keys", "count_dense": "count_dense_keys",
                   "count_hash": "count_hash_keys", "count_buckets": "count_buckets"}[kernel]
    (st, table), got = profiled(gpu, lambda: gpu.count_keys(device(keys), k, table=True))
    check_rows(st, table, want.stats, want.kmers, want.counts, (k, n, "keys"))
    check_path(got, {keys_kernel: 1}, (k, n, "keys"))
    if k == 13:
        # 3/4 kept (more than the first collect buffer's 2^20 rows): at 2^21 - 1 rows HASH runs the fused insert; at
        # 2^21 PARTITION counts the list, and the list (fewer than 2^21 keys) is counted by HASH
        pattern = "N" * 12 + "B"
        want = R.count_query(words, 1, n_bases, words.size, k, pattern=pattern, faithful=False)
        assert n // 2 < want.total < 1 << 21
        path = {"filter_collect": 2, "count_hash" if n < 1 << 21 else "count_hash_keys": 1}
        assert expected_path(k, n, AUTO, True, want.total) == path
        (st, table), got = profiled(gpu, lambda: gpu.count(seq, k, pattern=pattern, table=True))
        check_rows(st, table, want.stats, want.kmers, want.counts, (k, n, pattern))
        check_path(got, path, (k, n, pattern))
        check_spectrum(gpu, seq, k, want, (k, n, pattern), pattern=pattern)
    seq.free()


# ---- count_keys with DENSE and a key that is not a k-mer --------------------------------------------
def test_dense_key_list_rejects_a_key_that_is_not_a_kmer(gpu):
    """count_dense_keys flags a key >= 4^k: DNAGPU_EARG with the message, no table, and the context stays usable."""
    rng = np.random.default_rng(6)
    for k, bad in ((5, 4**5), (16, 1 << 32)):
        good = rng.integers(0, 4**k, size=10_000, dtype=np.uint64)
        keys = np.concatenate([good, np.array([bad], dtype=np.uint64)])
        rng.shuffle(keys)
        out, got = profiled(gpu, lambda: gpu.count_keys(device(keys), k, table=True, method=DENSE), error=True)
        assert out.code == EARG, (k, out)
        assert f"a key is not a {k}-mer (>= 4^k)" in str(out), (k, out)
        check_path(got, {"count_dense_keys": 1}, k)
        if k == 5:
            stats, kmers, counts = oracle_keys(good)
            st, table = gpu.count_keys(device(good), k, table=True, method=DENSE)
            check_rows(st, table, stats, kmers, counts, k)
        ordinary_query_is_right(gpu)
