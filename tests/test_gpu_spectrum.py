"""The k-mer abundance spectrum (dnagpu_count_spectrum / dnagpu_count_kmers_spectrum) against the CPU oracle.

The reference spectrum is the oracle's GROUP BY kmer binned as `SELECT least(count, H), count(*) ... GROUP BY 1`:
numpy.bincount(numpy.minimum(counts, H)).  Every case also checks sum(hist) == distinct, hist[0] == unique and that
the stats equal those of dnagpu_count on the same query.  The inputs are the ones the count tests use to reach the
rare paths of every count method: keys around the bin limits of the bucket count, a bucket passed on to the table
kernel whose table spills, optimistic partition regions that overflow and are redone, and the k = 32 'G' x 32 key."""
import numpy as np
import pytest
import torch

import dnagpu
from dnagpu import Dna, DnaError
from oracle import ref_cpu as R

pytestmark = pytest.mark.gpu

HS = [1, 2, 3, 15, 16, 17, 1000, 1 << 20]
METHODS = [("auto", {}), ("dense", {"method": dnagpu.COUNT_DENSE}), ("hash", {"method": dnagpu.COUNT_HASH}),
           ("partition", {"method": dnagpu.COUNT_PARTITION}),
           ("partition_exact", {"method": dnagpu.COUNT_PARTITION, "exact": True})]
M64 = (1 << 64) - 1
PART_MUL = 0xD6E8FEB86659FD93  # partition.cuh kPartMul: the partition digits are the top bits of x * kPartMul


def ref_hist(counts, H):
    counts = np.asarray(counts, dtype=np.uint64)
    return np.bincount(np.minimum(counts, np.uint64(H)).astype(np.int64), minlength=H + 1)[1:].astype(np.uint64)


def check_hist(st, hist, want_stats, want_counts, H, what=None):
    assert (st.total, st.distinct, st.unique) == tuple(want_stats), what
    assert hist.dtype == np.uint64 and hist.size == H, what
    assert np.array_equal(hist, ref_hist(want_counts, H)), what
    assert int(hist.sum()) == st.distinct, what
    if H >= 2:
        assert int(hist[0]) == st.unique, what


def spectrum(gpu, seq, k, H, **kw):
    """count_spectrum, checked against the stats of count on the same query"""
    st, hist = gpu.count_spectrum(seq, k, max_count=H, **kw)
    plain, _ = gpu.count(seq, k, **kw)
    assert (st.total, st.distinct, st.unique) == (plain.total, plain.distinct, plain.unique), (k, H, kw)
    return st, hist


def key_reads(gpu, keys):
    """one 32-base read per key (stride 1 word): at k = 32 the only k-mer of a read is its word"""
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    return gpu.upload_reads(keys, keys.size, 32, 1)


# ---- the two worked examples ----------------------------------------------------------------------
def test_kats(gpu):
    for dna, k, want in (("ATCGATCGATCGATCGACG", 5, {1: 2, 3: 3, 4: 1}), ("ACGTACGTACGTAG", 8, {1: 3, 2: 2})):
        for H in (4, 5, 1000):
            hist = dnagpu.kmer_spectrum(dna, k, max_count=H, ctx=gpu)
            got = {c + 1: int(v) for c, v in enumerate(hist) if v}
            assert got == {min(c, H): v for c, v in want.items()}, (dna, k, H)
        st, hist = gpu.count_kmers_spectrum(Dna(dna), k, max_count=3)
        assert int(hist.sum()) == st.distinct and int(hist[0]) == st.unique


# ---- every method, every k class, every bin limit -------------------------------------------------
@pytest.mark.parametrize("k", [1, 3, 7, 8, 12, 13, 16, 21, 31, 32])
def test_every_method_and_bin_limit(gpu, k):
    n = 150_001
    words = R.synth_seq(40 + k, n)                 # planted repeats + G x 64 / A x 64 windows
    seq = gpu.upload(Dna.from_words(words, n))
    want = R.count_query(words, 1, n, words.size, k, faithful=False)
    for name, kw in METHODS:
        for H in HS:
            st, hist = spectrum(gpu, seq, k, H, **kw)
            check_hist(st, hist, want.stats, want.counts, H, (k, name, H))
    seq.free()


# ---- layouts and WHERE clauses --------------------------------------------------------------------
def _clauses(k):
    pattern = "S" + "N" * (k - 2) + "W"
    return [("AC", None, False), (None, pattern, False), ("AC", pattern, False), ("AC", pattern, True),
            (None, pattern, True)]


@pytest.mark.parametrize("k", [5, 12, 21, 31])
def test_layouts_with_where_clauses(gpu, k):
    rng = np.random.default_rng(k)
    n = 300_000
    words = R.synth_seq(77, n)
    single = gpu.upload(Dna.from_words(words, n))
    n_reads, bpr, stride = 20_000, 150, 5
    reads = R.synth_reads(3, n_reads, bpr, stride)
    fixed = gpu.upload_reads(reads, n_reads, bpr, stride)
    lens = [int(x) for x in rng.integers(1, 400, size=300)] + [3, 9, 10, 11, 5000]
    dnas = []
    for m in lens:
        w = rng.integers(0, 2**64, size=(m + 31) // 32, dtype=np.uint64)
        if m % 32:
            w[-1] &= np.uint64((1 << (2 * (m % 32))) - 1)
        dnas.append(Dna.from_words(w, m))
    ragged = gpu.upload_ragged(dnas)
    for prefix, pattern, planes in [(None, None, False)] + _clauses(k):
        pk = R.kmer_make(prefix) if prefix else None
        cases = [("single", single, R.count_query(words, 1, n, words.size, k, prefix=pk, pattern=pattern, faithful=False)),
                 ("reads", fixed, R.count_query(reads, n_reads, bpr, stride, k, prefix=pk, pattern=pattern,
                                                faithful=False)),
                 ("ragged", ragged, R.count_ragged([(d.words, d.length) for d in dnas], k, prefix=pk, pattern=pattern,
                                                   faithful=False))]
        for name, seq, want in cases:
            for H in (2, 16, 1000):
                for mname, kw in METHODS[:4]:
                    st, hist = spectrum(gpu, seq, k, H, prefix=prefix, pattern=pattern, planes=planes, **kw)
                    check_hist(st, hist, want.stats, want.counts, H, (name, prefix, pattern, planes, mname, H))
    for s in (single, fixed, ragged):
        s.free()


# ---- the rare paths -------------------------------------------------------------------------------
def test_multiplicities_around_the_bin_limits(gpu):
    """k_count_buckets_bins holds at most 15 copies of a key in a bin and passes heavier buckets on to
    k_count_buckets: its cumulative spectrum and the table kernel's direct one must meet at every limit."""
    rng = np.random.default_rng(21)
    parts = [rng.integers(0, 2**64, size=2_600_000, dtype=np.uint64)]
    for copies, n_keys in ((2, 200_000), (3, 50_000), (7, 20_000), (14, 5_000), (15, 5_000), (16, 5_000),
                           (17, 5_000), (18, 2_000), (40, 2_000), (300, 300), (2000, 40), (3073, 3), (5000, 5)):
        parts.append(np.repeat(rng.integers(0, 2**64, size=n_keys, dtype=np.uint64), copies))
    keys = np.concatenate(parts)
    rng.shuffle(keys)
    seq = key_reads(gpu, keys)
    _, counts = np.unique(keys, return_counts=True)
    want = (keys.size, counts.size, int((counts == 1).sum()))
    for name, kw in METHODS:
        for H in HS:
            st, hist = spectrum(gpu, seq, 32, H, **kw)
            check_hist(st, hist, want, counts, H, (name, H))
    seq.free()


def test_passed_bucket_that_spills(gpu):
    """12 000 distinct keys that share the top 24 bits of the partition hash all land in one bucket: more keys than
    the shared-memory table has slots, so the table kernel spills into its HBM table.  Plus a few hot keys."""
    rng = np.random.default_rng(12)
    inv = pow(PART_MUL, -1, 1 << 64)
    top = 0x5A5A5A << 40
    crafted = np.array([((top | int(r)) * inv) & M64 for r in rng.choice(1 << 40, size=12_000, replace=False)],
                       dtype=np.uint64)
    hot = rng.integers(0, 2**64, size=5, dtype=np.uint64)
    keys = np.concatenate([np.repeat(crafted, rng.integers(1, 4, size=crafted.size)), np.repeat(hot, 100_000),
                           rng.integers(0, 2**64, size=3_000_000, dtype=np.uint64)])
    rng.shuffle(keys)
    seq = key_reads(gpu, keys)
    _, counts = np.unique(keys, return_counts=True)
    want = (keys.size, counts.size, int((counts == 1).sum()))
    for name, kw in METHODS:
        for H in (2, 3, 16, 1000, 1 << 20):
            st, hist = spectrum(gpu, seq, 32, H, **kw)
            check_hist(st, hist, want, counts, H, (name, H))
    seq.free()


def test_overflowing_partition_regions_are_counted_once(gpu):
    """Poly-A / poly-G runs overflow an optimistic level-1 region: the query is redone with the exact level 1, and the
    spectrum of the first attempt must not remain."""
    n = 6_000_003
    words = R.synth_seq(55, n)
    words[10_000:70_000] = 0
    words[100_000:130_000] = np.uint64(M64)
    seq = gpu.upload(Dna.from_words(words, n))
    for k in (21, 31, 32):
        want = R.count_query(words, 1, n, words.size, k, faithful=False, threads=8)
        for H in (2, 17, 10_000, 1 << 20):
            for name, kw in (METHODS[0], METHODS[3], METHODS[4]):
                st, hist = spectrum(gpu, seq, k, H, **kw)
                check_hist(st, hist, want.stats, want.counts, H, (k, name, H))
        st, hist = gpu.count_kmers_spectrum(Dna.from_words(words, n), k, max_count=1000)
        check_hist(st, hist, want.stats, want.counts, 1000, (k, "host"))
    seq.free()
    poly = gpu.upload(Dna("A" * 3_000_000))
    for H in (1, 2, 10_000, 1 << 20):
        st, hist = spectrum(gpu, poly, 31, H, method=dnagpu.COUNT_PARTITION)
        check_hist(st, hist, (3_000_000 - 30, 1, 0), [3_000_000 - 30], H, H)
    poly.free()


def test_k32_sentinel(gpu):
    """'G' x 32 has the bit pattern of the tables' EMPTY marker and is counted aside: one group of its own."""
    for s in ("G" * 32, "G" * 40 + "ACGT" * 20 + "G" * 33, "ACGT" * 20, "G" * 100_000 + "ACGT" * 50 + "G" * 40):
        words, n = R.encode_dna(s)
        want = R.count_query(words, 1, n, words.size, 32)
        seq = gpu.upload(Dna(s))
        for name, kw in METHODS:
            for H in (1, 2, 11, 12, 1000, 1 << 20):
                st, hist = spectrum(gpu, seq, 32, H, **kw)
                check_hist(st, hist, want.stats, want.counts, H, (s[:50], name, H))
        seq.free()


def test_empty_and_tiny_inputs(gpu):
    st, hist = gpu.count_kmers_spectrum(Dna("ACG"), 5, max_count=4)
    assert (st.total, st.distinct, st.unique) == (0, 0, 0) and not hist.any()
    st, hist = gpu.count_kmers_spectrum(Dna("ACGTACGT"), 4, prefix="GG", max_count=4)   # WHERE keeps nothing
    assert (st.total, st.distinct, st.unique) == (0, 0, 0) and not hist.any()
    st, hist = gpu.count_kmers_spectrum(Dna("A"), 1, max_count=1)
    assert hist.tolist() == [1]


# ---- owner shares ---------------------------------------------------------------------------------
def _pieces(words, n, cuts):
    bounds = [0] + list(cuts) + [n]
    tensors, first, starts = [], [], []
    n_words = (n + 31) // 32
    for a, b in zip(bounds[:-1], bounds[1:]):
        w0, w1 = a // 32, min(n_words, (b + 31 + 31) // 32)
        piece = np.concatenate([words[w0:w1], np.zeros(3, np.uint64)])
        if len(piece) % 2:
            piece = np.concatenate([piece, np.zeros(1, np.uint64)])
        tensors.append(torch.from_numpy(piece.view(np.int64)).cuda())
        first.append(a)
        starts.append(b - a)
    return tensors, first, starts


@pytest.mark.parametrize("G", [2, 3, 4, 8])
@pytest.mark.parametrize("k", [14, 31, 32])
def test_owner_shares_add_up(gpu, G, k):
    n, seed, H = 3_000_000, 5, 1000     # seed 5 contains 'G' x 32
    words = R.synth_seq(seed, n)
    seq = gpu.synth(n, seed)
    st0, whole = gpu.count_spectrum(seq, k, max_count=H)
    want = R.count_query(words, 1, n, words.size, k, faithful=False, threads=8)
    check_hist(st0, whole, want.stats, want.counts, H, k)
    total = np.zeros(H, dtype=np.uint64)
    for part in range(G):
        st, hist = spectrum(gpu, seq, k, H, owner=(G, part))
        assert int(hist.sum()) == st.distinct
        total += hist
    assert np.array_equal(total, whole)
    seq.free()
    tensors, first, starts = _pieces(words, n, [32 * 20_000, 32 * 41_000, 32 * 70_000])
    torch.cuda.synchronize()
    total[:] = 0
    P = len(tensors)
    for part in range(G):
        ring = [(part + i) % P for i in range(P)]
        pseq = gpu.wrap_pieces([tensors[i].data_ptr() for i in ring], [first[i] for i in ring],
                               [starts[i] for i in ring], n, keep=tensors)
        st, hist = spectrum(gpu, pseq, k, H, owner=(G, part))
        total += hist
        pseq.free()
    assert np.array_equal(total, whole)


def _n_gpus():
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.skipif(_n_gpus() < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("k", [13, 31, 32])
def test_multi_gpu_context_equals_one_gpu(gpu, k):
    n, H = 5_000_000, 10_000
    words = R.synth_seq(5, n)
    dna = Dna.from_words(words, n)
    st1, want = gpu.count_kmers_spectrum(dna, k, max_count=H)
    ctx = dnagpu.Context(devices=list(range(min(_n_gpus(), 8))))
    st, hist = ctx.count_kmers_spectrum(dna, k, max_count=H)
    ctx.close()
    assert (st.total, st.distinct, st.unique) == (st1.total, st1.distinct, st1.unique)
    assert np.array_equal(hist, want)


# ---- full size ------------------------------------------------------------------------------------
def test_full_size_config3(gpu):
    """BASELINE configs[3]: 3.1 Gbp, k = 31.  The aggregates against the oracle's golden answer, and the whole
    spectrum against a bincount of the device counts of the same query's table (a path that shares no spectrum
    code)."""
    import json
    import os
    from conftest import ROOT
    with open(os.path.join(ROOT, "tests", "golden", "big_expected.json")) as f:
        e = json.load(f)["c4"]
    H = 10_000
    seq = gpu.synth(e["n_bases"], e["seed"], e["repeat_every"])
    st, hist = gpu.count_spectrum(seq, e["k"], max_count=H)
    assert (st.total, st.distinct, st.unique) == (e["total"], e["distinct"], e["unique"])
    assert int(hist.sum()) == e["distinct"] and int(hist[0]) == e["unique"]
    st2, table = gpu.count(seq, e["k"], table=True)
    seq.free()
    assert table.rows == e["distinct"]
    _, counts_addr = table.device_pointers()
    d_counts = dnagpu._device_view(counts_addr, table.rows, gpu.device)
    want = torch.bincount(torch.clamp(d_counts, max=H), minlength=H + 1)[1:].cpu().numpy().astype(np.uint64)
    del d_counts
    table.free()
    assert np.array_equal(hist, want)


def test_kmer_with_more_than_2e32_copies(gpu):
    """S1 . A^m . S2 with ~ 2^32 + 2^20 copies of A^31: count(X) = count(S1 . A^64 . S2) + (m - 64) copies of A^31
    (the small twin has the same S1 and S2 words).  The key lands in the last bin; the passed-on bucket runs the
    64-bit k_count_buckets."""
    if gpu.device_info()["hbm_total"] < 90 * (1 << 30):
        pytest.skip("a GROUP BY of a 4.3e9-copy k-mer needs about 90 GiB of device memory")
    k, H = 31, 10_000
    rng = np.random.default_rng(3)
    w1 = rng.integers(0, 2**64, size=1000, dtype=np.uint64)
    w2 = rng.integers(0, 2**64, size=1000, dtype=np.uint64)
    m = (1 << 32) + (1 << 20) + k - 1
    m += (-m) % 32
    small = np.concatenate([w1, np.zeros(2, np.uint64), w2])
    n_small = small.size * 32
    want = R.count_query(small, 1, n_small, small.size, k, faithful=False)
    key = 0  # A^31
    i = int(np.searchsorted(want.kmers, np.uint64(key)))
    assert want.kmers[i] == key
    counts = want.counts.copy()
    counts[i] += np.uint64(m - 64)
    stats = (want.total + m - 64, want.distinct, want.unique)
    big = np.zeros(w1.size + m // 32 + w2.size, dtype=np.uint64)
    big[:w1.size] = w1
    big[w1.size + m // 32:] = w2
    dna = Dna.from_words(big, big.size * 32)
    del big
    seq = gpu.upload(dna)
    del dna
    st, hist = gpu.count_spectrum(seq, k, max_count=H)
    seq.free()
    check_hist(st, hist, stats, counts, H)
    assert int(hist[H - 1]) >= 1


# ---- errors ---------------------------------------------------------------------------------------
def test_errors(gpu):
    seq = gpu.upload(Dna("ACGTACGTAC"))
    for H in (0, (1 << 20) + 1):
        with pytest.raises(DnaError, match="max_count must be between 1 and 1048576") as e:
            gpu.count_spectrum(seq, 3, max_count=H)
        assert e.value.code == 20
        with pytest.raises(DnaError, match="max_count must be between 1 and 1048576"):
            gpu.count_kmers_spectrum(Dna("ACGTACGTAC"), 3, max_count=H)
    rc = gpu.lib.dnagpu_count_spectrum(gpu.handle, seq.handle, 3, None, None, 10, None, None)
    assert rc == 20
    words = np.zeros(1, dtype=np.uint64)
    rc = gpu.lib.dnagpu_count_kmers_spectrum(gpu.handle, words.ctypes.data, 10, 3, None, 10, None, None)
    assert rc == 20
    with pytest.raises(DnaError, match="Invalid k value: must be between 1 and 32"):
        gpu.count_spectrum(seq, 0, max_count=10)
    with pytest.raises(DnaError, match="Invalid k value: must be between 1 and 32"):
        gpu.count_kmers_spectrum(Dna("ACGTACGTAC"), 0, max_count=10)
    with pytest.raises(DnaError, match="Invalid character in qkmer pattern: X"):
        gpu.count_spectrum(seq, 3, pattern="NXN", max_count=10)
    with pytest.raises(DnaError, match="Qkmer pattern and kmer lengths do not match"):
        gpu.count_spectrum(seq, 3, pattern="NNNN", max_count=10)
    seq.free()
