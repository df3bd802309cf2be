"""The bucket count without a hash table (k_count_buckets_bins) on the bucket shapes its look-back depends on.

The compare phase of that kernel stores no rank: a key is compared with the three slots before it in the staging
area whatever they hold, and with further ones, up to the start of its bin, only when the third holds a key of its
bin.  That is exact because
the bin and the bucket are both functions of the key, so a slot outside the key's bin -- another bin, another
warp's region, a stale key of an earlier bucket, the sentinel in front of the first bin -- never holds an equal key.

Every case here is a batch of 31-base reads, one k-mer per read, so that the k-mers, and with them the buckets and
the bins, are chosen exactly.  Each is counted with the partition method, plain and with the spectrum (counts 1..15
and "16 or more": the 15-copy limit of a bin), and compared with the CPU oracle.  The helpers restate the kernels'
hashes: the bucket is the top bits of part_hash (plan_bits: one level below 2^22 keys), the bin is bin_of; warp w
owns the bins 128 w .. 128 w + 127 and 1024 + 128 w .. + 127, staged in that order."""
import numpy as np
import pytest

import dnagpu
from oracle import ref_cpu as R

pytestmark = pytest.mark.gpu

K = 31
PART = dnagpu.COUNT_PARTITION
H = 16                   # spectrum bins 1 .. 15 and ">= 16"
BINS, WARPS = 2048, 8    # sub-bins of a bucket, warps of a CTA
CAP, HEAVY = 3072, 15    # keys a CTA stages, keys a bin holds
KPART = np.uint64(0xD6E8FEB86659FD93)


def bucket_bits(n):
    return max(1, min(22, int(np.ceil(np.log2(max(1, -(-n // 2048)))))))


def bucket_of(keys, b):
    return (keys * KPART) >> np.uint64(64 - b)


def bin_of(keys):
    h = (keys & np.uint64(0xFFFFFFFF)) ^ (keys >> np.uint64(32))
    return ((h * np.uint64(0x9E3779B1)) & np.uint64(0xFFFFFFFF)) >> np.uint64(21)


def warp_bins(w):
    return list(range(128 * w, 128 * w + 128)) + list(range(1024 + 128 * w, 1024 + 128 * w + 128))


class Pool:
    """Distinct random k-mers by (bucket, bin), each handed out once."""

    def __init__(self, rng, b, n=1 << 21):
        keys = np.unique(rng.integers(0, 1 << (2 * K), size=n, dtype=np.uint64))
        rng.shuffle(keys)
        self.keys = keys
        self.bucket, self.bin = bucket_of(keys, b), bin_of(keys)
        group = self.bucket * np.uint64(BINS) + self.bin
        self.order = np.argsort(group, kind="stable")
        self.start = np.searchsorted(group[self.order], np.arange((BINS << b) + 1, dtype=np.uint64))
        self.used = np.zeros(keys.size, dtype=bool)

    def take(self, n, bucket, avoid=()):
        """n keys of `bucket` in any bin but those in `avoid`"""
        ok = ~self.used & (self.bucket == np.uint64(bucket)) & ~np.isin(self.bin, np.asarray(avoid, dtype=np.uint64))
        return self._use(np.flatnonzero(ok)[:n], n)

    def in_bin(self, n, bucket, b):
        """n keys of `bucket` in bin b"""
        g = bucket * BINS + b
        idx = self.order[self.start[g]:self.start[g + 1]]
        return self._use(idx[~self.used[idx]][:n], n)

    def _use(self, idx, n):
        assert idx.size == n, "pool too small"
        self.used[idx] = True
        return self.keys[idx]


def copies_of(rng, keys, total):
    """keys repeated 1 to 3 times, `total` entries"""
    out = np.repeat(keys, rng.integers(1, 4, size=keys.size))[:total]
    assert out.size == total
    return out


def check(gpu, rng, keys):
    """count + count_spectrum of the reads `keys` (shuffled), method PARTITION, against the oracle"""
    keys = np.array(keys, dtype=np.uint64)
    rng.shuffle(keys)
    n = keys.size
    want = R.count_query(keys, n, K, 1, K, faithful=False)
    assert want.total == n
    seq = gpu.upload_reads(keys, n, K, 1)
    try:
        st, _ = gpu.count(seq, K, method=PART)
        assert (st.total, st.distinct, st.unique) == want.stats
        st, hist = gpu.count_spectrum(seq, K, max_count=H, method=PART)
        assert (st.total, st.distinct, st.unique) == want.stats
        counts = np.minimum(want.counts, np.uint64(H)).astype(np.int64)
        assert np.array_equal(hist, np.bincount(counts, minlength=H + 1)[1:].astype(np.uint64))
    finally:
        seq.free()
    return want


@pytest.mark.parametrize("size", [1, 4 * 256, 6 * 256, 8 * 256, CAP, CAP + 1])
def test_bucket_sizes(gpu, size):
    """One bucket of `size` keys, one per row count of BINS_DISPATCH; CAP + 1 keys are passed on.  The full buckets
    are balanced so that every warp's region is exactly full (bin b holds 1 + (b & 1) keys): they stay here."""
    rng = np.random.default_rng(size)
    pool = Pool(rng, 1)
    assert bucket_bits(size + 64) == 1
    if size >= CAP:
        keys = []
        for b in range(BINS):  # odd bins: one k-mer twice or two k-mers, in turn
            got = pool.in_bin(1 + (b & 1), 0, b)
            keys.append(np.repeat(got[:1], 2) if b % 4 == 1 else got)
        keys = np.concatenate(keys)
        assert keys.size == CAP
        assert all(np.isin(bin_of(keys), warp_bins(w)).sum() == CAP // WARPS for w in range(WARPS))
        if size > CAP:
            keys = np.concatenate([keys, keys[:1]])
    else:
        keys = copies_of(rng, pool.take(size, 0), size)
    keys = np.concatenate([keys, copies_of(rng, pool.take(64, 1), 64)])
    assert (bucket_of(keys, 1) == 0).sum() == size
    check(gpu, rng, keys)


@pytest.mark.parametrize("copies", [HEAVY, HEAVY + 1])
def test_heavy_key(gpu, copies):
    """A k-mer of 15 copies stays in the bin count (its last copy looks back 14 slots), one of 16 passes the bucket
    on.  The heavy keys sit in bin 0, the first bin of the stage (its first copies look back into the sentinel slots in
    front), and in bin 2047, the last one."""
    rng = np.random.default_rng(copies)
    pool = Pool(rng, 1)
    heavy = np.concatenate([pool.in_bin(1, 0, 0), pool.in_bin(1, 0, BINS - 1)])
    rest = copies_of(rng, pool.take(1200, 0, avoid=(0, BINS - 1)), 2000)
    keys = np.concatenate([np.repeat(heavy, [copies, HEAVY]), rest, copies_of(rng, pool.take(64, 1), 64)])
    want = check(gpu, rng, keys)
    assert int(want.counts.max()) == copies


def test_warp_region_boundaries(gpu):
    """Every warp's region exactly full, so that the regions abut: the last bin of warp w's region (1024 + 128 w +
    127) holds one k-mer 15 times, and the first bin of warp w + 1's region (128 (w + 1)) one k-mer 3 times.  The
    first keys of a region look back into the heavy bin before it, which must count nothing."""
    rng = np.random.default_rng(7)
    pool = Pool(rng, 1)
    keys = []
    for w in range(WARPS):
        bins = warp_bins(w)
        last, first = bins[-1], bins[0]
        keys.append(np.repeat(pool.in_bin(1, 0, last), HEAVY))
        keys.append(np.repeat(pool.in_bin(1, 0, first), 3))
        others = [b for b in bins if b not in (first, last)]
        doubles = CAP // WARPS - HEAVY - 3 - len(others)  # bins of two keys, the others get one
        for i, b in enumerate(others):
            got = pool.in_bin(1 + (i < doubles), 0, b)
            keys.append(got if i % 3 else np.repeat(got[:1], got.size))
    keys = np.concatenate(keys)
    assert keys.size == CAP
    assert all(np.isin(bin_of(keys), warp_bins(w)).sum() == CAP // WARPS for w in range(WARPS))
    keys = np.concatenate([keys, copies_of(rng, pool.take(64, 1), 64)])
    check(gpu, rng, keys)


def test_many_buckets_per_cta(gpu):
    """1024 buckets, more than the grid of the bin count (4 CTAs per SM), so every CTA counts several buckets and
    its stage holds the keys of earlier buckets.  Many k-mers repeat (up to 20 copies), so that look-backs past
    three slots are common and some buckets are passed on."""
    rng = np.random.default_rng(11)
    n_distinct = 600_000
    keys = np.unique(rng.integers(0, 1 << (2 * K), size=n_distinct + 1000, dtype=np.uint64))[:n_distinct]
    reps = np.where(rng.random(n_distinct) < 0.05, rng.integers(4, 21, size=n_distinct),
                    rng.integers(1, 4, size=n_distinct))
    keys = np.repeat(keys, reps)
    n = keys.size
    assert bucket_bits(n) == 10 and (1 << 10) > 148 * 4
    check(gpu, rng, keys)
