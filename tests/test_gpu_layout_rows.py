"""The calls that return rows, on every input layout, against the CPU oracle.

These calls are generate_kmers (dnagpu_extract), its ordered WHERE scan (dnagpu_filter), the unordered collect
(dnagpu_collect), owner bucketing (dnagpu_partition), the shuffle send of the multi-GPU GROUP BY (dnagpu_shuffle_*)
and the seq scan over a stored kmer column (dnagpu_filter_keys).  Each kernel behind the first five is a template
over the layout of its input: one sequence (kSingle), fixed-stride reads (kFixed) or a ragged batch of values
(kRagged), and each layout finds a row's words with its own arithmetic.  The layouts here sit on the edges of that
arithmetic:

- single: lengths around a packed word (32 bases) and a Shift-And run (128 starts + k - 1 bases), and 2 * 10^5 bases
  with 'G' x 64 and 'A' x 64 planted;
- limit: one sequence with a start limit (dnagpu_seq_set_start_limit) of 1, 31, 32, 33, 127, 128, 129 and n - 1 rows;
- reads: 1 to 129 rows per read, at a stride of the read's words and wider (the words in between hold garbage), and
  reads shorter than k;
- ragged: values shorter than k at the start, in the middle and at the end, a 5003-base value among short ones,
  a batch of values all shorter than k, and a single value;
- ragged_abi: a ragged batch uploaded through the C ABI with word_offsets that leave gaps of garbage, run in
  descending order and let two rows share one value's words.

The expected rows of a batch are the oracle's rows of each value, concatenated in value order: the row order of
generate_kmers over a table (test.sql:140-150).  A start limit of L keeps the k-mers that start in the first L
bases, i.e. the rows of the sequence cut to L + k - 1 bases.  Ordered results are compared as arrays, unordered ones
sorted, every comparison bit-exact.  The per-launch profile (dnagpu_profile_dump) shows which kernels each call
ran, and the alignment of the output view shows which store width dnagpu_extract used."""
import ctypes as C

import numpy as np
import pytest
import torch

import dnagpu
from dnagpu import Dna, DnaError
from dnagpu.distributed import owner_digits
from oracle import ref_cpu as R

pytestmark = pytest.mark.gpu

M64 = (1 << 64) - 1
EARG, ECAPACITY = 20, 21
SENT = -7            # fills output buffers around the rows: a word no call may write
LAYOUTS = ["single", "limit", "reads", "ragged", "ragged_abi"]
PARTS = [1, 2, 3, 4, 5, 8, 16, 64]
IUPAC_SET = {"A": 1, "T": 2, "C": 4, "G": 8, "U": 0, "W": 3, "S": 12, "M": 5, "K": 10, "R": 9, "Y": 6,
             "B": 14, "D": 11, "H": 7, "V": 13, "N": 15}   # bit = base code: A 00, T 01, C 10, G 11


# ---- helpers ----------------------------------------------------------------------------------------
def profiled(gpu, fn):
    """Run fn with per-launch profiling on -> (its result, {launch name: launches})."""
    gpu.profile(True)
    gpu.profile_reset()
    try:
        out = fn()
        names = {name: int(v["launches"]) for name, v in gpu.profile_dump().items()}
    finally:
        gpu.profile(False)
        gpu.profile_reset()
    return out, names


def host(t):
    return t.cpu().numpy().view(np.uint64)


def filled(n, value=SENT):
    """A device int64 buffer of n words holding `value`, ready before the library's stream touches it."""
    t = torch.full((n,), value, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    return t


def last_error(gpu):
    return gpu.lib.dnagpu_last_error(gpu.handle).decode()


def raw_rows(gpu, fn, seq, k, ptr, cap, prefix=None, pattern=None, planes=False):
    """dnagpu_extract / _filter / _collect through the C ABI -> (rc, *n_out)."""
    n = C.c_uint64(12345)
    if fn == "dnagpu_extract":
        rc = gpu.lib.dnagpu_extract(gpu.handle, seq.handle, k, ptr, cap, C.byref(n))
    else:
        w, _keep = dnagpu._where(prefix, pattern, planes)
        rc = getattr(gpu.lib, fn)(gpu.handle, seq.handle, k, C.byref(w) if w is not None else None, ptr, cap,
                                  C.byref(n))
    return rc, n.value


def words_of(n):
    return (n + 31) // 32


def val(rng, n, fill=None):
    """One dna value -> (words, n_bases): random bases, or all 'G' / all 'A'."""
    w = words_of(n)
    if fill == "G":
        words = np.full(w, M64, dtype=np.uint64)
    elif fill == "A":
        words = np.zeros(w, dtype=np.uint64)
    else:
        words = rng.integers(0, 2**64, size=w, dtype=np.uint64)
    return cut(words, n)


def cut(words, n):
    """The first n bases of a packed value (the bits past them zero, as dna_in leaves them)."""
    words = words[:words_of(n)].copy()
    if n % 32:
        words[-1] &= np.uint64((1 << (2 * (n % 32))) - 1)
    return words, n


def expect(values, k, prefix=None, pattern=None):
    """The oracle's rows of a batch: each value's rows, in value order."""
    if prefix is None and pattern is None:
        parts = [R.generate_kmers(w, n, k, window=True) for w, n in values]
    else:
        pk = R.kmer_make(prefix) if prefix else None
        parts = [R.filter_kmers(w, n, k, prefix=pk, pattern=pattern) for w, n in values]
    return np.concatenate(parts) if parts else np.zeros(0, dtype=np.uint64)


# ---- the layouts ------------------------------------------------------------------------------------
def single_cases(gpu, k):
    rng = np.random.default_rng(100 + k)
    cases = []
    for n in sorted({k, k + 1, 31, 32, 33, 63, 65, 126 + k, 127 + k, 128 + k, 200_003}):
        words, _ = val(rng, n)
        if n > 10_000:
            words[100:102] = np.uint64(M64)     # 'G' x 64
            words[200:202] = 0                  # 'A' x 64
        cases.append((f"single n={n}", gpu.upload(Dna.from_words(words, n)), [(words, n)]))
    return cases


def limit_cases(gpu, k):
    rng = np.random.default_rng(200 + k)
    n = 100_003
    words, _ = val(rng, n)
    words[50:52] = np.uint64(M64)
    cases = []
    for limit in (1, 31, 32, 33, 127, 128, 129, n - k):    # n - k = the rows of the sequence - 1
        seq = gpu.upload(Dna.from_words(words, n))
        seq.set_start_limit(limit)
        assert seq.kmer_count(k) == limit
        cases.append((f"limit {limit}", seq, [cut(words, limit + k - 1)]))
    return cases


def reads_batch(rng, n_reads, bases, extra):
    """n_reads reads of `bases` bases, `extra` words of garbage after each; read 0 is all 'G', read 1 all 'A'."""
    wpr = words_of(bases)
    stride = max(wpr + extra, 1)
    arr = rng.integers(0, 2**64, size=(n_reads, stride), dtype=np.uint64)
    values = [val(rng, bases, "G" if r == 0 else "A" if r == 1 else None) for r in range(n_reads)]
    for r, (w, _) in enumerate(values):
        arr[r, :wpr] = w
    return arr.reshape(-1), stride, values


# (rows per read, reads, garbage words after each read): total rows = 1, 2, 0, 1, 0, 3, 1 mod 4; 1295 items in the
# 259-read batches of 129 rows (5 items a read), not a multiple of 256
READS = [(1, 257, 0), (31, 258, 2), (32, 257, 0), (33, 257, 1), (128, 259, 0), (129, 259, 3), (129, 2001, 0),
         (0, 300, 1)]


def reads_cases(gpu, k):
    rng = np.random.default_rng(300 + k)
    cases = []
    for rows, n_reads, extra in READS:
        bases = rows + k - 1
        words, stride, values = reads_batch(rng, n_reads, bases, extra)
        cases.append((f"reads {n_reads}x{bases} stride {stride}", gpu.upload_reads(words, n_reads, bases, stride),
                      values))
    return cases


def short_len(rng, k):
    return int(rng.integers(0, k))   # 0 .. k - 1 bases: no rows


def ragged_cases(gpu, k):
    rng = np.random.default_rng(400 + k)
    head = [short_len(rng, k), short_len(rng, k), k, k + 1, 31, 32, 33, 1, short_len(rng, k), short_len(rng, k),
            short_len(rng, k), 5003] + [int(x) for x in rng.integers(1, 200, size=150)] + [127 + k]
    tail = [short_len(rng, k), short_len(rng, k)]
    rows = sum(max(0, n - k + 1) for n in head + [40])
    cases = []
    for d in range(4):   # one value between head and tail brings the rows to each residue mod 4
        lens = head + [(d - rows) % 4 + 4 + k - 1] + tail
        values = [val(rng, n) for n in lens] + [val(rng, 40, "G")]
        values[-1], values[-3] = values[-3], values[-1]   # 'G' x 40 before the two short values at the end
        cases.append((f"ragged rows={d} mod 4", gpu.upload_ragged([Dna.from_words(*v) for v in values]), values))
    values = [val(rng, short_len(rng, k)) for _ in range(40)]
    cases.append(("ragged all shorter than k", gpu.upload_ragged([Dna.from_words(*v) for v in values]), values))
    values = [val(rng, 777)]
    cases.append(("ragged one value", gpu.upload_ragged([Dna.from_words(*v) for v in values]), values))
    return cases


def upload_ragged_abi(gpu, pool, offsets, lengths):
    offs = np.ascontiguousarray(offsets, dtype=np.uint64)
    n_bases = np.ascontiguousarray(lengths, dtype=np.uint64)
    pool = np.ascontiguousarray(pool, dtype=np.uint64)
    h = C.c_void_p()
    gpu._ok(gpu.lib.dnagpu_seq_upload_ragged(gpu.handle, pool.ctypes.data, offs.ctypes.data, n_bases.ctypes.data,
                                             offs.size, C.byref(h)))
    return dnagpu.Seq(gpu, h)


def ragged_abi_cases(gpu, k):
    """Values laid out in memory last row first, garbage words between them; rows 2 and 4 share one value's words,
    and so do rows 0 and 11."""
    rng = np.random.default_rng(500 + k)
    vals = [val(rng, n) for n in (300, short_len(rng, k), 5003, 77, k, 129 + k, 64, short_len(rng, k), 1000)]
    vals.append(val(rng, 40, "G"))
    row_value = [0, 1, 2, 3, 2, 4, 5, 6, 7, 8, 9, 0]
    pool = [rng.integers(0, 2**64, size=5, dtype=np.uint64)]
    at, where = 5, [0] * len(vals)
    for v in reversed(range(len(vals))):
        words, _ = vals[v]
        gap = rng.integers(0, 2**64, size=int(rng.integers(1, 4)), dtype=np.uint64)
        where[v] = at
        pool += [words, gap]
        at += words.size + gap.size
    assert where == sorted(where, reverse=True)
    seq = upload_ragged_abi(gpu, np.concatenate(pool), [where[v] for v in row_value], [vals[v][1] for v in row_value])
    return [("ragged through the C ABI", seq, [vals[v] for v in row_value])]


def build(gpu, layout, k):
    """-> [(label, seq, [(words, n_bases) per value])]"""
    cases = {"single": single_cases, "limit": limit_cases, "reads": reads_cases, "ragged": ragged_cases,
             "ragged_abi": ragged_abi_cases}[layout](gpu, k)
    for _, seq, _ in cases:
        # the first call for a k builds a ragged batch's row offsets (launches ragged_rows and scan); a count-only
        # extraction does it here, so that the profiles of the tests show each call's own launches
        assert raw_rows(gpu, "dnagpu_extract", seq, k, None, 0)[0] in (0, ECAPACITY)
    return cases


def free(cases):
    for _, seq, _ in cases:
        seq.free()


def clauses(k, values):
    """(name, prefix, pattern): ~1/4 and ~1/16 kept by a prefix, a prefix of length k (equality with a k-mer of the
    input), a sparse IUPAC pattern, N...NB (~3/4 kept: a tile's staging area nearly full), U (nothing) and none."""
    big = max(values, key=lambda v: v[1], default=None)
    eq = "A" * k
    if big is not None and big[1] >= k:
        eq = R.decode_kmer(int(R.generate_kmers(*big, k, window=True)[0]), k)
    sparse = ["N"] * k
    sparse[0] = "A"
    if k > 1:
        sparse[-1] = "K"
    if k > 2:
        sparse[k // 2] = "S"
    out = [("none", None, None), ("A", "A", None)]
    if k >= 2:
        out.append(("AC", "AC", None))
    return out + [("equal", eq, None), ("sparse", None, "".join(sparse)), ("3/4", None, "N" * (k - 1) + "B"),
                  ("U", None, "U" + "N" * (k - 1))]


def forms(layout):
    """Single sequences and reads run the Shift-And scan by default and the plane test on request; ragged
    batches always run the plane test."""
    return (False,) if layout.startswith("ragged") else (False, True)


# ---- A. extraction, both store widths ---------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 2, 15, 16, 17, 31, 32])
@pytest.mark.parametrize("layout", LAYOUTS)
def test_extract_both_store_widths(gpu, layout, k):
    """dnagpu_extract into a fresh tensor (32-byte aligned: k_extract4, four rows per 32-byte store) and into a view
    at a 16-byte offset (k_extract, two rows per 16-byte store), with every row count mod 4.  The words around the
    rows keep their sentinel.  An 8-byte offset is DNAGPU_EARG and a short buffer DNAGPU_ECAPACITY with the need,
    both before any launch."""
    cases = build(gpu, layout, k)
    mods = set()
    for label, seq, values in cases:
        want = expect(values, k)
        n = want.size
        what = (label, k)
        assert seq.kmer_count(k) == n, what
        mods.add(n % 4)
        out, got = profiled(gpu, lambda: gpu.extract(seq, k))
        assert out.data_ptr() % 32 == 0, what
        assert np.array_equal(host(out), want), what
        assert got == ({"extract": 1} if n else {}), (what, got)

        buf = filled(n + 6)
        view = buf[2:]
        assert view.data_ptr() % 32 == 16, what
        res, got = profiled(gpu, lambda: gpu.extract(seq, k, out=view))
        assert res.numel() == n and (n == 0 or res.data_ptr() == view.data_ptr()), what
        h = host(buf)
        assert np.array_equal(h[2:2 + n], want), what
        assert (h[:2].view(np.int64) == SENT).all() and (h[2 + n:].view(np.int64) == SENT).all(), what
        assert got == ({"extract": 1} if n else {}), (what, got)
        if n == 0:
            continue
        buf = filled(n + 6)
        (rc, need), got = profiled(gpu, lambda: raw_rows(gpu, "dnagpu_extract", seq, k, buf[1:].data_ptr(), n + 5))
        assert rc == EARG and "16-byte aligned" in last_error(gpu) and got == {}, (what, rc, got)
        for ptr, cap in ((buf[2:].data_ptr(), n - 1), (None, 0)):
            (rc, need), got = profiled(gpu, lambda: raw_rows(gpu, "dnagpu_extract", seq, k, ptr, cap))
            assert rc == ECAPACITY and need == n and got == {}, (what, cap, rc, need, got)
        gpu.synchronize()
        assert (host(buf).view(np.int64) == SENT).all(), what
    if layout in ("single", "reads", "ragged"):
        assert mods == {0, 1, 2, 3}, (layout, k, mods)
    free(cases)


# ---- B. the ordered WHERE scan ----------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 2, 16, 31, 32])
@pytest.mark.parametrize("layout", LAYOUTS)
def test_filter_ordered_rows(gpu, layout, k):
    """dnagpu_filter: the kept rows in oracle order for every clause, with the Shift-And scan and the plane test
    (k_filter_count + k_filter_write; ragged batches only take the plane test); the count-only call
    (NULL d_out) gives their number.  No clause falls through to extraction."""
    cases = build(gpu, layout, k)
    for label, seq, values in cases:
        n = seq.kmer_count(k)
        for cname, prefix, pattern in clauses(k, values):
            want = expect(values, k, prefix, pattern)
            if cname == "U":
                assert want.size == 0
            for planes in forms(layout):
                what = (label, k, cname, planes)
                out, got = profiled(gpu, lambda: gpu.filter(seq, k, prefix=prefix, pattern=pattern, planes=planes))
                assert np.array_equal(host(out), want), what
                if n == 0:
                    assert got == {}, (what, got)
                elif cname == "none":
                    assert got == {"extract": 1}, (what, got)
                else:
                    assert got.get("filter_count", 0) >= 1 and "extract" not in got, (what, got)
                    assert got.get("filter_write", 0) == (1 if want.size else 0), (what, got)
                rc, need = raw_rows(gpu, "dnagpu_filter", seq, k, None, 0, prefix, pattern, planes)
                assert rc == 0 and need == want.size, (what, rc, need)
    free(cases)


# ---- C. the unordered collect -----------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 16, 31, 32])
@pytest.mark.parametrize("layout", LAYOUTS)
def test_collect_unordered_rows_and_capacity(gpu, layout, k):
    """dnagpu_collect returns the rows of the ordered scan in any order.  A tile writes its rows only when they fit
    under cap, so: cap = the need succeeds; cap = need - 1 is DNAGPU_ECAPACITY with the need in *n_out and nothing
    written at or past cap; cap = 0 with a NULL buffer counts only."""
    cases = build(gpu, layout, k)
    for label, seq, values in cases:
        n = seq.kmer_count(k)
        for cname, prefix, pattern in clauses(k, values):
            want = np.sort(expect(values, k, prefix, pattern))
            for planes in forms(layout):
                what = (label, k, cname, planes)
                out, got = profiled(gpu, lambda: gpu.collect(seq, k, prefix=prefix, pattern=pattern, planes=planes))
                assert np.array_equal(np.sort(host(out)), want), what
                assert (got == {}) if n == 0 else got.get("filter_collect", 0) >= 1, (what, got)
                if cname not in ("none", "A", "3/4") or want.size == 0:
                    continue
                need = want.size
                buf = filled(need + 3)
                rc, m = raw_rows(gpu, "dnagpu_collect", seq, k, buf.data_ptr(), need, prefix, pattern, planes)
                gpu.synchronize()
                h = host(buf)
                assert rc == 0 and m == need, (what, rc, m)
                assert np.array_equal(np.sort(h[:need]), want), what
                assert (h[need:].view(np.int64) == SENT).all(), what
                buf = filled(need + 3)
                rc, m = raw_rows(gpu, "dnagpu_collect", seq, k, buf.data_ptr(), need - 1, prefix, pattern, planes)
                gpu.synchronize()
                assert rc == ECAPACITY and m == need, (what, rc, m)
                assert (host(buf)[need - 1:].view(np.int64) == SENT).all(), what
                rc, m = raw_rows(gpu, "dnagpu_collect", seq, k, None, 0, prefix, pattern, planes)
                assert rc == 0 and m == need, (what, rc, m)
    free(cases)


# ---- D. owner bucketing -----------------------------------------------------------------------------
_TAU = (0, 3, 6, 9, 13, 16, 19, 22, 26, 29)
_SUB = (0x06E, 0x2D1, 0x1B4)
_TAPS = [sum(1 << _TAU[p] for p in range(10) if sub >> p & 1) for sub in _SUB]


def owner_np(keys, n_parts):
    """owner_of (csrc/kernels.cuh) over a uint64 array: for 2, 4 and 8 parts bit i of the rank is the parity of the
    k-mer's low 32 bits under tap set i; otherwise the top bits of (low 32 bits * 0x85EBCA6B mod 2^32) * n_parts."""
    x = np.asarray(keys, dtype=np.uint64) & np.uint64(0xFFFFFFFF)
    lin = {2: 1, 4: 2, 8: 3}.get(n_parts, 0)
    if lin:
        r = np.zeros(x.shape, dtype=np.uint64)
        for i in range(lin):
            r |= (np.bitwise_count(x & np.uint64(_TAPS[i])).astype(np.uint64) & np.uint64(1)) << np.uint64(i)
        return r
    h = (x * np.uint64(0x85EBCA6B)) & np.uint64(0xFFFFFFFF)
    return (h * np.uint64(n_parts)) >> np.uint64(32)


def test_owner_of_port_matches_the_library(gpu):
    """The numpy owner_of used below agrees with dnagpu_owner_of on keys with and without high bits set."""
    rng = np.random.default_rng(7)
    keys = np.concatenate([np.array([0, M64, 1, 1 << 31, 1 << 32, (1 << 32) - 1, 1 << 63, M64 ^ 0xFFFFFFFF],
                                    dtype=np.uint64),
                           rng.integers(0, 2**64, size=2000, dtype=np.uint64),
                           rng.integers(0, 2**32, size=1000, dtype=np.uint64)])
    for n_parts in PARTS + [6, 7, 63]:
        want = np.array([dnagpu.owner_of(int(x), n_parts) for x in keys], dtype=np.uint64)
        assert np.array_equal(owner_np(keys, n_parts), want), n_parts
        assert want.max() < n_parts


def raw_partition(gpu, seq, k, n_parts, ptr, cap, prefix=None, pattern=None):
    counts = np.zeros(max(n_parts, 1) + 1, dtype=np.uint64)
    w, _keep = dnagpu._where(prefix, pattern)
    rc = gpu.lib.dnagpu_partition(gpu.handle, seq.handle, k, C.byref(w) if w is not None else None, n_parts, ptr, cap,
                                  counts.ctypes.data_as(dnagpu._lib.u64p))
    return rc, counts[:n_parts]


@pytest.mark.parametrize("k", [3, 17, 32])
@pytest.mark.parametrize("layout", LAYOUTS)
def test_partition_buckets_every_key(gpu, layout, k):
    """dnagpu_partition (k_partition_count + k_partition_write) with and without a clause: every key of bucket p is
    owned by p, bucket p is the multiset of the oracle's rows owned by p, and the counts equal the count-only call.
    n_parts 0 and 65 are DNAGPU_EARG; a short buffer is DNAGPU_ECAPACITY and stays unwritten."""
    cases = build(gpu, layout, k)
    for label, seq, values in cases:
        n = seq.kmer_count(k)
        for prefix, pattern in ((None, None), ("C", "N" * (k - 1) + "B")):
            want = expect(values, k, prefix, pattern)
            for n_parts in PARTS:
                what = (label, k, prefix, n_parts)
                (buf, counts), got = profiled(gpu, lambda: gpu.partition(seq, k, n_parts, prefix=prefix,
                                                                         pattern=pattern))
                own = owner_np(want, n_parts)
                assert np.array_equal(counts, np.bincount(own.astype(np.int64), minlength=n_parts)), what
                assert np.array_equal(counts, gpu.partition_counts(seq, k, n_parts, prefix=prefix, pattern=pattern))
                h = host(buf)
                h_own = owner_np(h, n_parts)
                assert np.array_equal(h_own, np.repeat(np.arange(n_parts, dtype=np.uint64), counts.astype(np.int64))), what
                o1, o2 = np.lexsort((h, h_own)), np.lexsort((want, own))
                assert np.array_equal(h[o1], want[o2]), what
                if n:
                    assert got.get("partition_count", 0) >= 1, (what, got)
                assert got.get("partition_write", 0) == (1 if want.size else 0), (what, got)
        if n:
            for bad in (0, 65):
                rc, _ = raw_partition(gpu, seq, k, bad, None, 0)
                assert rc == EARG and "n_parts must be between 1 and 64" in last_error(gpu), (label, bad)
            buf = filled(n + 2)
            rc, counts = raw_partition(gpu, seq, k, 5, buf.data_ptr(), n - 1)
            assert rc == ECAPACITY and int(counts.sum()) == n, (label, rc, counts)
            gpu.synchronize()
            assert (host(buf).view(np.int64) == SENT).all(), label
    free(cases)


# ---- E. the shuffle send on batches -----------------------------------------------------------------
def batch_blocks(gpu, layout, k, G):
    """A batch of reads or ragged values cut into G contiguous row blocks (one per rank) -> (values, seqs)."""
    rng = np.random.default_rng(600 + 10 * k + G)
    if layout == "reads":
        bases = 150
        words, stride, values = reads_batch(rng, 3001, bases, 1)
        cuts = [0, 1234, 3001] if G == 2 else [0, 1, 1700, 3001]   # G = 3: rank 0 holds read 0 ('G' x 150) alone
        seqs = [gpu.upload_reads(words[a * stride:b * stride], b - a, bases, stride) for a, b in zip(cuts, cuts[1:])]
        return values, seqs
    lens = [int(x) for x in rng.integers(0, 400, size=1200)] + [5003, 3, 0]
    values = [val(rng, n) for n in lens]
    for at, n in ((5, 40), (700, 33), (1100, 40)):
        values.insert(at, val(rng, n, "G"))
    cuts = [0, 600, len(values)] if G == 2 else [0, 2, 900, len(values)]
    seqs = [gpu.upload_ragged([Dna.from_words(*v) for v in values[a:b]]) for a, b in zip(cuts, cuts[1:])]
    return values, seqs


@pytest.mark.parametrize("k", [17, 32])
@pytest.mark.parametrize("G", [2, 3])
@pytest.mark.parametrize("layout", ["reads", "ragged"])
def test_shuffle_send_on_batches(gpu, layout, G, k):
    """G ranks emulated on one device, each holding a contiguous block of a batch: dnagpu_shuffle_send -> _count
    per owner (the owner's digit slices of every rank, peer-major), and dnagpu_shuffle_hist -> _scatter_to ->
    _count (stores straight into each owner's buffer).  The keys sent and received are the oracle's rows without
    'G' x 32, which goes to the side counter; tables, aggregates and side rows add up to the oracle's count."""
    values, seqs = batch_blocks(gpu, layout, k, G)
    n_rows = sum(s.kmer_count(k) for s in seqs)
    assert n_rows == expect(values, k).size
    for prefix, pattern in ((None, None), ("G", "N" * (k - 1) + "B")):
        what = (layout, G, k, prefix)
        want = R.count_ragged(values, k, prefix=R.kmer_make(prefix) if prefix else None, pattern=pattern,
                              faithful=False)
        rows = expect(values, k, prefix, pattern)
        n_side = int((rows == np.uint64(M64)).sum())
        assert (n_side > 0) == (k == 32), what   # 'G' x 32 passes both clauses
        rows = np.sort(rows[rows != np.uint64(M64)])
        plan = gpu.shuffle_plan(n_rows, G)
        ranges = [owner_digits(plan, o) for o in range(G)]

        sends, kept_all, side_all = [], 0, 0
        for seq in seqs:
            buf = torch.empty(seq.kmer_count(k) + 2, dtype=torch.int64, device="cuda")
            (counts, kept, side), got = profiled(gpu, lambda: gpu.shuffle_send(seq, k, plan, buf, prefix=prefix,
                                                                               pattern=pattern))
            assert got.get("part_hist") == 1 and got.get("part_scatter") == 1, (what, got)
            sends.append((buf, counts, np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)))
            kept_all += kept
            side_all += side
        assert (kept_all, side_all) == (want.total, n_side), what
        sent = np.concatenate([host(buf[:int(offs[-1])]) for buf, _, offs in sends])
        assert np.array_equal(np.sort(sent), rows), what
        tot, kk_all, cc_all = [0, 0, 0], [], []
        for lo, hi in ranges:
            pieces = [int(c) for _, counts, _ in sends for c in counts[lo:hi]]
            recv = torch.cat([buf[int(offs[lo]):int(offs[hi])] for buf, _, offs in sends])
            torch.cuda.synchronize()
            st, table = gpu.shuffle_count(recv, np.array(pieces, dtype=np.uint64), hi - lo, plan, k, table=True)
            assert st.total == sum(pieces), what
            tot = [tot[0] + st.total, tot[1] + st.distinct, tot[2] + st.unique]
            a, b = table.fetch()
            table.free()
            kk_all.append(a)
            cc_all.append(b)
        assert (tot[0] + side_all, tot[1] + (side_all > 0), tot[2] + (side_all == 1)) == want.stats, what
        kk, cc = np.concatenate(kk_all), np.concatenate(cc_all)
        if side_all:
            kk, cc = np.append(kk, np.uint64(M64)), np.append(cc, np.uint64(side_all))
        order = np.argsort(kk)
        assert np.array_equal(kk[order], want.kmers) and np.array_equal(cc[order], want.counts), what

        counts = np.stack([gpu.shuffle_hist(s, k, plan, prefix=prefix, pattern=pattern) for s in seqs])
        assert np.array_equal(counts, np.stack([c for _, c, _ in sends])), what
        recv = [filled(int(counts[:, a:b].sum()) + 2, -1) for a, b in ranges]   # -1 = 'G' x 32: never stored
        kept_all = side_all = 0
        for r, seq in enumerate(seqs):
            dest = np.zeros(plan.n_digits, dtype=np.uint64)
            for o, (a, b) in enumerate(ranges):
                block = counts[:, a:b]
                within = np.concatenate([[0], np.cumsum(block[r])[:-1]]).astype(np.uint64)
                dest[a:b] = np.uint64(recv[o].data_ptr()) + np.uint64(8) * (np.uint64(int(block[:r].sum())) + within)
            (kept, side), got = profiled(gpu, lambda: gpu.shuffle_scatter_to(seq, k, plan, dest, prefix=prefix,
                                                                             pattern=pattern))
            assert got.get("part_scatter_peer") == 1, (what, got)
            kept_all += kept
            side_all += side
        assert (kept_all, side_all) == (want.total, n_side), what
        got_rows = np.concatenate([host(t) for t in recv])
        assert np.array_equal(np.sort(got_rows[got_rows != np.uint64(M64)]), rows), what
        assert all(int((t == -1).sum()) == 2 for t in recv), what   # every slot written, the two pad words not
        distinct = unique = 0
        for o, (a, b) in enumerate(ranges):
            st = gpu.shuffle_count_addr(recv[o].data_ptr(), counts[:, a:b].reshape(-1), b - a, plan, k)
            distinct += st.distinct
            unique += st.unique
        assert (distinct + (side_all > 0), unique + (side_all == 1)) == (want.distinct, want.unique), what
    for s in seqs:
        s.free()


# ---- F. the seq scan over a stored kmer column ------------------------------------------------------
def keep_np(col, prefix, pattern):
    """WHERE kmer ^@ prefix AND pattern @> kmer over a column of k-mers, position by position."""
    keep = np.ones(col.size, dtype=bool)
    if prefix:
        pb, pl = R.kmer_make(prefix)
        keep &= (col & np.uint64(M64 if pl == 32 else (1 << (2 * pl)) - 1)) == np.uint64(pb)
    if pattern:
        for j, ch in enumerate(pattern):
            base = (col >> np.uint64(2 * j)) & np.uint64(3)
            keep &= ((np.uint64(IUPAC_SET[ch]) >> base) & np.uint64(1)).astype(bool)
    return keep


@pytest.mark.parametrize("k", [1, 2, 16, 31, 32])
def test_filter_keys_around_the_tile(gpu, k):
    """dnagpu_filter_keys (k_filter_keys_count + k_filter_keys_write, 2048-key tiles) on columns of 1, 2047, 2048,
    2049 and 3 * 2048 + 5 k-mers: rows in column order, the count-only call, DNAGPU_ECAPACITY with the need, and the
    reference's errors for a prefix or a pattern longer than k."""
    rng = np.random.default_rng(700 + k)
    sample = []
    for size in (1, 2047, 2048, 2049, 3 * 2048 + 5):
        col = rng.integers(0, 4**k if k < 32 else 2**64, size=size, dtype=np.uint64)
        if k == 32:
            col[::97] = np.uint64(M64)    # 'G' x 32: every bit set
        dev = torch.from_numpy(col.view(np.int64)).cuda()
        torch.cuda.synchronize()
        for cname, prefix, pattern in clauses(k, [(col[:1], k)]) + [("C + 3/4", "C", "N" * (k - 1) + "B")]:
            what = (k, size, cname)
            want = col[keep_np(col, prefix, pattern)]
            out, got = profiled(gpu, lambda: gpu.filter_keys(dev, k, prefix=prefix, pattern=pattern))
            assert np.array_equal(host(out), want), what
            if prefix or pattern:
                assert got.get("filter_keys_count", 0) >= 1, (what, got)
                assert got.get("filter_keys_write", 0) == (1 if want.size else 0), (what, got)
            w, _keep = dnagpu._where(prefix, pattern)
            wp = C.byref(w) if w is not None else None
            n = C.c_uint64()
            rc = gpu.lib.dnagpu_filter_keys(gpu.handle, dev.data_ptr(), size, k, wp, None, 0, C.byref(n))
            assert rc == 0 and n.value == want.size, (what, rc, n.value)
            if want.size:
                buf = filled(want.size + 2)
                rc = gpu.lib.dnagpu_filter_keys(gpu.handle, dev.data_ptr(), size, k, wp, buf.data_ptr(),
                                                want.size - 1, C.byref(n))
                assert rc == ECAPACITY and n.value == want.size, (what, rc, n.value)
                gpu.synchronize()
                assert (host(buf).view(np.int64) == SENT).all(), what
            if pattern and len(sample) < 400:
                sample.append((pattern, prefix, col[:40], keep_np(col[:40], prefix, pattern)))
        if k < 32:
            with pytest.raises(DnaError, match="Prefix length cannot exceed kmer length") as e:
                gpu.filter_keys(dev, k, prefix="A" * (k + 1))
            assert e.value.code == 2
            with pytest.raises(DnaError, match="Qkmer pattern and kmer lengths do not match") as e:
                gpu.filter_keys(dev, k, pattern="N" * (k + 1))
            assert e.value.code == 3
    for pattern, prefix, keys, keep in sample:   # the numpy predicate against the reference's functions
        pk = R.kmer_make(prefix) if prefix else None
        for x, kept in zip(keys, keep):
            ref = R.contains(pattern, int(x), k) and (pk is None or R.starts_with(int(x), k, *pk))
            assert ref == kept, (k, pattern, prefix, int(x))
