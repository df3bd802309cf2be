"""dnagpu -- Python face of libdnagpu, the B200 k-mer hot path of the `dna` extension.

The functions keep the names and argument meaning of the reference's SQL
surface (dna--1.0.sql): `generate_kmers(dna, k)` (dna.c:743-837), the `^@`
(`starts_with`, dna.c:842-866) and `@>` (`contains`, dna.c:1091-1135) operators
as WHERE clauses, and `GROUP BY kmer` + total/distinct/unique
(README.md:107-135).  All of the work happens in CUDA kernels behind the C ABI
in include/dnagpu.h; this package only marshals buffers.  Nothing here falls
back to the CPU: without the built library or without a B200 it raises.
"""
import ctypes as C
import weakref
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import CountOpts, ShufflePlan, Stats, Where
from .types import Dna, DnaError, Kmer, Qkmer, QKMER_ALPHABET, kmer_strings

COUNT_AUTO, COUNT_DENSE, COUNT_HASH, COUNT_PARTITION = 0, 1, 2, 3
COUNT_FLAG_EXACT = 1  # DNAGPU_COUNT_FLAG_EXACT: exact two-pass partition levels from the start
MAX_K = 32

__all__ = ["Context", "Seq", "Table", "Dna", "Kmer", "Qkmer", "DnaError", "KmerArray",
           "generate_kmers", "filter_kmers", "count_kmers", "kmer_stats", "kmer_spectrum", "owner_of",
           "default_context", "QKMER_ALPHABET"]


def _check(lib, ctx_handle, rc):
    if rc != 0:
        msg = lib.dnagpu_last_error(ctx_handle)
        raise DnaError((msg or lib.dnagpu_strerror(rc)).decode(), code=rc)


WHERE_FLAG_PLANES = 1  # DNAGPU_WHERE_FLAG_PLANES: the per-position plane test instead of the Shift-And automaton


def _where(prefix, pattern, planes=False):
    """(Kmer|str|None, Qkmer|str|None) -> (Where struct or None, keepalive)."""
    if prefix is None and pattern is None:
        return None, None
    w = Where()
    w.flags = WHERE_FLAG_PLANES if planes else 0
    keep = None
    if prefix is not None:
        prefix = Kmer(prefix)
        w.prefix_bits, w.prefix_len = prefix.bits, prefix.length
    if pattern is not None:
        keep = str(pattern).encode("ascii", "replace")  # validated by the library (dna.c:876-900)
        w.qkmer = keep
    return w, keep


@dataclass
class KmerArray:
    """Rows of kmers of one length k: `bits[i]` is Kmer.bit_sequence (dna.c:61-65)."""
    bits: np.ndarray
    k: int

    def __len__(self):
        return int(self.bits.size)

    def __iter__(self):
        return (Kmer(bits=int(b), length=self.k) for b in self.bits)

    def strings(self):
        return kmer_strings(self.bits, self.k)


class Seq:
    """Device-resident packed dna value(s)."""

    def __init__(self, ctx, handle, keep=None):
        self.ctx, self.handle, self._keep = ctx, handle, keep
        ctx._children.add(self)

    def kmer_count(self, k):
        return int(self.ctx.lib.dnagpu_seq_kmer_count(self.handle, k))

    @property
    def n_words(self):
        return int(self.ctx.lib.dnagpu_seq_words(self.handle))

    @property
    def device_ptr(self):
        return int(self.ctx.lib.dnagpu_seq_device_words(self.handle) or 0)

    def set_start_limit(self, n):
        _check(self.ctx.lib, self.ctx.handle, self.ctx.lib.dnagpu_seq_set_start_limit(self.handle, n))

    def download(self):
        out = np.empty(self.n_words, dtype=np.uint64)
        _check(self.ctx.lib, self.ctx.handle,
               self.ctx.lib.dnagpu_seq_download(self.ctx.handle, self.handle, out.ctypes.data, out.size))
        return out

    def free(self):
        if self.handle:
            self.ctx.lib.dnagpu_seq_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Table:
    """The grouped result of GROUP BY kmer: rows of (kmer, count), unordered."""

    def __init__(self, ctx, handle):
        self.ctx, self.handle = ctx, handle
        ctx._children.add(self)

    @property
    def rows(self):
        return int(self.ctx.lib.dnagpu_table_rows(self.handle))

    @property
    def k(self):
        return int(self.ctx.lib.dnagpu_table_k(self.handle))

    def fetch(self, offset=0, n=None):
        n = self.rows - offset if n is None else n
        kmers = np.empty(n, dtype=np.uint64)
        counts = np.empty(n, dtype=np.uint64)
        _check(self.ctx.lib, self.ctx.handle,
               self.ctx.lib.dnagpu_table_fetch(self.ctx.handle, self.handle, offset, n,
                                               kmers.ctypes.data, counts.ctypes.data))
        return kmers, counts

    def sorted(self):
        """(kmers, counts) ordered by kmer bits: how parity tests compare results."""
        kmers, counts = self.fetch()
        order = np.argsort(kmers, kind="stable")
        return kmers[order], counts[order]

    def device_pointers(self):
        a, b = C.c_void_p(), C.c_void_p()
        _check(self.ctx.lib, self.ctx.handle, self.ctx.lib.dnagpu_table_device(self.handle, C.byref(a), C.byref(b)))
        return int(a.value or 0), int(b.value or 0)

    def free(self):
        if self.handle:
            self.ctx.lib.dnagpu_table_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Index:
    """Sorted k-mer index over a stored kmer column (dnagpu_index_*): the SP-GiST replacement."""

    def __init__(self, ctx, handle):
        self.ctx, self.handle = ctx, handle
        ctx._children.add(self)

    @property
    def rows(self):
        return int(self.ctx.lib.dnagpu_index_rows(self.handle))

    @property
    def k(self):
        return int(self.ctx.lib.dnagpu_index_k(self.handle))

    def _rows_of(self, call):
        """Run a search: count first, then fetch into an exactly sized torch int64 CUDA tensor."""
        import torch
        n = C.c_uint64()
        self.ctx._ok(call(None, 0, C.byref(n)))
        out = torch.empty(max(int(n.value), 1), dtype=torch.int64, device=f"cuda:{self.ctx.device}")
        if n.value:
            self.ctx._ok(call(out.data_ptr(), out.numel(), C.byref(n)))
        self.ctx._before_torch()
        return out[:n.value]

    def equal(self, kmer):
        """WHERE kmer_sequence = kmer -> row numbers, ascending."""
        kmer = Kmer(kmer)
        return self._rows_of(lambda p, cap, n: self.ctx.lib.dnagpu_index_equal(self.ctx.handle, self.handle, kmer.bits,
                                                                               kmer.length, p, cap, n))

    def search(self, prefix=None, pattern=None):
        """WHERE kmer_sequence ^@ prefix AND pattern @> kmer_sequence -> row numbers, ascending."""
        w, _keep = _where(prefix, pattern)
        wp = C.byref(w) if w is not None else None
        return self._rows_of(lambda p, cap, n: self.ctx.lib.dnagpu_index_search(self.ctx.handle, self.handle, wp, p, cap, n))

    def sorted_column(self):
        """(sort keys ascending, row of each entry) as torch int64 CUDA tensors viewing the index's memory."""
        import torch
        a, b = C.c_void_p(), C.c_void_p()
        self.ctx._ok(self.ctx.lib.dnagpu_index_device(self.handle, C.byref(a), C.byref(b)))
        n = self.rows
        if n == 0:
            e = torch.empty(0, dtype=torch.int64, device=f"cuda:{self.ctx.device}")
            return e, e.clone()
        return _device_view(a.value, n, self.ctx.device), _device_view(b.value, n, self.ctx.device)

    def free(self):
        if self.handle:
            self.ctx.lib.dnagpu_index_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:  # noqa: BLE001 - interpreter shutdown
            pass


def _device_view(addr, n, device):
    """A torch int64 tensor over n u64 at a raw device address (no ownership)."""
    import torch

    class _Iface:
        __cuda_array_interface__ = {"shape": (int(n),), "typestr": "<i8", "data": (int(addr), False), "version": 3}
    return torch.as_tensor(_Iface(), device=f"cuda:{device}")


class Context:
    """One GPU, one stream (dnagpu_ctx).  `torch_stream=True` issues the library's
    work on torch's current stream so torch tensors can be passed in and out."""

    def __init__(self, device=0, torch_stream=False, devices=None):
        """devices=[d0, d1, ...]: one context over several GPUs of the box (dnagpu_create_multi): it behaves like a
        context on d0, and the host-buffer GROUP BY (count_kmers / count_kmers_ptr) uses all of them."""
        self.lib = _lib.load()
        self._children = weakref.WeakSet()  # live Seq / Table / Index objects (freed by close())
        h = C.c_void_p()
        if devices is not None:
            device = devices[0]
            rc = self.lib.dnagpu_create_multi(C.byref(h), (C.c_int * len(devices))(*devices), len(devices))
        else:
            rc = self.lib.dnagpu_create(C.byref(h), device)
        if rc != 0:
            raise DnaError(self.lib.dnagpu_last_error(None).decode(), code=rc)
        self.handle = h
        self.device = device
        self.shares_torch_stream = bool(torch_stream)
        if torch_stream:
            import torch
            with torch.cuda.device(device):
                s = torch.cuda.current_stream().cuda_stream
            # handle 0 is torch's legacy default stream; NULL would mean "the library's own stream", so lend
            # cudaStreamLegacy (0x1), which names the same stream explicitly
            _check(self.lib, self.handle, self.lib.dnagpu_set_stream(self.handle, C.c_void_p(s if s else 1)))

    def _after_torch(self):
        """Call before handing a torch tensor to the library: unless the ctx runs on torch's stream, whatever torch
        queued to produce the tensor (a copy from pageable memory, torch.cat, a fill) must have finished first."""
        if not self.shares_torch_stream:
            import torch
            torch.cuda.current_stream(self.device).synchronize()

    def _before_torch(self):
        """Call before returning a torch tensor the library wrote: unless the ctx runs on torch's stream, the
        kernel that fills it is still queued on the library's own (non-blocking) stream, which torch's streams do
        not order against."""
        if not self.shares_torch_stream:
            self.synchronize()

    def close(self):
        """dnagpu_destroy.  Seq / Table / Index objects that are still alive are freed first (their device memory
        belongs to the context); using them afterwards raises, dropping them is harmless."""
        if getattr(self, "handle", None):
            for child in list(getattr(self, "_children", ())):
                child.free()
            self.lib.dnagpu_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ok(self, rc):
        _check(self.lib, self.handle, rc)

    def synchronize(self):
        self._ok(self.lib.dnagpu_synchronize(self.handle))

    def device_info(self):
        name = C.create_string_buffer(128)
        sm, fr, tot = C.c_int(), C.c_uint64(), C.c_uint64()
        self._ok(self.lib.dnagpu_device_info(self.handle, name, 128, C.byref(sm), C.byref(fr), C.byref(tot)))
        return {"name": name.value.decode(), "sm_count": sm.value, "hbm_free": fr.value, "hbm_total": tot.value}

    # ---- inputs ---------------------------------------------------------------
    def upload(self, dna):
        dna = Dna(dna) if not isinstance(dna, Dna) else dna
        h = C.c_void_p()
        self._ok(self.lib.dnagpu_seq_upload(self.handle, dna.words.ctypes.data, dna.length, C.byref(h)))
        self.synchronize()  # dna.words may be freed by the caller afterwards
        return Seq(self, h)

    def upload_words(self, words_ptr, n_bases):
        """Upload from a raw host pointer (e.g. pinned memory); asynchronous."""
        h = C.c_void_p()
        self._ok(self.lib.dnagpu_seq_upload(self.handle, words_ptr, n_bases, C.byref(h)))
        return Seq(self, h)

    def upload_reads_ptr(self, words_ptr, n_reads, bases_per_read, stride_words):
        """Upload a fixed-stride batch from a raw host pointer (pinned memory); asynchronous."""
        h = C.c_void_p()
        self._ok(self.lib.dnagpu_seq_upload_reads(self.handle, words_ptr, n_reads, bases_per_read, stride_words,
                                                  C.byref(h)))
        return Seq(self, h)

    def upload_reads(self, words, n_reads, bases_per_read, stride_words):
        words = np.ascontiguousarray(words, dtype=np.uint64)
        h = C.c_void_p()
        self._ok(self.lib.dnagpu_seq_upload_reads(self.handle, words.ctypes.data, n_reads, bases_per_read,
                                                  stride_words, C.byref(h)))
        self.synchronize()
        return Seq(self, h)

    def upload_ragged(self, dnas):
        """A table of dna values of different lengths (rows of `dna_sequences`)."""
        dnas = [d if isinstance(d, Dna) else Dna(d) for d in dnas]
        n_bases = np.array([d.length for d in dnas], dtype=np.uint64)
        n_words = (n_bases + np.uint64(31)) // np.uint64(32)
        offs = np.zeros(len(dnas), dtype=np.uint64)
        if len(dnas) > 1:
            offs[1:] = np.cumsum(n_words)[:-1]
        words = (np.concatenate([d.words[:int(w)] for d, w in zip(dnas, n_words)])
                 if dnas else np.zeros(0, dtype=np.uint64))
        words = np.ascontiguousarray(words, dtype=np.uint64)
        h = C.c_void_p()
        self._ok(self.lib.dnagpu_seq_upload_ragged(self.handle, words.ctypes.data, offs.ctypes.data,
                                                   n_bases.ctypes.data, len(dnas), C.byref(h)))
        return Seq(self, h)

    def synth(self, n_bases, seed, repeat_every=8):
        h = C.c_void_p()
        self._ok(self.lib.dnagpu_seq_synth(self.handle, n_bases, seed, repeat_every, C.byref(h)))
        return Seq(self, h)

    def synth_range(self, n_bases_total, seed, repeat_every, first_base, n_starts, overlap_k):
        h = C.c_void_p()
        self._ok(self.lib.dnagpu_seq_synth_range(self.handle, n_bases_total, seed, repeat_every, first_base,
                                                 n_starts, overlap_k, C.byref(h)))
        return Seq(self, h)

    def synth_reads(self, first_read, n_reads, bases_per_read, stride_words, seed, repeat_every=8):
        h = C.c_void_p()
        self._ok(self.lib.dnagpu_seq_synth_reads(self.handle, first_read, n_reads, bases_per_read,
                                                 stride_words, seed, repeat_every, C.byref(h)))
        return Seq(self, h)

    def wrap(self, tensor, n_bases):
        """Borrow a torch int64/uint64 CUDA tensor holding packed words (+ >= 1 zero pad word)."""
        self._after_torch()
        h = C.c_void_p()
        self._ok(self.lib.dnagpu_seq_wrap(self.handle, tensor.data_ptr(), n_bases, tensor.numel(), C.byref(h)))
        return Seq(self, h, keep=tensor)

    def wrap_pieces(self, addrs, first_bases, n_starts, n_bases_total, keep=None):
        """One dna value resident as base-range pieces at raw device addresses (local or peer-mapped), walked in the
        order given: dnagpu_seq_wrap_pieces."""
        n = len(addrs)
        ptrs = (C.c_void_p * n)(*[C.c_void_p(int(a)) for a in addrs])
        fb = np.ascontiguousarray(first_bases, dtype=np.uint64)
        ns = np.ascontiguousarray(n_starts, dtype=np.uint64)
        h = C.c_void_p()
        self._ok(self.lib.dnagpu_seq_wrap_pieces(self.handle, ptrs, fb.ctypes.data_as(_lib.u64p),
                                                 ns.ctypes.data_as(_lib.u64p), n, n_bases_total, C.byref(h)))
        return Seq(self, h, keep=keep)

    def fill_words(self, addr, seq, n_words_alloc):
        """Copy a Seq's packed words to a raw device address (a peer-allocated shard) and zero the rest of the
        n_words_alloc words there; on torch's current stream."""
        import torch
        n = min(seq.n_words, n_words_alloc)
        dst = _device_view(addr, n_words_alloc, self.device)
        if n:
            dst[:n].copy_(_device_view(seq.device_ptr, n, self.device))
        dst[n:].zero_()
        if not self.shares_torch_stream:
            torch.cuda.current_stream(self.device).synchronize()

    def upload_to(self, addr, host_tensor, n_words_alloc):
        """H2D of packed words from a (pinned) torch int64 host tensor to a raw device address; the tail is zeroed."""
        import torch
        n = min(host_tensor.numel(), n_words_alloc)
        dst = _device_view(addr, n_words_alloc, self.device)
        dst[:n].copy_(host_tensor[:n], non_blocking=True)
        dst[n:].zero_()
        if not self.shares_torch_stream:
            torch.cuda.current_stream(self.device).synchronize()

    def wrap_reads(self, tensor, n_reads, bases_per_read, stride_words):
        self._after_torch()
        h = C.c_void_p()
        self._ok(self.lib.dnagpu_seq_wrap_reads(self.handle, tensor.data_ptr(), n_reads, bases_per_read,
                                                stride_words, tensor.numel(), C.byref(h)))
        return Seq(self, h, keep=tensor)

    # ---- ingest codec (dna_in / dna_out on the device) --------------------------------------
    def encode_dna(self, text):
        """ASCII -> Dna, validated and packed on the GPU (dna_make, dna.c:178-202)."""
        raw = text if isinstance(text, (bytes, bytearray)) else text.encode("ascii", "replace")
        words = np.empty((len(raw) + 31) // 32, dtype=np.uint64)
        self._ok(self.lib.dnagpu_encode_dna(self.handle, bytes(raw), len(raw), words.ctypes.data))
        return Dna.from_words(words, len(raw))

    def seq_from_text(self, text):
        raw = text if isinstance(text, (bytes, bytearray)) else text.encode("ascii", "replace")
        h = C.c_void_p()
        self._ok(self.lib.dnagpu_seq_from_text(self.handle, bytes(raw), len(raw), C.byref(h)))
        return Seq(self, h)

    def decode_dna(self, dna):
        buf = C.create_string_buffer(dna.length + 1)
        self._ok(self.lib.dnagpu_decode_dna(self.handle, dna.words.ctypes.data, dna.length, buf))
        return buf.raw[:dna.length].decode()

    # ---- generate_kmers ----------------------------------------------------------
    def generate_kmers(self, dna, k):
        """Host in, host out: `SELECT * FROM generate_kmers(dna, k)` (dna.c:743-837)."""
        dna = dna if isinstance(dna, Dna) else Dna(dna)
        rows = max(0, dna.length - k + 1) if 1 <= k <= 32 else 0
        out = np.empty(rows, dtype=np.uint64)
        n = C.c_uint64()
        self._ok(self.lib.dnagpu_generate_kmers(self.handle, dna.words.ctypes.data, dna.length, k,
                                                out.ctypes.data, out.size, C.byref(n)))
        return KmerArray(out[:n.value], k)

    def extract(self, seq, k, out=None):
        """Device in, device out; returns a torch int64 CUDA tensor of the rows."""
        import torch
        rows = seq.kmer_count(k)
        if not 1 <= k <= 32:
            self._ok(self.lib.dnagpu_extract(self.handle, seq.handle, k, None, 0, C.byref(C.c_uint64())))
        if out is None:
            out = torch.empty(max(rows, 2), dtype=torch.int64, device=f"cuda:{self.device}")
        n = C.c_uint64()
        self._ok(self.lib.dnagpu_extract(self.handle, seq.handle, k, out.data_ptr(), out.numel(), C.byref(n)))
        self._before_torch()
        return out[:n.value]

    # ---- WHERE ^@ / @> ---------------------------------------------------------------
    def filter_kmers(self, dna, k, prefix=None, pattern=None):
        """`SELECT * FROM generate_kmers(dna,k) AS k(kmer) WHERE kmer ^@ prefix AND pattern @> kmer`."""
        dna = dna if isinstance(dna, Dna) else Dna(dna)
        w, _keep = _where(prefix, pattern)
        wp = C.byref(w) if w is not None else None
        n = C.c_uint64()
        rc = self.lib.dnagpu_filter_kmers(self.handle, dna.words.ctypes.data, dna.length, k, wp, None, 0, C.byref(n))
        if rc not in (0, 21):  # 21 = ECAPACITY: *n_out holds the need
            self._ok(rc)
        out = np.empty(n.value, dtype=np.uint64)
        if n.value:
            self._ok(self.lib.dnagpu_filter_kmers(self.handle, dna.words.ctypes.data, dna.length, k, wp,
                                                  out.ctypes.data, out.size, C.byref(n)))
        return KmerArray(out[:n.value], k)

    def filter_count(self, seq, k, prefix=None, pattern=None):
        w, _keep = _where(prefix, pattern)
        n = C.c_uint64()
        self._ok(self.lib.dnagpu_filter(self.handle, seq.handle, k, C.byref(w) if w is not None else None,
                                        None, 0, C.byref(n)))
        return int(n.value)

    def filter(self, seq, k, prefix=None, pattern=None, planes=False):
        """Rows of generate_kmers that pass the WHERE clause, in sequence order (torch int64 CUDA tensor).
        One pass into a buffer sized for 1/8 of the rows; a second, exactly sized pass only if that was too small."""
        import torch
        w, _keep = _where(prefix, pattern, planes)
        wp = C.byref(w) if w is not None else None
        n = C.c_uint64()
        guess = seq.kmer_count(k) if w is None else max(1024, seq.kmer_count(k) // 8)
        for _ in range(2):
            out = torch.empty(max(int(guess), 2), dtype=torch.int64, device=f"cuda:{self.device}")
            rc = self.lib.dnagpu_filter(self.handle, seq.handle, k, wp, out.data_ptr(), out.numel(), C.byref(n))
            if rc != 21:  # DNAGPU_ECAPACITY: n holds the need
                self._ok(rc)
                self._before_torch()
                return out[:n.value]
            guess = n.value
        self._ok(rc)

    def collect(self, seq, k, prefix=None, pattern=None, planes=False):
        """The rows that pass the WHERE clause in no particular order (one predicate scan): torch int64 CUDA tensor."""
        import torch
        w, _keep = _where(prefix, pattern, planes)
        wp = C.byref(w) if w is not None else None
        n = C.c_uint64()
        guess = seq.kmer_count(k) if w is None else max(1024, seq.kmer_count(k) // 8)
        for _ in range(2):
            out = torch.empty(max(int(guess), 2), dtype=torch.int64, device=f"cuda:{self.device}")
            rc = self.lib.dnagpu_collect(self.handle, seq.handle, k, wp, out.data_ptr(), out.numel(), C.byref(n))
            if rc != 21:  # DNAGPU_ECAPACITY: n holds the need
                self._ok(rc)
                self._before_torch()
                return out[:n.value]
            guess = n.value
        self._ok(rc)

    def filter_keys(self, keys, k, prefix=None, pattern=None):
        """The same predicates over a materialised kmer column (torch int64 CUDA tensor), rows in column order."""
        self._after_torch()
        import torch
        w, _keep = _where(prefix, pattern)
        wp = C.byref(w) if w is not None else None
        n = C.c_uint64()
        guess = keys.numel() if w is None else max(1024, keys.numel() // 8)
        for _ in range(2):
            out = torch.empty(max(int(guess), 2), dtype=torch.int64, device=f"cuda:{self.device}")
            rc = self.lib.dnagpu_filter_keys(self.handle, keys.data_ptr(), keys.numel(), k, wp, out.data_ptr(),
                                             out.numel(), C.byref(n))
            if rc != 21:
                self._ok(rc)
                self._before_torch()
                return out[:n.value]
            guess = n.value
        self._ok(rc)

    def index_build(self, keys, k):
        """CREATE INDEX ... ON column(kmer): keys = torch int64 CUDA tensor of Kmer.bit_sequence, all of length k."""
        self._after_torch()
        h = C.c_void_p()
        self._ok(self.lib.dnagpu_index_build(self.handle, keys.data_ptr(), keys.numel(), k, C.byref(h)))
        return Index(self, h)

    # ---- GROUP BY kmer ------------------------------------------------------------------
    @staticmethod
    def _opts(method, load_factor, expected_keys, exact=False, owner=None):
        if method == COUNT_AUTO and not load_factor and not expected_keys and not exact and owner is None:
            return None
        o = CountOpts()
        o.method, o.load_factor, o.expected_keys = method, load_factor or 0.0, expected_keys or 0
        o.flags = COUNT_FLAG_EXACT if exact else 0
        if owner is not None:
            o.owner_parts, o.owner_part = owner
        return o

    def count(self, seq, k, prefix=None, pattern=None, table=False, method=COUNT_AUTO,
              load_factor=0.0, expected_keys=0, exact=False, owner=None, planes=False):
        """GROUP BY kmer over device-resident sequences -> (Stats, Table | None).
        owner=(n_parts, part): only the k-mers dnagpu_owner_of assigns to `part` (one GPU's share of a multi-GPU count)."""
        w, _keep = _where(prefix, pattern, planes)
        o = self._opts(method, load_factor, expected_keys, exact, owner)
        st, th = Stats(), C.c_void_p()
        self._ok(self.lib.dnagpu_count(self.handle, seq.handle, k, C.byref(w) if w is not None else None,
                                       C.byref(o) if o is not None else None, C.byref(st),
                                       C.byref(th) if table else None))
        return st, (Table(self, th) if table else None)

    def count_spectrum(self, seq, k, prefix=None, pattern=None, max_count=10000, method=COUNT_AUTO, exact=False,
                       owner=None, planes=False):
        """The abundance spectrum of `count`'s query -> (Stats, uint64 array h of max_count entries): h[c-1] distinct
        k-mers occur exactly c times (c < max_count), h[max_count-1] occur max_count times or more."""
        w, _keep = _where(prefix, pattern, planes)
        o = self._opts(method, 0.0, 0, exact, owner)
        st, hist = Stats(), np.zeros(max(int(max_count), 1), dtype=np.uint64)
        self._ok(self.lib.dnagpu_count_spectrum(self.handle, seq.handle, k, C.byref(w) if w is not None else None,
                                                C.byref(o) if o is not None else None, max_count,
                                                hist.ctypes.data, C.byref(st)))
        return st, hist

    def count_kmers_spectrum(self, dna, k, prefix=None, pattern=None, max_count=10000):
        """Host in: `SELECT least(count, max_count), count(*) FROM (... GROUP BY kmer) GROUP BY 1` as count_spectrum
        returns it.  On a multi-GPU context every GPU counts its share."""
        dna = dna if isinstance(dna, Dna) else Dna(dna)
        w, _keep = _where(prefix, pattern)
        st, hist = Stats(), np.zeros(max(int(max_count), 1), dtype=np.uint64)
        self._ok(self.lib.dnagpu_count_kmers_spectrum(self.handle, dna.words.ctypes.data, dna.length, k,
                                                      C.byref(w) if w is not None else None, max_count,
                                                      hist.ctypes.data, C.byref(st)))
        return st, hist

    def count_keys(self, keys, k, table=False, method=COUNT_AUTO, load_factor=0.0, expected_keys=0):
        self._after_torch()
        o = self._opts(method, load_factor, expected_keys)
        st, th = Stats(), C.c_void_p()
        self._ok(self.lib.dnagpu_count_keys(self.handle, keys.data_ptr(), keys.numel(), k,
                                            C.byref(o) if o is not None else None, C.byref(st),
                                            C.byref(th) if table else None))
        return st, (Table(self, th) if table else None)

    def count_kmers(self, dna, k, prefix=None, pattern=None, table=True):
        """Host in: `SELECT kmer, count(*) FROM generate_kmers(dna,k) [WHERE ...] GROUP BY kmer`."""
        dna = dna if isinstance(dna, Dna) else Dna(dna)
        w, _keep = _where(prefix, pattern)
        st, th = Stats(), C.c_void_p()
        self._ok(self.lib.dnagpu_count_kmers(self.handle, dna.words.ctypes.data, dna.length, k,
                                             C.byref(w) if w is not None else None, C.byref(st),
                                             C.byref(th) if table else None))
        return st, (Table(self, th) if table else None)

    def count_kmers_ptr(self, words_ptr, n_bases, k, prefix=None, pattern=None):
        """The C-ABI host call on a raw host pointer (pinned memory): stats only."""
        w, _keep = _where(prefix, pattern)
        st = Stats()
        self._ok(self.lib.dnagpu_count_kmers(self.handle, words_ptr, n_bases, k,
                                             C.byref(w) if w is not None else None, C.byref(st), None))
        return st

    def count_reads_ptr(self, words_ptr, n_reads, bases_per_read, stride_words, k, prefix=None, pattern=None,
                        planes=False):
        """The C-ABI host call for a batch of reads on a raw host pointer: stats only."""
        w, _keep = _where(prefix, pattern, planes)
        st = Stats()
        self._ok(self.lib.dnagpu_count_reads(self.handle, words_ptr, n_reads, bases_per_read, stride_words, k,
                                             C.byref(w) if w is not None else None, C.byref(st), None))
        return st

    def count_reads(self, words, n_reads, bases_per_read, stride_words, k, prefix=None, pattern=None,
                    table=True):
        words = np.ascontiguousarray(words, dtype=np.uint64)
        w, _keep = _where(prefix, pattern)
        st, th = Stats(), C.c_void_p()
        self._ok(self.lib.dnagpu_count_reads(self.handle, words.ctypes.data, n_reads, bases_per_read,
                                             stride_words, k, C.byref(w) if w is not None else None,
                                             C.byref(st), C.byref(th) if table else None))
        return st, (Table(self, th) if table else None)

    # ---- owner routing ---------------------------------------------------------------------
    def partition_counts(self, seq, k, n_parts, prefix=None, pattern=None):
        w, _keep = _where(prefix, pattern)
        counts = np.zeros(n_parts, dtype=np.uint64)
        self._ok(self.lib.dnagpu_partition(self.handle, seq.handle, k, C.byref(w) if w is not None else None,
                                           n_parts, None, 0, counts.ctypes.data_as(_lib.u64p)))
        return counts

    def partition(self, seq, k, n_parts, prefix=None, pattern=None, out=None):
        """Bucket the k-mers by owner rank -> (torch int64 tensor, per-owner counts)."""
        import torch
        w, _keep = _where(prefix, pattern)
        wp = C.byref(w) if w is not None else None
        counts = np.zeros(n_parts, dtype=np.uint64)
        if out is None:
            bound = seq.kmer_count(k) if w is None else int(self.partition_counts(seq, k, n_parts, prefix, pattern).sum())
            out = torch.empty(max(bound, 2), dtype=torch.int64, device=f"cuda:{self.device}")
        self._ok(self.lib.dnagpu_partition(self.handle, seq.handle, k, wp, n_parts, out.data_ptr(), out.numel(),
                                           counts.ctypes.data_as(_lib.u64p)))
        return out[:int(counts.sum())], counts

    # ---- fused owner routing (partition level 1 = exchange layout) ---------------------------------
    def shuffle_plan(self, n_rows_total, n_parts):
        plan = ShufflePlan()
        self._ok(self.lib.dnagpu_shuffle_plan_make(n_rows_total, n_parts, C.byref(plan)))
        return plan

    def shuffle_send(self, seq, k, plan, out, prefix=None, pattern=None):
        """-> (digit_counts[n_digits], rows_kept, side_rows); keys by digit in `out` (torch int64 tensor)."""
        w, _keep = _where(prefix, pattern)
        counts = np.zeros(plan.n_digits, dtype=np.uint64)
        kept, side = C.c_uint64(), C.c_uint64()
        self._ok(self.lib.dnagpu_shuffle_send(self.handle, seq.handle, k, C.byref(w) if w is not None else None,
                                              C.byref(plan), out.data_ptr(), out.numel(),
                                              counts.ctypes.data_as(_lib.u64p), C.byref(kept), C.byref(side)))
        return counts, int(kept.value), int(side.value)

    def shuffle_count(self, keys, piece_counts, n_groups, plan, k, table=False):
        self._after_torch()
        piece_counts = np.ascontiguousarray(piece_counts, dtype=np.uint64)
        st, th = Stats(), C.c_void_p()
        self._ok(self.lib.dnagpu_shuffle_count(self.handle, keys.data_ptr() if keys is not None else None,
                                               piece_counts.ctypes.data_as(_lib.u64p), piece_counts.size, n_groups,
                                               C.byref(plan), k, C.byref(st), C.byref(th) if table else None))
        return st, (Table(self, th) if table else None)

    # ---- exchange fused into the scatter kernel (peer memory) ------------------------------------
    def peer_alloc(self, n_bytes):
        """-> (device address, 64-byte IPC handle) of a receive buffer other ranks can map."""
        p, h = C.c_void_p(), C.create_string_buffer(64)
        self._ok(self.lib.dnagpu_peer_alloc(self.handle, n_bytes, C.byref(p), h))
        return int(p.value), h.raw

    def peer_open(self, handle):
        p = C.c_void_p()
        self._ok(self.lib.dnagpu_peer_open(self.handle, handle, C.byref(p)))
        return int(p.value)

    def peer_close(self, addr):
        self._ok(self.lib.dnagpu_peer_close(self.handle, C.c_void_p(addr)))

    def peer_free(self, addr):
        self._ok(self.lib.dnagpu_peer_free(self.handle, C.c_void_p(addr)))

    def shuffle_hist(self, seq, k, plan, prefix=None, pattern=None):
        w, _keep = _where(prefix, pattern)
        counts = np.zeros(plan.n_digits, dtype=np.uint64)
        self._ok(self.lib.dnagpu_shuffle_hist(self.handle, seq.handle, k, C.byref(w) if w is not None else None,
                                              C.byref(plan), counts.ctypes.data_as(_lib.u64p)))
        return counts

    def shuffle_scatter_to(self, seq, k, plan, digit_dest, prefix=None, pattern=None):
        w, _keep = _where(prefix, pattern)
        digit_dest = np.ascontiguousarray(digit_dest, dtype=np.uint64)
        kept, side = C.c_uint64(), C.c_uint64()
        self._ok(self.lib.dnagpu_shuffle_scatter_to(self.handle, seq.handle, k, C.byref(w) if w is not None else None,
                                                    C.byref(plan), digit_dest.ctypes.data_as(_lib.u64p),
                                                    C.byref(kept), C.byref(side)))
        return int(kept.value), int(side.value)

    def shuffle_hist_keys(self, keys, plan):
        self._after_torch()
        counts = np.zeros(plan.n_digits, dtype=np.uint64)
        self._ok(self.lib.dnagpu_shuffle_hist_keys(self.handle, keys.data_ptr(), keys.numel(), C.byref(plan),
                                                   counts.ctypes.data_as(_lib.u64p)))
        return counts

    def shuffle_scatter_keys_to(self, keys, plan, digit_dest):
        self._after_torch()
        digit_dest = np.ascontiguousarray(digit_dest, dtype=np.uint64)
        side = C.c_uint64()
        self._ok(self.lib.dnagpu_shuffle_scatter_keys_to(self.handle, keys.data_ptr(), keys.numel(), C.byref(plan),
                                                         digit_dest.ctypes.data_as(_lib.u64p), C.byref(side)))
        return int(side.value)

    def shuffle_count_addr(self, addr, piece_counts, n_groups, plan, k):
        """dnagpu_shuffle_count on a raw device address (a peer-allocated receive buffer)."""
        piece_counts = np.ascontiguousarray(piece_counts, dtype=np.uint64)
        st = Stats()
        self._ok(self.lib.dnagpu_shuffle_count(self.handle, C.c_void_p(addr), piece_counts.ctypes.data_as(_lib.u64p),
                                               piece_counts.size, n_groups, C.byref(plan), k, C.byref(st), None))
        return st

    # ---- profiling ----------------------------------------------------------------------------
    def profile(self, on=True):
        self._ok(self.lib.dnagpu_profile_enable(self.handle, 1 if on else 0))

    def profile_reset(self):
        self._ok(self.lib.dnagpu_profile_reset(self.handle))

    def profile_query(self, prefix=""):
        ms, n = C.c_double(), C.c_uint64()
        self._ok(self.lib.dnagpu_profile_query(self.handle, prefix.encode(), C.byref(ms), C.byref(n)))
        return ms.value, int(n.value)

    def profile_dump(self):
        import json
        buf = C.create_string_buffer(1 << 16)
        self._ok(self.lib.dnagpu_profile_dump(self.handle, buf, len(buf)))
        return json.loads(buf.value.decode())


def owner_of(kmer_bits, n_parts):
    return int(_lib.load().dnagpu_owner_of(int(kmer_bits), n_parts))


_default = None


def default_context():
    global _default
    if _default is None:
        _default = Context(0)
    return _default


# ---- the SQL surface as plain functions ---------------------------------------------------
def generate_kmers(dna, k, ctx=None):
    """`SELECT * FROM generate_kmers(dna, k)` (dna--1.0.sql:188-191)."""
    return (ctx or default_context()).generate_kmers(dna, k)


def filter_kmers(dna, k, prefix=None, pattern=None, ctx=None):
    """`... WHERE kmer ^@ prefix` / `... WHERE pattern @> kmer` (test.sql:67, 86)."""
    return (ctx or default_context()).filter_kmers(dna, k, prefix=prefix, pattern=pattern)


def count_kmers(dna, k, prefix=None, pattern=None, ctx=None):
    """`SELECT kmer, count(*) ... GROUP BY kmer` -> dict {kmer text: count} (README.md:107-116)."""
    st, table = (ctx or default_context()).count_kmers(dna, k, prefix=prefix, pattern=pattern, table=True)
    kmers, counts = table.sorted()
    table.free()
    return dict(zip(kmer_strings(kmers, k), (int(c) for c in counts)))


def kmer_stats(dna, k, prefix=None, pattern=None, ctx=None):
    """total / distinct / unique of README.md:122-130 -> (total, distinct, unique)."""
    st, _ = (ctx or default_context()).count_kmers(dna, k, prefix=prefix, pattern=pattern, table=False)
    return int(st.total), int(st.distinct), int(st.unique)


def kmer_spectrum(dna, k, prefix=None, pattern=None, max_count=10000, ctx=None):
    """The k-mer abundance spectrum -> uint64 array h: h[c-1] distinct k-mers occur c times, the last entry
    max_count times or more (`SELECT least(count, max_count), count(*) ... GROUP BY 1`)."""
    _, hist = (ctx or default_context()).count_kmers_spectrum(dna, k, prefix=prefix, pattern=pattern,
                                                             max_count=max_count)
    return hist
