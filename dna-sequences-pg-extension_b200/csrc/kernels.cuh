/*
 * kernels.cuh -- sm_100a device code of libdnagpu.
 *
 * The reference (/root/reference/dna.c) produces each k-mer by decoding k
 * bases to chars and re-encoding them (dna.c:803-825).  Because the `dna`
 * words (dna.c:116-123) and the `kmer` word (dna.c:406-412) are the same
 * little-endian 2-bit stream, k-mer i is simply bits [2i, 2i+2k) of the packed
 * stream: a funnel shift over two adjacent words and a mask.  Everything here
 * is built on that window; there is no dense contraction, so no tensor cores.
 *
 * Two thread mappings are used:
 *   row mapping   one thread = two consecutive output rows (ordered 16-byte
 *                 streaming stores; extraction is HBM-write-bound).
 *   item mapping  one thread = one packed word = up to 32 consecutive start
 *                 positions of one sequence, rolled out of two registers
 *                 (count / filter / partition; order-free or CTA-ordered).
 */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/dnagpu_synth.h"

namespace dnagpu {

constexpr int kThreads = 256;
constexpr uint64_t kEmpty = ~0ull; /* hash-slot sentinel; a real k-mer only for k = 32 ('G' x 32) */

enum Layout { kSingle = 0, kFixed = 1, kRagged = 2, kPieces = 3 /* host side only: see OwnedView */ };

/* Device view of a dnagpu_seq for one value of k. */
struct SeqView {
    const uint64_t *words;
    uint64_t n_seqs;
    uint64_t stride;       /* words between consecutive sequences (fixed)          */
    uint64_t rows_per_seq; /* generate_kmers rows of each sequence (single/fixed)  */
    uint64_t items_per_seq;/* ceil(rows_per_seq / 32)                              */
    uint64_t n_rows;       /* total rows                                           */
    uint64_t n_items;      /* total items                                          */
    /* ragged only */
    const uint64_t *word_off; /* first word of sequence s                           */
    const uint64_t *row_off;  /* exclusive prefix of rows, n_seqs + 1 entries       */
    const uint64_t *item_off; /* exclusive prefix of items, n_seqs + 1 entries      */
};

/* WHERE kmer ^@ prefix AND qkmer @> kmer as four "allowed" bit planes.
 * Bit 2j of plane X is set iff base X is allowed at position j (IUPAC set of
 * dna.c:1064-1086 intersected with the prefix base of dna.c:859-863);
 * positions >= k and every odd bit are set in all planes. */
struct Pred {
    uint64_t ma, mt, mc, mg;
};

/* Device counters of one GROUP BY (u64 each). */
enum { C_TOTAL = 0, C_DISTINCT, C_UNIQUE, C_SIDE, C_OVERFLOW, C_CURSOR, C_L1OVF, C_L2OVF, C_PASSED, C_COUNT };

__host__ __device__ __forceinline__ uint64_t mix64(uint64_t x)
{ /* murmur3 fmix64 */
    x ^= x >> 33;
    x *= 0xff51afd7ed558ccdull;
    x ^= x >> 33;
    x *= 0xc4ceb9fe1a85ec53ull;
    x ^= x >> 33;
    return x;
}
/* Owner rank of a k-mer among n_parts GPUs -- a function of the k-mer's low word (its first 16 bases; the whole
 * k-mer for k <= 16), because the multi-GPU count tests EVERY start position of the sequence for ownership
 * (k_collect_owned) and keeps one in n_parts.  Independent of the partition digits (64-bit multiply-shift over the
 * whole k-mer) and of the bucket / bin hashes (fold of both words, another multiplier).
 *   n_parts = 2, 4, 8 (the machines that exist): bit i of the rank is the parity of the low word under kOwnTap[i]
 *     -- a GF(2)-linear hash, five taps per bit out of a pool of ten bit offsets that mixes both bits of ten of the
 *     sixteen bases (any XOR of the three tap sets keeps >= 5 taps).  Linear means bit-parallel: the funnel shift
 *     of a packed word by a tap offset holds that tap for all 32 start positions at once, so the ownership of 32
 *     starts costs ~ 40 instructions instead of 32 x (shift, multiply, compare, select).
 *   any other n_parts: multiplicative hash of the low word, top bits -> rank; one IMAD per start position. */
constexpr uint32_t kOwnerMul = 0x85EBCA6Bu;
constexpr int kOwnPool = 10;
__host__ __device__ constexpr int own_tau(int p)
{ /* bit offsets of the pool inside the low word */
    return p == 0 ? 0 : p == 1 ? 3 : p == 2 ? 6 : p == 3 ? 9 : p == 4 ? 13 : p == 5 ? 16 : p == 6 ? 19 : p == 7 ? 22 : p == 8 ? 26 : 29;
}
__host__ __device__ constexpr uint32_t own_sub(int i)
{ /* pool members of rank bit i */
    return i == 0 ? 0x06Eu : i == 1 ? 0x2D1u : 0x1B4u;
}
__host__ __device__ constexpr uint32_t own_tap(int i)
{
    uint32_t m = 0;
    for (int p = 0; p < kOwnPool; ++p)
        if (own_sub(i) >> p & 1u) m |= 1u << own_tau(p);
    return m;
}
/* rank bits of the linear form: 1, 2, 3 for 2, 4, 8 owners; 0 = multiplicative form */
__host__ __device__ __forceinline__ int owner_lin_bits(uint32_t n_parts) { return n_parts == 2 ? 1 : n_parts == 4 ? 2 : n_parts == 8 ? 3 : 0; }
__host__ __device__ __forceinline__ uint32_t owner_hash(uint64_t kmer) { return (uint32_t)kmer * kOwnerMul; }
__host__ __device__ __forceinline__ uint32_t parity32(uint32_t x)
{
#ifdef __CUDA_ARCH__
    return (uint32_t)__popc(x) & 1u;
#else
    return (uint32_t)__builtin_popcount(x) & 1u;
#endif
}
__host__ __device__ __forceinline__ uint32_t owner_of(uint64_t kmer, uint32_t n_parts)
{
    const int lin = owner_lin_bits(n_parts);
    if (lin) {
        const uint32_t x = (uint32_t)kmer;
        uint32_t r = parity32(x & own_tap(0));
        if (lin > 1) r |= parity32(x & own_tap(1)) << 1;
        if (lin > 2) r |= parity32(x & own_tap(2)) << 2;
        return r;
    }
    return (uint32_t)(((uint64_t)owner_hash(kmer) * (uint64_t)n_parts) >> 32);
}

__device__ __forceinline__ bool pred_ok(const Pred &p, uint64_t x)
{
    /* per even bit: hi ? (lo ? G : C) : (lo ? T : A) -- three LOP3 per 32-bit half */
    uint64_t lo = x, hi = x >> 1;
    uint64_t s0 = (lo & p.mt) | (~lo & p.ma);
    uint64_t s1 = (lo & p.mg) | (~lo & p.mc);
    uint64_t m = (hi & s1) | (~hi & s0);
    /* odd bits of the planes are 1, but hi/lo garbage on odd bits selects among
     * ones only, so m has all odd bits set; all even bits set <=> every position ok */
    return m == ~0ull;
}

__device__ __forceinline__ uint64_t ld_nc(const uint64_t *p) { return __ldg(p); }

__device__ __forceinline__ void st_cs_v2(uint64_t *p, uint64_t a, uint64_t b)
{
    asm volatile("st.global.cs.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(a), "l"(b) : "memory");
}
__device__ __forceinline__ void st_cs(uint64_t *p, uint64_t a)
{
    asm volatile("st.global.cs.u64 [%0], %1;" ::"l"(p), "l"(a) : "memory");
}

/* bits [s, s+64) of the 128-bit value w1:w0, s in [0, 64) */
__device__ __forceinline__ uint64_t window(uint64_t w0, uint64_t w1, unsigned s)
{
    uint32_t a0 = (uint32_t)w0, a1 = (uint32_t)(w0 >> 32), a2 = (uint32_t)w1,
             a3 = (uint32_t)(w1 >> 32);
    if (s >= 32) {
        a0 = a1;
        a1 = a2;
        a2 = a3;
        s -= 32;
    }
    uint32_t lo = __funnelshift_r(a0, a1, s), hi = __funnelshift_r(a1, a2, s);
    return ((uint64_t)hi << 32) | lo;
}

/* ---- locating rows and items ------------------------------------------------ */
__device__ __forceinline__ uint64_t upper_seq(const uint64_t *off, uint64_t n_seqs, uint64_t g)
{ /* largest s with off[s] <= g (off has n_seqs + 1 entries, off[n_seqs] > g) */
    uint64_t lo = 0, hi = n_seqs;
    while (hi - lo > 1) {
        uint64_t mid = (lo + hi) >> 1;
        if (off[mid] <= g) lo = mid; else hi = mid;
    }
    return lo;
}

/* row g -> (pointer to the word holding its first base, bit shift) */
template <int L>
__device__ __forceinline__ const uint64_t *locate_row(const SeqView &sv, uint64_t g, unsigned &s)
{
    uint64_t base_word, pos;
    if (L == kSingle) {
        base_word = 0;
        pos = g;
    } else if (L == kFixed) {
        uint64_t r = g / sv.rows_per_seq;
        pos = g - r * sv.rows_per_seq;
        base_word = r * sv.stride;
    } else {
        uint64_t r = upper_seq(sv.row_off, sv.n_seqs, g);
        pos = g - sv.row_off[r];
        base_word = sv.word_off[r];
    }
    s = (unsigned)(pos & 31) * 2;
    return sv.words + base_word + (pos >> 5);
}

/* item t -> (pointer to its word, number of starts c in [1,32], first row index) */
template <int L>
__device__ __forceinline__ const uint64_t *locate_item(const SeqView &sv, uint64_t t, int &c,
                                                       uint64_t &row0)
{
    if (L == kSingle) {
        uint64_t left = sv.n_rows - t * 32;
        c = left < 32 ? (int)left : 32;
        row0 = t * 32;
        return sv.words + t;
    } else if (L == kFixed) {
        uint64_t r, qi;
        if (sv.n_items <= 0xffffffffull) {
            uint32_t r32 = (uint32_t)t / (uint32_t)sv.items_per_seq;
            r = r32;
            qi = (uint32_t)t - r32 * (uint32_t)sv.items_per_seq;
        } else {
            r = t / sv.items_per_seq;
            qi = t - r * sv.items_per_seq;
        }
        uint64_t left = sv.rows_per_seq - qi * 32;
        c = left < 32 ? (int)left : 32;
        row0 = r * sv.rows_per_seq + qi * 32;
        return sv.words + r * sv.stride + qi;
    } else {
        uint64_t r = upper_seq(sv.item_off, sv.n_seqs, t);
        uint64_t qi = t - sv.item_off[r];
        uint64_t rows = sv.row_off[r + 1] - sv.row_off[r];
        uint64_t left = rows - qi * 32;
        c = left < 32 ? (int)left : 32;
        row0 = sv.row_off[r] + qi * 32;
        return sv.words + sv.word_off[r] + qi;
    }
}

/* Roll the c start positions of an item out of two registers.  f(x, j) gets the
 * UNMASKED 64-bit window at start j (caller masks for the key). */
template <int UNROLL, class F>
__device__ __forceinline__ void roll_item(uint64_t w0, uint64_t w1, int c, F &&f)
{
    uint64_t cur = w0, nxt = w1;
#pragma unroll UNROLL
    for (int j = 0; j < 32; ++j) {
        if (j < c) f(cur, j);
        cur = (cur >> 2) | (nxt << 62);
        nxt >>= 2;
    }
}

/* ---- block helpers ------------------------------------------------------------ */
__device__ __forceinline__ uint64_t warp_sum(uint64_t v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ uint32_t warp_sum32(uint32_t v)
{
    return __reduce_add_sync(0xffffffffu, v);
}

/* block-wide exclusive scan of one u32 per thread (kThreads threads); returns
 * the exclusive prefix and writes the block total to *total. */
__device__ __forceinline__ uint32_t block_exscan(uint32_t v, uint32_t *total)
{
    __shared__ uint32_t warp_tot[kThreads / 32];
    __shared__ uint32_t block_tot;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t n = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += n;
    }
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        uint32_t t = lane < kThreads / 32 ? warp_tot[lane] : 0, ti = t;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t n = __shfl_up_sync(0xffffffffu, ti, o);
            if (lane >= o) ti += n;
        }
        if (lane < kThreads / 32) warp_tot[lane] = ti - t;
        if (lane == 31) block_tot = ti;
    }
    __syncthreads();
    uint32_t ex = warp_tot[wid] + inc - v;
    *total = block_tot;
    __syncthreads();
    return ex;
}

/* =================================================================================
 * K1  generate_kmers (dna.c:743-837): ordered extraction, row mapping.
 * Each thread produces kPairs pairs of consecutive rows; a warp's store
 * instruction writes 512 contiguous bytes.  8 B written + 0.25 B read per row.
 * ================================================================================= */
constexpr int kPairsPerThread = 4;

template <int L>
__global__ void __launch_bounds__(kThreads) k_extract(SeqView sv, uint64_t mask,
                                                      uint64_t *__restrict__ out)
{
    const uint64_t n_rows = sv.n_rows;
    const uint64_t tile = (uint64_t)blockIdx.x * (kThreads * kPairsPerThread);
    uint64_t x0[kPairsPerThread], x1[kPairsPerThread];
#pragma unroll
    for (int u = 0; u < kPairsPerThread; ++u) {
        uint64_t g = 2 * (tile + (uint64_t)u * kThreads + threadIdx.x);
        x0[u] = x1[u] = 0;
        if (g < n_rows) {
            unsigned s;
            const uint64_t *w = locate_row<L>(sv, g, s);
            uint64_t w0 = ld_nc(w), w1 = ld_nc(w + 1);
            x0[u] = window(w0, w1, s) & mask;
            if (g + 1 < n_rows) {
                if (L == kSingle) { /* g even: row g+1 starts in the same word */
                    x1[u] = window(w0, w1, s + 2) & mask;
                } else {
                    const uint64_t *v = locate_row<L>(sv, g + 1, s);
                    x1[u] = window(ld_nc(v), ld_nc(v + 1), s) & mask;
                }
            }
        }
    }
#pragma unroll
    for (int u = 0; u < kPairsPerThread; ++u) {
        uint64_t g = 2 * (tile + (uint64_t)u * kThreads + threadIdx.x);
        if (g + 1 < n_rows) st_cs_v2(out + g, x0[u], x1[u]);
        else if (g < n_rows) st_cs(out + g, x0[u]);
    }
}

/* The same with 256-bit stores (sm_100: STG.E.ENL2.256): one thread = FOUR consecutive rows = one full
 * 32-byte sector, a warp's store instruction writes 1 KB.  Needs a 32-byte aligned output. */
constexpr int kQuadsPerThread = 2;

__device__ __forceinline__ void st_v4(uint64_t *p, uint64_t a, uint64_t b, uint64_t c, uint64_t d)
{
    asm volatile("st.global.cs.v4.u64 [%0], {%1, %2, %3, %4};" ::"l"(p), "l"(a), "l"(b), "l"(c), "l"(d) : "memory");
}

template <int L>
__global__ void __launch_bounds__(kThreads) k_extract4(SeqView sv, uint64_t mask, uint64_t *__restrict__ out)
{
    const uint64_t n_rows = sv.n_rows;
    const uint64_t tile = (uint64_t)blockIdx.x * (kThreads * kQuadsPerThread);
    uint64_t x[kQuadsPerThread][4];
#pragma unroll
    for (int u = 0; u < kQuadsPerThread; ++u) {
        const uint64_t g = 4 * (tile + (uint64_t)u * kThreads + threadIdx.x);
#pragma unroll
        for (int j = 0; j < 4; ++j) x[u][j] = 0;
        if (g < n_rows) {
            if (L == kSingle) { /* g is a multiple of 4: the four rows start in the same packed word */
                unsigned s;
                const uint64_t *w = locate_row<L>(sv, g, s);
                const uint64_t w0 = ld_nc(w), w1 = ld_nc(w + 1);
#pragma unroll
                for (int j = 0; j < 4; ++j) x[u][j] = window(w0, w1, s + 2 * j) & mask;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (g + j < n_rows) {
                        unsigned s;
                        const uint64_t *w = locate_row<L>(sv, g + j, s);
                        x[u][j] = window(ld_nc(w), ld_nc(w + 1), s) & mask;
                    }
            }
        }
    }
#pragma unroll
    for (int u = 0; u < kQuadsPerThread; ++u) {
        const uint64_t g = 4 * (tile + (uint64_t)u * kThreads + threadIdx.x);
        if (g + 3 < n_rows) {
            st_v4(out + g, x[u][0], x[u][1], x[u][2], x[u][3]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (g + j < n_rows) st_cs(out + g + j, x[u][j]);
        }
    }
}

/* =================================================================================
 * K2  generate_kmers ... WHERE ^@ / @> : ordered compaction in three launches.
 *   k_filter_count  per-CTA match counts (item mapping, predicate on 2-bit planes)
 *   k_scan_u64      exclusive scan of the CTA counts
 *   k_filter_write  recompute, rank inside the CTA, stage in shared memory, store
 *                   each CTA's matches as one contiguous, coalesced run.
 * ================================================================================= */
/* The WHERE clause over the 32 start positions of one item, branch-free.  The low plane (the
 * packed words themselves) and the high plane (the same 128 bits shifted right by one) are
 * formed once; the window of start j is then two constant-amount funnel shifts per plane, and
 * the test is three LOP3 per 32-bit half (pred_ok's select tree) + one AND + one compare.
 * Bit j of the result is set iff start j < c passes. */
template <int L>
__device__ __forceinline__ uint32_t item_match_mask(const SeqView &sv, const Pred &p, uint64_t t,
                                                    uint64_t &w0, uint64_t &w1, int &c)
{
    uint64_t row0;
    const uint64_t *w = locate_item<L>(sv, t, c, row0);
    w0 = ld_nc(w);
    w1 = ld_nc(w + 1);
    const uint32_t a[5] = {(uint32_t)w0, (uint32_t)(w0 >> 32), (uint32_t)w1, (uint32_t)(w1 >> 32), 0u};
    const uint32_t h[5] = {__funnelshift_r(a[0], a[1], 1), __funnelshift_r(a[1], a[2], 1),
                           __funnelshift_r(a[2], a[3], 1), a[3] >> 1, 0u};
    const uint32_t mal = (uint32_t)p.ma, mah = (uint32_t)(p.ma >> 32), mtl = (uint32_t)p.mt,
                   mth = (uint32_t)(p.mt >> 32), mcl = (uint32_t)p.mc, mch = (uint32_t)(p.mc >> 32),
                   mgl = (uint32_t)p.mg, mgh = (uint32_t)(p.mg >> 32);
    uint32_t m = 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        const int q = (2 * j) >> 5, s = (2 * j) & 31; /* compile-time after unrolling */
        const uint32_t xl = s ? __funnelshift_r(a[q], a[q + 1], s) : a[q];
        const uint32_t xh = s ? __funnelshift_r(a[q + 1], a[q + 2], s) : a[q + 1];
        const uint32_t hl = s ? __funnelshift_r(h[q], h[q + 1], s) : h[q];
        const uint32_t hh = s ? __funnelshift_r(h[q + 1], h[q + 2], s) : h[q + 1];
        const uint32_t s0l = (xl & mtl) | (~xl & mal), s1l = (xl & mgl) | (~xl & mcl);
        const uint32_t s0h = (xh & mth) | (~xh & mah), s1h = (xh & mgh) | (~xh & mch);
        const uint32_t ml = (hl & s1l) | (~hl & s0l), mh = (hh & s1h) | (~hh & s0h);
        m |= (uint32_t)((ml & mh) == 0xffffffffu) << j;
    }
    return c >= 32 ? m : (m & ((1u << c) - 1u));
}

constexpr int kFilterTiles = 4; /* tiles of kThreads items one CTA walks (fewer, longer-lived CTAs) */

template <int L>
__global__ void __launch_bounds__(kThreads) k_filter_count(SeqView sv, Pred p,
                                                           uint64_t *__restrict__ tile_counts)
{
    __shared__ uint32_t wsum[kFilterTiles][kThreads / 32];
    const uint64_t n_tiles = (sv.n_items + kThreads - 1) / kThreads;
#pragma unroll
    for (int i = 0; i < kFilterTiles; ++i) {
        const uint64_t tile = (uint64_t)blockIdx.x * kFilterTiles + i;
        const uint64_t t = tile * kThreads + threadIdx.x;
        uint32_t n = 0;
        if (t < sv.n_items) {
            uint64_t w0, w1;
            int c;
            n = __popc(item_match_mask<L>(sv, p, t, w0, w1, c));
        }
        n = warp_sum32(n);
        if ((threadIdx.x & 31) == 0) wsum[i][threadIdx.x >> 5] = n;
    }
    __syncthreads();
    if (threadIdx.x < kFilterTiles) {
        const uint64_t tile = (uint64_t)blockIdx.x * kFilterTiles + threadIdx.x;
        uint32_t s = 0;
#pragma unroll
        for (int w = 0; w < kThreads / 32; ++w) s += wsum[threadIdx.x][w];
        if (tile < n_tiles) tile_counts[tile] = s;
    }
}

template <int L>
__global__ void __launch_bounds__(kThreads) k_filter_write(SeqView sv, Pred p, uint64_t mask,
                                                           const uint64_t *__restrict__ tile_off,
                                                           uint64_t *__restrict__ out)
{
    extern __shared__ uint64_t stage[]; /* kThreads * 32 entries */
    const uint64_t n_tiles = (sv.n_items + kThreads - 1) / kThreads;
    for (int i = 0; i < kFilterTiles; ++i) {
        const uint64_t tile = (uint64_t)blockIdx.x * kFilterTiles + i;
        if (tile >= n_tiles) break; /* uniform */
        const uint64_t t = tile * kThreads + threadIdx.x;
        uint32_t m = 0;
        uint64_t w0 = 0, w1 = 0;
        int c = 0;
        if (t < sv.n_items) m = item_match_mask<L>(sv, p, t, w0, w1, c);
        uint32_t total;
        uint32_t rank = block_exscan(__popc(m), &total);
        while (m) {
            int j = __ffs(m) - 1;
            m &= m - 1;
            stage[rank++] = window(w0, w1, 2 * j) & mask;
        }
        __syncthreads();
        uint64_t *dst = out + tile_off[tile];
        for (uint32_t q = threadIdx.x; q < total; q += kThreads) st_cs(dst + q, stage[q]);
        __syncthreads();
    }
}

/* Unordered single-pass form for GROUP BY (row order is irrelevant there): a tile claims its output range
 * with one atomicAdd on a cursor.  Tiles that would run past `cap` write nothing; the cursor still ends at
 * the exact number of matches, so the caller can re-run with a buffer of the right size. */
template <int L>
__global__ void __launch_bounds__(kThreads) k_filter_collect(SeqView sv, Pred p, uint64_t mask, uint64_t cap,
                                                             unsigned long long *__restrict__ cursor,
                                                             uint64_t *__restrict__ out)
{
    extern __shared__ uint64_t stage[]; /* kThreads * 32 entries */
    __shared__ unsigned long long base_s;
    const uint64_t n_tiles = (sv.n_items + kThreads - 1) / kThreads;
    for (int i = 0; i < kFilterTiles; ++i) {
        const uint64_t tile = (uint64_t)blockIdx.x * kFilterTiles + i;
        if (tile >= n_tiles) break; /* uniform */
        const uint64_t t = tile * kThreads + threadIdx.x;
        uint32_t m = 0;
        uint64_t w0 = 0, w1 = 0;
        int c = 0;
        if (t < sv.n_items) m = item_match_mask<L>(sv, p, t, w0, w1, c);
        uint32_t total;
        uint32_t rank = block_exscan(__popc(m), &total);
        if (threadIdx.x == 0 && total) base_s = atomicAdd(cursor, (unsigned long long)total);
        while (m) {
            int j = __ffs(m) - 1;
            m &= m - 1;
            stage[rank++] = window(w0, w1, 2 * j) & mask;
        }
        __syncthreads();
        if (total && base_s + total <= cap) {
            uint64_t *dst = out + base_s;
            for (uint32_t q = threadIdx.x; q < total; q += kThreads) st_cs(dst + q, stage[q]);
        }
        __syncthreads();
    }
}

/* ---- the same WHERE clause as a Shift-And automaton over the base stream ------------------------------
 * SURVEY 7 K2(b); replaces the per-base loop of contains() (dna.c:1114-1125).  State D has one bit per pattern
 * position, pattern position i at bit i + 32 - k, so that a full match is the SIGN bit for every k:
 *     t = F & M[base];   F = (t << 1) | (1 << (32 - k));   match of the k-mer ENDING at this base = t >> 31
 * with M[b] = the positions whose IUPAC set (intersected with the ^@ prefix base) allows base b.  Per base:
 * two instructions to turn the 2-bit base into a table offset, one shared-memory load of M[b] (four words in
 * four banks: any mix of lanes is one wavefront), LOP3, IADD3, and one funnel shift that collects the match
 * bits -- 6 instructions against the ~ 19 per START position of the plane test above.  A thread walks a run
 * of up to kSaItems consecutive items (128 starts) of one sequence = up to 159 bases, the first k-1 of them
 * warm-up: a 150-base read is exactly one run.  End-position matches are turned into start-position masks
 * by one 160-bit funnel shift by k-1, after which rank / stage / store work as in the plane form. */
constexpr int kSaItems = 4;
constexpr int kSaStage = 2048; /* staged matches per round (16 KB: five CTAs per SM; a selective clause needs one round) */

struct SaPred {
    uint32_t m[4]; /* M[A], M[T], M[C], M[G], left-aligned */
    uint32_t inj;  /* 1 << (32 - k) */
    uint32_t two;  /* the constant 2, as a run-time value: keeps the two multiply-adds of a step on the FMA pipe */
};

/* 32 bases of one half-word pair: steps the automaton, returns the 32 end-match bits (bit j = base j) */
/* Integer SASS splits over two pipes of half the issue rate each (B300_MICROARCH.md: IMAD on the FMA pipe;
 * LOP3 / SHF / IADD3 on the ALU pipe, one warp instruction per two clocks per SM sub-partition): a step written
 * with shifts and adds is five ALU-pipe instructions = 10 clocks.  Here the state update and the match bit come
 * from ONE 32 x 32 -> 64 multiply-add (low word = 2t + inj = the next F, high word = bit 31 of t = the match) and
 * the match bits are collected by a second multiply-add (e = 2e + match): 3 ALU + 2 FMA + 1 LDS per base. */
__device__ __forceinline__ uint32_t sa_word(uint64_t w, uint32_t lut_sa, uint32_t inj, uint32_t two, uint32_t &F)
{
    const uint32_t lo = (uint32_t)w, hi = (uint32_t)(w >> 32);
    uint32_t e = 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        const uint32_t h = j < 16 ? lo : hi;
        const int s = 2 * (j & 15);
        /* shared-memory address of M[base]: base * 4 OR-ed into the 16-byte aligned table address (one LOP3) */
        const uint32_t addr = ((s >= 2 ? h >> (s - 2) : h << 2) & 12u) | lut_sa;
        uint32_t m;
        asm("ld.shared.u32 %0, [%1];" : "=r"(m) : "r"(addr));
        const uint32_t t = (F | inj) & m; /* F carries 2t of the step before; bit 32 - k of it is never set */
        uint64_t p;
        asm("mul.wide.u32 %0, %1, %2;" : "=l"(p) : "r"(t), "r"(two));
        F = (uint32_t)p;
        asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(e) : "r"(e), "r"(two), "r"((uint32_t)(p >> 32)));
    }
    return __brev(e);
}

/* run r -> (first word, starts valid in the run); runs never span sequences */
template <int L>
__device__ __forceinline__ const uint64_t *locate_run(const SeqView &sv, uint64_t r, uint32_t &valid)
{
    static_assert(L == kSingle || L == kFixed, "Shift-And runs: single sequences and fixed-stride reads");
    if (L == kSingle) {
        const uint64_t left = sv.n_rows - r * (32 * kSaItems);
        valid = left < 32 * kSaItems ? (uint32_t)left : 32 * kSaItems;
        return sv.words + r * kSaItems;
    }
    const uint64_t runs_per_seq = (sv.items_per_seq + kSaItems - 1) / kSaItems;
    const uint64_t q = r / runs_per_seq, ri = r - q * runs_per_seq;
    const uint64_t left = sv.rows_per_seq - ri * (32 * kSaItems);
    valid = left < 32 * kSaItems ? (uint32_t)left : 32 * kSaItems;
    return sv.words + q * sv.stride + ri * kSaItems;
}

template <int L>
__device__ __forceinline__ uint64_t n_runs_of(const SeqView &sv)
{
    if (L == kSingle) return (sv.n_items + kSaItems - 1) / kSaItems;
    return sv.n_seqs * ((sv.items_per_seq + kSaItems - 1) / kSaItems);
}

/* start-position match masks of one run; w[] receives its packed words */
template <int L>
__device__ __forceinline__ void sa_run_masks(const SeqView &sv, uint32_t lut, uint32_t inj, uint32_t two, int k, uint64_t r,
                                             uint64_t (&w)[kSaItems + 1], uint32_t (&sm)[kSaItems])
{
    uint32_t valid;
    const uint64_t *p = locate_run<L>(sv, r, valid);
    const int n_items = (int)((valid + 31) >> 5);
#pragma unroll
    for (int i = 0; i <= kSaItems; ++i) w[i] = i <= n_items ? ld_nc(p + i) : 0; /* + the halo word */
    uint32_t F = 0, e[kSaItems + 1]; /* the injected bit is OR-ed in at the start of every step */
#pragma unroll
    for (int i = 0; i <= kSaItems; ++i) e[i] = i <= n_items ? sa_word(w[i], lut, inj, two, F) : 0u;
#pragma unroll
    for (int i = 0; i < kSaItems; ++i) {
        const uint32_t m = __funnelshift_r(e[i], e[i + 1], k - 1); /* the k-mer starting at s ends at s + k - 1 */
        const int c = (int)valid - 32 * i;
        sm[i] = c >= 32 ? m : c > 0 ? (m & ((1u << c) - 1u)) : 0u;
    }
}

/* MODE: kSaCollect = unordered, a tile claims its output range from `cursor` (tiles past `cap` write nothing but
 * still count); kSaCount = matches per tile -> tile_io[tile]; kSaWrite = the tile's rows, in sequence order, at
 * out + tile_io[tile] (the exclusive scan of the counts).  A tile = kThreads runs = 32768 start positions. */
enum { kSaCollect = 0, kSaCount = 1, kSaWrite = 2 };

template <int L, int MODE>
__global__ void __launch_bounds__(kThreads) k_filter_sa(SeqView sv, SaPred sp, uint64_t mask, int k, uint64_t cap,
                                                        unsigned long long *__restrict__ cursor,
                                                        uint64_t *__restrict__ tile_io, uint64_t *__restrict__ out)
{
    extern __shared__ uint64_t stage[]; /* kSaStage entries (none for kSaCount) */
    __shared__ __align__(16) uint32_t lut[4];
    __shared__ unsigned long long base_s;
    if (threadIdx.x < 4) lut[threadIdx.x] = sp.m[threadIdx.x];
    __syncthreads();
    const uint32_t lut_sa = (uint32_t)__cvta_generic_to_shared(lut);
    const uint64_t n_runs = n_runs_of<L>(sv);
    const uint64_t r = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    uint64_t w[kSaItems + 1];
    uint32_t sm[kSaItems] = {0, 0, 0, 0};
    if (r < n_runs) sa_run_masks<L>(sv, lut_sa, sp.inj, sp.two, k, r, w, sm);
    uint32_t n = 0;
#pragma unroll
    for (int i = 0; i < kSaItems; ++i) n += __popc(sm[i]);
    uint32_t total;
    const uint32_t rank0 = block_exscan(n, &total);
    if (MODE == kSaCount) {
        if (threadIdx.x == 0) tile_io[blockIdx.x] = total;
        return;
    }
    if (threadIdx.x == 0) {
        if (MODE == kSaWrite) base_s = tile_io[blockIdx.x];
        else if (total) base_s = atomicAdd(cursor, (unsigned long long)total);
    }
    __syncthreads();
    if (total == 0 || (MODE == kSaCollect && base_s + total > cap)) return; /* uniform; the cursor still counts what did not fit */
    uint64_t *dst = out + base_s;
    for (uint32_t round = 0; round < total; round += kSaStage) { /* one round unless > 2048 rows of the tile match */
        uint32_t rank = rank0;
#pragma unroll
        for (int i = 0; i < kSaItems; ++i) {
            uint32_t m = sm[i];
            while (m) {
                const int j = __ffs(m) - 1;
                m &= m - 1;
                if (rank >= round && rank < round + kSaStage) stage[rank - round] = window(w[i], w[i + 1], 2 * j) & mask;
                ++rank;
            }
        }
        __syncthreads();
        const uint32_t cnt = min((uint32_t)kSaStage, total - round);
        for (uint32_t q = threadIdx.x; q < cnt; q += kThreads) st_cs(dst + round + q, stage[q]);
        __syncthreads();
    }
}

/* the same predicates over a materialised kmer column (seq scan of test.sql:220-262) */
constexpr int kKeysPerThread = 8;
__global__ void __launch_bounds__(kThreads) k_filter_keys_count(const uint64_t *__restrict__ keys,
                                                                uint64_t n, Pred p,
                                                                uint64_t *__restrict__ tile_counts)
{
    __shared__ uint32_t wsum[kThreads / 32];
    uint64_t base = (uint64_t)blockIdx.x * (kThreads * kKeysPerThread);
    uint32_t cnt = 0;
#pragma unroll
    for (int u = 0; u < kKeysPerThread; ++u) {
        uint64_t i = base + (uint64_t)u * kThreads + threadIdx.x;
        if (i < n) cnt += pred_ok(p, ld_nc(keys + i));
    }
    cnt = warp_sum32(cnt);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t s = 0;
#pragma unroll
        for (int i = 0; i < kThreads / 32; ++i) s += wsum[i];
        tile_counts[blockIdx.x] = s;
    }
}

__global__ void __launch_bounds__(kThreads) k_filter_keys_write(const uint64_t *__restrict__ keys,
                                                                uint64_t n, Pred p,
                                                                const uint64_t *__restrict__ tile_off,
                                                                uint64_t *__restrict__ out)
{
    /* loads are coalesced (key u * 256 + t of the tile sits with thread t); output order must follow INPUT
     * order, i.e. row-major over (u, t): per-warp match counts of every row go to shared memory once, each
     * thread then walks the 8 x 8 counts for its offsets; matches are staged and stored as one run */
    __shared__ uint64_t stage[kThreads * kKeysPerThread];
    __shared__ uint32_t wc[kKeysPerThread * (kThreads / 32)]; /* 64 (row, warp) counts, then their prefix */
    __shared__ uint32_t total_s;
    static_assert(kKeysPerThread * (kThreads / 32) == 64, "one warp scans two counts per lane");
    const uint64_t base = (uint64_t)blockIdx.x * (kThreads * kKeysPerThread);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint64_t x[kKeysPerThread];
    uint32_t bal[kKeysPerThread];
#pragma unroll
    for (int u = 0; u < kKeysPerThread; ++u) {
        const uint64_t i = base + (uint64_t)u * kThreads + threadIdx.x;
        x[u] = i < n ? ld_nc(keys + i) : 0;
    }
#pragma unroll
    for (int u = 0; u < kKeysPerThread; ++u) {
        const uint64_t i = base + (uint64_t)u * kThreads + threadIdx.x;
        bal[u] = __ballot_sync(0xffffffffu, i < n && pred_ok(p, x[u]));
        if (lane == 0) wc[u * (kThreads / 32) + wid] = __popc(bal[u]);
    }
    __syncthreads();
    if (wid == 0) { /* exclusive scan of the 64 counts, row-major = input order */
        const uint32_t a = wc[2 * lane], b = wc[2 * lane + 1];
        uint32_t inc = a + b;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += y;
        }
        wc[2 * lane] = inc - a - b;
        wc[2 * lane + 1] = inc - b;
        if (lane == 31) total_s = inc;
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < kKeysPerThread; ++u)
        if (bal[u] & (1u << lane))
            stage[wc[u * (kThreads / 32) + wid] + __popc(bal[u] & ((1u << lane) - 1u))] = x[u];
    __syncthreads();
    const uint32_t total = total_s;
    uint64_t *dst = out + tile_off[blockIdx.x];
    for (uint32_t q = threadIdx.x; q < total; q += kThreads) st_cs(dst + q, stage[q]);
}

/* exclusive scan of n u64 values by ONE CTA of 1024 threads walking chunks with a
 * carry; out[n] receives the grand total.  Inputs here are CTA counts / per-row
 * counts (<= a few million entries). */
__global__ void __launch_bounds__(1024) k_scan_u64(const uint64_t *__restrict__ in, uint64_t n,
                                                   uint64_t *__restrict__ out)
{
    __shared__ uint64_t wtot[32];
    __shared__ uint64_t carry_s;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (uint64_t base = 0; base < n; base += 1024) {
        uint64_t i = base + threadIdx.x;
        uint64_t v = i < n ? in[i] : 0, inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint64_t y = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += y;
        }
        if (lane == 31) wtot[wid] = inc;
        __syncthreads();
        if (wid == 0) { /* exclusive scan of the 32 warp totals */
            uint64_t t = wtot[lane], ti = t;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                uint64_t y = __shfl_up_sync(0xffffffffu, ti, o);
                if (lane >= o) ti += y;
            }
            wtot[lane] = ti - t;
        }
        __syncthreads();
        uint64_t ex = carry_s + wtot[wid] + inc - v;
        if (i < n) out[i] = ex;
        __syncthreads(); /* everyone has read carry_s */
        if (threadIdx.x == 1023) carry_s = ex + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) out[n] = carry_s;
}

/* =================================================================================
 * K4  GROUP BY kmer, hash variant: HBM open-addressing table of 16-byte slots
 * {key, count}.  Insert = atomicCAS on the key, then atomicAdd on the count of
 * the SAME 32-byte sector; the value the add returns gives distinct (old == 0)
 * and unique (+1 at old == 0, -1 at old == 1) without ever scanning the table.
 * ================================================================================= */
struct Slot {
    unsigned long long key;
    unsigned long long count;
};

__global__ void __launch_bounds__(kThreads) k_table_init(Slot *__restrict__ slots, uint64_t cap)
{
    uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * kThreads;
    for (; i < cap; i += stride)
        asm volatile("st.global.cs.v2.u64 [%0], {%1, %2};" ::"l"(slots + i), "l"(kEmpty), "l"(0ull)
                     : "memory");
}

struct Tally { /* per-thread partial aggregates */
    uint32_t total, distinct;
    int32_t unique;
    uint32_t side;
};

__device__ __forceinline__ void hash_insert(Slot *__restrict__ slots, uint64_t cap, uint64_t x,
                                            Tally &ty, unsigned long long *ctr)
{
    if (x == kEmpty) { /* only reachable for k = 32: 'G' x 32 gets a side counter */
        ty.side++;
        return;
    }
    uint64_t i = __umul64hi(mix64(x), cap);
    for (uint64_t probes = 0; probes < cap; ++probes) {
        unsigned long long old = atomicCAS(&slots[i].key, (unsigned long long)kEmpty,
                                           (unsigned long long)x);
        if (old == kEmpty || old == x) {
            unsigned long long c = atomicAdd(&slots[i].count, 1ull);
            ty.distinct += (c == 0);
            ty.unique += (c == 0) - (c == 1);
            return;
        }
        if (++i == cap) i = 0;
    }
    atomicExch(&ctr[C_OVERFLOW], 1ull);
}

__device__ __forceinline__ void tally_flush(const Tally &ty, unsigned long long *ctr)
{
    uint32_t t = warp_sum32(ty.total), d = warp_sum32(ty.distinct), s = warp_sum32(ty.side);
    int32_t u = (int32_t)__reduce_add_sync(0xffffffffu, ty.unique);
    if ((threadIdx.x & 31) == 0) {
        if (t) atomicAdd(&ctr[C_TOTAL], (unsigned long long)t);
        if (d) atomicAdd(&ctr[C_DISTINCT], (unsigned long long)d);
        if (u) atomicAdd(&ctr[C_UNIQUE], (unsigned long long)(long long)u);
        if (s) atomicAdd(&ctr[C_SIDE], (unsigned long long)s);
    }
}

template <int L, bool FILTER>
__global__ void __launch_bounds__(kThreads) k_count_hash(SeqView sv, Pred p, uint64_t mask,
                                                         Slot *__restrict__ slots, uint64_t cap,
                                                         unsigned long long *__restrict__ ctr)
{
    uint64_t t = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    Tally ty = {0, 0, 0, 0};
    if (t < sv.n_items) {
        int c;
        uint64_t row0;
        const uint64_t *w = locate_item<L>(sv, t, c, row0);
        uint64_t w0 = ld_nc(w), w1 = ld_nc(w + 1);
        roll_item<4>(w0, w1, c, [&](uint64_t x, int) {
            if (FILTER && !pred_ok(p, x)) return;
            ty.total++;
            hash_insert(slots, cap, x & mask, ty, ctr);
        });
    }
    tally_flush(ty, ctr);
}

/* count an already materialised key list (receive side of the owner exchange) */
__global__ void __launch_bounds__(kThreads) k_count_hash_keys(const uint64_t *__restrict__ keys,
                                                              uint64_t n, Slot *__restrict__ slots,
                                                              uint64_t cap,
                                                              unsigned long long *__restrict__ ctr)
{
    uint64_t base = (uint64_t)blockIdx.x * (kThreads * kKeysPerThread);
    Tally ty = {0, 0, 0, 0};
    uint64_t x[kKeysPerThread];
#pragma unroll
    for (int u = 0; u < kKeysPerThread; ++u) {
        uint64_t i = base + (uint64_t)u * kThreads + threadIdx.x;
        x[u] = i < n ? ld_nc(keys + i) : 0;
    }
#pragma unroll
    for (int u = 0; u < kKeysPerThread; ++u) {
        uint64_t i = base + (uint64_t)u * kThreads + threadIdx.x;
        if (i < n) {
            ty.total++;
            hash_insert(slots, cap, x[u], ty, ctr);
        }
    }
    tally_flush(ty, ctr);
}

/* K5 for the hash table: compact occupied slots into (kmers[], counts[]) rows */
__global__ void __launch_bounds__(kThreads) k_table_compact(const Slot *__restrict__ slots,
                                                            uint64_t cap,
                                                            uint64_t *__restrict__ kmers,
                                                            uint64_t *__restrict__ counts,
                                                            unsigned long long *__restrict__ ctr)
{
    uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * kThreads;
    const int lane = threadIdx.x & 31;
    for (uint64_t b = i - lane; b < cap; b += stride) { /* warp-uniform trip count */
        uint64_t idx = b + lane;
        Slot s = {kEmpty, 0};
        if (idx < cap) {
            const ulonglong2 v = __ldg(reinterpret_cast<const ulonglong2 *>(slots + idx));
            s.key = v.x;
            s.count = v.y;
        }
        bool occ = s.key != kEmpty;
        unsigned bal = __ballot_sync(0xffffffffu, occ);
        if (bal) {
            unsigned long long basepos = 0;
            if (lane == 0) basepos = atomicAdd(&ctr[C_CURSOR], (unsigned long long)__popc(bal));
            basepos = __shfl_sync(0xffffffffu, basepos, 0);
            if (occ) {
                uint64_t pos = basepos + __popc(bal & ((1u << lane) - 1));
                kmers[pos] = s.key;
                counts[pos] = s.count;
            }
        }
    }
}

/* ---- abundance spectrum: how many groups have count c, c = 1 .. H-1, and how many H or more ------------------
 * Device layout of the histogram (u64): [0, kSpecCum) the cumulative part C[j] (k_count_buckets_bins: groups of count
 * >= j, j = 1 .. 15), then H direct bins, bin c-1 for count min(c, H) (every kernel that sees a final count). */
constexpr int kSpecCum = 16;
constexpr uint32_t kSpecMaxCount = 1u << 20;
constexpr uint32_t kSpecSmemBins = 1024; /* per-CTA shared bins of the small counts; the rest go to global atomics */
constexpr int kSpecSmem = kSpecSmemBins * (int)sizeof(uint32_t);

struct SpecBins {
    uint32_t *s;             /* shared: s[c] for 1 <= c < n_s */
    uint32_t n_s;
    unsigned long long *hist; /* the direct bins */
    uint32_t h;
    __device__ __forceinline__ SpecBins(uint32_t *smem, unsigned long long *direct, uint32_t max_count)
        : s(smem), n_s(min(max_count + 1, kSpecSmemBins)), hist(direct), h(max_count)
    {
    }
    __device__ __forceinline__ void zero() /* the caller syncs */
    {
        for (uint32_t i = threadIdx.x; i < n_s; i += blockDim.x) s[i] = 0;
    }
    __device__ __forceinline__ void add(uint64_t c)
    {
        const uint32_t b = (uint32_t)min(c, (uint64_t)h);
        if (b < n_s)
            atomicAdd(&s[b], 1u);
        else
            atomicAdd(&hist[b - 1], 1ull);
    }
    __device__ __forceinline__ void flush() /* after a barrier */
    {
        for (uint32_t i = 1 + threadIdx.x; i < n_s; i += blockDim.x)
            if (s[i]) atomicAdd(&hist[i - 1], (unsigned long long)s[i]);
    }
};

/* the spectrum of a hash table (the HBM table of DNAGPU_COUNT_HASH, the spill table of the bucket count): every
 * occupied slot holds its group's final count */
__global__ void __launch_bounds__(kThreads) k_table_spectrum(const Slot *__restrict__ slots, uint64_t cap,
                                                             unsigned long long *__restrict__ hist, uint32_t max_count)
{
    extern __shared__ uint32_t spec_smem[];
    SpecBins sb(spec_smem, hist, max_count);
    sb.zero();
    __syncthreads();
    const uint64_t stride = (uint64_t)gridDim.x * kThreads;
    for (uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x; i < cap; i += stride) {
        const ulonglong2 v = __ldg(reinterpret_cast<const ulonglong2 *>(slots + i));
        if (v.x != kEmpty) sb.add(v.y);
    }
    __syncthreads();
    sb.flush();
}

/* =================================================================================
 * K3  GROUP BY kmer, dense variant: 4^k direct-indexed counters (k <= 16).
 *   k <= 7   per-CTA shared-memory histograms, replicated R ways by lane so that
 *            lanes of a warp never meet on one address (tiny k = few bins),
 *            flushed once per CTA with global atomics; persistent grid.
 *   k >= 8   red.global.add straight into the (L2-resident up to k = 12) table.
 * ================================================================================= */
template <typename CT>
__device__ __forceinline__ void red_add(CT *p, CT v);
template <>
__device__ __forceinline__ void red_add<uint32_t>(uint32_t *p, uint32_t v)
{
    asm volatile("red.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
template <>
__device__ __forceinline__ void red_add<unsigned long long>(unsigned long long *p,
                                                            unsigned long long v)
{
    asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

template <int L, bool FILTER, typename CT>
__global__ void __launch_bounds__(kThreads) k_count_dense_smem(SeqView sv, Pred p, uint64_t mask,
                                                               uint32_t n_bins, uint32_t rep_shift,
                                                               CT *__restrict__ table,
                                                               unsigned long long *__restrict__ ctr)
{
    extern __shared__ uint32_t hist[]; /* n_bins << rep_shift counters */
    const uint32_t n_ctr = n_bins << rep_shift;
    const uint32_t rep = (threadIdx.x & 31) & ((1u << rep_shift) - 1);
    for (uint32_t i = threadIdx.x; i < n_ctr; i += kThreads) hist[i] = 0;
    __syncthreads();
    uint32_t total = 0;
    /* persistent grid: a CTA walks chunks of kThreads items (host sizes the grid so
     * that one CTA sees < 2^32 k-mers, the range of a shared-memory bin) */
    for (uint64_t t = (uint64_t)blockIdx.x * kThreads + threadIdx.x; t < sv.n_items;
         t += (uint64_t)gridDim.x * kThreads) {
        int c;
        uint64_t row0;
        const uint64_t *w = locate_item<L>(sv, t, c, row0);
        uint64_t w0 = ld_nc(w), w1 = ld_nc(w + 1);
        roll_item<8>(w0, w1, c, [&](uint64_t x, int) {
            if (FILTER && !pred_ok(p, x)) return;
            total++;
            atomicAdd(&hist[((uint32_t)(x & mask) << rep_shift) | rep], 1u);
        });
    }
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < n_bins; b += kThreads) {
        uint32_t s = 0;
        for (uint32_t r = 0; r < (1u << rep_shift); ++r) s += hist[(b << rep_shift) | r];
        if (s) red_add<CT>(table + b, (CT)s);
    }
    total = warp_sum32(total);
    if ((threadIdx.x & 31) == 0 && total) atomicAdd(&ctr[C_TOTAL], (unsigned long long)total);
}

template <int L, bool FILTER, typename CT>
__global__ void __launch_bounds__(kThreads) k_count_dense(SeqView sv, Pred p, uint64_t mask,
                                                          CT *__restrict__ table,
                                                          unsigned long long *__restrict__ ctr)
{
    uint64_t t = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    uint32_t total = 0;
    if (t < sv.n_items) {
        int c;
        uint64_t row0;
        const uint64_t *w = locate_item<L>(sv, t, c, row0);
        uint64_t w0 = ld_nc(w), w1 = ld_nc(w + 1);
        roll_item<8>(w0, w1, c, [&](uint64_t x, int) {
            if (FILTER && !pred_ok(p, x)) return;
            total++;
            red_add<CT>(table + (x & mask), (CT)1);
        });
    }
    total = warp_sum32(total);
    if ((threadIdx.x & 31) == 0 && total) atomicAdd(&ctr[C_TOTAL], (unsigned long long)total);
}

template <typename CT>
__global__ void __launch_bounds__(kThreads) k_count_dense_keys(const uint64_t *__restrict__ keys,
                                                               uint64_t n, uint64_t n_bins,
                                                               CT *__restrict__ table,
                                                               unsigned long long *__restrict__ ctr)
{
    uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * kThreads;
    uint32_t total = 0;
    for (; i < n; i += stride) {
        uint64_t x = ld_nc(keys + i);
        if (x < n_bins) {
            red_add<CT>(table + x, (CT)1);
            total++;
        } else {
            atomicExch(&ctr[C_OVERFLOW], 1ull); /* not a k-mer of this k */
        }
    }
    total = warp_sum32(total);
    if ((threadIdx.x & 31) == 0 && total) atomicAdd(&ctr[C_TOTAL], (unsigned long long)total);
}

/* K5 for the dense table: distinct / unique, and optional compaction.  The SPEC form also bins every non-zero
 * counter into the direct part of the spectrum (kSpecSmem bytes of dynamic shared memory). */
template <typename CT, bool SPEC = false>
__global__ void __launch_bounds__(kThreads) k_dense_stats(const CT *__restrict__ table,
                                                          uint64_t n_bins,
                                                          unsigned long long *__restrict__ ctr,
                                                          unsigned long long *__restrict__ spec_direct = nullptr,
                                                          uint32_t max_count = 0)
{
    extern __shared__ uint32_t spec_smem[];
    SpecBins sb(spec_smem, spec_direct, max_count);
    if constexpr (SPEC) {
        sb.zero();
        __syncthreads();
    }
    uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * kThreads;
    uint32_t d = 0, u = 0;
    for (; i < n_bins; i += stride) {
        CT c = table[i];
        d += (c != 0);
        u += (c == 1);
        if constexpr (SPEC)
            if (c) sb.add((uint64_t)c);
    }
    if constexpr (SPEC) {
        __syncthreads();
        sb.flush();
    }
    d = warp_sum32(d);
    u = warp_sum32(u);
    if ((threadIdx.x & 31) == 0) {
        if (d) atomicAdd(&ctr[C_DISTINCT], (unsigned long long)d);
        if (u) atomicAdd(&ctr[C_UNIQUE], (unsigned long long)u);
    }
}

template <typename CT>
__global__ void __launch_bounds__(kThreads) k_dense_compact(const CT *__restrict__ table,
                                                            uint64_t n_bins,
                                                            uint64_t *__restrict__ kmers,
                                                            uint64_t *__restrict__ counts,
                                                            unsigned long long *__restrict__ ctr)
{
    uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * kThreads;
    const int lane = threadIdx.x & 31;
    for (uint64_t b = i - lane; b < n_bins; b += stride) {
        uint64_t idx = b + lane;
        uint64_t c = idx < n_bins ? (uint64_t)table[idx] : 0;
        unsigned bal = __ballot_sync(0xffffffffu, c != 0);
        if (bal) {
            unsigned long long basepos = 0;
            if (lane == 0) basepos = atomicAdd(&ctr[C_CURSOR], (unsigned long long)__popc(bal));
            basepos = __shfl_sync(0xffffffffu, basepos, 0);
            if (c) {
                uint64_t pos = basepos + __popc(bal & ((1u << lane) - 1));
                kmers[pos] = idx;
                counts[pos] = c;
            }
        }
    }
}

/* =================================================================================
 * K6  owner routing for the multi-GPU GROUP BY: bucket k-mers by
 * owner_of(kmer).  Pass 1 counts per owner; pass 2 claims one contiguous
 * run per (CTA, owner) with a single atomic per owner, ranks inside the CTA in
 * shared memory, and writes each run coalesced.
 * ================================================================================= */
constexpr int kMaxParts = 64;

template <int L, bool FILTER>
__global__ void __launch_bounds__(kThreads) k_partition_count(SeqView sv, Pred p, uint64_t mask,
                                                              uint32_t n_parts,
                                                              unsigned long long *__restrict__ part_counts)
{
    __shared__ uint32_t cnt[kMaxParts];
    if (threadIdx.x < kMaxParts) cnt[threadIdx.x] = 0;
    __syncthreads();
    for (uint64_t t = (uint64_t)blockIdx.x * kThreads + threadIdx.x; t < sv.n_items;
         t += (uint64_t)gridDim.x * kThreads) {
        int c;
        uint64_t row0;
        const uint64_t *w = locate_item<L>(sv, t, c, row0);
        uint64_t w0 = ld_nc(w), w1 = ld_nc(w + 1);
        roll_item<8>(w0, w1, c, [&](uint64_t x, int) {
            if (FILTER && !pred_ok(p, x)) return;
            atomicAdd(&cnt[owner_of(x & mask, n_parts)], 1u);
        });
    }
    __syncthreads();
    if (threadIdx.x < n_parts && cnt[threadIdx.x])
        atomicAdd(&part_counts[threadIdx.x], (unsigned long long)cnt[threadIdx.x]);
}

template <int L, bool FILTER>
__global__ void __launch_bounds__(kThreads) k_partition_write(SeqView sv, Pred p, uint64_t mask,
                                                              uint32_t n_parts,
                                                              const uint64_t *__restrict__ part_off,
                                                              unsigned long long *__restrict__ cursors,
                                                              uint64_t *__restrict__ out)
{
    extern __shared__ uint64_t stage[]; /* kThreads * 32 k-mers */
    __shared__ uint32_t cnt[kMaxParts], loc[kMaxParts + 1], fill[kMaxParts];
    __shared__ uint64_t gbase[kMaxParts];
    if (threadIdx.x < kMaxParts) cnt[threadIdx.x] = 0, fill[threadIdx.x] = 0;
    __syncthreads();
    uint64_t t = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    uint64_t w0 = 0, w1 = 0;
    int c = 0;
    if (t < sv.n_items) {
        uint64_t row0;
        const uint64_t *w = locate_item<L>(sv, t, c, row0);
        w0 = ld_nc(w);
        w1 = ld_nc(w + 1);
        roll_item<8>(w0, w1, c, [&](uint64_t x, int) {
            if (FILTER && !pred_ok(p, x)) return;
            atomicAdd(&cnt[owner_of(x & mask, n_parts)], 1u);
        });
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t a = 0;
        for (uint32_t o = 0; o < n_parts; ++o) {
            loc[o] = a;
            a += cnt[o];
        }
        loc[n_parts] = a;
    }
    if (threadIdx.x < n_parts && cnt[threadIdx.x])
        gbase[threadIdx.x] = part_off[threadIdx.x] +
                             atomicAdd(&cursors[threadIdx.x], (unsigned long long)cnt[threadIdx.x]);
    __syncthreads();
    roll_item<8>(w0, w1, c, [&](uint64_t x, int) {
        if (FILTER && !pred_ok(p, x)) return;
        uint64_t key = x & mask;
        uint32_t o = owner_of(key, n_parts);
        stage[loc[o] + atomicAdd(&fill[o], 1u)] = key;
    });
    __syncthreads();
    const uint32_t total = loc[n_parts];
    for (uint32_t i = threadIdx.x; i < total; i += kThreads) {
        uint32_t o = 0;
        while (i >= loc[o + 1]) ++o; /* n_parts is small */
        out[gbase[o] + (i - loc[o])] = stage[i];
    }
}

/* ---- ragged batches: rows / items per sequence for a given k ---------------- */
__global__ void __launch_bounds__(kThreads) k_ragged_rows(const uint64_t *__restrict__ n_bases,
                                                          uint64_t n_seqs, int k,
                                                          uint64_t *__restrict__ rows,
                                                          uint64_t *__restrict__ items)
{
    uint64_t s = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (s >= n_seqs) return;
    uint64_t n = n_bases[s];
    uint64_t r = n >= (uint64_t)k ? n - k + 1 : 0; /* Q2: never the wrap of dna.c:781 */
    rows[s] = r;
    items[s] = (r + 31) >> 5;
}

/* =================================================================================
 * Ingest codec (SURVEY 8(f2)): dna_in / dna_out on the device.
 *   encode  validate_dna_sequence + encode_dna (dna.c:159-171, 114-128): one thread packs 32 ASCII
 *           bases into one word (two 16-byte loads, 8 B stored); the position of the first byte that
 *           is not one of A T C G goes to *first_bad through atomicMin (the reference reports the first).
 *   decode  decode_dna (dna.c:135-152): one thread unpacks one word into 32 characters.
 * 1 B read + 0.25 B written per base: HBM-bound streaming.
 * ================================================================================= */
__device__ __forceinline__ uint32_t base_code(uint32_t c, bool &ok)
{
    const uint32_t idx = (c >> 1) & 3u;                      /* A 0, C 1, T 2, G 3 */
    ok = ((0x47544341u >> (8 * idx)) & 0xffu) == c;           /* exactly 'A' 'C' 'T' 'G' (upper case only) */
    return (0xD8u >> (2 * idx)) & 3u;                         /* -> A 00, T 01, C 10, G 11 (dna.c:119-123) */
}

__global__ void __launch_bounds__(kThreads) k_encode_dna(const unsigned char *__restrict__ text, uint64_t n_bases,
                                                         uint64_t *__restrict__ words,
                                                         unsigned long long *__restrict__ first_bad)
{
    const uint64_t w = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    const uint64_t n_words = (n_bases + 31) >> 5;
    if (w >= n_words) return;
    const uint64_t first = w << 5;
    uint32_t chunk[8]; /* 32 characters */
    if (first + 32 <= n_bases) {
        const uint4 a = __ldg(reinterpret_cast<const uint4 *>(text + first));
        const uint4 b = __ldg(reinterpret_cast<const uint4 *>(text + first + 16));
        chunk[0] = a.x; chunk[1] = a.y; chunk[2] = a.z; chunk[3] = a.w;
        chunk[4] = b.x; chunk[5] = b.y; chunk[6] = b.z; chunk[7] = b.w;
    } else { /* the last, partial word: the tail reads as 'A' (code 00), i.e. zero padding (dna.c:186) */
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            uint32_t v = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint64_t i = first + 4 * q + j;
                v |= (uint32_t)(i < n_bases ? text[i] : (unsigned char)'A') << (8 * j);
            }
            chunk[q] = v;
        }
    }
    uint64_t word = 0;
    uint32_t bad = 32;
#pragma unroll
    for (int q = 7; q >= 0; --q) {
#pragma unroll
        for (int j = 3; j >= 0; --j) {
            bool ok;
            const uint32_t code = base_code((chunk[q] >> (8 * j)) & 0xffu, ok);
            word = (word << 2) | code;
            if (!ok) bad = 4 * q + j; /* descending loop: the smallest offending index survives */
        }
    }
    words[w] = word;
    if (bad < 32 && first + bad < n_bases) atomicMin(first_bad, (unsigned long long)(first + bad));
}

__global__ void __launch_bounds__(kThreads) k_decode_dna(const uint64_t *__restrict__ words, uint64_t n_bases,
                                                         unsigned char *__restrict__ text)
{
    const uint64_t w = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    const uint64_t n_words = (n_bases + 31) >> 5;
    if (w >= n_words) return;
    const uint64_t word = ld_nc(words + w), first = w << 5;
    uint32_t chunk[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        uint32_t v = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t code = (uint32_t)(word >> (2 * (4 * q + j))) & 3u;
            v |= ((0x47435441u >> (8 * code)) & 0xffu) << (8 * j); /* 00 A, 01 T, 10 C, 11 G (dna.c:142-147) */
        }
        chunk[q] = v;
    }
    if (first + 32 <= n_bases) {
        *reinterpret_cast<uint4 *>(text + first) = make_uint4(chunk[0], chunk[1], chunk[2], chunk[3]);
        *reinterpret_cast<uint4 *>(text + first + 16) = make_uint4(chunk[4], chunk[5], chunk[6], chunk[7]);
    } else {
        for (uint64_t i = first; i < n_bases; ++i) text[i] = (unsigned char)(chunk[(i - first) >> 2] >> (8 * ((i - first) & 3)));
    }
}

/* ---- synthetic inputs on the device (include/dnagpu_synth.h) ----------------- */
__global__ void __launch_bounds__(kThreads) k_synth_seq(uint64_t seed, uint32_t R, uint64_t n_bases,
                                                        uint64_t first_word, uint64_t n_words,
                                                        uint64_t *__restrict__ words)
{
    uint64_t j = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * kThreads;
    for (; j < n_words; j += stride) words[j] = dnagpu_synth_seq_word(seed, R, n_bases, first_word + j);
}

__global__ void __launch_bounds__(kThreads) k_synth_reads(uint64_t seed, uint32_t R,
                                                          uint64_t first_read, uint64_t n_reads,
                                                          uint32_t bases_per_read,
                                                          uint32_t stride_words,
                                                          uint64_t *__restrict__ words)
{
    uint64_t j = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * kThreads;
    const uint64_t n_words = n_reads * stride_words;
    for (; j < n_words; j += stride) {
        uint64_t r = j / stride_words;
        uint32_t t = (uint32_t)(j - r * stride_words);
        words[j] = dnagpu_synth_read_word(seed, R, bases_per_read, stride_words, first_read + r, t);
    }
}

} /* namespace dnagpu */
