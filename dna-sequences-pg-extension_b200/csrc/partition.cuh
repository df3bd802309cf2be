/*
 * partition.cuh -- GROUP BY kmer for large inputs: radix partition + shared-memory count.
 *
 * Why: an open-addressing table in HBM costs one random 32-byte-sector atomic per k-mer;
 * ncu (profiles/r01a_*) shows 122 B of DRAM traffic per insert at 1.9 TB/s -- random
 * access, not arithmetic, is the bound (15 Gkmer/s on 100 Mbp, 9 Gkmer/s on 3.1 Gbp).
 * Shared-memory atomics, by contrast, run at > 1 T updates/s chip-wide (k <= 7 dense
 * kernel).  So: move the k-mers with STREAMING traffic until every bucket fits in
 * shared memory, then count there.
 *
 *   level 1   k-mers (from packed words, WHERE fused) or a key list -> P1 <= 2048
 *             partitions by the top bits of mix64(kmer): histogram pass (exact sizes,
 *             no slack, no overflow), then scatter: a CTA ranks a tile of 8192 or 16384 keys by
 *             partition in shared memory and writes one contiguous run per partition.
 *   level 2   the same inside every partition on the next hash bits (P2 <= 2048), so
 *             that a bucket holds ~1-3 K keys.  Skipped when level 1 is already enough.
 *   count     one CTA per bucket (persistent grid): 4096-slot shared-memory table,
 *             atomicCAS to claim a slot (a claim IS the first occurrence; the counter
 *             holds only the extra ones), then distinct / unique / rows from a scan of
 *             the 48 KB table.  A key that finds the table full (more distinct keys in
 *             a bucket than slots) spills to a small HBM table -- same Slot / hash_insert
 *             as the plain hash variant -- so any key distribution stays correct.
 *
 * Algorithmic traffic: 8 B written + 8 B read per key and level, + 8 B read per hist2
 * pass and for the count = 40 B/key for two levels from packed input (56 B/key from a key
 * list), all of it coalesced.
 */
#pragma once
#include "kernels.cuh"

namespace dnagpu {

constexpr int kScatThreads = 512;          /* scatter CTA: 512 threads x 16 keys             */
constexpr int kScatPer = 16;
constexpr int kTileKeys = kScatThreads * kScatPer; /* 8192 keys staged per scatter tile (64 KB) */
constexpr int kSuperTile = kTileKeys * 8;  /* keys per CTA in a histogram pass              */
constexpr int kMaxFan = 2048;              /* partitions per level                          */
/* the 16384-key tile (one CTA per SM).  From packed words (level 1): 1024 threads x 16 keys -- 32 warps instead of 16
 * to cover the latency of the shared-memory atomics and of the dependent shifts (ncu r02c: short-scoreboard and wait
 * stalls at 25 % occupancy; r02h: 16.96 -> 15.75 ms on the headline workload).  From a key list (level 2): 512 x 32,
 * which measured 2.5 % faster there than 1024 x 16 (17.46 vs 17.90 ms). */
constexpr int kBigPer = 16, kBigThreads = 1024;        /* k_part_scatter_seq  */
constexpr int kBigPerKeys = 32, kBigThreadsKeys = 512; /* k_part_scatter_keys */
constexpr int kBucketSlots = 4096; /* shared-memory table of the count kernel (power of two) */
constexpr int kBucketSlotBits = 12;
static_assert((1 << kBucketSlotBits) == kBucketSlots, "kBucketSlotBits must be log2(kBucketSlots)");
constexpr uint64_t kSlotMul = 0x9E3779B97F4A7C15ull;
constexpr uint64_t kPartMul = 0xD6E8FEB86659FD93ull;

/* Partition hash: multiply-shift (universal for the TOP bits, which is all the digits use).
 * One 64-bit multiply instead of mix64's two: the scatter kernels are issue-bound. */
__device__ __forceinline__ uint64_t part_hash(uint64_t x) { return x * kPartMul; }
__device__ __forceinline__ uint32_t digit_of(uint64_t h, int shift, uint32_t fan_mask)
{
    return (uint32_t)(h >> shift) & fan_mask;
}

/* ---- tiles of a partitioned key array ------------------------------------------- */
/* tiles[p] = ceil(size_p / tile_keys) */
__global__ void __launch_bounds__(kThreads) k_part_tiles(const uint64_t *__restrict__ parent_beg,
                                                         const uint64_t *__restrict__ parent_end,
                                                         uint64_t n_parents, uint64_t tile_keys,
                                                         uint64_t *__restrict__ tiles)
{
    uint64_t p = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (p < n_parents) tiles[p] = (parent_end[p] - parent_beg[p] + tile_keys - 1) / tile_keys;
}

/* CTA -> (parent partition, key range).  A partition is keys[parent_beg[p] .. parent_end[p]): exact
 * layouts pass (off, off + 1), the optimistic level 1 passes region starts and fill marks. */
/* Tile table: what a CTA needs to know about its tile in ONE 16-byte load.  A CTA that found its parent by binary
 * search over tile_off spent ten DEPENDENT global loads (~ 1.5 us, with nothing else resident on the SM to cover them)
 * before its first key: ncu r02c put 14 % of the instructions and 21 % of the stall samples of the level-2 scatter
 * there (17.46 -> 15.47 ms on the headline workload with the parent looked up, r02i).  The table is zeroed first, so
 * the CTAs past the last tile (the grid is an upper bound) see cnt = 0. */
struct __align__(16) TileInfo {
    uint64_t beg;    /* first key of the tile */
    uint32_t cnt;    /* keys in the tile      */
    uint32_t parent; /* partition it lies in  */
};

__global__ void __launch_bounds__(kThreads) k_tile_table(const uint64_t *__restrict__ parent_beg,
                                                         const uint64_t *__restrict__ parent_end,
                                                         const uint64_t *__restrict__ tile_off, uint64_t n_parents,
                                                         uint64_t tile_keys, uint64_t max_tiles, TileInfo *__restrict__ table)
{
    const uint64_t p = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (p >= n_parents) return;
    const uint64_t t0 = tile_off[p], t1 = min(tile_off[p + 1], max_tiles), pb = parent_beg[p], pe = parent_end[p];
    for (uint64_t t = t0; t < t1; ++t) {
        const uint64_t beg = pb + (t - t0) * tile_keys;
        TileInfo ti;
        ti.beg = beg;
        ti.cnt = (uint32_t)(min(beg + tile_keys, pe) - beg);
        ti.parent = (uint32_t)p;
        table[t] = ti;
    }
}

/* -> false when the CTA has no tile */
__device__ __forceinline__ bool tile_range(const uint64_t *parent_beg, const uint64_t *parent_end,
                                           const uint64_t *tile_off, uint64_t n_parents, uint64_t tile_keys,
                                           uint64_t &parent, uint64_t &beg, uint64_t &end, const TileInfo *table = nullptr)
{
    if (table) {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(table + blockIdx.x));
        beg = ((uint64_t)v.y << 32) | v.x;
        end = beg + v.z;
        parent = v.w;
        return v.z != 0;
    }
    if (blockIdx.x >= tile_off[n_parents]) return false; /* the grid is an upper bound on the tiles */
    parent = n_parents == 1 ? 0 : upper_seq(tile_off, n_parents, blockIdx.x);
    uint64_t t = blockIdx.x - tile_off[parent];
    beg = parent_beg[parent] + t * tile_keys;
    end = min(beg + tile_keys, parent_end[parent]);
    return true;
}

/* optimistic layouts: region d starts at d * cap */
__global__ void __launch_bounds__(kThreads) k_region_begs(uint64_t cap, uint64_t n, uint64_t *__restrict__ beg)
{
    const uint64_t d = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (d < n) beg[d] = d * cap;
}

/* optimistic level 1: end[d] = beg[d] + keys actually stored in region d */
__global__ void __launch_bounds__(kThreads) k_region_ends(const unsigned long long *__restrict__ cur,
                                                          const uint64_t *__restrict__ beg, uint64_t cap,
                                                          uint32_t n, uint64_t *__restrict__ end)
{
    uint32_t d = blockIdx.x * kThreads + threadIdx.x;
    if (d < n) end[d] = beg[d] + min((uint64_t)cur[d], cap);
}

/* ---- histogram passes ---------------------------------------------------------------- */
template <int L, bool FILTER>
__global__ void __launch_bounds__(kThreads) k_part_hist_seq(SeqView sv, Pred p, uint64_t mask, int shift,
                                                            uint32_t fan,
                                                            unsigned long long *__restrict__ hist)
{
    __shared__ uint32_t h[kMaxFan];
    for (uint32_t i = threadIdx.x; i < fan; i += kThreads) h[i] = 0;
    __syncthreads();
    const uint32_t fm = fan - 1;
    for (uint64_t t = (uint64_t)blockIdx.x * kThreads + threadIdx.x; t < sv.n_items;
         t += (uint64_t)gridDim.x * kThreads) {
        int c;
        uint64_t row0;
        const uint64_t *w = locate_item<L>(sv, t, c, row0);
        uint64_t w0 = ld_nc(w), w1 = ld_nc(w + 1);
        roll_item<8>(w0, w1, c, [&](uint64_t x, int) {
            if (FILTER && !pred_ok(p, x)) return;
            x &= mask;
            if (x == kEmpty) return; /* 'G' x 32: side counter, added by the scatter pass */
            atomicAdd(&h[digit_of(part_hash(x), shift, fm)], 1u);
        });
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < fan; i += kThreads)
        if (h[i]) atomicAdd(&hist[i], (unsigned long long)h[i]);
}

/* children of every parent partition: hist[(parent % n_groups) * fan + digit].  n_groups < n_parents
 * when the same partition arrived in several pieces (one per peer rank) that must merge. */
__global__ void __launch_bounds__(kThreads) k_part_hist_keys(const uint64_t *__restrict__ keys,
                                                             const uint64_t *__restrict__ parent_off,
                                                             const uint64_t *__restrict__ parent_end,
                                                             const uint64_t *__restrict__ tile_off,
                                                             uint64_t n_parents, uint64_t n_groups, int shift,
                                                             uint32_t fan,
                                                             unsigned long long *__restrict__ hist,
                                                             const TileInfo *__restrict__ tile_table = nullptr)
{
    __shared__ uint32_t h[kMaxFan];
    uint64_t parent, beg, end;
    if (!tile_range(parent_off, parent_end, tile_off, n_parents, kSuperTile, parent, beg, end, tile_table)) return;
    for (uint32_t i = threadIdx.x; i < fan; i += kThreads) h[i] = 0;
    __syncthreads();
    const uint32_t fm = fan - 1;
    for (uint64_t base = beg; base < end; base += kThreads * 8) {
        uint64_t x[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            uint64_t i = base + (uint64_t)u * kThreads + threadIdx.x;
            x[u] = i < end ? ld_nc(keys + i) : kEmpty;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u)
            if (x[u] != kEmpty) atomicAdd(&h[digit_of(part_hash(x[u]), shift, fm)], 1u);
    }
    __syncthreads();
    unsigned long long *dst = hist + (parent % n_groups) * fan;
    for (uint32_t i = threadIdx.x; i < fan; i += kThreads)
        if (h[i]) atomicAdd(&dst[i], (unsigned long long)h[i]);
}

/* ---- scatter passes ------------------------------------------------------------------------ */
/* Shared state of one scatter tile: cur[d] counts the keys of digit d (the value atomicAdd
 * returns is the key's rank inside its digit), then holds the digit's start in the stage;
 * gdelta[d] turns a stage position into the global output index. */
struct ScatterSmem {
    uint32_t cur[kMaxFan + 1]; /* cur[fan] = dummy bin of the keys that are not scattered */
    uint32_t warp_tot[1024 / 32 + 1];
    long long gdelta[kMaxFan];
};

/* After counting: exclusive scan of cur[] (it becomes the stage start of every digit) and
 * one global atomicAdd per non-empty digit to claim its output run.  The atomics' results
 * stay in registers (gd[]) so that their latency hides behind the placing phase; the
 * caller hands them to scatter_publish() before the flush. */
constexpr long long kNoDest = (long long)0x8000000000000000ull; /* a run that found its region full */

/* THREADS = threads of the CTA (512 in the local scatters, 256 in the owned one): each plans kMaxFan / THREADS digits */
template <int THREADS = kScatThreads>
struct ScatterClaimT { /* what scatter_plan leaves in registers for scatter_publish */
    static constexpr int kPlanPer = kMaxFan / THREADS;
    unsigned long long at[kPlanPer]; /* value returned by the claim of digit base + i: NOT looked at before the publish */
    uint32_t n[kPlanPer], ex[kPlanPer];
};
using ScatterClaim = ScatterClaimT<kScatThreads>;

template <int THREADS = kScatThreads>
__device__ __forceinline__ uint32_t scatter_plan(ScatterSmem &s, uint32_t fan,
                                                 unsigned long long *__restrict__ child_cur, ScatterClaimT<THREADS> &cl)
{
    constexpr int kPlanPer = ScatterClaimT<THREADS>::kPlanPer;
    uint32_t sum = 0;
    const uint32_t base = threadIdx.x * kPlanPer;
#pragma unroll
    for (int i = 0; i < kPlanPer; ++i) {
        cl.n[i] = base + i < fan ? s.cur[base + i] : 0;
        sum += cl.n[i];
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    if (lane == 31) s.warp_tot[wid] = inc;
    __syncthreads();
    uint32_t woff = 0, total = 0;
#pragma unroll
    for (int i = 0; i < THREADS / 32; ++i) {
        uint32_t t = s.warp_tot[i];
        if (i < wid) woff += t;
        total += t;
    }
    uint32_t ex = woff + inc - sum;
#pragma unroll
    for (int i = 0; i < kPlanPer; ++i) {
        cl.at[i] = 0;
        cl.ex[i] = ex;
        if (base + i < fan) {
            s.cur[base + i] = ex;
            if (cl.n[i]) cl.at[i] = atomicAdd(&child_cur[base + i], (unsigned long long)cl.n[i]);
        }
        ex += cl.n[i];
    }
    if (threadIdx.x == 0) s.cur[fan] = 0;
    __syncthreads();
    return total;
}

/* After the placing phase: where every digit's run goes.  With cap != 0 (optimistic layout) a run that
 * finds its region full gets no destination and raises `full_flag`: the caller re-runs exactly. */
template <int THREADS = kScatThreads>
__device__ __forceinline__ void scatter_publish(ScatterSmem &s, uint32_t fan, const uint64_t *__restrict__ child_off,
                                                const ScatterClaimT<THREADS> &cl, uint64_t cap = 0,
                                                unsigned long long *__restrict__ ctr = nullptr, int full_flag = C_L1OVF)
{
    constexpr int kPlanPer = ScatterClaimT<THREADS>::kPlanPer;
    const uint32_t base = threadIdx.x * kPlanPer;
#pragma unroll
    for (int i = 0; i < kPlanPer; ++i) {
        if (base + i < fan && cl.n[i]) {
            if (cap && cl.at[i] + cl.n[i] > cap) {
                s.gdelta[base + i] = kNoDest;
                atomicExch(&ctr[full_flag], 1ull);
            } else {
                s.gdelta[base + i] = (long long)(child_off[base + i] + cl.at[i]) - (long long)cl.ex[i];
            }
        }
    }
}

/* stage -> global: consecutive threads copy consecutive stage entries, i.e. whole runs.  The digit of
 * a staged key is recomputed (one multiply) rather than kept in a side array: the kernel is bound by
 * L1 data-pipe wavefronts (ncu: 67 % busy), not by ALU work. */
template <int PER = kScatPer, int THREADS = kScatThreads>
__device__ __forceinline__ void scatter_flush(const ScatterSmem &s, const uint64_t *stage, uint32_t total,
                                              int shift, uint32_t fm, uint64_t *__restrict__ out)
{
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        const uint32_t i = (uint32_t)u * THREADS + threadIdx.x;
        if (i < total) {
            const uint64_t x = stage[i];
            const long long g = s.gdelta[digit_of(part_hash(x), shift, fm)];
            if (g != kNoDest) out[(uint64_t)(g + (long long)i)] = x;
        }
    }
}

/* the 16384-key tile of kBigThreads threads: one thread = PER = kBigPer consecutive start positions, half
 * a packed word; one CTA per SM.
 * Straight-line code: a key that is not scattered (past the end, rejected by the WHERE
 * clause, or the k = 32 sentinel) is ranked into the dummy bin cur[fan] and its stores
 * are predicated off, so the unrolled loops carry no branches. */
template <int L, bool FILTER>
__global__ void __launch_bounds__(kBigThreads, 1) k_part_scatter_seq(SeqView sv, Pred p, uint64_t mask, int shift,
                                                                      uint32_t fan,
                                                                      const uint64_t *__restrict__ child_off,
                                                                      unsigned long long *__restrict__ child_cur,
                                                                      uint64_t *__restrict__ out,
                                                                      unsigned long long *__restrict__ ctr,
                                                                      uint64_t cap)
{
    constexpr int PER = kBigPer, THREADS = kBigThreads;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *stage = reinterpret_cast<uint64_t *>(smem_raw);
    ScatterSmem &s = *reinterpret_cast<ScatterSmem *>(smem_raw + sizeof(uint64_t) * (PER * THREADS));
    for (uint32_t i = threadIdx.x; i <= fan; i += THREADS) s.cur[i] = 0;
    __syncthreads();
    const uint32_t fm = fan - 1;
    constexpr int SPLIT = 32 / PER; /* threads sharing one packed word */
    constexpr uint32_t TILE = PER * THREADS;
    const uint64_t t = (uint64_t)blockIdx.x * (THREADS / SPLIT) + (threadIdx.x / SPLIT);
    const int half = threadIdx.x % SPLIT;
    uint64_t a0 = 0, a1 = 0; /* the PER windows of this thread start at bit 0 of a0 */
    int c = 0;
    uint32_t side = 0, kept = 0;
    uint32_t rk[PER / 2]; /* two 16-bit ranks per register; the digit is recomputed */
    if (t < sv.n_items) {
        uint64_t row0;
        int cc;
        const uint64_t *w = locate_item<L>(sv, t, cc, row0);
        uint64_t w0 = ld_nc(w), w1 = ld_nc(w + 1);
        a0 = half ? (w0 >> 32) | (w1 << 32) : w0;
        a1 = half ? (w1 >> 32) : w1;
        c = min(PER, max(0, cc - PER * half));
    }
    uint32_t real_mask = 0; /* bit j: start j is scattered */
    {
        uint64_t cur = a0, nxt = a1;
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const uint64_t x = cur & mask;
            const bool keep = (j < c) & (!FILTER || pred_ok(p, cur));
            const bool real = keep & (x != kEmpty);
            kept += keep;
            side += keep & !real;
            real_mask |= (uint32_t)real << j;
            const uint32_t d = real ? digit_of(part_hash(x), shift, fm) : fan;
            const uint32_t r = atomicAdd(&s.cur[d], 1u);
            rk[j >> 1] = (j & 1) ? __byte_perm(rk[j >> 1], r, 0x5410) : r;
            cur = (cur >> 2) | (nxt << 62);
            nxt >>= 2;
        }
    }
    __syncthreads();
    ScatterClaimT<THREADS> cl;
    const uint32_t total = scatter_plan<THREADS>(s, fan, child_cur, cl);
    {
        uint64_t cur = a0, nxt = a1;
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const uint64_t x = cur & mask;
            const uint32_t r = (j & 1) ? (rk[j >> 1] >> 16) : (rk[j >> 1] & 0xffffu);
            const uint32_t d = digit_of(part_hash(x), shift, fm);
            const uint32_t pos = (s.cur[d] + r) & (TILE - 1);
            if (real_mask & (1u << j)) stage[pos] = x;
            cur = (cur >> 2) | (nxt << 62);
            nxt >>= 2;
        }
    }
    scatter_publish<THREADS>(s, fan, child_off, cl, cap, ctr);
    __syncthreads();
    scatter_flush<PER, THREADS>(s, stage, total, shift, fm, out);
    kept = warp_sum32(kept);
    side = warp_sum32(side);
    if ((threadIdx.x & 31) == 0) {
        if (kept) atomicAdd(&ctr[C_TOTAL], (unsigned long long)kept);
        if (side) atomicAdd(&ctr[C_SIDE], (unsigned long long)side);
    }
}

/* scatter the keys of every parent partition into its children: out[child_off[parent*fan+d] ...].
 * COUNT_SIDE: first level over a raw key list (the caller's keys may hold 'G' x 32). */
template <bool COUNT_SIDE, int PER = kScatPer, int THREADS = kScatThreads>
__global__ void __launch_bounds__(THREADS, (PER * THREADS == 8192 ? 2 : 1)) k_part_scatter_keys(const uint64_t *__restrict__ keys,
                                                                       const uint64_t *__restrict__ parent_off,
                                                                       const uint64_t *__restrict__ parent_end,
                                                                       const uint64_t *__restrict__ tile_off,
                                                                       uint64_t n_parents, uint64_t n_groups, int shift,
                                                                       uint32_t fan,
                                                                       const uint64_t *__restrict__ child_off,
                                                                       unsigned long long *__restrict__ child_cur,
                                                                       uint64_t *__restrict__ out,
                                                                       unsigned long long *__restrict__ ctr,
                                                                       uint64_t cap = 0, int full_flag = C_L2OVF,
                                                                       const TileInfo *__restrict__ tile_table = nullptr)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *stage = reinterpret_cast<uint64_t *>(smem_raw);
    ScatterSmem &s = *reinterpret_cast<ScatterSmem *>(smem_raw + sizeof(uint64_t) * (PER * THREADS));
    constexpr uint32_t TILE = PER * THREADS;
    uint64_t parent, beg, end;
    if (!tile_range(parent_off, parent_end, tile_off, n_parents, TILE, parent, beg, end, tile_table)) return;
    for (uint32_t i = threadIdx.x; i <= fan; i += THREADS) s.cur[i] = 0;
    __syncthreads();
    const uint32_t fm = fan - 1;
    uint64_t x[PER];
    uint32_t rk[PER / 2]; /* two 16-bit ranks per register; the digit is recomputed */
    uint32_t side = 0, kept = 0;
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        uint64_t i = beg + (uint64_t)u * THREADS + threadIdx.x;
        x[u] = i < end ? ld_nc(keys + i) : kEmpty;
        if (COUNT_SIDE) {
            kept += (i < end);
            side += (i < end) & (x[u] == kEmpty);
        }
    }
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        const uint32_t d = x[u] != kEmpty ? digit_of(part_hash(x[u]), shift, fm) : fan;
        const uint32_t r = atomicAdd(&s.cur[d], 1u);
        rk[u >> 1] = (u & 1) ? __byte_perm(rk[u >> 1], r, 0x5410) : r;
    }
    __syncthreads();
    ScatterClaimT<THREADS> cl;
    const uint32_t total = scatter_plan<THREADS>(s, fan, child_cur + (parent % n_groups) * fan, cl);
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        const uint32_t r = (u & 1) ? (rk[u >> 1] >> 16) : (rk[u >> 1] & 0xffffu);
        const uint32_t d = x[u] != kEmpty ? digit_of(part_hash(x[u]), shift, fm) : fan;
        const uint32_t pos = (s.cur[d] + r) & (TILE - 1);
        if (d != fan) stage[pos] = x[u];
    }
    scatter_publish<THREADS>(s, fan, child_off + (parent % n_groups) * fan, cl, cap, ctr, full_flag);
    __syncthreads();
    scatter_flush<PER, THREADS>(s, stage, total, shift, fm, out);
    if (COUNT_SIDE) {
        kept = warp_sum32(kept);
        side = warp_sum32(side);
        if ((threadIdx.x & 31) == 0) {
            if (kept) atomicAdd(&ctr[C_TOTAL], (unsigned long long)kept);
            if (side) atomicAdd(&ctr[C_SIDE], (unsigned long long)side);
        }
    }
}

/* ---- multi-GPU: every GPU reads the WHOLE sequence and keeps the k-mers it owns ------------------------
 * The sequence is resident as base-range shards, one per GPU, each with its (k-1)-base overlap and each
 * mapped into every GPU's address space (peer memory over NVLink).  What crosses NVLink is the 2-bit
 * packed bases (0.25 B per start position) instead of 8-byte k-mers: GPU g walks all pieces -- its own
 * first, the others in ring order so that no shard is read by everybody at once -- tests every start
 * position for owner_of(kmer) == g on the window's low word, and appends the k-mers it keeps
 * to a key list in its own HBM (k_collect_owned).  From there the single-GPU pipeline runs unchanged on
 * local data: optimistic level 1 from the key list, level 2, bucket count.  There is no exchange step
 * and nothing to merge.
 *
 * A CTA of 256 threads examines a tile of 256 * WPT packed words of ONE piece (WPT = n_parts / 2, so that it keeps
 * ~ 4096 k-mers; the pieces are padded to whole tiles in the walk order).  The tile's words are staged once in shared
 * memory (one coalesced read, peer or local).  Every thread builds the ownership masks of its WPT consecutive words
 * (bit-parallel for 2 / 4 / 8 owners, see owner_of), one warp scan places the thread in its warp's segment of a
 * shared-memory list (+ a shared overflow area), and ONE loop over the thread's set bits appends a 16-bit code
 * (word << 5 | bit) per owned start -- nineteen instructions per trip, the only divergent part (ncu: 24.7 of 32
 * lanes active over the whole kernel).  The CTA then claims
 * its range of the global list with ONE atomic and the warps expand their codes into k-mers from the staged words,
 * lane per slot: balanced, coalesced 8-byte stores.  ~ 19 KB of shared memory, 32 registers: eight CTAs per SM hide
 * the microseconds a peer load takes. */
constexpr int kMaxPieces = 16;
constexpr int kOwnThreads = 256;
constexpr int kOwnSeg = 576;                                     /* list slots of one warp (mean <= 512, sigma ~ 22) */
constexpr int kOwnOvf = 512;                                     /* shared overflow slots                            */
constexpr int kOwnList = (kOwnThreads / 32) * kOwnSeg + kOwnOvf; /* 5120 codes                                       */

struct OwnedView {
    const uint64_t *ptr[kMaxPieces];  /* first packed word of piece i (local or peer-mapped)                      */
    uint64_t vfirst[kMaxPieces + 1];  /* this GPU walks the items in the order of its piece list: [vfirst[i], vfirst[i+1]), */
    uint64_t nitems[kMaxPieces];      /* of which the first nitems[i] exist (the rest pads the piece to whole tiles) */
    uint64_t gfirst[kMaxPieces];      /* index of the piece's first item (= packed word) in the whole sequence     */
    uint64_t n_rows;                  /* generate_kmers rows of the whole sequence                                */
    uint32_t n_pieces;
};

/* What a kernel needs to tell its owner's k-mers: the hash range of the multiplicative form (lo, span_m1 = its
 * length - 1, so that one owner's whole range of 2^32 hashes fits), or for the linear form the XOR seeds of the
 * rank bits (inv[i] = ~0 when bit i of the rank is 0: the chain then ends in "bit matches") and the taps in force
 * (en, bit p: tap p lies inside the k-mer, i.e. own_tau(p) < 2k). */
struct OwnRange {
    uint32_t lo, span_m1, en, inv[3];
};
__host__ inline OwnRange own_range_of(uint32_t n_parts, uint32_t part, int k)
{
    OwnRange r;
    const uint64_t lo = (((uint64_t)part << 32) + n_parts - 1) / n_parts, hi = (((uint64_t)(part + 1) << 32) + n_parts - 1) / n_parts;
    r.lo = (uint32_t)lo; /* owner r holds the hashes [ceil(r 2^32 / G), ceil((r + 1) 2^32 / G)): what (hash * G) >> 32 == r says */
    r.span_m1 = (uint32_t)(hi - lo - 1);
    r.en = 0;
    for (int p = 0; p < kOwnPool; ++p)
        if (own_tau(p) < 2 * k) r.en |= 1u << p;
    for (int i = 0; i < 3; ++i) r.inv[i] = (part >> i & 1u) ? 0u : ~0u;
    return r;
}

/* Ownership of the 32 starts of the item (w0, low word a2 of its neighbour) as a mask.  MASKLO: k < 16, the low
 * word of a start's window holds bases past the k-mer.
 *   LIN = 0: bit j = start j; per start the funnel shift, hash - lo in one IMAD, compare, select (+ half an add).
 *   LIN = 1..3: bit 2j = start j, bit 2j + 1 = start 16 + j (the two 32-bit halves of the 64 bit positions, of which
 *     the even ones are starts, interleaved): per pool tap one funnel shift per half, per rank bit one XOR chain. */
template <int LIN, bool MASKLO>
__device__ __forceinline__ uint32_t owned_mask(uint64_t w0, uint32_t a2, uint32_t mask_lo, const OwnRange &own)
{
    const uint32_t a0 = (uint32_t)w0, a1 = (uint32_t)(w0 >> 32);
    if (LIN == 0) {
        uint32_t km = 0;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const uint32_t lo = j == 0 ? a0 : j < 16 ? __funnelshift_r(a0, a1, 2 * j) : j == 16 ? a1
                                                                                                 : __funnelshift_r(a1, a2, 2 * j - 32);
            const uint32_t t = (MASKLO ? lo & mask_lo : lo) * kOwnerMul - own.lo;
            km |= (uint32_t)(t <= own.span_m1) << j;
        }
        return km;
    }
    uint32_t f0[3] = {own.inv[0], own.inv[1], own.inv[2]}, f1[3] = {own.inv[0], own.inv[1], own.inv[2]};
#pragma unroll
    for (int p = 0; p < kOwnPool; ++p) {
        bool used = false;
#pragma unroll
        for (int i = 0; i < LIN; ++i) used |= (own_sub(i) >> p & 1u) != 0;
        if (!used) continue;
        uint32_t s0 = own_tau(p) ? __funnelshift_r(a0, a1, own_tau(p)) : a0;
        uint32_t s1 = own_tau(p) ? __funnelshift_r(a1, a2, own_tau(p)) : a1;
        if (MASKLO) {
            const uint32_t on = 0u - (own.en >> p & 1u);
            s0 &= on;
            s1 &= on;
        }
#pragma unroll
        for (int i = 0; i < LIN; ++i)
            if (own_sub(i) >> p & 1u) f0[i] ^= s0, f1[i] ^= s1;
    }
    uint32_t o0 = f0[0], o1 = f1[0];
#pragma unroll
    for (int i = 1; i < LIN; ++i) o0 &= f0[i], o1 &= f1[i];
    return (o0 & 0x55555555u) | ((o1 & 0x55555555u) << 1);
}
/* the mask of the first `n` starts (n < 32) in the layout of owned_mask<LIN> */
template <int LIN>
__device__ __forceinline__ uint32_t first_starts(uint32_t n)
{
    const uint32_t vm = (1u << n) - 1u;
    if (LIN == 0) return vm;
    auto spread = [](uint32_t x) { /* bit j -> bit 2j, j < 16 */
        x = (x | x << 8) & 0x00FF00FFu;
        x = (x | x << 4) & 0x0F0F0F0Fu;
        x = (x | x << 2) & 0x33333333u;
        return (x | x << 1) & 0x55555555u;
    };
    return spread(vm & 0xFFFFu) | spread(vm >> 16) << 1;
}
/* bit offset (2 * start) of the window a mask bit stands for */
template <int LIN>
__device__ __forceinline__ uint32_t start_shift(uint32_t bit)
{
    return LIN == 0 ? 2 * bit : (bit & 30u) | (bit & 1u) << 5;
}

/* virtual item v -> packed words and number of valid starts (0: padding) */
__device__ __forceinline__ int owned_item(const OwnedView &ov, uint64_t v, uint64_t &w0, uint64_t &w1)
{
    uint32_t i = 0;
    while (i + 1 < ov.n_pieces && v >= ov.vfirst[i + 1]) ++i;
    const uint64_t off = v - ov.vfirst[i];
    if (off >= ov.nitems[i]) return 0;
    const uint64_t *w = ov.ptr[i] + off;
    w0 = ld_nc(w);
    w1 = ld_nc(w + 1);
    const uint64_t left = ov.n_rows - (ov.gfirst[i] + off) * 32;
    return left < 32 ? (int)left : 32;
}

/* The owned k-mers of the sequence as a key list (unordered).  `cursor` ends at the number of owned rows even
 * when tiles past `cap` wrote nothing; a tile whose shared-memory list overflowed (a long run of one k-mer owned
 * by this GPU) raises C_L1OVF: the caller then uses k_collect_owned_any. */
template <int WPT, int LIN, bool MASKLO>
__global__ void __launch_bounds__(kOwnThreads) k_collect_owned(OwnedView ov, uint64_t mask, OwnRange own, uint64_t cap,
                                                               unsigned long long *__restrict__ ctr,
                                                               uint64_t *__restrict__ out)
{
    constexpr int T = kOwnThreads * WPT; /* words of a tile; vfirst[] are multiples of T */
    static_assert(T <= 2048 && (WPT == 1 || WPT == 2 || WPT == 4), "a code holds 11 bits of word index");
    __shared__ __align__(16) uint64_t words[T + 2];
    __shared__ uint16_t codes[kOwnList];
    __shared__ uint32_t n_ovf_s, wtot_s[kOwnThreads / 32];
    __shared__ unsigned long long base_s;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) n_ovf_s = 0;
    const uint64_t v0 = (uint64_t)blockIdx.x * T;
    uint32_t pi = 0;
    while (pi + 1 < ov.n_pieces && v0 >= ov.vfirst[pi + 1]) ++pi;
    const uint64_t off0 = v0 - ov.vfirst[pi];
    const uint64_t have = ov.nitems[pi] > off0 ? ov.nitems[pi] - off0 : 0;
    const uint32_t n_valid = have < (uint64_t)T ? (uint32_t)have : (uint32_t)T; /* uniform */
    if (n_valid == 0) return;
    {
        const uint64_t *src = ov.ptr[pi] + off0;
#pragma unroll
        for (int it = 0; it < WPT; ++it) {
            const uint32_t idx = it * kOwnThreads + tid;
            words[idx] = idx <= n_valid ? ld_nc(src + idx) : 0ull; /* [n_valid]: the last item's neighbour (overlap or pad word) */
        }
        if (tid == 0 && n_valid == (uint32_t)T) words[T] = ld_nc(src + T);
    }
    __syncthreads();
    const uint32_t mask_lo = (uint32_t)mask;
    /* starts from the tile's first word to the end of the sequence (>= 1 per existing item) */
    const uint64_t left0_64 = ov.n_rows - (ov.gfirst[pi] + off0) * 32;
    const uint32_t left0 = left0_64 < (uint64_t)T * 32 ? (uint32_t)left0_64 : (uint32_t)T * 32;
    /* 1. the masks of this thread's WPT consecutive words */
    const uint32_t i0 = tid * WPT;
    uint32_t km[WPT];
    {
        uint64_t w[WPT];
        if (WPT == 4) {
            const uint4 x = *reinterpret_cast<const uint4 *>(&words[i0]), y = *reinterpret_cast<const uint4 *>(&words[i0 + 2]);
            w[0] = (uint64_t)x.y << 32 | x.x, w[1] = (uint64_t)x.w << 32 | x.z;
            w[WPT - 2] = (uint64_t)y.y << 32 | y.x, w[WPT - 1] = (uint64_t)y.w << 32 | y.z;
        } else if (WPT == 2) {
            const uint4 x = *reinterpret_cast<const uint4 *>(&words[i0]);
            w[0] = (uint64_t)x.y << 32 | x.x, w[WPT - 1] = (uint64_t)x.w << 32 | x.z;
        } else {
            w[0] = words[i0];
        }
        /* the low word after the thread's last: the next lane's first (lane 31 reads it) */
        uint32_t nxt = __shfl_down_sync(0xffffffffu, (uint32_t)w[0], 1);
        if (lane == 31) nxt = (uint32_t)words[i0 + WPT];
#pragma unroll
        for (int it = 0; it < WPT; ++it) {
            const uint32_t idx = i0 + it;
            km[it] = 0;
            if (idx < n_valid) {
                km[it] = owned_mask<LIN, MASKLO>(w[it], it + 1 < WPT ? (uint32_t)w[it + 1 < WPT ? it + 1 : it] : nxt, mask_lo, own);
                const uint32_t left = left0 - idx * 32;
                if (left < 32) km[it] &= first_starts<LIN>(left);
            }
        }
    }
    /* 2. the thread's place in the warp's segment */
    uint32_t n = 0;
#pragma unroll
    for (int it = 0; it < WPT; ++it) n += __popc(km[it]);
    uint32_t inc = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (uint32_t)o) inc += y;
    }
    uint32_t p = inc - n;
    const uint32_t wcur = __shfl_sync(0xffffffffu, inc, 31);
    /* 3. one loop over all set bits of the thread: masks move down as they empty */
    {
        const uint32_t seg_addr = (uint32_t)__cvta_generic_to_shared(&codes[warp * kOwnSeg]);
        uint32_t m0 = km[0], m1 = WPT > 1 ? km[WPT > 1 ? 1 : 0] : 0, m2 = WPT > 2 ? km[WPT > 2 ? 2 : 0] : 0, m3 = WPT > 3 ? km[WPT > 3 ? 3 : 0] : 0;
        uint32_t code0 = i0 << 5;
#pragma unroll 1
        for (; n; --n) {
            if (m0 == 0) {
#pragma unroll 1
                do {
                    m0 = m1, m1 = m2, m2 = m3, m3 = 0;
                    code0 += 32;
                } while (m0 == 0);
            }
            const uint32_t code = code0 | (uint32_t)(__ffs(m0) - 1);
            m0 &= m0 - 1;
            if (p < (uint32_t)kOwnSeg) { /* (the address spelled out: the compiler rebuilds the array base per store) */
                asm volatile("st.shared.u16 [%0], %1;" ::"r"(seg_addr + 2 * p), "h"((uint16_t)code) : "memory");
            } else {
                const uint32_t q = atomicAdd(&n_ovf_s, 1u);
                if (q < (uint32_t)kOwnOvf) codes[(kOwnThreads / 32) * kOwnSeg + q] = (uint16_t)code;
            }
            ++p;
        }
    }
    const uint32_t wn = min(wcur, (uint32_t)kOwnSeg);
    if (lane == 0) wtot_s[warp] = wn;
    __syncthreads();
    const uint32_t n_ovf = n_ovf_s, on = min(n_ovf, (uint32_t)kOwnOvf);
    uint32_t before = 0, total = on;
#pragma unroll
    for (int i = 0; i < kOwnThreads / 32; ++i) {
        const uint32_t t = wtot_s[i];
        if (i < (int)warp) before += t;
        total += t;
    }
    if (tid == 0) {
        if (n_ovf > (uint32_t)kOwnOvf) atomicExch(&ctr[C_L1OVF], 1ull); /* keys were dropped */
        base_s = total ? atomicAdd(&ctr[C_CURSOR], (unsigned long long)total) : 0ull;
    }
    __syncthreads();
    if (total == 0 || base_s + total > cap) return; /* uniform */
    /* 4. codes -> k-mers, lane per slot */
    uint64_t *dst = out + base_s;
    auto kmer_of = [&](uint32_t code) {
        const uint32_t idx = code >> 5;
        return window(words[idx], words[idx + 1], start_shift<LIN>(code & 31u)) & mask;
    };
    for (uint32_t q = lane; q < wn; q += 32) dst[before + q] = kmer_of(codes[warp * kOwnSeg + q]);
    for (uint32_t q = tid; q < on; q += kOwnThreads) dst[total - on + q] = kmer_of(codes[(kOwnThreads / 32) * kOwnSeg + q]);
}

/* The same list for ANY input (the exact fallback: heavily repeated sequences): appended warp by warp through the
 * cursor, nothing staged, nothing dropped. */
template <int LIN>
__global__ void __launch_bounds__(kScatThreads) k_collect_owned_any(OwnedView ov, uint64_t mask, OwnRange own, uint64_t cap,
                                                                    unsigned long long *__restrict__ cursor,
                                                                    uint64_t *__restrict__ out)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t n_vitems = ov.vfirst[ov.n_pieces];
    for (uint64_t vb = (uint64_t)blockIdx.x * kScatThreads; vb < n_vitems; vb += (uint64_t)gridDim.x * kScatThreads) {
        const uint64_t v = vb + threadIdx.x;
        uint64_t w0 = 0, w1 = 0;
        uint32_t km = 0;
        if (v < n_vitems) {
            const int c = owned_item(ov, v, w0, w1);
            if (c > 0) km = owned_mask<LIN, true>(w0, (uint32_t)w1, (uint32_t)mask, own);
            if (c < 32) km &= first_starts<LIN>((uint32_t)c);
        }
        const uint32_t n = __popc(km);
        uint32_t inc = n;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= (uint32_t)o) inc += y;
        }
        const uint32_t wtotal = __shfl_sync(0xffffffffu, inc, 31);
        unsigned long long base = 0;
        if (lane == 31 && wtotal) base = atomicAdd(cursor, (unsigned long long)wtotal);
        base = __shfl_sync(0xffffffffu, base, 31);
        if (base + wtotal > cap) continue; /* warp-uniform */
        uint64_t p = base + inc - n;
        while (km) {
            const int j = __ffs(km) - 1;
            km &= km - 1;
            out[p++] = window(w0, w1, start_shift<LIN>((uint32_t)j)) & mask;
        }
    }
}

/* ---- count: one bucket at a time in a shared-memory table ------------------------------------- */
constexpr int kPre = kBucketSlots / 2 / kThreads; /* keys per thread fetched one bucket ahead (covers the mean bucket) */

/* slot inside a bucket: fold the key and multiply once (32-bit); the digits came from
 * a different multiplier over the unfolded key, so the two are independent in practice */
__device__ __forceinline__ uint32_t bucket_slot(uint64_t x)
{
    return (((uint32_t)x ^ (uint32_t)(x >> 32)) * 0x9E3779B1u) >> (32 - kBucketSlotBits);
}

struct BucketTally {
    uint32_t distinct;
    int32_t unique;
};

/* distinct / unique are accounted at insert time: a claim is a new distinct AND unique key; the
 * first extra occurrence (the add returns 0) takes the key out of the unique set.  No scan. */
template <class CT>
__device__ __forceinline__ void bucket_insert(unsigned long long *tk, CT *tc, uint64_t x, bool spill_ok,
                                              Slot *__restrict__ spill, uint64_t spill_cap, BucketTally &bt,
                                              Tally &ty, unsigned long long *ctr)
{
    uint32_t sl = bucket_slot(x);
    int probes = 0;
    for (;;) {
        unsigned long long old = atomicCAS(&tk[sl], (unsigned long long)kEmpty, (unsigned long long)x);
        if (old == kEmpty) {
            bt.distinct++;
            bt.unique++;
            return;
        }
        if (old == x) {
            bt.unique -= (atomicAdd(&tc[sl], (CT)1) == 0);
            return;
        }
        sl = (sl + 1) & (kBucketSlots - 1);
        if (++probes == kBucketSlots) { /* table full of other keys: count it in HBM */
            if (spill_ok) hash_insert(spill, spill_cap, x, ty, ctr);
            return;
        }
    }
}

/* CT, the per-slot count of extra occurrences: uint32_t unless the call has 2^32 - 1 or more keys, where one key
 * can occur 2^32 + 1 times and a 32-bit count would wrap (unsigned long long, 16 bytes per slot).
 * SPEC (not with EMIT): a bucket's keys are all in that bucket, so once it has drained every occupied slot holds its
 * group's final count; those are binned into the direct part of the spectrum (kSpecSmem more bytes of dynamic shared
 * memory, after the table).  Spilled keys are binned from the spill table afterwards. */
template <bool EMIT, class CT = uint32_t, bool SPEC = false>
__global__ void __launch_bounds__(kThreads) k_count_buckets(const uint64_t *__restrict__ keys,
                                                            const uint64_t *__restrict__ bucket_off,
                                                            const uint64_t *__restrict__ bucket_end,
                                                            uint64_t n_buckets, Slot *__restrict__ spill,
                                                            uint64_t spill_cap,
                                                            unsigned long long *__restrict__ ctr,
                                                            uint64_t *__restrict__ out_kmers,
                                                            uint64_t *__restrict__ out_counts,
                                                            const uint32_t *__restrict__ list = nullptr,
                                                            const unsigned long long *__restrict__ list_n = nullptr,
                                                            unsigned long long *__restrict__ spec_direct = nullptr,
                                                            uint32_t max_count = 0)
{
    static_assert(!(EMIT && SPEC), "the emitting pass re-runs a count whose spectrum is already taken");
    /* with a list: only the buckets list[0 .. *list_n) (the ones k_count_buckets_bins passed on) */
    if (list) n_buckets = *list_n;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned long long *tk = reinterpret_cast<unsigned long long *>(smem_raw);                /* keys   */
    CT *tc = reinterpret_cast<CT *>(smem_raw + sizeof(uint64_t) * kBucketSlots); /* extras */
    __shared__ unsigned long long row_base;
#define SPEC_BINS SpecBins(reinterpret_cast<uint32_t *>(smem_raw + (sizeof(uint64_t) + sizeof(CT)) * kBucketSlots), \
                           spec_direct, max_count)
    if constexpr (SPEC) SPEC_BINS.zero(); /* before the first barrier of the loop; flushed after the last */
    Tally ty = {0, 0, 0, 0}; /* spilled keys account themselves through hash_insert */
    BucketTally bt = {0, 0};
    uint64_t b = blockIdx.x;
    uint64_t beg = 0, end = 0;
    uint64_t pre[kPre];
    if (b < n_buckets) {
        const uint64_t id = list ? list[b] : b;
        beg = bucket_off[id];
        end = bucket_end[id];
#pragma unroll
        for (int u = 0; u < kPre; ++u) {
            uint64_t i = beg + (uint64_t)u * kThreads + threadIdx.x;
            pre[u] = i < end ? ld_nc(keys + i) : kEmpty;
        }
    }
    while (b < n_buckets) {
        const uint64_t nb = b + gridDim.x;
        uint64_t nbeg = 0, nend = 0;
        if (nb < n_buckets) {
            const uint64_t id = list ? list[nb] : nb;
            nbeg = bucket_off[id];
            nend = bucket_end[id];
        }
        { /* 48 (64) KB of 16-byte stores */
            ulonglong2 *k2 = reinterpret_cast<ulonglong2 *>(tk);
            uint4 *c4 = reinterpret_cast<uint4 *>(tc);
#pragma unroll
            for (int i = 0; i < kBucketSlots / 2 / kThreads; ++i)
                k2[i * kThreads + threadIdx.x] = make_ulonglong2(kEmpty, kEmpty);
#pragma unroll
            for (int i = 0; i < kBucketSlots * (int)sizeof(CT) / 16 / kThreads; ++i)
                c4[i * kThreads + threadIdx.x] = make_uint4(0, 0, 0, 0);
        }
        __syncthreads();
        /* EMIT re-runs the count: rows of spilled keys come from the spill table itself.
         * The shared-memory CAS pipe is what bounds this kernel, and a CAS issued for one lane costs as
         * much as one issued for 32.  So probing is organised in ROUNDS: first probes of all prefetched
         * keys go out back to back; then, while any lane of the warp still has a key that met a different
         * key, every such lane re-probes its OLDEST pending key in the same instruction.  Rounds needed =
         * the largest per-lane total of extra probes, not the sum of per-key maxima. */
        {
            uint32_t sl[kPre], pending = 0;
#pragma unroll
            for (int u = 0; u < kPre; ++u) sl[u] = bucket_slot(pre[u]);
            unsigned long long old[kPre];
#pragma unroll
            for (int u = 0; u < kPre; ++u) {
                old[u] = pre[u];
                if (pre[u] != kEmpty)
                    old[u] = atomicCAS(&tk[sl[u]], (unsigned long long)kEmpty, (unsigned long long)pre[u]);
            }
#pragma unroll
            for (int u = 0; u < kPre; ++u) {
                if (pre[u] == kEmpty) continue;
                if (old[u] == kEmpty) {
                    bt.distinct++;
                    bt.unique++;
                } else if (old[u] == pre[u]) {
                    bt.unique -= (atomicAdd(&tc[sl[u]], (CT)1) == 0);
                } else {
                    pending |= 1u << u;
                }
            }
            uint64_t key = 0;
            uint32_t slot = 0, probes = 0;
            int cur = -1;
            while (__any_sync(0xffffffffu, pending != 0)) {
                if (pending) {
                    const int u = __ffs(pending) - 1;
                    if (u != cur) { /* next pending key of this lane: fetch it out of the register arrays */
                        cur = u;
                        probes = 0;
#pragma unroll
                        for (int v = 0; v < kPre; ++v)
                            if (v == u) {
                                key = pre[v];
                                slot = sl[v];
                            }
                    }
                    slot = (slot + 1) & (kBucketSlots - 1);
                    const unsigned long long o = atomicCAS(&tk[slot], (unsigned long long)kEmpty, (unsigned long long)key);
                    if (o == kEmpty) {
                        bt.distinct++;
                        bt.unique++;
                        pending &= pending - 1;
                    } else if (o == key) {
                        bt.unique -= (atomicAdd(&tc[slot], (CT)1) == 0);
                        pending &= pending - 1;
                    } else if (++probes == kBucketSlots) { /* table full of other keys: count it in HBM */
                        if (!EMIT) hash_insert(spill, spill_cap, key, ty, ctr);
                        pending &= pending - 1;
                    }
                }
            }
        }
        for (uint64_t i = beg + (uint64_t)kPre * kThreads + threadIdx.x; i < end; i += kThreads)
            bucket_insert(tk, tc, ld_nc(keys + i), !EMIT, spill, spill_cap, bt, ty, ctr);
        /* next bucket's keys fly while this one drains and the table is re-initialised */
#pragma unroll
        for (int u = 0; u < kPre; ++u) {
            uint64_t i = nbeg + (uint64_t)u * kThreads + threadIdx.x;
            pre[u] = i < nend ? ld_nc(keys + i) : kEmpty;
        }
        __syncthreads();
        if (EMIT) {
            uint32_t mine = 0;
            for (int i = threadIdx.x; i < kBucketSlots; i += kThreads) mine += (tk[i] != kEmpty);
            uint32_t total;
            uint32_t rank = block_exscan(mine, &total);
            if (threadIdx.x == 0) row_base = atomicAdd(&ctr[C_CURSOR], (unsigned long long)total);
            __syncthreads();
            uint64_t pos = row_base + rank;
            for (int i = threadIdx.x; i < kBucketSlots; i += kThreads)
                if (tk[i] != kEmpty) {
                    out_kmers[pos] = tk[i];
                    out_counts[pos] = (uint64_t)tc[i] + 1;
                    pos++;
                }
            __syncthreads();
        }
        if constexpr (SPEC) {
            SpecBins sb = SPEC_BINS;
            for (int i = threadIdx.x; i < kBucketSlots; i += kThreads)
                if (tk[i] != kEmpty) sb.add((uint64_t)tc[i] + 1);
            __syncthreads(); /* before the next bucket clears the table */
        }
        b = nb;
        beg = nbeg;
        end = nend;
    }
    if constexpr (SPEC) {
        __syncthreads();
        SPEC_BINS.flush();
    }
#undef SPEC_BINS
    uint32_t d = warp_sum32(bt.distinct);
    int32_t u = (int32_t)__reduce_add_sync(0xffffffffu, bt.unique);
    if ((threadIdx.x & 31) == 0) {
        if (d) atomicAdd(&ctr[C_DISTINCT], (unsigned long long)d);
        if (u) atomicAdd(&ctr[C_UNIQUE], (unsigned long long)(long long)u);
    }
    ty.total = 0; /* totals were taken by the scatter pass */
    tally_flush(ty, ctr);
}

/* ---- bucket count without a hash table: bin, place, compare -------------------------------------
 * The aggregates (distinct, unique) of a bucket need no table.  The bucket's keys are spread over
 * kBins sub-bins by an independent hash with a RETURNING shared-memory add (11.6 lane-ops/clk/SM
 * against 3.1 for the 64-bit CAS of the table, profiles/r01e_microbench); the value returned is the
 * key's rank r inside its bin.  Each warp scans the counts of its own bins with shuffles, the keys
 * are placed bin by bin into a staging area (slot = start of the bin + r), and every staged key is
 * compared with the slots before it (the first three branch-free; further ones, up to the bin's start,
 * only when the third holds a key of its bin):
 *     e = earlier keys equal to mine;  repeats += (e >= 1);  second += (e == 1);
 *     distinct = keys - repeats;  unique = distinct - second  (unique iff no second occurrence).
 * No rank is stored for the compare: the bin and the bucket are both functions of the key, so a slot
 * outside my bin -- another bin, another warp's region, or a stale key of an earlier bucket -- never
 * holds a key equal to mine, and looking back past the start of the bin cannot change e.
 * No probe chains, no 48 KB table to clear, three barriers per bucket.  The kernel is bound by issue
 * slots, so it is written as straight-line code: lanes past the end of a bucket work on dummy bins and
 * slots, and the rank / place / load phases are instantiated per number of key rows (BINS_DISPATCH).
 * A bucket this cannot hold -- more than kBinCap keys, a warp's region overflowing, or a bin with
 * more than kBinHeavy keys (a k-mer with many copies) -- is appended to `list` and counted by the
 * table kernel afterwards (k_count_buckets with the list). */
constexpr int kBins = 2048;
constexpr int kBinPer = 12;                      /* keys per thread held in registers            */
constexpr int kBinCap = kBinPer * kThreads;      /* 3072 keys staged per bucket                  */
constexpr int kBinWarpCap = kBinCap / (kThreads / 32); /* staging slots of the bins of one warp  */
constexpr int kBinHeavy = 15;                    /* rank fits 4 bits, position 12 bits           */
static_assert(kBins == 8 * kThreads && kBinCap <= 4096, "packing of k_count_buckets_bins");

__device__ __forceinline__ uint32_t bin_of(uint64_t x)
{
    return (((uint32_t)x ^ (uint32_t)(x >> 32)) * 0x9E3779B1u) >> 21;
}

/* phases A and C for a bucket of at most ROWS x kThreads keys: straight-line code, the lanes past the end of
 * the bucket work on their dummy entries */
template <int ROWS>
__device__ __forceinline__ void bins_rank(const uint64_t (&x)[kBinPer], uint32_t (&f)[kBinPer / 2], uint32_t n,
                                          uint32_t tid, uint32_t lane, uint32_t *cnt)
{
#pragma unroll
    for (int u = 0; u < ROWS; ++u) {
        const uint32_t bin = u * kThreads + tid < n ? bin_of(x[u]) : kBins + lane;
        const uint32_t v = bin | (atomicAdd(&cnt[bin], 1u) << 12);
        f[u >> 1] = (u & 1) ? __byte_perm(f[u >> 1], v, 0x5410) : v;
    }
}

template <int ROWS>
__device__ __forceinline__ void bins_load(uint64_t (&x)[kBinPer], const uint64_t *__restrict__ src, uint32_t n, uint32_t tid)
{
#pragma unroll
    for (int u = 0; u < ROWS; ++u)
        if (u * kThreads + tid < n) x[u] = ld_nc(src + u * kThreads);
}

template <int ROWS>
__device__ __forceinline__ void bins_place(const uint64_t (&x)[kBinPer], const uint32_t (&f)[kBinPer / 2],
                                           const uint16_t *st, uint64_t *stage)
{
#pragma unroll
    for (int u = 0; u < ROWS; ++u) {
        const uint32_t v = (u & 1) ? (f[u >> 1] >> 16) : (f[u >> 1] & 0xffffu);
        stage[st[v & 0xfffu] + (v >> 12)] = x[u];
    }
}

#define BINS_DISPATCH(n, CALL)                                   \
    do {                                                         \
        if ((n) <= 4 * kThreads) { constexpr int ROWS = 4; CALL; } \
        else if ((n) <= 6 * kThreads) { constexpr int ROWS = 6; CALL; } \
        else if ((n) <= 8 * kThreads) { constexpr int ROWS = 8; CALL; } \
        else { constexpr int ROWS = kBinPer; CALL; }               \
    } while (0)

/* SPEC also takes the cumulative spectrum C[j] (groups of count >= j) of the buckets it counts, into spec_cum[j]:
 * a group of count m has exactly one key with e = j - 1 for each j = 1 .. m, so C[1] = keys - repeats, C[2] = second,
 * and C[j >= 3] = keys with e = j - 1 (rare: repeated k-mers only).  A bin holds at most kBinHeavy keys: j <= 15. */
template <bool SPEC = false>
__global__ void __launch_bounds__(kThreads, 4) k_count_buckets_bins(const uint64_t *__restrict__ keys,
                                                                    const uint64_t *__restrict__ bucket_off,
                                                                    const uint64_t *__restrict__ bucket_end,
                                                                    uint64_t n_buckets,
                                                                    unsigned long long *__restrict__ ctr,
                                                                    uint32_t *__restrict__ list,
                                                                    unsigned long long *__restrict__ list_n,
                                                                    unsigned long long *__restrict__ spec_cum = nullptr)
{
    static_assert(kBinHeavy < kSpecCum, "the cumulative spectrum of a bin");
    uint32_t *scum = nullptr; /* keys with e = j - 1 >= 2, by j */
    if constexpr (SPEC) {
        __shared__ uint32_t scum_s[kSpecCum];
        scum = scum_s;
        if (threadIdx.x < kSpecCum) scum[threadIdx.x] = 0; /* before the first barrier */
    }
    /* every array ends in dummy entries, one per lane (+ 15 for a dummy's meaningless 4-bit rank): the lanes
     * past the end of a bucket's last row work on those instead of branching around the atomics and the stores */
    /* 4 slots in front: the compare phase looks back 3.  The dummy slots stage[kBinCap ..] hold whatever the lanes
     * past the end of a bucket place there; the compare phase reads only slots before base + wtotal <= kBinCap. */
    __shared__ __align__(16) uint64_t stage_raw[4 + kBinCap + 48];
    uint64_t *const stage = stage_raw + 4;
    __shared__ __align__(16) uint32_t cnt[kBins + 32];
    __shared__ __align__(16) uint16_t st[kBins + 32]; /* start of the bin in `stage` */
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t repeats = 0, second = 0; /* keys with >= 1 / exactly 1 equal key before them in their bin */
    unsigned long long placed = 0;    /* thread 0: keys of the buckets counted here */
    for (int i = tid; i < kBins + 32; i += kThreads) cnt[i] = 0;
    /* kEmpty never reaches a bucket ('G' x 32 is counted on the side), so a slot never written since the launch
     * never equals a key: the look-back may read it */
    for (int i = tid; i < 4 + kBinCap + 48; i += kThreads) stage_raw[i] = kEmpty;
    if (tid < 32) st[kBins + tid] = (uint16_t)(kBinCap + tid);
    uint64_t b = blockIdx.x;
    uint32_t n = 0;
    uint64_t x[kBinPer];
#pragma unroll
    for (int u = 0; u < kBinPer; ++u) x[u] = 0;
    if (b < n_buckets) {
        const uint64_t beg = bucket_off[b];
        n = (uint32_t)min(bucket_end[b] - beg, (uint64_t)kBinCap + 1);
        if (n <= kBinCap) BINS_DISPATCH(n, bins_load<ROWS>(x, keys + beg + tid, n, tid));
    }
    __syncthreads();
    while (b < n_buckets) {
        const uint64_t nb = b + gridDim.x;
        uint64_t nbeg = 0;
        uint32_t nn = 0;
        if (nb < n_buckets) {
            nbeg = bucket_off[nb];
            nn = (uint32_t)min(bucket_end[nb] - nbeg, (uint64_t)kBinCap + 1);
        }
        bool pass_on = n > kBinCap; /* uniform */
        uint32_t wtotal = 0;        /* keys in the bins of this warp */
        if (!pass_on) {
            uint32_t f[kBinPer / 2]; /* two 16-bit fields per register: rank (4 bits, on top) and bin (12 bits) */
            /* A: rank of every key inside its bin */
            BINS_DISPATCH(n, bins_rank<ROWS>(x, f, n, tid, lane, cnt));
            __syncthreads();
            /* B: the owner of the bins 4 tid .. 4 tid + 3 and kBins / 2 + 4 tid .. + 3 (a 16-byte lane stride: no
             * bank conflict) reads their counts and clears them; warp scan -> starts.  Warp w's region of the stage
             * holds its bins 128 w .. 128 w + 127 and kBins / 2 + 128 w .. in thread order. */
            uint32_t *const cnt_lo = &cnt[4 * tid], *const cnt_hi = &cnt[kBins / 2 + 4 * tid];
            const uint4 c0 = *reinterpret_cast<const uint4 *>(cnt_lo);
            const uint4 c1 = *reinterpret_cast<const uint4 *>(cnt_hi);
            *reinterpret_cast<uint4 *>(cnt_lo) = make_uint4(0, 0, 0, 0);
            *reinterpret_cast<uint4 *>(cnt_hi) = make_uint4(0, 0, 0, 0);
            const uint32_t s1 = c0.x, s2 = s1 + c0.y, s3 = s2 + c0.z, s4 = s3 + c0.w, s5 = s4 + c1.x, s6 = s5 + c1.y,
                           s7 = s6 + c1.z, mine = s7 + c1.w;
            const uint32_t worst = max(max(max(c0.x, c0.y), max(c0.z, c0.w)), max(max(c1.x, c1.y), max(c1.z, c1.w)));
            uint32_t inc = mine;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += y;
            }
            wtotal = __shfl_sync(0xffffffffu, inc, 31);
            const bool bad = wtotal > (uint32_t)kBinWarpCap || worst > (uint32_t)kBinHeavy;
            const uint32_t p = warp * kBinWarpCap + inc - mine;
            /* (harmless when bad: the bucket is passed on and st is not read) */
            *reinterpret_cast<uint2 *>(&st[4 * tid]) = make_uint2(p | ((p + s1) << 16), (p + s2) | ((p + s3) << 16));
            *reinterpret_cast<uint2 *>(&st[kBins / 2 + 4 * tid]) =
                make_uint2((p + s4) | ((p + s5) << 16), (p + s6) | ((p + s7) << 16));
            pass_on = __syncthreads_or(bad);
            if (!pass_on) {
                /* C: place */
                BINS_DISPATCH(n, bins_place<ROWS>(x, f, st, stage));
                if (tid == 0) placed += n;
            }
        }
        /* the next bucket's keys fly during the compare phase */
        if (nn <= kBinCap) BINS_DISPATCH(nn, bins_load<ROWS>(x, keys + nbeg + tid, nn, tid));
        if (n <= kBinCap) { /* uniform: the barriers above were taken */
            __syncthreads();
            if (!pass_on) {
                /* D: a key against the keys placed before it in its bin.  A warp walks the region of its own
                 * bins; a slot outside the bin never equals the key, so it needs no bound. */
                const uint32_t base = warp * kBinWarpCap;
                for (uint32_t q = base + lane; q < base + wtotal; q += 32) {
                    /* three look-backs without a branch: neighbouring lanes read neighbouring slots */
                    const uint64_t key = stage[q], k1 = stage[q - 1], k2 = stage[q - 2], k3 = stage[q - 3];
                    uint32_t e = (uint32_t)(k1 == key) + (uint32_t)(k2 == key) + (uint32_t)(k3 == key);
                    const uint32_t bin = bin_of(key);
                    if (bin_of(k3) == bin) { /* rare (rank >= 3): kept out of line (the rolled loop's set-up was 13 % of the kernel's instructions, ncu r02c) */
                        /* the rank from the bin's start, which phase B left in st (walking on while the slots
                         * hold keys of the bin measured 2 % slower at k = 14, where many k-mers repeat) */
                        const uint32_t r = q - st[bin];
#pragma unroll 1
                        for (uint32_t j = 4; j <= r; ++j) e += stage[q - j] == key;
                    }
                    repeats += e >= 1;
                    second += e == 1;
                    if constexpr (SPEC)
                        if (e >= 2) atomicAdd(&scum[e + 1], 1u);
                }
            }
        }
        if (pass_on && tid == 0) list[atomicAdd(list_n, 1ull)] = (uint32_t)b;
        b = nb;
        n = nn;
    }
    /* distinct = keys - repeats; unique = distinct - second (a key is unique iff it has no second occurrence) */
    repeats = warp_sum32(repeats);
    second = warp_sum32(second);
    if (lane == 0 && (repeats | second)) {
        atomicAdd(&ctr[C_DISTINCT], (unsigned long long)(-(long long)repeats));
        atomicAdd(&ctr[C_UNIQUE], (unsigned long long)(-(long long)repeats - (long long)second));
    }
    if (tid == 0 && placed) {
        atomicAdd(&ctr[C_DISTINCT], placed);
        atomicAdd(&ctr[C_UNIQUE], placed);
    }
    if constexpr (SPEC) {
        if (lane == 0 && (repeats | second)) {
            atomicAdd(&spec_cum[1], (unsigned long long)(-(long long)repeats));
            atomicAdd(&spec_cum[2], (unsigned long long)second);
        }
        if (tid == 0 && placed) atomicAdd(&spec_cum[1], placed);
        __syncthreads();
        if (tid >= 3 && tid < kSpecCum && scum[tid]) atomicAdd(&spec_cum[tid], (unsigned long long)scum[tid]);
    }
}

/* ---- multi-CTA exclusive scan (bucket offsets: up to 4 M entries) ------------------------------ */
constexpr int kScanPer = 8; /* 1024 threads x 8 = 8192 entries per CTA */
__global__ void __launch_bounds__(1024) k_scan_block(const uint64_t *__restrict__ in, uint64_t n,
                                                     uint64_t *__restrict__ out,
                                                     uint64_t *__restrict__ block_sums)
{
    __shared__ uint64_t wtot[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint64_t base = ((uint64_t)blockIdx.x * 1024 + threadIdx.x) * kScanPer;
    uint64_t v[kScanPer], sum = 0;
#pragma unroll
    for (int i = 0; i < kScanPer; ++i) {
        v[i] = base + i < n ? in[base + i] : 0;
        sum += v[i];
    }
    uint64_t inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint64_t y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    if (lane == 31) wtot[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        uint64_t t = wtot[lane], ti = t;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint64_t y = __shfl_up_sync(0xffffffffu, ti, o);
            if (lane >= o) ti += y;
        }
        wtot[lane] = ti - t;
        if (lane == 31) block_sums[blockIdx.x] = ti;
    }
    __syncthreads();
    uint64_t ex = wtot[wid] + inc - sum;
#pragma unroll
    for (int i = 0; i < kScanPer; ++i) {
        if (base + i < n) out[base + i] = ex;
        ex += v[i];
    }
}

__global__ void __launch_bounds__(1024) k_scan_add(uint64_t *__restrict__ out, uint64_t n,
                                                   const uint64_t *__restrict__ block_off)
{
    const uint64_t add = block_off[blockIdx.x];
    const uint64_t base = ((uint64_t)blockIdx.x * 1024 + threadIdx.x) * kScanPer;
#pragma unroll
    for (int i = 0; i < kScanPer; ++i)
        if (base + i < n) out[base + i] += add;
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) out[n] = block_off[gridDim.x];
}

} /* namespace dnagpu */
