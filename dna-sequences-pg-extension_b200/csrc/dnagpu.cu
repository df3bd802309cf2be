/*
 * dnagpu.cu -- the C ABI of libdnagpu (include/dnagpu.h) over the sm_100a
 * kernels in kernels.cuh.  Host-side logic only: argument checks that mirror
 * the reference's ereport(ERROR) sites, device memory, launch geometry.
 *
 * There is no CPU implementation of any operation in this file: when no
 * sm_100 device is usable dnagpu_create fails and nothing else can run.
 */
#include "../../include/dnagpu.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <thread>
#include <unordered_set>
#include <vector>

#include "kernels.cuh"
#include "partition.cuh"
#include "index.cuh"

using namespace dnagpu;

/* ---- objects ----------------------------------------------------------------- */
struct ProfRec {
    std::string name;
    cudaEvent_t e0, e1;
};

struct dnagpu_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    unsigned long long *d_ctr = nullptr; /* C_COUNT + kMaxParts*2 u64 device counters */
    int bins_ctas_per_sm = 4;            /* resident CTAs of k_count_buckets_bins (occupancy query) */
    unsigned long long *h_ctr = nullptr; /* pinned mirror */
    /* the abundance spectrum of the running query (dnagpu_count_spectrum): kSpecCum + spec_h u64 (kernels.cuh), grown on
     * demand; spec_h = 0 outside such a query.  spec_side = the copies of 'G' x 32 (k = 32), a group of its own. */
    unsigned long long *d_spec = nullptr;
    uint32_t spec_alloc = 0, spec_h = 0;
    uint64_t spec_side = 0;
    cudaStream_t copy_stream = nullptr; /* H2D of the host-buffer calls, overlapped with level 1 */
    /* dnagpu_create_multi: the contexts of devices[1..] (this one is devices[0]) and one shard buffer per GPU */
    std::vector<dnagpu_ctx *> peers;
    std::vector<uint64_t *> shard_buf; /* plain cudaMalloc (peer-accessible), grown on demand */
    std::vector<uint64_t> shard_cap;   /* words */
    bool profiling = false;
    bool plane_filter = false; /* DNAGPU_WHERE_FLAG_PLANES of the running query */
    bool force_exact = false; /* DNAGPU_COUNT_FLAG_EXACT of the running query: no optimistic partition regions */
    std::vector<ProfRec> prof;
    /* live child handles: dnagpu_destroy releases their device memory and orphans them (ctx = NULL), so a
     * *_free that comes after the destroy only deletes the host struct */
    std::unordered_set<dnagpu_seq *> seqs;
    std::unordered_set<dnagpu_table *> tables;
    std::unordered_set<dnagpu_index *> indexes;
    char err[512] = {0};
};

struct dnagpu_seq {
    dnagpu_ctx *ctx = nullptr;
    int layout = kSingle;
    uint64_t *d_words = nullptr;
    bool own_words = true;
    uint64_t n_words_alloc = 0; /* incl. pad */
    uint64_t n_words = 0;       /* payload words (download) */
    uint64_t n_seqs = 1;
    uint64_t bases = 0;  /* per sequence (single / fixed) */
    uint64_t stride = 0; /* words per sequence (fixed) */
    uint64_t start_limit = 0;
    /* ragged */
    std::vector<uint64_t> h_n_bases;
    uint64_t *d_word_off = nullptr, *d_n_bases = nullptr;
    /* pieces (kPieces): base-range shards, possibly in peer memory */
    std::vector<const uint64_t *> piece_ptr;
    std::vector<uint64_t> piece_first, piece_starts;
    int cached_k = 0;
    uint64_t *d_row_off = nullptr, *d_item_off = nullptr;
    uint64_t cached_rows = 0, cached_items = 0;
};

struct dnagpu_table {
    dnagpu_ctx *ctx = nullptr;
    int k = 0;
    uint64_t rows = 0;
    uint64_t *d_kmers = nullptr, *d_counts = nullptr;
    std::vector<dnagpu_table *> parts; /* multi-GPU result: the per-GPU tables (disjoint key sets), in order */
};

struct dnagpu_index {
    dnagpu_ctx *ctx = nullptr;
    int k = 0;
    uint64_t rows = 0;
    uint64_t *d_skeys = nullptr, *d_rows = nullptr; /* sort keys ascending; the row each came from */
};

static thread_local char g_err[512] = "";

static int fail(dnagpu_ctx *ctx, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    snprintf(g_err, sizeof g_err, "%s", buf);
    if (ctx) snprintf(ctx->err, sizeof ctx->err, "%s", buf);
    return code;
}

#define CU(ctx, call)                                                                        \
    do {                                                                                     \
        cudaError_t e_ = (call);                                                             \
        if (e_ != cudaSuccess)                                                               \
            return fail(ctx, e_ == cudaErrorMemoryAllocation ? DNAGPU_ENOMEM : DNAGPU_ECUDA, \
                        "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

/* every launch goes through here so that profiling sees it */
template <class F>
static int launch(dnagpu_ctx *ctx, const char *name, F &&f)
{
    if (ctx->profiling) {
        ProfRec r;
        r.name = name;
        CU(ctx, cudaEventCreate(&r.e0));
        CU(ctx, cudaEventCreate(&r.e1));
        CU(ctx, cudaEventRecord(r.e0, ctx->stream));
        f();
        CU(ctx, cudaEventRecord(r.e1, ctx->stream));
        ctx->prof.push_back(r);
    } else {
        f();
    }
    CU(ctx, cudaGetLastError());
    return DNAGPU_OK;
}
#define TRY(x)                         \
    do {                               \
        int rc_ = (x);                 \
        if (rc_ != DNAGPU_OK) return rc_; \
    } while (0)

static int dalloc(dnagpu_ctx *ctx, void **p, uint64_t bytes)
{
    *p = nullptr;
    if (bytes == 0) bytes = 16;
    cudaError_t e = cudaMallocAsync(p, bytes, ctx->stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, DNAGPU_ENOMEM, "device allocation of %llu bytes failed: %s",
                    (unsigned long long)bytes, cudaGetErrorString(e));
    }
    return DNAGPU_OK;
}
static void dfree(dnagpu_ctx *ctx, void *p)
{
    if (p) cudaFreeAsync(p, ctx->stream);
}
/* scope guard for scratch buffers */
struct Scratch {
    dnagpu_ctx *ctx;
    std::vector<void *> ptrs;
    explicit Scratch(dnagpu_ctx *c) : ctx(c) {}
    ~Scratch()
    {
        for (void *p : ptrs) dfree(ctx, p);
    }
    int get(void **p, uint64_t bytes)
    {
        int rc = dalloc(ctx, p, bytes);
        if (rc == DNAGPU_OK) ptrs.push_back(*p);
        return rc;
    }
    void release(void *p) { ptrs.erase(std::remove(ptrs.begin(), ptrs.end(), p), ptrs.end()); }
};

static int scan_any(dnagpu_ctx *ctx, Scratch &sc, const uint64_t *in, uint64_t n, uint64_t *out);
static int read_u64(dnagpu_ctx *ctx, const uint64_t *d, uint64_t *h);

static inline uint64_t rows_of(uint64_t n_bases, int k)
{
    return n_bases >= (uint64_t)k ? n_bases - (uint64_t)k + 1 : 0; /* Q2 (dna.c:781) */
}
static inline uint64_t words_of(uint64_t n_bases) { return (n_bases + 31) / 32; }
static inline uint64_t kmer_mask(int k) { return k >= 32 ? ~0ull : ((1ull << (2 * k)) - 1); }
static inline unsigned grid_for(uint64_t n, uint64_t per_cta)
{
    uint64_t g = (n + per_cta - 1) / per_cta;
    return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(g, 0x7fffffffull));
}

/* ---- context ------------------------------------------------------------------ */
extern "C" int dnagpu_version(void) { return DNAGPU_VERSION; }

extern "C" const char *dnagpu_strerror(int code)
{
    switch (code) {
    case DNAGPU_OK: return "ok";
    case DNAGPU_EINVAL_K: return "Invalid k value: must be between 1 and 32";        /* dna.c:773 */
    case DNAGPU_EPREFIX_LEN: return "Prefix length cannot exceed kmer length";       /* dna.c:855 */
    case DNAGPU_EQKMER_LEN: return "Qkmer pattern and kmer lengths do not match";    /* dna.c:1107 */
    case DNAGPU_EQKMER_CHAR: return "Invalid character in qkmer pattern";            /* dna.c:894 */
    case DNAGPU_EQKMER_EMPTY: return "qkmer pattern cannot be empty";                /* dna.c:878 */
    case DNAGPU_EQKMER_TOOLONG: return "Qkmer pattern length cannot exceed 32 characters"; /* dna.c:884 */
    case DNAGPU_EPREFIX_BITS: return "prefix kmer has bits set beyond its length";
    case DNAGPU_EDNA_CHAR: return "Invalid character in DNA sequence";                /* dna.c:166 */
    case DNAGPU_EDNA_EMPTY: return "DNA sequence cannot be empty";                    /* dna.c:161 */
    case DNAGPU_EARG: return "invalid argument";
    case DNAGPU_ECAPACITY: return "output buffer too small";
    case DNAGPU_ENOMEM: return "out of device or pinned host memory";
    case DNAGPU_ECUDA: return "CUDA error";
    case DNAGPU_ENODEVICE: return "no usable sm_100 GPU";
    case DNAGPU_EINTERNAL: return "internal error";
    }
    return "unknown error";
}

extern "C" int dnagpu_create(dnagpu_ctx **out, int device)
{
    if (!out) return fail(nullptr, DNAGPU_EARG, "dnagpu_create: out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(nullptr, DNAGPU_ENODEVICE, "no CUDA device: %s (libdnagpu has no CPU path)",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= n)
        return fail(nullptr, DNAGPU_EARG, "device %d out of range (0..%d)", device, n - 1);
    cudaDeviceProp prop;
    CU(nullptr, cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(nullptr, DNAGPU_ENODEVICE,
                    "device %d (%s) is sm_%d%d; libdnagpu is built for sm_100a only", device,
                    prop.name, prop.major, prop.minor);
    dnagpu_ctx *ctx = new (std::nothrow) dnagpu_ctx();
    if (!ctx) return fail(nullptr, DNAGPU_ENOMEM, "out of host memory");
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    CU(nullptr, cudaSetDevice(device));
    CU(nullptr, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    /* keep freed scratch in the stream-ordered pool: repeated queries reuse it */
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    const size_t ctr_bytes = (C_COUNT + 2 * kMaxParts) * sizeof(unsigned long long);
    CU(nullptr, cudaMalloc((void **)&ctx->d_ctr, ctr_bytes));
    CU(nullptr, cudaMallocHost((void **)&ctx->h_ctr, ctr_bytes));
    /* opt in to the 64 KB staging tiles */
    const int smem = kThreads * 32 * (int)sizeof(uint64_t);
#define SMEM_ATTR(kern) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)
    SMEM_ATTR(k_filter_write<kSingle>);
    SMEM_ATTR(k_filter_write<kFixed>);
    SMEM_ATTR(k_filter_write<kRagged>);
    SMEM_ATTR(k_filter_collect<kSingle>);
    SMEM_ATTR(k_filter_collect<kFixed>);
    SMEM_ATTR(k_filter_collect<kRagged>);
    SMEM_ATTR((k_filter_sa<kSingle, kSaCollect>));
    SMEM_ATTR((k_filter_sa<kFixed, kSaCollect>));
    SMEM_ATTR((k_filter_sa<kSingle, kSaWrite>));
    SMEM_ATTR((k_filter_sa<kFixed, kSaWrite>));
    SMEM_ATTR((k_partition_write<kSingle, false>));
    SMEM_ATTR((k_partition_write<kSingle, true>));
    SMEM_ATTR((k_partition_write<kFixed, false>));
    SMEM_ATTR((k_partition_write<kFixed, true>));
    SMEM_ATTR((k_partition_write<kRagged, false>));
    SMEM_ATTR((k_partition_write<kRagged, true>));
    SMEM_ATTR((k_count_dense_smem<kSingle, false, uint32_t>));
    SMEM_ATTR((k_count_dense_smem<kSingle, true, uint32_t>));
    SMEM_ATTR((k_count_dense_smem<kFixed, false, uint32_t>));
    SMEM_ATTR((k_count_dense_smem<kFixed, true, uint32_t>));
    SMEM_ATTR((k_count_dense_smem<kRagged, false, uint32_t>));
    SMEM_ATTR((k_count_dense_smem<kRagged, true, uint32_t>));
    SMEM_ATTR((k_count_dense_smem<kSingle, false, unsigned long long>));
    SMEM_ATTR((k_count_dense_smem<kSingle, true, unsigned long long>));
    SMEM_ATTR((k_count_dense_smem<kFixed, false, unsigned long long>));
    SMEM_ATTR((k_count_dense_smem<kFixed, true, unsigned long long>));
    SMEM_ATTR((k_count_dense_smem<kRagged, false, unsigned long long>));
    SMEM_ATTR((k_count_dense_smem<kRagged, true, unsigned long long>));
#undef SMEM_ATTR
    {
        const int psmem = kTileKeys * (int)sizeof(uint64_t) + (int)sizeof(ScatterSmem);
#define PSMEM_ATTR(kern) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, psmem)
        PSMEM_ATTR(k_part_scatter_keys<false>);
        {
            const int psmem32 = 32 * kScatThreads * (int)sizeof(uint64_t) + (int)sizeof(ScatterSmem);
#define PSMEM32_ATTR(kern) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, psmem32)
            PSMEM32_ATTR((k_part_scatter_keys<false, kBigPerKeys, kBigThreadsKeys>));
            PSMEM32_ATTR((k_part_scatter_keys<true, kBigPerKeys, kBigThreadsKeys>));
            PSMEM32_ATTR((k_part_scatter_seq<kSingle, false>));
            PSMEM32_ATTR((k_part_scatter_seq<kSingle, true>));
            PSMEM32_ATTR((k_part_scatter_seq<kFixed, false>));
            PSMEM32_ATTR((k_part_scatter_seq<kFixed, true>));
            PSMEM32_ATTR((k_part_scatter_seq<kRagged, false>));
            PSMEM32_ATTR((k_part_scatter_seq<kRagged, true>));
#undef PSMEM32_ATTR
        }
        PSMEM_ATTR(k_part_scatter_keys<true>);
#undef PSMEM_ATTR
        {
            int per_sm = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_count_buckets_bins<false>, kThreads, 0) == cudaSuccess &&
                per_sm > 0)
                ctx->bins_ctas_per_sm = per_sm;
        }
        cudaFuncSetAttribute(k_sort_scatter<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SortSmem));
        cudaFuncSetAttribute(k_sort_scatter<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SortSmem));
        const int bsmem = kBucketSlots * 12, bsmem64 = kBucketSlots * 16;
        cudaFuncSetAttribute(k_count_buckets<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bsmem);
        cudaFuncSetAttribute(k_count_buckets<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bsmem);
        cudaFuncSetAttribute(k_count_buckets<false, unsigned long long>, cudaFuncAttributeMaxDynamicSharedMemorySize, bsmem64);
        cudaFuncSetAttribute(k_count_buckets<true, unsigned long long>, cudaFuncAttributeMaxDynamicSharedMemorySize, bsmem64);
        cudaFuncSetAttribute(k_count_buckets<false, uint32_t, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             bsmem + kSpecSmem);
        cudaFuncSetAttribute(k_count_buckets<false, unsigned long long, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             bsmem64 + kSpecSmem);
    }
    CU(nullptr, cudaGetLastError());
    *out = ctx;
    return DNAGPU_OK;
}

extern "C" int dnagpu_create_multi(dnagpu_ctx **out, const int *devices, int n_devices)
{
    if (!out || !devices || n_devices < 1 || n_devices > kMaxPieces)
        return fail(nullptr, DNAGPU_EARG, "dnagpu_create_multi: need 1..%d devices", kMaxPieces);
    *out = nullptr;
    for (int a = 0; a < n_devices; ++a)
        for (int b = a + 1; b < n_devices; ++b)
            if (devices[a] == devices[b]) return fail(nullptr, DNAGPU_EARG, "device %d is listed twice", devices[a]);
    dnagpu_ctx *ctx = nullptr;
    TRY(dnagpu_create(&ctx, devices[0]));
    for (int d = 1; d < n_devices; ++d) {
        dnagpu_ctx *p = nullptr;
        int rc = dnagpu_create(&p, devices[d]);
        if (rc != DNAGPU_OK) {
            dnagpu_destroy(ctx);
            return rc;
        }
        ctx->peers.push_back(p);
    }
    /* every GPU reads every other GPU's shard: peer access for all ordered pairs */
    for (int a = 0; a < n_devices; ++a) {
        cudaSetDevice(devices[a]);
        for (int b = 0; b < n_devices; ++b) {
            if (a == b) continue;
            int can = 0;
            cudaDeviceCanAccessPeer(&can, devices[a], devices[b]);
            cudaError_t e = can ? cudaDeviceEnablePeerAccess(devices[b], 0) : cudaErrorPeerAccessUnsupported;
            if (e == cudaErrorPeerAccessAlreadyEnabled) {
                cudaGetLastError();
                e = cudaSuccess;
            }
            if (e != cudaSuccess) {
                cudaGetLastError();
                dnagpu_destroy(ctx);
                return fail(nullptr, DNAGPU_ENODEVICE, "GPU %d cannot map the memory of GPU %d (%s): no multi-GPU context",
                            devices[a], devices[b], cudaGetErrorString(e));
            }
        }
    }
    cudaSetDevice(devices[0]);
    ctx->shard_buf.assign((size_t)n_devices, nullptr);
    ctx->shard_cap.assign((size_t)n_devices, 0);
    *out = ctx;
    return DNAGPU_OK;
}

extern "C" int dnagpu_device_count(const dnagpu_ctx *ctx) { return ctx ? 1 + (int)ctx->peers.size() : 0; }

static void seq_release(dnagpu_seq *s);
static void table_release(dnagpu_table *t);
static void index_release(dnagpu_index *ix);

extern "C" void dnagpu_destroy(dnagpu_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    /* handles the caller still holds: their device memory goes now, the host structs stay valid (orphaned)
     * until the caller frees them -- dnagpu_*_free after dnagpu_destroy is legal and touches no CUDA state */
    for (dnagpu_seq *c : ctx->seqs) seq_release(c);
    for (dnagpu_table *c : ctx->tables) table_release(c);
    for (dnagpu_index *c : ctx->indexes) index_release(c);
    ctx->seqs.clear();
    ctx->tables.clear();
    ctx->indexes.clear();
    cudaStreamSynchronize(ctx->stream);
    for (size_t d = 0; d < ctx->shard_buf.size(); ++d)
        if (ctx->shard_buf[d]) {
            cudaSetDevice(d == 0 ? ctx->device : ctx->peers[d - 1]->device);
            cudaFree(ctx->shard_buf[d]);
        }
    for (dnagpu_ctx *p : ctx->peers) dnagpu_destroy(p);
    ctx->peers.clear();
    cudaSetDevice(ctx->device);
    for (auto &r : ctx->prof) {
        cudaEventDestroy(r.e0);
        cudaEventDestroy(r.e1);
    }
    if (ctx->d_ctr) cudaFree(ctx->d_ctr);
    if (ctx->d_spec) cudaFree(ctx->d_spec);
    if (ctx->h_ctr) cudaFreeHost(ctx->h_ctr);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" const char *dnagpu_last_error(const dnagpu_ctx *ctx) { return ctx ? ctx->err : g_err; }

extern "C" int dnagpu_set_stream(dnagpu_ctx *ctx, void *cuda_stream)
{
    if (!ctx) return fail(nullptr, DNAGPU_EARG, "ctx is NULL");
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    if (cuda_stream) {
        ctx->stream = (cudaStream_t)cuda_stream;
        ctx->own_stream = false;
    } else {
        CU(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        ctx->own_stream = true;
    }
    return DNAGPU_OK;
}

extern "C" int dnagpu_synchronize(dnagpu_ctx *ctx)
{
    if (!ctx) return fail(nullptr, DNAGPU_EARG, "ctx is NULL");
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return DNAGPU_OK;
}

extern "C" int dnagpu_device_info(dnagpu_ctx *ctx, char *name, size_t cap, int *sm_count,
                                  uint64_t *hbm_free, uint64_t *hbm_total)
{
    if (!ctx) return fail(nullptr, DNAGPU_EARG, "ctx is NULL");
    cudaDeviceProp prop;
    CU(ctx, cudaGetDeviceProperties(&prop, ctx->device));
    if (name && cap) snprintf(name, cap, "%s", prop.name);
    if (sm_count) *sm_count = prop.multiProcessorCount;
    size_t f = 0, t = 0;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemGetInfo(&f, &t));
    if (hbm_free) *hbm_free = f;
    if (hbm_total) *hbm_total = t;
    return DNAGPU_OK;
}

extern "C" int dnagpu_host_alloc(dnagpu_ctx *ctx, void **out, uint64_t bytes)
{
    if (!ctx || !out) return fail(ctx, DNAGPU_EARG, "dnagpu_host_alloc: NULL argument");
    *out = nullptr;
    cudaError_t e = cudaMallocHost(out, bytes ? bytes : 16);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, DNAGPU_ENOMEM, "pinned allocation of %llu bytes failed: %s",
                    (unsigned long long)bytes, cudaGetErrorString(e));
    }
    return DNAGPU_OK;
}
extern "C" void dnagpu_host_free(dnagpu_ctx *ctx, void *p)
{
    (void)ctx;
    if (p) cudaFreeHost(p);
}

/* ---- sequences ------------------------------------------------------------------ */
static int seq_new(dnagpu_ctx *ctx, dnagpu_seq **out, dnagpu_seq **s)
{
    if (!ctx || !out) return fail(ctx, DNAGPU_EARG, "NULL ctx or output pointer");
    *out = nullptr;
    *s = new (std::nothrow) dnagpu_seq();
    if (!*s) return fail(ctx, DNAGPU_ENOMEM, "out of host memory");
    (*s)->ctx = ctx;
    ctx->seqs.insert(*s);
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) {
        ctx->seqs.erase(*s);
        delete *s;
        *s = nullptr;
        return fail(ctx, DNAGPU_ECUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
    }
    return DNAGPU_OK;
}

/* allocate payload + zeroed pad (>= 1 word, total even => 16-byte granules) */
static int seq_alloc_words(dnagpu_seq *s, uint64_t payload_words)
{
    dnagpu_ctx *ctx = s->ctx;
    s->n_words = payload_words;
    s->n_words_alloc = (payload_words + 2 + 1) & ~1ull;
    TRY(dalloc(ctx, (void **)&s->d_words, s->n_words_alloc * 8));
    CU(ctx, cudaMemsetAsync(s->d_words + payload_words, 0, (s->n_words_alloc - payload_words) * 8,
                            ctx->stream));
    return DNAGPU_OK;
}

/* give the device memory of a handle back and cut it loose from its ctx (the host struct stays) */
static void seq_release(dnagpu_seq *s)
{
    dnagpu_ctx *ctx = s->ctx;
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (s->own_words) dfree(ctx, s->d_words);
    dfree(ctx, s->d_word_off);
    dfree(ctx, s->d_n_bases);
    dfree(ctx, s->d_row_off);
    dfree(ctx, s->d_item_off);
    s->d_words = s->d_word_off = s->d_n_bases = s->d_row_off = s->d_item_off = nullptr;
    s->ctx = nullptr;
}

extern "C" void dnagpu_seq_free(dnagpu_seq *s)
{
    if (!s) return;
    if (s->ctx) {
        s->ctx->seqs.erase(s);
        seq_release(s);
    }
    delete s;
}

/* a child handle must belong to the (live) ctx it is used with */
#define CHECK_OWNED(ctx, child, what)                                                              \
    do {                                                                                           \
        if ((child)->ctx != (ctx))                                                                 \
            return fail(ctx, DNAGPU_EARG, what " belongs to another context or its context was destroyed"); \
    } while (0)

extern "C" int dnagpu_seq_upload(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_bases,
                                 dnagpu_seq **out)
{
    dnagpu_seq *s;
    TRY(seq_new(ctx, out, &s));
    if (!words && n_bases) {
        dnagpu_seq_free(s);
        return fail(ctx, DNAGPU_EARG, "dnagpu_seq_upload: words is NULL");
    }
    s->layout = kSingle;
    s->bases = n_bases;
    int rc = seq_alloc_words(s, words_of(n_bases));
    if (rc == DNAGPU_OK && s->n_words) {
        cudaError_t e = cudaMemcpyAsync(s->d_words, words, s->n_words * 8, cudaMemcpyHostToDevice,
                                        ctx->stream);
        /* "Copies; the caller keeps ownership": from pinned memory the copy is truly asynchronous, so it
         * must have left the caller's buffer before the call returns */
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = fail(ctx, DNAGPU_ECUDA, "H2D copy: %s", cudaGetErrorString(e));
    }
    if (rc != DNAGPU_OK) {
        dnagpu_seq_free(s);
        return rc;
    }
    *out = s;
    return DNAGPU_OK;
}

extern "C" int dnagpu_seq_upload_reads(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_reads,
                                       uint32_t bases_per_read, uint32_t stride_words,
                                       dnagpu_seq **out)
{
    dnagpu_seq *s;
    TRY(seq_new(ctx, out, &s));
    if ((!words && n_reads) || stride_words < words_of(bases_per_read)) {
        dnagpu_seq_free(s);
        return fail(ctx, DNAGPU_EARG, "dnagpu_seq_upload_reads: NULL words or stride < words per read");
    }
    s->layout = kFixed;
    s->n_seqs = n_reads;
    s->bases = bases_per_read;
    s->stride = stride_words;
    int rc = seq_alloc_words(s, n_reads * stride_words);
    if (rc == DNAGPU_OK && s->n_words) {
        cudaError_t e = cudaMemcpyAsync(s->d_words, words, s->n_words * 8, cudaMemcpyHostToDevice,
                                        ctx->stream);
        /* "Copies; the caller keeps ownership": from pinned memory the copy is truly asynchronous, so it
         * must have left the caller's buffer before the call returns */
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = fail(ctx, DNAGPU_ECUDA, "H2D copy: %s", cudaGetErrorString(e));
    }
    if (rc != DNAGPU_OK) {
        dnagpu_seq_free(s);
        return rc;
    }
    *out = s;
    return DNAGPU_OK;
}

extern "C" int dnagpu_seq_upload_ragged(dnagpu_ctx *ctx, const uint64_t *words,
                                        const uint64_t *word_offsets, const uint64_t *n_bases,
                                        uint64_t n_seqs, dnagpu_seq **out)
{
    dnagpu_seq *s;
    TRY(seq_new(ctx, out, &s));
    if (n_seqs && (!words || !word_offsets || !n_bases)) {
        dnagpu_seq_free(s);
        return fail(ctx, DNAGPU_EARG, "dnagpu_seq_upload_ragged: NULL argument");
    }
    s->layout = kRagged;
    s->n_seqs = n_seqs;
    s->h_n_bases.assign(n_bases, n_bases + n_seqs);
    uint64_t total_words = 0;
    for (uint64_t i = 0; i < n_seqs; ++i)
        total_words = std::max(total_words, word_offsets[i] + words_of(n_bases[i]));
    int rc = seq_alloc_words(s, total_words);
    if (rc == DNAGPU_OK) rc = dalloc(ctx, (void **)&s->d_word_off, (n_seqs + 1) * 8);
    if (rc == DNAGPU_OK) rc = dalloc(ctx, (void **)&s->d_n_bases, (n_seqs + 1) * 8);
    if (rc == DNAGPU_OK && n_seqs) {
        cudaError_t e = cudaSuccess;
        if (total_words)
            e = cudaMemcpyAsync(s->d_words, words, total_words * 8, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(s->d_word_off, word_offsets, n_seqs * 8, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(s->d_n_bases, n_bases, n_seqs * 8, cudaMemcpyHostToDevice, ctx->stream);
        /* the offsets/lengths arrays are the caller's: finish before returning */
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = fail(ctx, DNAGPU_ECUDA, "H2D copy: %s", cudaGetErrorString(e));
    }
    if (rc != DNAGPU_OK) {
        dnagpu_seq_free(s);
        return rc;
    }
    *out = s;
    return DNAGPU_OK;
}

extern "C" int dnagpu_seq_synth_range(dnagpu_ctx *ctx, uint64_t n_bases_total, uint64_t seed,
                                      uint32_t repeat_every, uint64_t first_base,
                                      uint64_t n_starts, int overlap_k, dnagpu_seq **out)
{
    dnagpu_seq *s;
    if (overlap_k < 1 || overlap_k > DNAGPU_MAX_K)
        return fail(ctx, DNAGPU_EINVAL_K, "%s", dnagpu_strerror(DNAGPU_EINVAL_K));
    if ((first_base & 31) || first_base > n_bases_total)
        return fail(ctx, DNAGPU_EARG, "first_base must be a multiple of 32 inside the sequence");
    TRY(seq_new(ctx, out, &s));
    uint64_t local = std::min(n_bases_total - first_base, n_starts + (uint64_t)overlap_k - 1);
    s->layout = kSingle;
    s->bases = local;
    s->start_limit = n_starts;
    int rc = seq_alloc_words(s, words_of(local));
    if (rc == DNAGPU_OK && s->n_words)
        rc = launch(ctx, "synth_seq", [&] {
            k_synth_seq<<<grid_for(s->n_words, kThreads), kThreads, 0, ctx->stream>>>(
                seed, repeat_every, n_bases_total, first_base / 32, s->n_words, s->d_words);
        });
    if (rc != DNAGPU_OK) {
        dnagpu_seq_free(s);
        return rc;
    }
    *out = s;
    return DNAGPU_OK;
}

extern "C" int dnagpu_seq_synth(dnagpu_ctx *ctx, uint64_t n_bases, uint64_t seed,
                                uint32_t repeat_every, dnagpu_seq **out)
{
    int rc = dnagpu_seq_synth_range(ctx, n_bases, seed, repeat_every, 0, n_bases, 1, out);
    if (rc == DNAGPU_OK) (*out)->start_limit = 0;
    return rc;
}

extern "C" int dnagpu_seq_synth_reads(dnagpu_ctx *ctx, uint64_t first_read, uint64_t n_reads,
                                      uint32_t bases_per_read, uint32_t stride_words,
                                      uint64_t seed, uint32_t repeat_every, dnagpu_seq **out)
{
    dnagpu_seq *s;
    if (stride_words < words_of(bases_per_read))
        return fail(ctx, DNAGPU_EARG, "stride_words < words per read");
    TRY(seq_new(ctx, out, &s));
    s->layout = kFixed;
    s->n_seqs = n_reads;
    s->bases = bases_per_read;
    s->stride = stride_words;
    int rc = seq_alloc_words(s, n_reads * stride_words);
    if (rc == DNAGPU_OK && s->n_words)
        rc = launch(ctx, "synth_reads", [&] {
            k_synth_reads<<<grid_for(s->n_words, kThreads), kThreads, 0, ctx->stream>>>(
                seed, repeat_every, first_read, n_reads, bases_per_read, stride_words, s->d_words);
        });
    if (rc != DNAGPU_OK) {
        dnagpu_seq_free(s);
        return rc;
    }
    *out = s;
    return DNAGPU_OK;
}

extern "C" int dnagpu_seq_wrap(dnagpu_ctx *ctx, const void *d_words, uint64_t n_bases,
                               uint64_t n_words_alloc, dnagpu_seq **out)
{
    dnagpu_seq *s;
    if (!d_words || ((uintptr_t)d_words & 15) || n_words_alloc < words_of(n_bases) + 1)
        return fail(ctx, DNAGPU_EARG,
                    "dnagpu_seq_wrap: need a 16-byte aligned device pointer with >= 1 pad word");
    TRY(seq_new(ctx, out, &s));
    s->layout = kSingle;
    s->bases = n_bases;
    s->d_words = (uint64_t *)d_words;
    s->own_words = false;
    s->n_words = words_of(n_bases);
    s->n_words_alloc = n_words_alloc;
    *out = s;
    return DNAGPU_OK;
}

extern "C" int dnagpu_seq_wrap_reads(dnagpu_ctx *ctx, const void *d_words, uint64_t n_reads,
                                     uint32_t bases_per_read, uint32_t stride_words,
                                     uint64_t n_words_alloc, dnagpu_seq **out)
{
    dnagpu_seq *s;
    if (!d_words || ((uintptr_t)d_words & 15) || stride_words < words_of(bases_per_read) ||
        n_words_alloc < n_reads * stride_words + 1)
        return fail(ctx, DNAGPU_EARG,
                    "dnagpu_seq_wrap_reads: need a 16-byte aligned device pointer with >= 1 pad word");
    TRY(seq_new(ctx, out, &s));
    s->layout = kFixed;
    s->n_seqs = n_reads;
    s->bases = bases_per_read;
    s->stride = stride_words;
    s->d_words = (uint64_t *)d_words;
    s->own_words = false;
    s->n_words = n_reads * stride_words;
    s->n_words_alloc = n_words_alloc;
    *out = s;
    return DNAGPU_OK;
}

extern "C" int dnagpu_seq_wrap_pieces(dnagpu_ctx *ctx, const void *const *d_words, const uint64_t *first_base,
                                      const uint64_t *n_starts, uint32_t n_pieces, uint64_t n_bases_total,
                                      dnagpu_seq **out)
{
    if (!ctx || !out || !d_words || !first_base || !n_starts || n_pieces < 1 || n_pieces > (uint32_t)kMaxPieces)
        return fail(ctx, DNAGPU_EARG, "dnagpu_seq_wrap_pieces: NULL argument or more than %d pieces", kMaxPieces);
    /* the ranges must tile the sequence: walk them in base order */
    std::vector<uint32_t> order(n_pieces);
    for (uint32_t i = 0; i < n_pieces; ++i) order[i] = i;
    std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return first_base[a] < first_base[b]; });
    uint64_t next = 0;
    for (uint32_t q = 0; q < n_pieces; ++q) {
        const uint32_t i = order[q];
        if (!d_words[i] || ((uintptr_t)d_words[i] & 15) || (first_base[i] & 31))
            return fail(ctx, DNAGPU_EARG, "piece %u: need a 16-byte aligned device pointer and a first base that is a multiple of 32", i);
        if (n_starts[i] == 0) continue; /* a GPU past the end of a short sequence */
        if (first_base[i] != next || ((n_starts[i] & 31) && next + n_starts[i] < n_bases_total))
            return fail(ctx, DNAGPU_EARG, "piece %u: the base ranges (multiples of 32) must tile the sequence", i);
        next += n_starts[i];
    }
    if (next < n_bases_total) return fail(ctx, DNAGPU_EARG, "the pieces cover %llu of %llu bases", (unsigned long long)next,
                                         (unsigned long long)n_bases_total);
    dnagpu_seq *s;
    TRY(seq_new(ctx, out, &s));
    s->layout = kPieces;
    s->bases = n_bases_total;
    s->own_words = false;
    s->n_words = 0;
    for (uint32_t i = 0; i < n_pieces; ++i) {
        s->piece_ptr.push_back((const uint64_t *)d_words[i]);
        s->piece_first.push_back(first_base[i]);
        s->piece_starts.push_back(n_starts[i]);
    }
    *out = s;
    return DNAGPU_OK;
}

extern "C" int dnagpu_seq_set_start_limit(dnagpu_seq *seq, uint64_t n_starts)
{
    if (!seq || seq->layout != kSingle)
        return fail(seq ? seq->ctx : nullptr, DNAGPU_EARG, "start limit applies to a single sequence");
    seq->start_limit = n_starts;
    return DNAGPU_OK;
}

extern "C" int dnagpu_seq_download(dnagpu_ctx *ctx, const dnagpu_seq *seq, uint64_t *words,
                                   uint64_t n_words)
{
    if (!ctx || !seq || (!words && n_words)) return fail(ctx, DNAGPU_EARG, "NULL argument");
    CHECK_OWNED(ctx, seq, "the sequence");
    if (n_words > seq->n_words) return fail(ctx, DNAGPU_EARG, "n_words exceeds the batch");
    CU(ctx, cudaSetDevice(ctx->device));
    if (n_words) CU(ctx, cudaMemcpyAsync(words, seq->d_words, n_words * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return DNAGPU_OK;
}

extern "C" uint64_t dnagpu_seq_words(const dnagpu_seq *seq) { return seq ? seq->n_words : 0; }

extern "C" const void *dnagpu_seq_device_words(const dnagpu_seq *seq)
{
    return seq ? seq->d_words : nullptr;
}

extern "C" uint64_t dnagpu_seq_kmer_count(const dnagpu_seq *seq, int k)
{
    if (!seq || k < 1 || k > DNAGPU_MAX_K) return 0;
    if (seq->layout == kSingle) {
        uint64_t r = rows_of(seq->bases, k);
        return seq->start_limit ? std::min(r, seq->start_limit) : r;
    }
    if (seq->layout == kFixed) return seq->n_seqs * rows_of(seq->bases, k);
    if (seq->layout == kPieces) return rows_of(seq->bases, k);
    uint64_t t = 0;
    for (uint64_t n : seq->h_n_bases) t += rows_of(n, k);
    return t;
}

/* the device view of a sequence for one k (ragged: builds and caches the prefix sums) */
static int make_view(dnagpu_ctx *ctx, const dnagpu_seq *cseq, int k, SeqView *v)
{
    dnagpu_seq *seq = const_cast<dnagpu_seq *>(cseq);
    CHECK_OWNED(ctx, seq, "the sequence");
    if (seq->layout == kPieces)
        return fail(ctx, DNAGPU_EARG, "a sequence in pieces is only accepted by dnagpu_count with an owner restriction");
    memset(v, 0, sizeof *v);
    v->words = seq->d_words;
    v->n_seqs = seq->n_seqs;
    v->stride = seq->stride;
    if (seq->layout != kRagged) {
        uint64_t r = rows_of(seq->bases, k);
        if (seq->layout == kSingle && seq->start_limit) r = std::min(r, seq->start_limit);
        v->rows_per_seq = r;
        v->items_per_seq = (r + 31) / 32;
        v->n_rows = r * seq->n_seqs;
        v->n_items = v->items_per_seq * seq->n_seqs;
        return DNAGPU_OK;
    }
    if (seq->cached_k != k) {
        const uint64_t n = seq->n_seqs;
        if (!seq->d_row_off) TRY(dalloc(ctx, (void **)&seq->d_row_off, (n + 1) * 8));
        if (!seq->d_item_off) TRY(dalloc(ctx, (void **)&seq->d_item_off, (n + 1) * 8));
        Scratch sc(ctx);
        uint64_t *rows, *items;
        TRY(sc.get((void **)&rows, (n + 1) * 8));
        TRY(sc.get((void **)&items, (n + 1) * 8));
        if (n)
            TRY(launch(ctx, "ragged_rows", [&] {
                k_ragged_rows<<<grid_for(n, kThreads), kThreads, 0, ctx->stream>>>(seq->d_n_bases, n, k,
                                                                                  rows, items);
            }));
        TRY(scan_any(ctx, sc, rows, n, seq->d_row_off));
        TRY(scan_any(ctx, sc, items, n, seq->d_item_off));
        CU(ctx, cudaMemcpyAsync(&ctx->h_ctr[0], seq->d_row_off + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(ctx, cudaMemcpyAsync(&ctx->h_ctr[1], seq->d_item_off + n, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        seq->cached_rows = ctx->h_ctr[0];
        seq->cached_items = ctx->h_ctr[1];
        seq->cached_k = k;
    }
    v->word_off = seq->d_word_off;
    v->row_off = seq->d_row_off;
    v->item_off = seq->d_item_off;
    v->n_rows = seq->cached_rows;
    v->n_items = seq->cached_items;
    return DNAGPU_OK;
}

/* ---- predicates ------------------------------------------------------------------- */
static int iupac_set(char c)
{ /* A=1 T=2 C=4 G=8, the sets of nucleotide_matches (dna.c:1064-1086); 'U' matches
     nothing because a kmer never decodes to 'U' (dna.c:1070, Q4) */
    switch (c) {
    case 'A': return 1;
    case 'T': return 2;
    case 'C': return 4;
    case 'G': return 8;
    case 'U': return 0;
    case 'W': return 1 | 2;
    case 'S': return 4 | 8;
    case 'M': return 1 | 4;
    case 'K': return 8 | 2;
    case 'R': return 1 | 8;
    case 'Y': return 4 | 2;
    case 'B': return 4 | 8 | 2;
    case 'D': return 1 | 8 | 2;
    case 'H': return 1 | 4 | 2;
    case 'V': return 1 | 4 | 8;
    case 'N': return 15;
    }
    return -1;
}

/* validate the literals (the reference does this when it coerces them:
 * qkmer_in -> validate_qkmer_pattern, dna.c:876-900) */
static int check_filter_literals(dnagpu_ctx *ctx, const dnagpu_where *f)
{
    if (!f) return DNAGPU_OK;
    if (f->flags & ~DNAGPU_WHERE_FLAG_PLANES) return fail(ctx, DNAGPU_EARG, "unknown bit in dnagpu_where.flags");
    if (f->prefix_len < 0 || f->prefix_len > DNAGPU_MAX_K)
        return fail(ctx, DNAGPU_EARG, "prefix_len out of range");
    if (f->prefix_len > 0 && f->prefix_len < 32 && (f->prefix_bits >> (2 * f->prefix_len)))
        return fail(ctx, DNAGPU_EPREFIX_BITS, "%s", dnagpu_strerror(DNAGPU_EPREFIX_BITS));
    if (f->qkmer) {
        size_t len = strlen(f->qkmer);
        if (len == 0) return fail(ctx, DNAGPU_EQKMER_EMPTY, "%s", dnagpu_strerror(DNAGPU_EQKMER_EMPTY));
        if (len > 32) return fail(ctx, DNAGPU_EQKMER_TOOLONG, "%s", dnagpu_strerror(DNAGPU_EQKMER_TOOLONG));
        for (size_t i = 0; i < len; ++i)
            if (iupac_set(f->qkmer[i]) < 0)
                return fail(ctx, DNAGPU_EQKMER_CHAR, "Invalid character in qkmer pattern: %c", f->qkmer[i]);
    }
    return DNAGPU_OK;
}

/* the per-row ERRORs (dna.c:854-856, 1106-1108) fire only when a row is evaluated */
static int build_pred(dnagpu_ctx *ctx, const dnagpu_where *f, int k, uint64_t n_rows, Pred *p,
                      bool *active)
{
    *active = false;
    p->ma = p->mt = p->mc = p->mg = ~0ull;
    if (ctx) ctx->plane_filter = f && (f->flags & DNAGPU_WHERE_FLAG_PLANES);
    if (!f || (f->prefix_len == 0 && !f->qkmer)) return DNAGPU_OK;
    if (n_rows == 0) return DNAGPU_OK;
    if (f->prefix_len > k) return fail(ctx, DNAGPU_EPREFIX_LEN, "%s", dnagpu_strerror(DNAGPU_EPREFIX_LEN));
    if (f->qkmer && (int)strlen(f->qkmer) != k)
        return fail(ctx, DNAGPU_EQKMER_LEN, "%s", dnagpu_strerror(DNAGPU_EQKMER_LEN));
    uint64_t plane[4] = {~0ull, ~0ull, ~0ull, ~0ull};
    for (int j = 0; j < k; ++j) {
        int set = f->qkmer ? iupac_set(f->qkmer[j]) : 15;
        if (j < f->prefix_len) set &= 1 << ((f->prefix_bits >> (2 * j)) & 3); /* Q1: len 32 = all 64 bits */
        for (int b = 0; b < 4; ++b)
            if (!(set & (1 << b))) plane[b] &= ~(1ull << (2 * j));
    }
    p->ma = plane[0];
    p->mt = plane[1];
    p->mc = plane[2];
    p->mg = plane[3];
    *active = true;
    return DNAGPU_OK;
}

static int check_k(dnagpu_ctx *ctx, int k)
{
    if (k <= 0 || k > DNAGPU_MAX_K) /* dna.c:772-773 */
        return fail(ctx, DNAGPU_EINVAL_K, "%s", dnagpu_strerror(DNAGPU_EINVAL_K));
    return DNAGPU_OK;
}

#define DISPATCH_LAYOUT(layout, CALL) \
    switch (layout) {                 \
    case kSingle: { constexpr int LY = kSingle; CALL; } break; \
    case kFixed: { constexpr int LY = kFixed; CALL; } break;   \
    default: { constexpr int LY = kRagged; CALL; } break;      \
    }

/* ---- ingest codec: dna_in / dna_out -------------------------------------------------------------- */
/* text (host) -> packed words resident on the device; the reference's checks and messages */
static int encode_to_device(dnagpu_ctx *ctx, const char *text, uint64_t n_bases, uint64_t *d_words /* n_words */)
{
    if (!text || n_bases == 0) /* dna.c:160-161 */
        return fail(ctx, DNAGPU_EDNA_EMPTY, "%s", dnagpu_strerror(DNAGPU_EDNA_EMPTY));
    Scratch sc(ctx);
    unsigned char *d_text;
    TRY(sc.get((void **)&d_text, n_bases + 32));
    CU(ctx, cudaMemcpyAsync(d_text, text, n_bases, cudaMemcpyHostToDevice, ctx->stream));
    unsigned long long *d_bad = ctx->d_ctr;
    CU(ctx, cudaMemsetAsync(d_bad, 0xff, 8, ctx->stream));
    TRY(launch(ctx, "encode_dna", [&] {
        k_encode_dna<<<grid_for(words_of(n_bases), kThreads), kThreads, 0, ctx->stream>>>(d_text, n_bases, d_words, d_bad);
    }));
    uint64_t bad;
    TRY(read_u64(ctx, (const uint64_t *)d_bad, &bad));
    if (bad != ~0ull) /* dna.c:165-166: the first offender, scanning left to right */
        return fail(ctx, DNAGPU_EDNA_CHAR, "Invalid character in DNA sequence: %c", text[bad]);
    return DNAGPU_OK;
}

extern "C" int dnagpu_encode_dna(dnagpu_ctx *ctx, const char *text, uint64_t n_bases, uint64_t *words)
{
    if (!ctx || !words) return fail(ctx, DNAGPU_EARG, "dnagpu_encode_dna: NULL argument");
    CU(ctx, cudaSetDevice(ctx->device));
    Scratch sc(ctx);
    uint64_t *d_words;
    TRY(sc.get((void **)&d_words, (words_of(n_bases) + 1) * 8));
    TRY(encode_to_device(ctx, text, n_bases, d_words));
    CU(ctx, cudaMemcpyAsync(words, d_words, words_of(n_bases) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return DNAGPU_OK;
}

extern "C" int dnagpu_seq_from_text(dnagpu_ctx *ctx, const char *text, uint64_t n_bases, dnagpu_seq **out)
{
    dnagpu_seq *s;
    TRY(seq_new(ctx, out, &s));
    s->layout = kSingle;
    s->bases = n_bases;
    int rc = seq_alloc_words(s, words_of(n_bases));
    if (rc == DNAGPU_OK) rc = encode_to_device(ctx, text, n_bases, s->d_words);
    if (rc != DNAGPU_OK) {
        dnagpu_seq_free(s);
        return rc;
    }
    *out = s;
    return DNAGPU_OK;
}

extern "C" int dnagpu_decode_dna(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_bases, char *text)
{
    if (!ctx || !text || (!words && n_bases)) return fail(ctx, DNAGPU_EARG, "dnagpu_decode_dna: NULL argument");
    CU(ctx, cudaSetDevice(ctx->device));
    text[n_bases] = '\0';
    if (n_bases == 0) return DNAGPU_OK;
    Scratch sc(ctx);
    uint64_t *d_words;
    unsigned char *d_text;
    TRY(sc.get((void **)&d_words, words_of(n_bases) * 8));
    TRY(sc.get((void **)&d_text, n_bases + 32));
    CU(ctx, cudaMemcpyAsync(d_words, words, words_of(n_bases) * 8, cudaMemcpyHostToDevice, ctx->stream));
    TRY(launch(ctx, "decode_dna", [&] {
        k_decode_dna<<<grid_for(words_of(n_bases), kThreads), kThreads, 0, ctx->stream>>>(d_words, n_bases, d_text);
    }));
    CU(ctx, cudaMemcpyAsync(text, d_text, n_bases, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return DNAGPU_OK;
}

/* ---- generate_kmers ----------------------------------------------------------------- */
extern "C" int dnagpu_extract(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k, uint64_t *d_out,
                              uint64_t cap, uint64_t *n_out)
{
    if (!ctx || !seq || !n_out) return fail(ctx, DNAGPU_EARG, "dnagpu_extract: NULL argument");
    TRY(check_k(ctx, k));
    CU(ctx, cudaSetDevice(ctx->device));
    SeqView v;
    TRY(make_view(ctx, seq, k, &v));
    *n_out = v.n_rows;
    if (v.n_rows == 0) return DNAGPU_OK;
    if (!d_out || cap < v.n_rows)
        return fail(ctx, DNAGPU_ECAPACITY, "generate_kmers needs room for %llu rows",
                    (unsigned long long)v.n_rows);
    if ((uintptr_t)d_out & 15) return fail(ctx, DNAGPU_EARG, "d_out must be 16-byte aligned");
    if (((uintptr_t)d_out & 31) == 0) { /* 256-bit stores */
        const unsigned grid = grid_for((v.n_rows + 3) / 4, (uint64_t)kThreads * kQuadsPerThread);
        DISPATCH_LAYOUT(seq->layout, TRY(launch(ctx, "extract", [&] {
            k_extract4<LY><<<grid, kThreads, 0, ctx->stream>>>(v, kmer_mask(k), d_out);
        })));
        return DNAGPU_OK;
    }
    const unsigned grid = grid_for((v.n_rows + 1) / 2, (uint64_t)kThreads * kPairsPerThread);
    DISPATCH_LAYOUT(seq->layout, TRY(launch(ctx, "extract", [&] {
        k_extract<LY><<<grid, kThreads, 0, ctx->stream>>>(v, kmer_mask(k), d_out);
    })));
    return DNAGPU_OK;
}

extern "C" int dnagpu_generate_kmers(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_bases,
                                     int k, uint64_t *out, uint64_t cap, uint64_t *n_out)
{
    if (!ctx || !n_out) return fail(ctx, DNAGPU_EARG, "dnagpu_generate_kmers: NULL argument");
    TRY(check_k(ctx, k));
    const uint64_t rows = rows_of(n_bases, k);
    *n_out = rows;
    if (rows == 0) return DNAGPU_OK;
    if (!out || cap < rows)
        return fail(ctx, DNAGPU_ECAPACITY, "generate_kmers needs room for %llu rows",
                    (unsigned long long)rows);
    dnagpu_seq *seq = nullptr;
    TRY(dnagpu_seq_upload(ctx, words, n_bases, &seq));
    uint64_t *d_out = nullptr;
    int rc = dalloc(ctx, (void **)&d_out, rows * 8);
    if (rc == DNAGPU_OK) rc = dnagpu_extract(ctx, seq, k, d_out, rows, n_out);
    if (rc == DNAGPU_OK) {
        cudaError_t e = cudaMemcpyAsync(out, d_out, rows * 8, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = fail(ctx, DNAGPU_ECUDA, "D2H copy: %s", cudaGetErrorString(e));
    }
    dfree(ctx, d_out);
    dnagpu_seq_free(seq);
    return rc;
}

/* ---- WHERE ^@ / @> -------------------------------------------------------------------- */
static int read_u64(dnagpu_ctx *ctx, const uint64_t *d, uint64_t *h)
{
    CU(ctx, cudaMemcpyAsync(&ctx->h_ctr[0], d, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    *h = ctx->h_ctr[0];
    return DNAGPU_OK;
}

/* matches per CTA tile + their exclusive scan; *n_match = total */
/* the Shift-And tables of a predicate: M[b] bit (i + 32 - k) = base b is allowed at pattern position i */
static SaPred sa_pred_of(const Pred &p, int k)
{
    const uint64_t plane[4] = {p.ma, p.mt, p.mc, p.mg};
    SaPred sp;
    for (int b = 0; b < 4; ++b) {
        uint32_t m = 0;
        for (int i = 0; i < k; ++i)
            if ((plane[b] >> (2 * i)) & 1) m |= 1u << (i + 32 - k);
        sp.m[b] = m;
    }
    sp.inj = 1u << (32 - k);
    sp.two = 2;
    return sp;
}

/* the ordered scan as a Shift-And automaton (single sequences and fixed-stride reads): count per tile, scan, write */
static bool sa_applies(const dnagpu_ctx *ctx, const dnagpu_seq *seq) { return seq->layout != kRagged && !ctx->plane_filter; }
static uint64_t sa_runs(const dnagpu_seq *seq, const SeqView &v)
{
    return seq->layout == kSingle ? (v.n_items + kSaItems - 1) / kSaItems
                                  : v.n_seqs * ((v.items_per_seq + kSaItems - 1) / kSaItems);
}
template <int MODE>
static int sa_launch(dnagpu_ctx *ctx, const char *name, const dnagpu_seq *seq, const SeqView &v, const Pred &p, int k,
                     uint64_t *tile_io, uint64_t *d_out)
{
    const SaPred sp = sa_pred_of(p, k);
    const unsigned tiles = grid_for(sa_runs(seq, v), kThreads);
    const int smem = MODE == kSaCount ? 0 : kSaStage * (int)sizeof(uint64_t);
    return launch(ctx, name, [&] {
        if (seq->layout == kSingle)
            k_filter_sa<kSingle, MODE><<<tiles, kThreads, smem, ctx->stream>>>(v, sp, kmer_mask(k), k, 0, nullptr, tile_io, d_out);
        else
            k_filter_sa<kFixed, MODE><<<tiles, kThreads, smem, ctx->stream>>>(v, sp, kmer_mask(k), k, 0, nullptr, tile_io, d_out);
    });
}

static int filter_scan(dnagpu_ctx *ctx, const dnagpu_seq *seq, const SeqView &v, const Pred &p, int k,
                       Scratch &sc, uint64_t **tile_off, uint64_t *n_match)
{
    if (sa_applies(ctx, seq)) {
        const unsigned tiles = grid_for(sa_runs(seq, v), kThreads);
        uint64_t *tile_cnt;
        TRY(sc.get((void **)&tile_cnt, ((uint64_t)tiles + 1) * 8));
        TRY(sc.get((void **)tile_off, ((uint64_t)tiles + 1) * 8));
        TRY(sa_launch<kSaCount>(ctx, "filter_count", seq, v, p, k, tile_cnt, nullptr));
        TRY(scan_any(ctx, sc, tile_cnt, tiles, *tile_off));
        return read_u64(ctx, *tile_off + tiles, n_match);
    }
    const unsigned tiles = grid_for(v.n_items, kThreads);
    uint64_t *tile_cnt;
    TRY(sc.get((void **)&tile_cnt, ((uint64_t)tiles + 1) * 8));
    TRY(sc.get((void **)tile_off, ((uint64_t)tiles + 1) * 8));
    DISPATCH_LAYOUT(seq->layout, TRY(launch(ctx, "filter_count", [&] {
        k_filter_count<LY><<<(tiles + kFilterTiles - 1) / kFilterTiles, kThreads, 0, ctx->stream>>>(v, p, tile_cnt);
    })));
    TRY(scan_any(ctx, sc, tile_cnt, tiles, *tile_off));
    return read_u64(ctx, *tile_off + tiles, n_match);
}

extern "C" int dnagpu_filter(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k,
                             const dnagpu_where *filter, uint64_t *d_out, uint64_t cap,
                             uint64_t *n_out)
{
    if (!ctx || !seq || !n_out) return fail(ctx, DNAGPU_EARG, "dnagpu_filter: NULL argument");
    TRY(check_k(ctx, k));
    TRY(check_filter_literals(ctx, filter));
    CU(ctx, cudaSetDevice(ctx->device));
    SeqView v;
    TRY(make_view(ctx, seq, k, &v));
    Pred p;
    bool active;
    TRY(build_pred(ctx, filter, k, v.n_rows, &p, &active));
    if (!active) {
        if (!d_out) {
            *n_out = v.n_rows;
            return DNAGPU_OK;
        }
        return dnagpu_extract(ctx, seq, k, d_out, cap, n_out);
    }
    *n_out = 0;
    if (v.n_rows == 0) return DNAGPU_OK;
    Scratch sc(ctx);
    uint64_t *tile_off, n_match;
    TRY(filter_scan(ctx, seq, v, p, k, sc, &tile_off, &n_match));
    *n_out = n_match;
    if (!d_out || n_match == 0) return DNAGPU_OK;
    if (cap < n_match)
        return fail(ctx, DNAGPU_ECAPACITY, "filter needs room for %llu rows", (unsigned long long)n_match);
    if (sa_applies(ctx, seq)) return sa_launch<kSaWrite>(ctx, "filter_write", seq, v, p, k, tile_off, d_out);
    const unsigned tiles = grid_for(v.n_items, kThreads);
    const int smem = kThreads * 32 * (int)sizeof(uint64_t);
    DISPATCH_LAYOUT(seq->layout, TRY(launch(ctx, "filter_write", [&] {
        k_filter_write<LY><<<(tiles + kFilterTiles - 1) / kFilterTiles, kThreads, smem, ctx->stream>>>(
            v, p, kmer_mask(k), tile_off, d_out);
    })));
    return DNAGPU_OK;
}

extern "C" int dnagpu_filter_kmers(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_bases,
                                   int k, const dnagpu_where *filter, uint64_t *out,
                                   uint64_t cap, uint64_t *n_out)
{
    if (!ctx || !n_out) return fail(ctx, DNAGPU_EARG, "dnagpu_filter_kmers: NULL argument");
    TRY(check_k(ctx, k));
    TRY(check_filter_literals(ctx, filter));
    dnagpu_seq *seq = nullptr;
    TRY(dnagpu_seq_upload(ctx, words, n_bases, &seq));
    uint64_t need = 0, *d_out = nullptr;
    int rc = dnagpu_filter(ctx, seq, k, filter, nullptr, 0, &need);
    *n_out = need;
    if (rc == DNAGPU_OK && need > 0) {
        if (!out || cap < need)
            rc = fail(ctx, DNAGPU_ECAPACITY, "filter needs room for %llu rows", (unsigned long long)need);
        if (rc == DNAGPU_OK) rc = dalloc(ctx, (void **)&d_out, need * 8);
        if (rc == DNAGPU_OK) rc = dnagpu_filter(ctx, seq, k, filter, d_out, need, n_out);
        if (rc == DNAGPU_OK) {
            cudaError_t e = cudaMemcpyAsync(out, d_out, need * 8, cudaMemcpyDeviceToHost, ctx->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
            if (e != cudaSuccess) rc = fail(ctx, DNAGPU_ECUDA, "D2H copy: %s", cudaGetErrorString(e));
        }
    }
    dfree(ctx, d_out);
    dnagpu_seq_free(seq);
    return rc;
}

extern "C" int dnagpu_filter_keys(dnagpu_ctx *ctx, const uint64_t *d_keys, uint64_t n, int k,
                                  const dnagpu_where *filter, uint64_t *d_out, uint64_t cap,
                                  uint64_t *n_out)
{
    if (!ctx || !n_out || (!d_keys && n)) return fail(ctx, DNAGPU_EARG, "dnagpu_filter_keys: NULL argument");
    TRY(check_k(ctx, k));
    TRY(check_filter_literals(ctx, filter));
    CU(ctx, cudaSetDevice(ctx->device));
    Pred p;
    bool active;
    TRY(build_pred(ctx, filter, k, n, &p, &active));
    *n_out = 0;
    if (n == 0) return DNAGPU_OK;
    if (!active) {
        *n_out = n;
        if (!d_out) return DNAGPU_OK;
        if (cap < n) return fail(ctx, DNAGPU_ECAPACITY, "filter needs room for %llu rows", (unsigned long long)n);
        CU(ctx, cudaMemcpyAsync(d_out, d_keys, n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
        return DNAGPU_OK;
    }
    Scratch sc(ctx);
    const unsigned tiles = grid_for(n, (uint64_t)kThreads * kKeysPerThread);
    uint64_t *tile_cnt, *tile_off, n_match;
    TRY(sc.get((void **)&tile_cnt, ((uint64_t)tiles + 1) * 8));
    TRY(sc.get((void **)&tile_off, ((uint64_t)tiles + 1) * 8));
    TRY(launch(ctx, "filter_keys_count", [&] {
        k_filter_keys_count<<<tiles, kThreads, 0, ctx->stream>>>(d_keys, n, p, tile_cnt);
    }));
    TRY(scan_any(ctx, sc, tile_cnt, tiles, tile_off));
    TRY(read_u64(ctx, tile_off + tiles, &n_match));
    *n_out = n_match;
    if (!d_out || n_match == 0) return DNAGPU_OK;
    if (cap < n_match)
        return fail(ctx, DNAGPU_ECAPACITY, "filter needs room for %llu rows", (unsigned long long)n_match);
    TRY(launch(ctx, "filter_keys_write", [&] {
        k_filter_keys_write<<<tiles, kThreads, 0, ctx->stream>>>(d_keys, n, p, tile_off, d_out);
    }));
    return DNAGPU_OK;
}

/* ---- GROUP BY kmer ---------------------------------------------------------------------- */
/* the spectrum starts over with the counters: every count, and every redo of one, begins here */
static int zero_spectrum(dnagpu_ctx *ctx)
{
    if (ctx->spec_h) CU(ctx, cudaMemsetAsync(ctx->d_spec, 0, (kSpecCum + (uint64_t)ctx->spec_h) * 8, ctx->stream));
    return DNAGPU_OK;
}
static int zero_counters(dnagpu_ctx *ctx)
{
    CU(ctx, cudaMemsetAsync(ctx->d_ctr, 0, (C_COUNT + 2 * kMaxParts) * 8, ctx->stream));
    return zero_spectrum(ctx);
}
static int fetch_counters(dnagpu_ctx *ctx)
{
    CU(ctx, cudaMemcpyAsync(ctx->h_ctr, ctx->d_ctr, (C_COUNT + 2 * kMaxParts) * 8,
                            cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return DNAGPU_OK;
}

static int table_new(dnagpu_ctx *ctx, int k, uint64_t rows, dnagpu_table **out)
{
    dnagpu_table *t = new (std::nothrow) dnagpu_table();
    if (!t) return fail(ctx, DNAGPU_ENOMEM, "out of host memory");
    t->ctx = ctx;
    ctx->tables.insert(t);
    t->k = k;
    t->rows = rows;
    int rc = dalloc(ctx, (void **)&t->d_kmers, rows * 8);
    if (rc == DNAGPU_OK) rc = dalloc(ctx, (void **)&t->d_counts, rows * 8);
    if (rc != DNAGPU_OK) {
        dnagpu_table_free(t);
        return rc;
    }
    *out = t;
    return DNAGPU_OK;
}

/* What the counting kernels consume: packed sequences or a materialised key list. */
struct CountInput {
    const dnagpu_seq *seq = nullptr;
    SeqView v;
    const uint64_t *d_keys = nullptr;
    uint64_t n = 0; /* rows (before WHERE) */
    bool filtered = false;
    Pred p;
};

static uint64_t pow4_capped(int k) { return k >= 32 ? UINT64_MAX : (1ull << (2 * k)); }

static int pick_method(const dnagpu_count_opts *opts, int k, uint64_t n)
{
    int m = opts ? opts->method : DNAGPU_COUNT_AUTO;
    if (m == DNAGPU_COUNT_DENSE && k > 16) m = DNAGPU_COUNT_HASH;
    if (m != DNAGPU_COUNT_AUTO) return m;
    /* measured on 1 Gbp (profiles/r01a_ksweep): shared-memory / L2-resident dense counters
     * (k <= 12) run at 200-1400 Gkmer/s; dense or hash tables that live in HBM (k >= 13)
     * drop to 15-30 Gkmer/s, where partition + shared-memory count wins by > 5x. */
    if (k <= 12 && pow4_capped(k) <= std::max<uint64_t>(1ull << 16, 8 * n)) return DNAGPU_COUNT_DENSE;
    if (n >= (1ull << 21)) return DNAGPU_COUNT_PARTITION;
    return DNAGPU_COUNT_HASH;
}

template <typename CT>
static int count_dense_t(dnagpu_ctx *ctx, const CountInput &in, int k, dnagpu_stats *stats,
                         dnagpu_table **table)
{
    const uint64_t bins = 1ull << (2 * k);
    const uint64_t mask = kmer_mask(k);
    Scratch sc(ctx);
    CT *tab;
    TRY(sc.get((void **)&tab, bins * sizeof(CT)));
    TRY(launch(ctx, "dense_init", [&] { cudaMemsetAsync(tab, 0, bins * sizeof(CT), ctx->stream); }));
    TRY(zero_counters(ctx));
    if (in.d_keys) {
        TRY(launch(ctx, "count_dense_keys", [&] {
            k_count_dense_keys<CT><<<grid_for(in.n, kThreads * 8), kThreads, 0, ctx->stream>>>(
                in.d_keys, in.n, bins, tab, ctx->d_ctr);
        }));
    } else if (k <= 7) {
        const uint32_t rep_shift = (uint32_t)std::min(5, 14 - 2 * k);
        const int smem = (int)((bins << rep_shift) * sizeof(uint32_t));
        /* persistent grid; enough CTAs that none sees 2^32 k-mers */
        uint64_t want = std::max<uint64_t>((uint64_t)ctx->sm_count * 4, in.v.n_items / (1ull << 26) + 1);
        const unsigned grid = (unsigned)std::min<uint64_t>(want, grid_for(in.v.n_items, kThreads));
        DISPATCH_LAYOUT(in.seq->layout, TRY(launch(ctx, "count_dense_smem", [&] {
            if (in.filtered)
                k_count_dense_smem<LY, true, CT><<<grid, kThreads, smem, ctx->stream>>>(
                    in.v, in.p, mask, (uint32_t)bins, rep_shift, tab, ctx->d_ctr);
            else
                k_count_dense_smem<LY, false, CT><<<grid, kThreads, smem, ctx->stream>>>(
                    in.v, in.p, mask, (uint32_t)bins, rep_shift, tab, ctx->d_ctr);
        })));
    } else {
        const unsigned grid = grid_for(in.v.n_items, kThreads);
        DISPATCH_LAYOUT(in.seq->layout, TRY(launch(ctx, "count_dense", [&] {
            if (in.filtered)
                k_count_dense<LY, true, CT><<<grid, kThreads, 0, ctx->stream>>>(in.v, in.p, mask, tab, ctx->d_ctr);
            else
                k_count_dense<LY, false, CT><<<grid, kThreads, 0, ctx->stream>>>(in.v, in.p, mask, tab, ctx->d_ctr);
        })));
    }
    const unsigned sgrid = (unsigned)std::min<uint64_t>(grid_for(bins, kThreads), (uint64_t)ctx->sm_count * 16);
    TRY(launch(ctx, "dense_stats", [&] {
        if (ctx->spec_h)
            k_dense_stats<CT, true><<<sgrid, kThreads, kSpecSmem, ctx->stream>>>(tab, bins, ctx->d_ctr,
                                                                                ctx->d_spec + kSpecCum, ctx->spec_h);
        else
            k_dense_stats<CT><<<sgrid, kThreads, 0, ctx->stream>>>(tab, bins, ctx->d_ctr);
    }));
    TRY(fetch_counters(ctx));
    if (ctx->h_ctr[C_OVERFLOW]) return fail(ctx, DNAGPU_EARG, "a key is not a %d-mer (>= 4^k)", k);
    stats->total = ctx->h_ctr[C_TOTAL];
    stats->distinct = ctx->h_ctr[C_DISTINCT];
    stats->unique = ctx->h_ctr[C_UNIQUE];
    if (table) {
        TRY(table_new(ctx, k, stats->distinct, table));
        if (stats->distinct)
            TRY(launch(ctx, "dense_compact", [&] {
                k_dense_compact<CT><<<sgrid, kThreads, 0, ctx->stream>>>(tab, bins, (*table)->d_kmers,
                                                                        (*table)->d_counts, ctx->d_ctr);
            }));
    }
    return DNAGPU_OK;
}

static int count_dense_any(dnagpu_ctx *ctx, const CountInput &in, int k, dnagpu_stats *stats, dnagpu_table **table)
{
    return in.n < 0xffffffffull ? count_dense_t<uint32_t>(ctx, in, k, stats, table)
                                : count_dense_t<unsigned long long>(ctx, in, k, stats, table);
}

/* a spectrum query bins the final counts of a hash table (the HBM table, the bucket count's spill table) */
static int table_spectrum(dnagpu_ctx *ctx, const Slot *slots, uint64_t cap)
{
    if (!ctx->spec_h) return DNAGPU_OK;
    const unsigned grid = (unsigned)std::min<uint64_t>(grid_for(cap, kThreads), (uint64_t)ctx->sm_count * 8);
    return launch(ctx, "table_spectrum", [&] {
        k_table_spectrum<<<grid, kThreads, kSpecSmem, ctx->stream>>>(slots, cap, ctx->d_spec + kSpecCum, ctx->spec_h);
    });
}

static int count_hash(dnagpu_ctx *ctx, const CountInput &in, int k, const dnagpu_count_opts *opts,
                      uint64_t n_keys_bound, dnagpu_stats *stats, dnagpu_table **table)
{
    double load = (opts && opts->load_factor > 0.0) ? opts->load_factor : 0.5;
    load = std::min(0.95, std::max(0.05, load));
    uint64_t expected = (opts && opts->expected_keys) ? opts->expected_keys
                                                      : std::min(n_keys_bound, pow4_capped(k));
    uint64_t cap = std::max<uint64_t>(1024, (uint64_t)((double)expected / load) + 1);
    size_t free_b = 0, total_b = 0;
    CU(ctx, cudaMemGetInfo(&free_b, &total_b));
    (void)total_b;
    Scratch sc(ctx);
    Slot *slots = nullptr;
    int rc = sc.get((void **)&slots, cap * sizeof(Slot));
    if (rc == DNAGPU_ENOMEM && !(opts && opts->load_factor > 0.0)) {
        /* default load does not fit: pack the table tighter before giving up */
        cap = std::max<uint64_t>(1024, (uint64_t)((double)expected / 0.85) + 1);
        rc = sc.get((void **)&slots, cap * sizeof(Slot));
    }
    TRY(rc);
    const unsigned igrid = (unsigned)std::min<uint64_t>(grid_for(cap, kThreads), (uint64_t)ctx->sm_count * 32);
    TRY(launch(ctx, "table_init", [&] { k_table_init<<<igrid, kThreads, 0, ctx->stream>>>(slots, cap); }));
    TRY(zero_counters(ctx));
    if (in.d_keys) {
        TRY(launch(ctx, "count_hash_keys", [&] {
            k_count_hash_keys<<<grid_for(in.n, (uint64_t)kThreads * kKeysPerThread), kThreads, 0, ctx->stream>>>(
                in.d_keys, in.n, slots, cap, ctx->d_ctr);
        }));
    } else {
        const unsigned grid = grid_for(in.v.n_items, kThreads);
        const uint64_t mask = kmer_mask(k);
        DISPATCH_LAYOUT(in.seq->layout, TRY(launch(ctx, "count_hash", [&] {
            if (in.filtered)
                k_count_hash<LY, true><<<grid, kThreads, 0, ctx->stream>>>(in.v, in.p, mask, slots, cap, ctx->d_ctr);
            else
                k_count_hash<LY, false><<<grid, kThreads, 0, ctx->stream>>>(in.v, in.p, mask, slots, cap, ctx->d_ctr);
        })));
    }
    TRY(fetch_counters(ctx));
    if (ctx->h_ctr[C_OVERFLOW])
        return fail(ctx, DNAGPU_EINTERNAL, "hash table of %llu slots overflowed (expected_keys too small)",
                    (unsigned long long)cap);
    TRY(table_spectrum(ctx, slots, cap));
    const uint64_t side = ctx->h_ctr[C_SIDE]; /* 'G' x 32, the one key equal to the sentinel */
    ctx->spec_side = side;
    const uint64_t in_table = ctx->h_ctr[C_DISTINCT];
    stats->total = ctx->h_ctr[C_TOTAL];
    stats->distinct = in_table + (side > 0);
    stats->unique = ctx->h_ctr[C_UNIQUE] + (side == 1);
    if (table) {
        TRY(table_new(ctx, k, stats->distinct, table));
        if (in_table) {
            const unsigned cgrid = (unsigned)std::min<uint64_t>(grid_for(cap, kThreads), (uint64_t)ctx->sm_count * 32);
            TRY(launch(ctx, "table_compact", [&] {
                k_table_compact<<<cgrid, kThreads, 0, ctx->stream>>>(slots, cap, (*table)->d_kmers,
                                                                    (*table)->d_counts, ctx->d_ctr);
            }));
        }
        if (side) {
            ctx->h_ctr[0] = kEmpty;
            ctx->h_ctr[1] = side;
            CU(ctx, cudaMemcpyAsync((*table)->d_kmers + in_table, &ctx->h_ctr[0], 8, cudaMemcpyHostToDevice, ctx->stream));
            CU(ctx, cudaMemcpyAsync((*table)->d_counts + in_table, &ctx->h_ctr[1], 8, cudaMemcpyHostToDevice, ctx->stream));
            CU(ctx, cudaStreamSynchronize(ctx->stream));
        }
    }
    return DNAGPU_OK;
}

/* exclusive scan of n u64 (out has n + 1 entries); multi-CTA above 16 K entries */
static int scan_any(dnagpu_ctx *ctx, Scratch &sc, const uint64_t *in, uint64_t n, uint64_t *out)
{
    if (n <= 16384)
        return launch(ctx, "scan", [&] { k_scan_u64<<<1, 1024, 0, ctx->stream>>>(in, n, out); });
    const unsigned blocks = grid_for(n, 1024 * kScanPer);
    uint64_t *sums, *offs;
    TRY(sc.get((void **)&sums, ((uint64_t)blocks + 1) * 8));
    TRY(sc.get((void **)&offs, ((uint64_t)blocks + 1) * 8));
    TRY(launch(ctx, "scan", [&] { k_scan_block<<<blocks, 1024, 0, ctx->stream>>>(in, n, out, sums); }));
    TRY(launch(ctx, "scan", [&] { k_scan_u64<<<1, 1024, 0, ctx->stream>>>(sums, blocks, offs); }));
    TRY(launch(ctx, "scan", [&] { k_scan_add<<<blocks, 1024, 0, ctx->stream>>>(out, n, offs); }));
    return DNAGPU_OK;
}

static int ceil_log2(uint64_t x)
{
    int b = 0;
    while (b < 63 && (1ull << b) < x) ++b;
    return b;
}
/* number of hash bits so that a bucket averages at most half the slots of the shared-memory table */
static int bucket_bits(uint64_t n)
{
    return std::max(1, std::min(22, ceil_log2((n + kBucketSlots / 2 - 1) / (kBucketSlots / 2)))); /* mean <= slots / 2 */
}

/* tile prefix sums of a partitioned key array: out_tile_off[n_parents + 1] */
static int part_tiles(dnagpu_ctx *ctx, Scratch &sc, const uint64_t *parent_off, const uint64_t *parent_end,
                      uint64_t n_parents, uint64_t tile_keys, uint64_t **out_tile_off, TileInfo **out_tile_table = nullptr,
                      uint64_t max_tiles = 0)
{
    if (out_tile_table) *out_tile_table = nullptr;
    uint64_t *tiles;
    TRY(sc.get((void **)&tiles, (n_parents + 1) * 8));
    TRY(sc.get((void **)out_tile_off, (n_parents + 1) * 8));
    TRY(launch(ctx, "part_tiles", [&] {
        k_part_tiles<<<grid_for(n_parents, kThreads), kThreads, 0, ctx->stream>>>(parent_off, parent_end, n_parents,
                                                                                tile_keys, tiles);
    }));
    TRY(scan_any(ctx, sc, tiles, n_parents, *out_tile_off));
    if (out_tile_table && n_parents > 1) { /* one 16-byte entry per CTA of the consumer (max_tiles = its grid) */
        TRY(sc.get((void **)out_tile_table, (max_tiles + 1) * sizeof(TileInfo)));
        CU(ctx, cudaMemsetAsync(*out_tile_table, 0, (max_tiles + 1) * sizeof(TileInfo), ctx->stream));
        TRY(launch(ctx, "part_tiles", [&] {
            k_tile_table<<<grid_for(n_parents, kThreads), kThreads, 0, ctx->stream>>>(parent_off, parent_end, *out_tile_off, n_parents,
                                                                                    tile_keys, max_tiles, *out_tile_table);
        }));
    }
    return DNAGPU_OK;
}

/* ---- GROUP BY kmer by radix partition + shared-memory count (partition.cuh) -------------------- */
/* bits of the two partition levels for n keys spread over n_parts owner ranks (1 = single GPU) */
static void plan_bits(uint64_t n, uint32_t n_parts, int *b1, int *b2)
{
    const int b = bucket_bits(n);
    if (n_parts <= 1) {
        /* the odd bit goes to level 1: level 2 moves twice the bytes per key and gains more from the longer runs of
         * the smaller fan-out (measured: 50.8 -> 49.9 ms) */
        *b1 = b <= 11 ? b : (b + 1) / 2;
        *b2 = std::max(0, std::min(11, b - *b1));
        return;
    }
    /* level 1 must separate the owners; level 2 merges the pieces that arrive from the peers.  Level 1
     * gets as FEW bits as two levels allow: its runs are what crosses NVLink, and they should be long. */
    *b1 = std::min(11, std::max(b - 11, ceil_log2(n_parts) + 2));
    *b2 = std::max(1, std::min(11, b - *b1));
}

/* ---- partition level 1: the launches shared by the local count and the multi-GPU exchange ---------------- */
/* The whole of a key list as the one parent partition the key kernels walk: its range {0, n} on the device.
 * Synchronises: h_ctr is pinned staging shared with the counters. */
static int root_range(dnagpu_ctx *ctx, Scratch &sc, uint64_t n, uint64_t **root)
{
    TRY(sc.get((void **)root, 2 * 8));
    ctx->h_ctr[0] = 0;
    ctx->h_ctr[1] = n;
    CU(ctx, cudaMemcpyAsync(*root, ctx->h_ctr, 16, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return DNAGPU_OK;
}

/* keys per digit of level 1 (1 << b1 digits) into hist (zeroed by the caller), from packed input (the WHERE clause
 * fused) or from a key list whose root_range is `root` */
static int l1_hist(dnagpu_ctx *ctx, Scratch &sc, const CountInput &in, int k, int b1, const uint64_t *root,
                   unsigned long long *hist)
{
    const uint32_t P1 = 1u << b1;
    const int shift1 = 64 - b1;
    if (in.d_keys) {
        uint64_t *tiles;
        TRY(part_tiles(ctx, sc, root, root + 1, 1, kSuperTile, &tiles));
        return launch(ctx, "part_hist", [&] {
            k_part_hist_keys<<<grid_for(in.n, kSuperTile), kThreads, 0, ctx->stream>>>(in.d_keys, root, root + 1, tiles, 1, 1,
                                                                                       shift1, P1, hist);
        });
    }
    const uint64_t mask = kmer_mask(k);
    const unsigned grid = (unsigned)std::min<uint64_t>(grid_for(in.v.n_items, kThreads), (uint64_t)ctx->sm_count * 8);
    DISPATCH_LAYOUT(in.seq->layout, TRY(launch(ctx, "part_hist", [&] {
        if (in.filtered)
            k_part_hist_seq<LY, true><<<grid, kThreads, 0, ctx->stream>>>(in.v, in.p, mask, shift1, P1, hist);
        else
            k_part_hist_seq<LY, false><<<grid, kThreads, 0, ctx->stream>>>(in.v, in.p, mask, shift1, P1, hist);
    })));
    return DNAGPU_OK;
}

/* Level-1 scatter of packed input: digit d's keys go to out[child_off[d] + child_cur[d] ...]; with cap != 0
 * (optimistic regions) a run that finds its region full is dropped and raises C_L1OVF.  16384-key tiles,
 * kBigThreads x kBigPer: measured from packed input they win over 8192-key tiles at every fan-out (256: 15 %,
 * 1024: 12 %, 2048: 2x).  out == NULL: child_off holds destination addresses / 8 (peer_dest), the stores go to
 * peer memory. */
static int l1_scatter_seq(dnagpu_ctx *ctx, int layout, const SeqView &v, const Pred &p, bool filtered, int k, int b1,
                          const uint64_t *child_off, unsigned long long *child_cur, uint64_t *out, uint64_t cap)
{
    const uint32_t P1 = 1u << b1;
    const int shift1 = 64 - b1;
    const uint64_t mask = kmer_mask(k);
    const int psmem = kBigPer * kBigThreads * (int)sizeof(uint64_t) + (int)sizeof(ScatterSmem);
    const unsigned grid = grid_for(v.n_items, kBigPer * kBigThreads / 32); /* packed items (32 starts) per tile */
    DISPATCH_LAYOUT(layout, TRY(launch(ctx, out ? "part_scatter" : "part_scatter_peer", [&] {
        if (filtered)
            k_part_scatter_seq<LY, true><<<grid, kBigThreads, psmem, ctx->stream>>>(v, p, mask, shift1, P1, child_off,
                                                                                   child_cur, out, ctx->d_ctr, cap);
        else
            k_part_scatter_seq<LY, false><<<grid, kBigThreads, psmem, ctx->stream>>>(v, p, mask, shift1, P1, child_off,
                                                                                    child_cur, out, ctx->d_ctr, cap);
    })));
    return DNAGPU_OK;
}

/* The same from a key list whose root_range is `root`; its 'G' x 32 keys are counted aside.  tile32: 16384-key tiles
 * (kBigThreadsKeys x kBigPerKeys) instead of 8192: measured from a key list they win 13 % at a fan-out of 2048, 1 % at
 * 1024 and lose 10 % at 256. */
static int l1_scatter_keys(dnagpu_ctx *ctx, Scratch &sc, const uint64_t *keys, uint64_t n, const uint64_t *root, bool tile32,
                           int b1, const uint64_t *child_off, unsigned long long *child_cur, uint64_t *out, uint64_t cap)
{
    const uint32_t P1 = 1u << b1;
    const int shift1 = 64 - b1;
    const uint64_t tile = tile32 ? 2 * kTileKeys : kTileKeys;
    uint64_t *tiles;
    TRY(part_tiles(ctx, sc, root, root + 1, 1, tile, &tiles));
    const int psmem = (int)tile * (int)sizeof(uint64_t) + (int)sizeof(ScatterSmem);
    return launch(ctx, out ? "part_scatter" : "part_scatter_peer", [&] {
        if (tile32)
            k_part_scatter_keys<true, kBigPerKeys, kBigThreadsKeys><<<grid_for(n, tile), kBigThreadsKeys, psmem, ctx->stream>>>(
                keys, root, root + 1, tiles, 1, 1, shift1, P1, child_off, child_cur, out, ctx->d_ctr, cap, C_L1OVF);
        else
            k_part_scatter_keys<true><<<grid_for(n, tile), kScatThreads, psmem, ctx->stream>>>(
                keys, root, root + 1, tiles, 1, 1, shift1, P1, child_off, child_cur, out, ctx->d_ctr, cap, C_L1OVF);
    });
}

/* Level 1: histogram, offsets (off1: device, P1 + 1 entries) and scatter into `out` (>= n + 2 keys).
 * The device counters C_TOTAL / C_SIDE receive the rows kept by the WHERE clause / the 'G' x 32 rows. */
static int part_level1(dnagpu_ctx *ctx, Scratch &sc, const CountInput &in, int k, int b1, uint64_t **keys_io,
                       uint64_t cap, uint64_t **off1_out, uint64_t *n_out)
{
    const uint32_t P1 = 1u << b1;
    uint64_t n = in.n;
    unsigned long long *hist1, *cur1;
    uint64_t *off1, *root = nullptr;
    TRY(sc.get((void **)&hist1, (uint64_t)P1 * 8));
    TRY(sc.get((void **)&cur1, (uint64_t)P1 * 8));
    TRY(sc.get((void **)&off1, ((uint64_t)P1 + 1) * 8));
    CU(ctx, cudaMemsetAsync(hist1, 0, (uint64_t)P1 * 8, ctx->stream));
    CU(ctx, cudaMemsetAsync(cur1, 0, (uint64_t)P1 * 8, ctx->stream));
    if (in.d_keys) TRY(root_range(ctx, sc, n, &root));
    TRY(l1_hist(ctx, sc, in, k, b1, root, hist1));
    TRY(scan_any(ctx, sc, (const uint64_t *)hist1, P1, off1));
    uint64_t *out = *keys_io;
    if (in.filtered || out) /* the WHERE clause decides how many keys there are; a caller's buffer must fit them */
        TRY(read_u64(ctx, off1 + P1, &n));
    if (!out) {
        TRY(sc.get((void **)&out, (n + 2) * 8));
        *keys_io = out;
    } else if (cap < n + 2) {
        *n_out = n;
        return fail(ctx, DNAGPU_ECAPACITY, "partition needs room for %llu keys (+2 pad)", (unsigned long long)n);
    }
    /* 8192-key tiles from a key list: this exact form counts lists under 2^24 keys, DNAGPU_COUNT_FLAG_EXACT queries and
     * the redo of an optimistic level 1 that found a region full */
    if (in.d_keys)
        TRY(l1_scatter_keys(ctx, sc, in.d_keys, in.n, root, false, b1, off1, cur1, out, 0));
    else
        TRY(l1_scatter_seq(ctx, in.seq->layout, in.v, in.p, in.filtered, k, b1, off1, cur1, out, 0));
    *off1_out = off1;
    *n_out = n;
    return DNAGPU_OK;
}

/* k_count_buckets over n keys in all: one key can occur n times, so past 2^32 - 1 keys the per-slot extras
 * counter is 64-bit (like count_dense_any's counters); every smaller call runs the 32-bit kernel */
template <bool EMIT, bool SPEC = false, class... A>
static void launch_count_buckets(dnagpu_ctx *ctx, uint64_t n, unsigned grid, A... a)
{
    const int spec_smem = SPEC ? kSpecSmem : 0;
    if (n < 0xffffffffull)
        k_count_buckets<EMIT, uint32_t, SPEC><<<grid, kThreads, kBucketSlots * 12 + spec_smem, ctx->stream>>>(a...);
    else
        k_count_buckets<EMIT, unsigned long long, SPEC><<<grid, kThreads, kBucketSlots * 16 + spec_smem, ctx->stream>>>(a...);
}

/* Level 2 (inside every parent; parents with equal parent % n_groups merge into the same children)
 * and the shared-memory count of every bucket.  Leaves distinct / unique in the device counters. */
static int part_finish_impl(dnagpu_ctx *ctx, Scratch &sc, const uint64_t *keys, uint64_t n, const uint64_t *parent_off,
                            const uint64_t *parent_end, uint64_t n_parents, uint64_t n_groups, int b1, int b2, int k,
                            dnagpu_stats *stats, uint64_t total_rows, dnagpu_table **table, bool optimistic2,
                            bool *regions_full)
{
    const int psmem = kTileKeys * (int)sizeof(uint64_t) + (int)sizeof(ScatterSmem);
    const uint64_t *bucket_keys = keys, *bucket_off = parent_off, *bucket_end = parent_end;
    uint64_t n_buckets = n_parents;
    *regions_full = false;
    if (b2 > 0) {
        const uint32_t P2 = 1u << b2;
        const int shift2 = 64 - b1 - b2;
        n_buckets = n_groups * P2;
        unsigned long long *hist2 = nullptr, *cur2;
        uint64_t *off2, *end2 = nullptr, *tiles_hist = nullptr, *tiles_scat, *bufB;
        TileInfo *tparent_hist = nullptr, *tparent_scat = nullptr;
        /* Optimistic level 2 (like level 1): hashing spreads a parent's keys evenly over its children, so every
         * bucket gets a fixed region of mean + 7 sigma and the histogram pass is skipped; a run that finds its
         * region full flags C_L2OVF and part_finish redoes level 2 with the exact histogram + scan. */
        const uint64_t mean2 = (n + n_buckets - 1) / n_buckets;
        const uint64_t cap2 = mean2 + 7 * (uint64_t)std::ceil(std::sqrt((double)mean2)) + 64;
        TRY(sc.get((void **)&cur2, n_buckets * 8));
        TRY(sc.get((void **)&off2, (n_buckets + 1) * 8));
        CU(ctx, cudaMemsetAsync(cur2, 0, n_buckets * 8, ctx->stream));
        if (optimistic2) {
            TRY(sc.get((void **)&end2, n_buckets * 8));
            TRY(sc.get((void **)&bufB, (n_buckets * cap2 + 2) * 8));
            TRY(launch(ctx, "part_tiles", [&] {
                k_region_begs<<<grid_for(n_buckets, kThreads), kThreads, 0, ctx->stream>>>(cap2, n_buckets, off2);
            }));
        } else {
            TRY(sc.get((void **)&hist2, n_buckets * 8));
            TRY(sc.get((void **)&bufB, (n + 2) * 8));
            CU(ctx, cudaMemsetAsync(hist2, 0, n_buckets * 8, ctx->stream));
            TRY(part_tiles(ctx, sc, parent_off, parent_end, n_parents, kSuperTile, &tiles_hist, &tparent_hist,
                           (uint64_t)grid_for(n, kSuperTile) + n_parents));
        }
        /* measured on the headline workload: at a fan-out of 2048 a (tile, digit) run of an 8192-key tile
         * is only 4 keys; 16384-key tiles (one CTA per SM) win 13 % there, are even at 1024 and lose 10 % at 256 */
        const bool per32 = P2 >= 1024;
        TRY(part_tiles(ctx, sc, parent_off, parent_end, n_parents, per32 ? 2 * kTileKeys : kTileKeys, &tiles_scat, &tparent_scat,
                       (uint64_t)grid_for(n, per32 ? 2 * kTileKeys : kTileKeys) + n_parents));
        if (!optimistic2) {
            TRY(launch(ctx, "part_hist2", [&] {
                k_part_hist_keys<<<grid_for(n, kSuperTile) + (unsigned)n_parents, kThreads, 0, ctx->stream>>>(
                    keys, parent_off, parent_end, tiles_hist, n_parents, n_groups, shift2, P2, hist2, tparent_hist);
            }));
            TRY(scan_any(ctx, sc, (const uint64_t *)hist2, n_buckets, off2));
        }
        const uint64_t cap = optimistic2 ? cap2 : 0;
        TRY(launch(ctx, "part_scatter2", [&] {
            if (per32) {
                const int psmem32 = 32 * kScatThreads * (int)sizeof(uint64_t) + (int)sizeof(ScatterSmem);
                k_part_scatter_keys<false, kBigPerKeys, kBigThreadsKeys><<<grid_for(n, 2 * kTileKeys) + (unsigned)n_parents, kBigThreadsKeys, psmem32,
                                                 ctx->stream>>>(keys, parent_off, parent_end, tiles_scat, n_parents, n_groups,
                                                                shift2, P2, off2, cur2, bufB, ctx->d_ctr, cap, C_L2OVF,
                                                                tparent_scat);
            } else {
                k_part_scatter_keys<false><<<grid_for(n, kTileKeys) + (unsigned)n_parents, kScatThreads, psmem, ctx->stream>>>(
                    keys, parent_off, parent_end, tiles_scat, n_parents, n_groups, shift2, P2, off2, cur2, bufB, ctx->d_ctr,
                    cap, C_L2OVF, tparent_scat);
            }
        }));
        bucket_keys = bufB;
        bucket_off = off2;
        bucket_end = off2 + 1;
        if (optimistic2) {
            TRY(launch(ctx, "part_tiles", [&] {
                k_region_ends<<<grid_for(n_buckets, kThreads), kThreads, 0, ctx->stream>>>(cur2, off2, cap2, (uint32_t)n_buckets,
                                                                                         end2);
            }));
            bucket_end = end2;
        }
    }
    const uint64_t spill_cap = std::max<uint64_t>(1ull << 16, n / 64);
    Slot *spill;
    TRY(sc.get((void **)&spill, spill_cap * sizeof(Slot)));
    TRY(launch(ctx, "table_init", [&] {
        k_table_init<<<(unsigned)std::min<uint64_t>(grid_for(spill_cap, kThreads), (uint64_t)ctx->sm_count * 8),
                       kThreads, 0, ctx->stream>>>(spill, spill_cap);
    }));
    const unsigned cgrid = (unsigned)std::min<uint64_t>(n_buckets, (uint64_t)ctx->sm_count * (16384 / kBucketSlots));
    /* the aggregates: bin / place / compare for every bucket that fits, the table kernel for the rest */
    uint32_t *passed;
    TRY(sc.get((void **)&passed, n_buckets * 4 + 16));
    const unsigned bgrid = (unsigned)std::min<uint64_t>(n_buckets, (uint64_t)ctx->sm_count * ctx->bins_ctas_per_sm);
    TRY(launch(ctx, "count_buckets", [&] {
        if (ctx->spec_h)
            k_count_buckets_bins<true><<<bgrid, kThreads, 0, ctx->stream>>>(bucket_keys, bucket_off, bucket_end, n_buckets,
                                                                            ctx->d_ctr, passed, ctx->d_ctr + C_PASSED,
                                                                            ctx->d_spec);
        else
            k_count_buckets_bins<<<bgrid, kThreads, 0, ctx->stream>>>(bucket_keys, bucket_off, bucket_end, n_buckets,
                                                                     ctx->d_ctr, passed, ctx->d_ctr + C_PASSED);
    }));
    TRY(launch(ctx, "count_buckets_passed", [&] {
        if (ctx->spec_h)
            launch_count_buckets<false, true>(ctx, n, cgrid, bucket_keys, bucket_off, bucket_end, n_buckets, spill,
                                              spill_cap, ctx->d_ctr, (uint64_t *)nullptr, (uint64_t *)nullptr,
                                              (const uint32_t *)passed, (const unsigned long long *)ctx->d_ctr + C_PASSED,
                                              ctx->d_spec + kSpecCum, ctx->spec_h);
        else
            launch_count_buckets<false>(ctx, n, cgrid, bucket_keys, bucket_off, bucket_end, n_buckets, spill, spill_cap,
                                        ctx->d_ctr, (uint64_t *)nullptr, (uint64_t *)nullptr, (const uint32_t *)passed,
                                        (const unsigned long long *)ctx->d_ctr + C_PASSED);
    }));
    TRY(fetch_counters(ctx));
    if (ctx->h_ctr[C_L2OVF]) { /* some keys were dropped: the caller redoes level 2 exactly */
        *regions_full = true;
        return DNAGPU_OK;
    }
    if (ctx->h_ctr[C_OVERFLOW])
        return fail(ctx, DNAGPU_EINTERNAL, "spill table of %llu slots overflowed", (unsigned long long)spill_cap);
    TRY(table_spectrum(ctx, spill, spill_cap));
    const uint64_t side = ctx->h_ctr[C_SIDE];
    ctx->spec_side = side;
    const uint64_t keyed = ctx->h_ctr[C_DISTINCT];
    stats->total = total_rows ? total_rows : ctx->h_ctr[C_TOTAL];
    stats->distinct = keyed + (side > 0);
    stats->unique = ctx->h_ctr[C_UNIQUE] + (side == 1);
    if (table) {
        TRY(table_new(ctx, k, stats->distinct, table));
        if (keyed) {
            CU(ctx, cudaMemsetAsync(ctx->d_ctr + C_CURSOR, 0, 8, ctx->stream));
            TRY(launch(ctx, "count_buckets_emit", [&] {
                launch_count_buckets<true>(ctx, n, cgrid, bucket_keys, bucket_off, bucket_end, n_buckets, spill, spill_cap,
                                           ctx->d_ctr, (*table)->d_kmers, (*table)->d_counts);
            }));
            TRY(launch(ctx, "table_compact", [&] { /* rows that spilled, appended after the bucket rows */
                k_table_compact<<<(unsigned)std::min<uint64_t>(grid_for(spill_cap, kThreads), (uint64_t)ctx->sm_count * 8),
                                  kThreads, 0, ctx->stream>>>(spill, spill_cap, (*table)->d_kmers,
                                                              (*table)->d_counts, ctx->d_ctr);
            }));
        }
        if (side) {
            ctx->h_ctr[0] = kEmpty;
            ctx->h_ctr[1] = side;
            CU(ctx, cudaMemcpyAsync((*table)->d_kmers + keyed, &ctx->h_ctr[0], 8, cudaMemcpyHostToDevice, ctx->stream));
            CU(ctx, cudaMemcpyAsync((*table)->d_counts + keyed, &ctx->h_ctr[1], 8, cudaMemcpyHostToDevice, ctx->stream));
        }
        CU(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return DNAGPU_OK;
}

static int part_finish(dnagpu_ctx *ctx, Scratch &sc, const uint64_t *keys, uint64_t n, const uint64_t *parent_off,
                       const uint64_t *parent_end, uint64_t n_parents, uint64_t n_groups, int b1, int b2, int k,
                       dnagpu_stats *stats, uint64_t total_rows, dnagpu_table **table)
{
    /* optimistic level 2 where no parents merge (one GPU) and the buckets are full-sized */
    const bool optimistic2 = !ctx->force_exact && b2 > 0 && n_groups == n_parents && (n >> (b1 + b2)) >= 512;
    bool full = false;
    TRY(part_finish_impl(ctx, sc, keys, n, parent_off, parent_end, n_parents, n_groups, b1, b2, k, stats, total_rows, table,
                         optimistic2, &full));
    if (!full) return DNAGPU_OK;
    /* the counters of the scatter passes before (rows kept, 'G' x 32 rows, level-1 flag) stay; the count starts over */
    CU(ctx, cudaMemsetAsync(ctx->d_ctr + C_DISTINCT, 0, 2 * 8, ctx->stream));
    CU(ctx, cudaMemsetAsync(ctx->d_ctr + C_OVERFLOW, 0, 2 * 8, ctx->stream));
    CU(ctx, cudaMemsetAsync(ctx->d_ctr + C_L2OVF, 0, 2 * 8, ctx->stream));
    TRY(zero_spectrum(ctx));
    if (table && *table) {
        dnagpu_table_free(*table);
        *table = nullptr;
    }
    return part_finish_impl(ctx, sc, keys, n, parent_off, parent_end, n_parents, n_groups, b1, b2, k, stats, total_rows, table,
                            false, &full);
}

/* Optimistic level 1 (unfiltered packed input): no histogram pass.  Hashing spreads the keys evenly, so
 * every partition gets a fixed region of mean + 12.5 % + 65536 keys; a (tile, digit) run that finds its region
 * full is dropped and flags C_L1OVF, and the caller redoes the query with the exact two-pass level 1
 * (only heavily repeated input -- e.g. a poly-A run of millions of bases -- ever gets there). */
struct L1Regions {
    uint64_t *keys = nullptr, *beg = nullptr, *end = nullptr;
    unsigned long long *cur = nullptr;
    uint64_t cap = 0;
    uint32_t P1 = 0;
    int b1 = 0;
};

static int l1_regions_begin(dnagpu_ctx *ctx, Scratch &sc, uint64_t n_rows, int b1, L1Regions *r)
{
    r->b1 = b1;
    r->P1 = 1u << b1;
    const uint64_t mean = n_rows >> b1; /* hashing is even; the slack is for k-mers with many copies */
    r->cap = mean + mean / 8 + std::min<uint64_t>(65536, std::max<uint64_t>(1024, mean / 2));
    TRY(sc.get((void **)&r->keys, ((uint64_t)r->P1 * r->cap + 2) * 8));
    TRY(sc.get((void **)&r->beg, (uint64_t)r->P1 * 8));
    TRY(sc.get((void **)&r->end, (uint64_t)r->P1 * 8));
    TRY(sc.get((void **)&r->cur, (uint64_t)r->P1 * 8));
    TRY(launch(ctx, "part_tiles", [&] {
        k_region_begs<<<grid_for(r->P1, kThreads), kThreads, 0, ctx->stream>>>(r->cap, r->P1, r->beg);
    }));
    CU(ctx, cudaMemsetAsync(r->cur, 0, (uint64_t)r->P1 * 8, ctx->stream));
    return DNAGPU_OK;
}

static int l1_regions_scatter(dnagpu_ctx *ctx, const L1Regions &r, int layout, const SeqView &v, int k)
{
    const Pred none = {~0ull, ~0ull, ~0ull, ~0ull};
    return l1_scatter_seq(ctx, layout, v, none, false, k, r.b1, r.beg, r.cur, r.keys, r.cap);
}

/* the same from a key list on the device (the owned k-mers of a multi-GPU count, a stored column): 16384-key tiles,
 * 'G' x 32 keys counted aside */
static int l1_regions_scatter_keys(dnagpu_ctx *ctx, Scratch &sc, const L1Regions &r, const uint64_t *d_keys, uint64_t n)
{
    uint64_t *root;
    TRY(root_range(ctx, sc, n, &root));
    return l1_scatter_keys(ctx, sc, d_keys, n, root, true, r.b1, r.beg, r.cur, r.keys, r.cap);
}

static int l1_regions_end(dnagpu_ctx *ctx, const L1Regions &r)
{
    return launch(ctx, "part_tiles", [&] {
        k_region_ends<<<grid_for(r.P1, kThreads), kThreads, 0, ctx->stream>>>(r.cur, r.beg, r.cap, r.P1, r.end);
    });
}

static int count_partition_exact(dnagpu_ctx *ctx, const CountInput &in, int k, dnagpu_stats *stats,
                                 dnagpu_table **table)
{
    Scratch sc(ctx);
    int b1, b2;
    plan_bits(in.n, 1, &b1, &b2);
    TRY(zero_counters(ctx));
    uint64_t *off1, n, *keys = nullptr;
    TRY(part_level1(ctx, sc, in, k, b1, &keys, 0, &off1, &n));
    if (in.filtered) { /* fewer keys than rows: the second level may not be needed any more */
        int e1, e2;
        plan_bits(n, 1, &e1, &e2);
        b2 = std::max(0, std::min(11, e1 + e2 - b1));
    }
    const uint64_t P1 = 1ull << b1;
    return part_finish(ctx, sc, keys, n, off1, off1 + 1, P1, P1, b1, b2, k, stats, 0, table);
}

static int count_partition(dnagpu_ctx *ctx, const CountInput &in, int k, dnagpu_stats *stats,
                           dnagpu_table **table)
{
    if (in.filtered || ctx->force_exact || (in.d_keys && in.n < (1ull << 24)))
        return count_partition_exact(ctx, in, k, stats, table);
    {
        Scratch sc(ctx);
        int b1, b2;
        plan_bits(in.n, 1, &b1, &b2);
        TRY(zero_counters(ctx));
        L1Regions r;
        TRY(l1_regions_begin(ctx, sc, in.n, b1, &r));
        if (in.d_keys)
            TRY(l1_regions_scatter_keys(ctx, sc, r, in.d_keys, in.n));
        else
            TRY(l1_regions_scatter(ctx, r, in.seq->layout, in.v, k));
        TRY(l1_regions_end(ctx, r));
        TRY(part_finish(ctx, sc, r.keys, in.n, r.beg, r.end, r.P1, r.P1, b1, b2, k, stats, 0, table));
        if (!ctx->h_ctr[C_L1OVF]) return DNAGPU_OK;
        if (table && *table) {
            dnagpu_table_free(*table);
            *table = nullptr;
        }
    }
    return count_partition_exact(ctx, in, k, stats, table); /* a region overflowed: heavily repeated input */
}

/* rc of a count; a failed count leaves no table behind */
static int free_table_on_error(int rc, dnagpu_table **table)
{
    if (rc != DNAGPU_OK && table && *table) {
        dnagpu_table_free(*table);
        *table = nullptr;
    }
    return rc;
}

/* the count itself, by the method pick_method chose */
static int count_by_method(dnagpu_ctx *ctx, const CountInput &in, int k, int method, const dnagpu_count_opts *opts,
                           uint64_t n_keys_bound, dnagpu_stats *stats, dnagpu_table **table)
{
    int rc;
    if (method == DNAGPU_COUNT_DENSE)
        rc = count_dense_any(ctx, in, k, stats, table);
    else if (method == DNAGPU_COUNT_PARTITION)
        rc = count_partition(ctx, in, k, stats, table);
    else
        rc = count_hash(ctx, in, k, opts, n_keys_bound, stats, table);
    return free_table_on_error(rc, table);
}

/* one chunk of a pipelined upload: H2D on the copy stream, the compute stream waits for it.  Never returns
 * early with an event outside `ev` (the callers destroy the events on every path). */
static int chunk_copy(dnagpu_ctx *ctx, std::vector<cudaEvent_t> &ev, uint64_t *dst, const uint64_t *src, uint64_t bytes)
{
    cudaEvent_t e;
    cudaError_t err = cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    if (err != cudaSuccess) return fail(ctx, DNAGPU_ECUDA, "cudaEventCreate: %s", cudaGetErrorString(err));
    ev.push_back(e);
    err = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->copy_stream);
    if (err == cudaSuccess) err = cudaEventRecord(e, ctx->copy_stream);
    if (err == cudaSuccess) err = cudaStreamWaitEvent(ctx->stream, e, 0);
    if (err != cudaSuccess) return fail(ctx, DNAGPU_ECUDA, "pipelined H2D copy: %s", cudaGetErrorString(err));
    return DNAGPU_OK;
}

/* The host-buffer query with the upload hidden behind level 1: the packed words are copied in chunks on
 * a second stream and every chunk is scattered as soon as it has landed (the optimistic level 1 needs no
 * histogram over the whole input first). */
static int count_kmers_pipelined(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_bases, int k,
                                 dnagpu_stats *stats, dnagpu_table **table, bool *done)
{
    *done = false;
    const uint64_t rows = rows_of(n_bases, k), n_words = words_of(n_bases);
    if (pick_method(nullptr, k, rows) != DNAGPU_COUNT_PARTITION) return DNAGPU_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    if (!ctx->copy_stream) CU(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    Scratch words_sc(ctx), sc(ctx); /* the words outlive the optimistic pass's scratch (see the redo below) */
    uint64_t *d_words;
    const uint64_t alloc_words = (n_words + 3) & ~1ull;
    TRY(words_sc.get((void **)&d_words, alloc_words * 8));
    CU(ctx, cudaMemsetAsync(d_words + n_words, 0, (alloc_words - n_words) * 8, ctx->stream));
    int b1, b2;
    plan_bits(rows, 1, &b1, &b2);
    TRY(zero_counters(ctx));
    L1Regions r;
    TRY(l1_regions_begin(ctx, sc, rows, b1, &r));
    CU(ctx, cudaStreamSynchronize(ctx->stream)); /* d_words (stream-ordered allocation) exists before the copy stream writes it */
    const int n_chunks = 8;
    const uint64_t chunk_words = ((n_words + n_chunks - 1) / n_chunks + 255) & ~255ull;
    std::vector<cudaEvent_t> ev;
    int rc = DNAGPU_OK;
    for (uint64_t w0 = 0; w0 < n_words && rc == DNAGPU_OK; w0 += chunk_words) {
        const uint64_t w1 = std::min(n_words, w0 + chunk_words);
        const uint64_t copy_end = std::min(n_words, w1 + 1); /* + the halo word of the chunk's last windows */
        rc = chunk_copy(ctx, ev, d_words + w0, words + w0, (copy_end - w0) * 8);
        if (rc != DNAGPU_OK) break;
        const uint64_t row0 = w0 * 32, row1 = std::min(rows, w1 * 32);
        if (row1 <= row0) continue;
        SeqView v;
        memset(&v, 0, sizeof v);
        v.words = d_words + w0;
        v.n_seqs = 1;
        v.rows_per_seq = v.n_rows = row1 - row0;
        v.items_per_seq = v.n_items = (v.n_rows + 31) / 32;
        rc = l1_regions_scatter(ctx, r, kSingle, v, k);
    }
    if (rc == DNAGPU_OK) rc = l1_regions_end(ctx, r);
    if (rc == DNAGPU_OK) rc = part_finish(ctx, sc, r.keys, rows, r.beg, r.end, r.P1, r.P1, b1, b2, k, stats, 0, table);
    /* on every path: the copy stream must be done with d_words before Scratch hands it back to the pool */
    cudaStreamSynchronize(ctx->copy_stream);
    if (rc != DNAGPU_OK) cudaStreamSynchronize(ctx->stream);
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
    TRY(rc);
    if (ctx->h_ctr[C_L1OVF]) { /* redo exactly, on the words that are resident now */
        if (table && *table) {
            dnagpu_table_free(*table);
            *table = nullptr;
        }
        /* the regions and buckets of the optimistic pass go back to the pool before the exact pass allocates its
         * own, so the redo needs no more device memory than an exact count of the resident words */
        for (void *p : sc.ptrs) dfree(ctx, p);
        sc.ptrs.clear();
        dnagpu_seq *seq = nullptr;
        TRY(dnagpu_seq_wrap(ctx, d_words, n_bases, alloc_words, &seq));
        rc = dnagpu_count(ctx, seq, k, nullptr, nullptr, stats, table);
        dnagpu_seq_free(seq);
        TRY(rc);
    }
    *done = true;
    return DNAGPU_OK;
}

/* One predicate scan, matches appended in no particular order. */
static int collect_launch(dnagpu_ctx *ctx, int layout, const SeqView &v, const Pred &p, int k, uint64_t *d_out, uint64_t cap)
{
    if (layout != kRagged && !ctx->plane_filter) { /* Shift-And over the base stream: 6 instructions per base */
        const SaPred sp = sa_pred_of(p, k);
        const uint64_t runs = layout == kSingle ? (v.n_items + kSaItems - 1) / kSaItems
                                                : v.n_seqs * ((v.items_per_seq + kSaItems - 1) / kSaItems);
        const int smem = kSaStage * (int)sizeof(uint64_t);
        return launch(ctx, "filter_collect", [&] {
            if (layout == kSingle)
                k_filter_sa<kSingle, kSaCollect><<<grid_for(runs, kThreads), kThreads, smem, ctx->stream>>>(
                    v, sp, kmer_mask(k), k, cap, ctx->d_ctr + C_CURSOR, nullptr, d_out);
            else
                k_filter_sa<kFixed, kSaCollect><<<grid_for(runs, kThreads), kThreads, smem, ctx->stream>>>(
                    v, sp, kmer_mask(k), k, cap, ctx->d_ctr + C_CURSOR, nullptr, d_out);
        });
    }
    const unsigned tiles = grid_for(v.n_items, kThreads);
    const int smem = kThreads * 32 * (int)sizeof(uint64_t);
    DISPATCH_LAYOUT(layout, TRY(launch(ctx, "filter_collect", [&] {
        k_filter_collect<LY><<<(tiles + kFilterTiles - 1) / kFilterTiles, kThreads, smem, ctx->stream>>>(
            v, p, kmer_mask(k), cap, ctx->d_ctr + C_CURSOR, d_out);
    })));
    return DNAGPU_OK;
}

static int collect_rows(dnagpu_ctx *ctx, const CountInput &in, int k, uint64_t *d_out, uint64_t cap, uint64_t *n_match)
{
    TRY(zero_counters(ctx));
    TRY(collect_launch(ctx, in.seq->layout, in.v, in.p, k, d_out, cap));
    return read_u64(ctx, (const uint64_t *)(ctx->d_ctr + C_CURSOR), n_match);
}

static int count_listed(dnagpu_ctx *ctx, const uint64_t *keys, uint64_t n_match, int k, const dnagpu_count_opts *opts,
                        dnagpu_stats *stats, dnagpu_table **table);

/* ---- multi-GPU: the k-mers of one owner out of the whole sequence (k_collect_owned + the key-list count) ----- */
/* the walk order of k_collect_owned: every piece padded to whole tiles of `tile` items */
static int owned_view(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k, uint64_t tile, OwnedView *ov)
{
    CHECK_OWNED(ctx, seq, "the sequence");
    memset(ov, 0, sizeof *ov);
    if (seq->layout == kSingle) {
        uint64_t r = rows_of(seq->bases, k);
        if (seq->start_limit) r = std::min(r, seq->start_limit);
        ov->ptr[0] = seq->d_words;
        ov->nitems[0] = (r + 31) / 32;
        ov->vfirst[1] = (ov->nitems[0] + tile - 1) / tile * tile;
        ov->n_rows = r;
        ov->n_pieces = 1;
        return DNAGPU_OK;
    }
    if (seq->layout != kPieces)
        return fail(ctx, DNAGPU_EARG, "an owner restriction applies to a single sequence (whole or in pieces)");
    const uint64_t rows = rows_of(seq->bases, k);
    ov->n_rows = rows;
    ov->n_pieces = (uint32_t)seq->piece_ptr.size();
    uint64_t v = 0;
    for (uint32_t i = 0; i < ov->n_pieces; ++i) {
        const uint64_t fb = seq->piece_first[i];
        const uint64_t starts = rows > fb ? std::min(seq->piece_starts[i], rows - fb) : 0;
        ov->ptr[i] = seq->piece_ptr[i];
        ov->gfirst[i] = fb / 32;
        ov->vfirst[i] = v;
        ov->nitems[i] = (starts + 31) / 32;
        v += (ov->nitems[i] + tile - 1) / tile * tile;
    }
    ov->vfirst[ov->n_pieces] = v;
    return DNAGPU_OK;
}

static int count_owned(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k, const dnagpu_count_opts *opts, dnagpu_stats *stats,
                       dnagpu_table **table)
{
    const uint32_t G = opts->owner_parts, me = opts->owner_part;
    if (G > (uint32_t)kMaxParts || me >= G) return fail(ctx, DNAGPU_EARG, "owner_part must be below owner_parts <= %d", kMaxParts);
    dnagpu_stats local;
    if (!stats) stats = &local;
    stats->total = stats->distinct = stats->unique = 0;
    if (table) *table = nullptr;
    const int wpt = G >= 8 ? 4 : G >= 4 ? 2 : 1; /* a CTA examines 256 * wpt words and keeps ~ 8192 * wpt / G k-mers */
    OwnedView ov;
    TRY(owned_view(ctx, seq, k, (uint64_t)kOwnThreads * wpt, &ov));
    if (ov.n_rows == 0) {
        if (table) TRY(table_new(ctx, k, 0, table));
        return DNAGPU_OK;
    }
    const OwnRange own = own_range_of(G, me, k); /* what owner_of maps to `me` */
    const int lin = owner_lin_bits(G);
    const uint64_t n_expect = ov.n_rows / G + 1;
    const uint64_t n_vitems = ov.vfirst[ov.n_pieces];
    const uint64_t mask = kmer_mask(k);
    /* 1. the owned k-mers as a key list: the staged kernel first, the one that takes any input if a tile's list
     *    overflowed (or the list ran past its guess: more than the expected share + 1.5 %) */
    Scratch sc(ctx);
    uint64_t cap = n_expect + n_expect / 64 + 65536, n_own = 0, *keys = nullptr;
    bool staged = !(opts->flags & DNAGPU_COUNT_FLAG_EXACT);
    for (int attempt = 0; attempt < 3; ++attempt) {
        TRY(sc.get((void **)&keys, (cap + 2) * 8));
        TRY(zero_counters(ctx));
        if (staged) {
            const unsigned grid = grid_for(n_vitems, (uint64_t)kOwnThreads * wpt);
#define OWNED_LAUNCH(WPT, LIN, ML) \
    k_collect_owned<WPT, LIN, ML><<<grid, kOwnThreads, 0, ctx->stream>>>(ov, mask, own, cap, ctx->d_ctr, keys)
            TRY(launch(ctx, "collect_owned", [&] {
                if (k < 16) {
                    if (lin == 3) OWNED_LAUNCH(4, 3, true); else if (lin == 2) OWNED_LAUNCH(2, 2, true); else if (lin == 1) OWNED_LAUNCH(1, 1, true);
                    else if (wpt == 4) OWNED_LAUNCH(4, 0, true); else if (wpt == 2) OWNED_LAUNCH(2, 0, true); else OWNED_LAUNCH(1, 0, true);
                } else {
                    if (lin == 3) OWNED_LAUNCH(4, 3, false); else if (lin == 2) OWNED_LAUNCH(2, 2, false); else if (lin == 1) OWNED_LAUNCH(1, 1, false);
                    else if (wpt == 4) OWNED_LAUNCH(4, 0, false); else if (wpt == 2) OWNED_LAUNCH(2, 0, false); else OWNED_LAUNCH(1, 0, false);
                }
            }));
#undef OWNED_LAUNCH
        } else {
            const unsigned grid = (unsigned)std::min<uint64_t>(grid_for(n_vitems, kScatThreads), (uint64_t)ctx->sm_count * 8);
#define OWNED_ANY(LIN) k_collect_owned_any<LIN><<<grid, kScatThreads, 0, ctx->stream>>>(ov, mask, own, cap, ctx->d_ctr + C_CURSOR, keys)
            TRY(launch(ctx, "collect_owned_any", [&] {
                if (lin == 3) OWNED_ANY(3); else if (lin == 2) OWNED_ANY(2); else if (lin == 1) OWNED_ANY(1); else OWNED_ANY(0);
            }));
#undef OWNED_ANY
        }
        TRY(fetch_counters(ctx));
        n_own = ctx->h_ctr[C_CURSOR];
        const bool dropped = staged && ctx->h_ctr[C_L1OVF];
        if (!dropped && n_own <= cap) break;
        if (attempt == 2) return fail(ctx, DNAGPU_EINTERNAL, "the owned k-mers could not be collected");
        sc.release(keys);
        dfree(ctx, keys);
        if (dropped) staged = false;   /* the cursor missed what was dropped: size the retry generously */
        cap = dropped ? std::max(cap, n_own + n_own / 2 + 65536) : n_own;
    }
    if (n_own == 0) {
        if (table) TRY(table_new(ctx, k, 0, table));
        return DNAGPU_OK;
    }
    /* 2. the single-GPU pipeline over the list (optimistic level 1 from keys, level 2, bucket count) */
    dnagpu_count_opts o2 = *opts;
    o2.owner_parts = o2.owner_part = 0;
    o2.method = DNAGPU_COUNT_AUTO;
    ctx->force_exact = (opts->flags & DNAGPU_COUNT_FLAG_EXACT) != 0;
    const int rc = count_listed(ctx, keys, n_own, k, &o2, stats, table);
    ctx->force_exact = false;
    return rc;
}

/* GROUP BY over a key list on the device (what a WHERE clause kept) */
static int count_listed(dnagpu_ctx *ctx, const uint64_t *keys, uint64_t n_match, int k, const dnagpu_count_opts *opts,
                        dnagpu_stats *stats, dnagpu_table **table)
{
    CountInput listed;
    listed.d_keys = keys;
    listed.n = n_match;
    dnagpu_count_opts o2 = opts ? *opts : dnagpu_count_opts{0, 0, 0.0, 0, 0, 0};
    return count_by_method(ctx, listed, k, pick_method(&o2, k, n_match), opts, n_match, stats, table);
}

static int count_any(dnagpu_ctx *ctx, CountInput &in, int k, const dnagpu_count_opts *opts,
                     dnagpu_stats *stats, dnagpu_table **table)
{
    dnagpu_stats local;
    if (!stats) stats = &local;
    stats->total = stats->distinct = stats->unique = 0;
    if (table) *table = nullptr;
    if (in.n == 0) {
        if (table) TRY(table_new(ctx, k, 0, table));
        return DNAGPU_OK;
    }
    const int method = pick_method(opts, k, in.n);
    struct ExactScope { /* the flag holds for this query only */
        dnagpu_ctx *c;
        ~ExactScope() { c->force_exact = false; }
    } exact_scope{ctx};
    ctx->force_exact = opts && (opts->flags & DNAGPU_COUNT_FLAG_EXACT);
    /* A selective WHERE clause: evaluate it once into an ordered key list (two cheap predicate
     * scans: count per tile, then write) and count that list, instead of dragging the whole
     * input through the partition / hash machinery only to drop most of it. */
    Scratch keep(ctx);
    if (in.filtered && in.seq && method != DNAGPU_COUNT_DENSE) {
        /* one predicate scan: matches are appended (unordered -- GROUP BY does not care) to a buffer sized
         * for a selectivity of 1/8; only a less selective clause needs the second, exactly sized scan */
        uint64_t n_match = 0, cap0 = std::min<uint64_t>(in.n, std::max<uint64_t>(1ull << 20, in.n / 8));
        uint64_t *keys;
        TRY(keep.get((void **)&keys, (cap0 + 2) * 8));
        for (int attempt = 0; attempt < 2; ++attempt) {
            TRY(collect_rows(ctx, in, k, keys, cap0, &n_match));
            if (n_match <= cap0) break;
            keep.release(keys);
            dfree(ctx, keys);
            cap0 = n_match;
            TRY(keep.get((void **)&keys, (cap0 + 2) * 8));
        }
        if (n_match == 0) {
            if (table) TRY(table_new(ctx, k, 0, table));
            return DNAGPU_OK;
        }
        if (n_match <= in.n / 2 || method == DNAGPU_COUNT_PARTITION) return count_listed(ctx, keys, n_match, k, opts, stats, table);
        if (method == DNAGPU_COUNT_HASH) /* not selective: fused insert into a table sized by n_match */
            return count_by_method(ctx, in, k, method, opts, n_match, stats, table);
    }
    return count_by_method(ctx, in, k, method, opts, in.n, stats, table);
}

extern "C" int dnagpu_collect(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k, const dnagpu_where *filter,
                              uint64_t *d_out, uint64_t cap, uint64_t *n_out)
{
    if (!ctx || !seq || !n_out || (cap && !d_out)) return fail(ctx, DNAGPU_EARG, "dnagpu_collect: NULL argument");
    TRY(check_k(ctx, k));
    TRY(check_filter_literals(ctx, filter));
    CU(ctx, cudaSetDevice(ctx->device));
    *n_out = 0;
    CountInput in;
    in.seq = seq;
    TRY(make_view(ctx, seq, k, &in.v));
    in.n = in.v.n_rows;
    TRY(build_pred(ctx, filter, k, in.n, &in.p, &in.filtered));
    if (in.n == 0) return DNAGPU_OK;
    TRY(collect_rows(ctx, in, k, d_out, cap, n_out));
    if (d_out && *n_out > cap)
        return fail(ctx, DNAGPU_ECAPACITY, "collect needs room for %llu rows", (unsigned long long)*n_out);
    return DNAGPU_OK; /* d_out == NULL: only the number of rows was asked for */
}

extern "C" int dnagpu_count(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k,
                            const dnagpu_where *filter, const dnagpu_count_opts *opts,
                            dnagpu_stats *stats, dnagpu_table **table)
{
    if (!ctx || !seq) return fail(ctx, DNAGPU_EARG, "dnagpu_count: NULL argument");
    TRY(check_k(ctx, k));
    TRY(check_filter_literals(ctx, filter));
    CU(ctx, cudaSetDevice(ctx->device));
    /* one owner of a sequence in pieces is the whole count of one GPU's ring; of a single sequence, no restriction */
    if (opts && (opts->owner_parts > 1 || (opts->owner_parts == 1 && seq->layout == kPieces))) {
        if (filter && (filter->prefix_len || filter->qkmer))
            return fail(ctx, DNAGPU_EARG, "an owner restriction cannot be combined with a WHERE clause");
        if (opts->method != DNAGPU_COUNT_AUTO && opts->method != DNAGPU_COUNT_PARTITION)
            return fail(ctx, DNAGPU_EARG, "an owner restriction needs method AUTO or PARTITION");
        return count_owned(ctx, seq, k, opts, stats, table);
    }
    CountInput in;
    in.seq = seq;
    TRY(make_view(ctx, seq, k, &in.v));
    in.n = in.v.n_rows;
    TRY(build_pred(ctx, filter, k, in.n, &in.p, &in.filtered));
    return count_any(ctx, in, k, opts, stats, table);
}

extern "C" int dnagpu_count_keys(dnagpu_ctx *ctx, const uint64_t *d_keys, uint64_t n, int k,
                                 const dnagpu_count_opts *opts, dnagpu_stats *stats,
                                 dnagpu_table **table)
{
    if (!ctx || (!d_keys && n)) return fail(ctx, DNAGPU_EARG, "dnagpu_count_keys: NULL argument");
    TRY(check_k(ctx, k));
    CU(ctx, cudaSetDevice(ctx->device));
    CountInput in;
    in.d_keys = d_keys;
    in.n = n;
    return count_any(ctx, in, k, opts, stats, table);
}

/* The abundance spectrum: the query dnagpu_count runs, with spec_h set so that every count method bins its final
 * counts on the way (see kernels.cuh for the device layout).  Here the parts are added up:
 *   cumulative part (k_count_buckets_bins):  groups of count c = C[c] - C[c+1] for c < H, count >= H = C[H];
 *   direct part (every other kernel):         already binned by min(count, H);
 *   'G' x 32 (k = 32):                        one group of count spec_side. */
extern "C" int dnagpu_count_spectrum(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k, const dnagpu_where *filter,
                                     const dnagpu_count_opts *opts, uint32_t max_count, uint64_t *hist,
                                     dnagpu_stats *stats)
{
    if (!ctx || !seq || !hist) return fail(ctx, DNAGPU_EARG, "dnagpu_count_spectrum: NULL argument");
    if (max_count < 1 || max_count > kSpecMaxCount)
        return fail(ctx, DNAGPU_EARG, "max_count must be between 1 and %u", kSpecMaxCount);
    TRY(check_k(ctx, k));
    TRY(check_filter_literals(ctx, filter));
    CU(ctx, cudaSetDevice(ctx->device));
    if (ctx->spec_alloc < max_count) {
        if (ctx->d_spec) CU(ctx, cudaFree(ctx->d_spec));
        ctx->d_spec = nullptr;
        ctx->spec_alloc = 0;
        CU(ctx, cudaMalloc((void **)&ctx->d_spec, (kSpecCum + (uint64_t)max_count) * 8));
        ctx->spec_alloc = max_count;
    }
    struct SpecScope { /* the spectrum is wanted by this query only */
        dnagpu_ctx *c;
        ~SpecScope() { c->spec_h = 0; }
    } spec_scope{ctx};
    ctx->spec_h = max_count;
    ctx->spec_side = 0;
    TRY(zero_spectrum(ctx)); /* a count that finds no rows launches nothing */
    dnagpu_stats st;
    TRY(dnagpu_count(ctx, seq, k, filter, opts, &st, nullptr));
    uint64_t cum[kSpecCum];
    CU(ctx, cudaMemcpyAsync(cum, ctx->d_spec, sizeof cum, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaMemcpyAsync(hist, ctx->d_spec + kSpecCum, (uint64_t)max_count * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    for (uint32_t c = 1; c < (uint32_t)kSpecCum && c <= max_count; ++c)
        hist[c - 1] += c < max_count ? cum[c] - (c + 1 < (uint32_t)kSpecCum ? cum[c + 1] : 0) : cum[c];
    if (ctx->spec_side) hist[std::min<uint64_t>(ctx->spec_side, max_count) - 1] += 1;
    if (stats) *stats = st;
    return DNAGPU_OK;
}

/* The host-buffer GROUP BY on every GPU of a multi context: shard d of the packed words goes to GPU d (H2D on
 * all PCIe links at once), then every GPU walks ALL shards through peer memory -- its own first, the others in
 * ring order -- and counts the k-mers it owns.  One host thread per GPU drives its (synchronous) count.  With
 * max_count > 0 every GPU takes the spectrum of its share instead of a table, and the spectra add into hist. */
static int count_kmers_multi(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_bases, int k, dnagpu_stats *stats,
                             dnagpu_table **table, uint32_t max_count = 0, uint64_t *hist = nullptr)
{
    const int G = 1 + (int)ctx->peers.size();
    std::vector<dnagpu_ctx *> cx(1, ctx);
    cx.insert(cx.end(), ctx->peers.begin(), ctx->peers.end());
    const uint64_t n_words = words_of(n_bases);
    const uint64_t per = ((n_bases + G - 1) / G + 31) / 32 * 32, end = (n_bases + 31) / 32 * 32;
    std::vector<uint64_t> first(G), starts(G);
    for (int d = 0; d < G; ++d) {
        first[d] = std::min<uint64_t>((uint64_t)d * per, end);
        starts[d] = n_bases > first[d] ? std::min(per, n_bases - first[d]) : 0;
        /* the piece: its bases + the 31-base overlap, >= 1 zero pad word, an even number of words */
        const uint64_t held = std::min(n_bases, first[d] + starts[d] + 31) - std::min(n_bases, first[d]);
        const uint64_t w_copy = std::min(words_of(held), n_words - std::min(n_words, first[d] / 32));
        const uint64_t w_alloc = (words_of(held) + 3) & ~1ull;
        CU(ctx, cudaSetDevice(cx[d]->device));
        if (ctx->shard_cap[d] < w_alloc) {
            if (ctx->shard_buf[d]) cudaFree(ctx->shard_buf[d]);
            ctx->shard_buf[d] = nullptr;
            ctx->shard_cap[d] = 0;
            cudaError_t e = cudaMalloc((void **)&ctx->shard_buf[d], w_alloc * 8);
            if (e != cudaSuccess) {
                cudaGetLastError();
                return fail(ctx, DNAGPU_ENOMEM, "shard of %llu bytes on GPU %d: %s", (unsigned long long)(w_alloc * 8),
                            cx[d]->device, cudaGetErrorString(e));
            }
            ctx->shard_cap[d] = w_alloc;
        }
        if (w_copy)
            CU(ctx, cudaMemcpyAsync(ctx->shard_buf[d], words + first[d] / 32, w_copy * 8, cudaMemcpyHostToDevice, cx[d]->stream));
        CU(ctx, cudaMemsetAsync(ctx->shard_buf[d] + w_copy, 0, (w_alloc - w_copy) * 8, cx[d]->stream));
    }
    for (int d = 0; d < G; ++d) { /* every shard must be resident before anybody reads it */
        CU(ctx, cudaSetDevice(cx[d]->device));
        CU(ctx, cudaStreamSynchronize(cx[d]->stream));
    }
    std::vector<int> rc((size_t)G, DNAGPU_OK);
    std::vector<dnagpu_stats> st((size_t)G);
    std::vector<dnagpu_table *> tb((size_t)G, nullptr);
    std::vector<std::vector<uint64_t>> hs((size_t)G, std::vector<uint64_t>(max_count));
    std::vector<std::thread> th;
    for (int d = 0; d < G; ++d)
        th.emplace_back([&, d] {
            cudaSetDevice(cx[d]->device);
            const void *ptr[kMaxPieces];
            uint64_t fb[kMaxPieces], ns[kMaxPieces];
            for (int i = 0; i < G; ++i) {
                const int p = (d + i) % G;
                ptr[i] = ctx->shard_buf[p];
                fb[i] = first[p];
                ns[i] = starts[p];
            }
            dnagpu_seq *seq = nullptr;
            rc[d] = dnagpu_seq_wrap_pieces(cx[d], ptr, fb, ns, (uint32_t)G, n_bases, &seq);
            if (rc[d] != DNAGPU_OK) return;
            dnagpu_count_opts o = {DNAGPU_COUNT_AUTO, 0, 0.0, 0, (uint32_t)G, (uint32_t)d};
            rc[d] = max_count ? dnagpu_count_spectrum(cx[d], seq, k, nullptr, &o, max_count, hs[d].data(), &st[d])
                              : dnagpu_count(cx[d], seq, k, nullptr, &o, &st[d], table ? &tb[d] : nullptr);
            dnagpu_seq_free(seq);
        });
    for (auto &t : th) t.join();
    CU(ctx, cudaSetDevice(ctx->device));
    for (int d = 0; d < G; ++d)
        if (rc[d] != DNAGPU_OK) {
            for (dnagpu_table *t : tb) dnagpu_table_free(t);
            return fail(ctx, rc[d], "GPU %d: %s", cx[d]->device, dnagpu_last_error(cx[d]));
        }
    stats->total = stats->distinct = stats->unique = 0;
    for (int d = 0; d < G; ++d) {
        stats->total += st[d].total;
        stats->distinct += st[d].distinct;
        stats->unique += st[d].unique;
    }
    if (max_count) {
        std::fill(hist, hist + max_count, 0);
        for (int d = 0; d < G; ++d)
            for (uint32_t c = 0; c < max_count; ++c) hist[c] += hs[d][c];
    }
    if (table) {
        dnagpu_table *t = new (std::nothrow) dnagpu_table();
        if (!t) {
            for (dnagpu_table *p : tb) dnagpu_table_free(p);
            return fail(ctx, DNAGPU_ENOMEM, "out of host memory");
        }
        t->ctx = ctx;
        ctx->tables.insert(t);
        t->k = k;
        t->rows = stats->distinct;
        t->parts = tb;
        *table = t;
    }
    return DNAGPU_OK;
}

extern "C" int dnagpu_count_kmers(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_bases, int k,
                                  const dnagpu_where *filter, dnagpu_stats *stats,
                                  dnagpu_table **table)
{
    if (!ctx) return fail(ctx, DNAGPU_EARG, "dnagpu_count_kmers: NULL ctx");
    TRY(check_k(ctx, k));
    TRY(check_filter_literals(ctx, filter));
    if (!ctx->peers.empty() && words && (!filter || (filter->prefix_len == 0 && !filter->qkmer)) &&
        rows_of(n_bases, k) >= (1ull << 21)) { /* smaller inputs are not worth the fan-out */
        dnagpu_stats local;
        if (table) *table = nullptr;
        return count_kmers_multi(ctx, words, n_bases, k, stats ? stats : &local, table);
    }
    if (words && (!filter || (filter->prefix_len == 0 && !filter->qkmer))) {
        dnagpu_stats local;
        bool done = false;
        if (table) *table = nullptr;
        TRY(count_kmers_pipelined(ctx, words, n_bases, k, stats ? stats : &local, table, &done));
        if (done) return DNAGPU_OK;
    }
    dnagpu_seq *seq = nullptr;
    TRY(dnagpu_seq_upload(ctx, words, n_bases, &seq));
    int rc = dnagpu_count(ctx, seq, k, filter, nullptr, stats, table);
    dnagpu_seq_free(seq);
    return rc;
}

extern "C" int dnagpu_count_kmers_spectrum(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_bases, int k,
                                           const dnagpu_where *filter, uint32_t max_count, uint64_t *hist,
                                           dnagpu_stats *stats)
{
    if (!ctx || !hist) return fail(ctx, DNAGPU_EARG, "dnagpu_count_kmers_spectrum: NULL argument");
    if (max_count < 1 || max_count > kSpecMaxCount)
        return fail(ctx, DNAGPU_EARG, "max_count must be between 1 and %u", kSpecMaxCount);
    TRY(check_k(ctx, k));
    TRY(check_filter_literals(ctx, filter));
    if (!ctx->peers.empty() && words && (!filter || (filter->prefix_len == 0 && !filter->qkmer)) &&
        rows_of(n_bases, k) >= (1ull << 21)) { /* the same fan-out rule as dnagpu_count_kmers */
        dnagpu_stats local;
        return count_kmers_multi(ctx, words, n_bases, k, stats ? stats : &local, nullptr, max_count, hist);
    }
    dnagpu_seq *seq = nullptr;
    TRY(dnagpu_seq_upload(ctx, words, n_bases, &seq));
    int rc = dnagpu_count_spectrum(ctx, seq, k, filter, nullptr, max_count, hist, stats);
    dnagpu_seq_free(seq);
    return rc;
}

/* Host reads + a WHERE clause: the upload goes in chunks on the copy stream while the predicate scan of the
 * previous chunk appends its matches to the key list; the list is counted at the end.  If the list overflows
 * its guess (a clause that keeps more than 1/8 of the rows) the query is redone on the resident words. */
static int count_reads_pipelined(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_reads, uint32_t bases_per_read,
                                 uint32_t stride_words, int k, const dnagpu_where *filter, dnagpu_stats *stats,
                                 dnagpu_table **table, bool *done)
{
    *done = false;
    const uint64_t rows_per_read = rows_of(bases_per_read, k), n = n_reads * rows_per_read;
    if (!words || n < (1ull << 24) || stride_words < words_of(bases_per_read) ||
        pick_method(nullptr, k, n) == DNAGPU_COUNT_DENSE)
        return DNAGPU_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    Pred p;
    bool active = false;
    TRY(build_pred(ctx, filter, k, n, &p, &active));
    if (!active) return DNAGPU_OK;
    if (!ctx->copy_stream) CU(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    Scratch sc(ctx);
    const uint64_t n_words = n_reads * stride_words, alloc_words = (n_words + 3) & ~1ull;
    const uint64_t cap = std::max<uint64_t>(1ull << 20, n / 8);
    uint64_t *d_words, *keys;
    TRY(sc.get((void **)&d_words, alloc_words * 8));
    TRY(sc.get((void **)&keys, (cap + 2) * 8));
    CU(ctx, cudaMemsetAsync(d_words + n_words, 0, (alloc_words - n_words) * 8, ctx->stream));
    TRY(zero_counters(ctx));
    CU(ctx, cudaStreamSynchronize(ctx->stream)); /* d_words exists before the copy stream writes it */
    const int n_chunks = 8;
    const uint64_t chunk_reads = (n_reads + n_chunks - 1) / n_chunks;
    std::vector<cudaEvent_t> ev;
    int rc = DNAGPU_OK;
    for (uint64_t r0 = 0; r0 < n_reads && rc == DNAGPU_OK; r0 += chunk_reads) {
        const uint64_t r1 = std::min(n_reads, r0 + chunk_reads);
        rc = chunk_copy(ctx, ev, d_words + r0 * stride_words, words + r0 * stride_words, (r1 - r0) * stride_words * 8);
        if (rc != DNAGPU_OK) break;
        SeqView v;
        memset(&v, 0, sizeof v);
        v.words = d_words + r0 * stride_words;
        v.n_seqs = r1 - r0;
        v.stride = stride_words;
        v.rows_per_seq = rows_per_read;
        v.items_per_seq = (rows_per_read + 31) / 32;
        v.n_rows = v.rows_per_seq * v.n_seqs;
        v.n_items = v.items_per_seq * v.n_seqs;
        if (v.n_rows) rc = collect_launch(ctx, kFixed, v, p, k, keys, cap);
    }
    uint64_t n_match = 0;
    if (rc == DNAGPU_OK) rc = read_u64(ctx, (const uint64_t *)(ctx->d_ctr + C_CURSOR), &n_match);
    /* on every path: the copy stream must be done with d_words before Scratch hands it back to the pool */
    cudaStreamSynchronize(ctx->copy_stream);
    if (rc != DNAGPU_OK) cudaStreamSynchronize(ctx->stream);
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
    TRY(rc);
    if (n_match > cap) { /* not selective after all: the ordinary path, on the words that are resident now */
        dnagpu_seq *seq = nullptr;
        TRY(dnagpu_seq_wrap_reads(ctx, d_words, n_reads, bases_per_read, stride_words, alloc_words, &seq));
        rc = dnagpu_count(ctx, seq, k, filter, nullptr, stats, table);
        dnagpu_seq_free(seq);
        TRY(rc);
    } else if (n_match == 0) {
        stats->total = stats->distinct = stats->unique = 0;
        if (table) TRY(table_new(ctx, k, 0, table));
    } else {
        TRY(count_listed(ctx, keys, n_match, k, nullptr, stats, table));
    }
    *done = true;
    return DNAGPU_OK;
}

extern "C" int dnagpu_count_reads(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_reads,
                                  uint32_t bases_per_read, uint32_t stride_words, int k,
                                  const dnagpu_where *filter, dnagpu_stats *stats,
                                  dnagpu_table **table)
{
    if (!ctx) return fail(ctx, DNAGPU_EARG, "dnagpu_count_reads: NULL ctx");
    TRY(check_k(ctx, k));
    TRY(check_filter_literals(ctx, filter));
    if (stats && filter) {
        if (table) *table = nullptr;
        bool done = false;
        TRY(count_reads_pipelined(ctx, words, n_reads, bases_per_read, stride_words, k, filter, stats, table, &done));
        if (done) return DNAGPU_OK;
    }
    dnagpu_seq *seq = nullptr;
    TRY(dnagpu_seq_upload_reads(ctx, words, n_reads, bases_per_read, stride_words, &seq));
    int rc = dnagpu_count(ctx, seq, k, filter, nullptr, stats, table);
    dnagpu_seq_free(seq);
    return rc;
}

/* ---- the grouped result -------------------------------------------------------------------- */
extern "C" uint64_t dnagpu_table_rows(const dnagpu_table *t) { return t ? t->rows : 0; }

/* rows [offset, offset + n) of a multi-GPU table: walk the per-GPU tables */
static int table_fetch_parts(dnagpu_ctx *ctx, const dnagpu_table *t, uint64_t offset, uint64_t n, uint64_t *kmers,
                             uint64_t *counts)
{
    uint64_t base = 0;
    for (const dnagpu_table *p : t->parts) {
        if (n == 0) break;
        if (offset < base + p->rows) {
            const uint64_t o = offset - base, m = std::min(n, p->rows - o);
            int rc = dnagpu_table_fetch(p->ctx, p, o, m, kmers, counts);
            if (rc != DNAGPU_OK) return fail(ctx, rc, "%s", dnagpu_last_error(p->ctx));
            offset += m;
            n -= m;
            if (kmers) kmers += m;
            if (counts) counts += m;
        }
        base += p->rows;
    }
    CU(ctx, cudaSetDevice(ctx->device));
    return DNAGPU_OK;
}
extern "C" int dnagpu_table_k(const dnagpu_table *t) { return t ? t->k : 0; }

extern "C" int dnagpu_table_fetch(dnagpu_ctx *ctx, const dnagpu_table *t, uint64_t offset,
                                  uint64_t n, uint64_t *kmers, uint64_t *counts)
{
    if (!ctx || !t) return fail(ctx, DNAGPU_EARG, "dnagpu_table_fetch: NULL argument");
    CHECK_OWNED(ctx, t, "the table");
    if (offset > t->rows || n > t->rows - offset) return fail(ctx, DNAGPU_EARG, "row range outside the table");
    if (!t->parts.empty()) return table_fetch_parts(ctx, t, offset, n, kmers, counts);
    CU(ctx, cudaSetDevice(ctx->device));
    if (n && kmers) CU(ctx, cudaMemcpyAsync(kmers, t->d_kmers + offset, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (n && counts) CU(ctx, cudaMemcpyAsync(counts, t->d_counts + offset, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return DNAGPU_OK;
}

extern "C" int dnagpu_table_device(const dnagpu_table *t, const uint64_t **d_kmers,
                                   const uint64_t **d_counts)
{
    if (!t) return fail(nullptr, DNAGPU_EARG, "table is NULL");
    if (!t->parts.empty()) return fail(t->ctx, DNAGPU_EARG, "the rows of a multi-GPU table live on several GPUs: use dnagpu_table_fetch");
    if (d_kmers) *d_kmers = t->d_kmers;
    if (d_counts) *d_counts = t->d_counts;
    return DNAGPU_OK;
}

static void table_release(dnagpu_table *t)
{
    if (!t->ctx) return;
    for (dnagpu_table *p : t->parts) dnagpu_table_free(p); /* the peers' contexts are still alive here */
    t->parts.clear();
    cudaSetDevice(t->ctx->device);
    dfree(t->ctx, t->d_kmers);
    dfree(t->ctx, t->d_counts);
    t->d_kmers = t->d_counts = nullptr;
    t->ctx = nullptr;
}

extern "C" void dnagpu_table_free(dnagpu_table *t)
{
    if (!t) return;
    if (t->ctx) {
        t->ctx->tables.erase(t);
        table_release(t);
    }
    delete t;
}

/* ---- owner routing --------------------------------------------------------------------------- */
extern "C" uint32_t dnagpu_owner_of(uint64_t kmer, uint32_t n_parts)
{
    return owner_of(kmer, n_parts ? n_parts : 1);
}

extern "C" int dnagpu_partition(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k,
                                const dnagpu_where *filter, uint32_t n_parts, uint64_t *d_out,
                                uint64_t cap, uint64_t *part_counts)
{
    if (!ctx || !seq || !part_counts) return fail(ctx, DNAGPU_EARG, "dnagpu_partition: NULL argument");
    if (n_parts < 1 || n_parts > (uint32_t)kMaxParts)
        return fail(ctx, DNAGPU_EARG, "n_parts must be between 1 and %d", kMaxParts);
    TRY(check_k(ctx, k));
    TRY(check_filter_literals(ctx, filter));
    CU(ctx, cudaSetDevice(ctx->device));
    SeqView v;
    TRY(make_view(ctx, seq, k, &v));
    Pred p;
    bool active;
    TRY(build_pred(ctx, filter, k, v.n_rows, &p, &active));
    for (uint32_t i = 0; i < n_parts; ++i) part_counts[i] = 0;
    if (v.n_rows == 0) return DNAGPU_OK;
    const uint64_t mask = kmer_mask(k);
    unsigned long long *d_cnt = ctx->d_ctr + C_COUNT, *d_cur = ctx->d_ctr + C_COUNT + kMaxParts;
    TRY(zero_counters(ctx));
    const unsigned pgrid = (unsigned)std::min<uint64_t>(grid_for(v.n_items, kThreads), (uint64_t)ctx->sm_count * 16);
    DISPATCH_LAYOUT(seq->layout, TRY(launch(ctx, "partition_count", [&] {
        if (active)
            k_partition_count<LY, true><<<pgrid, kThreads, 0, ctx->stream>>>(v, p, mask, n_parts, d_cnt);
        else
            k_partition_count<LY, false><<<pgrid, kThreads, 0, ctx->stream>>>(v, p, mask, n_parts, d_cnt);
    })));
    TRY(fetch_counters(ctx));
    uint64_t total = 0;
    uint64_t offs[kMaxParts];
    for (uint32_t i = 0; i < n_parts; ++i) {
        part_counts[i] = ctx->h_ctr[C_COUNT + i];
        offs[i] = total;
        total += part_counts[i];
    }
    if (!d_out) return DNAGPU_OK;
    if (cap < total)
        return fail(ctx, DNAGPU_ECAPACITY, "partition needs room for %llu rows", (unsigned long long)total);
    if (total == 0) return DNAGPU_OK;
    Scratch sc(ctx);
    uint64_t *d_off;
    TRY(sc.get((void **)&d_off, kMaxParts * 8));
    memcpy(ctx->h_ctr, offs, n_parts * 8); /* pinned staging */
    CU(ctx, cudaMemcpyAsync(d_off, ctx->h_ctr, n_parts * 8, cudaMemcpyHostToDevice, ctx->stream));
    const unsigned grid = grid_for(v.n_items, kThreads);
    const int smem = kThreads * 32 * (int)sizeof(uint64_t);
    DISPATCH_LAYOUT(seq->layout, TRY(launch(ctx, "partition_write", [&] {
        if (active)
            k_partition_write<LY, true><<<grid, kThreads, smem, ctx->stream>>>(v, p, mask, n_parts, d_off, d_cur, d_out);
        else
            k_partition_write<LY, false><<<grid, kThreads, smem, ctx->stream>>>(v, p, mask, n_parts, d_off, d_cur, d_out);
    })));
    CU(ctx, cudaStreamSynchronize(ctx->stream)); /* h_ctr staging is reused by the next call */
    return DNAGPU_OK;
}

/* ---- multi-GPU GROUP BY with the owner routing fused into partition level 1 ---------------------- */
extern "C" int dnagpu_shuffle_plan_make(uint64_t n_rows_total, uint32_t n_parts, dnagpu_shuffle_plan *plan)
{
    if (!plan || n_parts < 1 || n_parts > (uint32_t)kMaxParts)
        return fail(nullptr, DNAGPU_EARG, "dnagpu_shuffle_plan_make: bad arguments");
    int b1, b2;
    plan_bits(n_rows_total, n_parts, &b1, &b2);
    plan->bits1 = b1;
    plan->bits2 = b2;
    plan->n_parts = n_parts;
    plan->n_digits = 1u << b1;
    return DNAGPU_OK;
}

extern "C" uint32_t dnagpu_shuffle_owner(const dnagpu_shuffle_plan *plan, uint32_t digit)
{
    return (uint32_t)(((uint64_t)digit * plan->n_parts) >> plan->bits1);
}

extern "C" int dnagpu_shuffle_send(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k, const dnagpu_where *filter,
                                   const dnagpu_shuffle_plan *plan, uint64_t *d_out, uint64_t cap,
                                   uint64_t *digit_counts, uint64_t *rows_kept, uint64_t *side_rows)
{
    if (!ctx || !seq || !plan || !d_out || !digit_counts)
        return fail(ctx, DNAGPU_EARG, "dnagpu_shuffle_send: NULL argument");
    TRY(check_k(ctx, k));
    TRY(check_filter_literals(ctx, filter));
    CU(ctx, cudaSetDevice(ctx->device));
    CountInput in;
    in.seq = seq;
    TRY(make_view(ctx, seq, k, &in.v));
    in.n = in.v.n_rows;
    TRY(build_pred(ctx, filter, k, in.n, &in.p, &in.filtered));
    for (uint32_t d = 0; d < plan->n_digits; ++d) digit_counts[d] = 0;
    if (rows_kept) *rows_kept = 0;
    if (side_rows) *side_rows = 0;
    if (in.n == 0) return DNAGPU_OK;
    Scratch sc(ctx);
    TRY(zero_counters(ctx));
    uint64_t *off1, n = 0, *keys = d_out;
    TRY(part_level1(ctx, sc, in, k, plan->bits1, &keys, cap, &off1, &n));
    std::vector<uint64_t> off((size_t)plan->n_digits + 1);
    CU(ctx, cudaMemcpyAsync(off.data(), off1, off.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    TRY(fetch_counters(ctx)); /* synchronises the stream */
    for (uint32_t d = 0; d < plan->n_digits; ++d) digit_counts[d] = off[d + 1] - off[d];
    if (rows_kept) *rows_kept = ctx->h_ctr[C_TOTAL];
    if (side_rows) *side_rows = ctx->h_ctr[C_SIDE];
    return DNAGPU_OK;
}

extern "C" int dnagpu_shuffle_count(dnagpu_ctx *ctx, const uint64_t *d_keys, const uint64_t *piece_counts,
                                    uint32_t n_pieces, uint32_t n_groups, const dnagpu_shuffle_plan *plan, int k,
                                    dnagpu_stats *stats, dnagpu_table **table)
{
    if (!ctx || !plan || !piece_counts || !stats || n_groups == 0 || n_pieces % n_groups)
        return fail(ctx, DNAGPU_EARG, "dnagpu_shuffle_count: bad arguments");
    TRY(check_k(ctx, k));
    CU(ctx, cudaSetDevice(ctx->device));
    stats->total = stats->distinct = stats->unique = 0;
    if (table) *table = nullptr;
    std::vector<uint64_t> off((size_t)n_pieces + 1, 0);
    for (uint32_t i = 0; i < n_pieces; ++i) off[i + 1] = off[i] + piece_counts[i];
    const uint64_t n = off[n_pieces];
    if (n == 0) {
        if (table) TRY(table_new(ctx, k, 0, table));
        return DNAGPU_OK;
    }
    if (!d_keys) return fail(ctx, DNAGPU_EARG, "dnagpu_shuffle_count: d_keys is NULL");
    Scratch sc(ctx);
    uint64_t *d_off;
    TRY(sc.get((void **)&d_off, off.size() * 8));
    CU(ctx, cudaMemcpyAsync(d_off, off.data(), off.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream)); /* `off` is a host temporary */
    TRY(zero_counters(ctx));
    return free_table_on_error(part_finish(ctx, sc, d_keys, n, d_off, d_off + 1, n_pieces, n_groups, plan->bits1, plan->bits2,
                                           k, stats, n, table),
                               table);
}

/* ---- the exchange fused into the scatter kernel: stores straight into peer memory ---------------- */
extern "C" int dnagpu_peer_alloc(dnagpu_ctx *ctx, uint64_t bytes, void **d_ptr, unsigned char handle[64])
{
    if (!ctx || !d_ptr || !handle) return fail(ctx, DNAGPU_EARG, "dnagpu_peer_alloc: NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CU(ctx, cudaSetDevice(ctx->device));
    *d_ptr = nullptr;
    cudaError_t e = cudaMalloc(d_ptr, bytes ? bytes : 16); /* IPC needs a plain allocation, not the pool */
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, DNAGPU_ENOMEM, "peer allocation of %llu bytes failed: %s", (unsigned long long)bytes,
                    cudaGetErrorString(e));
    }
    cudaIpcMemHandle_t h;
    e = cudaIpcGetMemHandle(&h, *d_ptr);
    if (e != cudaSuccess) {
        cudaFree(*d_ptr);
        *d_ptr = nullptr;
        cudaGetLastError();
        return fail(ctx, DNAGPU_ECUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e));
    }
    memcpy(handle, &h, 64);
    return DNAGPU_OK;
}

extern "C" int dnagpu_peer_open(dnagpu_ctx *ctx, const unsigned char handle[64], void **d_ptr)
{
    if (!ctx || !d_ptr || !handle) return fail(ctx, DNAGPU_EARG, "dnagpu_peer_open: NULL argument");
    CU(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    cudaError_t e = cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, DNAGPU_ECUDA, "cudaIpcOpenMemHandle: %s (is peer access available between the GPUs?)",
                    cudaGetErrorString(e));
    }
    return DNAGPU_OK;
}

extern "C" int dnagpu_peer_close(dnagpu_ctx *ctx, void *d_ptr)
{
    if (!ctx) return fail(ctx, DNAGPU_EARG, "ctx is NULL");
    CU(ctx, cudaSetDevice(ctx->device));
    if (d_ptr) CU(ctx, cudaIpcCloseMemHandle(d_ptr));
    return DNAGPU_OK;
}

extern "C" int dnagpu_peer_free(dnagpu_ctx *ctx, void *d_ptr)
{
    if (!ctx) return fail(ctx, DNAGPU_EARG, "ctx is NULL");
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    if (d_ptr) CU(ctx, cudaFree(d_ptr));
    return DNAGPU_OK;
}

/* shared front end of the two fused-exchange calls */
static int shuffle_input(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k, const dnagpu_where *filter, CountInput *in)
{
    TRY(check_k(ctx, k));
    TRY(check_filter_literals(ctx, filter));
    CU(ctx, cudaSetDevice(ctx->device));
    in->seq = seq;
    TRY(make_view(ctx, seq, k, &in->v));
    in->n = in->v.n_rows;
    return build_pred(ctx, filter, k, in->n, &in->p, &in->filtered);
}

/* keys per digit of level 1 (host array of plan->n_digits entries) of a sequence or a key list */
static int shuffle_hist(dnagpu_ctx *ctx, const CountInput &in, int k, const dnagpu_shuffle_plan *plan, uint64_t *digit_counts)
{
    const uint32_t P1 = plan->n_digits;
    for (uint32_t d = 0; d < P1; ++d) digit_counts[d] = 0;
    if (in.n == 0) return DNAGPU_OK;
    Scratch sc(ctx);
    unsigned long long *hist1;
    uint64_t *root = nullptr;
    TRY(sc.get((void **)&hist1, (uint64_t)P1 * 8));
    CU(ctx, cudaMemsetAsync(hist1, 0, (uint64_t)P1 * 8, ctx->stream));
    if (in.d_keys) TRY(root_range(ctx, sc, in.n, &root));
    TRY(l1_hist(ctx, sc, in, k, plan->bits1, root, hist1));
    CU(ctx, cudaMemcpyAsync(digit_counts, hist1, (uint64_t)P1 * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return DNAGPU_OK;
}

extern "C" int dnagpu_shuffle_hist(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k, const dnagpu_where *filter,
                                   const dnagpu_shuffle_plan *plan, uint64_t *digit_counts)
{
    if (!ctx || !seq || !plan || !digit_counts) return fail(ctx, DNAGPU_EARG, "dnagpu_shuffle_hist: NULL argument");
    CountInput in;
    TRY(shuffle_input(ctx, seq, k, filter, &in));
    return shuffle_hist(ctx, in, k, plan, digit_counts);
}

/* The scatter kernels add "index of the run" to a base pointer; with a NULL base and addresses / 8 as indices the
 * same kernels store to arbitrary (peer) destinations per digit.  -> that index table and a zeroed cursor per digit. */
static int peer_dest(dnagpu_ctx *ctx, Scratch &sc, const dnagpu_shuffle_plan *plan, const uint64_t *digit_dest,
                     uint64_t **d_idx, unsigned long long **cur1)
{
    const uint32_t P1 = plan->n_digits;
    std::vector<uint64_t> idx(P1);
    for (uint32_t d = 0; d < P1; ++d) {
        if (digit_dest[d] & 7) return fail(ctx, DNAGPU_EARG, "destination of digit %u is not 8-byte aligned", d);
        idx[d] = digit_dest[d] >> 3;
    }
    TRY(sc.get((void **)d_idx, ((uint64_t)P1 + 1) * 8));
    TRY(sc.get((void **)cur1, (uint64_t)P1 * 8));
    CU(ctx, cudaMemcpyAsync(*d_idx, idx.data(), (uint64_t)P1 * 8, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemsetAsync(*cur1, 0, (uint64_t)P1 * 8, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream)); /* idx is a host temporary */
    return DNAGPU_OK;
}

extern "C" int dnagpu_shuffle_scatter_to(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k, const dnagpu_where *filter,
                                         const dnagpu_shuffle_plan *plan, const uint64_t *digit_dest,
                                         uint64_t *rows_kept, uint64_t *side_rows)
{
    if (!ctx || !seq || !plan || !digit_dest)
        return fail(ctx, DNAGPU_EARG, "dnagpu_shuffle_scatter_to: NULL argument");
    CountInput in;
    TRY(shuffle_input(ctx, seq, k, filter, &in));
    if (rows_kept) *rows_kept = 0;
    if (side_rows) *side_rows = 0;
    if (in.n == 0) return DNAGPU_OK;
    Scratch sc(ctx);
    uint64_t *d_idx;
    unsigned long long *cur1;
    TRY(peer_dest(ctx, sc, plan, digit_dest, &d_idx, &cur1));
    TRY(zero_counters(ctx));
    TRY(l1_scatter_seq(ctx, seq->layout, in.v, in.p, in.filtered, k, plan->bits1, d_idx, cur1, nullptr, 0));
    TRY(fetch_counters(ctx)); /* synchronises: every store of this rank has been issued and retired */
    if (rows_kept) *rows_kept = ctx->h_ctr[C_TOTAL];
    if (side_rows) *side_rows = ctx->h_ctr[C_SIDE];
    return DNAGPU_OK;
}

/* the same two steps from a key list on the device */
extern "C" int dnagpu_shuffle_hist_keys(dnagpu_ctx *ctx, const uint64_t *d_keys, uint64_t n,
                                        const dnagpu_shuffle_plan *plan, uint64_t *digit_counts)
{
    if (!ctx || !plan || !digit_counts || (n && !d_keys))
        return fail(ctx, DNAGPU_EARG, "dnagpu_shuffle_hist_keys: NULL argument");
    CU(ctx, cudaSetDevice(ctx->device));
    CountInput in;
    in.d_keys = d_keys;
    in.n = n;
    return shuffle_hist(ctx, in, 0, plan, digit_counts);
}

extern "C" int dnagpu_shuffle_scatter_keys_to(dnagpu_ctx *ctx, const uint64_t *d_keys, uint64_t n,
                                              const dnagpu_shuffle_plan *plan, const uint64_t *digit_dest,
                                              uint64_t *side_rows)
{
    if (!ctx || !plan || !digit_dest || (n && !d_keys))
        return fail(ctx, DNAGPU_EARG, "dnagpu_shuffle_scatter_keys_to: NULL argument");
    CU(ctx, cudaSetDevice(ctx->device));
    if (side_rows) *side_rows = 0;
    if (n == 0) return DNAGPU_OK;
    Scratch sc(ctx);
    uint64_t *d_idx, *root;
    unsigned long long *cur1;
    TRY(peer_dest(ctx, sc, plan, digit_dest, &d_idx, &cur1));
    TRY(root_range(ctx, sc, n, &root));
    TRY(zero_counters(ctx));
    TRY(l1_scatter_keys(ctx, sc, d_keys, n, root, true, plan->bits1, d_idx, cur1, nullptr, 0));
    TRY(fetch_counters(ctx)); /* synchronises: every store of this rank has been issued and retired */
    if (side_rows) *side_rows = ctx->h_ctr[C_SIDE];
    return DNAGPU_OK;
}

/* ---- sorted k-mer index (the SP-GiST replacement) ------------------------------------------------ */
/* Stable LSD radix sort of n (key, value) pairs over key bits [0, bits).  a* hold the input, b* are
 * scratch of the same size; *in_a tells where the result is.  vals may be NULL (keys only). */
static int radix_sort(dnagpu_ctx *ctx, Scratch &sc, uint64_t *ak, uint64_t *av, uint64_t *bk, uint64_t *bv, uint64_t n,
                      int bits, bool *in_a)
{
    *in_a = true;
    if (n < 2 || bits <= 0) return DNAGPU_OK;
    const uint64_t chunks = (n + kSortChunk - 1) / kSortChunk;
    const unsigned grid = (unsigned)std::min<uint64_t>(chunks, (uint64_t)ctx->sm_count * 4);
    const uint64_t per_cta = (chunks + grid - 1) / grid * kSortChunk;
    uint64_t *cnt, *off;
    TRY(sc.get((void **)&cnt, 256ull * grid * 8));
    TRY(sc.get((void **)&off, (256ull * grid + 1) * 8));
    for (int shift = 0; shift < bits; shift += 8) {
        const uint64_t *src_k = *in_a ? ak : bk, *src_v = *in_a ? av : bv;
        uint64_t *dst_k = *in_a ? bk : ak, *dst_v = *in_a ? bv : av;
        TRY(launch(ctx, "sort_hist", [&] { k_sort_hist<<<grid, kSortThreads, 0, ctx->stream>>>(src_k, n, per_cta, shift, cnt); }));
        TRY(scan_any(ctx, sc, cnt, 256ull * grid, off));
        TRY(launch(ctx, "sort_scatter", [&] {
            if (av)
                k_sort_scatter<true><<<grid, kSortThreads, sizeof(SortSmem), ctx->stream>>>(src_k, src_v, n, per_cta, shift, off,
                                                                                          dst_k, dst_v);
            else
                k_sort_scatter<false><<<grid, kSortThreads, sizeof(SortSmem), ctx->stream>>>(src_k, nullptr, n, per_cta, shift,
                                                                                           off, dst_k, nullptr);
        }));
        *in_a = !*in_a;
    }
    return DNAGPU_OK;
}

extern "C" int dnagpu_index_build(dnagpu_ctx *ctx, const uint64_t *d_keys, uint64_t n, int k, dnagpu_index **index)
{
    if (!ctx || !index || (n && !d_keys)) return fail(ctx, DNAGPU_EARG, "dnagpu_index_build: NULL argument");
    *index = nullptr;
    TRY(check_k(ctx, k));
    CU(ctx, cudaSetDevice(ctx->device));
    dnagpu_index *ix = new (std::nothrow) dnagpu_index;
    if (!ix) return fail(ctx, DNAGPU_ENOMEM, "out of host memory");
    ix->ctx = ctx;
    ctx->indexes.insert(ix);
    ix->k = k;
    ix->rows = n;
    int rc = DNAGPU_OK;
    uint64_t *tk = nullptr, *tv = nullptr;
    {
        Scratch sc(ctx);
        rc = dalloc(ctx, (void **)&ix->d_skeys, (n + 2) * 8);
        if (rc == DNAGPU_OK) rc = dalloc(ctx, (void **)&ix->d_rows, (n + 2) * 8);
        if (rc == DNAGPU_OK && n) rc = dalloc(ctx, (void **)&tk, (n + 2) * 8);
        if (rc == DNAGPU_OK && n) rc = dalloc(ctx, (void **)&tv, (n + 2) * 8);
        if (rc == DNAGPU_OK && n) {
            const unsigned grid = (unsigned)std::min<uint64_t>(grid_for(n, kThreads), (uint64_t)ctx->sm_count * 16);
            rc = launch(ctx, "index_keys", [&] { k_index_keys<<<grid, kThreads, 0, ctx->stream>>>(d_keys, n, k, ix->d_skeys, ix->d_rows); });
            bool in_a = true;
            if (rc == DNAGPU_OK) rc = radix_sort(ctx, sc, ix->d_skeys, ix->d_rows, tk, tv, n, 2 * k, &in_a);
            if (rc == DNAGPU_OK && !in_a) {
                std::swap(ix->d_skeys, tk);
                std::swap(ix->d_rows, tv);
            }
        }
        if (rc == DNAGPU_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess)
            rc = fail(ctx, DNAGPU_ECUDA, "index build: %s", cudaGetErrorString(cudaGetLastError()));
    }
    dfree(ctx, tk);
    dfree(ctx, tv);
    if (rc != DNAGPU_OK) {
        dnagpu_index_free(ix);
        return rc;
    }
    *index = ix;
    return DNAGPU_OK;
}

static void index_release(dnagpu_index *ix)
{
    if (!ix->ctx) return;
    cudaSetDevice(ix->ctx->device);
    dfree(ix->ctx, ix->d_skeys);
    dfree(ix->ctx, ix->d_rows);
    ix->d_skeys = ix->d_rows = nullptr;
    ix->ctx = nullptr;
}

extern "C" void dnagpu_index_free(dnagpu_index *ix)
{
    if (!ix) return;
    if (ix->ctx) {
        ix->ctx->indexes.erase(ix);
        index_release(ix);
    }
    delete ix;
}

extern "C" uint64_t dnagpu_index_rows(const dnagpu_index *ix) { return ix ? ix->rows : 0; }
extern "C" int dnagpu_index_k(const dnagpu_index *ix) { return ix ? ix->k : 0; }

extern "C" int dnagpu_index_device(const dnagpu_index *ix, const uint64_t **d_sort_keys, const uint64_t **d_rows)
{
    if (!ix) return fail(nullptr, DNAGPU_EARG, "index is NULL");
    if (d_sort_keys) *d_sort_keys = ix->d_skeys;
    if (d_rows) *d_rows = ix->d_rows;
    return DNAGPU_OK;
}

/* positions [beg, end) of the sorted column whose sort key lies in [lo, hi] */
static int index_bounds(dnagpu_ctx *ctx, const dnagpu_index *ix, uint64_t lo, uint64_t hi, uint64_t *beg, uint64_t *end)
{
    uint64_t *d_out = (uint64_t *)(ctx->d_ctr + C_COUNT); /* two spare counters */
    TRY(launch(ctx, "index_bounds", [&] { k_index_bounds<<<1, 32, 0, ctx->stream>>>(ix->d_skeys, ix->rows, lo, hi, d_out); }));
    CU(ctx, cudaMemcpyAsync(ctx->h_ctr, d_out, 16, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    *beg = ctx->h_ctr[0];
    *end = ctx->h_ctr[1];
    return DNAGPU_OK;
}

/* hand out `n` row numbers (device, unordered unless `ordered`) in ascending order, like a bitmap heap scan */
static int index_emit(dnagpu_ctx *ctx, const dnagpu_index *ix, uint64_t *d_found, uint64_t n, bool ordered,
                      uint64_t *d_rows, uint64_t cap, uint64_t *n_out)
{
    *n_out = n;
    if (!d_rows || n == 0) return DNAGPU_OK;
    if (cap < n) return fail(ctx, DNAGPU_ECAPACITY, "index search needs room for %llu rows", (unsigned long long)n);
    if (ordered || n == 1) {
        CU(ctx, cudaMemcpyAsync(d_rows, d_found, n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    } else {
        Scratch sc(ctx);
        uint64_t *a, *b;
        TRY(sc.get((void **)&a, (n + 2) * 8));
        TRY(sc.get((void **)&b, (n + 2) * 8));
        CU(ctx, cudaMemcpyAsync(a, d_found, n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
        bool in_a = true;
        TRY(radix_sort(ctx, sc, a, nullptr, b, nullptr, n, ceil_log2(std::max<uint64_t>(ix->rows, 2)), &in_a));
        CU(ctx, cudaMemcpyAsync(d_rows, in_a ? a : b, n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return DNAGPU_OK;
}

extern "C" int dnagpu_index_equal(dnagpu_ctx *ctx, const dnagpu_index *ix, uint64_t kmer_bits, int kmer_len,
                                  uint64_t *d_rows, uint64_t cap, uint64_t *n_out)
{
    if (!ctx || !ix || !n_out) return fail(ctx, DNAGPU_EARG, "dnagpu_index_equal: NULL argument");
    CHECK_OWNED(ctx, ix, "the index");
    CU(ctx, cudaSetDevice(ctx->device));
    *n_out = 0;
    /* kmer_eq compares the lengths first (dna.c:655-668): a k-mer of another length equals no row */
    if (ix->rows == 0 || kmer_len != ix->k || (kmer_bits & ~kmer_mask(ix->k))) return DNAGPU_OK;
    const uint64_t s = sort_key_of(kmer_bits, ix->k);
    uint64_t beg, end;
    TRY(index_bounds(ctx, ix, s, s, &beg, &end));
    /* rows of one key are in input order: the sort is stable */
    return index_emit(ctx, ix, ix->d_rows + beg, end - beg, true, d_rows, cap, n_out);
}

extern "C" int dnagpu_index_search(dnagpu_ctx *ctx, const dnagpu_index *ix, const dnagpu_where *where, uint64_t *d_rows,
                                   uint64_t cap, uint64_t *n_out)
{
    if (!ctx || !ix || !n_out) return fail(ctx, DNAGPU_EARG, "dnagpu_index_search: NULL argument");
    CHECK_OWNED(ctx, ix, "the index");
    CU(ctx, cudaSetDevice(ctx->device));
    *n_out = 0;
    TRY(check_filter_literals(ctx, where));
    const int k = ix->k;
    Pred p;
    bool active = false;
    TRY(build_pred(ctx, where, k, ix->rows, &p, &active)); /* the reference's length errors, raised when a row exists */
    if (ix->rows == 0) return DNAGPU_OK;
    /* the leading positions that allow exactly one base select one range of the sorted column */
    uint64_t lead = 0;
    int n_lead = 0;
    bool rest = false; /* constraints after the leading run */
    if (active) {
        const uint64_t plane[4] = {p.ma, p.mt, p.mc, p.mg};
        bool leading = true;
        for (int j = 0; j < k; ++j) {
            int set = 0;
            for (int b = 0; b < 4; ++b) set |= (int)((plane[b] >> (2 * j)) & 1) << b;
            if (set == 0) return DNAGPU_OK; /* a position nothing can match (e.g. 'U', dna.c:1064-1086) */
            const bool one = (set & (set - 1)) == 0;
            if (leading && one) {
                const int base = set == 1 ? 0 : set == 2 ? 1 : set == 4 ? 2 : 3;
                lead = (lead << 2) | (uint64_t)base;
                ++n_lead;
            } else {
                leading = false;
                if (set != 15) rest = true;
            }
        }
    }
    const int free_bits = 2 * (k - n_lead);
    const uint64_t lo = free_bits >= 64 ? 0 : lead << free_bits;
    const uint64_t hi = free_bits >= 64 ? ~0ull : lo | (free_bits ? ((1ull << free_bits) - 1) : 0);
    uint64_t beg = 0, end = ix->rows;
    if (n_lead) TRY(index_bounds(ctx, ix, lo, hi, &beg, &end));
    if (end == beg) return DNAGPU_OK;
    if (!rest) return index_emit(ctx, ix, ix->d_rows + beg, end - beg, n_lead == k, d_rows, cap, n_out);
    /* remaining positions: evaluate the predicate on the range only */
    Scratch sc(ctx);
    uint64_t found_cap = d_rows ? std::min<uint64_t>(end - beg, std::max<uint64_t>(cap, 1)) : 0, *found = nullptr, n_found = 0;
    TRY(sc.get((void **)&found, (found_cap + 2) * 8));
    TRY(zero_counters(ctx));
    const unsigned grid = (unsigned)std::min<uint64_t>(grid_for(end - beg, kThreads), (uint64_t)ctx->sm_count * 16);
    TRY(launch(ctx, "index_match", [&] {
        k_index_match<<<grid, kThreads, 0, ctx->stream>>>(ix->d_skeys, ix->d_rows, beg, end, k, p, found_cap,
                                                        ctx->d_ctr + C_CURSOR, found);
    }));
    TRY(read_u64(ctx, (const uint64_t *)(ctx->d_ctr + C_CURSOR), &n_found));
    if (d_rows && n_found > found_cap) {
        *n_out = n_found;
        return fail(ctx, DNAGPU_ECAPACITY, "index search needs room for %llu rows", (unsigned long long)n_found);
    }
    return index_emit(ctx, ix, found, n_found, false, d_rows, cap, n_out);
}

/* ---- profiling --------------------------------------------------------------------------------- */
extern "C" int dnagpu_profile_enable(dnagpu_ctx *ctx, int on)
{
    if (!ctx) return fail(nullptr, DNAGPU_EARG, "ctx is NULL");
    ctx->profiling = on != 0;
    return DNAGPU_OK;
}

extern "C" int dnagpu_profile_reset(dnagpu_ctx *ctx)
{
    if (!ctx) return fail(nullptr, DNAGPU_EARG, "ctx is NULL");
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    for (auto &r : ctx->prof) {
        cudaEventDestroy(r.e0);
        cudaEventDestroy(r.e1);
    }
    ctx->prof.clear();
    return DNAGPU_OK;
}

extern "C" int dnagpu_profile_query(dnagpu_ctx *ctx, const char *prefix, double *total_ms,
                                    uint64_t *launches)
{
    if (!ctx) return fail(nullptr, DNAGPU_EARG, "ctx is NULL");
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    double ms = 0;
    uint64_t n = 0;
    const size_t plen = prefix ? strlen(prefix) : 0;
    for (auto &r : ctx->prof) {
        if (plen && r.name.compare(0, plen, prefix) != 0) continue;
        float t = 0;
        CU(ctx, cudaEventElapsedTime(&t, r.e0, r.e1));
        ms += t;
        n++;
    }
    if (total_ms) *total_ms = ms;
    if (launches) *launches = n;
    return DNAGPU_OK;
}

extern "C" int dnagpu_profile_dump(dnagpu_ctx *ctx, char *buf, size_t cap)
{
    if (!ctx || !buf || !cap) return fail(ctx, DNAGPU_EARG, "NULL argument");
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    std::vector<std::string> names;
    for (auto &r : ctx->prof)
        if (std::find(names.begin(), names.end(), r.name) == names.end()) names.push_back(r.name);
    std::string js = "{";
    for (size_t i = 0; i < names.size(); ++i) {
        double ms = 0;
        uint64_t n = 0;
        for (auto &r : ctx->prof)
            if (r.name == names[i]) {
                float t = 0;
                cudaEventElapsedTime(&t, r.e0, r.e1);
                ms += t;
                n++;
            }
        char item[256];
        snprintf(item, sizeof item, "%s\"%s\": {\"ms\": %.6f, \"launches\": %llu}", i ? ", " : "",
                 names[i].c_str(), ms, (unsigned long long)n);
        js += item;
    }
    js += "}";
    if (js.size() + 1 > cap) return fail(ctx, DNAGPU_ECAPACITY, "profile buffer too small");
    memcpy(buf, js.c_str(), js.size() + 1);
    return DNAGPU_OK;
}
