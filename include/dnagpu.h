/*
 * dnagpu.h -- C ABI of libdnagpu: the B200 (sm_100a) implementation of the
 * k-mer hot path of the `dna` PostgreSQL extension.
 *
 * This header is the drop-in boundary.  Everything in it is plain C: opaque
 * handles, pointers and sizes; no C++ or torch types, no exceptions, no
 * longjmp across the boundary.  Host code (the dna.c fmgr glue, the C bench
 * harness, the ctypes binding used by the tests) sees only this file.
 *
 * What each entry point replaces in the reference (/root/reference):
 *
 *   dnagpu_generate_kmers / dnagpu_extract
 *       generate_kmers(dna, int) -- SRF, dna.c:743-837 (SQL: dna--1.0.sql:188-191).
 *       Input is `Dna.bit_sequence` + `Dna.length` exactly as stored
 *       (dna.c:42-47); output element i is `Kmer.bit_sequence` of the i-th
 *       k-mer (dna.c:61-65), `Kmer.length` == k for every element.
 *   dnagpu_filter_kmers / dnagpu_filter
 *       generate_kmers(...) WHERE kmer ^@ prefix AND qkmer @> kmer:
 *       starts_with(), dna.c:842-866 (operator ^@, dna--1.0.sql:193-201) and
 *       contains(), dna.c:1091-1135 with nucleotide_matches(), dna.c:1064-1086
 *       (operator @>, dna--1.0.sql:268-276).  Rows come back in sequence order.
 *   dnagpu_count_kmers / dnagpu_count / dnagpu_count_keys + dnagpu_table_*
 *       SELECT kmer, count(*) ... GROUP BY kmer  and the outer
 *       sum(count) / count(*) / count(*) FILTER (WHERE count = 1)
 *       (README.md:107-135, test.sql:95-119,140-154), i.e. PostgreSQL's
 *       HashAggregate driven by kmer_hash (dna.c:722-735) and kmer_eq
 *       (dna.c:655-668,686-696; opclass dna--1.0.sql:204-212).
 *   dnagpu_count_kmers_spectrum / dnagpu_count_spectrum
 *       SELECT least(count, H), count(*) FROM (... GROUP BY kmer) g GROUP BY 1: the abundance spectrum of
 *       the same GROUP BY, binned on the GPU (unique is its first bin, distinct its sum).
 *   dnagpu_collect
 *       the same WHERE clauses when the row order does not matter (the input of
 *       a GROUP BY or of the exchange between GPUs): one predicate scan.
 *   dnagpu_filter_keys
 *       the same two operators as a seq scan over a stored kmer column
 *       (SELECT ... WHERE kmer_sequence ^@ / @> / =, test.sql:186-262).
 *   dnagpu_index_build / dnagpu_index_equal / dnagpu_index_search
 *       CREATE INDEX ... USING spgist (kmer_sequence spgist_kmer_ops) and the index
 *       scans it serves (dna.c:1137-1737, dna--1.0.sql:278-330, test.sql:186-262).
 *   dnagpu_encode_dna / dnagpu_seq_from_text / dnagpu_decode_dna
 *       dna_in -> dna_make: validate_dna_sequence (dna.c:159-171) + encode_dna
 *       (dna.c:114-128); dna_out -> decode_dna (dna.c:135-152).
 *   dnagpu_partition / dnagpu_owner_of, dnagpu_shuffle_*, dnagpu_peer_*
 *       no reference counterpart (the reference is single-process); these are
 *       the owner-routing / exchange steps of the multi-GPU GROUP BY.
 *
 * Errors: every call returns an int status (0 = ok).  Argument errors carry
 * the reference's own ereport() texts (see dnagpu_strerror), so glue can do
 * `ereport(ERROR, (errmsg("%s", dnagpu_last_error(ctx))))`.
 *
 * Threading: a ctx is single-threaded (like a PostgreSQL backend); distinct
 * contexts may be used from distinct threads.  All work of a ctx is issued on
 * one CUDA stream (its own, or one lent with dnagpu_set_stream).
 *
 * There is no CPU fallback: without a usable sm_100 device dnagpu_create fails
 * with DNAGPU_ENODEVICE and nothing else can be called.
 */
#ifndef DNAGPU_H
#define DNAGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DNAGPU_VERSION 100 /* 1.0.0 */
#define DNAGPU_MAX_K 32

/* ---- status codes -------------------------------------------------------- */
enum {
    DNAGPU_OK = 0,
    /* argument errors that mirror an ereport(ERROR) of the reference */
    DNAGPU_EINVAL_K = 1,      /* dna.c:772-773  "Invalid k value: must be between 1 and 32" */
    DNAGPU_EPREFIX_LEN = 2,   /* dna.c:854-856  "Prefix length cannot exceed kmer length" */
    DNAGPU_EQKMER_LEN = 3,    /* dna.c:1106-1108 "Qkmer pattern and kmer lengths do not match" */
    DNAGPU_EQKMER_CHAR = 4,   /* dna.c:893-895  "Invalid character in qkmer pattern: %c" */
    DNAGPU_EQKMER_EMPTY = 5,  /* dna.c:877-879  "qkmer pattern cannot be empty" */
    DNAGPU_EQKMER_TOOLONG = 6,/* dna.c:883-885  "Qkmer pattern length cannot exceed 32 characters" */
    DNAGPU_EPREFIX_BITS = 7,  /* prefix has bits set above 2*prefix_len (cannot come from kmer_make) */
    DNAGPU_EDNA_CHAR = 8,     /* dna.c:165-166  "Invalid character in DNA sequence: %c" (first offender) */
    DNAGPU_EDNA_EMPTY = 9,    /* dna.c:160-161  "DNA sequence cannot be empty" */
    /* library errors */
    DNAGPU_EARG = 20,         /* NULL pointer, misaligned device pointer, bad size ... */
    DNAGPU_ECAPACITY = 21,    /* caller's output buffer is too small; *n_out holds the need */
    DNAGPU_ENOMEM = 22,       /* device or pinned-host allocation failed */
    DNAGPU_ECUDA = 23,        /* a CUDA call failed; text in dnagpu_last_error */
    DNAGPU_ENODEVICE = 24,    /* no usable sm_100 GPU / driver */
    DNAGPU_EINTERNAL = 25     /* invariant violated (e.g. hash table overflow) */
};

typedef struct dnagpu_ctx dnagpu_ctx;     /* one GPU, one stream, scratch memory   */
typedef struct dnagpu_seq dnagpu_seq;     /* device-resident packed dna value(s)   */
typedef struct dnagpu_table dnagpu_table; /* device-resident GROUP BY kmer result  */

/*
 * WHERE-clause predicates fused into extraction.  Both optional; both given =
 * AND.  `prefix_bits`/`prefix_len` are the two fields of the prefix `Kmer`
 * (dna.c:61-65) as kmer_make() builds them; `qkmer` is `Qkmer.sequence`
 * (dna.c:81-84), a NUL-terminated IUPAC string.
 */
/* How an unordered predicate scan (dnagpu_collect, the WHERE clause of a GROUP BY) evaluates the clause: by
 * default as a Shift-And automaton over the base stream (6 instructions per base); with this flag as the
 * per-start-position test on four "allowed" bit planes (~ 19 instructions per start position), which the
 * ordered scans (dnagpu_filter*) and ragged batches always use.  Same rows either way. */
#define DNAGPU_WHERE_FLAG_PLANES 1

typedef struct dnagpu_where {
    uint64_t prefix_bits; /* Kmer.bit_sequence of the ^@ right operand          */
    int32_t prefix_len;   /* Kmer.length of it; 0 = no ^@ predicate             */
    int32_t flags;        /* DNAGPU_WHERE_FLAG_*; 0 = default                    */
    const char *qkmer;    /* @> left operand; NULL = no @> predicate            */
} dnagpu_where;

/* sum(count), count(*), count(*) FILTER (WHERE count = 1) over the groups. */
typedef struct dnagpu_stats {
    uint64_t total;
    uint64_t distinct;
    uint64_t unique;
} dnagpu_stats;

/* How GROUP BY is executed.  AUTO picks by k and input size (see DESIGN.md). */
enum {
    DNAGPU_COUNT_AUTO = 0,
    DNAGPU_COUNT_DENSE = 1,     /* direct-indexed 4^k counters (k <= 16)        */
    DNAGPU_COUNT_HASH = 2,      /* HBM open-addressing table, CAS + add         */
    DNAGPU_COUNT_PARTITION = 3  /* two-level radix partition, then one shared-memory table per bucket */
};

/* DNAGPU_COUNT_PARTITION sizes its partitions optimistically (fixed regions of mean + slack, no histogram
 * pass; a full region makes the library redo that level exactly).  This flag takes the exact two-pass form
 * from the start: same result, for inputs known to be heavily repeated -- and for the tests of that path. */
#define DNAGPU_COUNT_FLAG_EXACT 1

typedef struct dnagpu_count_opts {
    int32_t method;        /* DNAGPU_COUNT_*                                    */
    int32_t flags;         /* DNAGPU_COUNT_FLAG_*; 0 = default                    */
    double load_factor;    /* hash table target load, 0 = default (0.5)         */
    uint64_t expected_keys;/* 0 = derive from input (n_kmers, 4^k)              */
    /* Multi-GPU: count only the k-mers that dnagpu_owner_of(kmer, owner_parts) assigns to owner_part
     * (0 parts = no restriction).  Every GPU of a box runs the same query over the same sequence --
     * resident as one piece per GPU, see dnagpu_seq_wrap_pieces -- with its own owner_part; the key sets
     * are disjoint, so the aggregates add and the grouped rows concatenate.  Single sequences only, no
     * WHERE clause.  owner_parts = 1 (owner_part 0) keeps every k-mer: on a sequence in pieces it counts
     * the whole sequence, on any other input it is the same as no restriction. */
    uint32_t owner_parts;
    uint32_t owner_part;
} dnagpu_count_opts;

/* ---- context ------------------------------------------------------------- */
int dnagpu_version(void);
const char *dnagpu_strerror(int code);
int dnagpu_create(dnagpu_ctx **out, int device);
/* One context over several GPUs of one box: one process, no IPC, the GPUs see each other's memory through
 * peer access (NVLink).  The context behaves like a single-GPU context on devices[0] for every call; the
 * host-buffer GROUP BY (dnagpu_count_kmers without a WHERE clause) uses ALL of them: the packed words are
 * cut into one base-range shard per GPU (with the (k-1)-base overlap), uploaded in parallel, and every GPU
 * counts the k-mers it owns out of the whole sequence (see dnagpu_count_opts.owner_parts).  The aggregates
 * are the sums, the table is the concatenation of the per-GPU tables.  n_devices <= 16. */
int dnagpu_create_multi(dnagpu_ctx **out, const int *devices, int n_devices);
/* GPUs behind the context (1 for dnagpu_create). */
int dnagpu_device_count(const dnagpu_ctx *ctx);
void dnagpu_destroy(dnagpu_ctx *ctx);
const char *dnagpu_last_error(const dnagpu_ctx *ctx);
/* Lend a cudaStream_t (e.g. torch's current stream); NULL = library's own. */
int dnagpu_set_stream(dnagpu_ctx *ctx, void *cuda_stream);
int dnagpu_synchronize(dnagpu_ctx *ctx);
/* Device facts for the harness: name (<= cap bytes), SM count, free/total HBM. */
int dnagpu_device_info(dnagpu_ctx *ctx, char *name, size_t cap, int *sm_count,
                       uint64_t *hbm_free, uint64_t *hbm_total);
/* Page-locked host memory.  The host-in/host-out calls below accept any host
 * pointer, but copies from/to memory obtained here run at full PCIe speed
 * (glue: detoast the dna value into such a buffer). */
int dnagpu_host_alloc(dnagpu_ctx *ctx, void **out, uint64_t bytes);
void dnagpu_host_free(dnagpu_ctx *ctx, void *p);

/* ---- packed sequences on the device -------------------------------------- */
/* One dna value: words = Dna.bit_sequence (ceil(n_bases/32) words, any 8-byte
 * aligned host pointer; 4-byte aligned is tolerated, see dna--1.0.sql:31),
 * n_bases = Dna.length.  Copies; the caller keeps ownership of `words`. */
int dnagpu_seq_upload(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_bases,
                      dnagpu_seq **out);
/* A batch of equal-length dna values (reads) at a fixed stride: read r's words
 * start at words[r*stride_words].  k-mers never span reads (each read is its
 * own generate_kmers call, test.sql:140-150). */
int dnagpu_seq_upload_reads(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_reads,
                            uint32_t bases_per_read, uint32_t stride_words,
                            dnagpu_seq **out);
/* A batch of dna values of different lengths (rows of a table): value s has
 * n_bases[s] bases and its words start at words[word_offsets[s]]. */
int dnagpu_seq_upload_ragged(dnagpu_ctx *ctx, const uint64_t *words,
                             const uint64_t *word_offsets, const uint64_t *n_bases,
                             uint64_t n_seqs, dnagpu_seq **out);
/* Synthetic inputs generated on the device (include/dnagpu_synth.h defines the
 * stream).  The *_range form builds the shard [first_base, first_base+n_starts)
 * of a longer sequence plus the (k-1)-base overlap needed for `overlap_k`
 * (first_base must be a multiple of 32); only k-mers that START inside the
 * shard are ever produced from it. */
int dnagpu_seq_synth(dnagpu_ctx *ctx, uint64_t n_bases, uint64_t seed,
                     uint32_t repeat_every, dnagpu_seq **out);
int dnagpu_seq_synth_range(dnagpu_ctx *ctx, uint64_t n_bases_total, uint64_t seed,
                           uint32_t repeat_every, uint64_t first_base,
                           uint64_t n_starts, int overlap_k, dnagpu_seq **out);
int dnagpu_seq_synth_reads(dnagpu_ctx *ctx, uint64_t first_read, uint64_t n_reads,
                           uint32_t bases_per_read, uint32_t stride_words,
                           uint64_t seed, uint32_t repeat_every, dnagpu_seq **out);
/* Borrow caller-owned device memory holding one packed sequence.  d_words must
 * be 16-byte aligned and n_words_alloc >= ceil(n_bases/32)+1 rounded up to an
 * even count, with every word at or past ceil(n_bases/32) equal to zero. */
int dnagpu_seq_wrap(dnagpu_ctx *ctx, const void *d_words, uint64_t n_bases,
                    uint64_t n_words_alloc, dnagpu_seq **out);
/* The same for a fixed-stride batch of reads (n_words_alloc >= n_reads*stride+1). */
int dnagpu_seq_wrap_reads(dnagpu_ctx *ctx, const void *d_words, uint64_t n_reads,
                          uint32_t bases_per_read, uint32_t stride_words,
                          uint64_t n_words_alloc, dnagpu_seq **out);
/* One dna value resident as n_pieces base-range pieces (multi-GPU: one shard per GPU, each mapped into this
 * GPU's address space -- its own memory, or peer memory opened with dnagpu_peer_open).  Piece i holds the
 * packed words of the bases from first_base[i] on and serves the k-mers that START in
 * [first_base[i], first_base[i] + n_starts[i]): it must reach 31 bases past that range (the (k-1)-base
 * overlap for any k <= 32) and end in one zero pad word, first_base[i] must be a multiple of 32, and the
 * ranges must tile [0, n_bases_total) when sorted.  The pieces are walked in the order given (put this GPU's
 * own piece first and the others in ring order, so that no shard is read by every GPU at once).  Such a
 * sequence is accepted by dnagpu_count with an owner restriction (dnagpu_count_opts.owner_parts) only. */
int dnagpu_seq_wrap_pieces(dnagpu_ctx *ctx, const void *const *d_words, const uint64_t *first_base,
                           const uint64_t *n_starts, uint32_t n_pieces, uint64_t n_bases_total,
                           dnagpu_seq **out);
/* Restrict a single sequence to the k-mers starting in its first n_starts
 * bases (multi-GPU shards with overlap).  0 = no restriction. */
int dnagpu_seq_set_start_limit(dnagpu_seq *seq, uint64_t n_starts);
/* Copy the packed words back (tests): n_words = all words of the batch. */
int dnagpu_seq_download(dnagpu_ctx *ctx, const dnagpu_seq *seq, uint64_t *words,
                        uint64_t n_words);
uint64_t dnagpu_seq_words(const dnagpu_seq *seq);
const void *dnagpu_seq_device_words(const dnagpu_seq *seq);
/* Number of rows generate_kmers(seq, k) returns, summed over the batch
 * (0 where length < k, never the reference's unsigned wrap of dna.c:781). */
uint64_t dnagpu_seq_kmer_count(const dnagpu_seq *seq, int k);
void dnagpu_seq_free(dnagpu_seq *seq);

/* ---- ingest codec: dna_in / dna_out (dna.c:114-171, 135-152) ------------------------ */
/* text (n_bases ASCII bytes, no NUL needed) -> packed words, validated like dna_make: upper-case A T C G
 * only, not empty; on DNAGPU_EDNA_CHAR the message names the first offending character. */
int dnagpu_encode_dna(dnagpu_ctx *ctx, const char *text, uint64_t n_bases, uint64_t *words);
/* the same, leaving the packed sequence on the device ready for the calls below (COPY ... FROM) */
int dnagpu_seq_from_text(dnagpu_ctx *ctx, const char *text, uint64_t n_bases, dnagpu_seq **out);
/* packed words -> text; writes n_bases characters and a terminating NUL */
int dnagpu_decode_dna(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_bases, char *text);

/* ---- generate_kmers -------------------------------------------------------- */
/* Host in, host out: what the fmgr glue calls on the SRF's first call.
 * out[i] = bit_sequence of k-mer i; *n_out = number written (or needed, with
 * DNAGPU_ECAPACITY, when cap is too small; out may be NULL to just ask). */
int dnagpu_generate_kmers(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_bases,
                          int k, uint64_t *out, uint64_t cap, uint64_t *n_out);
/* Device in, device out (d_out 16-byte aligned). */
int dnagpu_extract(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k, uint64_t *d_out,
                   uint64_t cap, uint64_t *n_out);

/* ---- generate_kmers ... WHERE ^@ / @> -------------------------------------- */
int dnagpu_filter_kmers(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_bases,
                        int k, const dnagpu_where *filter, uint64_t *out,
                        uint64_t cap, uint64_t *n_out);
/* d_out may be NULL: then only the number of matching rows is computed. */
int dnagpu_filter(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k,
                  const dnagpu_where *filter, uint64_t *d_out, uint64_t cap,
                  uint64_t *n_out);
/* The rows that pass the WHERE clause in NO particular order -- what a GROUP BY or an exchange
 * between GPUs needs; one predicate scan instead of the two of the ordered form.  Writes at most
 * cap rows; with more matches than cap returns DNAGPU_ECAPACITY and *n_out = the number needed.
 * d_out may be NULL (cap 0): then only the number of matching rows is computed. */
int dnagpu_collect(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k, const dnagpu_where *filter,
                   uint64_t *d_out, uint64_t cap, uint64_t *n_out);
/* The same predicates over a materialised kmer column (k the same for all
 * rows): keeps input order.  d_out may alias nothing and may be NULL. */
int dnagpu_filter_keys(dnagpu_ctx *ctx, const uint64_t *d_keys, uint64_t n, int k,
                       const dnagpu_where *filter, uint64_t *d_out, uint64_t cap,
                       uint64_t *n_out);

/* ---- GROUP BY kmer ---------------------------------------------------------- */
/* filter may be NULL; opts may be NULL (AUTO); table may be NULL when only the
 * three aggregates are wanted. */
int dnagpu_count_kmers(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_bases, int k,
                       const dnagpu_where *filter, dnagpu_stats *stats,
                       dnagpu_table **table);
/* The table form of the query (test.sql:140-150): one row per read, k-mers
 * never span rows, counts merge across rows. */
int dnagpu_count_reads(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_reads,
                       uint32_t bases_per_read, uint32_t stride_words, int k,
                       const dnagpu_where *filter, dnagpu_stats *stats,
                       dnagpu_table **table);
int dnagpu_count(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k,
                 const dnagpu_where *filter, const dnagpu_count_opts *opts,
                 dnagpu_stats *stats, dnagpu_table **table);
/* Count an already materialised k-mer list on the device (the receive side of
 * the multi-GPU exchange, or a stored kmer column). */
int dnagpu_count_keys(dnagpu_ctx *ctx, const uint64_t *d_keys, uint64_t n, int k,
                      const dnagpu_count_opts *opts, dnagpu_stats *stats,
                      dnagpu_table **table);

/* The abundance spectrum of the same query (jellyfish histo): with H = max_count, 1 <= H <= 2^20,
 *   hist[c-1] = the number of distinct k-mers that occur exactly c times, c = 1 .. H-1;
 *   hist[H-1] = the number that occur H times or more  (SQL: GROUP BY least(count, H)).
 * hist is H uint64 in host memory.  stats receives what dnagpu_count returns, so sum(hist) == distinct and, for
 * H >= 2, hist[0] == unique.  WHERE clause, layouts, methods, flags and the owner restriction are those of
 * dnagpu_count; no table is built: the spectrum is binned on the device by the count itself, and H integers come
 * back.  'G' x 32 (k = 32) is one group like any other.  A bad max_count or a NULL hist: DNAGPU_EARG. */
int dnagpu_count_spectrum(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k, const dnagpu_where *filter,
                          const dnagpu_count_opts *opts, uint32_t max_count, uint64_t *hist, dnagpu_stats *stats);
/* The same from host words (what the SQL glue calls).  On a dnagpu_create_multi context and without a WHERE clause,
 * every GPU counts the k-mers it owns (as dnagpu_count_kmers does) and the spectra add. */
int dnagpu_count_kmers_spectrum(dnagpu_ctx *ctx, const uint64_t *words, uint64_t n_bases, int k,
                                const dnagpu_where *filter, uint32_t max_count, uint64_t *hist,
                                dnagpu_stats *stats);

/* The grouped result.  Rows are (kmer bits, count); order is unspecified (as
 * for a HashAggregate) but fixed for the life of the table. */
uint64_t dnagpu_table_rows(const dnagpu_table *table);
int dnagpu_table_k(const dnagpu_table *table);
int dnagpu_table_fetch(dnagpu_ctx *ctx, const dnagpu_table *table, uint64_t offset,
                       uint64_t n, uint64_t *kmers, uint64_t *counts);
/* Device pointers of the compacted rows (valid until dnagpu_table_free).  Not available for the table of a
 * multi-GPU count (its rows live on several GPUs): DNAGPU_EARG. */
int dnagpu_table_device(const dnagpu_table *table, const uint64_t **d_kmers,
                        const uint64_t **d_counts);
void dnagpu_table_free(dnagpu_table *table);

/* ---- multi-GPU owner routing ------------------------------------------------- */
/* Owner rank of a k-mer among n_parts ranks (pure function; host-callable).  A function of the k-mer's first
 * 16 bases: for 2, 4 and 8 ranks a GF(2)-linear hash (parities under three tap masks; the rank among 2 or 4 is
 * the low bits of the rank among 8), for any other count a multiplicative hash. */
uint32_t dnagpu_owner_of(uint64_t kmer, uint32_t n_parts);
/* Extract (+filter) and bucket the k-mers by owner: bucket p occupies
 * d_out[offset_p, offset_p + part_counts[p]) with offset_p the exclusive prefix
 * sum of part_counts (host array of n_parts entries, written by the call).
 * d_out may be NULL to obtain only the counts. */
int dnagpu_partition(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k,
                     const dnagpu_where *filter, uint32_t n_parts, uint64_t *d_out,
                     uint64_t cap, uint64_t *part_counts);

/*
 * The faster multi-GPU form: the owner routing IS level 1 of the radix partition.  Every rank
 * partitions its shard by the top `bits1` bits of the partition hash into n_digits buckets laid
 * out in digit order; owner(digit) = digit * n_parts >> bits1, so what goes to one owner is ONE
 * contiguous slice of d_out and the all-to-all needs no separate bucketing pass.  The receiver
 * gets, from every peer, the pieces of the digits it owns (n_groups of them per peer, in digit
 * order, peer-major) and finishes with level 2 + the shared-memory count; pieces of the same digit
 * merge.  All ranks must build the plan from the same (n_rows_total, n_parts).
 */
typedef struct dnagpu_shuffle_plan {
    int32_t bits1, bits2; /* hash bits of partition level 1 (exchange) and level 2 (local) */
    uint32_t n_parts;     /* owner ranks                                                  */
    uint32_t n_digits;    /* 1 << bits1                                                   */
} dnagpu_shuffle_plan;
int dnagpu_shuffle_plan_make(uint64_t n_rows_total, uint32_t n_parts, dnagpu_shuffle_plan *plan);
uint32_t dnagpu_shuffle_owner(const dnagpu_shuffle_plan *plan, uint32_t digit);
/* Extract (+filter) this rank's k-mers and lay them out by digit in d_out (cap >= rows + 2).
 * digit_counts (host, n_digits entries) receives the keys per digit; rows_kept the rows that
 * passed the WHERE clause; side_rows the 'G' x 32 rows (k = 32), which are not in d_out. */
int dnagpu_shuffle_send(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k, const dnagpu_where *filter,
                        const dnagpu_shuffle_plan *plan, uint64_t *d_out, uint64_t cap,
                        uint64_t *digit_counts, uint64_t *rows_kept, uint64_t *side_rows);
/* Count what arrived: n_pieces = n_peers * n_groups pieces of piece_counts[i] keys each, stored
 * back to back in d_keys; piece i holds digit (i % n_groups) of this owner. */
int dnagpu_shuffle_count(dnagpu_ctx *ctx, const uint64_t *d_keys, const uint64_t *piece_counts,
                         uint32_t n_pieces, uint32_t n_groups, const dnagpu_shuffle_plan *plan, int k,
                         dnagpu_stats *stats, dnagpu_table **table);

/*
 * The exchange fused INTO the scatter kernel (no all-to-all at all): each rank allocates its
 * receive buffer with dnagpu_peer_alloc, the ranks swap the 64-byte handles (any side channel,
 * e.g. torch.distributed.all_gather_object) and map each other's buffers with dnagpu_peer_open.
 * A step is then: dnagpu_shuffle_hist -> all-gather of the per-digit counts (so that every rank
 * can compute where its piece of every digit starts inside the owner's buffer, pieces laid out
 * peer-major in digit order) -> dnagpu_shuffle_scatter_to, whose kernel stores every run of keys
 * straight into the owner's memory over NVLink (st.global on peer-mapped addresses) ->
 * a barrier -> dnagpu_shuffle_count on the local receive buffer.
 */
int dnagpu_peer_alloc(dnagpu_ctx *ctx, uint64_t bytes, void **d_ptr, unsigned char handle[64]);
int dnagpu_peer_open(dnagpu_ctx *ctx, const unsigned char handle[64], void **d_ptr);
int dnagpu_peer_close(dnagpu_ctx *ctx, void *d_ptr);
int dnagpu_peer_free(dnagpu_ctx *ctx, void *d_ptr);
/* keys per digit of this rank's shard (host array of plan->n_digits entries) */
int dnagpu_shuffle_hist(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k, const dnagpu_where *filter,
                        const dnagpu_shuffle_plan *plan, uint64_t *digit_counts);
/* scatter: the keys of digit d go to the device address digit_dest[d] (local or peer-mapped,
 * 8-byte aligned), digit_counts[d] of them */
int dnagpu_shuffle_scatter_to(dnagpu_ctx *ctx, const dnagpu_seq *seq, int k, const dnagpu_where *filter,
                              const dnagpu_shuffle_plan *plan, const uint64_t *digit_dest,
                              uint64_t *rows_kept, uint64_t *side_rows);
/* The same two steps over a key list already on the device (e.g. what dnagpu_collect kept of
 * a selective WHERE clause): keys per digit, then the stores.  side_rows = the 'G' x 32 rows
 * (k = 32) of the list, which are not stored. */
int dnagpu_shuffle_hist_keys(dnagpu_ctx *ctx, const uint64_t *d_keys, uint64_t n,
                             const dnagpu_shuffle_plan *plan, uint64_t *digit_counts);
int dnagpu_shuffle_scatter_keys_to(dnagpu_ctx *ctx, const uint64_t *d_keys, uint64_t n,
                                   const dnagpu_shuffle_plan *plan, const uint64_t *digit_dest,
                                   uint64_t *side_rows);

/* ---- index over a stored kmer column -------------------------------------------
 * Replaces the reference's SP-GiST operator class (spgist_kmer_ops: config / choose /
 * picksplit / inner_consistent / leaf_consistent, dna.c:1137-1737, dna--1.0.sql:278-330)
 * for the queries it serves (test.sql:186-262):  kmer = x,  kmer ^@ prefix,  qkmer @> kmer.
 * The index is the column sorted by base string (base 0 most significant) with the row
 * number of every entry; a prefix is one contiguous range.  Searches return 0-based row
 * numbers of the indexed column in ascending order (the order of a bitmap heap scan) and,
 * unlike the reference's trie (1021 of 1025 rows, test.sql:186-214), exactly the rows a
 * sequential scan returns.  d_rows may be NULL: then only the number of rows is computed;
 * too small a buffer gives DNAGPU_ECAPACITY with *n_out = the number needed. */
typedef struct dnagpu_index dnagpu_index;
int dnagpu_index_build(dnagpu_ctx *ctx, const uint64_t *d_keys, uint64_t n, int k, dnagpu_index **index);
uint64_t dnagpu_index_rows(const dnagpu_index *index);
int dnagpu_index_k(const dnagpu_index *index);
/* the sorted column (sort keys: the 2-bit groups of Kmer.bit_sequence in reverse order) and the rows */
int dnagpu_index_device(const dnagpu_index *index, const uint64_t **d_sort_keys, const uint64_t **d_rows);
/* WHERE kmer = x: kmer_eq compares the lengths too (dna.c:655-668) */
int dnagpu_index_equal(dnagpu_ctx *ctx, const dnagpu_index *index, uint64_t kmer_bits, int kmer_len,
                       uint64_t *d_rows, uint64_t cap, uint64_t *n_out);
/* WHERE kmer ^@ prefix AND qkmer @> kmer (either may be absent); same errors as dnagpu_filter_keys */
int dnagpu_index_search(dnagpu_ctx *ctx, const dnagpu_index *index, const dnagpu_where *where,
                        uint64_t *d_rows, uint64_t cap, uint64_t *n_out);
void dnagpu_index_free(dnagpu_index *index);

/* ---- per-kernel device timing (CUDA events on the ctx stream) --------------- */
int dnagpu_profile_enable(dnagpu_ctx *ctx, int on);
int dnagpu_profile_reset(dnagpu_ctx *ctx);
/* Total device milliseconds and launch count of kernels whose name starts with
 * `prefix` ("" = all) since the last reset.  Synchronises the stream. */
int dnagpu_profile_query(dnagpu_ctx *ctx, const char *prefix, double *total_ms,
                         uint64_t *launches);
/* JSON object {"kernel": {"ms": x, "launches": n}, ...} into buf. */
int dnagpu_profile_dump(dnagpu_ctx *ctx, char *buf, size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* DNAGPU_H */
