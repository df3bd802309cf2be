/*
 * dna_gpu.c -- PostgreSQL-side glue: the fmgr entry points of the k-mer path re-pointed at
 * libdnagpu.  Built as part of the extension's .so in place of the corresponding functions
 * of the reference's dna.c (same symbol names, same SQL declarations, dna--1.0.sql:188-191),
 * so `CREATE EXTENSION dna` and every existing query keep working.
 *
 *   generate_kmers(dna, int) SETOF kmer   drop-in for dna.c:743-837.  Rows are extracted on the GPU in
 *       windows of GLUE_WINDOW_ROWS start positions, refilled as the executor pulls rows (the SRF protocol
 *       is row-at-a-time by design), so backend memory stays bounded for any sequence length.
 *   generate_kmers_where(dna, int, kmer, qkmer) SETOF kmer   the same rows with the WHERE clause pushed
 *       down:  ... WHERE k.kmer ^@ prefix AND pattern @> k.kmer  (test.sql:67-73, 86-92; starts_with
 *       dna.c:842-866, contains dna.c:1091-1135).  A NULL prefix / pattern means "no such predicate".
 *   kmer_stats(dna, int [, kmer, qkmer], OUT total, OUT distinct, OUT uniq)   the README's total / distinct /
 *       unique query (README.md:122-130) without ever materialising the k-mers in the executor.
 *   count_kmers(dna, int [, kmer, qkmer]) SETOF (kmer, count)   the GROUP BY of README.md:107-116; the grouped
 *       rows stay on the GPU and are fetched in windows.
 *   kmer_spectrum(dna, int [, kmer, qkmer], int H) SETOF (count, kmers)   the abundance spectrum of that GROUP BY
 *       (how many k-mers occur c times, the last row H or more times), binned on the GPU: H integers come back.
 *   kmer_stats_agg(dna, int)   aggregate: the table form of the query (test.sql:140-150,
 *       FROM dna_sequences d, generate_kmers(d.sequence, k) ... GROUP BY) in one pass over the table: the
 *       transition function appends every value to a ragged batch, the final function counts the batch on
 *       the GPU (k-mers never span rows, counts merge across rows).
 *
 * GPU handles that live across calls (the table of count_kmers) are released from a memory-context reset
 * callback, so a query that is cancelled or fails between two rows leaks nothing.
 *
 * There is no PostgreSQL in the build image (no pg_config, no server headers).  The tests
 * compile this file, together with the reference's dna.c, against the PostgreSQL API shim
 * they own and drive it through the fmgr / SRF / aggregate protocol on the GPU (tests/test_gpu_pg_glue.py);
 * pg/Makefile builds the real extension on a machine that has PGXS.  INTEGRATION.md has the steps.
 */
#include "postgres.h"

#include "fmgr.h"
#include "funcapi.h"
#include "access/htup_details.h"
#include "utils/builtins.h"
#include "utils/memutils.h"

#include "../../include/dnagpu.h"

#ifndef DNAGPU_GLUE_NO_MODULE_MAGIC /* dna.c already carries PG_MODULE_MAGIC when linked together */
PG_MODULE_MAGIC;
#endif

#ifndef GLUE_WINDOW_ROWS
#define GLUE_WINDOW_ROWS (4u << 20) /* rows materialised in the backend at a time: 32 MB (+ 32 MB of counts) */
#endif

/* the reference's value layouts (dna.c:42-47, 61-65, 81-84) */
typedef struct Dna {
    char vl_len_[4];
    uint64_t length;
    uint64_t bit_sequence[FLEXIBLE_ARRAY_MEMBER];
} Dna;
typedef struct Kmer {
    int32 length;
    uint64_t bit_sequence;
} Kmer;
typedef struct Qkmer {
    char vl_len_[4];
    char sequence[FLEXIBLE_ARRAY_MEMBER];
} Qkmer;

/* One CUDA context per backend process, created on first use: contexts do not survive the
 * postmaster's fork, and most backends never touch a dna value. */
static dnagpu_ctx *backend_ctx = NULL;
static int live_tables = 0; /* GPU tables held across calls (tests watch this) */

/* Which GPUs the backend uses: "0" (default), or a list such as "0,1,2,3,4,5,6,7" -- then the context spans them
 * (dnagpu_create_multi) and the GROUP BY entry points (kmer_stats, count_kmers without a WHERE clause) shard the
 * sequence over all of them; everything else runs on the first.  Read once, when the backend first touches a dna
 * value.  In an installed extension this is the string GUC dna_gpu.devices (DefineCustomStringVariable in
 * _PG_init, PGC_BACKEND); the environment variable DNAGPU_DEVICES stands in for it here. */
static int
gpu_devices(int *devs, int max)
{
    const char *spec = getenv("DNAGPU_DEVICES");
    int         n = 0;

    while (spec && *spec && n < max)
    {
        char       *end;
        long        v = strtol(spec, &end, 10);

        if (end == spec || v < 0 || v > 1023)
            ereport(ERROR, (errmsg("dnagpu: invalid device list \"%s\"", getenv("DNAGPU_DEVICES"))));
        devs[n++] = (int) v;
        spec = *end == ',' ? end + 1 : end;
        if (*end != ',' && *end != '\0')
            ereport(ERROR, (errmsg("dnagpu: invalid device list \"%s\"", getenv("DNAGPU_DEVICES"))));
    }
    return n;
}

static dnagpu_ctx *
gpu(void)
{
    if (backend_ctx == NULL)
    {
        int         devs[16];
        int         n = gpu_devices(devs, 16);
        int         rc = n > 1 ? dnagpu_create_multi(&backend_ctx, devs, n) : dnagpu_create(&backend_ctx, n == 1 ? devs[0] : 0);

        if (rc != DNAGPU_OK)
            ereport(ERROR, (errmsg("dnagpu: %s", dnagpu_last_error(NULL))));
    }
    return backend_ctx;
}

int
dna_gpu_device_count(void)
{
    return backend_ctx ? dnagpu_device_count(backend_ctx) : 0; /* GPUs of the backend's context, 0 before first use (tests) */
}

int
dna_gpu_live_tables(void)
{
    return live_tables;
}

static void
check_k(int k)
{
    if (k <= 0 || k > 32)       /* dna.c:772-773, same text */
        ereport(ERROR, (errmsg("Invalid k value: must be between 1 and 32")));
}

static uint64_t
rows_of(uint64_t length, int k)
{
    /* dna.c:781 computes length - k + 1 unsigned; a sequence shorter than k has no rows */
    return length >= (uint64_t) k ? length - (uint64_t) k + 1 : 0;
}

/* the optional (kmer, qkmer) arguments 2 and 3 -> dnagpu_where; NULL = predicate absent */
static const dnagpu_where *
where_args(FunctionCallInfo fcinfo, dnagpu_where *w)
{
    memset(w, 0, sizeof *w);
    if (PG_NARGS() < 4)
        return NULL;
    if (!PG_ARGISNULL(2))
    {
        Kmer       *prefix = (Kmer *) PG_GETARG_POINTER(2);

        w->prefix_bits = prefix->bit_sequence;
        w->prefix_len = prefix->length;
    }
    if (!PG_ARGISNULL(3))
        w->qkmer = ((Qkmer *) PG_GETARG_VARLENA_P(3))->sequence;
    return (w->prefix_len || w->qkmer) ? w : NULL;
}

/* =====================================================================================================
 * generate_kmers / generate_kmers_where: windows of start positions, refilled as rows are pulled
 * ===================================================================================================== */
typedef struct GenerateState
{
    Dna        *dna;            /* detoasted into multi_call_memory_ctx */
    int         k;
    uint64_t    rows_total;     /* start positions of the whole value */
    uint64_t    next_start;     /* first start position of the NEXT window (multiple of 32) */
    uint64_t   *bits;           /* rows of the current window */
    uint64_t    n_bits, pos;    /* rows in the window, rows handed out */
    bool        filtered;
    dnagpu_where where;
    char        pattern[36];    /* copy of the qkmer text (the argument is only valid during the first call) */
} GenerateState;

/* load the next non-empty window; false when the value is exhausted */
static bool
generate_refill(GenerateState *st)
{
    while (st->next_start < st->rows_total)
    {
        const uint64_t start = st->next_start;
        const uint64_t starts = Min((uint64_t) GLUE_WINDOW_ROWS, st->rows_total - start);
        const uint64_t sub_bases = starts + (uint64_t) st->k - 1;   /* the window's starts + the (k-1)-base overlap */
        const uint64_t *words = st->dna->bit_sequence + start / 32;
        uint64_t    got = 0;
        int         rc;

        st->next_start = start + starts;
        if (st->filtered)
            rc = dnagpu_filter_kmers(gpu(), words, sub_bases, st->k, &st->where, st->bits, GLUE_WINDOW_ROWS, &got);
        else
            rc = dnagpu_generate_kmers(gpu(), words, sub_bases, st->k, st->bits, GLUE_WINDOW_ROWS, &got);
        if (rc != DNAGPU_OK)
            ereport(ERROR, (errmsg("%s", dnagpu_last_error(backend_ctx))));
        st->n_bits = got;
        st->pos = 0;
        if (got)
            return true;
    }
    return false;
}

static Datum
generate_common(FunctionCallInfo fcinfo, bool with_where)
{
    FuncCallContext *funcctx;
    GenerateState *st;

    if (SRF_IS_FIRSTCALL())
    {
        MemoryContext oldcontext;
        dnagpu_where w;
        const dnagpu_where *wp;

        funcctx = SRF_FIRSTCALL_INIT();
        oldcontext = MemoryContextSwitchTo(funcctx->multi_call_memory_ctx);
        st = (GenerateState *) palloc0(sizeof(GenerateState));
        st->dna = (Dna *) PG_GETARG_VARLENA_P(0);
        st->k = PG_GETARG_INT32(1);
        check_k(st->k);
        st->rows_total = rows_of(st->dna->length, st->k);
        wp = with_where ? where_args(fcinfo, &w) : NULL;
        if (wp)
        {
            st->filtered = true;
            st->where = *wp;
            if (wp->qkmer)
            {
                strncpy(st->pattern, wp->qkmer, sizeof st->pattern - 1);
                st->where.qkmer = st->pattern;
            }
        }
        /* the varlena may be 4-byte aligned (dna--1.0.sql:31): the library copies bytewise */
        st->bits = (uint64_t *) MemoryContextAllocHuge(funcctx->multi_call_memory_ctx,
                                                       sizeof(uint64_t) * Max((uint64_t) 1, Min((uint64_t) GLUE_WINDOW_ROWS, st->rows_total)));
        funcctx->user_fctx = st;
        MemoryContextSwitchTo(oldcontext);
    }

    funcctx = SRF_PERCALL_SETUP();
    st = (GenerateState *) funcctx->user_fctx;

    if (st->pos < st->n_bits || generate_refill(st))
    {
        Kmer       *kmer = (Kmer *) palloc0(sizeof(Kmer));

        kmer->length = st->k;
        kmer->bit_sequence = st->bits[st->pos++];
        SRF_RETURN_NEXT(funcctx, PointerGetDatum(kmer));
    }
    SRF_RETURN_DONE(funcctx);
}

PG_FUNCTION_INFO_V1(generate_kmers);
Datum
generate_kmers(PG_FUNCTION_ARGS)
{
    return generate_common(fcinfo, false);
}

PG_FUNCTION_INFO_V1(generate_kmers_where);
Datum
generate_kmers_where(PG_FUNCTION_ARGS)
{
    if (PG_ARGISNULL(0) || PG_ARGISNULL(1))     /* not STRICT (the predicates may be NULL): no rows for a NULL value */
    {
        FuncCallContext *funcctx = SRF_IS_FIRSTCALL() ? SRF_FIRSTCALL_INIT() : SRF_PERCALL_SETUP();

        SRF_RETURN_DONE(funcctx);
    }
    return generate_common(fcinfo, true);
}

/* =====================================================================================================
 * kmer_stats(dna, int [, kmer, qkmer])
 * ===================================================================================================== */
static Datum
stats_tuple(FunctionCallInfo fcinfo, const dnagpu_stats *st, const char *fn)
{
    TupleDesc   tupdesc;
    Datum       values[3];
    bool        nulls[3] = {false, false, false};

    if (get_call_result_type(fcinfo, NULL, &tupdesc) != TYPEFUNC_COMPOSITE)
        ereport(ERROR, (errmsg("%s must be called in a context that accepts a record", fn)));
    values[0] = Int64GetDatum((int64) st->total);
    values[1] = Int64GetDatum((int64) st->distinct);
    values[2] = Int64GetDatum((int64) st->unique);
    return HeapTupleGetDatum(heap_form_tuple(BlessTupleDesc(tupdesc), values, nulls));
}

PG_FUNCTION_INFO_V1(kmer_stats);
Datum
kmer_stats(PG_FUNCTION_ARGS)
{
    Dna        *dna;
    int         k, rc;
    dnagpu_stats st;
    dnagpu_where w;
    const dnagpu_where *wp;

    if (PG_ARGISNULL(0) || PG_ARGISNULL(1))
        PG_RETURN_NULL();
    dna = (Dna *) PG_GETARG_VARLENA_P(0);
    k = PG_GETARG_INT32(1);
    check_k(k);
    wp = where_args(fcinfo, &w);
    rc = dnagpu_count_kmers(gpu(), dna->bit_sequence, dna->length, k, wp, &st, NULL);
    if (rc != DNAGPU_OK)
        ereport(ERROR, (errmsg("%s", dnagpu_last_error(backend_ctx))));
    PG_FREE_IF_COPY(dna, 0);
    PG_RETURN_DATUM(stats_tuple(fcinfo, &st, "kmer_stats"));
}

/* =====================================================================================================
 * count_kmers(dna, int [, kmer, qkmer]) SETOF (kmer, count): SELECT kmer, count(*) FROM generate_kmers(...)
 * [WHERE ...] GROUP BY kmer (README.md:107-116, test.sql:95-104) as one function.  The first call groups on
 * the GPU; the grouped rows stay there and come over in windows.  Row order is unspecified, like a HashAggregate's.
 * ===================================================================================================== */
typedef struct CountState
{
    dnagpu_table *table;        /* lives on the GPU across calls: freed at the end or by the reset callback */
    uint64_t    rows_total, next_row;
    uint64_t   *kmers;
    uint64_t   *counts;
    uint64_t    n, pos;
    int         k;
    MemoryContextCallback cb;
} CountState;

static void
count_state_release(void *arg)
{
    CountState *st = (CountState *) arg;

    if (st->table)
    {
        dnagpu_table_free(st->table);
        st->table = NULL;
        live_tables--;
    }
}

PG_FUNCTION_INFO_V1(count_kmers);
Datum
count_kmers(PG_FUNCTION_ARGS)
{
    FuncCallContext *funcctx;
    CountState *st;

    if (PG_ARGISNULL(0) || PG_ARGISNULL(1))
    {
        funcctx = SRF_IS_FIRSTCALL() ? SRF_FIRSTCALL_INIT() : SRF_PERCALL_SETUP();
        SRF_RETURN_DONE(funcctx);
    }
    if (SRF_IS_FIRSTCALL())
    {
        MemoryContext oldcontext;
        Dna        *dna;
        int         rc;
        dnagpu_stats stats;
        dnagpu_where w;
        const dnagpu_where *wp;
        TupleDesc   tupdesc;
        uint64_t    win;

        funcctx = SRF_FIRSTCALL_INIT();
        oldcontext = MemoryContextSwitchTo(funcctx->multi_call_memory_ctx);
        dna = (Dna *) PG_GETARG_VARLENA_P(0);
        st = (CountState *) palloc0(sizeof(CountState));
        st->k = PG_GETARG_INT32(1);
        check_k(st->k);
        if (get_call_result_type(fcinfo, NULL, &tupdesc) != TYPEFUNC_COMPOSITE)
            ereport(ERROR, (errmsg("count_kmers must be called in a context that accepts a record")));
        funcctx->tuple_desc = BlessTupleDesc(tupdesc);
        wp = where_args(fcinfo, &w);

        /* the callback is registered BEFORE the table exists: an ereport from here on finds it */
        st->cb.func = count_state_release;
        st->cb.arg = st;
        MemoryContextRegisterResetCallback(funcctx->multi_call_memory_ctx, &st->cb);
        rc = dnagpu_count_kmers(gpu(), dna->bit_sequence, dna->length, st->k, wp, &stats, &st->table);
        if (rc != DNAGPU_OK)
            ereport(ERROR, (errmsg("%s", dnagpu_last_error(backend_ctx))));
        live_tables++;
        st->rows_total = dnagpu_table_rows(st->table);
        win = Max((uint64_t) 1, Min((uint64_t) GLUE_WINDOW_ROWS, st->rows_total));
        st->kmers = (uint64_t *) MemoryContextAllocHuge(funcctx->multi_call_memory_ctx, sizeof(uint64_t) * win);
        st->counts = (uint64_t *) MemoryContextAllocHuge(funcctx->multi_call_memory_ctx, sizeof(uint64_t) * win);
        funcctx->user_fctx = st;
        MemoryContextSwitchTo(oldcontext);
    }

    funcctx = SRF_PERCALL_SETUP();
    st = (CountState *) funcctx->user_fctx;

    if (st->pos == st->n && st->next_row < st->rows_total)
    {
        const uint64_t n = Min((uint64_t) GLUE_WINDOW_ROWS, st->rows_total - st->next_row);
        int         rc = dnagpu_table_fetch(backend_ctx, st->table, st->next_row, n, st->kmers, st->counts);

        if (rc != DNAGPU_OK)
            ereport(ERROR, (errmsg("%s", dnagpu_last_error(backend_ctx))));
        st->next_row += n;
        st->n = n;
        st->pos = 0;
        if (st->next_row == st->rows_total)
            count_state_release(st);    /* the last window is in backend memory */
    }
    if (st->pos < st->n)
    {
        Kmer       *kmer = (Kmer *) palloc0(sizeof(Kmer));
        Datum       values[2];
        bool        nulls[2] = {false, false};

        kmer->length = st->k;
        kmer->bit_sequence = st->kmers[st->pos];
        values[0] = PointerGetDatum(kmer);
        values[1] = Int64GetDatum((int64) st->counts[st->pos]);
        st->pos++;
        SRF_RETURN_NEXT(funcctx, HeapTupleGetDatum(heap_form_tuple((TupleDesc) funcctx->tuple_desc, values, nulls)));
    }
    count_state_release(st);
    SRF_RETURN_DONE(funcctx);
}

/* =====================================================================================================
 * kmer_spectrum(dna, int [, kmer, qkmer], int H) SETOF (count, kmers): the k-mer abundance spectrum,
 *   SELECT least(count, H) AS count, count(*) AS kmers
 *   FROM (SELECT kmer, count(*) FROM generate_kmers(seq, k) AS k(kmer) [WHERE ...] GROUP BY kmer) g
 *   GROUP BY 1 ORDER BY 1;
 * One row per non-zero bin in ascending count; count = H means "H or more".  The first call runs the whole query
 * and keeps at most H rows in backend memory, so no GPU handle outlives it.
 * ===================================================================================================== */
typedef struct SpectrumState
{
    uint64_t   *count;
    uint64_t   *kmers;
    uint64_t    n, pos;
} SpectrumState;

PG_FUNCTION_INFO_V1(kmer_spectrum);
Datum
kmer_spectrum(PG_FUNCTION_ARGS)
{
    FuncCallContext *funcctx;
    SpectrumState *st;
    const int   h_arg = PG_NARGS() - 1;

    if (PG_ARGISNULL(0) || PG_ARGISNULL(1) || PG_ARGISNULL(h_arg))
    {
        funcctx = SRF_IS_FIRSTCALL() ? SRF_FIRSTCALL_INIT() : SRF_PERCALL_SETUP();
        SRF_RETURN_DONE(funcctx);
    }
    if (SRF_IS_FIRSTCALL())
    {
        MemoryContext oldcontext;
        Dna        *dna;
        int         k, rc;
        int32       h;
        uint64_t   *hist;
        uint64_t    c;
        dnagpu_stats stats;
        dnagpu_where w;
        const dnagpu_where *wp;
        TupleDesc   tupdesc;

        funcctx = SRF_FIRSTCALL_INIT();
        oldcontext = MemoryContextSwitchTo(funcctx->multi_call_memory_ctx);
        dna = (Dna *) PG_GETARG_VARLENA_P(0);
        k = PG_GETARG_INT32(1);
        h = PG_GETARG_INT32(h_arg);
        check_k(k);
        if (get_call_result_type(fcinfo, NULL, &tupdesc) != TYPEFUNC_COMPOSITE)
            ereport(ERROR, (errmsg("kmer_spectrum must be called in a context that accepts a record")));
        funcctx->tuple_desc = BlessTupleDesc(tupdesc);
        wp = where_args(fcinfo, &w);
        /* an H out of range is reported by the library; it writes nothing then */
        hist = (uint64_t *) palloc0(sizeof(uint64_t) * (h >= 1 && h <= (1 << 20) ? (uint64_t) h : 1));
        rc = dnagpu_count_kmers_spectrum(gpu(), dna->bit_sequence, dna->length, k, wp, (uint32_t) h, hist, &stats);
        if (rc != DNAGPU_OK)
            ereport(ERROR, (errmsg("%s", dnagpu_last_error(backend_ctx))));
        st = (SpectrumState *) palloc0(sizeof(SpectrumState));
        st->count = (uint64_t *) palloc(sizeof(uint64_t) * (uint64_t) h);
        st->kmers = (uint64_t *) palloc(sizeof(uint64_t) * (uint64_t) h);
        for (c = 1; c <= (uint64_t) h; c++)
            if (hist[c - 1])
            {
                st->count[st->n] = c;
                st->kmers[st->n] = hist[c - 1];
                st->n++;
            }
        pfree(hist);
        funcctx->user_fctx = st;
        MemoryContextSwitchTo(oldcontext);
    }

    funcctx = SRF_PERCALL_SETUP();
    st = (SpectrumState *) funcctx->user_fctx;
    if (st->pos < st->n)
    {
        Datum       values[2];
        bool        nulls[2] = {false, false};

        values[0] = Int64GetDatum((int64) st->count[st->pos]);
        values[1] = Int64GetDatum((int64) st->kmers[st->pos]);
        st->pos++;
        SRF_RETURN_NEXT(funcctx, HeapTupleGetDatum(heap_form_tuple((TupleDesc) funcctx->tuple_desc, values, nulls)));
    }
    SRF_RETURN_DONE(funcctx);
}

/* =====================================================================================================
 * kmer_stats_agg(dna, int): the table form (test.sql:140-150).
 *   SELECT (kmer_stats_agg(sequence, 10)).* FROM dna_sequences;
 * sfunc appends the detoasted value to a ragged batch in the aggregate's memory context; finalfunc uploads
 * the batch once and counts it (dnagpu_seq_upload_ragged + dnagpu_count): one GPU query for the whole table.
 * ===================================================================================================== */
typedef struct AggState
{
    int         k;
    uint64_t    n_seqs, cap_seqs;
    uint64_t    n_words, cap_words;
    uint64_t   *words;          /* the values' packed words back to back, each followed by one zero word */
    uint64_t   *word_off;       /* first word of value s */
    uint64_t   *n_bases;        /* Dna.length of value s */
} AggState;

PG_FUNCTION_INFO_V1(kmer_stats_agg_trans);
Datum
kmer_stats_agg_trans(PG_FUNCTION_ARGS)
{
    MemoryContext aggctx, oldcontext;
    AggState   *st;
    Dna        *dna;
    uint64_t    w;

    if (!AggCheckCallContext(fcinfo, &aggctx))
        ereport(ERROR, (errmsg("kmer_stats_agg_trans called in non-aggregate context")));
    st = PG_ARGISNULL(0) ? NULL : (AggState *) PG_GETARG_POINTER(0);
    if (PG_ARGISNULL(1) || PG_ARGISNULL(2))     /* NULL rows contribute nothing, like generate_kmers(NULL, k) */
    {
        if (st)
            PG_RETURN_POINTER(st);
        PG_RETURN_NULL();
    }
    oldcontext = MemoryContextSwitchTo(aggctx);
    if (st == NULL)
    {
        st = (AggState *) palloc0(sizeof(AggState));
        st->k = PG_GETARG_INT32(2);
        check_k(st->k);
        st->cap_seqs = 1024;
        st->cap_words = 1 << 16;
        st->words = (uint64_t *) MemoryContextAllocHuge(aggctx, st->cap_words * sizeof(uint64_t));
        st->word_off = (uint64_t *) MemoryContextAllocHuge(aggctx, st->cap_seqs * sizeof(uint64_t));
        st->n_bases = (uint64_t *) MemoryContextAllocHuge(aggctx, st->cap_seqs * sizeof(uint64_t));
    }
    else if (PG_GETARG_INT32(2) != st->k)
        ereport(ERROR, (errmsg("kmer_stats_agg: k must be the same for every row")));
    dna = (Dna *) PG_GETARG_VARLENA_P(1);
    w = (dna->length + 31) / 32;
    if (st->n_seqs == st->cap_seqs)
    {
        st->cap_seqs *= 2;
        st->word_off = (uint64_t *) repalloc_huge(st->word_off, st->cap_seqs * sizeof(uint64_t));
        st->n_bases = (uint64_t *) repalloc_huge(st->n_bases, st->cap_seqs * sizeof(uint64_t));
    }
    if (st->n_words + w + 1 > st->cap_words)
    {
        while (st->n_words + w + 1 > st->cap_words)
            st->cap_words *= 2;
        st->words = (uint64_t *) repalloc_huge(st->words, st->cap_words * sizeof(uint64_t));
    }
    memcpy(st->words + st->n_words, dna->bit_sequence, w * sizeof(uint64_t));   /* bytewise: 4-byte aligned varlena */
    st->words[st->n_words + w] = 0;
    st->word_off[st->n_seqs] = st->n_words;
    st->n_bases[st->n_seqs] = dna->length;
    st->n_seqs++;
    st->n_words += w + 1;
    MemoryContextSwitchTo(oldcontext);
    PG_FREE_IF_COPY(dna, 1);
    PG_RETURN_POINTER(st);
}

PG_FUNCTION_INFO_V1(kmer_stats_agg_final);
Datum
kmer_stats_agg_final(PG_FUNCTION_ARGS)
{
    AggState   *st;
    dnagpu_stats stats = {0, 0, 0};

    if (!AggCheckCallContext(fcinfo, NULL))
        ereport(ERROR, (errmsg("kmer_stats_agg_final called in non-aggregate context")));
    st = PG_ARGISNULL(0) ? NULL : (AggState *) PG_GETARG_POINTER(0);
    if (st != NULL && st->n_seqs > 0)
    {
        dnagpu_seq *seq = NULL;
        int         rc = dnagpu_seq_upload_ragged(gpu(), st->words, st->word_off, st->n_bases, st->n_seqs, &seq);

        if (rc == DNAGPU_OK)
        {
            rc = dnagpu_count(backend_ctx, seq, st->k, NULL, NULL, &stats, NULL);
            dnagpu_seq_free(seq);   /* before any ereport: the handle is not in a memory context */
        }
        if (rc != DNAGPU_OK)
            ereport(ERROR, (errmsg("%s", dnagpu_last_error(backend_ctx))));
    }
    PG_RETURN_DATUM(stats_tuple(fcinfo, &stats, "kmer_stats_agg"));
}
