-- Additions to dna--1.0.sql for the GPU build.  generate_kmers keeps its declaration
-- (dna--1.0.sql:188-191); only the implementation behind MODULE_PATHNAME changes.

-- generate_kmers(...) WHERE kmer ^@ prefix AND pattern @> kmer  (test.sql:67-73, 86-92) with the clause pushed
-- down to the GPU; a NULL prefix / pattern means "no such predicate".  Not STRICT for that reason.
CREATE OR REPLACE FUNCTION generate_kmers_where(dna, integer, kmer, qkmer)
    RETURNS SETOF kmer
    AS 'MODULE_PATHNAME', 'generate_kmers_where'
    LANGUAGE C IMMUTABLE PARALLEL SAFE;

-- total / distinct / unique of README.md:122-130 computed on the GPU in one call
CREATE OR REPLACE FUNCTION kmer_stats(dna, integer, OUT total bigint, OUT "distinct" bigint, OUT uniq bigint)
    RETURNS record
    AS 'MODULE_PATHNAME', 'kmer_stats'
    LANGUAGE C IMMUTABLE STRICT PARALLEL SAFE;
CREATE OR REPLACE FUNCTION kmer_stats(dna, integer, kmer, qkmer, OUT total bigint, OUT "distinct" bigint, OUT uniq bigint)
    RETURNS record
    AS 'MODULE_PATHNAME', 'kmer_stats'
    LANGUAGE C IMMUTABLE PARALLEL SAFE;

-- SELECT kmer, count(*) FROM generate_kmers(seq, k) [WHERE ...] GROUP BY kmer  (README.md:107-116) in one call
CREATE OR REPLACE FUNCTION count_kmers(dna, integer, OUT kmer kmer, OUT count bigint)
    RETURNS SETOF record
    AS 'MODULE_PATHNAME', 'count_kmers'
    LANGUAGE C IMMUTABLE STRICT PARALLEL SAFE;
CREATE OR REPLACE FUNCTION count_kmers(dna, integer, kmer, qkmer, OUT kmer kmer, OUT count bigint)
    RETURNS SETOF record
    AS 'MODULE_PATHNAME', 'count_kmers'
    LANGUAGE C IMMUTABLE PARALLEL SAFE;

-- The k-mer abundance spectrum in one call: one row per non-zero bin, count = H meaning "H or more", i.e.
--   SELECT least(count, H) AS count, count(*) AS kmers
--   FROM (SELECT kmer, count(*) FROM generate_kmers(seq, k) AS k(kmer) [WHERE ...] GROUP BY kmer) g
--   GROUP BY 1 ORDER BY 1;
CREATE OR REPLACE FUNCTION kmer_spectrum(dna, integer, integer, OUT count bigint, OUT kmers bigint)
    RETURNS SETOF record
    AS 'MODULE_PATHNAME', 'kmer_spectrum'
    LANGUAGE C IMMUTABLE STRICT PARALLEL SAFE;
CREATE OR REPLACE FUNCTION kmer_spectrum(dna, integer, kmer, qkmer, integer, OUT count bigint, OUT kmers bigint)
    RETURNS SETOF record
    AS 'MODULE_PATHNAME', 'kmer_spectrum'
    LANGUAGE C IMMUTABLE PARALLEL SAFE;

-- The table form (test.sql:140-150) as an aggregate: one GPU query for the whole table.
--   SELECT (kmer_stats_agg(sequence, 10)).* FROM dna_sequences;
CREATE OR REPLACE FUNCTION kmer_stats_agg_trans(internal, dna, integer)
    RETURNS internal
    AS 'MODULE_PATHNAME', 'kmer_stats_agg_trans'
    LANGUAGE C IMMUTABLE;
CREATE OR REPLACE FUNCTION kmer_stats_agg_final(internal, OUT total bigint, OUT "distinct" bigint, OUT uniq bigint)
    RETURNS record
    AS 'MODULE_PATHNAME', 'kmer_stats_agg_final'
    LANGUAGE C IMMUTABLE;
CREATE AGGREGATE kmer_stats_agg(dna, integer) (
    SFUNC = kmer_stats_agg_trans,
    STYPE = internal,
    FINALFUNC = kmer_stats_agg_final
);
