/*
 * itsx_b200.h -- C ABI of libitsx_b200.so, the B200 (sm_100a) implementation of the ITSxpress
 * hot path:  exact dereplication -> profile-HMM search -> boundary selection -> trim/re-expand.
 *
 * Every entry point below replaces one process boundary / Python loop of the reference
 * (citations are into the upstream tree, itsxpress/...):
 *
 *   itsx_profiles_*      create_runtime_hmm()                       main.py:176-231
 *                        + hmmsearch's own reading of that file     SeqSample.py:191-209
 *   itsx_derep*          `vsearch --fastx_uniques --strand both`    SeqSample.py:93-131 (argv :106-116)
 *                        + Dedup.parse (read -> representative)     SeqSample.py:542-562
 *   itsx_search*         `hmmsearch --domtblout -T 10 --F1 1e-6 --F2 1e-6 --F3 1e-6`
 *                                                                  SeqSample.py:178-225 (argv :191-209)
 *   itsx_hits            the domtbl rows ItsPosition.parse consumes SeqSample.py:431-461 (cols :445-450)
 *   itsx_positions       ItsPosition._score / get_position          SeqSample.py:400-429, 463-498
 *   itsx_trim_*          Dedup._get_trimmed_seq_generator /         SeqSample.py:792-884
 *                        Dedup._get_paired_seq_generator            SeqSample.py:564-711
 *   itsx_merge_*         `vsearch --fastq_mergepairs` (paired input, the step in front of derep)
 *                                                                  SeqSample.py:266-365 (argv :314-349)
 *   itsx_gzip_*          gzip.open(..., "wt") of the output writers    SeqSample.py:767-788, 926-949
 *
 * Conventions: plain C, no callbacks, no exceptions across the boundary.  Functions return
 * 0 on success and a negative ITSX_E* code on failure; itsx_last_error() gives the text.
 * Caller buffers are caller-owned and may live in host memory (pageable or pinned) OR in device
 * memory of the context's GPU (copies use cudaMemcpyDefault; the multi-GPU driver passes torch tensors);
 * the library's own device memory sits behind itsx_ctx (one ctx per host thread / per GPU).  Calls run on the
 * library's stream and return after it drained: make a device buffer's producer finish first.  There is NO CPU fallback: without a usable CUDA device
 * itsx_create() fails with ITSX_ENODEV.
 */
#ifndef ITSX_B200_H
#define ITSX_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ITSX_OK        0
#define ITSX_ENODEV   -1   /* no CUDA device / wrong architecture */
#define ITSX_ECUDA    -2   /* CUDA runtime error (text in itsx_last_error) */
#define ITSX_EINVAL   -3   /* bad argument / call order */
#define ITSX_EIO      -4   /* cannot read a profile file */
#define ITSX_ECOLLIDE -5   /* unresolvable 64-bit key collision in derep (two independent hashes) */
#define ITSX_ELIMIT   -6   /* a fixed capacity was exceeded (domains per hit, model length) */
#define ITSX_EFORMAT  -7   /* malformed FASTQ (host scanner); text in itsx_host_last_error */

#define ITSX_MAXM      45  /* longest profile the DP kernels hold in registers (all ITSx_db profiles) */
#define ITSX_MAXDOM     8  /* envelopes kept per (sequence, profile) hit */
#define ITSX_CLUSTER_MAXD 64  /* largest edit band of itsx_cluster: reads up to ~6.4 kb at id 0.99 */

typedef struct itsx_ctx itsx_ctx;

/* hmmsearch thresholds as the reference passes them (SeqSample.py:191-209) */
typedef struct {
    float  T;        /* -T 10        per-sequence bit-score threshold              */
    double F1;       /* --F1 1e-6    MSV + bias filter P-value                      */
    double F2;       /* --F2 1e-6    Viterbi filter: runs on F2 < P(MSV + bias) <= F1, i.e. never when F1 == F2 */
    double F3;       /* --F3 1e-6    Forward filter P-value                         */
    double domE;     /* 10.0         per-domain conditional E-value (hmmsearch default) */
    int32_t resolve_multidomain; /* 1 (default): regions flagged multidomain are resolved like p7_domaindef does
                                  * (200 stochastic tracebacks, RNG seed 42, single-linkage clustering);
                                  * 0: such a region is rescored as one envelope */
    int32_t keep_rows;  /* what stays on the device until domZ is known (hmmsearch prints a domain iff
                         * P x domZ <= domE, domZ = reported hits of the profile over the WHOLE run):
                         *   1  every domain row (itsx_hits gives the full domtbl-equivalent table),
                         *   2  compact: a row whose P x domz_upper <= domE is printed whatever domZ turns out to
                         *      be, so ItsPosition's arg-max over those rows is taken at once; only rows that are
                         *      still undecided AND would beat that winner are kept.  Positions are identical;
                         *      itsx_hits then returns only the kept rows.  Memory per searched sequence drops
                         *      from ~3.5 KB (54 rows of 64 B) to < 100 B,
                         *   0  (default) 1 up to 200 000 searched sequences, 2 above. */
    int64_t domz_upper; /* upper bound of any profile's domZ for mode 2; 0 = the number of sequences this context
                         * searches (a sharded run passes the sample's read count) */
} itsx_search_params;

/* one domtbl-equivalent row (only the fields ItsPosition reads, plus diagnostics) */
typedef struct {
    int32_t seq;           /* index of the target among the searched (unique) sequences */
    int32_t prof;          /* index of the profile in load order (= runtime HMM file order) */
    int32_t ienv, jenv;    /* env from / env to, 1-based inclusive  (domtbl cols 19, 20) */
    int32_t tlen;          /* target length                         (domtbl col 2) */
    int32_t dom_idx;       /* 0-based index of the domain within its hit */
    float   bitscore;      /* domain bit score                      (domtbl col 13, before %.1f) */
    float   envsc;         /* envelope Forward score, nats */
    float   domcorrection; /* null2 correction, nats */
    float   seq_score;     /* per-sequence bit score of the hit */
    double  lnP;           /* ln P-value of the domain score */
    double  seq_lnP;       /* ln P-value of the hit (row order key within a profile) */
    int32_t is_multidomain;/* envelope comes from a region flagged multidomain */
    int32_t reported;      /* passes -T and domE (rows returned by itsx_hits always have 1) */
} itsx_dom_row;

/* counters of the last itsx_search (for GCUPS accounting and parity tests) */
typedef struct {
    int64_t n_seq, n_prof, n_pairs;
    int64_t n_past_msv, n_past_bias, n_past_fwd, n_hits_reported;
    int64_t n_domains, n_domains_reported, n_multidomain_regions, n_dom_overflow;
    double  msv_cells, bias_rows, fwd_cells, bck_cells, env_cells;   /* DP cells actually computed */
    /* device time per stage, milliseconds, CUDA events on the library's stream */
    float   ms_msv, ms_bias, ms_fwd, ms_mdom, ms_env, ms_final, ms_total;   /* ms_mdom: multidomain regions */
    float   reserved;
    /* selected left / right boundaries (ItsPosition winners) whose envelope came out of a region flagged
     * multidomain -- the only rows whose coordinates depend on the stochastic-traceback ensemble (DESIGN.md 2) */
    int64_t n_selected_multidomain;
    /* Viterbi filter (runs only when F2 < F1): pairs it was run on, pairs left after it, DP cells, device time */
    int64_t n_vit_run, n_past_vit;
    double  vit_cells;
    float   ms_vit, reserved2;
} itsx_search_stats;

typedef struct {
    int64_t n_reads, n_unique, n_collided;     /* n_collided: reads resolved by the second hash */
    int64_t bytes_ascii;                       /* sequence bytes hashed */
    float   ms_pack, ms_hash, ms_insert, ms_verify, ms_compact, ms_total;
} itsx_derep_stats;

/* ---- context ---------------------------------------------------------------------- */
int  itsx_create(int device, itsx_ctx **out);
void itsx_destroy(itsx_ctx *ctx);
const char *itsx_last_error(const itsx_ctx *ctx);   /* ctx may be NULL: error of the last failed create */
int  itsx_device_info(const itsx_ctx *ctx, int *sm_count, int *cc_major, int *cc_minor, int64_t *mem_bytes);
void *itsx_stream(const itsx_ctx *ctx);             /* the cudaStream_t all work is enqueued on */
int  itsx_sync(itsx_ctx *ctx);
/* page-locked host staging buffers (for callers that want DMA-able inputs/outputs) */
void *itsx_pinned_alloc(size_t bytes);
void itsx_pinned_free(void *p);

/* ---- profiles: replaces create_runtime_hmm + hmmsearch's file reader --------------- */
int  itsx_profiles_clear(itsx_ctx *ctx);
/* Append the profiles of a HMMER3/f ASCII file whose NAME starts with one of `prefixes`
 * (nprefix == 0: all), in file order (main.py:217-229).  Returns the number appended. */
int  itsx_profiles_append_file(itsx_ctx *ctx, const char *path, const char *const *prefixes, int nprefix);
int  itsx_profiles_count(const itsx_ctx *ctx);
const char *itsx_profile_name(const itsx_ctx *ctx, int p);
int  itsx_profile_M(const itsx_ctx *ctx, int p);
/* side[p]: 0 = left-boundary profile, 1 = right-boundary profile, -1 = ignored
 * (ItsPosition's prefix dispatch, SeqSample.py:388-398). */
int  itsx_profiles_set_sides(itsx_ctx *ctx, const int8_t *side, int n);
/* configured MSV byte profile for parity tests: cost[(M+1)*16], scalars {bias, base, tbm, tec} */
int  itsx_profile_msv(const itsx_ctx *ctx, int p, uint8_t *cost, int32_t *scalars4);

/* ---- dereplication ------------------------------------------------------------------ */
/* seq: reads packed back to back (ASCII, any case, IUPAC allowed); off[nreads+1].
 * rep_index[i] = index of the first read of i's class {s, revcomp(s)}; strand[i] = 0 '+', 1 '-'
 * (either output pointer may be NULL).  The reads and their representatives stay resident on
 * the device for itsx_search / itsx_trim_*. */
int  itsx_derep(itsx_ctx *ctx, const uint8_t *seq, const int64_t *off, int64_t nreads,
                int32_t *rep_index, uint8_t *strand, int64_t *n_unique);
/* clusters in first-occurrence order: first_read[u], abundance[u], u < n_unique */
int  itsx_derep_clusters(itsx_ctx *ctx, int32_t *first_read, int32_t *abundance);
/* 64-bit canonical key (strand-independent, case-insensitive) of every unique, same order as
 * itsx_derep_clusters: the owner rank of a class in the hash-partitioned multi-GPU derep is key % G. */
int  itsx_derep_unique_keys(itsx_ctx *ctx, uint64_t *keys);
/* the read -> representative map of the last derep (what Dedup.parse rebuilds from uc.txt, SeqSample.py:542-562):
 * rep_index[i] = first read of i's class, strand[i], uid[i] = dense class index in first-occurrence order (= row of
 * itsx_positions / itsx_derep_clusters).  Any may be NULL. */
int  itsx_derep_map(itsx_ctx *ctx, int32_t *rep_index, uint8_t *strand, int32_t *uid);
int  itsx_derep_get_stats(const itsx_ctx *ctx, itsx_derep_stats *st);
/* test hook: keep only the low `bits` bits of the 64-bit key (forces collisions); 64 = normal */
int  itsx_derep_set_key_bits(itsx_ctx *ctx, int bits);

/* ---- profile-HMM search --------------------------------------------------------------- */
void itsx_search_default_params(itsx_search_params *prm);
/* search the representatives of the last itsx_derep (device resident) */
int  itsx_search(itsx_ctx *ctx, const itsx_search_params *prm);
/* search caller-supplied sequences (the `_search(rep.fa)` entry): ASCII, off[nseq+1] */
int  itsx_search_seqs(itsx_ctx *ctx, const uint8_t *seq, const int64_t *off, int64_t nseq,
                      const itsx_search_params *prm);
int  itsx_search_get_stats(const itsx_ctx *ctx, itsx_search_stats *st);
/* reported rows in hmmsearch order (profile; ln P of the hit, then sequence index; domain
 * position).  rows may be NULL to query *n. */
int  itsx_hits(itsx_ctx *ctx, itsx_dom_row *rows, int64_t cap, int64_t *n);
int  itsx_nreported(itsx_ctx *ctx, int32_t *per_profile);           /* domZ per profile */
/* ItsPosition per searched sequence; -1 encodes None.  Any pointer may be NULL.
 * score10 = the "%.1f"-printed score in integer tenths (INT32_MIN when absent). */
int  itsx_positions(itsx_ctx *ctx, int32_t *start, int32_t *stop, int32_t *tlen,
                    int32_t *left_score10, int32_t *left_from, int32_t *left_to,
                    int32_t *right_score10, int32_t *right_from, int32_t *right_to);

/* multi-GPU: add other ranks' per-profile reported-hit counts (domZ is global per hmmsearch
 * run) between itsx_search_stage1 and itsx_search_stage2.  itsx_search == stage1 + stage2. */
int  itsx_search_stage1(itsx_ctx *ctx, const itsx_search_params *prm);
int  itsx_search_seqs_stage1(itsx_ctx *ctx, const uint8_t *seq, const int64_t *off, int64_t nseq,
                             const itsx_search_params *prm);
int  itsx_search_shard(itsx_ctx *ctx, int64_t first_unique, int64_t n_unique_local); /* restrict to a slice */
int  itsx_nreported_set(itsx_ctx *ctx, const int32_t *per_profile_global);
int  itsx_search_stage2(itsx_ctx *ctx);
/* install a position table computed elsewhere (all-gathered shards / a test fixture) */
int  itsx_positions_set(itsx_ctx *ctx, const int32_t *start, const int32_t *stop, const int32_t *tlen,
                        int64_t n);

/* ---- trim + re-expansion ---------------------------------------------------------------- */
/* Install a read -> unique map computed elsewhere (Dedup built from a uc.txt on disk, SeqSample.py:542-562,
 * or another rank's derep): uid[i] in [0, n_unique) or -1 (read absent from the map -> dropped,
 * SeqSample.py:817).  Replaces the map left by the last itsx_derep; the position table installed with
 * itsx_positions_set / itsx_search must then have n_unique rows. */
int  itsx_trim_set_map(itsx_ctx *ctx, const int32_t *uid, int64_t nreads, int64_t n_unique);
/* mode: 0 = single-end / merged record[start:stop]           (SeqSample.py:862)
 *       2 = paired R1  [start:stop] or [start:] if stop>tlen  (SeqSample.py:639-645)
 *       1 = paired R2  [tlen-stop : tlen-start]               (SeqSample.py:640,648-655)
 * Bounds for every read of the last itsx_derep in input order; keep[i] = 1 iff the read's
 * representative has both boundaries and start < stop (SeqSample.py:814-825).
 * off_other: offsets of the R1/R2 file being sliced when it is not the dereplicated one
 * (NULL: slice the dereplicated reads themselves).  Returns the number kept in *n_kept. */
int  itsx_trim_bounds(itsx_ctx *ctx, int mode, const int64_t *off_other, int64_t nreads,
                      uint8_t *keep, int32_t *lo, int32_t *hi, int64_t *n_kept);
/* gather the kept slices of (seq, qual) into back-to-back output buffers on the device and copy
 * them out: out_off[n_kept+1], out_seq/out_qual sized >= total (query with NULLs first via
 * *total).  seq/qual: the records being sliced (host), off: their offsets. */
int  itsx_trim_gather(itsx_ctx *ctx, int mode, const uint8_t *seq, const uint8_t *qual, const int64_t *off,
                      int64_t nreads, int64_t *n_kept, int64_t *total,
                      int32_t *kept_index, int64_t *out_off, uint8_t *out_seq, uint8_t *out_qual);

/* the same for the RESIDENT reads (itsx_reads_upload / itsx_quals_upload, after itsx_search or itsx_shard_apply): the
 * gathered slices stay on the device; itsx_run_fetch copies them out */
int  itsx_trim_gather_resident(itsx_ctx *ctx, int mode, int64_t *n_kept, int64_t *total);

/* ---- paired-end merge (SURVEY 8f row 2) ------------------------------------------------------------------
 * Replaces the `vsearch --fastq_mergepairs R1 --reverse R2 --fastqout seq.fq --fastq_maxdiffs 40 --fastq_maxee 2
 * [--fastq_allowmergestagger] --fastq_qmax 93` process of SeqSamplePairedNotInterleaved._merge_reads
 * (SeqSample.py:266-365; constants definitions.py:79,82). */
enum { ITSX_MERGE_OK = 0, ITSX_MERGE_REPEAT, ITSX_MERGE_STAGGERED, ITSX_MERGE_MAXDIFFS, ITSX_MERGE_MAXDIFFPCT,
       ITSX_MERGE_NOKMERS, ITSX_MERGE_MINSCORE, ITSX_MERGE_MINOVLEN, ITSX_MERGE_MAXEE, ITSX_MERGE_BADQUAL };
typedef struct {
    int32_t maxdiffs;        /* --fastq_maxdiffs 40           definitions.py:79, SeqSample.py:322 */
    int32_t allow_stagger;   /* --fastq_allowmergestagger     SeqSample.py:328 */
    int32_t qmax;            /* --fastq_qmax 93               definitions.py:82, SeqSample.py:330 */
    int32_t minovlen, qmaxout, qminout, ascii;   /* vsearch defaults the reference leaves alone: 10, 41, 0, 33 */
    int32_t reserved;
    double  maxee;           /* --fastq_maxee 2               SeqSample.py:324 */
    double  maxdiffpct;      /* vsearch default 100 */
} itsx_merge_params;
typedef struct {
    int64_t n_pairs, n_merged;
    int64_t by_reason[16];   /* pairs per ITSX_MERGE_* outcome (what vsearch prints as its merge statistics) */
    int64_t bytes_in, bytes_out;   /* bases + qualities read / written by the merge kernel */
    float   ms_kernel;       /* merge_kernel alone, CUDA events on the library's stream */
} itsx_merge_stats;
void itsx_merge_default_params(itsx_merge_params *prm);
/* fseq/fqual with foff[npairs+1]: R1 records; rseq/rqual with roff[npairs+1]: R2 records as they stand in the file
 * (the library reverse-complements).  merged_len[i] = length of pair i's merged read or 0, reason[i] = ITSX_MERGE_*
 * (either may be NULL).  *n_merged pairs with *total bases stay resident for itsx_merge_fetch.  A quality value
 * outside [0, qmax] -- where vsearch stops with a fatal error -- returns ITSX_EFORMAT. */
int  itsx_merge_pairs(itsx_ctx *ctx, const uint8_t *fseq, const uint8_t *fqual, const int64_t *foff,
                      const uint8_t *rseq, const uint8_t *rqual, const int64_t *roff, int64_t npairs,
                      const itsx_merge_params *prm, int32_t *merged_len, uint8_t *reason, int64_t *n_merged,
                      int64_t *total);
/* merged reads of the last itsx_merge_pairs in input order, packed back to back: merged_index[n_merged] = pair
 * index (the title vsearch writes is R1's), out_off[n_merged+1], out_seq / out_qual [total].  Any may be NULL. */
int  itsx_merge_fetch(itsx_ctx *ctx, int32_t *merged_index, int64_t *out_off, uint8_t *out_seq, uint8_t *out_qual);
int  itsx_merge_get_stats(const itsx_ctx *ctx, itsx_merge_stats *st);

/* ---- gzip reader (inflate_host.cpp, host only) -----------------------------------------------------------------
 * Replaces gzip.open(path, "rt") under SeqIO.parse (SeqSample.py:742-752, 767-788; main.py:295-330), used like gzread:
 * itsx_gz_open over the bytes of a gzip file (one or more members; the memory must stay valid until itsx_gz_close),
 * then itsx_gz_read until it returns 0.  `threads` > 1 inflates ONE deflate stream on several host cores (chunks that
 * find their own block starts, 16-bit symbols with markers for the unknown window, resolved front to back); 1 is a
 * single-core decoder, 0 = every core.  itsx_gz_read fills dst with up to cap bytes and returns how many (it may return
 * fewer than cap before the end), 0 at the end of the stream, or
 * ITSX_EFORMAT for anything that is not a valid gzip stream (CRC-32 and ISIZE of every member are checked; the error is
 * sticky).  `hist`: how many bytes right in front of dst are the output of the preceding calls, untouched (0 when dst is a
 * fresh buffer): with 32 KB of them in place the stream is decoded straight into dst, otherwise through a bounce buffer
 * until the call itself has written that much. */
typedef struct itsx_gz itsx_gz;
itsx_gz *itsx_gz_open(const uint8_t *src, int64_t n, int threads);
int64_t  itsx_gz_read(itsx_gz *h, uint8_t *dst, int64_t cap, int64_t hist);
int      itsx_gz_eof(const itsx_gz *h);
/* chunking of the multi-core mode (compressed bytes per chunk, least input worth several cores; the tests shrink them) and
 * its counters (what = 0: batches decoded on several cores, 1: chunks decoded again because a block start was none) */
int      itsx_gz_tune(itsx_gz *h, int64_t chunk_min, int64_t chunk_max, int64_t par_min);
int64_t  itsx_gz_stat(const itsx_gz *h, int what);
void     itsx_gz_close(itsx_gz *h);

/* ---- gzip writer (deflate.cu) ------------------------------------------------------------------------------------
 * Replaces the compression inside the reference's output writers: gzip.open(outfile, "wt") around SeqIO.write in
 * Dedup.create_trimmed_seqs / create_paired_trimmed_seqs (SeqSample.py:767-788, 926-949) and the .fastq.gz files of the
 * QIIME 2 actions (q2_itsxpress.py:311-333).  src[n] (host or device) becomes a multi-member gzip stream in dst (every
 * 1 MiB of input one member of 32 byte-aligned dynamic-Huffman deflate blocks, with its CRC-32 and ISIZE; a valid gzip
 * file that any reader inflates to src).  cap must be at least itsx_gzip_bound(n); *dst_n receives the stream's length. */
int64_t itsx_gzip_bound(int64_t n);
int  itsx_gzip_compress(itsx_ctx *ctx, const uint8_t *src, int64_t n, uint8_t *dst, int64_t cap, int64_t *dst_n);

/* ---- whole path, host buffers in / host buffers out (the calls bench.py's e2e leg times) --
 * Together they replace main.py:534-624 for one sample: deduplicate -> _search -> ItsPosition -> Dedup ->
 * create_trimmed_seqs (SeqSample.py:93-131, 178-225, 380-498, 517-562, 792-949). */
typedef struct {
    int64_t n_reads, n_unique, n_kept, out_bytes;
    float   ms_h2d, ms_derep, ms_search, ms_trim, ms_d2h, ms_total;
    float   ms_gather, reserved;     /* re-expansion of the kept slices (itsx_run_trim, resident runs with qualities) */
} itsx_run_stats;
/* derep + search + positions + single-end trim bounds.  Outputs: rep_index[nreads], keep[nreads],
 * lo[nreads], hi[nreads] (any may be NULL). */
int  itsx_run(itsx_ctx *ctx, const uint8_t *seq, const int64_t *off, int64_t nreads,
              const itsx_search_params *prm, int32_t *rep_index, uint8_t *keep, int32_t *lo, int32_t *hi,
              itsx_run_stats *st);
/* the same followed by the re-expansion: bases AND qualities go in, the kept reads' trimmed bases and qualities come
 * back packed in input order -- what Dedup.create_trimmed_seqs writes (SeqSample.py:792-949) minus the titles, which
 * never leave the host.  Output buffers must hold the worst case: kept_index[nreads], out_off[nreads + 1],
 * out_seq / out_qual [off[nreads]] (every read kept whole); st->n_kept / st->out_bytes say how much was written.
 * rep_index may be NULL. */
int  itsx_run_trim(itsx_ctx *ctx, const uint8_t *seq, const uint8_t *qual, const int64_t *off, int64_t nreads,
                   const itsx_search_params *prm, int32_t *rep_index, int32_t *kept_index, int64_t *out_off,
                   uint8_t *out_seq, uint8_t *out_qual, itsx_run_stats *st);
/* the same with the reads already resident (itsx_reads_upload [+ itsx_quals_upload]): kernels only.  With the
 * qualities resident the run ends with the re-expansion and itsx_run_fetch copies its result out. */
int  itsx_reads_upload(itsx_ctx *ctx, const uint8_t *seq, const int64_t *off, int64_t nreads);
int  itsx_quals_upload(itsx_ctx *ctx, const uint8_t *qual);      /* qual[off[nreads]] of the resident reads */
/* Streamed upload -- a FASTQ file too large to sit parsed in host memory (BASELINE configs[3]: 70 GB of text) arrives in
 * chunks: the host reader parses a chunk into pinned buffers while the previous one is on its way (the reference streams
 * the file through Biopython the same way, SeqSample.py:742-752, 908-949).  begin (hints size the first allocation) ->
 * append chunk after chunk (off[nreads + 1] chunk-relative, off[0] = 0; qual may be NULL) -> end.  The reads are then
 * resident exactly as after itsx_reads_upload [+ itsx_quals_upload].  itsx_reads_append returns once the chunk's
 * buffers are free again. */
int  itsx_reads_begin(itsx_ctx *ctx, int64_t nreads_hint, int64_t bases_hint);
int  itsx_reads_append(itsx_ctx *ctx, const uint8_t *seq, const uint8_t *qual, const int64_t *off, int64_t nreads);
int  itsx_reads_end(itsx_ctx *ctx, int64_t *nreads, int64_t *total_bases);
/* ... and the chunked way out: keep filter + re-expansion of the resident reads [first, first + count) only (mode 0);
 * kept_index is relative to `first`.  Output buffers: worst case count / count + 1 / the range's bases. */
int  itsx_trim_gather_range(itsx_ctx *ctx, int mode, int64_t first, int64_t count, int64_t *n_kept, int64_t *total,
                            int32_t *kept_index, int64_t *out_off, uint8_t *out_seq, uint8_t *out_qual);
/* Several samples in one pass (the loop over samples of q2_itsxpress.py:273-333 runs one vsearch and one hmmsearch PER
 * SAMPLE: classes never span samples and domZ is per sample): sample_of_read[nreads] in [0, n_samples) for the resident
 * reads, set before itsx_derep_resident.  The search then counts reported hits per (sample, profile) -- itsx_nreported /
 * itsx_nreported_set carry n_samples x n_profiles values, sample-major -- and every later call works on the concatenated
 * reads in input order.  Reset by the next itsx_reads_upload. */
int  itsx_reads_set_samples(itsx_ctx *ctx, const int32_t *sample_of_read, int32_t n_samples);
/* exact dereplication of the resident reads (what itsx_derep does after its upload); build_search_set = 0 skips the
 * re-coding of the representatives for a context that will not search them (the block side of a sharded run) */
int  itsx_derep_resident(itsx_ctx *ctx, int build_search_set, int64_t *n_unique);
int  itsx_run_resident(itsx_ctx *ctx, const itsx_search_params *prm, itsx_run_stats *st);
int  itsx_run_fetch(itsx_ctx *ctx, int64_t *n_kept, int64_t *total, int32_t *kept_index, int64_t *out_off,
                    uint8_t *out_seq, uint8_t *out_qual);
/* ---- clustering below 100 % identity: replaces `vsearch --cluster_size --id X --strand both` (SeqSample.py:133-176) ----
 * Runs on the exact classes of the resident derep (itsx_derep / itsx_derep_resident).  Classes are taken in
 * `order` (unique indices in processing order; NULL = abundance descending, then first occurrence).  ed is unit-cost
 * Levenshtein distance over the derep's normalised residues, min over both strands of the later class ('+' on a tie);
 * with L the longer length a pair is accepted iff (L - ed) / L >= id.  A class becomes a centroid iff no earlier centroid
 * accepts it; otherwise it joins the accepted earlier centroid of highest identity, the earliest on a tie.  Exhaustive:
 * no k-mer heuristics, terminal gaps count (DESIGN.md §6).
 * Afterwards the search set is the centroids' first reads in processing order (row r = r-th centroid), and the resident
 * read -> row map that itsx_trim_* / itsx_derep_map read gives every read its centroid's row; itsx_derep_clusters still
 * returns the exact classes.  ITSX_ELIMIT when the longest class allows more than ITSX_CLUSTER_MAXD edits.
 * Several samples (itsx_reads_set_samples): per_sample = 1 clusters every sample on its own in the same call, and with
 * sample ids set per_sample = 0 is ITSX_EINVAL; without sample ids per_sample has no effect.  A class is then compared
 * only with classes of its own sample (the sample id seeds the index keys, and a hit of another sample is dropped before
 * verification), so each sample gets exactly the centroids, per-class centroid / strand / ed and relative order of
 * centroid rows that a call on that sample alone gives with `order` restricted to it.  `order` is any permutation of
 * the unique indices (the samples need not be contiguous in it; the default order restricts to the default order of
 * each sample alone), centroid rows follow it across samples, and every centroid row of the search set keeps its
 * sample, so itsx_search counts domZ per (sample, profile) over the centroids. */
typedef struct {
    double  id;             /* identity threshold, 0.5 < id <= 1 */
    int32_t strand_both;    /* must be 1 */
    int32_t per_sample;     /* 1: cluster each sample on its own when sample ids are set (else they are refused) */
} itsx_cluster_params;
typedef struct {
    int64_t n_unique, n_centroids;
    int64_t n_segments;     /* pigeonhole index entries */
    int64_t n_candidates;   /* candidate pairs emitted by the index lookups (with repeats) */
    int64_t n_verified;     /* distinct candidate pairs given to the banded edit distance */
    int64_t n_accepted;     /* pairs within the identity threshold */
    int64_t n_rounds;       /* resolution rounds */
    int32_t d_max;          /* D(L) of the longest class */
    int32_t n_len_slots;    /* partner lengths looked up per class and strand */
    float   ms_index, ms_candidates, ms_verify, ms_resolve, ms_remap, ms_total;
} itsx_cluster_stats;
int  itsx_cluster(itsx_ctx *ctx, const itsx_cluster_params *prm, const int32_t *order, int64_t *n_centroids);
/* per unique (first-occurrence order): row of its centroid, strand relative to it (0 '+', 1 '-'), ed to it; per row:
 * the unique index of the centroid.  Any pointer may be NULL. */
int  itsx_cluster_fetch(itsx_ctx *ctx, int32_t *centroid_row_of_unique, uint8_t *strand_of_unique, int32_t *ed_of_unique,
                        int32_t *unique_of_row);
int  itsx_cluster_get_stats(const itsx_ctx *ctx, itsx_cluster_stats *st);
/* test hook: keep only the low `bits` bits of the segment keys of itsx_cluster (forces key collisions, also between
 * samples); 64 = normal */
int  itsx_cluster_set_key_bits(itsx_ctx *ctx, int bits);
/* host only: dmax[L] = the largest ed with (L - ed) / L >= id for L = 0 .. lmax (the acceptance table of itsx_cluster) */
int  itsx_cluster_dtable(double id, int32_t lmax, int32_t *dmax);
/* number of kernel launches issued by this ctx so far (bench.py's gpu_launches) */
int64_t itsx_launch_count(const itsx_ctx *ctx);

/* ---- one sample sharded over the G GPUs of a box (SURVEY 8e) ---------------------------------------------------
 * vsearch --fastx_uniques and hmmsearch are global over a sample (SeqSample.py:106-116, 191-209): first occurrence
 * of a class, per-profile domZ.  A rank holds a contiguous block of the reads in a LOCAL context and the classes
 * whose key64 % G equals its rank in an OWNER context; the host driver (itsxpress_b200/distributed.py) moves the
 * buffers below with two NCCL all-to-alls and one all-reduce.  Every buffer may be device memory.
 *   local:  itsx_reads_upload, itsx_derep_resident(0), itsx_shard_plan, itsx_shard_pack
 *   owner:  itsx_shard_owner_derep, itsx_search_stage1, [all-reduce nreported], itsx_nreported_set,
 *           itsx_search_stage2, itsx_shard_answers
 *   local:  itsx_shard_apply, itsx_trim_bounds / itsx_trim_gather */
/* per destination rank g: records (local uniques owned by g) and their bases; one D2H of 2 G counters */
int  itsx_shard_plan(itsx_ctx *local, int G, int64_t *rec_counts, int64_t *byte_counts);
/* rec[n_unique_local]: (global read index of the unique's first read) | (length << 32), grouped by owner, ascending
 * index inside a group; bases[sum byte_counts]: their bases back to back in the same order */
int  itsx_shard_pack(itsx_ctx *local, int64_t first_global_index, uint64_t *rec, uint8_t *bases);
/* the records / bases received from all ranks in source-rank order (= ascending global read index) become the owner
 * context's read set: exact derep (first arrival = first occurrence), the classes become its search set */
int  itsx_shard_owner_derep(itsx_ctx *owner, const uint64_t *rec, int64_t nrec, const uint8_t *bases, int64_t nbytes,
                            int64_t *n_own);
/* after itsx_search_stage2: ans[nrec][4] = {global index of the class representative | strand << 31, start, stop,
 * tlen} (-1 = None) per received record, arrival order */
int  itsx_shard_answers(itsx_ctx *owner, int64_t nrec, int32_t *ans);
/* the answers that came back (same order as itsx_shard_pack's records) become the local context's position table
 * (one row per local unique); rep_global[nreads] / strand[nreads] (may be NULL): the global class representative
 * and strand of every read of the block */
int  itsx_shard_apply(itsx_ctx *local, const int32_t *ans, int64_t n_unique_local, int64_t *rep_global,
                      uint8_t *strand);

/* ---- host-side FASTQ scanner / packer / formatter (multi-threaded C++, no GPU involved) -------------
 * Replace Biopython's SeqIO.parse / SeqIO.write on the path (SeqSample.py:746-757, 912-945): a decompressed
 * 4-line FASTQ buffer -> offset arrays (title after '@' right-stripped, sequence, quality), packed byte
 * streams for itsx_derep / itsx_trim_*, and FASTQ text from the slices itsx_trim_gather returns. */
const char *itsx_host_last_error(void);
/* cap == 0: count records only.  Returns the record count or ITSX_EFORMAT / ITSX_EINVAL. */
int64_t itsx_fastq_index(const uint8_t *buf, int64_t nbytes, int64_t cap, int64_t *t_off, int32_t *t_len,
                         int64_t *s_off, int32_t *s_len, int64_t *q_off);
/* Where a chunked reader may cut a piece of a 4-line FASTQ file that starts at a record boundary: the offset behind the
 * last line whose number is a multiple of four (0: fewer than four lines).  Lines are counted, not recognised -- a quality
 * line may begin with '@' (SeqSample.py:742-752 streams through Biopython, which counts too). */
int64_t itsx_fastq_cut(const uint8_t *buf, int64_t nbytes);
/* out_off[n+1] = prefix sums of len; out (may be NULL) = segments packed back to back.  Returns total bytes. */
int64_t itsx_bytes_gather(const uint8_t *buf, const int64_t *off, const int32_t *len, int64_t n, uint8_t *out,
                          int64_t *out_off);
/* The files vsearch hands to the next stage (SeqSample.py:104-119; SURVEY.md Appendix B), from the arrays itsx_derep returns:
 * itsx_fastq_labels = Biopython's record.id of every record (title.split(None, 1)[0]) as (offset into buf, length);
 * itsx_uc_format = uc.txt of --fastx_uniques (S / H rows per cluster in `order`, then the C rows);
 * itsx_repfa_format = rep.fa (>label, sequence wrapped at `width` = 80).  Both return the bytes written to dst or ITSX_ELIMIT. */
int64_t itsx_fastq_labels(const uint8_t *buf, const int64_t *t_off, const int64_t *t_len, int64_t n, int64_t *lab_off,
                          int32_t *lab_len);
int64_t itsx_uc_format(const int32_t *rep, const uint8_t *strand, const int64_t *len, int64_t n, const int64_t *order, int64_t nc,
                       const uint8_t *buf, const int64_t *lab_off, const int32_t *lab_len, uint8_t *dst, int64_t cap);
int64_t itsx_repfa_format(const uint8_t *buf, const int64_t *s_off, const int64_t *s_len, const int64_t *lab_off,
                          const int32_t *lab_len, const int64_t *order, int64_t nc, int32_t width, uint8_t *dst, int64_t cap);
/* domtbl.txt body -- hmmsearch --domtblout rows (SeqSample.py:190; the six fields ItsPosition reads at :445-450 carry the
 * computed values) -- from the rows of itsx_hits.  Labels: byte strings with offsets (no terminators); Z = searched
 * sequences, nreported = itsx_nreported (domZ).  Returns the bytes written to dst, ITSX_ELIMIT if cap is too small. */
int64_t itsx_domtbl_format(const itsx_dom_row *rows, int64_t nrows, const uint8_t *seq_lab, const int64_t *seq_off,
                           const uint8_t *prof_lab, const int64_t *prof_off, const int32_t *prof_M, const int32_t *nreported,
                           double Z, uint8_t *dst, int64_t cap);
/* '@title\nseq\n+\nqual\n' for nkeep records (dst == NULL: size query); pre_ and suf_ (lp, ls bytes) are stitched to
 * every record's bases and qualities (--trim-ccs, SeqSample.py:601-622).  Returns the number of bytes. */
int64_t itsx_fastq_format(const uint8_t *buf, const int64_t *t_off, const int32_t *t_len, const int32_t *keep_idx,
                          int64_t nkeep, const int64_t *out_off, const uint8_t *out_seq, const uint8_t *out_qual,
                          const uint8_t *pre_s, const uint8_t *pre_q, int32_t lp, const uint8_t *suf_s,
                          const uint8_t *suf_q, int32_t ls, uint8_t *dst);

#ifdef __cplusplus
}
#endif
#endif
