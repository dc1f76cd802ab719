/*
 * mcx.h -- C ABI of libmcx.so, the B200 (sm_100a) replacement for the translated marker search of
 * MicrobeCensus.  Plain pointers and sizes only; no C++/torch types cross this boundary.
 *
 * What each entry point replaces in the reference (/root/reference/microbe_census/microbe_census.py = mc.py):
 *
 *   mcx_create / mcx_destroy     loading of data/rapdb_2.15 by the RAPsearch2 child process
 *                                (command line built at mc.py:375; DB made by prerapsearch,
 *                                training/search_reads.py:50)
 *   mcx_set_params               args['read_length'|'quality_offset'|'min_quality'|'mean_quality'|
 *                                'max_unknown'|'filter_dups'] (mc.py:189-224) and the per-family cutoff
 *                                rows find_opt_pars() returns (mc.py:61-72)
 *   mcx_push_reads[_packed][_dev] process_seqfile()'s per-read filter chain (mc.py:328-356) and
 *                                quality_filter() (mc.py:265-279); the reads are what the reference
 *                                writes to its FASTA tempfile (mc.py:352)
 *   mcx_qc_counts                the too_short / low_qual / dups / read_id counters (mc.py:336, 363-367)
 *   mcx_search                   search_seqs() (mc.py:369-389, the rapsearch child) + classify_reads()
 *                                (mc.py:432-460) + aggregate_hits() (mc.py:462-472), with the `-n` cut
 *                                (mc.py:356) applied as a quota of kept reads
 *   mcx_result                   args['sampled_reads'] (mc.py:362), "reads hit marker proteins"
 *                                (mc.py:386), "reads assigned" (mc.py:459) and agg_hits (mc.py:620)
 *   mcx_get_hits                 the lines of the .m8 file RAPsearch2 writes (mc.py:391-398)
 *   mcx_last_error               stderr of the child (mc.py:389)
 *
 * All functions return 0 on success or a negative MCX_E* code; nothing throws across the ABI.
 * A context is bound to one CUDA device and is not re-entrant.  There is no CPU fallback: every
 * entry point that computes fails with MCX_ECUDA when no usable device is present.
 */
#ifndef MCX_H
#define MCX_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MCX_OK        0
#define MCX_EINVAL   -1   /* bad argument */
#define MCX_ECUDA    -2   /* CUDA runtime error / no device */
#define MCX_ESTATE   -3   /* call out of order */
#define MCX_ENOMEM   -4   /* a device buffer overflowed; the message names it */

#define MCX_N_FAM    30
#define MCX_LEN_BINS 1280 /* subject lengths are < 1280 (max 1183) */

typedef struct mcx_ctx mcx_ctx;

/* marker database: caller-owned host arrays, copied by mcx_create */
typedef struct {
    int32_t        n_subj;
    const int32_t *off;      /* n_subj + 1 residue offsets */
    const uint8_t *res;      /* residue codes 0..19 (ARNDCQEGHILKMFPSTWYV), 20 = X */
    const uint8_t *fam;      /* family index 0..29 per subject */
} mcx_db;

/* cutoffs of one family at the current read length (one pars.map row) */
typedef struct {
    double  min_cov;         /* aln_cov      */
    double  max_aaid;        /* max_aaid     */
    int32_t min_raw;         /* smallest raw score whose printed bit score reaches score_cutoff */
    int32_t stat;            /* 0 hits, 1 cov, 2 aln */
} mcx_cutoff;

typedef struct {
    int32_t read_length;     /* -l : one of the 20 lengths of read_len.map */
    int32_t has_quality;     /* 1 for FASTQ input */
    int32_t quality_offset;  /* 33 / 64 style offset (args['quality_offset']) */
    int32_t min_quality;     /* -q */
    int32_t mean_quality;    /* -m */
    int32_t max_unknown;     /* -u */
    int32_t filter_dups;     /* -d */
    int32_t min_report_raw;  /* raw score floor of reported HSPs (RAPsearch2 -e 1 at this length) */
    mcx_cutoff cut[MCX_N_FAM];
} mcx_params;

typedef struct {
    int64_t n_reads;         /* reads pushed */
    int64_t kept;            /* reads passing all filters (before the -n cut) */
    int64_t too_short, low_qual, dups;
} mcx_qc;

typedef struct {
    int64_t sampled_reads;   /* reads searched (kept reads up to the quota) */
    int64_t too_short, low_qual, dups;   /* counted up to the read that filled the quota */
    int64_t reads_with_hits; /* reads with at least one reported HSP */
    int64_t reads_classified;
    int64_t n_hsp;           /* reported HSPs ("m8 lines") */
    int64_t n_seed_hits;     /* seeds whose ungapped extension reached the report floor */
    int64_t n_gapped;        /* gapped X-drop extensions run */
    int64_t gapped_cells;    /* DP cells evaluated by them */
    int64_t n_capped_reads;  /* reads with more than 500 reportable lines (RAPsearch2 -v 500: the lowest were dropped) */
    int64_t fam_hits[MCX_N_FAM];          /* classified reads per family */
    int64_t fam_aln[MCX_N_FAM];           /* sum of aln-len per family */
    int64_t aln_by_len[MCX_N_FAM * MCX_LEN_BINS]; /* sum of aln-len per (family, subject length) */
} mcx_result;

/* one reported HSP, the fields of an m8 line before formatting */
typedef struct {
    int32_t read;            /* index among the pushed reads */
    int32_t subject;
    int32_t frame;           /* 0..2 forward, 3..5 reverse complement */
    int32_t score;           /* raw */
    int32_t aln, ident, mism, gapo;
    int32_t q0, q1;          /* 0-based inclusive aa range on the frame */
    int32_t t0, t1;          /* 0-based inclusive aa range on the subject */
} mcx_hit;

int  mcx_create(mcx_ctx **out, const mcx_db *db, int device);
void mcx_destroy(mcx_ctx *ctx);
int  mcx_set_params(mcx_ctx *ctx, const mcx_params *p);
/* run on the caller's CUDA stream (a cudaStream_t, e.g. torch.cuda.current_stream().cuda_stream) instead of
 * the context's own; lets the caller bracket calls with its own CUDA events */
int  mcx_set_stream(mcx_ctx *ctx, void *cuda_stream);

/* Reads as 2-bit bases + mask in bit-planes of 32 bases -- the layout the reads have in HBM and the one the host
 * reader (libmcxio) and the synthetic generator produce.  Read i of lengths[i] bases owns 3 G words, G =
 * ceil(lengths[i] / 32), stored back to back in read order: lo[G], hi[G], mask[G].  Bit k of lo / hi = low / high bit of
 * the code of base k (T 0, C 1, A 2, G 3); a mask bit marks a base that is not an upper-case A, C, G or T, and under it
 * lo = 0 means 'N' (the character mc.py:269 counts), lo = 1 anything else (hi = 0); bits past the length are zero.
 * quals (NULL for FASTA) holds one byte per base, all reads back to back; n_words / n_bases are the sizes of the two
 * arrays (= sum of 3 G / sum of lengths).  Host pointers; pinned memory (mcx_host_alloc) makes the call asynchronous: it
 * returns once the copies are queued on the context's copy stream, and mcx_search consumes the reads chunk by chunk as
 * they arrive, so the copy of later reads overlaps the search of earlier ones.  The buffers must stay valid and
 * unchanged until the next call that waits for them (mcx_search, or any mcx_qc_* call).  Replaces any reads pushed before. */
int  mcx_push_reads_packed(mcx_ctx *ctx, const uint32_t *packed, int64_t n_words, const uint32_t *lengths,
                           const uint8_t *quals, int64_t n_bases, int64_t n);
/* same with device-resident buffers (no copy; d_quals 16-byte aligned; the buffers stay the caller's) */
int  mcx_push_reads_packed_dev(mcx_ctx *ctx, const uint32_t *d_packed, int64_t n_words, const uint32_t *d_lengths,
                               const uint8_t *d_quals, int64_t n_bases, int64_t n);
/* Reads as ASCII bytes, read i = bases[offsets[i] .. offsets[i+1]); quals may be NULL (FASTA) and
 * otherwise shares the offsets.  Host pointers (pinned or pageable).  The device packs them into the layout above
 * (k_pack_ascii).  Replaces any reads pushed before. */
int  mcx_push_reads(mcx_ctx *ctx, const uint8_t *bases, const uint8_t *quals,
                    const int64_t *offsets, int64_t n);
/* same with device-resident buffers (no host->device copy; d_quals 16-byte aligned) */
int  mcx_push_reads_dev(mcx_ctx *ctx, const uint8_t *d_bases, const uint8_t *d_quals,
                        const int64_t *d_offsets, int64_t n, int64_t total_bytes);
/* page-locked host memory for the push buffers (cudaHostAlloc, portable across the GPUs of the box) */
int  mcx_host_alloc(void **out, size_t bytes);
void mcx_host_free(void *p);

/* verdict counts over ALL pushed reads.  Forces the QC of every pushed read (and so waits for every copy of the
 * push): a caller that does not need them before the search should not ask -- mcx_result carries the counts the
 * reference prints (up to the read that filled -n). */
int  mcx_qc_counts(mcx_ctx *ctx, mcx_qc *out);
/* Per-read verdicts of the pushed reads (0 keep, 1 too short, 2 low quality, 3 duplicate) and, optionally,
 * the 128-bit strand-canonical fingerprints of the untrimmed reads (2 x uint64 per read) to host memory;
 * mcx_qc_import replaces the verdicts (e.g. duplicates decided across GPUs, mc.py:345) and rebuilds the kept list. */
int  mcx_qc_export(mcx_ctx *ctx, uint8_t *code, uint64_t *fingerprints);
int  mcx_qc_import(mcx_ctx *ctx, const uint8_t *code);
/* The same without leaving the device: *d_code = the n verdict bytes, *d_fingerprints (optional) = n records of 24 bytes
 * {uint64 a, uint64 b, uint32 read index, uint32 0}, both in HBM and owned by the context.  The caller may rewrite the
 * verdicts in place (on the context's stream or after synchronising) and then calls mcx_qc_refresh to rebuild the kept
 * list.  Used by the cross-GPU duplicate exchange, which never brings fingerprints to the host. */
int  mcx_qc_device(mcx_ctx *ctx, void **d_code, void **d_fingerprints, int64_t *n);
int  mcx_qc_refresh(mcx_ctx *ctx);
/* -d over several pushes (batches of one run): the context remembers the fingerprints of the reads it has kept -- after
 * every mcx_search with filter_dups set, and on the owner side of mcx_dedup_owner -- and later pushes are tested against
 * them as well (mc.py:345 keeps one set for the whole run).  mcx_set_params and mcx_dedup_reset forget them (start of a run). */
int  mcx_dedup_reset(mcx_ctx *ctx);
/* -d across GPUs (one context per GPU, reads sharded; mc.py:345 decided over all of them).  Three compute steps on the
 * device with two all-to-all transfers by the caller in between (NCCL; microbecensus_b200/distributed.py):
 *   mcx_dedup_begin   QC of all pushed reads, fingerprints, records {uint64 a, uint64 b, int64 global index << 1 |
 *                     passed-QC} of the long-enough reads grouped by owner rank (a mod world); *d_send = the records
 *                     (device memory of the context), send_counts[world] = records per owner (host);
 *   mcx_dedup_owner   d_recv = the m records this rank owns (device memory of the caller); sorts them by (fingerprint,
 *                     global index) and marks every record behind the first QC-passing read of its fingerprint;
 *                     *d_marks = m bytes in the order of d_recv (device memory of the context);
 *   mcx_dedup_finish  d_marks_back = the marks of this rank's own records in the order of *d_send; rewrites the
 *                     verdicts (3 = duplicate) and recounts.
 * first_index = global index of this rank's first read. */
int  mcx_dedup_begin(mcx_ctx *ctx, int world, int64_t first_index, void **d_send, int64_t *send_counts);
int  mcx_dedup_owner(mcx_ctx *ctx, const void *d_recv, int64_t m, void **d_marks);
int  mcx_dedup_finish(mcx_ctx *ctx, const void *d_marks_back);
/* search the first `quota` kept reads (quota < 0: all of them) */
int  mcx_search(mcx_ctx *ctx, int64_t quota);
int  mcx_result_get(mcx_ctx *ctx, mcx_result *out);
/* reported HSPs of the last search, ordered by (read, subject, score desc); *n receives the total */
int  mcx_get_hits(mcx_ctx *ctx, mcx_hit *out, int64_t cap, int64_t *n);
/* per pushed read: subject of the best passing hit or -1 */
int  mcx_get_classified(mcx_ctx *ctx, int32_t *best_subject, int64_t n);

/* device time (ms, CUDA events on the context's stream) of the stages of the last push/search:
 * [0] h2d copy, [1] k_qc + compaction, [2] k_probe + k_resolve, [3] gapped stage (k_gap_*), [4] sort, [5] classifier (k_cls_*),
 * [6] d2h, [7] k_seed + k_walk, [8] k_frames, [9] k_seg, [10] k_qc alone (part of [1]), [11] -d: fingerprints + sort + marks
 * (part of [1]); and the number of kernel launches.  [0] is the span of the copies on the copy stream: they overlap
 * the other stages. */
int  mcx_timings(mcx_ctx *ctx, float ms[12], int64_t *launches);
/* the seed stage kernel by kernel: [0] k_probe (filter), [1] k_resolve (tables + postings), [2] k_seed, [3] k_walk;
 * [0] + [1] = mcx_timings [2], [2] + [3] = mcx_timings [7] */
int  mcx_timings_detail(mcx_ctx *ctx, float ms[4]);
/* queue lengths of the last search (what the kernels between the stages worked on; the roofline figures of bench.py are
 * formed from them): [0] frames with a low-entropy window (k_seg), [1] records of the filter-pass queue, [2] of the
 * candidate queue, [3] of the seed queue ([1]-[3] include the few records a warp reserved and left empty), [4] ungapped
 * HSPs at or above the report floor; [5] gapped extensions the screening pass (k_gap_screen) handed to the complete DP
 * (k_gap_dp), [6] extensions whose live window outgrew k_gap_dp's ring and went to the fallback (k_gap_dir); [7] reserved
 * (0).  The environment variables MCX_GAP_SCREEN_ROWS (1..32), MCX_GAP_SCREEN_COLS (1..48) and MCX_GAP_DP_COLS (1..56)
 * lower the limits at which these hand-offs happen (tests of the later paths; the results do not depend on them). */
int  mcx_search_counters(mcx_ctx *ctx, int64_t out[8]);

/* Measurement aid (SURVEY 8d): issue rate of the DPX instructions an affine-gap cell uses (viaddmax_s32 /
 * vimax3_s32_relu, independent chains on every SM), in 1e9 thread-instructions per second.  The DPX-bound cell rate
 * that the gapped stage's GCUPS is quoted against is this number / 3 (two viaddmax + one vimax3 per cell). */
int  mcx_dpx_peak(mcx_ctx *ctx, double *gops_per_s);

/* Measurement aid (SURVEY 8d, "seeding: L2/HBM random-access transaction rate"): rate of independent 4-byte loads at
 * random words of the 32 MB presence filter (one 32-byte L2 sector each), in 1e9 loads per second -- the access pattern
 * of the seed-word probes with nothing else in the way.  k_probe's probes/s are quoted against it. */
int  mcx_l2_peak(mcx_ctx *ctx, double *gsectors_per_s);

const char *mcx_last_error(mcx_ctx *ctx);
const char *mcx_version(void);

#ifdef __cplusplus
}
#endif
#endif
