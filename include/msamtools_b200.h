/*
 * msamtools_b200.h -- C ABI of the B200-native msamtools hot path.
 *
 * One shared library (libmsamtools_b200.so, CUDA sm_100a) replaces the three
 * in-process streaming kernels of the reference and the helpers under them:
 *
 *   reference (pull model, state in `global`)          this ABI (push model, state in msg_ctx)
 *   ------------------------------------------------   ----------------------------------------
 *   mFilterFile                msam_filter.c:98-190    msg_push + msg_pull_kept / msg_pull_records
 *   mWriteBestHitBamPool*      msam_filter.c:192-263   (hit_mode in msg_config)
 *   bam_cigar2details          mBamVector.c:23-38      (decode/filter kernel) msg_pull_stats
 *   bam_get_summary            mBamVector.c:40-133     (decode/filter kernel) msg_pull_stats
 *   mEstimateInsertCountOnFile msam_profile.c:204-243  msg_push (want_profile)
 *   mEstimateInsertCountOnPool msam_profile.c:65-200   msg_push (want_profile)
 *   mInsertCountToAbundanceMatrix msam_profile.c:248-425  msg_finish_profile
 *   mEstimateCoverageOnFile    msam_coverage.c:106-139 msg_push (want_coverage)
 *   mUpdateCoverageForAlignment msam_coverage.c:33-87  msg_push (want_coverage)
 *   mWriteCoverageSummaryToStream msam_coverage.c:189-219 (numbers) msg_finish_coverage
 *
 * Conventions
 *   - plain pointers and sizes only; no CUDA or torch types cross this boundary.
 *   - every function returns 0 on success or a negative MSG_E* code; nothing in
 *     the library calls exit(). msg_last_error() gives the text the CLI prints
 *     after "Fatal Error: " (mirrors mDie, mCommon.c:22-31).
 *   - the caller owns all host buffers; the library owns device memory/streams.
 *   - a context is NOT thread-safe; calls on one context must be serialised.
 *   - there is no CPU fallback: msg_create fails (MSG_ENODEV) without a GPU.
 *
 * Input layout ("raw chunk"): the uncompressed BAM record stream exactly as it
 * sits inside the BGZF payload -- for each record `int32 block_size` followed
 * by block_size bytes (SAM spec 4.2) -- plus a host-built index
 * rec_off[0..nrec] of byte offsets of each record's block_size field
 * (rec_off[nrec] = end of the last record).  A chunk must end on a QNAME
 * boundary (see msg_split_point) so that no read group straddles chunks/GPUs --
 * except on a context created with `collate`, which takes records in any order.
 *
 * Collating contexts (msg_config.collate = 1 or MSG_COLLATE_RANKS)
 *   - chunks need not end on a QNAME boundary; a read's records may be spread over any number of pushes, and a read
 *     may have any number of records.
 *   - msg_push* append the records' heads (everything but SEQ/QUAL) to device memory and complete before returning.
 *     More than 2^32-2 records (or 64 GiB of heads) in one scope: MSG_ERANGE; no room on the device: MSG_ENOMEM.
 *   - the first msg_finish_profile / msg_finish_coverage / msg_pull_counts after pushes groups everything held by
 *     QNAME (equal l_read_name and bytes) and runs the pipeline once for every consumer; later calls reuse it.
 *     A push after that starts a new scope whose records add to the same accumulators.  msg_reset drops held records.
 *   - integers equal, and f64 values agree to rounding with, those of the same records reordered so that each
 *     QNAME's records are contiguous and keep their input order.
 *   - msg_kept_count, msg_pull_kept, msg_pull_records and msg_pull_stats return MSG_ESTATE.
 *   - errors found after grouping (MSG_ENOTAG, MSG_ENOAS, MSG_EFORMAT) name the record's input ordinal (0-based,
 *     counted over the scope's pushes) in msg_last_error.
 *
 * Collating across ranks (msg_config.collate = MSG_COLLATE_RANKS, n_ranks > 1)
 *   - one read's records may be pushed on different ranks, in any order and any number of pushes.  The input is rank
 *     0's pushes, then rank 1's, and so on: a record's global input ordinal is the number of records pushed by lower
 *     ranks in this scope plus its ordinal among this rank's pushes.
 *   - at the first collation point after pushes the ranks exchange record heads over NCCL (send/recv) so that every
 *     QNAME lands on exactly one rank (rank floor(hash * n_ranks / 2^64) of its 64-bit QNAME hash); each rank then
 *     collates and runs the pipeline on what it received, and msg_finish_profile / msg_finish_coverage combine the
 *     ranks as usual.  Each rank holds about 1/n_ranks of the heads.
 *   - results equal those of one collating GPU fed the concatenation: integers exactly, f64 values to rounding, the
 *     same PropSharing iteration count; they are bit-identical on every rank.
 *   - msg_finish_profile, msg_finish_coverage and msg_pull_counts are COLLECTIVE: every rank must make each such
 *     call, in the same order, including ranks that pushed nothing.  msg_reset must be called on every rank.
 *   - more than 2^32-2 records over all ranks in one scope, or 64 GiB of heads for one rank: MSG_ERANGE on every rank
 *     before any record moves; a rank without room for what it receives: MSG_ENOMEM on every rank, naming that rank.
 *   - a push-time MSG_EFORMAT names the ordinal within this rank's pushes.  Errors found after grouping name the
 *     global input ordinal and its source, "(input record G: rank r, record k of its pushes)", on the rank that found
 *     them; every other rank returns the same code with "record error on rank q".
 *   - with n_ranks == 1 it is collate = 1.  Not with exact.
 */
#ifndef MSAMTOOLS_B200_H
#define MSAMTOOLS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSG_ABI_VERSION 2

/* error codes */
#define MSG_OK         0
#define MSG_EINVAL    -1   /* bad argument / bad config                           */
#define MSG_ENODEV    -2   /* no CUDA device / driver                             */
#define MSG_ECUDA     -3   /* CUDA runtime error (text in msg_last_error)         */
#define MSG_ENOMEM    -4
#define MSG_ENOTAG    -5   /* neither NM nor MD present  (msam_filter.c:150-152)  */
#define MSG_ENOAS     -6   /* AS missing on a best-hit candidate (msam_filter.c:220-221) */
#define MSG_EFORMAT   -7   /* malformed record (offsets run past the chunk)       */
#define MSG_ERANGE    -8   /* output buffer too small                             */
#define MSG_ENCCL     -9   /* NCCL error                                          */
#define MSG_ESTATE   -10   /* call out of order                                   */

/* hit_mode: which pool writer the reference would pick, msam_filter.c:88-93 */
#define MSG_HIT_NONE    0  /* mWriteBamPool               */
#define MSG_HIT_BEST    1  /* mWriteBestHitBamPool        */
#define MSG_HIT_UNIQUE  2  /* mWriteUniqueBestHitBamPool  */

/* collate: 1 = group by QNAME on one GPU; MSG_COLLATE_RANKS = also across the ranks of a multi-GPU run */
#define MSG_COLLATE_RANKS      2

/* share_type: msam_profile.c:5-8 (same numeric values) */
#define MSG_MULTI_ALL          1
#define MSG_MULTI_EQUAL        2
#define MSG_MULTI_PROPORTIONAL 3
#define MSG_MULTI_IGNORE       4

typedef struct msg_ctx msg_ctx;   /* opaque; one per GPU */

/*
 * Mirrors the fields of msam_global (msam.h:19-52) that the three streaming
 * kernels read, plus the mFilterFile arguments (msam_filter.c:98).
 */
typedef struct msg_config {
    uint32_t abi_version;        /* = MSG_ABI_VERSION */

    /* ---- stage 1: filter (msam_filter.c) ---- */
    uint8_t  do_filter;          /* 0: every record goes straight to profile/coverage
                                       (plain `msamtools profile` / `coverage`)        */
    uint8_t  hit_mode;           /* MSG_HIT_*                                          */
    uint8_t  invert;             /* -v                                                 */
    uint8_t  keep_unmapped;      /* -k                                                 */
    uint8_t  rescore;            /* --rescore                                          */
    uint8_t  collate;            /* records may come in any order (e.g. sorted by coordinate): the context keeps their
                                    heads (no SEQ/QUAL) on the device and groups them by QNAME at the first
                                    msg_finish_profile / msg_finish_coverage after pushes.  Needs want_profile and/or
                                    want_coverage; not with want_records / want_kept / want_stats.  1 needs
                                    n_ranks == 1; MSG_COLLATE_RANKS (2) also groups across ranks (see above).
                                    Results equal those of the same records regrouped stably by QNAME (see above).    */
    uint8_t  exact;              /* bit-exact abundances: every feature's --multi=equal shares and PropSharing increments
                                    are added in the input order of their inserts, with the reference's IEEE operations,
                                    instead of by f64 atomics.  Abundances, EM deltas, iterations and purged count are then
                                    bit-identical to the reference's (for any chunking and push kind; with collate, to the
                                    reference on the grouped order).  Effect only with share_type MSG_MULTI_EQUAL or
                                    MSG_MULTI_PROPORTIONAL.  Needs n_ranks == 1 (msg_create returns MSG_EINVAL otherwise);
                                    works with collate.  Costs a transposition of the lists per finish after pushes
                                    and a serial sum per feature in each iteration (DESIGN.md §9).                      */
    uint8_t  reserved0[1];
    int32_t  min_length;         /* -l  (MIN_LENGTH, msam_filter.c:449-457)            */
    int32_t  ppt;                /* 10*-p or --ppt (PPT, msam_filter.c:420-437)        */
    int32_t  max_clip;           /* 100 - z; 100 when -z absent (MAX_CLIP, :439-447)   */

    /* ---- stage 2 consumers of the (filtered) record stream ---- */
    uint8_t  want_kept;          /* keep the kept-record index list for msg_pull_kept; with 0, best-hit + profile
                                    runs as one fused pass and only msg_kept_count is available          */
    uint8_t  want_records;       /* materialise filtered record bytes (msg_pull_records) */
    uint8_t  want_profile;       /* msam_profile.c                                     */
    uint8_t  want_coverage;      /* msam_coverage.c                                    */
    uint8_t  want_stats;         /* keep per-record (alen,qlen,qclip,edit,AS) for msg_pull_stats */
    uint8_t  share_type;         /* MSG_MULTI_*                                        */
    uint8_t  debug_force_slow;   /* testing: route every record through the global-memory parser */
    uint8_t  coverage_summary;   /* want_coverage: only the per-target summary of msam_coverage.c:189-219 is needed (`coverage
                                    --summary`): one bit per position instead of a depth cell; msg_pull_coverage unavailable */

    int32_t  n_targets;          /* header->n_targets                                  */
    int32_t  n_features;         /* global->n_features (== n_targets when fmap NULL)   */
    const int32_t  *fmap;        /* [n_targets] seq -> feature, NULL = identity (msam_profile.c:845-852) */
    const uint32_t *target_len;  /* [n_targets]; required for want_coverage            */

    /* ---- placement ---- */
    int32_t  device;             /* CUDA device ordinal                                */
    int32_t  n_ranks;            /* 1 = single GPU; >1 enables the NCCL allreduce      */
    int32_t  rank;
    const void *nccl_unique_id;  /* 128 bytes from msg_nccl_unique_id (rank 0), NULL if n_ranks==1 */
} msg_config;

/* header statistics of `msamtools profile` (msam_profile.c:886-903) */
typedef struct msg_profile_stats {
    uint32_t mapped_inserts;     /* return value of mEstimateInsertCountOnFile  :204 */
    uint32_t uniq_mapper_count;  /* global->uniq_mapper_count                        */
    uint32_t multi_mapper_count; /* global->multi_mapper_count                       */
    uint32_t purged_insert_count;/* global->purged_insert_count            :394-404  */
    int32_t  em_iterations;      /* last k of the PropSharing loop         :331      */
    int32_t  em_converged;       /* 1 if delta < 1e-10 was hit             :383      */
    double   em_delta[20];       /* DELTA^2 per iteration (index k-1)      :381      */
    uint64_t multi_lists;        /* |multi_mappers| summed over all ranks            */
    uint64_t multi_entries;      /* total list entries (this rank)                   */
} msg_profile_stats;

/* ------------------------------------------------------------------ lifecycle */
int  msg_create(const msg_config *cfg, msg_ctx **out);
void msg_destroy(msg_ctx *ctx);
const char *msg_last_error(const msg_ctx *ctx);   /* ctx may be NULL: last create error */
int  msg_abi_version(void);
int  msg_device_count(void);

/* ------------------------------------------------------------------ host index helpers (CPU, no GPU needed) */
/* Walk the block_size chain (sam_read1's framing, msam_helper.c:267).  Writes
 * up to cap offsets + the end offset; *nrec gets the number of whole records.
 * Returns MSG_EFORMAT if a record runs past nbytes (partial trailing record is
 * reported through *consumed < nbytes and is not an error when allow_partial). */
int  msg_index_records(const uint8_t *raw, size_t nbytes, uint64_t *rec_off, size_t cap,
                       size_t *nrec, size_t *consumed, int allow_partial);
/* Largest k <= want such that records k-1 and k have different QNAMEs and record
 * k-1 is mapped with tid >= 0 (so both the filter's and the profile's prev_read
 * equal QNAME(k-1): msam_filter.c:120-121,170; msam_profile.c:223-232).
 * Returns 0 if no such point exists in (0, want]. */
size_t msg_split_point(const uint8_t *raw, const uint64_t *rec_off, size_t nrec, size_t want);

/* ------------------------------------------------------------------ data path */
/* Host buffers (pinned or pageable).  H2D copy + all kernels for this chunk.  A pinned, mapped, 16-byte
 * aligned buffer (msg_host_alloc) is not copied when the fused filter->profile pass applies
 * (do_filter, hit_mode, want_profile and no kept/records/coverage): the decode kernel reads its
 * windows of each record in place over PCIe (msg_timing.zero_copy_chunks; MSG_ZERO_COPY=0 disables). */
int  msg_push(msg_ctx *ctx, const uint8_t *raw, size_t nbytes,
              const uint64_t *rec_off, size_t nrec);
/* Same, but the chunk already lives in device memory (device pointers).      */
int  msg_push_device(msg_ctx *ctx, const uint8_t *d_raw, size_t nbytes,
                     const uint64_t *d_rec_off, size_t nrec);
/*
 * Asynchronous, double-buffered push -- the streaming loop of the reference (one record at a time through mSamRead,
 * msam_filter.c:116-125, msam_helper.c:246-268) becomes a pipeline of chunks: the call queues the chunk's transfers
 * and kernels and returns without waiting for them, so that the host can inflate / index the next chunk meanwhile.
 *   - at most TWO chunks are in flight.  The call first completes the chunk pushed two calls earlier; its buffers
 *     (raw, rec_off) may be recycled once this call returns.  A host that rotates three buffers never waits for the
 *     GPU; with two it calls msg_wait before refilling.  msg_wait (and every result / finish / reset call)
 *     completes everything in flight.
 *   - staged chunks are copied on a second stream into one of two device slots while the previous chunk's kernels
 *     run; pinned 16-byte aligned buffers (msg_host_alloc) are decoded in place over PCIe instead.
 *   - errors of a chunk (MSG_ENOTAG, MSG_ENOAS, MSG_EFORMAT) are reported by the call that completes it.
 *   - contexts that need host decisions per chunk (record output, kept list, coverage, stats, profile without
 *     best-hit) complete the chunk before returning: for them msg_push_async == msg_push.
 *   - "results of the LAST pushed chunk" below refer to the last COMPLETED chunk.
 */
int  msg_push_async(msg_ctx *ctx, const uint8_t *raw, size_t nbytes,
                    const uint64_t *rec_off, size_t nrec);
int  msg_push_device_async(msg_ctx *ctx, const uint8_t *d_raw, size_t nbytes,
                           const uint64_t *d_rec_off, size_t nrec);
int  msg_wait(msg_ctx *ctx);
/* Device staging owned by the library, for callers that want to fill HBM once
 * and push the same resident chunk repeatedly (benchmarks).                   */
int  msg_device_alloc(msg_ctx *ctx, size_t nbytes, void **d_ptr);
int  msg_device_free(msg_ctx *ctx, void *d_ptr);
int  msg_device_upload(msg_ctx *ctx, void *d_dst, const void *h_src, size_t nbytes);
/* Pinned (page-locked) host staging for msg_push callers: H2D copies from it run at full PCIe rate
 * and asynchronously.  Usable before any context exists (device = CUDA ordinal).               */
int  msg_host_alloc(int device, size_t nbytes, void **h_ptr);
int  msg_host_free(void *h_ptr);
int  msg_sync(msg_ctx *ctx);
/* Forget accumulated profile/coverage/kept state (keeps allocations).        */
int  msg_reset(msg_ctx *ctx);

/* ---- results of the LAST pushed chunk ---- */
/* kept records in reference output order (msam_filter.c:186,247-263) as indices
 * into the chunk's rec_off[]. */
int  msg_kept_count(msg_ctx *ctx, size_t *n_kept);
int  msg_pull_kept(msg_ctx *ctx, uint32_t *idx, size_t cap, size_t *n_kept);
/* filtered record bytes, reference output order; with rescore the AS tag is
 * rewritten as the reference does (msam_filter.c:160-168). */
int  msg_pull_records(msg_ctx *ctx, uint8_t *out, size_t cap, size_t *nbytes, size_t *nrec);
/* per-record alignment summary (mAlignmentSummary, mBamVector.h:38-47) and AS.
 * Any pointer may be NULL.  flags: bit0 entered pool, bit1 has AS, bit2 QNAME
 * equals previous record's, bit3 parsed by the slow path. */
int  msg_pull_stats(msg_ctx *ctx, size_t nrec, int32_t *alen, int32_t *qlen, int32_t *qclip,
                    int32_t *edit, int32_t *score, uint8_t *flags);

/* ---- accumulated over all pushed chunks ---- */
/* raw counters before the abundance step: ui_insert_count (doubled, u32) and
 * d_insert_count; either may be NULL.  Local to this rank (no allreduce).    */
int  msg_pull_counts(msg_ctx *ctx, uint32_t *ui, double *d);
/* mInsertCountToAbundanceMatrix: U = ui/2 (+ d | proportional loop).  With n_ranks > 1 every rank
 * must call it and gets the same result: proportional mode combines the ranks inside one
 * cooperative kernel over CUDA-IPC peer memory, the other modes (or MSG_NO_P2P=1) through NCCL.
 * On a MSG_COLLATE_RANKS context with n_ranks > 1, msg_pull_counts and msg_finish_coverage are
 * collective too (the first of these calls after pushes exchanges the records).                  */
int  msg_finish_profile(msg_ctx *ctx, double *abundance /*[n_features]*/, msg_profile_stats *st);
/* per target: covered flag, #positions with depth != 0, sum of depths
 * (msam_coverage.c:189-219).  With n_ranks > 1: allreduce first.             */
int  msg_finish_coverage(msg_ctx *ctx, uint8_t *covered, int64_t *touched, int64_t *sum /*[n_targets]*/);
/* per-position depth of one target (msam_coverage.c:143-187), after msg_finish_coverage */
int  msg_pull_coverage(msg_ctx *ctx, int32_t tid, int32_t *depth /*[target_len[tid]]*/);

/* ------------------------------------------------------------------ timing / accounting */
typedef struct msg_timing {
    double   decode_ms;      /* dominant kernel: decode + filter statistics (sum over launches) */
    uint64_t decode_launches;
    double   total_ms;       /* all kernels of msg_push*, sum                                    */
    uint64_t kernel_launches;/* every kernel launched by this context                           */
    uint64_t h2d_bytes, d2h_bytes;
    uint64_t alg_bytes;      /* sum over pushed records of A(rec) (DESIGN.md)                    */
    uint64_t slow_records;   /* records parsed by the global-memory slow path                    */
    uint64_t fused_chunks;   /* chunks that went through the fused besthit->profile pass          */
    uint64_t fused_fallbacks;/* ... of which the guard sent to the general pipeline               */
    uint64_t zero_copy_chunks;/* msg_push chunks decoded straight from pinned host memory (no bulk H2D) */
} msg_timing;
int  msg_get_timing(msg_ctx *ctx, msg_timing *t, int reset);
/* CUDA-event stopwatch on the context's own stream (the stream every kernel of this
 * context is launched on): msg_mark records event `slot` (0..7); msg_elapsed_ms
 * synchronises and returns the device time between two marks.                      */
int  msg_mark(msg_ctx *ctx, int slot);
int  msg_elapsed_ms(msg_ctx *ctx, int slot_from, int slot_to, double *ms);

/* ------------------------------------------------------------------ multi-GPU */
int  msg_nccl_unique_id(void *id128 /* 128 bytes out */);

#ifdef __cplusplus
}
#endif
#endif /* MSAMTOOLS_B200_H */
