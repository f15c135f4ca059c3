/*
 * msamtools_main.c -- drop-in `msamtools {filter,profile,coverage}` whose hot path runs on the GPU
 * through libmsamtools_b200 (include/msamtools_b200.h).
 *
 * What is mirrored from the reference, by file:line --
 *   command dispatch and usage                  msamtools.c:8-49
 *   filter options, validation order, messages  msam_filter.c:304-458 (messages go to stdout, then "\n" on stderr, exit 1)
 *   output modes "w"/"wh"/"wb"/"wbu"            msam_filter.c:464-470, msam_helper.c:238-241
 *   QNAME grouping pre-flight + status strings  msam_helper.c:88-137,295-484
 *   @PG / '#' provenance                        msam_helper.c:139-184
 *   profile options, prefix matching, --genome, --mincount, Unknown, units, header statistics, "%.8g" table
 *                                               msam_profile.c:434-499,503-1015; mMatrix.c:168-179,359-376
 *   coverage options and both writers           msam_coverage.c:143-219,223-390
 *   error convention "Fatal Error: ...", exit 1 mCommon.c:3-31
 * The help glossaries are written for this build; option names and semantics are the reference's.
 * `summary` is outside the accelerated path (SURVEY.md 8) and is not provided.
 */
#include <math.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <pthread.h>
#include <sys/stat.h>
#include <time.h>
#include <unistd.h>
#include <zlib.h>

#include "../../../include/msamtools_b200.h"
#include "../host/bamio.h"
#include "../host/gzpar.h"
#include "../host/keyorder.h"
#include "../host/margs.h"
#include "../host/recwalk.h"

#define PROGRAM "msamtools"
#define PACKAGE_VERSION "1.1.3-b200"
#define MSAM_GIT_COMMIT "b200-native"

#define QNAME_GROUP_CHECK_RECORDS 10000
#define COORD_ORDER_CHECK_RECORDS 100000
#define COORD_ORDER_MIN_RECORDS   10000

static void warm_join(void);
static void mQuit(const char *fmt, ...)
{
    va_list ap;
    warm_join();
    va_start(ap, fmt); vfprintf(stderr, fmt, ap); va_end(ap);
    fprintf(stderr, "\n");
    exit(EXIT_FAILURE);
}
static void mDie(const char *fmt, ...)
{
    va_list ap;
    warm_join();                            /* never exit() under a CUDA start-up still running on the warm-up thread */
    fflush(stdout);
    fprintf(stderr, "Fatal Error: ");
    va_start(ap, fmt); vfprintf(stderr, fmt, ap); va_end(ap);
    fprintf(stderr, "\n");
    exit(EXIT_FAILURE);
}

/* MSAMTOOLS_TIMING=1: wall time of each host phase on stderr ("# phase <command> <name>: <seconds>") */
static void phase(const char *cmd, const char *name)
{
    static int on = -1; static struct timespec t0;
    struct timespec t;
    if (on < 0) { on = getenv("MSAMTOOLS_TIMING") != NULL; clock_gettime(CLOCK_MONOTONIC, &t0); }
    if (!on) return;
    clock_gettime(CLOCK_MONOTONIC, &t);
    if (name) {
        struct timespec rt; clock_gettime(CLOCK_REALTIME, &rt);
        fprintf(stderr, "# phase %s %s: %.3f s (ends at %02d.%03d)\n", cmd, name, (t.tv_sec - t0.tv_sec) + 1e-9 * (t.tv_nsec - t0.tv_nsec),
                (int)(rt.tv_sec % 60), (int)(rt.tv_nsec / 1000000));
    }
    t0 = t;
}

/* worker threads for inflate / deflate / formatting: MSAMTOOLS_THREADS, default the online cores, at most 16 */
static int host_threads(void)
{
    long n = sysconf(_SC_NPROCESSORS_ONLN);
    if (getenv("MSAMTOOLS_THREADS")) n = atol(getenv("MSAMTOOLS_THREADS"));
    return n > 16 ? 16 : (n < 1 ? 1 : (int)n);
}

static void print_help(const char *sub, void **argtable)
{   /* mPrintHelp, msam_helper.c:49-57 */
    fprintf(stdout, "Usage:\n------\n\n%s %s", PROGRAM, sub);
    arg_print_syntax(stdout, argtable, "\n");
    fprintf(stdout, "\nGeneral options:\n----------------\n\nThese options specify the input/output formats of BAM/SAM files \n(same meaning as in 'samtools view'):\n");
    arg_print_glossary(stdout, argtable, "  %-25s %s\n");
}

static void multiple_file_error(const char *sub, void **argtable)
{
    fprintf(stderr, "Multiple input files not supported in %s.\n", sub);
    fprintf(stderr, "Use 'samtools merge' to combine BAM/SAM files.\n");
    print_help(sub, argtable);
    mQuit("");
}

static char *command_line(int argc, char *argv[])
{   /* mBuildCommandLine: PROGRAM + the sub-command's argv */
    char **full = malloc(sizeof(char *) * (size_t)(argc + 1));
    full[0] = (char *)PROGRAM;
    for (int i = 0; i < argc; i++) full[i + 1] = argv[i];
    char *s = bio_stringify_argv(argc + 1, full);
    free(full);
    if (!s) mDie("Cannot construct command line for provenance");
    return s;
}

/* ============================================================ record chunks */
typedef struct {
    uint8_t *raw; size_t len, cap;        /* record stream; len may include a partial trailing record (bulk reader) */
    uint64_t *off; size_t n, offcap;      /* off[0..n]: whole records indexed so far, off[n] = end of the last one */
    int fixed;                            /* 1: raw is a fixed-capacity (possibly pinned) buffer, never realloc'ed */
    int pinned;
    size_t k;                             /* records handed to the GPU (a QNAME boundary) */
} chunk_t;

static void input_die(bio_file *in)
{   /* the reference ends the stream silently on sam_read1 < -1 and htslib prints the reason; a drop-in that keeps going
       after a corrupt block would write a partial result with exit status 0, so this one stops */
    mDie("Cannot read input: %s", bio_error(in));
}

static void chunk_reserve_off(chunk_t *c, size_t n)
{
    if (n + 2 > c->offcap) { c->offcap = c->offcap ? c->offcap * 2 : 1 << 16; while (n + 2 > c->offcap) c->offcap *= 2; c->off = realloc(c->off, c->offcap * sizeof(uint64_t)); if (!c->off) mDie("Out of memory"); }
}

/* record-wise: append records until the chunk holds `want_records` / `want_bytes` or the input ends */
static void chunk_fill(chunk_t *c, bio_file *in, const bio_hdr *h, size_t want_records, size_t want_bytes, int *eof)
{
    while (!*eof && c->n < want_records && c->len < want_bytes) {
        chunk_reserve_off(c, c->n + 1);
        c->off[c->n] = c->len;
        int rc = bio_read_record(in, h, &c->raw, &c->cap, &c->len);
        if (rc < 0) input_die(in);
        if (rc == 0) { *eof = 1; break; }
        c->n++;
    }
    chunk_reserve_off(c, c->n);
    c->off[c->n] = c->len;
}

static double g_walk_sec;
/* bulk (BAM): inflate straight into the fixed-capacity buffer, then walk the block_size chain over the new bytes */
static void chunk_fill_bulk(chunk_t *c, bio_file *in, int32_t n_targets, size_t want_records, size_t want_bytes, int *eof)
{
    if (want_bytes > c->cap) want_bytes = c->cap;
    while (!*eof && c->n < want_records && c->len < want_bytes) {
        int rc = bio_read_raw(in, c->raw, c->cap, &c->len);
        if (rc < 0) input_die(in);
        if (rc == 0) { *eof = 1; break; }
        struct timespec w0, w1; clock_gettime(CLOCK_MONOTONIC, &w0);
        const int wrc = rw_index(c->raw, (size_t)c->off[c->n], c->len, n_targets, host_threads(), &c->off, &c->n, &c->offcap);
        if (wrc == -1) mDie("Cannot read input: corrupt BAM record");
        if (wrc) mDie("Out of memory");
        clock_gettime(CLOCK_MONOTONIC, &w1); g_walk_sec += (w1.tv_sec - w0.tv_sec) + 1e-9 * (w1.tv_nsec - w0.tv_nsec);
        if (rc == 2) break;                                  /* buffer full */
    }
    if (*eof && (size_t)c->off[c->n] != c->len) mDie("Cannot read input: truncated BAM record");
}

static int names_differ(const chunk_t *c, size_t a, size_t b)
{
    const uint8_t *x = c->raw + c->off[a], *y = c->raw + c->off[b];
    return x[12] != y[12] || memcmp(x + 36, y + 36, x[12]) != 0;
}

/* ============================================================ QNAME grouping pre-flight (msam_helper.c:295-484) */
typedef enum { QN_NOT_REQUIRED = 0, QN_HEADER_CONFIRMED, QN_SAMPLE_OK, QN_SAMPLE_WARNING } qn_status;
typedef struct { qn_status status; size_t qname_records_checked, input_records_checked, mapped_records_checked; } qn_result;

static void qn_format(const qn_result *r, char *buf, size_t n)
{   /* mFormatQNameCheck, msam_helper.c:88-137 */
    switch (r->status) {
    case QN_NOT_REQUIRED: snprintf(buf, n, "QNAME grouping check: not required for this operation"); break;
    case QN_HEADER_CONFIRMED: snprintf(buf, n, "QNAME grouping check: confirmed by input header SO:queryname"); break;
    case QN_SAMPLE_OK:
        if (r->input_records_checked < QNAME_GROUP_CHECK_RECORDS)
            snprintf(buf, n, "QNAME grouping check: no QNAME grouping violation detected in all %zu records", r->qname_records_checked);
        else
            snprintf(buf, n, "QNAME grouping check: no QNAME grouping violation detected in first %zu records", r->qname_records_checked);
        break;
    default:
        snprintf(buf, n, "QNAME grouping check: WARNING - no QNAME grouping violation detected in first %zu records; %zu mapped records among the "
                 "first %zu input records were consistent with coordinate ordering", r->qname_records_checked, r->mapped_records_checked, r->input_records_checked);
    }
}

typedef struct { char **key; size_t *last; size_t cap, n; } nameset;
static uint64_t fnv1a(const char *s) { uint64_t h = 1469598103934665603ull; for (; *s; s++) { h ^= (uint8_t)*s; h *= 1099511628211ull; } return h; }
static size_t *nameset_slot(nameset *s, const char *k, int insert)
{
    if (s->cap == 0) { s->cap = 1 << 15; s->key = calloc(s->cap, sizeof(char *)); s->last = calloc(s->cap, sizeof(size_t)); }
    size_t i = fnv1a(k) & (s->cap - 1);
    while (s->key[i]) { if (!strcmp(s->key[i], k)) return &s->last[i]; i = (i + 1) & (s->cap - 1); }
    if (!insert) return NULL;
    s->key[i] = strdup(k); s->n++;
    return &s->last[i];
}

/* works on the first chunk, which the caller fills with >= COORD_ORDER_CHECK_RECORDS records (or the whole input) */
static qn_result qname_preflight(const bio_hdr *h, const chunk_t *c)
{
    qn_result r = { QN_SAMPLE_OK, 0, 0, 0 };
    char *so = bio_hdr_find_hd_tag(h, "SO");
    if (so) {
        if (!strcmp(so, "queryname")) { free(so); r.status = QN_HEADER_CONFIRMED; return r; }
        if (!strcmp(so, "coordinate")) {
            free(so);
            mDie("Input SAM/BAM declares 'SO:coordinate', but this operation requires records to be grouped by QNAME.\n"
                 "             Please name-sort the input, for example with 'samtools sort -n input.bam -o input.name_sorted.bam'.");
        }
        free(so);
    }
    nameset closed = { 0 };
    const char *cur = NULL; size_t cur_first = 0;
    int coord_ordered = 1, coord_relevant = 0, have_prev = 0; int32_t ptid = -1, ppos = -1;
    size_t lim = c->n < COORD_ORDER_CHECK_RECORDS ? c->n : COORD_ORDER_CHECK_RECORDS;
    for (size_t i = 0; i < lim; i++) {
        const uint8_t *rec = c->raw + c->off[i];
        const char *qname = (const char *)rec + 36;
        size_t recno = i + 1;
        r.input_records_checked++;
        if (recno <= QNAME_GROUP_CHECK_RECORDS) {
            r.qname_records_checked++;
            if (!cur) { cur = qname; cur_first = recno; }
            else if (strcmp(qname, cur) != 0) {
                *nameset_slot(&closed, cur, 1) = recno - 1;
                size_t *re = nameset_slot(&closed, qname, 0);
                if (re)
                    mDie("SAM/BAM file is not grouped by QNAME. Read '%s' reappears at record %zu after its previous group ended at record %zu "
                         "(%zu intervening records). Please name-sort the input, for example with 'samtools sort -n input.bam -o input.name_sorted.bam'.",
                         qname, recno, *re, recno - *re - 1);
                cur = qname; cur_first = recno;
            }
        }
        uint32_t flag = (uint32_t)rec[18] | (uint32_t)rec[19] << 8;
        int32_t tid = (int32_t)((uint32_t)rec[4] | (uint32_t)rec[5] << 8 | (uint32_t)rec[6] << 16 | (uint32_t)rec[7] << 24);
        int32_t pos = (int32_t)((uint32_t)rec[8] | (uint32_t)rec[9] << 8 | (uint32_t)rec[10] << 16 | (uint32_t)rec[11] << 24);
        if (!(flag & 4) && tid >= 0) {
            r.mapped_records_checked++;
            if (have_prev && (tid < ptid || (tid == ptid && pos < ppos))) coord_ordered = 0;
            ptid = tid; ppos = pos; have_prev = 1;
        }
        if (flag & (1 | 256 | 2048)) coord_relevant = 1;
    }
    (void)cur_first;
    for (size_t i = 0; i < closed.cap; i++) free(closed.key[i]);
    free(closed.key); free(closed.last);
    if (coord_ordered && coord_relevant && r.mapped_records_checked >= COORD_ORDER_MIN_RECORDS) {
        char w[1024];
        r.status = QN_SAMPLE_WARNING;
        qn_format(&r, w, sizeof w);
        fprintf(stderr, "WARNING: %s\n", w);
    }
    return r;
}

/* ============================================================ the GPU streaming loop shared by the three commands */
typedef struct {
    msg_config cfg;
    bio_file *in; bio_hdr *hdr;
    chunk_t chunk; int eof;               /* filled with the first records by the QNAME pre-flight */
    bio_file *out; bio_hdr *out_hdr;      /* filter only */
    const char *path;
} run_t;

/* chunk size: records / bytes per push (MSAMTOOLS_CHUNK_RECORDS / MSAMTOOLS_CHUNK_MB override, for tests and tuning) */
static size_t env_size(const char *name, size_t dflt, size_t unit) { const char *e = getenv(name); return e && atol(e) > 0 ? (size_t)atol(e) * unit : dflt; }
#define CHUNK_RECORDS env_size("MSAMTOOLS_CHUNK_RECORDS", (size_t)1 << 19, 1)
#define CHUNK_BYTES   env_size("MSAMTOOLS_CHUNK_MB", (size_t)128 << 20, (size_t)1 << 20)
#define CHUNK_SLACK   env_size("MSAMTOOLS_CHUNK_SLACK_KB", (size_t)32 << 20, (size_t)1 << 10)   /* a buffer holds a chunk plus this: the last batch of
                                                                                             blocks is cut to fit (the override is for tests) */
#define NBUF 3

static void gpu_die(msg_ctx *ctx) { mDie("%s", msg_last_error(ctx)); }

/* Reader thread <-> GPU thread: a ring of NBUF chunk buffers.  The reader fills buffer i (BGZF blocks are inflated on
 * worker threads straight into it, msam_helper.c:246-268 becomes bulk ingest), cuts it at a QNAME boundary, moves the
 * tail behind the cut to the front of buffer i+1 and posts it; the GPU thread pushes posted chunks with msg_push_async
 * and gives a buffer back two pushes later (the library may still be reading it until then). */
typedef struct {
    run_t *r;
    chunk_t buf[NBUF];
    int state[NBUF];                      /* 0 free, 1 posted */
    int posted_last;                      /* the posted chunk with this index is the final one (-1: not yet known) */
    int bulk, pin;                        /* pin: page-lock the chunk buffers (msg_host_alloc) */
    size_t cap;                           /* capacity of every fixed buffer */
    pthread_mutex_t mu; pthread_cond_t cv;
} ring_t;

static size_t choose_cut(chunk_t *c, int eof)
{   /* records to hand over: everything at EOF, else the last QNAME boundary msg_split_point accepts (0: need more input) */
    if (eof) return c->n;
    if (c->n < 2) return 0;
    size_t k = msg_split_point(c->raw, c->off, c->n, c->n - 1);
    return k;
}

static void ring_buffer_alloc(ring_t *g, int i, int pin);

static void *reader_main(void *arg)
{
    ring_t *g = arg; run_t *r = g->r;
    int cur = 0;
    for (;;) {
        chunk_t *c = &g->buf[cur];
        size_t want_n = CHUNK_RECORDS, want_b = CHUNK_BYTES;
        size_t k;
        for (;;) {
            if (g->bulk) chunk_fill_bulk(c, r->in, r->hdr->n_targets, want_n, want_b, &r->eof);
            else chunk_fill(c, r->in, r->hdr, want_n, want_b, &r->eof);
            k = choose_cut(c, r->eof);
            if (k || r->eof) break;
            /* no mapped record closes a QNAME group in the whole chunk: read on (growable buffers), or cut at any QNAME change */
            if (!c->fixed && c->n < 8 * CHUNK_RECORDS && c->len < 8 * CHUNK_BYTES) { want_n = c->n * 2; want_b = c->len * 2; continue; }
            for (k = c->n - 1; k > 0 && !names_differ(c, k - 1, k); k--) ;
            if (k) break;
            if (c->fixed && c->len + (1 << 17) < c->cap) { want_n = c->n * 2; want_b = c->cap; continue; }
            mDie("A single QNAME group exceeds the chunk buffer (%zu records, %zu bytes)", c->n, c->len);
        }
        c->k = k;
        const int last = r->eof && k == c->n;
        const int nxt = (cur + 1) % NBUF;
        pthread_mutex_lock(&g->mu);                          /* post first: the GPU thread only reads raw[0, off[k]) */
        g->state[cur] = 1;
        if (last) g->posted_last = cur;
        pthread_cond_broadcast(&g->cv);
        pthread_mutex_unlock(&g->mu);
        if (!last) {
            /* the records behind the cut (and a partial trailing record) open the next buffer */
            pthread_mutex_lock(&g->mu);
            while (g->state[nxt]) pthread_cond_wait(&g->cv, &g->mu);
            pthread_mutex_unlock(&g->mu);
            ring_buffer_alloc(g, nxt, g->pin);
            chunk_t *d = &g->buf[nxt];
            const size_t base = (size_t)c->off[k], tail = c->len - base;
            if (!d->fixed && tail > d->cap) { d->raw = realloc(d->raw, tail + (1 << 20)); d->cap = tail + (1 << 20); if (!d->raw) mDie("Out of memory"); }
            if (tail > d->cap) mDie("A single QNAME group exceeds the chunk buffer");
            memcpy(d->raw, c->raw + base, tail);
            d->len = tail; d->n = c->n - k;
            chunk_reserve_off(d, d->n + 1);
            for (size_t i = 0; i <= d->n; i++) d->off[i] = c->off[k + i] - base;
        }
        if (last) return NULL;
        cur = nxt;
    }
}

/* ---- record output (filter): a writer thread packs BGZF blocks / formats SAM and writes while the GPU thread is
 * already on the next chunk.  Two output buffers; the order of chunks is the order of posts. */
typedef struct {
    run_t *r;
    uint8_t *buf[2]; size_t cap[2], len[2];
    int pinned[2], want_pinned;           /* page-locked output buffers (device -> host copies by DMA) when the input buffers are */
    int state[2];                         /* 0 free, 1 posted */
    int done, failed;
    double t_write;
    pthread_mutex_t mu; pthread_cond_t cv;
} wring_t;

static int emit_records(run_t *r, const uint8_t *buf, size_t nb)
{
    if (bio_is_bam(r->out)) return bio_write_raw(r->out, buf, nb);      /* the bytes already are BAM records: blocks are packed on the worker threads */
    for (size_t o = 0; o < nb;) {
        const uint8_t *p = buf + o;
        uint32_t bs = (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24;
        if (bio_write_record(r->out, r->out_hdr, p, 4 + (size_t)bs)) return -1;
        o += 4 + (size_t)bs;
    }
    return 0;
}

static void *writer_main(void *arg)
{
    wring_t *w = arg;
    struct timespec ta, tb;
    for (int cur = 0;; cur ^= 1) {
        pthread_mutex_lock(&w->mu);
        while (!w->state[cur] && !w->done) pthread_cond_wait(&w->cv, &w->mu);
        const int have = w->state[cur];
        pthread_mutex_unlock(&w->mu);
        if (!have) return NULL;
        clock_gettime(CLOCK_MONOTONIC, &ta);
        const int rc = emit_records(w->r, w->buf[cur], w->len[cur]);
        clock_gettime(CLOCK_MONOTONIC, &tb);
        w->t_write += (tb.tv_sec - ta.tv_sec) + 1e-9 * (tb.tv_nsec - ta.tv_nsec);
        pthread_mutex_lock(&w->mu);
        if (rc) w->failed = 1;
        w->state[cur] = 0;
        pthread_cond_broadcast(&w->cv);
        pthread_mutex_unlock(&w->mu);
    }
}

/* kept records of the chunk just pushed -> output buffer `*wcur` (the writer thread takes it from there; w->r == NULL: no
 * thread, written here) */
static void pull_kept_records(run_t *r, msg_ctx *ctx, wring_t *w, int *wcur)
{
    size_t nb = 0, nr = 0;
    const int i = *wcur;
    if (msg_pull_records(ctx, NULL, 0, &nb, &nr)) gpu_die(ctx);
    pthread_mutex_lock(&w->mu);
    while (w->state[i]) pthread_cond_wait(&w->cv, &w->mu);
    const int failed = w->failed;
    pthread_mutex_unlock(&w->mu);
    if (failed) mDie("Cannot write alignment record");
    if (nb > w->cap[i]) {
        if (w->pinned[i]) msg_host_free(w->buf[i]); else free(w->buf[i]);
        w->buf[i] = NULL; w->pinned[i] = 0;
        w->cap[i] = nb + nb / 4 + 4096;
        if (w->want_pinned) {
            /* kept records never exceed the chunk (--rescore may add an AS tag per record: then the buffer is simply replaced) */
            void *pm = NULL;
            const size_t pcap = w->cap[i] > CHUNK_BYTES + CHUNK_SLACK ? w->cap[i] : CHUNK_BYTES + CHUNK_SLACK;
            if (msg_host_alloc(r->cfg.device, pcap, &pm) == MSG_OK) { w->buf[i] = pm; w->cap[i] = pcap; w->pinned[i] = 1; }
        }
        if (!w->buf[i]) { w->buf[i] = malloc(w->cap[i]); if (!w->buf[i]) mDie("Out of memory"); }
    }
    if (msg_pull_records(ctx, w->buf[i], w->cap[i], &nb, &nr)) gpu_die(ctx);
    w->len[i] = nb;
    if (!w->r) { if (emit_records(r, w->buf[i], nb)) mDie("Cannot write alignment record"); return; }
    pthread_mutex_lock(&w->mu);
    w->state[i] = 1;
    pthread_cond_broadcast(&w->cv);
    pthread_mutex_unlock(&w->mu);
    *wcur ^= 1;
}

/* ---- CUDA start-up off the critical path: runtime + context creation (hundreds of ms) overlaps reading the header */
static pthread_t g_warm_thread; static int g_warm_started;
static void *warm_main(void *arg)
{
    void *p = NULL;
    if (msg_host_alloc((int)(intptr_t)arg, 4096, &p) == MSG_OK) msg_host_free(p);
    return NULL;
}
static void warm_start(void)
{
    int dev = getenv("MSAMTOOLS_DEVICE") ? atoi(getenv("MSAMTOOLS_DEVICE")) : 0;
    if (getenv("MSAMTOOLS_NO_WARMUP")) return;
    g_warm_started = pthread_create(&g_warm_thread, NULL, warm_main, (void *)(intptr_t)dev) == 0;
}
static void warm_join(void) { if (g_warm_started) { g_warm_started = 0; pthread_join(g_warm_thread, NULL); } }

static void ring_buffer_alloc(ring_t *g, int i, int pin)
{   /* BAM: fixed-capacity buffers the inflate workers write into directly; pinned (so that H2D copies run asynchronously
       at full PCIe rate) once the input is large enough to pay for page-locking them */
    chunk_t *c = &g->buf[i];
    if (!g->bulk || c->raw) return;
    c->fixed = 1; c->cap = g->cap;
    void *pmem = NULL;
    if (pin && msg_host_alloc(g->r->cfg.device, c->cap, &pmem) == MSG_OK) { c->raw = pmem; c->pinned = 1; }
    else { c->raw = malloc(c->cap); if (!c->raw) mDie("Out of memory"); }
    chunk_reserve_off(c, 1);
    c->off[0] = 0;
}

static msg_ctx *run_stream(run_t *r)
{
    msg_ctx *ctx = NULL;
    r->cfg.abi_version = MSG_ABI_VERSION;
    r->cfg.n_ranks = 1;
    if (getenv("MSAMTOOLS_DEVICE")) r->cfg.device = atoi(getenv("MSAMTOOLS_DEVICE"));
    warm_join();
    if (msg_create(&r->cfg, &ctx)) mDie("%s", msg_last_error(NULL));
    double t_push = 0; size_t n_pushed = 0;
    struct timespec ta, tb;
    wring_t w; memset(&w, 0, sizeof w);
    pthread_mutex_init(&w.mu, NULL); pthread_cond_init(&w.cv, NULL);
    int wcur = 0;

    if (!r->eof) chunk_fill(&r->chunk, r->in, r->hdr, r->chunk.n + 1, (size_t)-1, &r->eof);      /* learn whether there is anything beyond the pre-flight sample */
    if (r->eof) {
        /* small input: everything is already in the pre-flight chunk, one synchronous push, no threads */
        chunk_t *c = &r->chunk;
        if (c->n) {
            clock_gettime(CLOCK_MONOTONIC, &ta);
            if (msg_push(ctx, c->raw, c->len, c->off, c->n)) gpu_die(ctx);
            clock_gettime(CLOCK_MONOTONIC, &tb);
            t_push += (tb.tv_sec - ta.tv_sec) + 1e-9 * (tb.tv_nsec - ta.tv_nsec); n_pushed += c->n;
            if (r->cfg.want_records) pull_kept_records(r, ctx, &w, &wcur);
        }
    } else {
        ring_t g; memset(&g, 0, sizeof g);
        g.r = r; g.posted_last = -1;
        g.bulk = bio_is_bam(r->in);
        pthread_mutex_init(&g.mu, NULL); pthread_cond_init(&g.cv, NULL);
        if (g.bulk) {
            struct stat sb;
            const char *e = getenv("MSAMTOOLS_PINNED");
            if (e) g.pin = atoi(e) != 0;
            else g.pin = r->path && strcmp(r->path, "-") != 0 && stat(r->path, &sb) == 0 && S_ISREG(sb.st_mode) && (size_t)sb.st_size >= ((size_t)192 << 20);
            /* (a pipe stays pageable: page-locking a buffer stalls the reader thread for ~0.1 s, and behind a pipe the staged
               copies are not what limits the stream) */
        }
        /* a chunk plus slack -- and never less than what the QNAME pre-flight already read (100 000 records: more than a chunk
           when records are long) */
        g.cap = CHUNK_BYTES + CHUNK_SLACK;
        if (r->chunk.len + CHUNK_SLACK > g.cap) g.cap = r->chunk.len + CHUNK_SLACK;
        ring_buffer_alloc(&g, 0, g.pin);                     /* the others are allocated by the reader thread when it first needs them */
        w.want_pinned = g.pin;
        {   /* the pre-flight records open buffer 0 */
            chunk_t *c = &g.buf[0], *s0 = &r->chunk;
            if (c->fixed) {
                if (s0->len > c->cap) mDie("Out of memory");
                memcpy(c->raw, s0->raw, s0->len);
            } else { c->raw = s0->raw; c->cap = s0->cap; s0->raw = NULL; }
            c->len = s0->len; c->n = s0->n;
            chunk_reserve_off(c, c->n + 1);
            memcpy(c->off, s0->off, (s0->n + 1) * sizeof(uint64_t));
        }
        pthread_t th, wth; int have_writer = 0;
        if (pthread_create(&th, NULL, reader_main, &g)) mDie("Cannot start the reader thread");
        if (r->cfg.want_records) { w.r = r; have_writer = pthread_create(&wth, NULL, writer_main, &w) == 0; if (!have_writer) w.r = NULL; }
        int cur = 0, inflight[2] = { -1, -1 };
        for (;;) {
            pthread_mutex_lock(&g.mu);
            while (!g.state[cur]) pthread_cond_wait(&g.cv, &g.mu);
            const int last = g.posted_last == cur;
            pthread_mutex_unlock(&g.mu);
            chunk_t *c = &g.buf[cur];
            if (c->k) {
                clock_gettime(CLOCK_MONOTONIC, &ta);
                if (msg_push_async(ctx, c->raw, (size_t)c->off[c->k], c->off, c->k)) gpu_die(ctx);
                if (r->cfg.want_records) pull_kept_records(r, ctx, &w, &wcur);      /* completes the chunk */
                clock_gettime(CLOCK_MONOTONIC, &tb);
                t_push += (tb.tv_sec - ta.tv_sec) + 1e-9 * (tb.tv_nsec - ta.tv_nsec); n_pushed += c->k;
            }
            /* the buffer pushed two calls ago is no longer referenced by the library */
            if (inflight[0] >= 0) {
                pthread_mutex_lock(&g.mu);
                g.state[inflight[0]] = 0;
                pthread_cond_broadcast(&g.cv);
                pthread_mutex_unlock(&g.mu);
            }
            inflight[0] = inflight[1]; inflight[1] = cur;
            if (last) break;
            cur = (cur + 1) % NBUF;
        }
        if (msg_wait(ctx)) gpu_die(ctx);
        pthread_join(th, NULL);
        if (have_writer) {
            pthread_mutex_lock(&w.mu);
            w.done = 1;
            pthread_cond_broadcast(&w.cv);
            pthread_mutex_unlock(&w.mu);
            pthread_join(wth, NULL);
            if (w.failed) mDie("Cannot write alignment record");
        }
        for (int i = 0; i < NBUF; i++) {
            if (g.buf[i].pinned) msg_host_free(g.buf[i].raw); else free(g.buf[i].raw);
            free(g.buf[i].off);
        }
        pthread_mutex_destroy(&g.mu); pthread_cond_destroy(&g.cv);
    }
    for (int i = 0; i < 2; i++) { if (w.pinned[i]) msg_host_free(w.buf[i]); else free(w.buf[i]); }
    pthread_mutex_destroy(&w.mu); pthread_cond_destroy(&w.cv);
    if (getenv("MSAMTOOLS_TIMING")) {      /* host-ingest vs GPU time, reported separately (BASELINE.json north_star) */
        uint64_t ib = 0; double isec = 0; msg_timing tm;
        bio_ingest_stats(r->in, &ib, &isec);
        msg_get_timing(ctx, &tm, 0);
        fprintf(stderr, "# timing: index walk %.3f s; record output %.3f s (writer thread)\n", g_walk_sec, w.t_write);
        fprintf(stderr, "# timing: host ingest %.3f GB in %.3f s (%.2f GB/s, read+inflate); push loop %.3f s (H2D %.3f GB, GPU kernels %.1f ms); %llu records\n",
                ib / 1e9, isec, isec > 0 ? ib / 1e9 / isec : 0.0, t_push, tm.h2d_bytes / 1e9, tm.total_ms, (unsigned long long)n_pushed);
    }
    return ctx;
}

static void open_input(run_t *r, const char *infile)
{
    r->path = infile;
    r->in = bio_open_read(infile);
    if (!r->in) mDie("Cannot open %s for reading", infile);
    warm_start();                                /* the device starts up while the header is read and parsed */
    bio_set_threads(r->in, host_threads());      /* BGZF blocks are inflated on worker threads */
    r->hdr = bio_read_header(r->in);
    if (!r->hdr) { if (bio_error(r->in)[0]) mDie("Cannot read header from %s: %s", infile, bio_error(r->in)); mDie("Cannot read header from %s", infile); }
}

/* ============================================================ filter */
static int filter_main(int argc, char *argv[])
{
    const char *sub = "filter";
    struct arg_lit *a_b = arg_lit0("b", NULL, "output BAM (default: false)");
    struct arg_lit *a_u = arg_lit0("u", NULL, "uncompressed BAM output (force -b) (default: false)");
    struct arg_lit *a_h = arg_lit0("h", NULL, "print header for the SAM output (default: false)");
    struct arg_lit *a_S = arg_lit0("S", NULL, "input is SAM (default: false)");
    struct arg_file *a_file = arg_filen(NULL, NULL, "<bamfile>", 1, 1, "input SAM/BAM file");
    struct arg_lit *a_help = arg_lit0(NULL, "help", "print this help and exit\n\nSpecific options:\n-----------------\n");
    struct arg_int *a_l = arg_int0("l", NULL, NULL, "min. length of alignment (default: 0)");
    struct arg_int *a_p = arg_int0("p", NULL, NULL, "min. sequence identity of alignment, in percent, integer in [0,100]; needs MD or NM (default: 0)");
    struct arg_int *a_ppt = arg_int0(NULL, "ppt", NULL, "min (positive) or max (negative) sequence identity in parts per thousand, integer in [-1000,1000]; needs MD or NM (default: 0)");
    struct arg_int *a_z = arg_int0("z", NULL, NULL, "min. percent of the query that must be aligned, integer in [0,100] (default: 0)");
    struct arg_lit *a_k = arg_lit0("k", "keep_unmapped", "report unmapped reads, when filtering using upper-limit thresholds (default: false)");
    struct arg_lit *a_v = arg_lit0("v", "invert", "invert the effect of the filter: report the complement among mapped alignments (default: false)");
    struct arg_lit *a_rescore = arg_lit0(NULL, "rescore", "rescore alignments using MD or NM fields, in that order (default: false)\n\n"
                                         "Special filters (need name-grouped input and AS, unless --rescore; cannot be combined with -v):\n");
    struct arg_lit *a_best = arg_lit0(NULL, "besthit", "keep all highest scoring hit(s) per read (default: false); input in any other order (e.g. sorted by\n"
                                      "coordinate) stays refused, as the output records would need SEQ/QUAL held on the GPU: filter it without\n"
                                      "--besthit and pipe it into 'profile --collate'");
    struct arg_lit *a_uniq = arg_lit0(NULL, "uniqhit", "keep only one highest scoring hit per read, only if it is unique (default: false)");
    struct arg_end *end = arg_end(16);
    void *argtable[] = { a_b, a_u, a_h, a_S, a_file, a_help, a_l, a_p, a_ppt, a_z, a_k, a_v, a_rescore, a_best, a_uniq, end };

    if (arg_nullcheck(argtable) != 0) mDie("insufficient memory");
    int nerrors = arg_parse(argc, argv, argtable);
    if (a_help->count > 0 || argc < 2) { print_help(sub, argtable); exit(EXIT_SUCCESS); }
    if (nerrors > 0) {
        arg_print_errors(stderr, end, PROGRAM);
        fprintf(stderr, "Use --help for usage instructions!\n");
        mQuit("");
    }
    if (a_file->count > 1) multiple_file_error(sub, argtable);

    int32_t PPT = 0, MAX_CLIP = 100, MIN_LENGTH = 0;
#define USAGE_FAIL(msg) do { fprintf(stdout, msg "\n"); print_help(sub, argtable); mQuit(""); } while (0)
    if (a_v->count > 0 && (a_best->count > 0 || a_uniq->count > 0)) USAGE_FAIL("--invert cannot be combined with --besthit or --uniqhit");
    else if (a_best->count > 0 && a_uniq->count > 0) USAGE_FAIL("--besthit cannot be combined with --uniqhit");
    else if (a_p->count > 0 && a_ppt->count > 0) USAGE_FAIL("-p cannot be combined with --ppt");
    else if (!a_l->count && !a_p->count && !a_ppt->count && !a_uniq->count && !a_best->count && !a_z->count)
        USAGE_FAIL("--mode filter needs -l, -p, --ppt, -z, --besthit or --uniqhit");
    else {
        if (a_p->count > 0) {
            int pid = a_p->ival[0];
            if (pid < 0 || pid > 100) USAGE_FAIL("-p must be in the range [0,100]");
            PPT = 10 * pid;
        } else if (a_ppt->count > 0) {
            PPT = a_ppt->ival[0];
            if (PPT < -1000 || PPT > 1000) USAGE_FAIL("--ppt must be in the range [-1000,1000]");
        }
        if (a_z->count > 0) {
            MAX_CLIP = 100 - a_z->ival[0];
            if (MAX_CLIP < 0 || MAX_CLIP > 100) USAGE_FAIL("-z must be in the range [0,100]");
        }
        if (a_l->count > 0) {
            MIN_LENGTH = a_l->ival[0];
            if (MIN_LENGTH < 0) USAGE_FAIL("-l must be a non-negative integer");
        }
    }
    char outmode[6] = "w";
    if (a_u->count > 0) strcat(outmode, "bu"); else if (a_b->count > 0) strcat(outmode, "b"); else if (a_h->count > 0) strcat(outmode, "h");

    run_t r; memset(&r, 0, sizeof r);
    phase(sub, NULL);
    open_input(&r, a_file->filename[0]);
    phase(sub, "open + header");
    const int hit = a_uniq->count > 0 ? MSG_HIT_UNIQUE : a_best->count > 0 ? MSG_HIT_BEST : MSG_HIT_NONE;
    qn_result qn = { QN_NOT_REQUIRED, 0, 0, 0 };
    if (hit) {
        chunk_fill(&r.chunk, r.in, r.hdr, COORD_ORDER_CHECK_RECORDS, (size_t)-1, &r.eof);
        qn = qname_preflight(r.hdr, &r.chunk);
    }
    /* provenance goes into a copy of the header (msam_filter.c:484-493) */
    r.out_hdr = bio_hdr_dup(r.hdr);
    if (!r.out_hdr) mDie("Cannot duplicate SAM header for output provenance");
    {
        char *cl = command_line(argc, argv), qmsg[1024], ds[1252];
        qn_format(&qn, qmsg, sizeof qmsg);
        snprintf(ds, sizeof ds, "git=%s; %s", MSAM_GIT_COMMIT, qmsg);
        if (bio_hdr_add_pg(r.out_hdr, PROGRAM, PROGRAM, PACKAGE_VERSION, cl, ds) < 0) mDie("Cannot add msamtools @PG record to SAM/BAM header");
        free(cl);
    }
    r.out = bio_open_write("-", outmode);
    if (!r.out) mDie("Cannot open - for writing");
    bio_set_threads(r.out, host_threads());
    if (bio_write_header(r.out, r.out_hdr) < 0) mDie("Cannot write SAM header");
    phase(sub, "pre-flight + output header");

    /* mFilterFileWrapper, msam_filter.c:79-84 */
    if (!(MIN_LENGTH > 0) && PPT == 0 && !(MAX_CLIP < 100) && !hit)
        mDie("'filter' command requires atleast one of --ppt, -l, -p, -z, --besthit or --uniqhit");

    r.cfg.do_filter = 1; r.cfg.hit_mode = (uint8_t)hit; r.cfg.invert = a_v->count > 0; r.cfg.keep_unmapped = a_k->count > 0;
    r.cfg.rescore = a_rescore->count > 0;
    r.cfg.min_length = MIN_LENGTH; r.cfg.ppt = PPT; r.cfg.max_clip = MAX_CLIP;
    r.cfg.want_records = 1;
    r.cfg.n_targets = r.hdr->n_targets; r.cfg.n_features = r.hdr->n_targets;
    msg_ctx *ctx = run_stream(&r);
    phase(sub, "stream");
    msg_destroy(ctx);
    bio_close(r.in);
    if (bio_close(r.out)) mDie("Cannot write output");
    phase(sub, "close");
    return 0;
}

/* ============================================================ profile */
static void print_insert_stats(gzp *s, int left, const char *type, int number, int total, const char *post)
{   /* mPrintInsertStats, msam_profile.c:434-470 */
    int width = 7;
    if (total > 0) width = 1 + log10(total);
    gzp_printf(s, "# ");
    if (left) gzp_printf(s, "%-20s: ", type); else gzp_printf(s, "%20s: ", type);
    if (strcmp(type, "Total inserts") == 0 && number == -1) gzp_printf(s, "%*s (", width, "NA"); else gzp_printf(s, "%*d (", width, number);
    if (total > 0) gzp_printf(s, "%6.2f", 100.0 * number / total); else gzp_printf(s, "%6s", "NA");
    gzp_printf(s, "%%)");
    if (post) gzp_printf(s, " %s\n", post); else gzp_printf(s, "\n");
}
static void print_insert_stats_double(gzp *s, const char *type, double number, int total, const char *post)
{   /* mPrintInsertStatsDouble, msam_profile.c:472-499 (always left aligned by its callers) */
    gzp_printf(s, "# ");
    gzp_printf(s, "%-20s: ", type);
    gzp_printf(s, "%10.7g (", number);
    if (total > 0) gzp_printf(s, "%6.2f", 100.0 * number / total); else gzp_printf(s, "%6s", "NA");
    gzp_printf(s, "%%)");
    if (post) gzp_printf(s, " %s\n", post); else gzp_printf(s, "\n");
}

/* the "<name>\t%.8g\n" rows of mWriteMatrixTransposedGzip (mMatrix.c:359-376): row ranges are formatted on worker threads
 * (same printf conversion, so the same text), then handed to the gzip writer in order */
typedef struct { char **name; const double *v; size_t a, b; char *buf; size_t len; int err; } row_job;
static void *row_worker(void *arg)
{
    row_job *j = arg;
    size_t cap = 1;
    for (size_t i = j->a; i < j->b; i++) cap += strlen(j->name[i]) + 40;
    char *d = j->buf = malloc(cap);
    if (!d) { j->err = 1; return NULL; }
    for (size_t i = j->a; i < j->b; i++) {
        const size_t l = strlen(j->name[i]);
        memcpy(d, j->name[i], l); d += l; *d++ = '\t';
        const double x = j->v[i];
        if (x == 0.0 && !signbit(x)) *d++ = '0';             /* what %.8g prints for +0 */
        else d += snprintf(d, 38, "%.8g", x);
        *d++ = '\n';
    }
    j->len = (size_t)(d - j->buf);
    return NULL;
}
static void write_rows(gzp *out, char **name, const double *v, size_t n, int threads)
{
    enum { SLAB = 1 << 16 };                                  /* rows per job: bounds the text held in memory */
    for (size_t base = 0; base < n;) {
        int t = threads;
        if ((size_t)t * SLAB > n - base) t = (int)((n - base + SLAB - 1) / SLAB);
        pthread_t th[16]; row_job job[16]; int spawned[16];
        for (int i = 0; i < t; i++) {
            size_t a = base + (size_t)i * SLAB, b = a + SLAB > n ? n : a + SLAB;
            job[i] = (row_job){ name, v, a, b, NULL, 0, 0 };
            spawned[i] = i && pthread_create(&th[i], NULL, row_worker, &job[i]) == 0;
        }
        for (int i = 0; i < t; i++) { if (spawned[i]) pthread_join(th[i], NULL); else row_worker(&job[i]); }
        for (int i = 0; i < t; i++) {
            if (job[i].err || gzp_write(out, job[i].buf, job[i].len)) mDie("Cannot write the profile");
            free(job[i].buf);
        }
        base += (size_t)t * SLAB;
    }
}

static int profile_main(int argc, char *argv[])
{
    const char *sub = "profile";
    struct arg_lit *a_S = arg_lit0("S", NULL, "input is SAM (default: false)");
    struct arg_file *a_file = arg_filen(NULL, NULL, "<bamfile>", 1, 1, "input SAM/BAM file");
    struct arg_lit *a_help = arg_lit0(NULL, "help", "print this help and exit\n\nSpecific options:\n-----------------\n");
    struct arg_str *a_out = arg_str1("o", NULL, "<file>", "name of output file (required)");
    struct arg_str *a_label = arg_str1(NULL, "label", NULL, "label to use for the profile; typically the sample id (required)");
    struct arg_str *a_genome = arg_str0(NULL, "genome", NULL, "tab-delimited genome definition file - 'genome-id<tab>seq-id' (default: none)");
    struct arg_int *a_mincount = arg_int0(NULL, "mincount", NULL, "minimum number of inserts mapped to a feature, below which the feature is counted as absent (default: 0)");
    struct arg_int *a_total = arg_int0(NULL, "total", NULL, "number of high-quality inserts (mate-pairs/paired-ends) that were input to the aligner (default: unknown)");
    struct arg_str *a_unit = arg_str0(NULL, "unit", NULL, "unit of abundance to report {ab | rel | fpkm | tpm} (default: rel)");
    struct arg_lit *a_pandas = arg_lit0(NULL, "pandas", "print two columns (ID, sample-label) as header compatible with python pandas (default)");
    struct arg_lit *a_nopandas = arg_lit0(NULL, "no-pandas", "use legacy profile header without the ID column");
    struct arg_lit *a_nolen = arg_lit0(NULL, "nolen", "do not normalize the abundance (only relevant for ab or rel) for sequence length (default: normalize)");
    struct arg_str *a_multi = arg_str0(NULL, "multi", NULL, "how to deal with multi-mappers {all | equal | proportional | ignore} (default: proportional)\n\n"
                                       "Inserts (all alignments of one QNAME) are counted per reference sequence, or per genome with --genome.\n"
                                       "An insert hitting N features adds 1 to each (all), 1/N to each (equal), a share proportional to the\n"
                                       "features' current abundances (proportional), or nothing (ignore). Input must be grouped by QNAME and\n"
                                       "already filtered (see 'filter').");
    struct arg_lit *a_collate = arg_lit0(NULL, "collate", "input need not be grouped by QNAME (e.g. sorted by coordinate): the records are grouped on the GPU\n"
                                         "(default: false; without it, input must be grouped by QNAME)");
    struct arg_end *end = arg_end(20);
    void *argtable[] = { a_S, a_file, a_help, a_out, a_label, a_genome, a_total, a_mincount, a_unit, a_pandas, a_nopandas, a_nolen, a_multi, a_collate, end };

    if (arg_nullcheck(argtable) != 0) mDie("insufficient memory");
    int nerrors = arg_parse(argc, argv, argtable);
    if (a_help->count > 0 || argc < 2) { print_help(sub, argtable); exit(EXIT_SUCCESS); }
    if (nerrors > 0) {
        arg_print_errors(stdout, end, PROGRAM);
        fprintf(stdout, "Use --help for usage instructions!\n");
        mQuit("");
    }
    if (a_file->count > 1) multiple_file_error(sub, argtable);
    if (a_label->count != 1 || a_out->count != 1) USAGE_FAIL("requires --label and -o");
    if (a_pandas->count > 0 && a_nopandas->count > 0) USAGE_FAIL("--pandas and --no-pandas cannot be used together");
    int total_inserts = -1;
    if (a_total->count > 0) { total_inserts = a_total->ival[0]; if (total_inserts <= 0) USAGE_FAIL("--total must be a positive integer"); }
    if (a_mincount->count > 0 && a_mincount->ival[0] < 0) USAGE_FAIL("--mincount must be a non-negative integer");

    run_t r; memset(&r, 0, sizeof r);
    phase(sub, NULL);
    open_input(&r, a_file->filename[0]);
    phase(sub, "open + header");
    chunk_fill(&r.chunk, r.in, r.hdr, COORD_ORDER_CHECK_RECORDS, (size_t)-1, &r.eof);
    qn_result qn = { QN_NOT_REQUIRED, 0, 0, 0 };
    if (a_collate->count == 0) qn = qname_preflight(r.hdr, &r.chunk);

    /* any prefix matches, first hit in this order (msam_profile.c:712-748) */
    int share_type = MSG_MULTI_PROPORTIONAL, unit_type = 1;
    if (a_multi->count > 0) {
        const char *types[5] = { "", "all", "equal", "proportional", "ignore" };
        share_type = -1;
        for (int i = 1; i <= 4; i++) if (strncmp(a_multi->sval[0], types[i], strlen(a_multi->sval[0])) == 0) { share_type = i; break; }
        if (share_type == -1) mDie("Do not understand --multi=%s", a_multi->sval[0]);
    }
    if (a_unit->count > 0) {
        const char *types[5] = { "", "relative", "fpkm", "tpm", "abundance" };
        unit_type = -1;
        for (int i = 1; i <= 4; i++) if (strncmp(a_unit->sval[0], types[i], strlen(a_unit->sval[0])) == 0) { unit_type = i; break; }
        if (unit_type == -1) mDie("Do not understand --unit=%s", a_unit->sval[0]);
    }
    int length_normalize = 1;
    if (unit_type == 1 || unit_type == 4) length_normalize = (a_nolen->count == 0);

    /* feature map: identity, or --genome in the reference's key order (msam_profile.c:757-852) */
    const int n_targets = r.hdr->n_targets;
    int32_t *fmap = malloc(sizeof(int32_t) * (size_t)(n_targets ? n_targets : 1));
    for (int i = 0; i < n_targets; i++) fmap[i] = -1;
    int n_features; char **feature_name; uint32_t *feature_len;
    keyorder *genomes = NULL;
    if (a_genome->count > 0) {
        char line[4096], gname[4096], sname[4096];
        FILE *def = fopen(a_genome->sval[0], "r");
        if (!def) mDie("Cannot open file %s", a_genome->sval[0]);
        genomes = ko_new();
        while (fgets(line, sizeof line, def)) {
            if (sscanf(line, "%s\t%s", gname, sname) != 2) mDie("GENOME DEFINITION LINE ERROR");
            ko_add(genomes, gname);
        }
        rewind(def);
        n_features = (int)ko_size(genomes);
        while (fgets(line, sizeof line, def)) {
            if (sscanf(line, "%s\t%s", gname, sname) != 2) mDie("GENOME DEFINITION LINE ERROR");
            long gid = ko_find(genomes, gname);
            int sid = bio_hdr_tid(r.hdr, sname);
            if (gid < 0) mDie("Genome '%s' not found in BAM file", gname);
            if (sid < 0) mDie("Sequence '%s' not found in BAM file", sname);
            fmap[sid] = (int32_t)gid;
        }
        fclose(def);
        feature_len = calloc((size_t)(n_features ? n_features : 1), sizeof(uint32_t));
        for (int i = 0; i < n_targets; i++) {
            if (fmap[i] == -1) mDie("Sequence '%s' not found in genome definition", r.hdr->target_name[i]);
            feature_len[fmap[i]] += r.hdr->target_len[i];
        }
        feature_name = malloc(sizeof(char *) * (size_t)(n_features ? n_features : 1));
        for (int i = 0; i < n_features; i++) feature_name[i] = (char *)ko_key(genomes, (size_t)i);
    } else {
        for (int i = 0; i < n_targets; i++) fmap[i] = i;
        n_features = n_targets; feature_name = r.hdr->target_name; feature_len = r.hdr->target_len;
    }

    r.cfg.do_filter = 0; r.cfg.want_profile = 1; r.cfg.share_type = (uint8_t)share_type;
    r.cfg.collate = a_collate->count > 0;
    /* MSAMTOOLS_EXACT=1: abundances bit-identical to the reference (--multi=equal / proportional; msg_config.exact) */
    r.cfg.exact = getenv("MSAMTOOLS_EXACT") && atoi(getenv("MSAMTOOLS_EXACT")) != 0;
    r.cfg.n_targets = n_targets; r.cfg.n_features = n_features; r.cfg.fmap = fmap;
    phase(sub, "pre-flight + feature map");
    msg_ctx *ctx = run_stream(&r);
    phase(sub, "stream");
    double *ab = calloc((size_t)n_features + 1, sizeof(double));      /* ab[0] = Unknown, ab[1..] features */
    msg_profile_stats st;
    if (msg_finish_profile(ctx, ab + 1, &st)) gpu_die(ctx);
    msg_destroy(ctx);
    phase(sub, "finish");
    if (share_type == MSG_MULTI_PROPORTIONAL) {                        /* stderr side channel, msam_profile.c:330,381-390,405 */
        fprintf(stderr, "# Start PropSharing:\n");
        for (int k = 1; k <= st.em_iterations; k++) {
            fprintf(stderr, "#     PropSharing Iteration: %2d; DELTA^2=%g", k, st.em_delta[k - 1]);
            if (k == st.em_iterations && st.em_converged) fprintf(stderr, ". CONVERGED!\n"); else fprintf(stderr, "\n");
        }
        fprintf(stderr, "# End   PropSharing!\n");
        fprintf(stderr, "# Purged %d inserts that mapped to features without unique inserts.\n", (int)st.purged_insert_count);
    }
    int mapped_inserts = (int)st.mapped_inserts;
    double purged_eq = 0;
    if (a_mincount->count > 0) {                                       /* msam_profile.c:858-869 */
        int mincount = a_mincount->ival[0];
        for (int i = 1; i <= n_features; i++) if (ab[i] < mincount) { purged_eq += ab[i]; ab[i] = 0; }
        fprintf(stderr, "# Purged %.7g insert-equivalents from low-abundance features based on --mincount.\n", purged_eq);
    }
    if (total_inserts > 0 && total_inserts < mapped_inserts) {
        fprintf(stderr, "# Ignoring 'unknown' fraction, as total inserts (%d) < mapped inserts (%d)!\n", total_inserts, mapped_inserts);
        total_inserts = -1;
    }
    gzp *out = gzp_open(a_out->sval[0], host_threads());
    if (!out) mDie("Cannot open %s for writing", a_out->sval[0]);
    {   /* mPrintProfileProvenanceGzip */
        char *cl = command_line(argc, argv), qmsg[1024];
        qn_format(&qn, qmsg, sizeof qmsg);
        gzp_printf(out, "# msamtools version: %s\n", PACKAGE_VERSION);
        gzp_printf(out, "# msamtools git commit: %s\n", MSAM_GIT_COMMIT);
        gzp_printf(out, "# Command line: %s\n", cl);
        gzp_printf(out, "# %s\n", qmsg);
        free(cl);
    }
    double purged_inserts = st.purged_insert_count + purged_eq;
    double effective = mapped_inserts - purged_inserts;
    if (share_type == MSG_MULTI_IGNORE) effective -= st.multi_mapper_count;
    print_insert_stats(out, 1, "Total inserts", total_inserts, total_inserts, NULL);
    print_insert_stats(out, 1, "Mapped inserts", mapped_inserts, total_inserts, NULL);
    print_insert_stats(out, 0, "- Multiple mapped ", (int)st.multi_mapper_count, total_inserts, NULL);
    print_insert_stats(out, 0, "- Uniquely mapped ", (int)st.uniq_mapper_count, total_inserts, NULL);
    print_insert_stats_double(out, "Purged inserts", purged_inserts, total_inserts, "due to ambiguous mapping or low abundance features");
    print_insert_stats_double(out, "Effective inserts", effective, total_inserts, NULL);
    if (total_inserts <= 0) gzp_printf(out, "# Estimated seq. length for 'Unknown': NA\n");
    if (total_inserts > 0) {                                           /* msam_profile.c:906-934 */
        ab[0] = total_inserts - mapped_inserts + purged_inserts;
        if (share_type == MSG_MULTI_IGNORE) ab[0] += st.multi_mapper_count;
        if (length_normalize) {
            int count = 0; uint64_t sum = 0;
            for (int i = 0; i < n_features; i++) { sum += feature_len[i]; count++; }
            uint32_t unknown_size = (uint32_t)(sum / (uint64_t)count);
            gzp_printf(out, "# Estimated seq. length for 'Unknown': %dbp\n", unknown_size);
            ab[0] = 1.0 * ab[0] / unknown_size;
        } else gzp_printf(out, "# Estimated seq. length for 'Unknown': NA\n");
    }
    if (length_normalize) for (int i = 0; i < n_features; i++) ab[i + 1] /= feature_len[i];
    if (unit_type == 2) {                                              /* fpkm */
        double f = total_inserts > 0 ? 1.0E9 / total_inserts : 1.0E9 / mapped_inserts;
        for (int i = 0; i <= n_features; i++) ab[i] *= f;
    } else if (unit_type == 3 || unit_type == 1) {                     /* tpm / rel: row-normalise incl. Unknown (mMatrix.c:168-179) */
        double sum = 0;
        for (int i = 0; i <= n_features; i++) sum += ab[i];
        for (int i = 0; i <= n_features; i++) ab[i] /= sum;
        if (unit_type == 3) for (int i = 0; i <= n_features; i++) ab[i] *= 1.0E6;
    }
    if (a_nopandas->count == 0) gzp_printf(out, "ID\t");                 /* mWriteMatrixTransposedGzip, mMatrix.c:359-376 */
    gzp_printf(out, "%s\n", a_label->sval[0]);
    gzp_printf(out, "%s\t%.8g\n", "Unknown", ab[0]);
    write_rows(out, feature_name, ab + 1, (size_t)n_features, host_threads());
    if (gzp_close(out)) mDie("Cannot write %s", a_out->sval[0]);
    phase(sub, "table");
    bio_close(r.in);
    return 0;
}

/* ============================================================ coverage */
/* the depth values of one sequence, `wordsize` per line (mWriteCoverageToStream, msam_coverage.c:160-185); depth == NULL: zeros */
static void write_depths(gzp *out, const int32_t *depth, int64_t tlen, int wordsize)
{
    enum { STEP = 8192 };
    if (tlen <= 0) { gzp_puts(out, "0\n"); return; }           /* the reference's loops print one value even then */
    for (int64_t base = 0; base < tlen; base += STEP) {
        const int64_t end = base + STEP < tlen ? base + STEP : tlen;
        char *d = gzp_reserve(out, (size_t)STEP * 12), *d0 = d;
        if (!d) mDie("Cannot write coverage");
        for (int64_t i = base; i < end; i++) {
            int32_t v = depth ? depth[i] : 0;
            if (v < 0) { *d++ = '-'; }
            uint32_t u = v < 0 ? 0u - (uint32_t)v : (uint32_t)v;
            char tmp[10]; int k = 0;
            do { tmp[k++] = (char)('0' + u % 10); u /= 10; } while (u);
            while (k) *d++ = tmp[--k];
            *d++ = (i == tlen - 1 || (i + 1) % wordsize == 0) ? '\n' : ' ';
        }
        gzp_commit(out, (size_t)(d - d0));
    }
}

static int coverage_main(int argc, char *argv[])
{
    const char *sub = "coverage";
    struct arg_lit *a_S = arg_lit0("S", NULL, "input is SAM (default: false)");
    struct arg_file *a_file = arg_filen(NULL, NULL, "<bamfile>", 1, 1, "input SAM/BAM file");
    struct arg_lit *a_help = arg_lit0(NULL, "help", "print this help and exit\n\nSpecific options:\n-----------------\n");
    struct arg_str *a_out = arg_str1("o", NULL, "<file>", "name of output file (required)");
    struct arg_lit *a_summary = arg_lit0(NULL, "summary", "do not report per-position coverage but report fraction of sequence covered (default: false)");
    struct arg_lit *a_skip = arg_lit0("x", "skipuncovered", "do not report coverage for sequences without aligned reads (default: false)");
    struct arg_int *a_w = arg_int0("w", "wordsize", NULL, "number of words (coverage values) per line (default: 17)");
    struct arg_lit *a_gz = arg_lit0("z", "gzip", "compress output file using gzip (default; option retained for backward compatibility)\n\n"
                                    "Coverage is aligned query-base depth per reference position: CIGAR M, = and X count, D and N do not.\n"
                                    "Output is always gzip-compressed; no '.gz' is appended to the file name.");
    struct arg_end *end = arg_end(20);
    void *argtable[] = { a_S, a_file, a_help, a_out, a_summary, a_skip, a_w, a_gz, end };
    int wordsize = 17;

    if (arg_nullcheck(argtable) != 0) mDie("insufficient memory");
    int nerrors = arg_parse(argc, argv, argtable);
    if (a_help->count > 0 || argc < 2) { print_help(sub, argtable); exit(EXIT_SUCCESS); }
    if (nerrors > 0) {
        arg_print_errors(stderr, end, PROGRAM);
        fprintf(stderr, "Use --help for usage instructions!\n");
        mQuit("");
    }
    if (a_file->count > 1) multiple_file_error(sub, argtable);
    if (a_w->count > 0) { wordsize = a_w->ival[0]; if (wordsize < 1) USAGE_FAIL("-w must be a non-zero positive integer"); }
    if (a_out->count != 1) USAGE_FAIL("requires -o");

    gzp *out = gzp_open(a_out->sval[0], host_threads());
    if (!out) mDie("Cannot open %s for writing", a_out->sval[0]);
    run_t r; memset(&r, 0, sizeof r);
    open_input(&r, a_file->filename[0]);
    const int T = r.hdr->n_targets;
    r.cfg.do_filter = 0; r.cfg.want_coverage = 1; r.cfg.coverage_summary = a_summary->count > 0; r.cfg.n_targets = T; r.cfg.n_features = T; r.cfg.target_len = r.hdr->target_len;
    msg_ctx *ctx = run_stream(&r);
    uint8_t *covered = calloc((size_t)(T ? T : 1), 1);
    int64_t *touched = calloc((size_t)(T ? T : 1), sizeof(int64_t)), *sum = calloc((size_t)(T ? T : 1), sizeof(int64_t));
    if (msg_finish_coverage(ctx, covered, touched, sum)) gpu_die(ctx);
    const int skip = a_skip->count > 0;
    if (a_summary->count > 0) {                                        /* mWriteCoverageSummaryToStream, msam_coverage.c:189-219 */
        for (int t = 0; t < T; t++) {
            int64_t tlen = r.hdr->target_len[t];
            if (!covered[t]) { if (!skip) gzp_printf(out, "%s\t%d\t%d\n", r.hdr->target_name[t], 0, 0); continue; }
            gzp_printf(out, "%s\t%.8f\t%.2f\n", r.hdr->target_name[t], 1.0 * touched[t] / tlen, 1.0 * sum[t] / tlen);
        }
    } else {                                                           /* mWriteCoverageToStream, msam_coverage.c:143-187 */
        int32_t *depth = NULL; size_t dcap = 0;
        for (int t = 0; t < T; t++) {
            int64_t tlen = r.hdr->target_len[t];
            if (!covered[t]) {
                if (!skip) {
                    gzp_printf(out, ">%s\n", r.hdr->target_name[t]);
                    write_depths(out, NULL, tlen, wordsize);
                }
                continue;
            }
            if ((size_t)tlen > dcap) { dcap = (size_t)tlen; depth = realloc(depth, dcap * sizeof(int32_t)); }
            if (msg_pull_coverage(ctx, t, depth)) gpu_die(ctx);
            gzp_printf(out, ">%s\n", r.hdr->target_name[t]);
            write_depths(out, depth, tlen, wordsize);
        }
        free(depth);
    }
    if (gzp_close(out)) mDie("Cannot write %s", a_out->sval[0]);
    msg_destroy(ctx);
    bio_close(r.in);
    return 0;
}

/* ============================================================ dispatch (msamtools.c:8-49) */
static int usage(FILE *out)
{
    fprintf(out, "\n");
    fprintf(out, "Program: %s (Metagenomics-related extension to samtools)\n", PROGRAM);
    fprintf(out, "Version: %s (git %s; GPU hot path libmsamtools_b200 ABI %d, own BAM/SAM I/O over zlib %s)\n", PACKAGE_VERSION, MSAM_GIT_COMMIT, msg_abi_version(), zlibVersion());
    fprintf(out, "\n");
    fprintf(out, "Usage:   %s <command> [options]\n\n", PROGRAM);
    fprintf(out, "Commands:\n");
    fprintf(out, " -- Filtering\n");
    fprintf(out, "     filter         filter alignments based on alignment statistics\n");
    fprintf(out, "\n");
    fprintf(out, " -- Profiling\n");
    fprintf(out, "     profile        estimate relative abundance profile of reference sequences or genomes in bam file\n");
    fprintf(out, "\n");
    fprintf(out, " -- Coverage\n");
    fprintf(out, "     coverage       estimate per-base or per-sequence read coverage of each reference sequence\n");
    fprintf(out, "\n");
    return 1;
}

int main(int argc, char *argv[])
{
    if (argc < 2) return usage(stderr);
    if (strcmp(argv[1], "filter") == 0) return filter_main(argc - 1, argv + 1);
    else if (strcmp(argv[1], "profile") == 0) return profile_main(argc - 1, argv + 1);
    else if (strcmp(argv[1], "coverage") == 0) return coverage_main(argc - 1, argv + 1);
    else if (strcmp(argv[1], "help") == 0) { usage(stdout); return 0; }
    else if (strcmp(argv[1], "summary") == 0) {
        fprintf(stderr, "[msamtools] 'summary' is not part of the GPU-accelerated path; use the CPU msamtools for it\n");
        return 1;
    } else {
        fprintf(stderr, "[msamtools] unrecognized command '%s'\n", argv[1]);
        usage(stderr);
        return 1;
    }
}
