/*
 * IMSAME_allvsall -- the reference's all-vs-all workflow (bin/all_vs_all_metagenomes_IMSAME.sh:27-58)
 * in ONE process: same arguments, same output files (OUT/X-Y.align and OUT/X-Y.r.align, byte for byte
 * what the script produces with the drop-in IMSAME and revComp), same resume rule (existing outputs
 * are kept) -- but every sample is parsed once, its reverse complement (src/reverseComplement.c, incl.
 * the reversed record order that renumbers db_seq) is built in memory instead of a temporary Y.r.EXT
 * file, and the comparisons run on a few long-lived CUDA contexts.  A sample is uploaded and packed
 * once per context (imsame_gpu_sample_create): it stays on the device as the database of later
 * comparisons, keeps the word table built for it as a query, and its reverse complement is made on the
 * device from the packed form (imsame_gpu_sample_revcomp).  The script starts 56 IMSAME and 28 revComp
 * processes for 8 samples and re-parses every file 14 times.
 *
 * usage: IMSAME_allvsall metagenomes_directory coverage similarity threads file_extension outpath
 *                        [-device D] [-gpus N] [-jobs J]
 *   -device D   first CUDA device (default 0)
 *   -gpus N     use the devices D .. D+N-1 (default 1)
 *   -jobs J     comparisons in flight (default N): J worker threads, each with its own CUDA context, go
 *               round-robin over the N devices.  J > N puts several workers on one GPU, so that one
 *               renders its records while another aligns.  The output files do not depend on N or J.
 *
 * A unit is one output file (X, Y, strand); the canonical order is the script's loop order.  A free worker
 * takes the next pending unit, preferring one whose query sample's word table it holds, then one whose
 * database read set it holds, then the lowest canonical index, and writes that unit's file itself.  The
 * [INFO] line of every unit goes to stdout in canonical order.  When a unit fails, no later unit is started,
 * every earlier one is finished and the units in flight complete; then the earliest failure is reported
 * exactly as with -jobs 1 (exit status 255).
 *
 * Each sample's two host parses (forward, revComp) are built once and shared.  The device read sets are
 * per worker (imsame_gpu_align_samples stores the word table in the query sample and points its context at
 * it) and held within a budget: half of the worker's share of the device's free memory once every context
 * exists (the other half stays free for the work buffers of the runs).  A read set that no pending or
 * running unit needs any more is released; to make room, the least recently used read sets that the unit
 * does not need are evicted.  A unit whose read sets do not fit the budget on their own, whose database is
 * larger than one segment (2^29 bases), or that still meets IMSAME_ENOMEM after everything else was
 * evicted, runs from host buffers (imsame_gpu_align).
 *
 * Environment: IMSAME_TRACE (phase times; one line per worker at the end: device, units, uploads, table
 * builds, evictions, host-path fallbacks, busy seconds), IMSAME_NO_RESIDENT (every unit from host buffers),
 * IMSAME_TEST_SAMPLE_BUDGET (test hook: the budget of every worker in bytes), IMSAME_TEST_FAIL_ALLOC (test hook of the
 * library: chosen device allocations of every context fail), IMSAME_FAST_EXIT.
 */
#define _GNU_SOURCE
#include <dirent.h>
#include <errno.h>
#include <inttypes.h>
#include <locale.h>
#include <math.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <time.h>
#include <unistd.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#include "imsame_host.h"
#include "imsame_job.h"

static void terror(const char *s) { /* src/commonFunctions.c:10-13 */
    printf("ERR**** %s ****\n", s);
    exit(-1);
}

static double now_s(void) {
    struct timespec t;
    clock_gettime(CLOCK_MONOTONIC, &t);
    return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec;
}

typedef struct {
    char *name;            /* file name without ".EXT" */
    pthread_mutex_t lock;  /* the parses below are built once, by the first worker that needs them */
    imsame_fasta fwd, rev; /* parsed forward sample / parsed revComp(sample): what the records are rendered from */
    int have_fwd, have_rev;
    const char *fwd_err, *rev_err; /* a parse failed: its terror text */
    int has_u;                     /* the file contains a 'U' (imsame_revcomp_load, imsame_revcomp_on_device) */
    int mirror;                    /* -1 unknown, else imsame_revcomp_on_device(fwd, rev, has_u) */
    int uses[2];                   /* pending or running units that need the forward / reverse read set (G.lock) */
} sample;

enum { U_PENDING, U_RUNNING, U_DONE, U_FAILED };

typedef struct {
    int i, j, rev; /* OUT/<i>-<j>[.r].align */
    int state;     /* G.lock */
    char *text;    /* U_DONE: the [INFO] line; U_FAILED: the terror text */
} unit;

/* A worker: one thread, one context, its own device read sets.  Read set x is the forward one of sample x / 2
 * (x even) or its reverse complement (x odd). */
typedef struct {
    int id, device;
    imsame_ctx *ctx;
    int ctx_rc;
    uint64_t budget, held; /* bytes of device read sets (estimates: set_bytes, table_bytes) */
    imsame_sample **dev;
    uint64_t *bytes, *last, tick;
    unsigned char *tab; /* [sample]: the forward read set carries its word table */
    uint64_t units, uploads, tables, evictions, fallbacks;
    double busy;
} worker;

static struct {
    pthread_mutex_t lock;
    pthread_barrier_t start;
    sample *sm;
    size_t n;
    unit *u;
    size_t nu, first, stop; /* units [0, first) are not pending; none at or after `stop` (earliest failure) starts */
    size_t printed;         /* [INFO] lines of units [0, printed) are out */
    uint64_t done;
    const char *dir, *ext, *out;
    imsame_job_opts jo;
    int no_resident, n_gpus, n_workers, omp_threads;
    long long test_budget; /* IMSAME_TEST_SAMPLE_BUDGET, -1 = none */
} G;

static int by_name(const void *a, const void *b) { return strcoll(((const sample *)a)->name, ((const sample *)b)->name); }

static int exists(const char *path) {
    struct stat st;
    return stat(path, &st) == 0 && S_ISREG(st.st_mode);
}

static void unit_path(const unit *u, char *path, size_t len) {
    snprintf(path, len, "%s/%s-%s%s.align", G.out, G.sm[u->i].name, G.sm[u->j].name, u->rev ? ".r" : "");
}

/* ---- host parses (shared, read-only once built) ---- */
static const char *need_forward(sample *s) {
    pthread_mutex_lock(&s->lock);
    if (!s->have_fwd && !s->fwd_err) {
        char path[4096];
        snprintf(path, sizeof path, "%s/%s.%s", G.dir, s->name, G.ext);
        if (imsame_fasta_load(path, 1, &s->fwd)) s->fwd_err = "Could not allocate memory for database vector";
        else s->have_fwd = 1;
    }
    const char *e = s->fwd_err;
    pthread_mutex_unlock(&s->lock);
    return e;
}

static const char *need_reverse(sample *s) {
    pthread_mutex_lock(&s->lock);
    if (!s->have_rev && !s->rev_err) {
        char path[4096];
        snprintf(path, sizeof path, "%s/%s.%s", G.dir, s->name, G.ext);
        switch (imsame_revcomp_load(path, &s->rev, &s->has_u)) {
            case 0: s->have_rev = 1; break;
            case 1: s->rev_err = "opening IN sequence FASTA file"; break;
            case 2: s->rev_err = "memory for Seq"; break;
            default: s->rev_err = "Could not allocate memory for database vector"; break;
        }
    }
    const char *e = s->rev_err;
    pthread_mutex_unlock(&s->lock);
    return e;
}

/* The device reverse complement works on the packed forward reads; revComp works on the text, and its filter is
   not the loader's (imsame_revcomp_is_mirror, host/fasta.c: '\r' / '-' / digits inside a record, 'U', header lines
   with several '>').  The device path is taken only when the parse of revComp's text IS the mirror image of the
   sample, otherwise that parse is uploaded.  (Both parses exist when this is asked.) */
static int sample_mirror(sample *s) {
    pthread_mutex_lock(&s->lock);
    if (s->mirror < 0) s->mirror = imsame_revcomp_on_device(&s->fwd, &s->rev, s->has_u) != 0;
    const int m = s->mirror;
    pthread_mutex_unlock(&s->lock);
    return m;
}

static void gpu_msg(char *msg, size_t ml, const char *what, int rc, imsame_ctx *ctx) {
    snprintf(msg, ml, "%s: %s / %s", what, imsame_gpu_strerror(rc), ctx ? imsame_gpu_last_cuda_error(ctx) : "");
}

/* ---- the per-worker device read sets ---- */
/* device bytes of a read set (capi_samples.inc: packed bases, read offsets, 64-base block index, word breaks) */
static uint64_t set_bytes(const imsame_fasta *f) {
    return f->total_len / 4 + f->total_len / 16 + 4 * (f->n_seqs + 2) + 4 * f->n_breaks + 1024;
}
/* its word table as a query: offsets over the 4^12 words + one 24-byte entry per word (qtable.cuh) */
static uint64_t table_bytes(const imsame_fasta *f) { return 4 * ((1ull << 24) + 1) + 24 * f->total_len; }

/* read set x leaves the worker's books; the caller frees what is returned */
static imsame_sample *take(worker *w, int x) {
    imsame_sample *s = w->dev[x];
    w->dev[x] = NULL;
    w->held -= w->bytes[x];
    w->bytes[x] = 0;
    if (!(x & 1)) w->tab[x / 2] = 0;
    return s;
}

static void drop(worker *w, int x) { imsame_gpu_sample_free(w->ctx, take(w, x)); }

static int kept(const int *keep, int nkeep, int x) {
    for (int k = 0; k < nkeep; k++)
        if (keep[k] == x) return 1;
    return 0;
}

/* evict least recently used read sets outside `keep` until `need` more bytes fit the budget (need = ~0: all) */
static void make_room(worker *w, const int *keep, int nkeep, uint64_t need) {
    while (need == ~0ull || w->held + need > w->budget) {
        int victim = -1;
        for (int x = 0; x < (int)(2 * G.n); x++)
            if (w->dev[x] && !kept(keep, nkeep, x) && (victim < 0 || w->last[x] < w->last[victim])) victim = x;
        if (victim < 0) return;
        drop(w, victim);
        w->evictions++;
    }
}

/* read set x from the host parse `src`, or (src == NULL) as the device reverse complement of read set x - 1.
   0: made; 1: IMSAME_ENOMEM even after evicting everything outside `keep`; -1: error (msg) */
static int make_set(worker *w, int x, const imsame_fasta *src, uint64_t bytes, const int *keep, int nkeep, const char *what,
                    char *msg, size_t ml) {
    for (int attempt = 0;; attempt++) {
        int rc;
        if (src) {
            imsame_seqinfo v;
            imsame_fasta_view(src, &v);
            rc = imsame_gpu_sample_create(w->ctx, &v, &w->dev[x]);
        } else {
            rc = imsame_gpu_sample_revcomp(w->ctx, w->dev[x - 1], &w->dev[x]);
        }
        if (!rc) {
            w->bytes[x] = bytes;
            w->held += bytes;
            w->uploads++;
            return 0;
        }
        w->dev[x] = NULL;
        if (rc != IMSAME_ENOMEM) {
            gpu_msg(msg, ml, what, rc, w->ctx);
            return -1;
        }
        if (attempt) return 1;
        make_room(w, keep, nkeep, ~0ull);
    }
}

/* the unit's query and database read sets on the worker's device: 0 (jo->q_sample / db_sample set), 1 (host
   buffers) or -1 (error, msg) */
static int place(worker *w, const unit *u, imsame_job_opts *jo, char *msg, size_t ml) {
    sample *si = &G.sm[u->i], *sj = &G.sm[u->j];
    const imsame_fasta *db = u->rev ? &sj->rev : &sj->fwd;
    if (db->total_len > (1ull << 29)) return 1; /* > one segment: before anything is uploaded */
    const int xq = 2 * u->i, xd = 2 * u->j + u->rev, xf = 2 * u->j;
    const int mirror = u->rev && sample_mirror(sj), via_fwd = mirror && !w->dev[xd];
    const int keep[3] = {xq, xd, xf}, nkeep = via_fwd ? 3 : 2;
    const uint64_t bq = set_bytes(&si->fwd) + table_bytes(&si->fwd), bd = set_bytes(db), bf = via_fwd ? set_bytes(&sj->fwd) : 0;
    if (bq + bd + bf > w->budget) return 1; /* not even alone */
    const uint64_t need = (w->dev[xq] ? 0 : bq) + (w->dev[xd] ? 0 : bd) + (via_fwd && !w->dev[xf] ? bf : 0);
    make_room(w, keep, nkeep, need);
    int rc = 0;
    if (!w->dev[xq]) rc = make_set(w, xq, &si->fwd, bq, keep, nkeep, "uploading a sample", msg, ml);
    if (!rc && !w->dev[xd]) {
        if (via_fwd) {
            if (!w->dev[xf]) rc = make_set(w, xf, &sj->fwd, bf, keep, nkeep, "uploading a sample", msg, ml);
            if (!rc) rc = make_set(w, xd, NULL, bd, keep, nkeep, "reverse complement of a sample", msg, ml);
        } else {
            rc = make_set(w, xd, db, bd, keep, nkeep, u->rev ? "reverse complement of a sample" : "uploading a sample", msg, ml);
        }
    }
    if (rc) return rc;
    w->last[xq] = ++w->tick;
    w->last[xd] = ++w->tick;
    jo->q_sample = w->dev[xq];
    jo->db_sample = w->dev[xd];
    return 0;
}

/* ---- one unit ---- */
static int unit_fail(unit *u, const char *msg) {
    u->text = strdup(msg);
    return 1;
}

static int run_unit(worker *w, unit *u) {
    sample *si = &G.sm[u->i], *sj = &G.sm[u->j];
    char msg[512];
    const char *e;
    if ((e = need_forward(si))) return unit_fail(u, e);
    if ((e = u->rev ? need_reverse(sj) : need_forward(sj))) return unit_fail(u, e);
    const imsame_fasta *q = &si->fwd, *db = u->rev ? &sj->rev : &sj->fwd;
    imsame_job_opts jo = G.jo;
    jo.device = w->device;
    jo.q_sample = NULL;
    jo.db_sample = NULL;
    int resident = 0;
    if (q->n_seqs > 0 && db->n_seqs > 0 && !G.no_resident) {
        if (!w->ctx) {
            gpu_msg(msg, sizeof msg, "no usable GPU", w->ctx_rc, NULL);
            return unit_fail(u, msg);
        }
        if (u->rev && (e = need_forward(sj))) return unit_fail(u, e);
        const int p = place(w, u, &jo, msg, sizeof msg);
        if (p < 0) return unit_fail(u, msg);
        resident = p == 0;
        if (!resident) w->fallbacks++;
    }
    char path[4096];
    unit_path(u, path, sizeof path);
    FILE *fout = fopen(path, "wt");
    const double t0 = now_s();
    uint64_t accepted = 0;
    char err[300];
    int rc = imsame_run_job(q, db, &jo, fout, &w->ctx, &accepted, err, sizeof err);
    for (int attempt = 0; rc == IMSAME_ENOMEM && resident && attempt < 2; attempt++) {
        /* nothing was written (the records are rendered only after the alignment and the traceback succeeded):
           retry once with every other read set evicted, then from host buffers with none left */
        const int keep[2] = {2 * u->i, 2 * u->j + u->rev};
        make_room(w, keep, attempt ? 0 : 2, ~0ull);
        if (attempt) {
            jo.q_sample = NULL;
            jo.db_sample = NULL;
            resident = 0;
            w->fallbacks++;
        }
        if (fout) fclose(fout);
        fout = fopen(path, "wt");
        rc = imsame_run_job(q, db, &jo, fout, &w->ctx, &accepted, err, sizeof err);
    }
    if (fout) fclose(fout);
    if (rc == IMSAME_EREADSIZE) return unit_fail(u, "Read size reached for gapped alignment.");
    if (rc) {
        snprintf(msg, sizeof msg, "GPU hot path failed: %s%s%s", imsame_gpu_strerror(rc), err[0] ? " / " : "", err);
        return unit_fail(u, msg);
    }
    if (resident && !w->tab[u->i]) {
        w->tab[u->i] = 1;
        w->tables++;
    }
    if (asprintf(&u->text,
                 "[INFO] %s vs %s%s: %" PRIu64 " reads (%" PRIu64 ") from the query were found in the database (%" PRIu64
                 "); Jaccard-index %Le; %.3f s\n",
                 si->name, sj->name, u->rev ? " (reverse complement)" : "", accepted, q->n_seqs, db->n_seqs,
                 (long double)accepted / ((db->n_seqs + q->n_seqs) - accepted), now_s() - t0) < 0)
        return unit_fail(u, "Could not allocate memory for the report");
    return 0;
}

/* ---- scheduling (G.lock held) ---- */
static long pick(const worker *w) {
    long best = -1;
    int best_score = -1;
    while (G.first < G.nu && G.u[G.first].state != U_PENDING) G.first++;
    for (size_t k = G.first; k < G.stop; k++) {
        const unit *u = &G.u[k];
        if (u->state != U_PENDING) continue;
        const int score = w->tab[u->i] ? 2 : w->dev[2 * u->j + u->rev] ? 1 : 0;
        if (score > best_score) {
            best = (long)k;
            best_score = score;
            if (score == 2) break;
        }
    }
    return best;
}

static void release_host(sample *s, int r) {
    if (s->uses[r]) return;
    if (r == 0 && s->have_fwd) { imsame_fasta_free(&s->fwd); s->have_fwd = 0; }
    if (r == 1 && s->have_rev) { imsame_fasta_free(&s->rev); s->have_rev = 0; }
}

static void finish(unit *u, int failed, size_t k) {
    if (failed) {
        u->state = U_FAILED;
        if (k < G.stop) G.stop = k;
    } else {
        u->state = U_DONE;
        G.done++;
        sample *si = &G.sm[u->i], *sj = &G.sm[u->j];
        si->uses[0]--;
        sj->uses[0]--;
        if (u->rev) sj->uses[1]--;
        release_host(si, 0);
        release_host(sj, 0);
        if (u->rev) release_host(sj, 1);
    }
    while (G.printed < G.nu && G.u[G.printed].state == U_DONE) {
        fputs(G.u[G.printed].text, stdout);
        free(G.u[G.printed].text);
        G.u[G.printed].text = NULL;
        G.printed++;
    }
    fflush(stdout);
}

static void *worker_main(void *arg) {
    worker *w = (worker *)arg;
    w->ctx_rc = imsame_gpu_create(&w->ctx, w->device); /* the contexts come up side by side */
    pthread_barrier_wait(&G.start);
    /* every context exists: the free memory is what the workers of a device share */
    uint64_t fr = 0, tot = 0;
    if (w->ctx && !imsame_gpu_mem_info(w->ctx, &fr, &tot)) {
        const int on_dev = G.n_workers / G.n_gpus + (w->id % G.n_gpus < G.n_workers % G.n_gpus);
        w->budget = fr / (uint64_t)on_dev / 2;
    }
    if (G.test_budget >= 0) w->budget = (uint64_t)G.test_budget;
    pthread_barrier_wait(&G.start);
#ifdef _OPENMP
    if (G.omp_threads > 0) omp_set_num_threads(G.omp_threads); /* record rendering: the host cores shared by the workers */
#endif
    imsame_sample **dead = (imsame_sample **)calloc(2 * G.n, sizeof(imsame_sample *));
    pthread_mutex_lock(&G.lock);
    for (;;) {
        const long k = pick(w);
        if (k < 0) break;
        unit *u = &G.u[k];
        u->state = U_RUNNING;
        /* read sets that no pending or running unit needs any more */
        int nd = 0;
        for (int x = 0; x < (int)(2 * G.n); x++)
            if (w->dev[x] && G.sm[x / 2].uses[x & 1] == 0) dead[nd++] = take(w, x); /* freed outside the lock */
        pthread_mutex_unlock(&G.lock);
        for (int d = 0; d < nd; d++) imsame_gpu_sample_free(w->ctx, dead[d]);
        const double t0 = now_s();
        const int failed = run_unit(w, u);
        w->busy += now_s() - t0;
        w->units++;
        pthread_mutex_lock(&G.lock);
        finish(u, failed, (size_t)k);
    }
    pthread_mutex_unlock(&G.lock);
    free(dead);
    return NULL;
}

/* -gpus / -jobs: an integer from 1 to 1024 */
static int count_arg(int argc, char **av, int i, const char *what) {
    char msg[128];
    snprintf(msg, sizeof msg, "%s must be an integer from 1 to 1024", what);
    if (i + 1 >= argc) terror(msg);
    char *end;
    errno = 0;
    const long v = strtol(av[i + 1], &end, 10);
    if (end == av[i + 1] || *end || errno || v < 1 || v > 1024) terror(msg);
    return (int)v;
}

int main(int argc, char **av) {
    if (argc < 7) {
        printf("***ERROR*** Use: %s metagenomes_directory coverage similarity threads file_extension outpath\n", av[0]);
        return 255;
    }
    setlocale(LC_ALL, "");
    const char *dir = av[1], *ext = av[5], *out = av[6];
    imsame_job_opts jo;
    memset(&jo, 0, sizeof jo);
    /* the script passes -coverage / -identity / -n_threads; everything else keeps IMSAME's defaults (src/IMSAME.c:44-49) */
    jo.mincoverage = (long double)atof(av[2]);
    jo.minidentity = (long double)atof(av[3]);
    jo.n_threads = (uint64_t)atoi(av[4]);
    jo.minevalue = 1 / powl(10, 20);
    jo.igap = -5;
    jo.egap = -2;
    jo.gpus = 1;
    jo.trace = getenv("IMSAME_TRACE") != NULL;
    int n_gpus = 1, n_jobs = 0;
    for (int i = 7; i < argc; i++) {
        if (strcmp(av[i], "-device") == 0 && i + 1 < argc) jo.device = atoi(av[i + 1]);
        if (strcmp(av[i], "-gpus") == 0) n_gpus = count_arg(argc, av, i, "-gpus");
        if (strcmp(av[i], "-jobs") == 0) n_jobs = count_arg(argc, av, i, "-jobs");
    }
    if (!n_jobs) n_jobs = n_gpus;
    if (jo.mincoverage <= 0) terror("Min-coverage must be larger than zero");
    if (jo.minidentity <= 0) terror("Min-identity must be larger than zero");

    /* `ls -d DIR/<name>.EXT`: names ending in ".EXT", in collation order */
    DIR *d = opendir(dir);
    if (!d) terror("Could not open the metagenomes directory");
    size_t n = 0, cap = 16, el = strlen(ext);
    sample *sm = (sample *)calloc(cap, sizeof(sample));
    if (!sm) terror("Could not allocate memory for the sample list");
    for (struct dirent *e; (e = readdir(d)) != NULL;) {
        const size_t l = strlen(e->d_name);
        if (e->d_name[0] == '.' || l < el + 2 || e->d_name[l - el - 1] != '.' || strcmp(e->d_name + l - el, ext) != 0) continue;
        if (n == cap) {
            cap *= 2;
            sm = (sample *)realloc(sm, cap * sizeof(sample));
            if (!sm) terror("Could not allocate memory for the sample list");
            memset(sm + n, 0, (cap - n) * sizeof(sample));
        }
        sm[n].name = strndup(e->d_name, l - el - 1);
        n++;
    }
    closedir(d);
    qsort(sm, n, sizeof(sample), by_name);
    for (size_t s = 0; s < n; s++) {
        pthread_mutex_init(&sm[s].lock, NULL);
        sm[s].mirror = -1;
    }

    G.sm = sm;
    G.n = n;
    G.dir = dir;
    G.ext = ext;
    G.out = out;
    G.jo = jo;
    G.no_resident = getenv("IMSAME_NO_RESIDENT") != NULL;
    const char *tb = getenv("IMSAME_TEST_SAMPLE_BUDGET"); /* test hook: small budgets make the eviction and fallback paths run */
    G.test_budget = tb ? atoll(tb) : -1;
    pthread_mutex_init(&G.lock, NULL);
    /* the units in canonical order (the script's loops); existing outputs are kept: bin/...sh:35,45 */
    G.u = (unit *)calloc(n > 1 ? n * (n - 1) : 1, sizeof(unit));
    if (!G.u) terror("Could not allocate memory for the sample list");
    for (size_t i = 0; i < n; i++)
        for (size_t j = i + 1; j < n; j++)
            for (int rev = 0; rev < 2; rev++) {
                unit *u = &G.u[G.nu];
                u->i = (int)i;
                u->j = (int)j;
                u->rev = rev;
                char path[4096];
                unit_path(u, path, sizeof path);
                if (exists(path)) continue;
                sm[i].uses[0]++;
                sm[j].uses[0]++; /* (a reverse unit: the forward parse decides the device path, the forward set feeds it) */
                if (rev) sm[j].uses[1]++;
                G.nu++;
            }
    G.stop = G.nu;

    const double t_all = now_s();
    G.n_gpus = n_gpus;
    G.n_workers = n_jobs < (int)G.nu ? n_jobs : (int)G.nu;
    worker *ws = (worker *)calloc(G.n_workers > 0 ? (size_t)G.n_workers : 1, sizeof(worker));
    pthread_t *th = (pthread_t *)calloc(G.n_workers > 0 ? (size_t)G.n_workers : 1, sizeof(pthread_t));
    if (!ws || !th) terror("Could not allocate memory for the workers");
#ifdef _OPENMP
    if (G.n_workers > 1) {
        G.omp_threads = omp_get_max_threads() / G.n_workers;
        if (G.omp_threads < 1) G.omp_threads = 1;
    }
#endif
    if (G.n_workers > 0) pthread_barrier_init(&G.start, NULL, (unsigned)G.n_workers);
    for (int w = 0; w < G.n_workers; w++) {
        ws[w].id = w;
        ws[w].device = jo.device + w % n_gpus;
        ws[w].dev = (imsame_sample **)calloc(2 * n, sizeof(imsame_sample *));
        ws[w].bytes = (uint64_t *)calloc(2 * n, sizeof(uint64_t));
        ws[w].last = (uint64_t *)calloc(2 * n, sizeof(uint64_t));
        ws[w].tab = (unsigned char *)calloc(n, 1);
        if (!ws[w].dev || !ws[w].bytes || !ws[w].last || !ws[w].tab) terror("Could not allocate memory for the workers");
    }
    for (int w = 0; w < G.n_workers; w++)
        if (pthread_create(&th[w], NULL, worker_main, &ws[w])) terror("Could not start a worker thread");
    for (int w = 0; w < G.n_workers; w++) pthread_join(th[w], NULL);
    if (jo.trace)
        for (int w = 0; w < G.n_workers; w++)
            fprintf(stderr,
                    "[imsame_allvsall] worker %d device %d: units %" PRIu64 ", uploads %" PRIu64 ", table builds %" PRIu64
                    ", evictions %" PRIu64 ", host-path fallbacks %" PRIu64 ", busy %.3f s\n",
                    w, ws[w].device, ws[w].units, ws[w].uploads, ws[w].tables, ws[w].evictions, ws[w].fallbacks, ws[w].busy);
    if (G.stop < G.nu) {
        fflush(stderr);
        terror(G.u[G.stop].text); /* the earliest failure: every unit before it is written and reported */
    }
    fprintf(stdout, "[INFO] %" PRIu64 " comparisons of %zu samples in %.3f s\n", G.done, n, now_s() - t_all);
    fflush(stdout);
    /* every output file is closed: as in IMSAME (imsame_main.c) the release of the device and host memory is left
       to the operating system unless IMSAME_FAST_EXIT=0 asks for the orderly one */
    const char *fast = getenv("IMSAME_FAST_EXIT");
    if (!(fast && fast[0] == '0')) {
        fflush(stderr);
        _exit(0);
    }
    for (int w = 0; w < G.n_workers; w++) {
        for (int x = 0; x < (int)(2 * n); x++)
            if (ws[w].dev[x]) imsame_gpu_sample_free(ws[w].ctx, ws[w].dev[x]);
        if (ws[w].ctx) imsame_gpu_destroy(ws[w].ctx);
        free(ws[w].dev);
        free(ws[w].bytes);
        free(ws[w].last);
        free(ws[w].tab);
    }
    free(ws);
    free(th);
    if (G.n_workers > 0) pthread_barrier_destroy(&G.start);
    for (size_t i = 0; i < n; i++) {
        if (sm[i].have_fwd) imsame_fasta_free(&sm[i].fwd);
        if (sm[i].have_rev) imsame_fasta_free(&sm[i].rev);
        pthread_mutex_destroy(&sm[i].lock);
        free(sm[i].name);
    }
    free(sm);
    free(G.u);
    return 0;
}
