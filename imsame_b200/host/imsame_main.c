/*
 * IMSAME -- drop-in command line for the reference binary (src/IMSAME.c:34-578):
 * same flags and defaults (init_args, :520-578), same `.align` record format
 * (src/alignmentFunctions.c:167-168), same [INFO] summary lines on stdout
 * (src/IMSAME.c:63,102,106,295,317,407,416,470-473), same error text / exit
 * status (terror, src/commonFunctions.c:10-13; --help exits 1).
 *
 * The host side stays in C: FASTA ingest, thresholds, reporting.  Index build,
 * scan, extension, NW, filter and first-hit selection (src/IMSAME.c:232-281 and
 * :409-467) run on the GPU through include/imsame_gpu.h; the alignment text of
 * the accepted reads comes from a device traceback rendered by host/render.c.
 * Records are written in ascending read order, which is the reference's own
 * order with -n_threads 1 and a legal interleaving of its threads otherwise.
 *
 * Opt-in additions that default to reference behaviour:
 *   -gpus N     shard the database by contiguous read ranges over N GPUs (default 1)
 *   -kmer K     seed length 4..16 (default 12 = the reference's FIXED_K; it has no such flag)
 *   -device D   first CUDA device to use (default 0)
 *   -out_rev F  also align the query against the reverse complement of the database and write those records to F:
 *               what `revComp db db.r; IMSAME ... -db db.r -out F` writes, in the same run.  The reverse read set is
 *               built by a host thread while the forward strand runs; where it is the mirror image of the database
 *               (imsame_revcomp_on_device) the database already on the GPU(s) is reverse complemented in place
 *               (imsame_gpu_align_revcomp), otherwise the reverse parse is uploaded.  stdout gains two lines after
 *               the Jaccard index, the numbers the second process would print; -out is what the run without the
 *               flag writes.  (Not in --help, whose text is the reference's.)
 */
#define _GNU_SOURCE
#include <inttypes.h>
#include <math.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <unistd.h>

#include "imsame_host.h"
#include "imsame_job.h"

static void terror(const char *s) { /* src/commonFunctions.c:10-13: message on STDOUT, exit(-1) */
    printf("ERR**** %s ****\n", s);
    exit(-1);
}

static double now_s(void) {
    struct timespec t;
    clock_gettime(CLOCK_MONOTONIC, &t);
    return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec;
}

#define SWEEP_ENTRIES (IMSAME_SWEEP_MAX - 1) /* set 0 is -coverage / -identity */

typedef struct {
    const char *query, *db, *out, *out_rev, *sweep;
    uint64_t n_threads;
    long double minevalue, mincoverage, minidentity;
    int igap, egap;
    int gpus, device, kmer;
    /* -sweep, parsed */
    int n_sweep;
    long double sweep_cov[SWEEP_ENTRIES], sweep_id[SWEEP_ENTRIES];
    char sweep_text[SWEEP_ENTRIES][2][64]; /* the values as given, for the summary lines */
} cli_args;

static void usage_and_exit(void) { /* src/IMSAME.c:526-538 */
    fprintf(stdout, "USAGE:\n");
    fprintf(stdout, "           IMSAME -query [query] -db [database]\n");
    fprintf(stdout, "OPTIONAL:\n");
    fprintf(stdout, "           -n_threads  [Integer:   0<n_threads] (default 4)\n");
    fprintf(stdout, "           -evalue     [Double:    0<=pval<1] (default: 1 * 10^-20)\n");
    fprintf(stdout, "           -coverage   [Double:    0<coverage<=1 (default: 0.5)\n");
    fprintf(stdout, "           -identity   [Double:    0<identity<=1 (default: 0.5)\n");
    fprintf(stdout, "           -igap       [Integer:   (default: 5)\n");
    fprintf(stdout, "           -egap       [Integer:   (default: 2)\n");
    fprintf(stdout, "           -out        [File path]\n");
    fprintf(stdout, "           --verbose   Turns verbose on\n");
    fprintf(stdout, "           --help      Shows help for program usage\n");
    exit(1);
}

/* one value of a -sweep entry: a whole number as atof reads it (strtod accepts exactly what atof converts) */
static int sweep_value(const char *b, const char *e, char *text, long double *v) {
    const size_t n = (size_t)(e - b);
    if (n == 0 || n >= 64) return 0;
    memcpy(text, b, n);
    text[n] = 0;
    char *end = NULL;
    (void)strtod(text, &end);
    if (end != text + n) return 0;
    *v = (long double)atof(text); /* double first, then widened, like -coverage / -identity */
    return 1;
}

static void parse_sweep(const char *list, cli_args *a) {
    const char *at = list;
    a->n_sweep = 0;
    for (;;) {
        const char *comma = strchr(at, ',');
        const char *end = comma ? comma : at + strlen(at);
        const char *colon = memchr(at, ':', (size_t)(end - at));
        if (a->n_sweep == SWEEP_ENTRIES) terror("-sweep takes at most 15 coverage:identity pairs");
        const int i = a->n_sweep;
        if (!colon || !sweep_value(at, colon, a->sweep_text[i][0], &a->sweep_cov[i]) ||
            !sweep_value(colon + 1, end, a->sweep_text[i][1], &a->sweep_id[i]))
            terror("-sweep expects a list of coverage:identity pairs, e.g. -sweep 0.5:0.7,0.5:0.9");
        if (a->sweep_cov[i] <= 0) terror("Min-coverage must be larger than zero");
        if (a->sweep_id[i] <= 0) terror("Min-identity must be larger than zero");
        a->n_sweep++;
        if (!comma) break;
        at = comma + 1;
    }
}

static void parse_args(int argc, char **av, cli_args *a) {
    /* defaults: src/IMSAME.c:44-49 */
    a->query = a->db = a->out = a->out_rev = a->sweep = NULL;
    a->n_sweep = 0;
    a->n_threads = 4;
    a->minevalue = 1 / powl(10, 20);
    a->mincoverage = 0.5;
    a->minidentity = 0.5;
    a->igap = -5;
    a->egap = -2;
    a->gpus = 1;
    a->device = 0;
    a->kmer = 12; /* FIXED_K, src/structs.h:15 */
    for (int i = 0; i < argc; i++) { /* the reference also scans av[0] and never skips values */
        const char *nxt = (i + 1 < argc) ? av[i + 1] : NULL;
        if (strcmp(av[i], "--help") == 0) usage_and_exit();
        if (strcmp(av[i], "-query") == 0 && nxt) a->query = nxt;
        if (strcmp(av[i], "-db") == 0 && nxt) a->db = nxt;
        if (strcmp(av[i], "-out") == 0 && nxt) a->out = nxt;
        if (strcmp(av[i], "-out_rev") == 0 && nxt) a->out_rev = nxt;
        if (strcmp(av[i], "-sweep") == 0 && nxt) a->sweep = nxt;
        if (strcmp(av[i], "-evalue") == 0 && nxt) {
            a->minevalue = (long double)atof(nxt); /* double first, then widened (:553) */
            if (a->minevalue < 0) terror("Min-e-value must be larger than zero");
        }
        if (strcmp(av[i], "-coverage") == 0 && nxt) {
            a->mincoverage = (long double)atof(nxt);
            if (a->mincoverage <= 0) terror("Min-coverage must be larger than zero");
        }
        if (strcmp(av[i], "-identity") == 0 && nxt) {
            a->minidentity = (long double)atof(nxt);
            if (a->minidentity <= 0) terror("Min-identity must be larger than zero");
        }
        if (strcmp(av[i], "-igap") == 0 && nxt) a->igap = -(atoi(nxt));
        if (strcmp(av[i], "-egap") == 0 && nxt) a->egap = -(atoi(nxt));
        if (strcmp(av[i], "-n_threads") == 0 && nxt) a->n_threads = (uint64_t)atoi(nxt);
        if (strcmp(av[i], "-gpus") == 0 && nxt) a->gpus = atoi(nxt);
        if (strcmp(av[i], "-device") == 0 && nxt) a->device = atoi(nxt);
        if (strcmp(av[i], "-kmer") == 0 && nxt) {
            a->kmer = atoi(nxt);
            if (a->kmer < 4 || a->kmer > 16) terror("The seed length must be between 4 and 16");
        }
    }
    if (a->sweep) {
        parse_sweep(a->sweep, a);
        if (a->gpus > 1) terror("-sweep runs on one GPU: it cannot be combined with -gpus above 1");
        if (a->out_rev) terror("-sweep cannot be combined with -out_rev");
    }
}

/* the CUDA context (0.8 s to create) comes up on its own thread while the FASTA files are parsed */
typedef struct {
    int device, rc;
    imsame_ctx *ctx;
} ctx_boot;
static void *ctx_boot_main(void *arg) {
    ctx_boot *b = (ctx_boot *)arg;
    b->rc = imsame_gpu_create(&b->ctx, b->device);
    return NULL;
}

/* -out_rev: revComp(db) as the loader sees it, built on its own thread while the forward strand is parsed and aligned */
typedef struct {
    const char *path;
    const imsame_fasta *fwd;
    imsame_fasta rev;
    int has_u, rc, started, joined;
    pthread_t thread;
} rev_load;
static void *rev_load_main(void *arg) {
    rev_load *r = (rev_load *)arg;
    r->rc = imsame_revcomp_load(r->path, &r->rev, &r->has_u);
    return NULL;
}
static const imsame_fasta *rev_wait(void *arg, int *on_device) {
    rev_load *r = (rev_load *)arg;
    if (!r->joined) {
        if (r->started) pthread_join(r->thread, NULL);
        else rev_load_main(r);
        r->joined = 1;
    }
    if (r->rc) return NULL;
    if (on_device) *on_device = imsame_revcomp_on_device(r->fwd, &r->rev, r->has_u);
    return &r->rev;
}

int main(int argc, char **av) {
    cli_args a;
    parse_args(argc, av, &a);
    FILE *fq = a.query ? fopen(a.query, "rt") : NULL;
    FILE *fd = a.db ? fopen(a.db, "rt") : NULL;
    FILE *fout = a.out ? fopen(a.out, "wt") : NULL; /* a failed -out open silently disables output (:549-550) */
    if (fq == NULL || fd == NULL) terror("A query and database is required");
    fclose(fq);
    fclose(fd);
    FILE *fout_rev = NULL;
    rev_load rl;
    memset(&rl, 0, sizeof rl);
    if (a.out_rev) {
        if ((fout_rev = fopen(a.out_rev, "wt")) == NULL) terror("Could not open the reverse-strand output file");
        rl.path = a.db;
        rl.started = pthread_create(&rl.thread, NULL, rev_load_main, &rl) == 0;
    }
    FILE *fout_sweep[SWEEP_ENTRIES];
    memset(fout_sweep, 0, sizeof fout_sweep);
    if (fout != NULL)
        for (int i = 0; i < a.n_sweep; i++) {
            char path[4096];
            snprintf(path, sizeof path, "%s.%d", a.out, i + 1);
            if ((fout_sweep[i] = fopen(path, "wt")) == NULL) terror("Could not open a -sweep output file");
        }

    double t0 = now_s();
    fprintf(stdout, "[INFO] Init. quick table\n");
    if (a.gpus < 1) a.gpus = 1;
    ctx_boot boot;
    pthread_t boot_thread;
    int booting = 0;
    memset(&boot, 0, sizeof boot);
    boot.device = a.device;
    if (a.gpus == 1 && a.n_threads > 0) booting = pthread_create(&boot_thread, NULL, ctx_boot_main, &boot) == 0;
    fprintf(stdout, "[INFO] Initialization took %e seconds \n", now_s() - t0);

    fprintf(stdout, "[INFO] Loading database\n");
    t0 = now_s();
    imsame_fasta db, q;
    if (imsame_fasta_load(a.db, 1, &db)) terror("Could not allocate memory for database vector");
    rl.fwd = &db;
    fprintf(stdout, "[INFO] Database loaded and of length %" PRIu64 ". Hash table building took %e seconds\n",
            db.total_len, now_s() - t0);
    t0 = now_s();
    fprintf(stdout, "[INFO] Loading query.\n");
    if (imsame_fasta_load(a.query, 0, &q)) terror("Could not allocate memory for query vector");
    fprintf(stdout, "[INFO] Query loaded and of length %" PRIu64 ". Took %e seconds\n", q.total_len, now_s() - t0);

    t0 = now_s();
    fprintf(stdout, "[INFO] Computing alignments.\n");
    /* src/IMSAME.c:414,430-452 + src/alignmentFunctions.c:88: every thread announces its range */
    if (a.n_threads > 0) {
        uint64_t per = (uint64_t)floorl((long double)q.n_seqs / (long double)a.n_threads);
        for (uint64_t t = 0; t < a.n_threads; t++)
            fprintf(stdout, "Going from %" PRIu64 " to %" PRIu64 "\n", t * per,
                    t == a.n_threads - 1 ? q.n_seqs : (t + 1) * per);
    }
    fflush(stdout);

    uint64_t accepted = 0;
    imsame_job_opts jo;
    memset(&jo, 0, sizeof jo);
    jo.n_threads = a.n_threads;
    jo.minevalue = a.minevalue;
    jo.mincoverage = a.mincoverage;
    jo.minidentity = a.minidentity;
    jo.igap = a.igap;
    jo.egap = a.egap;
    jo.gpus = a.gpus;
    jo.kmer = a.kmer;
    jo.device = a.device;
    jo.trace = getenv("IMSAME_TRACE") != NULL; /* phase wall times on stderr (not part of the reference's output) */
    imsame_rev_job rj;
    memset(&rj, 0, sizeof rj);
    if (a.out_rev) {
        rj.out = fout_rev;
        rj.wait = rev_wait;
        rj.arg = &rl;
        jo.rev = &rj;
    }
    imsame_sweep_job sj;
    uint64_t sweep_accepted[SWEEP_ENTRIES] = {0};
    int sweep_rc[SWEEP_ENTRIES] = {0};
    memset(&sj, 0, sizeof sj);
    if (a.n_sweep) {
        sj.n = a.n_sweep;
        sj.coverage = a.sweep_cov;
        sj.identity = a.sweep_id;
        sj.out = fout_sweep;
        sj.accepted = sweep_accepted;
        sj.rc = sweep_rc;
        jo.sweep = &sj;
    }
    char err[300];
    imsame_ctx *ctx = NULL;
    if (booting) {
        const double tw = now_s();
        pthread_join(boot_thread, NULL);
        if (jo.trace) fprintf(stderr, "[imsame] waited %.3f s for the CUDA context after parsing the FASTA files\n", now_s() - tw);
        ctx = boot.rc == IMSAME_OK ? boot.ctx : NULL; /* on failure run_job tries again and reports */
    }
    int rc = imsame_run_job(&q, &db, &jo, fout, ctx ? &ctx : NULL, &accepted, err, sizeof err);
    if (rc == IMSAME_EREADSIZE) terror("Read size reached for gapped alignment."); /* src/alignmentFunctions.c:155 */
    if (rc) {
        char msg[512];
        snprintf(msg, sizeof msg, "GPU hot path failed: %s%s%s", imsame_gpu_strerror(rc), err[0] ? " / " : "", err);
        terror(msg);
    }

    fprintf(stdout, "[INFO] Alignments computed in %e seconds.\n", now_s() - t0);
    fprintf(stdout,
            "[INFO] %" PRIu64 " reads (%" PRIu64 ") from the query were found in the database (%" PRIu64
            ") at a minimum e-value of %Le and minimum coverage of %d%%.\n",
            accepted, q.n_seqs, db.n_seqs, (long double)a.minevalue, (int)(100 * a.mincoverage));
    fprintf(stdout, "[INFO] The Jaccard-index is: %Le\n",
            (long double)accepted / ((db.n_seqs + q.n_seqs) - accepted));
    if (a.out_rev) {
        /* what the second process of the workflow (IMSAME -db revComp(db)) would report; revComp writes one record
           per '>' byte, so its read count is the reverse parse's own */
        const imsame_fasta *rdb = rev_wait(&rl, NULL);
        if (rl.rc == 1) terror("opening IN sequence FASTA file");
        if (rl.rc == 2) terror("memory for Seq");
        if (rl.rc == 3) terror("Could not allocate memory for database vector");
        if (rj.rc == IMSAME_EREADSIZE) terror("Read size reached for gapped alignment.");
        if (rj.rc) {
            char msg[512];
            snprintf(msg, sizeof msg, "GPU hot path failed: %s%s%s", imsame_gpu_strerror(rj.rc), err[0] ? " / " : "", err);
            terror(msg);
        }
        fprintf(stdout,
                "[INFO] %" PRIu64 " reads (%" PRIu64 ") from the query were found in the reverse complement of the database (%" PRIu64
                ") at a minimum e-value of %Le and minimum coverage of %d%%.\n",
                rj.accepted, q.n_seqs, rdb->n_seqs, (long double)a.minevalue, (int)(100 * a.mincoverage));
        fprintf(stdout, "[INFO] The Jaccard-index against the reverse complement is: %Le\n",
                (long double)rj.accepted / ((rdb->n_seqs + q.n_seqs) - rj.accepted));
    }
    int exit_status = 0;
    for (int i = 0; i < a.n_sweep; i++) {
        fprintf(stdout, "[INFO] Sweep %d of %d: -coverage %s -identity %s\n", i + 1, a.n_sweep, a.sweep_text[i][0],
                a.sweep_text[i][1]);
        if (sweep_rc[i]) { /* that run's terror line (src/commonFunctions.c:10-13); the process ends with its status */
            printf("ERR**** Read size reached for gapped alignment. ****\n");
            exit_status = 255;
            continue;
        }
        fprintf(stdout,
                "[INFO] %" PRIu64 " reads (%" PRIu64 ") from the query were found in the database (%" PRIu64
                ") at a minimum e-value of %Le and minimum coverage of %d%%.\n",
                sweep_accepted[i], q.n_seqs, db.n_seqs, (long double)a.minevalue, (int)(100 * a.sweep_cov[i]));
        fprintf(stdout, "[INFO] The Jaccard-index is: %Le\n",
                (long double)sweep_accepted[i] / ((db.n_seqs + q.n_seqs) - sweep_accepted[i]));
    }
    fprintf(stdout, "[INFO] Deallocating heap memory.\n");
    if (fout != NULL) fclose(fout);
    if (fout_rev != NULL) fclose(fout_rev);
    for (int i = 0; i < a.n_sweep; i++)
        if (fout_sweep[i] != NULL) fclose(fout_sweep[i]);
    fflush(stdout);
    /* Everything the caller can observe is on disk / on stdout now: the process ends here and leaves the device
       memory, the pinned buffers and the parsed reads to the operating system instead of releasing them piece by
       piece (the orderly release of a cfg2 run took 0.15 s in one run and 3.1 s in the next on the same box,
       profiles/r02_cli_e2e_cfg2_v4.log).  IMSAME_FAST_EXIT=0 releases everything in order (leak checkers). */
    const char *fast = getenv("IMSAME_FAST_EXIT");
    if (!(fast && fast[0] == '0')) {
        fflush(stderr);
        _exit(exit_status);
    }
    t0 = now_s();
    if (ctx) imsame_gpu_destroy(ctx);
    if (jo.trace) fprintf(stderr, "[imsame] context destroyed in %.3f s\n", now_s() - t0);
    t0 = now_s();
    imsame_fasta_free(&db);
    imsame_fasta_free(&q);
    if (a.out_rev) imsame_fasta_free(&rl.rev);
    if (jo.trace) fprintf(stderr, "[imsame] host read sets freed in %.3f s\n", now_s() - t0);
    return exit_status;
}
