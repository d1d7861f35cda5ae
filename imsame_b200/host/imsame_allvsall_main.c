/*
 * IMSAME_allvsall -- the reference's all-vs-all workflow (bin/all_vs_all_metagenomes_IMSAME.sh:27-58)
 * in ONE process: same arguments, same output files (OUT/X-Y.align and OUT/X-Y.r.align, byte for byte
 * what the script produces with the drop-in IMSAME and revComp), same resume rule (existing outputs
 * are kept) -- but every sample is parsed once, its reverse complement (src/reverseComplement.c, incl.
 * the reversed record order that renumbers db_seq) is built in memory instead of a temporary Y.r.EXT
 * file, and all 2 * n(n-1)/2 comparisons share one CUDA context.  Every sample is also uploaded and packed
 * ONCE (imsame_gpu_sample_create): it stays on the device as the database of later comparisons, keeps the word
 * table built for it as a query, and its reverse complement is made on the device from the packed form
 * (imsame_gpu_sample_revcomp).  The script starts 56 IMSAME and 28 revComp processes for 8 samples and
 * re-parses every file 14 times.
 *
 * usage: IMSAME_allvsall metagenomes_directory coverage similarity threads file_extension outpath [-device D]
 */
#define _GNU_SOURCE
#include <dirent.h>
#include <inttypes.h>
#include <locale.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <time.h>
#include <unistd.h>

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
    imsame_fasta fwd, rev; /* parsed forward sample / parsed revComp(sample): what the records are rendered from */
    int have_fwd, have_rev;
    imsame_sample *dfwd, *drev; /* the same two read sets resident on the device */
    int has_u;                  /* the file contains a 'U' (imsame_revcomp_load, imsame_revcomp_on_device) */
} sample;

static int by_name(const void *a, const void *b) { return strcoll(((const sample *)a)->name, ((const sample *)b)->name); }

static int exists(const char *path) {
    struct stat st;
    return stat(path, &st) == 0 && S_ISREG(st.st_mode);
}

static void need_forward(sample *s, const char *dir, const char *ext) {
    if (s->have_fwd) return;
    char path[4096];
    snprintf(path, sizeof path, "%s/%s.%s", dir, s->name, ext);
    if (imsame_fasta_load(path, 1, &s->fwd)) terror("Could not allocate memory for database vector");
    s->have_fwd = 1;
}

static void need_reverse(sample *s, const char *dir, const char *ext) {
    if (s->have_rev) return;
    char path[4096];
    snprintf(path, sizeof path, "%s/%s.%s", dir, s->name, ext);
    switch (imsame_revcomp_load(path, &s->rev, &s->has_u)) {
        case 1: terror("opening IN sequence FASTA file");
        case 2: terror("memory for Seq");
        case 3: terror("Could not allocate memory for database vector");
    }
    s->have_rev = 1;
}

static void gpu_fail(const char *what, int rc, imsame_ctx *ctx) {
    char msg[512];
    snprintf(msg, sizeof msg, "%s: %s / %s", what, imsame_gpu_strerror(rc), ctx ? imsame_gpu_last_cuda_error(ctx) : "");
    terror(msg);
}

/* the device copies (lazily, once per sample) */
static void need_forward_dev(sample *s, imsame_ctx *ctx) {
    if (s->dfwd) return;
    imsame_seqinfo v;
    imsame_fasta_view(&s->fwd, &v);
    const int rc = imsame_gpu_sample_create(ctx, &v, &s->dfwd);
    if (rc) gpu_fail("uploading a sample", rc, ctx);
}

static void need_reverse_dev(sample *s, imsame_ctx *ctx) {
    if (s->drev) return;
    int rc;
    /* The device reverse complement works on the packed forward reads; revComp works on the text, and its filter is
       not the loader's (imsame_revcomp_is_mirror, host/fasta.c: '\r' / '-' / digits inside a record, 'U', header lines
       with several '>').  Both parses are in memory for the renderer anyway: the device path is taken only when
       the parse of revComp's text IS the mirror image of the sample, otherwise that parse is uploaded. */
    if (!(s->have_fwd && s->have_rev && imsame_revcomp_on_device(&s->fwd, &s->rev, s->has_u))) {
        imsame_seqinfo v;
        imsame_fasta_view(&s->rev, &v);
        rc = imsame_gpu_sample_create(ctx, &v, &s->drev);
    } else {
        need_forward_dev(s, ctx);
        rc = imsame_gpu_sample_revcomp(ctx, s->dfwd, &s->drev);
    }
    if (rc) gpu_fail("reverse complement of a sample", rc, ctx);
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
    for (int i = 7; i + 1 < argc; i++)
        if (strcmp(av[i], "-device") == 0) jo.device = atoi(av[i + 1]);
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

    imsame_ctx *ctx = NULL;
    const double t_all = now_s();
    uint64_t jobs = 0;
    for (size_t i = 0; i < n; i++)
        for (size_t j = i + 1; j < n; j++)
            for (int rev = 0; rev < 2; rev++) {
                char path[4096];
                snprintf(path, sizeof path, "%s/%s-%s%s.align", out, sm[i].name, sm[j].name, rev ? ".r" : "");
                if (exists(path)) continue; /* resume: bin/...sh:35,45 */
                need_forward(&sm[i], dir, ext);
                if (rev) need_reverse(&sm[j], dir, ext); else need_forward(&sm[j], dir, ext);
                const imsame_fasta *q = &sm[i].fwd, *db = rev ? &sm[j].rev : &sm[j].fwd;
                if (q->n_seqs > 0 && db->n_seqs > 0 && !getenv("IMSAME_NO_RESIDENT")) {
                    if (!ctx) {
                        const int crc = imsame_gpu_create(&ctx, jo.device);
                        if (crc) gpu_fail("no usable GPU", crc, NULL);
                    }
                    if (rev && !sm[j].have_fwd) need_forward(&sm[j], dir, ext);
                    need_forward_dev(&sm[i], ctx);
                    if (rev) need_reverse_dev(&sm[j], ctx); else need_forward_dev(&sm[j], ctx);
                    jo.q_sample = sm[i].dfwd;
                    jo.db_sample = rev ? sm[j].drev : sm[j].dfwd;
                    if ((rev ? db->total_len : db->total_len) > (1ull << 29)) jo.q_sample = NULL, jo.db_sample = NULL; /* > one segment */
                } else {
                    jo.q_sample = NULL;
                    jo.db_sample = NULL;
                }
                FILE *fout = fopen(path, "wt");
                const double t0 = now_s();
                uint64_t accepted = 0;
                char err[300];
                const int rc = imsame_run_job(q, db, &jo, fout, &ctx, &accepted, err, sizeof err);
                if (fout) fclose(fout);
                if (rc == IMSAME_EREADSIZE) terror("Read size reached for gapped alignment.");
                if (rc) {
                    char msg[512];
                    snprintf(msg, sizeof msg, "GPU hot path failed: %s%s%s", imsame_gpu_strerror(rc), err[0] ? " / " : "", err);
                    terror(msg);
                }
                jobs++;
                fprintf(stdout,
                        "[INFO] %s vs %s%s: %" PRIu64 " reads (%" PRIu64 ") from the query were found in the database (%" PRIu64
                        "); Jaccard-index %Le; %.3f s\n",
                        sm[i].name, sm[j].name, rev ? " (reverse complement)" : "", accepted, q->n_seqs, db->n_seqs,
                        (long double)accepted / ((db->n_seqs + q->n_seqs) - accepted), now_s() - t0);
                fflush(stdout);
            }
    fprintf(stdout, "[INFO] %" PRIu64 " comparisons of %zu samples in %.3f s\n", jobs, n, now_s() - t_all);
    fflush(stdout);
    /* every output file is closed: as in IMSAME (imsame_main.c) the release of the device and host memory is left
       to the operating system unless IMSAME_FAST_EXIT=0 asks for the orderly one */
    const char *fast = getenv("IMSAME_FAST_EXIT");
    if (!(fast && fast[0] == '0')) {
        fflush(stderr);
        _exit(0);
    }
    for (size_t i = 0; i < n; i++) {
        imsame_gpu_sample_free(ctx, sm[i].dfwd);
        imsame_gpu_sample_free(ctx, sm[i].drev);
    }
    if (ctx) imsame_gpu_destroy(ctx);
    for (size_t i = 0; i < n; i++) {
        if (sm[i].have_fwd) imsame_fasta_free(&sm[i].fwd);
        if (sm[i].have_rev) imsame_fasta_free(&sm[i].rev);
        free(sm[i].name);
    }
    free(sm);
    return 0;
}
