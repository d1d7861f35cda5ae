/* imsame_job.c -- see imsame_job.h */
#define _GNU_SOURCE
#include "imsame_job.h"

#include <inttypes.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#ifdef _OPENMP
#include <omp.h>
#endif

static double now_s(void) {
    struct timespec t;
    clock_gettime(CLOCK_MONOTONIC, &t);
    return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec;
}

/* contexts of a multi-GPU job come up side by side (0.5 - 1 s each) */
typedef struct {
    int device, kmer, rc;
    imsame_ctx *ctx;
} ctx_job;

static void *ctx_main(void *arg) {
    ctx_job *j = (ctx_job *)arg;
    j->rc = imsame_gpu_create(&j->ctx, j->device);
    if (!j->rc) j->rc = imsame_gpu_set_kmer(j->ctx, j->kmer);
    return NULL;
}

/* one traceback on the GPU: the ops and cells of the accepted reads of a record array; with -cigar also their
   alignments (imsame_gpu_align_traceback) */
typedef struct {
    uint64_t *ops_off, *cigar_off;
    uint32_t *ops, *cell, *cigar;
    imsame_aln *aln;
} tb_layer;

static void tb_layer_free(tb_layer *L) {
    imsame_gpu_free(L->ops);
    imsame_gpu_free(L->cigar);
    free(L->ops_off);
    free(L->cell);
    free(L->cigar_off);
    free(L->aln);
    memset(L, 0, sizeof *L);
}

static int tb_layer_run(imsame_ctx **ctx, const imsame_job_opts *o, const imsame_fasta *q, const imsame_fasta *db,
                        const imsame_params *p, const imsame_best *best, tb_layer *L, char *err, size_t errlen, double *tp) {
    imsame_seqinfo qv, dv;
    imsame_fasta_view(q, &qv);
    imsame_fasta_view(db, &dv);
    memset(L, 0, sizeof *L);
    int rc = IMSAME_OK;
    if (!*ctx && (rc = imsame_gpu_create(ctx, o->device))) return rc;
    L->ops_off = (uint64_t *)malloc((q->n_seqs + 1) * sizeof(uint64_t));
    L->cell = (uint32_t *)malloc(4 * q->n_seqs * sizeof(uint32_t));
    rc = (L->ops_off && L->cell) ? imsame_gpu_traceback(*ctx, &dv, &qv, p, best, L->ops_off, &L->ops, L->cell) : IMSAME_ENOMEM;
    if (!rc && o->cigar) {
        L->cigar_off = (uint64_t *)malloc((q->n_seqs + 1) * sizeof(uint64_t));
        L->aln = (imsame_aln *)malloc(q->n_seqs * sizeof(imsame_aln));
        rc = (L->cigar_off && L->aln) ? imsame_gpu_align_traceback(*ctx, &dv, &qv, p, 1, best, L->aln, L->cigar_off, &L->cigar)
                                      : IMSAME_ENOMEM;
    }
    if (rc) {
        if (err && errlen) snprintf(err, errlen, "%s", imsame_gpu_last_cuda_error(*ctx));
        tb_layer_free(L);
    } else if (o->trace) {
        fprintf(stderr, "[imsame] traceback (GPU) %.3f s\n", now_s() - *tp);
        *tp = now_s();
    }
    return rc;
}

/* rendering of the records of the accepted reads of `best` (db: what best[].db_seq indexes); the path of read r is in
   layers[layer_of ? layer_of[r] : 0] */
static int render_records(const imsame_job_opts *o, const imsame_fasta *qf, const imsame_fasta *dbf, const imsame_best *best,
                          const tb_layer *layers, const uint8_t *layer_of, FILE *fout, double *tp) {
    const imsame_fasta q = *qf, db = *dbf;
    int rc = IMSAME_OK;
    {
        /* records are rendered by all host threads, each into its own buffer for a contiguous range of
           reads, and written in ascending read order (the reference's order with -n_threads 1) */
        int nt = 1;
#ifdef _OPENMP
        nt = omp_get_max_threads();
#endif
        if (nt > 64) nt = 64;
        if ((uint64_t)nt > q.n_seqs) nt = (int)q.n_seqs;
        char *bufs[64];
        size_t lens[64];
        int failed = 0;
        memset(bufs, 0, sizeof bufs);
        memset(lens, 0, sizeof lens);
#pragma omp parallel for schedule(static, 1) num_threads(nt)
        for (int t = 0; t < nt; t++) {
            const uint64_t r0 = q.n_seqs * (uint64_t)t / (uint64_t)nt, r1 = q.n_seqs * (uint64_t)(t + 1) / (uint64_t)nt;
            /* -cigar: at most xlen + ylen ops of at most 5 characters and six numbers */
            const size_t rec_max = (o->cigar ? 11 : 6) * (2 * (size_t)IMSAME_MAX_READ_SIZE) + 768;
            size_t cap = 1 << 20, len = 0;
            char *buf = (char *)malloc(cap);
            for (uint64_t r = r0; r < r1 && buf; r++) {
                if (!best[r].accepted) continue;
                if (cap - len < rec_max) {
                    cap = cap * 2 + rec_max;
                    char *nb2 = (char *)realloc(buf, cap);
                    if (!nb2) { free(buf); buf = NULL; break; }
                    buf = nb2;
                }
                const tb_layer *L = layers + (layer_of ? layer_of[r] : 0);
                const uint64_t s = best[r].db_seq;
                const uint32_t xlen = (uint32_t)(db.start_pos[s + 1] - db.start_pos[s]);
                const uint32_t ylen = (uint32_t)(q.start_pos[r + 1] - q.start_pos[r]);
                len += (size_t)imsame_format_header(buf + len, r, s, best[r].length, best[r].identities, ylen);
                if (o->cigar) len += imsame_format_cigar_columns(buf + len, &L->aln[r], L->cigar + L->cigar_off[r],
                                                                 L->cigar_off[r + 1] - L->cigar_off[r]);
                len += (size_t)imsame_render_alignment(buf + len, db.sequences + db.start_pos[s], xlen,
                                                       q.sequences + q.start_pos[r], ylen, L->cell[4 * r], L->cell[4 * r + 1],
                                                       L->ops + L->ops_off[r], L->ops_off[r + 1] - L->ops_off[r]);
            }
            if (!buf) {
#pragma omp atomic write
                failed = 1;
            }
            bufs[t] = buf;
            lens[t] = len;
        }
        for (int t = 0; t < nt; t++) {
            if (!failed && bufs[t]) fwrite(bufs[t], 1, lens[t], fout);
            free(bufs[t]);
        }
        if (failed) rc = IMSAME_ENOMEM;
        if (o->trace) { fprintf(stderr, "[imsame] render + write %.3f s\n", now_s() - *tp); *tp = now_s(); }
    }
    return rc;
}

/* traceback on the GPU + rendering of the records of the accepted reads of `best` */
static int write_records(imsame_ctx **ctx, const imsame_job_opts *o, const imsame_fasta *q, const imsame_fasta *db,
                         const imsame_params *p, const imsame_best *best, FILE *fout, char *err, size_t errlen, double *tp) {
    tb_layer L;
    int rc = tb_layer_run(ctx, o, q, db, p, best, &L, err, errlen, tp);
    if (rc) return rc;
    rc = render_records(o, q, db, best, &L, NULL, fout, tp);
    tb_layer_free(&L);
    return rc;
}

/* the records of n_sets record arrays (best + t * nq) into fouts[t] (NULL: none).  Most sets share most winners: each
   distinct (read, db_seq) winner is traced once.  Layer L holds the L-th distinct winner of every read (in set order),
   so that at most n_sets tracebacks together trace every distinct pair exactly once. */
static int write_sweep_records(imsame_ctx **ctx, const imsame_job_opts *o, const imsame_fasta *q, const imsame_fasta *db,
                               const imsame_params *p, const imsame_best *best, int n_sets, FILE *const *fouts, char *err,
                               size_t errlen, double *tp) {
    const uint64_t nq = q->n_seqs;
    uint8_t *layer_of = (uint8_t *)calloc((size_t)n_sets * nq, 1);
    imsame_best *lb = (imsame_best *)malloc(nq * sizeof(imsame_best));
    if (!layer_of || !lb) { free(layer_of); free(lb); return IMSAME_ENOMEM; }
    int n_layers = 0;
    for (uint64_t r = 0; r < nq; r++) {
        uint64_t seen[IMSAME_SWEEP_MAX];
        int k = 0;
        for (int t = 0; t < n_sets; t++) {
            const imsame_best *b = best + (uint64_t)t * nq + r;
            if (!fouts[t] || !b->accepted) continue;
            int j = 0;
            while (j < k && seen[j] != b->db_seq) j++;
            if (j == k) seen[k++] = b->db_seq;
            layer_of[(uint64_t)t * nq + r] = (uint8_t)j;
        }
        if (k > n_layers) n_layers = k;
    }
    tb_layer layers[IMSAME_SWEEP_MAX];
    memset(layers, 0, sizeof layers);
    int rc = IMSAME_OK;
    for (int L = 0; L < n_layers && !rc; L++) {
        memset(lb, 0, nq * sizeof(imsame_best));
        for (uint64_t r = 0; r < nq; r++)
            for (int t = 0; t < n_sets && !lb[r].accepted; t++) {
                const imsame_best *b = best + (uint64_t)t * nq + r;
                if (fouts[t] && b->accepted && layer_of[(uint64_t)t * nq + r] == L) lb[r] = *b;
            }
        rc = tb_layer_run(ctx, o, q, db, p, lb, &layers[L], err, errlen, tp);
    }
    for (int t = 0; t < n_sets && !rc; t++)
        if (fouts[t]) rc = render_records(o, q, db, best + (uint64_t)t * nq, layers, layer_of + (uint64_t)t * nq, fouts[t], tp);
    for (int L = 0; L < n_layers; L++) tb_layer_free(&layers[L]);
    free(layer_of);
    free(lb);
    return rc;
}

/* o->sweep: the job's thresholds as set 0 of the sweep, the sweep's entries as sets 1 .. n; with o->q_sample / db_sample
   imsame_gpu_align_samples_sweep, else imsame_gpu_align_sweep from the host buffers */
static int sweep_job(const imsame_fasta *q, const imsame_fasta *db, const imsame_job_opts *o, const imsame_params *p,
                     int kmer, FILE *fout, imsame_ctx **ctx_cache, uint64_t *accepted_out, char *err, size_t errlen) {
    imsame_sweep_job *sw = o->sweep;
    const int n_sets = 1 + sw->n;
    if (n_sets > IMSAME_SWEEP_MAX || o->gpus > 1 || o->rev) return IMSAME_EARG;
    double tp = now_s();
    imsame_seqinfo qv, dv;
    imsame_fasta_view(q, &qv);
    imsame_fasta_view(db, &dv);
    imsame_params ps[IMSAME_SWEEP_MAX];
    for (int t = 0; t < n_sets; t++) {
        ps[t] = *p;
        if (t) { ps[t].min_coverage = sw->coverage[t - 1]; ps[t].min_identity = sw->identity[t - 1]; }
    }
    const uint64_t nq = q->n_seqs;
    imsame_best *best = (imsame_best *)calloc((size_t)n_sets * nq, sizeof(imsame_best));
    if (!best) return IMSAME_ENOMEM;
    int set_rc[IMSAME_SWEEP_MAX];
    imsame_ctx *ctx = (ctx_cache && *ctx_cache) ? *ctx_cache : NULL;
    int rc = IMSAME_OK;
    if (!ctx && (rc = imsame_gpu_create(&ctx, o->device))) { free(best); return rc; }
    if (ctx_cache) *ctx_cache = ctx;
    rc = imsame_gpu_set_kmer(ctx, kmer);
    if (!rc) {
        if (o->q_sample && o->db_sample) rc = imsame_gpu_align_samples_sweep(ctx, o->db_sample, o->q_sample, ps, n_sets, best, set_rc, NULL);
        else rc = imsame_gpu_align_sweep(ctx, &dv, &qv, ps, n_sets, best, set_rc, NULL);
    }
    if (rc && err && errlen) snprintf(err, errlen, "%s", imsame_gpu_last_cuda_error(ctx));
    if (!rc) rc = set_rc[0];  /* the main set's read-size stop ends the job as without the sweep */
    if (!rc) {
        if (o->trace) { fprintf(stderr, "[imsame] align (%d threshold sets) %.3f s\n", n_sets, now_s() - tp); tp = now_s(); }
        FILE *fouts[IMSAME_SWEEP_MAX];
        for (int t = 0; t < n_sets; t++) {
            uint64_t acc = 0;
            for (uint64_t r = 0; r < nq; r++) acc += best[(uint64_t)t * nq + r].accepted;
            if (t) { sw->accepted[t - 1] = acc; sw->rc[t - 1] = set_rc[t]; }
            else *accepted_out = acc;
            fouts[t] = t ? (sw->out ? sw->out[t - 1] : NULL) : fout;
            if (set_rc[t] || acc == 0) fouts[t] = NULL;
        }
        rc = write_sweep_records(&ctx, o, q, db, p, best, n_sets, fouts, err, errlen, &tp);
    }
    if (ctx && !(ctx_cache && *ctx_cache == ctx)) imsame_gpu_destroy(ctx);
    free(best);
    return rc;
}

/* o->kmers: the job's seed length as entry 0, the list's as entries 1 .. n (imsame_gpu_align_kmers); the records of
   every entry are traced together, a winner that several entries share once (write_sweep_records) */
_Static_assert(IMSAME_KMERS_MAX <= IMSAME_SWEEP_MAX, "write_sweep_records takes every entry");
static int kmers_job(const imsame_fasta *q, const imsame_fasta *db, const imsame_job_opts *o, const imsame_params *p,
                     int kmer, FILE *fout, imsame_ctx **ctx_cache, uint64_t *accepted_out, char *err, size_t errlen) {
    imsame_kmers_job *kj = o->kmers;
    const int n_k = 1 + kj->n;
    if (n_k > IMSAME_KMERS_MAX || o->gpus > 1 || o->rev || o->sweep || o->q_sample) return IMSAME_EARG;
    double tp = now_s();
    imsame_seqinfo qv, dv;
    imsame_fasta_view(q, &qv);
    imsame_fasta_view(db, &dv);
    int ks[IMSAME_KMERS_MAX];
    ks[0] = kmer;
    for (int t = 1; t < n_k; t++) ks[t] = kj->k[t - 1];
    const uint64_t nq = q->n_seqs;
    imsame_best *best = (imsame_best *)calloc((size_t)n_k * nq, sizeof(imsame_best));
    if (!best) return IMSAME_ENOMEM;
    int k_rc[IMSAME_KMERS_MAX];
    imsame_ctx *ctx = (ctx_cache && *ctx_cache) ? *ctx_cache : NULL;
    int rc = IMSAME_OK;
    if (!ctx && (rc = imsame_gpu_create(&ctx, o->device))) { free(best); return rc; }
    if (ctx_cache) *ctx_cache = ctx;
    rc = imsame_gpu_align_kmers(ctx, &dv, &qv, p, n_k, ks, best, k_rc, NULL);
    if (rc && err && errlen) snprintf(err, errlen, "%s", imsame_gpu_last_cuda_error(ctx));
    if (!rc) rc = k_rc[0]; /* the main entry's read-size stop ends the job as without the list */
    if (!rc) {
        if (o->trace) { fprintf(stderr, "[imsame] align (%d seed lengths) %.3f s\n", n_k, now_s() - tp); tp = now_s(); }
        FILE *fouts[IMSAME_KMERS_MAX];
        for (int t = 0; t < n_k; t++) {
            uint64_t acc = 0;
            for (uint64_t r = 0; r < nq; r++) acc += best[(uint64_t)t * nq + r].accepted;
            if (t) { kj->accepted[t - 1] = acc; kj->rc[t - 1] = k_rc[t]; }
            else *accepted_out = acc;
            fouts[t] = t ? (kj->out ? kj->out[t - 1] : NULL) : fout;
            if (k_rc[t] || acc == 0) fouts[t] = NULL;
        }
        rc = write_sweep_records(&ctx, o, q, db, p, best, n_k, fouts, err, errlen, &tp);
    }
    if (ctx && !(ctx_cache && *ctx_cache == ctx)) imsame_gpu_destroy(ctx);
    free(best);
    return rc;
}

/* the reverse strand (o->rev) on the contexts of the forward one: ctxs[0 .. ng) (ctxs == &ctx when ng == 1) */
static int reverse_strand(imsame_ctx **ctxs, int ng, const imsame_job_opts *o, const imsame_fasta *q, imsame_params *p,
                          char *err, size_t errlen, double *tp) {
    imsame_rev_job *rv = o->rev;
    int on_device = 0;
    const imsame_fasta *rdb = rv->wait(rv->arg, &on_device);
    if (!rdb) return IMSAME_EARG;
    if (o->trace) { fprintf(stderr, "[imsame] reverse strand ready (%s) %.3f s\n", on_device ? "device" : "upload", now_s() - *tp); *tp = now_s(); }
    if (rdb->n_seqs == 0) return IMSAME_OK;
    imsame_best *best = (imsame_best *)calloc(q->n_seqs, sizeof(imsame_best));
    if (!best) return IMSAME_ENOMEM;
    imsame_seqinfo qv, rv_view;
    imsame_fasta_view(q, &qv);
    imsame_fasta_view(rdb, &rv_view);
    int rc;
    if (on_device) {  /* the forward database is still resident: mirrored there (rdb has its shape) */
        rc = imsame_gpu_align_revcomp(ctxs, ng, best, NULL);
    } else {          /* revComp's text parses into something else: upload that parse, as a second process would */
        int nr = ng;
        if ((uint64_t)nr > rdb->n_seqs) nr = (int)rdb->n_seqs;
        rc = nr == 1 ? imsame_gpu_align(ctxs[0], &rv_view, &qv, p, best, NULL)
                     : imsame_gpu_align_sharded(ctxs, nr, &rv_view, &qv, p, best, NULL);
    }
    if (rc && err && errlen) snprintf(err, errlen, "%s", imsame_gpu_last_cuda_error(ctxs[0]));
    if (o->trace) { fprintf(stderr, "[imsame] align reverse strand %.3f s\n", now_s() - *tp); *tp = now_s(); }
    uint64_t accepted = 0;
    if (!rc) {
        for (uint64_t r = 0; r < q->n_seqs; r++) accepted += best[r].accepted;
        if (rv->out != NULL && accepted > 0) rc = write_records(&ctxs[0], o, q, rdb, p, best, rv->out, err, errlen, tp);
    }
    rv->accepted = accepted;
    free(best);
    return rc;
}

int imsame_run_job(const imsame_fasta *qf, const imsame_fasta *dbf, const imsame_job_opts *o, FILE *fout,
                   imsame_ctx **ctx_cache, uint64_t *accepted_out, char *err, size_t errlen) {
    const imsame_fasta q = *qf, db = *dbf;
    double tp = now_s();
    uint64_t accepted = 0;
    if (err && errlen) err[0] = 0;
    *accepted_out = 0;
    if (!(o->n_threads > 0 && q.n_seqs > 0 && db.n_seqs > 0)) return IMSAME_OK;
    imsame_best *best = (imsame_best *)calloc(q.n_seqs ? q.n_seqs : 1, sizeof(imsame_best));
    if (!best) return IMSAME_ENOMEM;
    imsame_seqinfo qv, dv;
    imsame_fasta_view(&q, &qv);
    imsame_fasta_view(&db, &dv);
    imsame_params p;
    memset(&p, 0, sizeof p);
    p.min_e_value = o->minevalue;
    p.min_coverage = o->mincoverage;
    p.min_identity = o->minidentity;
    p.igap = o->igap;
    p.egap = o->egap;
    p.n_threads = o->n_threads;
    const int kmer = o->kmer ? o->kmer : 12; /* FIXED_K, src/structs.h:15 */
    if (o->sweep) {
        free(best);
        return sweep_job(&q, &db, o, &p, kmer, fout, ctx_cache, accepted_out, err, errlen);
    }
    if (o->kmers) {
        free(best);
        return kmers_job(&q, &db, o, &p, kmer, fout, ctx_cache, accepted_out, err, errlen);
    }

    int ng = o->gpus < 1 ? 1 : o->gpus;
    if ((uint64_t)ng > db.n_seqs) ng = (int)db.n_seqs;
    imsame_ctx *ctx = NULL; /* device `o->device`: alignment (shard 0) and traceback; kept if the caller caches */
    imsame_ctx **ctxs = NULL; /* ng > 1: the shards' contexts, kept until the reverse strand is done (o->rev) */
    int rc = IMSAME_OK;
    if (ctx_cache && *ctx_cache) ctx = *ctx_cache;
    if (ng == 1) {
        if (!ctx && (rc = imsame_gpu_create(&ctx, o->device))) { free(best); return rc; }
        if (ctx_cache) *ctx_cache = ctx;
        rc = imsame_gpu_set_kmer(ctx, kmer);
        if (!rc) {
            if (o->q_sample && o->db_sample) rc = imsame_gpu_align_samples(ctx, o->db_sample, o->q_sample, &p, best, NULL);
            else rc = imsame_gpu_align(ctx, &dv, &qv, &p, best, NULL);
        }
        if (rc && err && errlen) snprintf(err, errlen, "%s", imsame_gpu_last_cuda_error(ctx));
    } else {
        /* the database sharded by contiguous read ranges over ng GPUs; the per-read first accepted hit is
           reduced with NCCL inside the library (imsame_gpu_align_sharded), replacing src/IMSAME.c:430-467 */
        ctx_job *jobs = (ctx_job *)calloc((size_t)ng, sizeof(ctx_job));
        pthread_t *th = (pthread_t *)calloc((size_t)ng, sizeof(pthread_t));
        ctxs = (imsame_ctx **)calloc((size_t)ng, sizeof(imsame_ctx *));
        if (!jobs || !th || !ctxs) {
            free(jobs); free(th); free(ctxs); free(best);
            return IMSAME_ENOMEM;
        }
        for (int g = 0; g < ng; g++) {
            jobs[g].device = o->device + g;
            jobs[g].kmer = kmer;
            if (g == 0 && ctx) { jobs[g].ctx = ctx; jobs[g].rc = imsame_gpu_set_kmer(ctx, kmer); continue; }
            if (pthread_create(&th[g], NULL, ctx_main, &jobs[g])) { ctx_main(&jobs[g]); th[g] = 0; }
        }
        for (int g = 0; g < ng; g++) {
            if (th[g]) pthread_join(th[g], NULL);
            ctxs[g] = jobs[g].ctx;
            if (jobs[g].rc && !rc) {
                rc = jobs[g].rc;
                if (err && errlen) snprintf(err, errlen, "device %d: %s", jobs[g].device, imsame_gpu_strerror(rc));
            }
        }
        if (o->trace) { fprintf(stderr, "[imsame] %d contexts %.3f s\n", ng, now_s() - tp); tp = now_s(); }
        if (!rc) {
            rc = imsame_gpu_align_sharded(ctxs, ng, &dv, &qv, &p, best, NULL);
            if (rc && err && errlen) snprintf(err, errlen, "%s", imsame_gpu_last_cuda_error(ctxs[0]));
        }
        if (!o->rev || rc)
            for (int g = 1; g < ng; g++) imsame_gpu_destroy(ctxs[g]);
        ctx = ctxs[0];
        if (ctx_cache && ctx) *ctx_cache = ctx;
        free(jobs);
        free(th);
        if (!o->rev || rc) { free(ctxs); ctxs = NULL; }
    }
    if (rc) { free(best); if (ctx && !(ctx_cache && *ctx_cache == ctx)) imsame_gpu_destroy(ctx); return rc; }
    for (uint64_t r = 0; r < q.n_seqs; r++) accepted += best[r].accepted;
    if (o->trace) { fprintf(stderr, "[imsame] align (all shards) %.3f s\n", now_s() - tp); tp = now_s(); }

    if (fout != NULL && accepted > 0) rc = write_records(&ctx, o, &q, &db, &p, best, fout, err, errlen, &tp);
    if (!rc && o->rev) {
        /* the forward records are complete: a read-size stop of the reverse strand leaves them as the first process
           of the two-process workflow would */
        if (ctxs) ctxs[0] = ctx;
        o->rev->rc = reverse_strand(ctxs ? ctxs : &ctx, ng, o, &q, &p, err, errlen, &tp);
        if (ctxs) ctx = ctxs[0];
    }
    if (ctxs) {
        for (int g = 1; g < ng; g++) imsame_gpu_destroy(ctxs[g]);
        free(ctxs);
    }
    if (ctx && !(ctx_cache && *ctx_cache == ctx)) imsame_gpu_destroy(ctx);
    free(best);
    *accepted_out = accepted;
    return rc;
}
