/*
 * imsame_job.h -- one IMSAME comparison (query sample vs database sample) on the GPU(s), shared by
 * the drop-in command line (imsame_main.c: one job per process, like the reference) and by the
 * in-process all-vs-all driver (imsame_allvsall_main.c: many jobs, one CUDA context).
 * Covers src/IMSAME.c:409-467 (fan-out, join, accepted count) and the record output of
 * src/alignmentFunctions.c:163-173.
 */
#ifndef IMSAME_JOB_H
#define IMSAME_JOB_H
#include "imsame_host.h"

/* The reverse strand in the same job (IMSAME -out_rev): the records of `IMSAME -db revComp(db)` against the
 * database still resident on the job's GPU(s) where the mirror rule holds (imsame_revcomp_on_device), else against
 * an upload of the reverse parse. */
typedef struct imsame_rev_job {
    FILE *out; /* its records */
    /* called once the forward records are written: the parse of revComp(db) (imsame_revcomp_load) with
       *on_device = imsame_revcomp_on_device(db, rev, has_u), or NULL when it could not be built */
    const imsame_fasta *(*wait)(void *arg, int *on_device);
    void *arg;
    uint64_t accepted; /* out: reads with a record against the reverse complement */
    int rc;            /* out: the reverse strand's result (the job returns the forward strand's) */
} imsame_rev_job;

/* More coverage/identity sets in the same run (IMSAME -sweep): sets 1 .. n of imsame_gpu_align_sweep, the job's own
 * thresholds being set 0, whose records and count the job reports as without a sweep.  One GPU, no samples, no rev. */
typedef struct imsame_sweep_job {
    int n;
    const long double *coverage, *identity; /* n each */
    FILE **out;                             /* n files for the records (NULL, or NULL entries: count only) */
    uint64_t *accepted;                     /* out: n */
    int *rc;                                /* out: n, IMSAME_OK or IMSAME_EREADSIZE */
} imsame_sweep_job;

typedef struct imsame_job_opts {
    uint64_t n_threads;
    long double minevalue, mincoverage, minidentity;
    int igap, egap; /* negated, as stored by the reference (src/IMSAME.c:565,568) */
    int gpus, device;
    int trace; /* phase wall times on stderr */
    int kmer;  /* seed length, 0 = the reference's FIXED_K (12) */
    /* optional (gpus == 1): the two read sets already resident on the device (imsame_gpu_sample_*); the host
       copies q / db are still what the records are rendered from */
    imsame_sample *q_sample;
    const imsame_sample *db_sample;
    /* optional (not with the samples): the reverse strand too, after the forward records are written */
    imsame_rev_job *rev;
    /* optional (gpus == 1, not with the samples or rev): more threshold sets in the same run */
    imsame_sweep_job *sweep;
} imsame_job_opts;

/* Aligns every read of q against db and writes the records of the accepted reads to fout (may be
 * NULL: only count); then, with o->rev, the same against revComp(db) into o->rev->out.  *ctx_cache (may be NULL) keeps the context of `device` alive between jobs when
 * gpus == 1.  Returns 0 or an IMSAME_E* code; err receives the CUDA detail. */
int imsame_run_job(const imsame_fasta *q, const imsame_fasta *db, const imsame_job_opts *o, FILE *fout,
                   imsame_ctx **ctx_cache, uint64_t *accepted, char *err, size_t errlen);

#endif
