/*
 * imsame_host.h -- host-side C pieces around the GPU hot path: FASTA ingest
 * (src/IMSAME.c:196-289,320-371), exact long-double threshold tables
 * (src/alignmentFunctions.c:139,163,384), record/alignment text output
 * (src/alignmentFunctions.c:167-168,230-271) and the synthetic generator used
 * by tests and bench.py.  No CUDA here.
 */
#ifndef IMSAME_HOST_H
#define IMSAME_HOST_H
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/imsame_gpu.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- FASTA ingest -------------------------------------------------------- */
typedef struct imsame_fasta {
    unsigned char *sequences; /* ACGT only */
    uint64_t *start_pos;      /* n_seqs + 1 entries (last = total_len) */
    uint64_t total_len, n_seqs;
    uint64_t *break_pos;
    uint64_t n_breaks;
} imsame_fasta;

int imsame_fasta_load(const char *path, int is_db, imsame_fasta *out);
/* the same parser on a FASTA image in memory */
int imsame_fasta_parse_mem(const unsigned char *buf, size_t len, int is_db, imsame_fasta *out);
typedef struct imsame_file_image {
    unsigned char *data;
    size_t len;
    int mapped;
} imsame_file_image;
int imsame_file_map(const char *path, imsame_file_image *img);
void imsame_file_unmap(imsame_file_image *img);
/* src/reverseComplement.c on a memory image; *out is malloc'ed */
int imsame_revcomp_mem(const unsigned char *buf, size_t n, unsigned char **out, size_t *out_len);
/* 1 when `rev` (parse of revComp's output) is exactly the mirror image of `fwd`: bases, read offsets, word breaks */
int imsame_revcomp_is_mirror(const imsame_fasta *fwd, const imsame_fasta *rev);
/* revComp(path) as the database loader sees it (`revComp path r.fa` + imsame_fasta_load(r.fa, 1), in memory): 0, or
 * 1 = the file could not be read, 2 = no memory for its reverse complement, 3 = none for the parse.  *has_u: the
 * file holds a 'U' or 'u'.  Then imsame_revcomp_on_device(fwd, rev, has_u) decides whether the device may derive the
 * reverse read set from the forward one (imsame_gpu_sample_revcomp, imsame_gpu_db_revcomp) or has to upload rev:
 * rev is the mirror image of fwd and the file had no U (which revComp turns into an A the loader keeps). */
int imsame_revcomp_load(const char *path, imsame_fasta *rev, int *has_u);
int imsame_revcomp_on_device(const imsame_fasta *fwd, const imsame_fasta *rev, int has_u);
void imsame_fasta_free(imsame_fasta *f);
void imsame_fasta_view(const imsame_fasta *f, imsame_seqinfo *v);

/* ---- exact thresholds ------------------------------------------------------ */
/* nmin[ylen], ylen in [0, IMSAME_MAX_READ_SIZE]: smallest n = 2*idents - t_len
 * with 0.333L*ylen*db_total_len*expl(-0.275*(4n)) < min_e_value; 65535 = never. */
void imsame_build_nmin(long double min_e_value, uint64_t db_total_len, uint16_t *nmin);
void imsame_build_nmin_upto(long double min_e_value, uint64_t db_total_len, uint16_t *nmin, uint64_t max_ylen);
/* lmin[ylen]: smallest length with (long double)length/ylen >= min_coverage */
void imsame_build_lmin(long double min_coverage, uint16_t *lmin);
/* imin[len], len in [0, 2*IMSAME_MAX_READ_SIZE]: smallest identities with
 * (long double)identities/len >= min_identity; 65535 = never. imin[0] = 65535 (NaN rejects). */
void imsame_build_imin(long double min_identity, uint16_t *imin);
/* the tables of n_sets coverage/identity pairs (imsame_gpu_align_sweep): lmin_sets / imin_sets hold n_sets
 * consecutive tables of IMSAME_MAX_READ_SIZE + 1 / 2 * IMSAME_MAX_READ_SIZE + 1 entries (imsame_build_lmin /
 * imsame_build_imin of each set); lmin_all / imin_all their elementwise maxima: a pair passes every set exactly
 * when it passes those. */
void imsame_build_sweep_tables(int n_sets, const long double *coverage, const long double *identity, uint16_t *lmin_sets,
                               uint16_t *imin_sets, uint16_t *lmin_all, uint16_t *imin_all);
/* -sweep C1:I1[,C2:I2...] of the command lines (IMSAME, IMSAME_allvsall): up to IMSAME_SWEEP_ENTRIES pairs, each value
 * a whole number as atof reads it and larger than zero.  Returns NULL, or the error text the command line reports. */
#define IMSAME_SWEEP_ENTRIES (IMSAME_SWEEP_MAX - 1) /* set 0 is -coverage / -identity */
typedef struct imsame_sweep_list {
    int n;
    long double coverage[IMSAME_SWEEP_ENTRIES], identity[IMSAME_SWEEP_ENTRIES];
    char text[IMSAME_SWEEP_ENTRIES][2][64]; /* the values as given, for the summary lines */
} imsame_sweep_list;
const char *imsame_parse_sweep(const char *list, imsame_sweep_list *s);
/* -kmers K1[,K2...] of IMSAME: up to IMSAME_KMERS_ENTRIES distinct seed lengths 4..16, none equal to `kmer` (the run's
 * own -kmer, entry 0 of imsame_gpu_align_kmers).  Returns NULL, or the error text the command line reports. */
#define IMSAME_KMERS_ENTRIES (IMSAME_KMERS_MAX - 1)
typedef struct imsame_kmer_list {
    int n;
    int k[IMSAME_KMERS_ENTRIES];
} imsame_kmer_list;
const char *imsame_parse_kmers(const char *list, int kmer, imsame_kmer_list *s);

/* ---- output ---------------------------------------------------------------- */
/* header line of a record, src/alignmentFunctions.c:167 */
int imsame_format_header(char *dst, uint64_t read, uint64_t db_seq, uint32_t length, uint32_t identities,
                         uint64_t ylen);
/* -cigar: dst = the end of a header just written by imsame_format_header; its first line gains the columns
 * " q_start q_end db_start db_end score CIGAR" of `a` (imsame_gpu_align_traceback).  Returns the bytes it grew by. */
size_t imsame_format_cigar_columns(char *dst, const imsame_aln *a, const uint32_t *ops, uint64_t n_ops);
/* alignment text from a device traceback (ops = run-length path from the best
 * cell back to the border, see csrc/traceback.cuh), src/alignmentFunctions.c:230-271,493-560.
 * Returns bytes written (without the terminating 0). dst needs 6*(xlen+ylen)+256 bytes. */
uint64_t imsame_render_alignment(char *dst, const unsigned char *X, uint32_t xlen, const unsigned char *Y,
                                 uint32_t ylen, uint32_t bx, uint32_t by, const uint32_t *ops,
                                 uint64_t n_ops);

/* ---- synthetic metagenomes (SURVEY.md 8(d)) ---------------------------------- */
typedef struct imsame_synth_pool imsame_synth_pool;
void imsame_synth_set_threads(int n);
imsame_synth_pool *imsame_synth_pool_create(uint64_t seed, uint32_t n_genomes, uint64_t genome_len);
void imsame_synth_pool_destroy(imsame_synth_pool *p);
void imsame_synth_db_reads(const imsame_synth_pool *p, uint64_t seed, uint64_t first, uint64_t count,
                           uint32_t L, unsigned char *out);
void imsame_synth_query_reads(const imsame_synth_pool *p, uint64_t seed, uint64_t first, uint64_t count,
                              uint32_t L, double divergence, uint32_t n_genomes_used, unsigned char *out);
int imsame_synth_write_fasta(const char *path, const unsigned char *seq, uint64_t n_reads, uint32_t L,
                             char prefix);

#ifdef __cplusplus
}
#endif
#endif
