/*
 * oracle/imsame_oracle.h -- TEST INFRASTRUCTURE ONLY.
 *
 * CPU restatement of the IMSAME read-vs-metagenome alignment hot path, written
 * from the behaviour of the reference sources (cited per function in the .c
 * file as `src/<file>:<lines>`, relative to the reference checkout).  Nothing
 * in the product (imsame_b200/, include/, the IMSAME binary) links, imports or
 * executes this code: only tests/, __graft_entry__.smoke() and the
 * cpu_baseline / --impl reference legs of bench.py may use it, and only as
 * the checker.
 *
 * Pinning: the reference ships no tests or golden vectors ("parity unpinned
 * by reference tests").  The restatement is pinned instead against the
 * reference itself, compiled unmodified from /root/reference/src into
 * oracle/_ref/ by oracle/build_ref.sh (see tests/test_oracle_vs_reference.py
 * and tests/golden/).
 */
#ifndef IMSAME_ORACLE_H
#define IMSAME_ORACLE_H
#include <stdint.h>
#include <stdio.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ORC_MAX_READ 3000 /* src/structs.h:19 MAX_READ_SIZE */

/* src/structs.h:40-45 SeqInfo plus what the reference keeps implicitly in its
 * k-mer table: the positions at which a dropped non-ACGT character resets the
 * database word (src/IMSAME.c:229-231). brk[i] = index (in `seq`) of the first
 * kept base after such a character. */
typedef struct {
    unsigned char *seq;  /* A/C/G/T only, reads concatenated, no separators */
    uint64_t *start;     /* n_seqs+1 entries; start[n_seqs] = total_len */
    uint64_t total_len;
    uint64_t n_seqs;
    uint64_t *brk;
    uint64_t n_brk;
} orc_seqs;

typedef struct {
    long double min_e_value, min_coverage, min_identity; /* src/alignmentFunctions.h:17-19 */
    int igap, egap;     /* negated, as stored in HashTableArgs (src/IMSAME.c:565,568) */
    uint64_t n_threads; /* only defines the chunk starts (src/IMSAME.c:414,433) */
    int k;              /* seed length; the reference has FIXED_K = 12 (the only pinned value), 4..14 accepted */
    /* database shards (multi-GPU tests): 0 = db is the whole database */
    uint64_t db_total_len_global; /* database->total_len used by the e-value (src/alignmentFunctions.c:384) */
} orc_params;

typedef struct {
    uint64_t db_seq;    /* index of the database read */
    uint64_t qpos_end;  /* curr_pos of the accepting k-mer (index of its last base in query->seq) */
    uint64_t db_pos;    /* llpos.pos of the accepting hit (index after the k-mer's last base) */
    uint32_t length, identities;
    int32_t score;
    uint32_t bx, by;    /* best border cell */
    uint8_t accepted;
} orc_best;

typedef struct {
    uint64_t hits, evalue_pass, nw_calls, accepted;
} orc_stats;

int orc_load_fasta(const char *path, int is_db, orc_seqs *out);
void orc_free_seqs(orc_seqs *s);

/* ungapped extension; returns n = 2*idents - t_len  (raw score = 4n) */
int64_t orc_extend(const orc_seqs *db, const orc_seqs *q, uint64_t pos_db, uint64_t pos_q,
                   uint64_t read, uint64_t db_seq);
int64_t orc_extend_k(const orc_seqs *db, const orc_seqs *q, uint64_t pos_db, uint64_t pos_q,
                     uint64_t read, uint64_t db_seq, int k);
long double orc_evalue(int64_t n, uint64_t ylen, uint64_t db_total_len);
long double orc_default_evalue(void);

/* full NW with back-pointers + traceback + rendering (reference formulation) */
int orc_nw_traceback(const unsigned char *X, uint64_t xlen, const unsigned char *Y, uint64_t ylen,
                     int igap, int egap, int32_t *score, uint32_t *bx, uint32_t *by,
                     uint32_t *length, uint32_t *identities, char *text /* may be NULL */,
                     uint64_t text_cap);
/* same results from a forward-carried (length, identities) DP without a table */
int orc_nw_forward(const unsigned char *X, uint64_t xlen, const unsigned char *Y, uint64_t ylen,
                   int igap, int egap, int32_t *score, uint32_t *bx, uint32_t *by,
                   uint32_t *length, uint32_t *identities);

/* reference scan order with early exit (src/alignmentFunctions.c:43-208);
 * writes the .align records to `out` if not NULL, in ascending read order per chunk */
int orc_align_sequential(const orc_seqs *db, const orc_seqs *q, const orc_params *p,
                         orc_best *best, FILE *out, orc_stats *st);
/* order-free min-key form: winner(r) = argmin (qpos_end asc, db_pos desc) over
 * e-value-passing hits whose pair passes the filter */
int orc_align_bulk(const orc_seqs *db, const orc_seqs *q, const orc_params *p, orc_best *best,
                   orc_stats *st);

/* Index-free checker for inputs the reference's own index cannot hold (imsame_sampled.c): the first
 * accepted hit, in the reference's scan order with its early exit, of the query reads reads[0..n_reads)
 * against `db` (the whole database or one contiguous shard of it; db_pos_base / db_seq_base make the
 * result global, p->db_total_len_global is the e-value's database length).  best[i] belongs to reads[i].
 * Streams the database once on all host threads (OpenMP).  Returns -5 where the reference would stop
 * with "Read size reached for gapped alignment." (src/alignmentFunctions.c:155). */
void orc_set_threads(int n);
int orc_align_sampled(const orc_seqs *db, const orc_seqs *q, const orc_params *p, const uint64_t *reads,
                      uint64_t n_reads, uint64_t db_pos_base, uint64_t db_seq_base, orc_best *best,
                      orc_stats *st);

#ifdef __cplusplus
}
#endif
#endif
