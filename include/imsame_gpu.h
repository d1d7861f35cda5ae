/*
 * imsame_gpu.h -- C ABI of the B200-native IMSAME alignment hot path.
 *
 * The reference (Bitlab-UMA/IMSAME) has no plugin or FFI interface: its hot
 * path is the pthread entry point
 *     void *computeAlignmentsByThread(void *HashTableArgs)     (src/alignmentFunctions.h:51,
 *                                                               src/alignmentFunctions.c:43-208)
 * fed by `HashTableArgs` (src/alignmentFunctions.h:10-30) and fanned out from
 * main (src/IMSAME.c:409-467) over a seed index built at src/IMSAME.c:232-281.
 * This library replaces exactly that: index build + query scan + ungapped
 * extension + NW/identity filter + first-accepted hit per read.  Everything is
 * plain pointers and sizes; no torch / C++ types cross the boundary.
 *
 * Error convention: functions return 0 or a negative IMSAME_E* code and never
 * call exit(); the CLI turns codes into the reference's `terror` text
 * (src/commonFunctions.c:10-13).  There is no CPU fallback: every entry point
 * that computes fails with IMSAME_ENODEV when no sm_100 device is usable.
 */
#ifndef IMSAME_GPU_H
#define IMSAME_GPU_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IMSAME_MAX_READ_SIZE 3000 /* src/structs.h:19 */
#define IMSAME_FIXED_K 12         /* src/structs.h:15 */

enum {
    IMSAME_OK = 0,
    IMSAME_ENODEV = -1,    /* no CUDA device / wrong architecture */
    IMSAME_ECUDA = -2,     /* CUDA runtime error (see imsame_gpu_last_cuda_error) */
    IMSAME_EARG = -3,      /* bad argument */
    IMSAME_ENOMEM = -4,    /* host or device allocation failed */
    IMSAME_EREADSIZE = -5, /* "Read size reached for gapped alignment." (src/alignmentFunctions.c:155) */
    IMSAME_ESTATE = -6,    /* call order violated (e.g. run before set_query) */
    IMSAME_ELIMIT = -7,    /* input exceeds an implementation limit (documented in DESIGN.md) */
    IMSAME_EPEER = -8,     /* sharded run: another shard failed (its own code is returned on its rank) */
    IMSAME_ENCCL = -9      /* NCCL missing or failed (see imsame_gpu_last_cuda_error) */
};

/* Replaces SeqInfo (src/structs.h:40-45), filled like src/IMSAME.c:199-226,323-347:
 * `sequences` holds upper-case A/C/G/T only, reads concatenated without
 * separators; start_pos[r] = offset of read r (n_seqs entries are read).
 * The reference keeps one more fact implicitly in its k-mer table: database
 * words are reset by dropped non-ACGT characters (src/IMSAME.c:229-231).
 * break_pos[] lists, ascending, the index of the first kept base after such a
 * character (NULL / 0 when the FASTA had none).  Ignored for the query. */
typedef struct imsame_seqinfo {
    const unsigned char *sequences;
    const uint64_t *start_pos;
    uint64_t total_len;
    uint64_t n_seqs;
    const uint64_t *break_pos;
    uint64_t n_breaks;
} imsame_seqinfo;

/* The value-carrying part of HashTableArgs (src/alignmentFunctions.h:10-30). */
typedef struct imsame_params {
    long double min_e_value;  /* hta->min_e_value  */
    long double min_coverage; /* hta->min_coverage */
    long double min_identity; /* hta->min_identity */
    int igap, egap;           /* negated, exactly as stored in hta (src/IMSAME.c:565,568) */
    uint64_t n_threads;       /* -n_threads: only defines chunk starts (src/IMSAME.c:414,433) */
    /* database sharding (multi-GPU): coordinates of this shard in the whole database */
    uint64_t db_total_len_global; /* 0 = this shard is the whole database */
    uint64_t db_pos_base;         /* global index of the shard's first base */
    uint64_t db_seq_base;         /* global index of the shard's first read */
} imsame_params;

/* Result per query read = what src/alignmentFunctions.c:163-173 would print. */
typedef struct imsame_best {
    uint64_t db_seq;      /* curr_db_seq (global) */
    uint64_t qpos_end;    /* curr_pos of the accepting k-mer */
    uint64_t db_pos;      /* aux->pos of the accepting hit (global) */
    uint32_t length;      /* ba.length */
    uint32_t identities;  /* ba.identities */
    uint32_t accepted;    /* 1 if the read produced a record */
    uint32_t reserved;
} imsame_best;

typedef struct imsame_stats {
    uint64_t n_query_kmers; /* entries of the query word table (K1) */
    uint64_t n_db_kmers;    /* database words scanned (K2) */
    uint64_t n_hits;        /* seed hits extended (K2) */
    uint64_t n_evalue_pass; /* hits below the e-value threshold (K2) */
    uint64_t n_pairs;       /* distinct (read, db_seq) candidates (K2b) */
    uint64_t n_pairs_dp;    /* candidates actually run through NW (K3) */
    uint64_t n_cells;       /* NW cells evaluated (K3): sum (xlen-1)(ylen-1) */
    uint64_t n_accepted;    /* reads with a record */
    float ms_pack_query, ms_k1, ms_pack_db, ms_k2, ms_k2b, ms_k3, ms_select;
    float ms_h2d, ms_d2h, ms_total;
    uint64_t h2d_bytes, d2h_bytes;
    uint32_t k2_launches, k3_launches, total_launches;
    uint32_t k3_packed_launches; /* of k3_launches: packed-word kernel (imsame_gpu_set_nw_mode) */
    float ms_comm;               /* NCCL reductions of a sharded run (imsame_gpu_run_sharded) */
    uint32_t scan_passes;        /* 1, or 2: early words first (imsame_gpu_set_passes) */
} imsame_stats;

typedef struct imsame_ctx imsame_ctx;

/* ---- lifetime ---------------------------------------------------------- */
int imsame_gpu_create(imsame_ctx **ctx, int device);
void imsame_gpu_destroy(imsame_ctx *ctx);
const char *imsame_gpu_strerror(int code);
const char *imsame_gpu_last_cuda_error(const imsame_ctx *ctx);
/* free and total memory of the context's device (cudaMemGetInfo) */
int imsame_gpu_mem_info(const imsame_ctx *ctx, uint64_t *free_bytes, uint64_t *total_bytes);
/* run all work of this context on an existing cudaStream_t (NULL = own non-blocking stream; pass
 * cudaStreamLegacy / cudaStreamPerThread to share a default stream with other libraries) */
int imsame_gpu_set_stream(imsame_ctx *ctx, void *cuda_stream);

/* ---- one call = src/IMSAME.c:232-281 + :409-467 ------------------------ */
/* Host buffers in, host records out (nq entries, caller-owned).  The database is uploaded on an internal copy
 * stream one segment (2^29 bases) ahead of its scan; nothing of the caller's buffers is in flight when the call
 * returns, whatever its result.  IMSAME_EREADSIZE exactly where the reference stops with "Read size reached for
 * gapped alignment.": an e-value-passing hit with a read of more than IMSAME_MAX_READ_SIZE bases that its query
 * read reaches before being accepted. */
int imsame_gpu_align(imsame_ctx *ctx, const imsame_seqinfo *db, const imsame_seqinfo *query,
                     const imsame_params *params, imsame_best *out, imsame_stats *stats);

/* ---- staged form (device-resident inputs; used for sharded databases) --- */
/* upload + 2-bit pack + build the query word table (K1) */
int imsame_gpu_set_query(imsame_ctx *ctx, const imsame_seqinfo *query, const imsame_params *params);
/* upload + 2-bit pack one database shard; stays resident until replaced.  Synchronous: the host buffers (pinned
 * or pageable) may be refilled or freed as soon as it returns; the same holds for imsame_gpu_set_query. */
int imsame_gpu_set_db(imsame_ctx *ctx, const imsame_seqinfo *db);
/* scan + extension + NW + filter over the resident shard. Results stay on the
 * device as one packed key per read (smaller = earlier in the reference's scan
 * order; IMSAME_KEY_NONE = no record) and one payload word.  d_keys/d_payload:
 * device buffers of nq uint64 each supplied by the caller (e.g. NCCL buffers),
 * or NULL to use the context's own. */
int imsame_gpu_run(imsame_ctx *ctx, const imsame_params *params, uint64_t *d_keys,
                   uint64_t *d_payload, imsame_stats *stats);
/* The same run in steps, for callers that exchange the keys between GPUs while it runs
 * (database shards: the earliest accepted hit of a read may live in another shard, and knowing
 * it early prunes this shard's later candidates exactly like the reference's early exit,
 * src/alignmentFunctions.c:172,189):
 *     run_begin(params, d_keys, d_payload)
 *     for seg in [0, n_segments):   run_scan(seg)           (all scans first: candidates are kept)
 *     for band in [0, n_bands):
 *         for seg in [0, n_segments): run_band(seg, band)   [caller: all-reduce(d_keys, MIN)]
 *     for seg in [0, n_segments):   run_select(seg)
 *     run_end(stats)                                        [caller: all-reduce(d_payload, MAX)]
 * Bands order a read's candidates by the position of their k-mer inside the read; run_end zeroes
 * every payload whose key is no longer the read's key, so the owner's payload survives a MAX. */
int imsame_gpu_n_segments(const imsame_ctx *ctx);
int imsame_gpu_n_bands(void);
int imsame_gpu_run_begin(imsame_ctx *ctx, const imsame_params *params, uint64_t *d_keys, uint64_t *d_payload);
int imsame_gpu_run_scan(imsame_ctx *ctx, int seg);
int imsame_gpu_run_band(imsame_ctx *ctx, int seg, int band);
int imsame_gpu_run_select(imsame_ctx *ctx, int seg);
int imsame_gpu_run_end(imsame_ctx *ctx, imsame_stats *stats);
/* after a min-reduction of the keys across shards: zero the payload of every
 * read this shard does not own, so that a max-reduction yields the owner's */
int imsame_gpu_mask_payload(imsame_ctx *ctx, const uint64_t *d_keys_reduced,
                            const uint64_t *d_keys_local, uint64_t *d_payload);
/* decode (reduced) device keys/payload into host records */
int imsame_gpu_fetch(imsame_ctx *ctx, const uint64_t *d_keys, const uint64_t *d_payload,
                     imsame_best *out);

#define IMSAME_KEY_NONE 0x7FFFFFFFFFFFFFFFull

/* ---- database sharded over several GPUs: the reduction lives in the library -------------------
 * Replaces the pthread fan-out + join of src/IMSAME.c:430-467 at the scale the reference cannot reach:
 * the database is cut into contiguous read ranges, one per GPU, the query and its word table are
 * replicated, and the per-read first accepted hit -- a minimum over the scan-order key -- is reduced
 * with ncclAllReduce(ncclUint64, ncclMin) over NVLink between k-mer-end bands (an accepted early hit
 * in one shard prunes the later candidates of that read in every shard, like the reference's early
 * exit, src/alignmentFunctions.c:172,189), followed by one ncclMax of the owner's payload.
 * NCCL is loaded at run time (libnccl.so.2; the one already in the process if there is one).
 *
 * One rank per context.  Ranks may live in one process (imsame_gpu_align_sharded does everything)
 * or in one process per GPU: rank 0 calls imsame_gpu_comm_id, hands the 128 bytes to the others by
 * any means (torch.distributed, MPI, a file), every rank calls imsame_gpu_comm_init, then
 * set_query / set_db(its shard) / imsame_gpu_run_sharded with params->db_*_base/global set. */
#define IMSAME_COMM_ID_BYTES 128
int imsame_gpu_comm_id(void *id /* IMSAME_COMM_ID_BYTES */);
int imsame_gpu_comm_init(imsame_ctx *ctx, const void *id, int n_ranks, int rank);
int imsame_gpu_comm_free(imsame_ctx *ctx);
/* imsame_gpu_run over this rank's resident shard with the key exchange every `exchange_every` bands
 * (<= 0: library default).  On return d_keys / d_payload (or the context's own buffers) hold the
 * REDUCED result on every rank; imsame_gpu_fetch decodes it.  Collective: every rank must call it. */
int imsame_gpu_run_sharded(imsame_ctx *ctx, const imsame_params *params, uint64_t *d_keys,
                           uint64_t *d_payload, int exchange_every, imsame_stats *stats);
/* The whole per-rank job in one collective call, like imsame_gpu_align: uploads the query (+ its word table) and
 * THIS rank's shard from host buffers -- the shard's segments one ahead of their scan, on a copy stream -- then
 * continues like imsame_gpu_run_sharded.  `shard` = this rank's contiguous read range with local start_pos;
 * params->db_total_len_global / db_pos_base / db_seq_base place it in the whole database. */
int imsame_gpu_align_shard(imsame_ctx *ctx, const imsame_seqinfo *shard, const imsame_seqinfo *query,
                           const imsame_params *params, uint64_t *d_keys, uint64_t *d_payload,
                           imsame_stats *stats);
/* One process, n GPUs: cut `db` into n contiguous read ranges, upload, build the query table on every
 * GPU, run sharded, decode into out (nq entries).  ctxs[i] must sit on n different devices; stats: n
 * entries or NULL.  The communicator is created on first use and kept in the contexts. */
int imsame_gpu_align_sharded(imsame_ctx *const *ctxs, int n, const imsame_seqinfo *db,
                             const imsame_seqinfo *query, const imsame_params *params, imsame_best *out,
                             imsame_stats *stats);

/* ---- the reverse strand of the resident database --------------------------------------------------
 * A read may come from either strand; the reference workflow aligns the query once more against revComp(db)
 * (src/reverseComplement.c) in a second process.  These calls give the records of `IMSAME -db revComp(db)` from
 * the database already on the device.
 *
 * The resident database (set_db, or what the last imsame_gpu_align / _align_shard left resident) becomes its reverse
 * complement in place: reads in reverse order, each reverse complemented, offsets and word breaks mirrored -- what
 * revComp + the loader give when imsame_revcomp_is_mirror holds (a break at a segment's first base, which changes
 * no word, is dropped).  Calling it again restores the forward database.  IMSAME_ESTATE without a resident
 * database, with a sample's (imsame_gpu_sample_revcomp) or while a run is in progress.
 * A per-rank caller of a sharded database sets, for the reverse strand, db_pos_base' = T - (db_pos_base + shard bases)
 * and db_seq_base' = N - (db_seq_base + shard reads) (T, N: bases and reads of the whole database). */
int imsame_gpu_db_revcomp(imsame_ctx *ctx);
/* The query, parameters and contexts of the previous imsame_gpu_align (n = 1) / imsame_gpu_align_sharded (same ctxs,
 * same order) call, aligned against the reverse complement of that call's database, which is still resident: no upload,
 * no word table rebuilt for the first pass.  out: nq records whose db_seq / db_pos count in the reverse database.
 * stats: n entries or NULL.  The database stays reversed.  IMSAME_ESTATE when the contexts do not hold the state of
 * such a call that succeeded; IMSAME_EARG when it had a non-zero db_pos_base / db_seq_base (the whole database is
 * then unknown); IMSAME_EREADSIZE exactly where the reference stops on revComp(db). */
int imsame_gpu_align_revcomp(imsame_ctx *const *ctxs, int n, imsame_best *out, imsame_stats *stats);

/* ---- several coverage / identity threshold sets in one run ------------------------------------------
 * Metagenomes are compared at more than one similarity level; the reference workflow runs one IMSAME process per
 * threshold.  Only the filter of the NW epilogue (src/alignmentFunctions.c:163) and the first-accepted selection
 * after it depend on -coverage / -identity: word table, seed hits, e-value test, candidate pairs and the NW result of
 * every pair are the same for every set, so one run gives the records of n_sets threshold sets.
 *   params[0 .. n_sets): full parameter sets that agree exactly in every field but min_coverage and min_identity
 *                        (e-value, gaps, n_threads, db_*); otherwise IMSAME_EARG.  1 <= n_sets <= IMSAME_SWEEP_MAX.
 *   out:                 n_sets x nq records; block t (out + t * nq) equals, field by field, what imsame_gpu_align
 *                        with params[t] returns.
 *   set_rc[t]:           IMSAME_OK, or IMSAME_EREADSIZE exactly where a separate imsame_gpu_align of set t stops with
 *                        "Read size reached for gapped alignment." (a candidate with a read of more than
 *                        IMSAME_MAX_READ_SIZE bases earlier in scan order than set t's final key); that set's block is
 *                        zeroed, the others are complete.  The call returns 0 when the run completed.
 *   stats:               one for the run (its n_accepted is set 0's), or NULL.
 * imsame_gpu_set_kmer / _set_passes / _set_nw_mode apply as to imsame_gpu_align; the context stays usable after
 * every error.  Device memory: 16 bytes per set and query read on top of imsame_gpu_align.  Not covered: databases
 * sharded over several GPUs, resident samples (imsame_gpu_align_samples), imsame_gpu_align_revcomp after a sweep
 * (IMSAME_ESTATE), and sweeping the e-value, the gaps or the seed length. */
#define IMSAME_SWEEP_MAX 16
int imsame_gpu_align_sweep(imsame_ctx *ctx, const imsame_seqinfo *db, const imsame_seqinfo *query,
                           const imsame_params *params, int n_sets, imsame_best *out, int *set_rc,
                           imsame_stats *stats);

/* ---- NW on explicit pairs (src/alignmentFunctions.c:389-560 in isolation) */
/* X[i] / Y[i]: ASCII reads; out5[i*5..] = score, bx, by, length, identities */
int imsame_gpu_nw_batch(imsame_ctx *ctx, uint32_t n_pairs, const unsigned char *const *X,
                        const uint32_t *xlen, const unsigned char *const *Y, const uint32_t *ylen,
                        int igap, int egap, int32_t *out5, float *ms_kernel);

/* How the database is scanned.  The reference walks the words of a query read left to right and stops at the
 * read's first accepted hit (src/alignmentFunctions.c:172,189); a read that is in the database is usually
 * accepted on one of its first words.  2 = "early words first": scan with the words that end inside the first
 * 6 of the 32 k-mer-end bands of their read, align those bands, then scan again with the later words of the
 * reads that are still without an accepted hit only (a third less scan work on config 2; identical records).
 * 1 = one scan with every word.  0 (default) = 2 when the expected number of seed hits per GPU (query bases x
 * database bases / 4^k) is at least 4e9, else 1.  Resident samples (imsame_gpu_align_samples) and callers that
 * step through a run themselves (imsame_gpu_run_begin ...) always get one pass.  In a sharded run the keys are
 * reduced between the passes; every rank must use the same setting (checked: IMSAME_ESTATE otherwise). */
int imsame_gpu_set_passes(imsame_ctx *ctx, int mode);

/* Which K3 kernel evaluates the pairs: 0 (default) = the packed-word kernel for every pair that fits it
 * (<= 321 query / 512 database bases, non-positive gap scores; nwp_core.cuh: pw_eligible) and the generic
 * kernel for the others, pair by pair; 1 = always the generic kernel.  Both give identical results; the
 * switch exists so tests and benchmarks can compare them. */
int imsame_gpu_set_nw_mode(imsame_ctx *ctx, int mode);

/* Seed length k (SURVEY 8(f) rank 4).  The reference has exactly one: FIXED_K = 12 (src/structs.h:15),
 * wired into its 12-dimensional Container (src/alignmentFunctions.h:4-6); that is the default here and
 * the only value with a reference to compare against.  Any 4 <= k <= 16 behaves like the reference
 * recompiled with FIXED_K = k over a flat 4^k table (word positions, phantom word, extension start
 * score k*POINT, t_len).  Call before imsame_gpu_set_query / imsame_gpu_align; a resident query table
 * built with another k is dropped.  The word table needs 2 * 4 * (4^k + 1) bytes of device memory
 * (134 MB at k = 12, 34 GB at k = 16). */
int imsame_gpu_set_kmer(imsame_ctx *ctx, int k);

/* ---- read sets resident on the device (all-vs-all, SURVEY 8(f) rank 3) ------------------------
 * bin/all_vs_all_metagenomes_IMSAME.sh:27-58 runs IMSAME once per ordered pair of samples and once
 * more against the reverse complement (revComp, src/reverseComplement.c): every sample is parsed,
 * indexed or scanned 14 times.  A sample is uploaded and packed ONCE here, serves as the database
 * of any number of comparisons, and keeps the word table built for it as a query.  Its reverse
 * complement is made on the device from the packed form: revComp writes the records in reverse order
 * (src/reverseComplement.c:56) and reverses each one, which together is the whole concatenated array
 * reversed and complemented; start offsets and word breaks are mirrored.  That equals revComp + the
 * loader exactly when the sample's records hold letters only, no U and one '>' per header line:
 * revComp keeps letters only (src/reverseComplement.c:65-70) whereas the database loader restarts its
 * seed word at every dropped character but '\n' (src/IMSAME.c:229-231), so a '\r', '-' or digit inside
 * a record is a word break of the sample but not of its reverse complement, and revComp turns U into
 * an A the loader keeps.  imsame_revcomp_is_mirror (imsame_b200/host/imsame_host.h) decides it on the
 * two parses; otherwise upload the parse of revComp's text with imsame_gpu_sample_create.
 * A sample used as a database must fit one segment (2^29 bases, IMSAME_ELIMIT otherwise).
 * A sample belongs to the context it was made with: imsame_gpu_align_samples points the context at the
 * query's buffers and stores the word table in the query sample, so two contexts never share one.
 * After any error of imsame_gpu_align_samples (IMSAME_ENOMEM included) the context and both samples stay
 * usable: free memory and call it again, or fall back to imsame_gpu_align. */
typedef struct imsame_sample imsame_sample;
int imsame_gpu_sample_create(imsame_ctx *ctx, const imsame_seqinfo *reads, imsame_sample **out);
int imsame_gpu_sample_revcomp(imsame_ctx *ctx, const imsame_sample *in, imsame_sample **out);
void imsame_gpu_sample_free(imsame_ctx *ctx, imsame_sample *s);
/* imsame_gpu_align with both read sets resident (same results).  The query's word table is built on
 * first use for (seed length, params->n_threads) and kept in the sample. */
int imsame_gpu_align_samples(imsame_ctx *ctx, const imsame_sample *db, imsame_sample *query,
                             const imsame_params *params, imsame_best *out, imsame_stats *stats);

/* ---- winners-only traceback (src/alignmentFunctions.c:493-546) ---------- */
/* For each accepted read of `best`, NW is recomputed on the device with one
 * back-pointer code per cell and walked back from the best border cell.  The
 * path comes back as run-length ops in traceback order (type << 28 | count:
 * 1 = diagonal steps, 2 = jump up a column: count bases of X over '-', 3 = jump
 * along a row: '-' over count bases of Y); ops of read r are
 * ops[ops_off[r] .. ops_off[r+1]) (ops_off has nq+1 entries).  cell_xy holds
 * 4 values per read: best cell (x, y) and the border cell where the walk ended.
 * `db` must be the shard that best[].db_seq (minus params->db_seq_base) indexes.
 * imsame_host.h: imsame_render_alignment() turns this into the reference's text. */
int imsame_gpu_traceback(imsame_ctx *ctx, const imsame_seqinfo *db, const imsame_seqinfo *query,
                         const imsame_params *params, const imsame_best *best, uint64_t *ops_off,
                         uint32_t **ops /* malloc'ed by the library, free with imsame_gpu_free */,
                         uint32_t *cell_xy);
void imsame_gpu_free(void *p);

/* pinned host memory helpers for callers that want full-speed copies */
void *imsame_gpu_host_alloc(uint64_t bytes);
void imsame_gpu_host_free(void *p);

#ifdef __cplusplus
}
#endif
#endif
