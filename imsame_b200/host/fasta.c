/*
 * fasta.c -- FASTA ingest producing the reference's in-memory form.
 *
 * Behaviour follows src/IMSAME.c:196-289 (database) and :320-371 (query):
 *   - a record starts at '>' ; the header is skipped up to the first '\n';
 *   - text before the first '>' is ignored;
 *   - characters are upper-cased; only A/C/G/T are stored, everything else is
 *     dropped (multi-line records therefore concatenate);
 *   - start_pos[r] = number of stored bases before record r;
 *   - for the database, a dropped character other than '\n' resets the seed
 *     word (src/IMSAME.c:229-231): the index of the next stored base is
 *     recorded in break_pos[] when it is not already a read start.
 * The file is mapped and parsed by all host threads with a class table instead of the
 * reference's char-at-a-time buffered reader (src/commonFunctions.c:15-23): it is cut
 * at "\n>" boundaries (always a record start: a header never spans a newline), every
 * thread first counts the bases / records / breaks of its piece, a prefix sum gives
 * each piece its place in the output arrays, and a second pass writes them.  The
 * reference reads 3.5 Mbp/s (with indexing); cfg2's 2.6 GB database FASTA would otherwise
 * take four times longer to parse than to align on the GPU.
 */
#include "imsame_host.h"
#include <fcntl.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#if defined(__SSE2__)
#include <emmintrin.h>
#endif

enum { C_BASE = 0, C_NL = 1, C_GT = 2, C_OTHER = 3 };

/* is ln[0, n) made of upper-case A/C/G/T only?  16 bytes per step where SSE2 exists (every x86-64) */
static int all_upper_acgt(const unsigned char *ln, size_t n) {
    size_t k = 0;
#if defined(__SSE2__)
    const __m128i a = _mm_set1_epi8('A'), c = _mm_set1_epi8('C'), g = _mm_set1_epi8('G'), t = _mm_set1_epi8('T');
    for (; k + 16 <= n; k += 16) {
        const __m128i v = _mm_loadu_si128((const __m128i *)(ln + k));
        const __m128i ok = _mm_or_si128(_mm_or_si128(_mm_cmpeq_epi8(v, a), _mm_cmpeq_epi8(v, c)),
                                        _mm_or_si128(_mm_cmpeq_epi8(v, g), _mm_cmpeq_epi8(v, t)));
        if (_mm_movemask_epi8(ok) != 0xFFFF) return 0;
    }
#endif
    for (; k < n; k++) {
        const unsigned char x = ln[k];
        if (!((x == 'A') | (x == 'C') | (x == 'G') | (x == 'T'))) return 0;
    }
    return 1;
}

typedef struct {
    uint64_t bases, recs, brks;
} piece_counts;

/* Parse buf[i, end).  For every piece but the first, buf[i] == '>'.  With seq == NULL only count;
 * otherwise write bases at seq[pos..], record starts at start[n..], breaks at brk[nb..]. */
static void parse_piece(const unsigned char *buf, size_t i, size_t end, int is_db, const unsigned char *cls,
                        const unsigned char *up, unsigned char *seq, uint64_t *start, uint64_t *brk, uint64_t pos,
                        uint64_t n, uint64_t nb, piece_counts *cnt) {
    const uint64_t pos0 = pos, n0 = n, nb0 = nb;
    while (i < end && buf[i] != '>') i++; /* text before the first header is ignored */
    while (i < end) {
        /* buf[i] == '>' */
        const uint64_t rec_start = pos;
        if (seq) start[n] = pos;
        n++;
        const unsigned char *nl = (const unsigned char *)memchr(buf + i, '\n', end - i);
        if (!nl) break;
        i = (size_t)(nl - buf) + 1;
        int pending = 0;
        while (i < end) {
            /* fast path: a whole line of nothing but A/C/G/T (any case) is classified with one pass and
               copied with another, without the per-character state machine below */
            if (!pending) {
                const unsigned char *le = (const unsigned char *)memchr(buf + i, '\n', end - i);
                const size_t ll = (le ? (size_t)(le - buf) : end) - i;
                unsigned bad = 0, lower = 0;
                if (!all_upper_acgt(buf + i, ll)) /* the common case needs no table */
                    for (size_t k = 0; k < ll; k++) { bad |= cls[buf[i + k]]; lower |= buf[i + k]; }
                if (!bad && ll) {
                    if (seq) {
                        if (lower & 0x20) for (size_t k = 0; k < ll; k++) seq[pos + k] = up[buf[i + k]];
                        else memcpy(seq + pos, buf + i, ll);
                    }
                    pos += ll;
                    i += ll + (le ? 1 : 0);
                    continue;
                }
            }
            const unsigned char c = buf[i];
            const unsigned k = cls[c];
            if (k == C_BASE) {
                if (pending) {
                    if (is_db && pos > rec_start) {
                        if (seq) brk[nb] = pos;
                        nb++;
                    }
                    pending = 0;
                }
                if (seq) seq[pos] = up[c];
                pos++;
            } else if (k == C_GT) {
                break;
            } else if (k == C_OTHER) {
                pending = 1;
            }
            i++;
        }
    }
    if (cnt) { cnt->bases = pos - pos0; cnt->recs = n - n0; cnt->brks = nb - nb0; }
}

/* parse a FASTA image held in memory (the file, or the output of imsame_revcomp_mem) */
int imsame_fasta_parse_mem(const unsigned char *buf, size_t flen, int is_db, imsame_fasta *out) {
    memset(out, 0, sizeof(*out));
    unsigned char cls[256], up[256];
    for (int c = 0; c < 256; c++) { cls[c] = C_OTHER; up[c] = (unsigned char)c; }
    cls['\n'] = C_NL;
    cls['>'] = C_GT;
    const char *b = "ACGTacgt";
    for (int i = 0; i < 8; i++) { cls[(unsigned char)b[i]] = C_BASE; up[(unsigned char)b[i]] = (unsigned char)b[i & 3]; }

    /* pieces: cut at "\n>" so that every piece but the first starts on a header */
    int np = 1;
#ifdef _OPENMP
    np = omp_get_max_threads();
#endif
    if (np > 256) np = 256;
    size_t piece = 1 << 20; /* >= 1 MB per piece */
    const char *tp = getenv("IMSAME_TEST_FASTA_PIECE"); /* test hook (tools/host_fuzz.c): many pieces on small inputs */
    if (tp && atol(tp) > 0) { piece = (size_t)atol(tp); np = 256; }
    if ((size_t)np > flen / piece + 1) np = (int)(flen / piece + 1);
    size_t cut[257];
    cut[0] = 0;
    for (int k = 1; k < np; k++) {
        size_t at = flen / (size_t)np * (size_t)k;
        if (at < cut[k - 1]) at = cut[k - 1];
        size_t found = flen;
        while (at < flen) {
            const unsigned char *g = (const unsigned char *)memchr(buf + at, '>', flen - at);
            if (!g) break;
            const size_t gi = (size_t)(g - buf);
            if (gi > 0 && buf[gi - 1] == '\n') { found = gi; break; }
            at = gi + 1;
        }
        cut[k] = found;
    }
    cut[np] = flen;

    piece_counts cnt[256];
    memset(cnt, 0, sizeof cnt);
#pragma omp parallel for schedule(static, 1)
    for (int k = 0; k < np; k++)
        parse_piece(buf, cut[k], cut[k + 1], is_db, cls, up, NULL, NULL, NULL, 0, 0, 0, &cnt[k]);
    uint64_t pos0[257], n0[257], nb0[257];
    pos0[0] = n0[0] = nb0[0] = 0;
    for (int k = 0; k < np; k++) {
        pos0[k + 1] = pos0[k] + cnt[k].bases;
        n0[k + 1] = n0[k] + cnt[k].recs;
        nb0[k + 1] = nb0[k] + cnt[k].brks;
    }
    unsigned char *seq = (unsigned char *)malloc((size_t)pos0[np] + 64);
    uint64_t *start = (uint64_t *)malloc((n0[np] + 2) * sizeof(uint64_t));
    uint64_t *brk = (uint64_t *)malloc((nb0[np] + 1) * sizeof(uint64_t));
    if (!seq || !start || !brk) { free(seq); free(start); free(brk); return IMSAME_ENOMEM; }
#pragma omp parallel for schedule(static, 1)
    for (int k = 0; k < np; k++)
        parse_piece(buf, cut[k], cut[k + 1], is_db, cls, up, seq, start, brk, pos0[k], n0[k], nb0[k], NULL);
    start[n0[np]] = pos0[np];
    out->sequences = seq;
    out->start_pos = start;
    out->break_pos = brk;
    out->total_len = pos0[np];
    out->n_seqs = n0[np];
    out->n_breaks = nb0[np];
    return IMSAME_OK;
}

/* whole file -> memory image (mapped when possible); release with imsame_file_unmap */
int imsame_file_map(const char *path, imsame_file_image *img) {
    memset(img, 0, sizeof(*img));
    const int fd = open(path, O_RDONLY);
    if (fd < 0) return IMSAME_EARG;
    struct stat st;
    if (fstat(fd, &st)) { close(fd); return IMSAME_EARG; }
    size_t flen = (size_t)st.st_size;
    unsigned char *buf = NULL;
    if (S_ISREG(st.st_mode) && flen > 0) {
        void *m = mmap(NULL, flen, PROT_READ, MAP_PRIVATE, fd, 0);
        if (m != MAP_FAILED) { buf = (unsigned char *)m; img->mapped = 1; madvise(m, flen, MADV_SEQUENTIAL | MADV_WILLNEED); }
    }
    if (!buf) { /* not mappable (or empty): read it */
        size_t cap = flen ? flen : (1 << 16), got = 0;
        buf = (unsigned char *)malloc(cap + 1);
        if (!buf) { close(fd); return IMSAME_ENOMEM; }
        for (;;) {
            if (got == cap) {
                cap *= 2;
                unsigned char *nb2 = (unsigned char *)realloc(buf, cap + 1);
                if (!nb2) { free(buf); close(fd); return IMSAME_ENOMEM; }
                buf = nb2;
            }
            const ssize_t r = read(fd, buf + got, cap - got);
            if (r < 0) { free(buf); close(fd); return IMSAME_EARG; }
            if (r == 0) break;
            got += (size_t)r;
        }
        flen = got;
    }
    close(fd);
    img->data = buf;
    img->len = flen;
    return IMSAME_OK;
}

void imsame_file_unmap(imsame_file_image *img) {
    if (img->data) {
        if (img->mapped) munmap(img->data, img->len); else free(img->data);
    }
    memset(img, 0, sizeof(*img));
}

int imsame_fasta_load(const char *path, int is_db, imsame_fasta *out) {
    memset(out, 0, sizeof(*out));
    imsame_file_image img;
    int rc = imsame_file_map(path, &img);
    if (rc) return rc;
    rc = imsame_fasta_parse_mem(img.data, img.len, is_db, out);
    imsame_file_unmap(&img);
    return rc;
}

/* The reference's reverse-complement tool on a memory image (src/reverseComplement.c:21-118):
 * records in REVERSE file order (:56); a record starts at every '>' byte (:47-52); the header line is
 * copied verbatim (:59-62); only letters are kept from the body (:65-70) and written
 * reverse-complemented on ONE line (:71-112) with A<->T, C<->G, U->A (case preserved), every other
 * letter unchanged.  *out is malloc'ed (free it). */
/* Threaded like the parser: the '>' bytes are located piece by piece (count, prefix sum, fill), every record's
 * output length is counted (header line + letters + '\n'), a suffix sum over the records gives each its place in
 * the output (records come out in reverse order), and a last pass writes them.  A header line that holds further
 * '>' bytes is copied once per '>' (every '>' starts a record, :47-52, and the header runs to the end of the
 * line, :59), so the output can be far longer than the input: hence the counting pass. */
static inline int is_letter(unsigned char c) { return (unsigned)((c | 0x20) - 'a') < 26u; }

/* header end (one past its '\n') and body end (the next '>' at or after the header end) of record r */
static inline void record_bounds(const unsigned char *buf, size_t n, const size_t *off, size_t nrec, size_t r, size_t *h, size_t *end) {
    const unsigned char *nl = (const unsigned char *)memchr(buf + off[r], '\n', n - off[r]);
    *h = nl ? (size_t)(nl - buf) + 1 : n;
    size_t k = r + 1;
    while (k < nrec && off[k] < *h) k++; /* '>' bytes inside the header line */
    *end = k < nrec ? off[k] : n;
}

int imsame_revcomp_mem(const unsigned char *buf, size_t n, unsigned char **out, size_t *out_len) {
    unsigned char comp[256];
    for (int c = 0; c < 256; c++) comp[c] = (unsigned char)c;
    comp['A'] = 'T'; comp['C'] = 'G'; comp['G'] = 'C'; comp['T'] = 'A'; comp['U'] = 'A';
    comp['a'] = 't'; comp['c'] = 'g'; comp['g'] = 'c'; comp['t'] = 'a'; comp['u'] = 'a';
    int np = 1;
#ifdef _OPENMP
    np = omp_get_max_threads();
#endif
    if (np > 256) np = 256;
    size_t piece = 1 << 20;
    const char *tp = getenv("IMSAME_TEST_FASTA_PIECE"); /* test hook, as in imsame_fasta_parse_mem */
    if (tp && atol(tp) > 0) { piece = (size_t)atol(tp); np = 256; }
    if ((size_t)np > n / piece + 1) np = (int)(n / piece + 1);
    /* 1. where the records start */
    size_t first[257];
    first[0] = 0;
#pragma omp parallel for schedule(static, 1) if (np > 1)
    for (int k = 0; k < np; k++) {
        const size_t a = n / (size_t)np * (size_t)k, b = k + 1 == np ? n : n / (size_t)np * (size_t)(k + 1);
        size_t c = 0;
        for (const unsigned char *g = buf + a; g < buf + b && (g = (const unsigned char *)memchr(g, '>', (size_t)(buf + b - g))) != NULL; g++) c++;
        first[k + 1] = c;
    }
    for (int k = 0; k < np; k++) first[k + 1] += first[k];
    const size_t nrec = first[np];
    size_t *off = (size_t *)malloc((nrec + 1) * sizeof(size_t));
    size_t *place = (size_t *)malloc((nrec + 1) * sizeof(size_t)); /* output length, then output offset, of record r */
    if (!off || !place) { free(off); free(place); return IMSAME_ENOMEM; }
#pragma omp parallel for schedule(static, 1) if (np > 1)
    for (int k = 0; k < np; k++) {
        const size_t a = n / (size_t)np * (size_t)k, b = k + 1 == np ? n : n / (size_t)np * (size_t)(k + 1);
        size_t w = first[k];
        for (const unsigned char *g = buf + a; g < buf + b && (g = (const unsigned char *)memchr(g, '>', (size_t)(buf + b - g))) != NULL; g++)
            off[w++] = (size_t)(g - buf);
    }
    /* 2. output length of every record */
#pragma omp parallel for schedule(static) if (np > 1)
    for (int64_t r = 0; r < (int64_t)nrec; r++) {
        size_t h, end, letters = 0;
        record_bounds(buf, n, off, nrec, (size_t)r, &h, &end);
        for (size_t k = h; k < end; k++) letters += (size_t)is_letter(buf[k]);
        place[r] = (h - off[r]) + letters + 1;
    }
    /* 3. records in REVERSE file order (:56): record r starts where the records after it end */
    size_t total = 0;
    for (size_t r = nrec; r-- > 0;) {
        const size_t len = place[r];
        place[r] = total;
        total += len;
    }
    unsigned char *dst = (unsigned char *)malloc(total + 16);
    if (!dst) { free(off); free(place); return IMSAME_ENOMEM; }
#pragma omp parallel for schedule(static) if (np > 1)
    for (int64_t r = 0; r < (int64_t)nrec; r++) {
        /* header = up to the first newline (fgets, :59), even if it holds another '>';
           body = up to the next '>' after the header (:65), letters only, reverse-complemented on one line */
        size_t h, end, w = place[r];
        record_bounds(buf, n, off, nrec, (size_t)r, &h, &end);
        memcpy(dst + w, buf + off[r], h - off[r]);
        w += h - off[r];
        for (size_t k = end; k-- > h;) {
            const unsigned char c = buf[k];
            dst[w] = comp[c];
            w += (size_t)is_letter(c);
        }
        dst[w] = '\n';
    }
    free(off);
    free(place);
    *out = dst;
    *out_len = total;
    return IMSAME_OK;
}

/* Is `rev` (the parse of revComp's output for a sample) exactly the mirror image of `fwd` (the parse of the sample):
 * the concatenated bases reversed and complemented, read offsets and word breaks mirrored?  Then -- and only then --
 * the device may derive the reverse-complemented read set from the packed forward one (csrc/capi_samples.inc).
 * It is not whenever revComp's text filter and the loader's disagree: revComp keeps letters only
 * (src/reverseComplement.c:65-70), so a '\r', '-', '*' or digit inside a record restarts the database's seed word in
 * the sample (src/IMSAME.c:229-231) but not in its reverse complement; 'U' comes back as an 'A' the loader keeps;
 * a header line with several '>' bytes comes out once per '>'. */
int imsame_revcomp_is_mirror(const imsame_fasta *fwd, const imsame_fasta *rev) {
    if (fwd->n_seqs != rev->n_seqs || fwd->total_len != rev->total_len || fwd->n_breaks != rev->n_breaks) return 0;
    const uint64_t n = fwd->n_seqs, total = fwd->total_len, nb = fwd->n_breaks;
    for (uint64_t i = 0; i <= n; i++)
        if (rev->start_pos[i] != total - fwd->start_pos[n - i]) return 0;
    for (uint64_t i = 0; i < nb; i++)
        if (rev->break_pos[i] != total - fwd->break_pos[nb - 1 - i]) return 0;
    unsigned char comp[256];
    memset(comp, 0, sizeof comp);
    comp['A'] = 'T'; comp['C'] = 'G'; comp['G'] = 'C'; comp['T'] = 'A';
    int differ = 0;
#pragma omp parallel for reduction(| : differ) schedule(static)
    for (int64_t i = 0; i < (int64_t)total; i++) differ |= rev->sequences[i] != comp[fwd->sequences[total - 1 - (uint64_t)i]];
    return !differ;
}

/* The in-memory form of `revComp path r.fa` + the database loader: the file mapped, reverse complemented
 * (imsame_revcomp_mem) and parsed with is_db = 1.  *has_u: the file holds a 'U' or 'u'. */
int imsame_revcomp_load(const char *path, imsame_fasta *rev, int *has_u) {
    memset(rev, 0, sizeof(*rev));
    imsame_file_image img;
    if (imsame_file_map(path, &img)) return 1;
    *has_u = memchr(img.data, 'U', img.len) != NULL || memchr(img.data, 'u', img.len) != NULL;
    unsigned char *rc = NULL;
    size_t rc_len = 0;
    const int e = imsame_revcomp_mem(img.data, img.len, &rc, &rc_len);
    imsame_file_unmap(&img);
    if (e) return 2;
    const int pe = imsame_fasta_parse_mem(rc, rc_len, 1, rev);
    free(rc);
    return pe ? 3 : 0;
}

/* revComp turns U into an A the loader keeps, so a file with a U never qualifies, whatever the parses say */
int imsame_revcomp_on_device(const imsame_fasta *fwd, const imsame_fasta *rev, int has_u) {
    return !has_u && imsame_revcomp_is_mirror(fwd, rev);
}

void imsame_fasta_free(imsame_fasta *f) {
    free(f->sequences);
    free(f->start_pos);
    free(f->break_pos);
    memset(f, 0, sizeof(*f));
}

void imsame_fasta_view(const imsame_fasta *f, imsame_seqinfo *v) {
    v->sequences = f->sequences;
    v->start_pos = f->start_pos;
    v->total_len = f->total_len;
    v->n_seqs = f->n_seqs;
    v->break_pos = f->break_pos;
    v->n_breaks = f->n_breaks;
}
