/*
 * oracle/imsame_oracle.c -- TEST INFRASTRUCTURE ONLY (see imsame_oracle.h).
 *
 * Plain-C restatement of the reference's hot path. Citations are
 * `src/<file>:<lines>` of the reference checkout. The product never links this.
 */
#define _GNU_SOURCE
#include "imsame_oracle.h"
#include <ctype.h>
#include <inttypes.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#define PT 4 /* src/structs.h:13 POINT */

/* ------------------------------------------------------------------------- */
/* FASTA ingest: src/IMSAME.c:196-289 (database) and :320-371 (query).        */
/* Only A/C/G/T (after toupper) are kept; the header line is skipped up to    */
/* '\n'; text before the first '>' is ignored. For the database, any dropped  */
/* character other than '\n' resets the k-mer word (:229-231) -> recorded as  */
/* a break; read starts reset it too (:283).                                  */
/* ------------------------------------------------------------------------- */
static int is_acgt(int c) { return c == 'A' || c == 'C' || c == 'G' || c == 'T'; }

int orc_load_fasta(const char *path, int is_db, orc_seqs *out) {
    FILE *f = fopen(path, "rb");
    if (!f) return -1;
    fseek(f, 0, SEEK_END);
    long flen = ftell(f);
    fseek(f, 0, SEEK_SET);
    unsigned char *buf = (unsigned char *)malloc((size_t)flen + 1);
    if (!buf) { fclose(f); return -2; }
    if (fread(buf, 1, (size_t)flen, f) != (size_t)flen) { fclose(f); free(buf); return -3; }
    fclose(f);
    uint64_t cap_s = 1024, cap_b = 16;
    out->seq = (unsigned char *)malloc((size_t)flen + 1);
    out->start = (uint64_t *)malloc(cap_s * sizeof(uint64_t));
    out->brk = (uint64_t *)malloc(cap_b * sizeof(uint64_t));
    out->n_seqs = out->n_brk = 0;
    uint64_t pos = 0;
    long i = 0;
    while (i < flen) {
        if (buf[i] != '>') { i++; continue; }
        if (out->n_seqs + 2 > cap_s) {
            cap_s *= 2;
            out->start = (uint64_t *)realloc(out->start, cap_s * sizeof(uint64_t));
        }
        out->start[out->n_seqs++] = pos;
        while (i < flen && buf[i] != '\n') i++; /* skip ID */
        int pending_break = 0;
        for (;;) {
            i++;
            if (i >= flen) break;
            int c = toupper(buf[i]);
            if (is_acgt(c)) {
                if (pending_break && is_db && pos > out->start[out->n_seqs - 1]) {
                    if (out->n_brk + 1 > cap_b) {
                        cap_b *= 2;
                        out->brk = (uint64_t *)realloc(out->brk, cap_b * sizeof(uint64_t));
                    }
                    out->brk[out->n_brk++] = pos;
                }
                pending_break = 0;
                out->seq[pos++] = (unsigned char)c;
            } else if (c != '\n') {
                pending_break = 1;
            }
            if (c == '>') break;
        }
    }
    out->total_len = pos;
    out->start[out->n_seqs] = pos;
    free(buf);
    return 0;
}

void orc_free_seqs(orc_seqs *s) {
    free(s->seq);
    free(s->start);
    free(s->brk);
    memset(s, 0, sizeof(*s));
}

/* ------------------------------------------------------------------------- */
/* Seed index over the database: src/IMSAME.c:232-281. Every k-mer that lies  */
/* inside one read and spans no break is stored with pos = index AFTER its    */
/* last base (:247,265). Lists are head-inserted, i.e. walked in DESCENDING   */
/* pos. Here: CSR in ascending order, walked backwards.                       */
/* ------------------------------------------------------------------------- */
typedef struct {
    int k;
    uint64_t n_codes;
    uint64_t *off;  /* n_codes+1 */
    uint64_t *pos;  /* ascending within a bucket */
    uint32_t *sid;
} orc_index;

static inline unsigned base2(unsigned char c) { /* src/IMSAME.c:55-59 */
    return c == 'A' ? 0u : c == 'C' ? 1u : c == 'G' ? 2u : 3u;
}

static int build_index(const orc_seqs *db, int k, orc_index *ix) {
    if (k < 4 || k > 14) return -1; /* 4^14 offsets = 2 GB of host memory */
    ix->k = k;
    ix->n_codes = 1ull << (2 * k);
    ix->off = (uint64_t *)calloc(ix->n_codes + 1, sizeof(uint64_t));
    uint64_t mask = ix->n_codes - 1;
    for (int pass = 0; pass < 2; pass++) {
        uint64_t bi = 0;
        for (uint64_t s = 0; s < db->n_seqs; s++) {
            uint64_t word = 0, code = 0;
            for (uint64_t x = db->start[s]; x < db->start[s + 1]; x++) {
                while (bi < db->n_brk && db->brk[bi] < x) bi++;
                if (bi < db->n_brk && db->brk[bi] == x) word = 0;
                code = ((code << 2) | base2(db->seq[x])) & mask;
                if (word < (uint64_t)k) word++;
                if (word == (uint64_t)k) {
                    if (pass == 0) ix->off[code + 1]++;
                    else {
                        uint64_t slot = ix->off[code]++;
                        ix->pos[slot] = x + 1;
                        ix->sid[slot] = (uint32_t)s;
                    }
                }
            }
        }
        if (pass == 0) {
            for (uint64_t c = 0; c < ix->n_codes; c++) ix->off[c + 1] += ix->off[c];
            uint64_t n = ix->off[ix->n_codes];
            ix->pos = (uint64_t *)malloc((n + 1) * sizeof(uint64_t));
            ix->sid = (uint32_t *)malloc((n + 1) * sizeof(uint32_t));
        } else {
            /* off[c] now holds the END of bucket c; shift back */
            for (uint64_t c = ix->n_codes; c > 0; c--) ix->off[c] = ix->off[c - 1];
            ix->off[0] = 0;
        }
    }
    return 0;
}

static void free_index(orc_index *ix) {
    free(ix->off);
    free(ix->pos);
    free(ix->sid);
}

/* ------------------------------------------------------------------------- */
/* Ungapped extension: src/alignmentFunctions.c:276-359.                      */
/* pos_db / pos_q = index after the seed's last base in each array.           */
/* ------------------------------------------------------------------------- */
int64_t orc_extend(const orc_seqs *db, const orc_seqs *q, uint64_t pos_db, uint64_t pos_q,
                   uint64_t read, uint64_t db_seq) {
    return orc_extend_k(db, q, pos_db, pos_q, read, db_seq, 12); /* FIXED_K, src/structs.h:15 */
}

/* the same with FIXED_K = k: what the reference would compute if recompiled with another seed length
 * (it cannot be: its Container is a 12-dimensional array, src/alignmentFunctions.h:4-6) */
int64_t orc_extend_k(const orc_seqs *db, const orc_seqs *q, uint64_t pos_db, uint64_t pos_q,
                     uint64_t read, uint64_t db_seq, int k) {
    /* read bounds (:280-294): end = index of the last base, or total_len for the last read */
    int64_t xs = (int64_t)db->start[db_seq];
    int64_t xe = db_seq == db->n_seqs - 1 ? (int64_t)db->total_len : (int64_t)db->start[db_seq + 1] - 1;
    int64_t ys = (int64_t)q->start[read];
    int64_t ye = read == q->n_seqs - 1 ? (int64_t)q->total_len : (int64_t)q->start[read + 1] - 1;
    int64_t cd = (int64_t)pos_db, cq = (int64_t)pos_q;
    int64_t end_x = cd - 1, start_x = end_x - k + 1;
    int64_t sc = (int64_t)k * PT, hi_r = sc, hi_l = sc; /* :301-303 */
    uint64_t idents = (uint64_t)k;
    /* forward (:318-333) */
    while (sc > 0 && cd < (int64_t)db->total_len && cq < (int64_t)q->total_len) {
        if (cd > xe || cq > ye) break;
        if (db->seq[cd] == q->seq[cq]) { sc += PT; idents++; } else sc -= PT;
        if (hi_r <= sc) { end_x = cd; hi_r = sc; }
        cd++; cq++;
    }
    /* backward (:335-357): restarts from hi_r, but hi_l keeps its initial 48 */
    cd = (int64_t)pos_db - k - 1;
    cq = (int64_t)pos_q - k - 1;
    sc = hi_r;
    while (sc > 0 && cd >= 0 && cq >= 0) {
        if (cd < xs || cq < ys) break;
        if (db->seq[cd] == q->seq[cq]) { sc += PT; idents++; } else sc -= PT;
        if (hi_l <= sc) { start_x = cd; hi_l = sc; }
        cd--; cq--;
    }
    int64_t t_len = end_x - start_x; /* :359 */
    return 2 * (int64_t)idents - t_len;
}

/* e-value: src/alignmentFunctions.c:373,384 (x87 long double, unsigned wrap) */
long double orc_evalue(int64_t n, uint64_t ylen, uint64_t db_total_len) {
    uint64_t raw_u = (uint64_t)(4 * n);
    long double rawscore = raw_u;
    long double t_len = (long double)ylen;
    return (long double)0.333 * t_len * db_total_len * expl(-0.275 * rawscore);
}

/* default -evalue: 1/powl(10,20) in long double, src/IMSAME.c:44 */
long double orc_default_evalue(void) {
    return 1 / powl(10, 20);
}

/* ------------------------------------------------------------------------- */
/* NW: src/alignmentFunctions.c:389-489, traceback :493-560, rendering and    */
/* identity count :230-271. X = database read (rows), Y = query read (cols).  */
/* ------------------------------------------------------------------------- */
typedef struct { int64_t s; uint32_t fx, fy; } tcell;
typedef struct { int64_t s; uint32_t x, y; } pcell;

int orc_nw_traceback(const unsigned char *X, uint64_t xlen, const unsigned char *Y, uint64_t ylen,
                     int igap, int egap, int32_t *score, uint32_t *bx, uint32_t *by,
                     uint32_t *length, uint32_t *identities, char *text, uint64_t text_cap) {
    if (xlen < 2 || ylen < 2 || xlen > ORC_MAX_READ || ylen > ORC_MAX_READ) return -1;
    tcell *T = (tcell *)malloc(xlen * ylen * sizeof(tcell));
    pcell *mc = (pcell *)malloc(ylen * sizeof(pcell));
    if (!T || !mc) return -2;
#define AT(i, j) T[(uint64_t)(i) * ylen + (j)]
    pcell bc = {INT64_MIN, 0, 0}, mf;
    for (uint64_t j = 0; j < ylen; j++) { /* :404-413 */
        AT(0, j).s = X[0] == Y[j] ? PT : -PT;
        mc[j].s = AT(0, j).s; mc[j].x = 0; mc[j].y = (uint32_t)j;
    }
    for (uint64_t i = 1; i < xlen; i++) {
        AT(i, 0).s = X[i] == Y[0] ? PT : -PT; /* :426-429 */
        mf.s = AT(i, 0).s; mf.x = (uint32_t)i; mf.y = 0;
        for (uint64_t j = 1; j < ylen; j++) {
            if (j > 1 && mf.s <= AT(i, j - 2).s) { /* :434-438 */
                mf.s = AT(i - 1, j - 2).s; mf.x = (uint32_t)(i - 1); mf.y = (uint32_t)(j - 2);
            }
            int64_t m = X[i] == Y[j] ? PT : -PT;
            int64_t d = AT(i - 1, j - 1).s + m;
            int64_t l = j > 1 ? mf.s + igap + ((int64_t)j - ((int64_t)mf.y + 1)) * egap + m : INT64_MIN;
            int64_t r = i > 1 ? mc[j - 1].s + igap + ((int64_t)i - ((int64_t)mc[j - 1].x + 1)) * egap + m
                              : INT64_MIN;
            tcell *c = &AT(i, j);
            if (d >= l && d >= r) { c->s = d; c->fx = (uint32_t)(i - 1); c->fy = (uint32_t)(j - 1); }
            else if (r > l) { c->s = r; c->fx = mc[j - 1].x; c->fy = mc[j - 1].y; }
            else { c->s = l; c->fx = mf.x; c->fy = mf.y; }
            if (i > 1 && j > 1 && AT(i - 2, j - 1).s > mc[j - 1].s) { /* :476-480 */
                mc[j - 1].s = AT(i - 2, j - 1).s; mc[j - 1].x = (uint32_t)(i - 2); mc[j - 1].y = (uint32_t)(j - 1);
            }
            if (i == xlen - 1 || j == ylen - 1) /* :481-484 */
                if (c->s >= bc.s) { bc.s = c->s; bc.x = (uint32_t)i; bc.y = (uint32_t)j; }
        }
    }
    /* traceback (:493-546): collect columns right-to-left */
    uint64_t cap = 2 * (xlen + ylen) + 8, n = 0;
    char *cx = (char *)malloc(cap), *cy = (char *)malloc(cap);
    uint32_t px = bc.x, py = bc.y, len = 0;
    uint32_t ux = px, uy = py;
    while (ux > 0 && uy > 0) {
        ux = AT(px, py).fx; uy = AT(px, py).fy;
        if (ux == px - 1 && uy == py - 1) { cx[n] = (char)X[px]; cy[n] = (char)Y[py]; n++; len++; }
        else if (px - ux > py - uy) {
            for (uint32_t k = px; k > ux; k--) { cx[n] = (char)X[k]; cy[n] = '-'; n++; len++; }
        } else {
            for (uint32_t k = py; k > uy; k--) { cx[n] = '-'; cy[n] = (char)Y[k]; n++; len++; }
        }
        px = ux; py = uy;
    }
    /* left overhang (:548-556) */
    uint32_t lead = ux > uy ? ux : uy;
    /* forward-ordered strands: lead, path, trailing dashes (:503-504) */
    uint64_t tx = xlen - 1 - bc.x, ty = ylen - 1 - bc.y;
    uint64_t Lx = lead + n + tx, Ly = lead + n + ty;
    char *sx = (char *)malloc(Lx + 1), *sy = (char *)malloc(Ly + 1);
    for (uint32_t k = 0; k < lead; k++) { sx[k] = ux >= uy ? '-' : ' '; sy[k] = ux >= uy ? ' ' : '-'; }
    for (uint64_t k = 0; k < n; k++) { sx[lead + k] = cx[n - 1 - k]; sy[lead + k] = cy[n - 1 - k]; }
    for (uint64_t k = 0; k < tx; k++) sx[lead + n + k] = '-';
    for (uint64_t k = 0; k < ty; k++) sy[lead + n + k] = '-';
    /* rendering + identity count (:233-271): blocks of 60, loop stops when either strand ends */
    uint32_t ids = 0;
    uint64_t w = 0, i = 0, j = 0;
    while (i < Lx && j < Ly) {
        uint64_t bi = i, bj = j, o;
        for (o = 0; o < 60 && i < Lx; o++, i++) if (text && w + 4 < text_cap) text[w++] = sx[i];
        if (text && w + 4 < text_cap) text[w++] = '\n';
        for (o = 0; o < 60 && j < Ly; o++, j++) if (text && w + 4 < text_cap) text[w++] = sy[j];
        if (text && w + 4 < text_cap) text[w++] = '\n';
        for (; bi < i; bi++, bj++) {
            int star = sx[bi] != '-' && bj < Ly && sy[bj] != '-' && sx[bi] == sy[bj];
            if (star) ids++;
            if (text && w + 4 < text_cap) text[w++] = star ? '*' : ' ';
        }
        if (text && w + 4 < text_cap) text[w++] = '\n';
    }
    if (text) { text[w++] = '\n'; text[w] = 0; }
    *score = (int32_t)bc.s; *bx = bc.x; *by = bc.y; *length = len; *identities = ids;
    free(sx); free(sy); free(cx); free(cy); free(T); free(mc);
#undef AT
    return 0;
}

/* Forward-carried form: each cell carries (length, identities) of its own
 * traceback path, so the filter needs no table (SURVEY.md section 8(a) A5).
 * diag: (len+1, id+match) from (i-1,j-1); jump to (px,py): len += max(i-px, j-py).
 * Cells on row 0 / column 0 carry (0,0). Rolling storage: three rows. */
int orc_nw_forward(const unsigned char *X, uint64_t xlen, const unsigned char *Y, uint64_t ylen,
                   int igap, int egap, int32_t *score, uint32_t *bx, uint32_t *by,
                   uint32_t *length, uint32_t *identities) {
    if (xlen < 2 || ylen < 2) return -1;
    typedef struct { int32_t s; uint32_t len, id; } fc;
    fc *row[3];
    for (int r = 0; r < 3; r++) row[r] = (fc *)calloc(ylen, sizeof(fc));
    struct { int32_t s; uint32_t x, len, id; } *mc = calloc(ylen, sizeof(*mc));
    fc *p2 = row[0], *p1 = row[1], *cu = row[2]; /* rows i-2, i-1, i */
    for (uint64_t j = 0; j < ylen; j++) {
        p1[j].s = X[0] == Y[j] ? PT : -PT; p1[j].len = p1[j].id = 0;
        mc[j].s = p1[j].s; mc[j].x = 0; mc[j].len = mc[j].id = 0;
    }
    int64_t bs = INT64_MIN; uint32_t bcx = 0, bcy = 0, bl = 0, bi = 0;
    for (uint64_t i = 1; i < xlen; i++) {
        cu[0].s = X[i] == Y[0] ? PT : -PT; cu[0].len = cu[0].id = 0;
        int32_t mfs = cu[0].s; uint32_t mfy = 0, mfl = 0, mfi = 0;
        for (uint64_t j = 1; j < ylen; j++) {
            if (j > 1 && mfs <= cu[j - 2].s) { mfs = p1[j - 2].s; mfy = (uint32_t)(j - 2); mfl = p1[j - 2].len; mfi = p1[j - 2].id; }
            int match = X[i] == Y[j];
            int32_t m = match ? PT : -PT;
            int64_t d = (int64_t)p1[j - 1].s + m;
            int64_t l = j > 1 ? (int64_t)mfs + igap + ((int64_t)j - ((int64_t)mfy + 1)) * egap + m : INT64_MIN;
            int64_t r = i > 1 ? (int64_t)mc[j - 1].s + igap + ((int64_t)i - ((int64_t)mc[j - 1].x + 1)) * egap + m : INT64_MIN;
            if (d >= l && d >= r) { cu[j].s = (int32_t)d; cu[j].len = p1[j - 1].len + 1; cu[j].id = p1[j - 1].id + (uint32_t)match; }
            else if (r > l) { cu[j].s = (int32_t)r; cu[j].len = mc[j - 1].len + (uint32_t)(i - mc[j - 1].x); cu[j].id = mc[j - 1].id; }
            else { cu[j].s = (int32_t)l; cu[j].len = mfl + (uint32_t)(j - mfy); cu[j].id = mfi; }
            if (i > 1 && j > 1 && p2[j - 1].s > mc[j - 1].s) { mc[j - 1].s = p2[j - 1].s; mc[j - 1].x = (uint32_t)(i - 2); mc[j - 1].len = p2[j - 1].len; mc[j - 1].id = p2[j - 1].id; }
            if ((i == xlen - 1 || j == ylen - 1) && cu[j].s >= bs) { bs = cu[j].s; bcx = (uint32_t)i; bcy = (uint32_t)j; bl = cu[j].len; bi = cu[j].id; }
        }
        fc *t = p2; p2 = p1; p1 = cu; cu = t;
    }
    *score = (int32_t)bs; *bx = bcx; *by = bcy; *length = bl; *identities = bi;
    for (int r = 0; r < 3; r++) free(row[r]);
    free(mc);
    return 0;
}

/* filter: src/alignmentFunctions.c:163 */
static int accept_pair(uint32_t length, uint32_t identities, uint64_t ylen, const orc_params *p) {
    return ((long double)length / ylen) >= p->min_coverage &&
           ((long double)identities / length) >= p->min_identity;
}

static void emit_record(FILE *out, uint64_t r, uint64_t s, uint32_t len, uint32_t id, uint64_t ylen,
                        const char *text) { /* :167-168 */
    uint64_t pi = 100ull * id / len, pc = 100ull * len / ylen;
    fprintf(out, "(%" PRIu64 ", %" PRIu64 ") : %d%% %d%% %" PRIu64 "\n $$$$$$$ \n", r, s,
            (int)(pi > 100 ? 100 : pi), (int)(pc > 100 ? 100 : pc), ylen);
    fprintf(out, "%s", text);
}

/* ------------------------------------------------------------------------- */
/* Query scan in reference order: src/alignmentFunctions.c:84-203, chunking   */
/* src/IMSAME.c:414,430-452.                                                  */
/* ------------------------------------------------------------------------- */
int orc_align_sequential(const orc_seqs *db, const orc_seqs *q, const orc_params *p,
                         orc_best *best, FILE *out, orc_stats *st) {
    if (p->k < 4 || p->k > 14) return -9; /* k != 12: no reference to compare against (orc_extend_k) */
    orc_index ix;
    if (build_index(db, p->k, &ix)) return -1;
    orc_stats z = {0, 0, 0, 0};
    char *text = out ? (char *)malloc(4 * (2 * ORC_MAX_READ + 64) * 3) : NULL;
    uint64_t text_cap = 4 * (2 * ORC_MAX_READ + 64) * 3;
    for (uint64_t r = 0; r < q->n_seqs; r++) memset(&best[r], 0, sizeof(orc_best));
    uint64_t T = p->n_threads ? p->n_threads : 1;
    uint64_t per = q->n_seqs / T;
    uint64_t mask = ix.n_codes - 1;
    for (uint64_t t = 0; t < T; t++) {
        uint64_t from = t * per, to = (t == T - 1) ? q->n_seqs : (t + 1) * per;
        if (from >= to) continue;
        uint64_t cr = from, cp = q->start[from], filled = 0, code = 0;
        int aligned = 0;
        while (cr < to && cp < q->total_len) {
            uint64_t up_to = cr < q->n_seqs - 1 ? q->start[cr + 1] - 1 : q->total_len;
            if (cp == up_to) { filled = 0; aligned = 0; cr++; continue; } /* :96-105: no advance */
            code = ((code << 2) | base2(q->seq[cp])) & mask;
            filled++;
            if (filled >= (uint64_t)p->k) {
                uint64_t lo = ix.off[code], hi = ix.off[code + 1];
                uint64_t ylen = q->start[cr + 1] - q->start[cr];
                for (uint64_t h = hi; h > lo && !aligned; h--) { /* descending pos */
                    uint64_t pos = ix.pos[h - 1], s = ix.sid[h - 1];
                    z.hits++;
                    int64_t n = orc_extend_k(db, q, pos, cp + 1, cr, s, p->k);
                    if (!(orc_evalue(n, ylen, p->db_total_len_global ? p->db_total_len_global : db->total_len) < p->min_e_value)) continue;
                    z.evalue_pass++;
                    uint64_t xlen = db->start[s + 1] - db->start[s];
                    if (xlen > ORC_MAX_READ || ylen > ORC_MAX_READ) { free_index(&ix); free(text); return -5; }
                    int32_t sc; uint32_t bx, by, len, id;
                    z.nw_calls++;
                    if (orc_nw_traceback(db->seq + db->start[s], xlen, q->seq + q->start[cr], ylen, p->igap,
                                         p->egap, &sc, &bx, &by, &len, &id, text, text_cap)) continue;
                    if (accept_pair(len, id, ylen, p)) {
                        z.accepted++;
                        orc_best *b = &best[cr];
                        b->db_seq = s; b->qpos_end = cp; b->db_pos = pos; b->length = len; b->identities = id;
                        b->score = sc; b->bx = bx; b->by = by; b->accepted = 1;
                        if (out) emit_record(out, cr, s, len, id, ylen, text);
                        aligned = 1;
                    }
                }
                if (aligned) {
                    if (cr == q->n_seqs - 1) break; /* reference reads start_pos[n_seqs] here; benign */
                    cp = q->start[cr + 1] - 2;       /* :190 */
                } else filled--;                     /* :192-194 slide */
            }
            cp++;
        }
    }
    if (st) *st = z;
    free(text);
    free_index(&ix);
    return 0;
}

/* ------------------------------------------------------------------------- */
/* Order-free form (SURVEY.md Appendix B): every read independently, all      */
/* hits, minimum key among accepted. Pair results are cached per read.        */
/* ------------------------------------------------------------------------- */
int orc_align_bulk(const orc_seqs *db, const orc_seqs *q, const orc_params *p, orc_best *best,
                   orc_stats *st) {
    if (p->k < 4 || p->k > 14) return -9;
    orc_index ix;
    if (build_index(db, p->k, &ix)) return -1;
    orc_stats z = {0, 0, 0, 0};
    uint64_t T = p->n_threads ? p->n_threads : 1, per = q->n_seqs / T;
    uint64_t mask = ix.n_codes - 1;
    /* small per-read pair cache */
    uint64_t ccap = 64, cn;
    struct pc { uint64_t s; uint32_t len, id, bx, by; int32_t sc; int ok; } *cache = malloc(ccap * sizeof(*cache));
    for (uint64_t r = 0; r < q->n_seqs; r++) {
        orc_best *b = &best[r];
        memset(b, 0, sizeof(*b));
        cn = 0;
        int first = 0;
        for (uint64_t t = 0; t < T; t++) if (r == t * per && (t == 0 || per > 0)) first = 1;
        if (per == 0) first = (r == 0);
        uint64_t ylen = q->start[r + 1] - q->start[r];
        int64_t lo = first ? (int64_t)q->start[r] : (int64_t)q->start[r] - 1;
        int64_t hi = r < q->n_seqs - 1 ? (int64_t)q->start[r + 1] - 2 : (int64_t)q->total_len - 1;
        for (int64_t e = lo + p->k - 1; e <= hi; e++) {
            uint64_t code = 0;
            for (int64_t x = e - p->k + 1; x <= e; x++) code = ((code << 2) | base2(q->seq[x])) & mask;
            for (uint64_t h = ix.off[code + 1]; h > ix.off[code]; h--) {
                uint64_t pos = ix.pos[h - 1], s = ix.sid[h - 1];
                z.hits++;
                /* key order: e ascending, pos descending; skip anything not better */
                if (b->accepted && !((uint64_t)e < b->qpos_end || ((uint64_t)e == b->qpos_end && pos > b->db_pos))) continue;
                int64_t n = orc_extend_k(db, q, pos, (uint64_t)e + 1, r, s, p->k);
                if (!(orc_evalue(n, ylen, p->db_total_len_global ? p->db_total_len_global : db->total_len) < p->min_e_value)) continue;
                z.evalue_pass++;
                uint64_t ci;
                for (ci = 0; ci < cn; ci++) if (cache[ci].s == s) break;
                if (ci == cn) {
                    if (cn == ccap) { ccap *= 2; cache = realloc(cache, ccap * sizeof(*cache)); }
                    uint64_t xlen = db->start[s + 1] - db->start[s];
                    cache[ci].s = s;
                    z.nw_calls++;
                    orc_nw_forward(db->seq + db->start[s], xlen, q->seq + q->start[r], ylen, p->igap, p->egap,
                                   &cache[ci].sc, &cache[ci].bx, &cache[ci].by, &cache[ci].len, &cache[ci].id);
                    cache[ci].ok = cache[ci].len > 0 && accept_pair(cache[ci].len, cache[ci].id, ylen, p);
                    cn++;
                }
                if (!cache[ci].ok) continue;
                b->db_seq = s; b->qpos_end = (uint64_t)e; b->db_pos = pos; b->length = cache[ci].len;
                b->identities = cache[ci].id; b->score = cache[ci].sc; b->bx = cache[ci].bx; b->by = cache[ci].by;
                b->accepted = 1;
            }
        }
        if (b->accepted) z.accepted++;
    }
    free(cache);
    if (st) *st = z;
    free_index(&ix);
    return 0;
}
