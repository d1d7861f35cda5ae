/*
 * thresholds.c -- the reference's three floating-point tests, turned into
 * integer tables on the host so the device never evaluates them.
 *
 *   e-value   src/alignmentFunctions.c:373,384 + test :139
 *   coverage  src/alignmentFunctions.c:163 (first operand)
 *   identity  src/alignmentFunctions.c:163 (second operand)
 *
 * All three are evaluated here in x87 `long double`, with the operand types
 * and the left-to-right evaluation order of the reference expression, and are
 * monotone in the integer they are tabulated over, so "value >= table[...]"
 * on the device decides exactly like the reference.
 */
#include "imsame_host.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>

/* e = (long double)0.333 * t_len * db_total_len * expl(-0.275 * rawscore), rawscore = 4n as
 * uint64 -> long double; QF_KARLIN / QF_LAMBDA are double literals (src/alignmentFunctions.h:1-2) */
static long double evalue_of(uint64_t n, uint64_t ylen, uint64_t db_total_len) {
    uint64_t raw_u = 4ull * n;
    long double rawscore = raw_u;
    long double t_len = (long double)ylen;
    return (long double)0.333 * t_len * db_total_len * expl(-0.275 * rawscore);
}

void imsame_build_nmin(long double min_e_value, uint64_t db_total_len, uint16_t *nmin) {
    imsame_build_nmin_upto(min_e_value, db_total_len, nmin, IMSAME_MAX_READ_SIZE);
}

/* reads longer than MAX_READ_SIZE still go through the e-value test: the reference only stops when such a
 * read reaches NW (src/alignmentFunctions.c:155), so the scan needs their thresholds too */
void imsame_build_nmin_upto(long double min_e_value, uint64_t db_total_len, uint16_t *nmin, uint64_t max_ylen) {
    const uint64_t n_max = 2ull * max_ylen + 64 < 65534 ? 2ull * max_ylen + 64 : 65534;
    for (uint64_t ylen = 0; ylen <= max_ylen; ylen++) {
        /* e is non-increasing in n: binary search for the first n with e < min */
        if (!(evalue_of(n_max, ylen, db_total_len) < min_e_value)) { nmin[ylen] = 65535; continue; }
        uint64_t lo = 0, hi = n_max; /* invariant: pass(hi) */
        while (lo < hi) {
            uint64_t mid = (lo + hi) / 2;
            if (evalue_of(mid, ylen, db_total_len) < min_e_value) hi = mid; else lo = mid + 1;
        }
        nmin[ylen] = (uint16_t)lo;
    }
}

void imsame_build_lmin(long double min_coverage, uint16_t *lmin) {
    const uint64_t len_max = 2ull * IMSAME_MAX_READ_SIZE;
    lmin[0] = 65535; /* ylen == 0 never reaches the filter */
    for (uint64_t ylen = 1; ylen <= IMSAME_MAX_READ_SIZE; ylen++) {
        uint64_t lo = 0, hi = len_max + 1;
        if (!(((long double)len_max / ylen) >= min_coverage)) { lmin[ylen] = 65535; continue; }
        hi = len_max;
        while (lo < hi) {
            uint64_t mid = (lo + hi) / 2;
            if (((long double)mid / ylen) >= min_coverage) hi = mid; else lo = mid + 1;
        }
        lmin[ylen] = (uint16_t)lo;
    }
}

void imsame_build_imin(long double min_identity, uint16_t *imin) {
    const uint64_t len_max = 2ull * IMSAME_MAX_READ_SIZE;
    imin[0] = 65535; /* 0/0 = NaN: comparison false */
    for (uint64_t len = 1; len <= len_max; len++) {
        if (!(((long double)len / len) >= min_identity)) { imin[len] = 65535; continue; }
        uint64_t lo = 0, hi = len;
        while (lo < hi) {
            uint64_t mid = (lo + hi) / 2;
            if (((long double)mid / len) >= min_identity) hi = mid; else lo = mid + 1;
        }
        imin[len] = (uint16_t)lo;
    }
}

void imsame_build_sweep_tables(int n_sets, const long double *coverage, const long double *identity, uint16_t *lmin_sets,
                               uint16_t *imin_sets, uint16_t *lmin_all, uint16_t *imin_all) {
    const uint64_t nl = IMSAME_MAX_READ_SIZE + 1, ni = 2 * IMSAME_MAX_READ_SIZE + 1;
    for (uint64_t i = 0; i < nl; i++) lmin_all[i] = 0;
    for (uint64_t i = 0; i < ni; i++) imin_all[i] = 0;
    for (int t = 0; t < n_sets; t++) {
        uint16_t *l = lmin_sets + (uint64_t)t * nl, *m = imin_sets + (uint64_t)t * ni;
        imsame_build_lmin(coverage[t], l);
        imsame_build_imin(identity[t], m);
        for (uint64_t i = 0; i < nl; i++) if (l[i] > lmin_all[i]) lmin_all[i] = l[i];
        for (uint64_t i = 0; i < ni; i++) if (m[i] > imin_all[i]) imin_all[i] = m[i];
    }
}

/* one value of a -sweep entry: a whole number as atof reads it (strtod accepts exactly what atof converts) */
static int sweep_value(const char *b, const char *e, char *text, long double *v) {
    const size_t n = (size_t)(e - b);
    if (n == 0 || n >= sizeof(((imsame_sweep_list *)0)->text[0][0])) return 0;
    memcpy(text, b, n);
    text[n] = 0;
    char *end = NULL;
    (void)strtod(text, &end);
    if (end != text + n) return 0;
    *v = (long double)atof(text); /* double first, then widened, like -coverage / -identity */
    return 1;
}

const char *imsame_parse_sweep(const char *list, imsame_sweep_list *s) {
    const char *at = list;
    s->n = 0;
    for (;;) {
        const char *comma = strchr(at, ',');
        const char *end = comma ? comma : at + strlen(at);
        const char *colon = memchr(at, ':', (size_t)(end - at));
        if (s->n == IMSAME_SWEEP_ENTRIES) return "-sweep takes at most 15 coverage:identity pairs";
        const int i = s->n;
        if (!colon || !sweep_value(at, colon, s->text[i][0], &s->coverage[i]) ||
            !sweep_value(colon + 1, end, s->text[i][1], &s->identity[i]))
            return "-sweep expects a list of coverage:identity pairs, e.g. -sweep 0.5:0.7,0.5:0.9";
        if (s->coverage[i] <= 0) return "Min-coverage must be larger than zero";
        if (s->identity[i] <= 0) return "Min-identity must be larger than zero";
        s->n++;
        if (!comma) break;
        at = comma + 1;
    }
    return NULL;
}

const char *imsame_parse_kmers(const char *list, int kmer, imsame_kmer_list *s) {
    const char *at = list;
    s->n = 0;
    for (;;) {
        const char *comma = strchr(at, ',');
        const char *end = comma ? comma : at + strlen(at);
        if (s->n == IMSAME_KMERS_ENTRIES) return "-kmers takes at most 12 seed lengths";
        long v = 0;
        const char *c = at;
        for (; c < end && *c >= '0' && *c <= '9' && c - at < 3; c++) v = 10 * v + (*c - '0');
        if (c == at || c != end) return "-kmers expects a list of seed lengths, e.g. -kmers 8,10,14";
        if (v < 4 || v > 16) return "The seed length must be between 4 and 16";
        if (v == kmer) return "-kmers must not repeat a seed length or give the -kmer one";
        for (int i = 0; i < s->n; i++)
            if (s->k[i] == v) return "-kmers must not repeat a seed length or give the -kmer one";
        s->k[s->n++] = (int)v;
        if (!comma) break;
        at = comma + 1;
    }
    return NULL;
}
