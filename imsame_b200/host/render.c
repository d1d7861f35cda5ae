/*
 * render.c -- record header and alignment text, from the device traceback.
 *
 * The reference renders inside build_alignment (src/alignmentFunctions.c:230-271)
 * from two right-aligned scratch strands filled by backtrackingNW (:493-560).
 * Here the path arrives as run-length ops (csrc/traceback.cuh) and the same
 * text is produced directly:
 *   - strands, left to right: left overhang (:548-556: dashes on the strand that
 *     still has bases before the end cell, spaces on the other), the path, then
 *     one '-' per base after the best cell on each strand (:503-504);
 *   - a diagonal step prints X[x] over Y[y]; a column jump prints the skipped
 *     bases of X over '-', a row jump '-' over the skipped bases of Y (:514-543);
 *   - blocks of ALIGN_LEN = 60 columns: X line, Y line, marker line ('*' where
 *     both strands hold the same base), repeated while BOTH strands have
 *     columns left (:233), then one empty line (:270).
 */
#include "imsame_host.h"
#include <string.h>

#define OP_TYPE(o) ((o) >> 28)
#define OP_COUNT(o) ((o) & 0x0FFFFFFFu)

int imsame_format_header(char *dst, uint64_t read, uint64_t db_seq, uint32_t length, uint32_t identities,
                         uint64_t ylen) {
    /* src/alignmentFunctions.c:167: integer percentages, clamped to 100 */
    uint64_t pi = 100ull * identities / length, pc = 100ull * length / ylen;
    return sprintf(dst, "(%llu, %llu) : %d%% %d%% %llu\n $$$$$$$ \n", (unsigned long long)read,
                   (unsigned long long)db_seq, (int)(pi > 100 ? 100 : pi), (int)(pc > 100 ? 100 : pc),
                   (unsigned long long)ylen);
}

size_t imsame_format_cigar_columns(char *dst, const imsame_aln *a, const uint32_t *ops, uint64_t n_ops) {
    /* dst holds the header of imsame_format_header, "...\n $$$$$$$ \n": the columns go before its first newline */
    static const char tail[] = "\n $$$$$$$ \n";
    const size_t lt = sizeof tail - 1;
    char *w = dst - lt;
    w += sprintf(w, " %u %u %u %u %d ", a->q_start, a->q_end, a->db_start, a->db_end, a->score);
    for (uint64_t k = 0; k < n_ops; k++) w += sprintf(w, "%u%c", ops[k] >> 4, "MIDNSHP=X"[ops[k] & 15]);
    memcpy(w, tail, lt + 1);
    return (size_t)(w + lt - dst);
}

uint64_t imsame_render_alignment(char *dst, const unsigned char *X, uint32_t xlen, const unsigned char *Y,
                                 uint32_t ylen, uint32_t bx, uint32_t by, const uint32_t *ops, uint64_t n_ops) {
    /* path length and end cell */
    uint64_t ncol = 0;
    uint32_t x = bx, y = by;
    for (uint64_t k = 0; k < n_ops; k++) {
        const uint32_t c = OP_COUNT(ops[k]);
        ncol += c;
        switch (OP_TYPE(ops[k])) {
            case 1: x -= c; y -= c; break;
            case 2: x -= c; y -= 1; break;
            default: y -= c; x -= 1; break;
        }
    }
    const uint32_t lead = x > y ? x : y;
    const uint64_t tx = xlen - 1 - bx, ty = ylen - 1 - by;
    const uint64_t Lx = lead + ncol + tx, Ly = lead + ncol + ty;
    /* strands are built at the tail of dst's own space: caller gives 4*(xlen+ylen)+256 bytes,
       text needs at most 3*(max(Lx,Ly)) + blocks*3 + 2; use separate stack-free buffers */
    char *sx = dst + 0, *sy;
    /* layout: [text ........][sx Lx][sy Ly] -- text grows from dst, strands live behind it */
    const uint64_t text_cap = 3 * (Lx > Ly ? Lx : Ly) + 3 * ((Lx > Ly ? Lx : Ly) / 60 + 2) + 8;
    sx = dst + text_cap;
    sy = sx + Lx + 1;
    memset(sx, x >= y ? '-' : ' ', lead);
    memset(sy, x >= y ? ' ' : '-', lead);
    /* path, written right to left */
    uint64_t at = lead + ncol;
    uint32_t px = bx, py = by;
    for (uint64_t k = 0; k < n_ops; k++) {
        const uint32_t c = OP_COUNT(ops[k]);
        switch (OP_TYPE(ops[k])) {
            case 1:
                for (uint32_t t = 0; t < c; t++) { at--; sx[at] = (char)X[px--]; sy[at] = (char)Y[py--]; }
                break;
            case 2:
                for (uint32_t t = 0; t < c; t++) { at--; sx[at] = (char)X[px--]; sy[at] = '-'; }
                py -= 1;
                break;
            default:
                for (uint32_t t = 0; t < c; t++) { at--; sx[at] = '-'; sy[at] = (char)Y[py--]; }
                px -= 1;
                break;
        }
    }
    memset(sx + lead + ncol, '-', tx);
    memset(sy + lead + ncol, '-', ty);
    /* blocks */
    uint64_t w = 0, i = 0, j = 0;
    while (i < Lx && j < Ly) {
        const uint64_t bi = i, bj = j;
        const uint64_t nx = Lx - i < 60 ? Lx - i : 60, ny = Ly - j < 60 ? Ly - j : 60;
        memcpy(dst + w, sx + i, nx); w += nx; i += nx;
        dst[w++] = '\n';
        memcpy(dst + w, sy + j, ny); w += ny; j += ny;
        dst[w++] = '\n';
        for (uint64_t t = 0; t < nx; t++) {
            const char a = sx[bi + t];
            const int star = a != '-' && bj + t < Ly && sy[bj + t] != '-' && a == sy[bj + t];
            dst[w++] = star ? '*' : ' ';
        }
        dst[w++] = '\n';
    }
    dst[w++] = '\n';
    dst[w] = 0;
    return w;
}
