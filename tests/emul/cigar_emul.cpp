// CPU emulation of K5 (cigar.cuh): the wavefront with 4-bit codes in the kernel's step-major layout (nw_core.cuh,
// TB = 2) -> cg_walk, stepped as a 32-lane warp.  Checked against the oracle's forward NW (score, best cell, length,
// identities) and against the 16-bit back-pointer path of the winners' traceback (nw_row TB = 1 -> tb_walk, itself
// pinned to the reference's text by tb_emul): the same path, op for op.  The CIGAR is replayed over the two reads:
// score, counts, coordinates, and the record's length / identities by the documented rule.
//   usage: cigar_emul <n_cases> <seed> [long_len]
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include "../../imsame_b200/csrc/cigar.cuh"
#include "../../imsame_b200/csrc/traceback.cuh"
extern "C" {
#include "../../oracle/imsame_oracle.h"
}
using namespace imsame;
static uint64_t rng_state;
static uint64_t rnd() { uint64_t z = (rng_state += 0x9E3779B97F4A7C15ull); z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27)) * 0x94D049BB133111EBull; return z ^ (z >> 31); }
static inline uint32_t code(unsigned char c) { return (c >> 1) & 3; }

// the kernel's warp, lanes in any order that respects the hand-over; both code forms written in one sweep
static NwBest run_pair(const unsigned char *X, int xlen, const unsigned char *Y, int ylen, int igap, int egap,
                       std::vector<uint32_t> &nib, std::vector<uint16_t> &tb, uint32_t &stride) {
    constexpr int S = CG_S;
    const int X1 = xlen - 1, Y1 = ylen - 1;
    nib.assign(cg_words(X1, Y1), 0xFFFFFFFFu);
    stride = tb_stride(ylen, S);
    tb.assign((size_t)X1 * stride + 64, 0xFFFF);
    std::vector<NwLink> carry(xlen + 1), carry_next(xlen + 1);
    NwBest best; best.s = NW_NEG * 2; best.i = best.j = best.p = 0;
    int pass = 0;
    for (int jb = 0; jb < Y1; jb += 32 * S, pass++) {
        int nl = (Y1 - jb + S - 1) / S; if (nl > 32) nl = 32;
        static NwLane<S> lanes[32], lanes2[32];
        NwLink outs[32];
        for (int l = 0; l < nl; l++) {
            int j0 = jb + l * S + 1;
            uint64_t halo = 0;
            for (int k = 0; k < S + 2; k++) { int j = j0 - 2 + k; uint64_t c = (j >= 0 && j < ylen) ? code(Y[j]) : 0; halo |= c << (2 * k); }
            nw_lane_init<S>(lanes[l], code(X[0]), halo, jb == 0 && l == 0, l);
            lanes2[l] = lanes[l];
        }
        for (int t = 0; t <= X1 + nl - 2; t++)
            for (int l = nl - 1; l >= 0; l--) {
                int i = t - l + 1;
                if (i < 1 || i > X1) continue;
                int j0 = jb + l * S + 1;
                NwLink in = (l == 0) ? (jb == 0 ? nw_first_link(code(X[i]), code(Y[0])) : carry[i]) : outs[l - 1];
                uint32_t mm = 0;
                for (int c = 0; c < S; c++) { int j = j0 + c; uint32_t y = j < ylen ? code(Y[j]) : 0; if (y != code(X[i])) mm |= 1u << (2 * c); }
                NwLink out, out2;
                const int cl = (Y1 - 1 - jb) % S; const bool owns = Y1 >= j0 && Y1 < j0 + S;
                uint32_t *w = nib.data() + ((uint64_t)pass * (X1 + 31) + t) * 32 + l;
                uint16_t *tbr = tb.data() + (size_t)(i - 1) * stride + (j0 - 1);
                if (t & 1) {
                    nw_row<S, 2>(lanes[l], lanes[l].r1, lanes[l].r0, in, out, i, j0, mm, igap, egap, X1, Y1, cl, owns, jb == 0 && l == 0, w);
                    nw_row<S, 1>(lanes2[l], lanes2[l].r1, lanes2[l].r0, in, out2, i, j0, mm, igap, egap, X1, Y1, cl, owns, jb == 0 && l == 0, tbr);
                } else {
                    nw_row<S, 2>(lanes[l], lanes[l].r0, lanes[l].r1, in, out, i, j0, mm, igap, egap, X1, Y1, cl, owns, jb == 0 && l == 0, w);
                    nw_row<S, 1>(lanes2[l], lanes2[l].r0, lanes2[l].r1, in, out2, i, j0, mm, igap, egap, X1, Y1, cl, owns, jb == 0 && l == 0, tbr);
                }
                outs[l] = out;
                if (l == 31) carry_next[i] = out;
            }
        for (int l = 0; l < nl; l++) if (best_better(lanes[l].best, best)) best = lanes[l].best;
        carry.swap(carry_next);
    }
    return best;
}

static std::string cigar_text(const uint32_t *ops, uint32_t n) {
    std::string s;
    for (uint32_t k = 0; k < n; k++) s += std::to_string(ops[k] >> 4) + "?MIDNSHP=X"[1 + (ops[k] & 15)];
    return s;
}

int main(int argc, char **argv) {
    int n = argc > 1 ? atoi(argv[1]) : 200; rng_state = argc > 2 ? strtoull(argv[2], 0, 10) : 1;
    const int long_x = argc > 3 ? atoi(argv[3]) : 700, long_y = argc > 3 ? atoi(argv[3]) : 900;
    const char B[4] = {'A', 'C', 'G', 'T'};
    int bad = 0;
    for (int it = 0; it < n; it++) {
        int xlen = 12 + rnd() % (it % 7 == 0 ? long_x : 300), ylen = 11 + rnd() % (it % 5 == 0 ? long_y : 300);
        if (it % 11 == 0) { xlen = 250; ylen = 250; }
        if (it % 13 == 0) xlen = 2 + rnd() % 6;
        if (it % 17 == 0) ylen = 2 + rnd() % 6;
        std::vector<unsigned char> X(xlen), Y(ylen);
        for (auto &c : X) c = B[rnd() & 3];
        int mode = it % 19 == 0 ? 4 : rnd() % 4;
        if (mode == 4) { ylen = xlen; Y = X; }  // identical reads
        else if (mode == 0) for (auto &c : Y) c = B[rnd() & 3];
        else {
            int off = (int)(rnd() % (xlen)) - xlen / 3; double pe = (mode == 1) ? 0.03 : (mode == 2 ? 0.15 : 0.30);
            int src = off;
            for (int j = 0; j < ylen; j++) {
                double u = (rnd() >> 11) * (1.0 / 9007199254740992.0);
                if (u < pe / 6) src += 1 + rnd() % 4;
                if (u > 1 - pe / 6) { Y[j] = B[rnd() & 3]; continue; }
                unsigned char c = (src >= 0 && src < xlen) ? X[src] : B[rnd() & 3];
                if (u > 0.5 && u < 0.5 + pe) c = B[rnd() & 3];
                Y[j] = c; src++;
            }
        }
        int igap = -(int)(rnd() % 8), egap = -(int)(rnd() % 4);
        if (it % 3 == 0) { igap = -5; egap = -2; }
        if (it % 23 == 0) { igap = 2; egap = 1; }  // positive gap scores: the path model holds for any sign
        int32_t os; uint32_t obx, oby, olen, oid;
        orc_nw_forward(X.data(), xlen, Y.data(), ylen, igap, egap, &os, &obx, &oby, &olen, &oid);
        std::vector<uint32_t> nib; std::vector<uint16_t> tb; uint32_t stride;
        NwBest b = run_pair(X.data(), xlen, Y.data(), ylen, igap, egap, nib, tb, stride);
        std::vector<uint32_t> ops(xlen + ylen), tops(xlen + ylen + 4);
        HitAln h;
        uint32_t nops = cg_walk(nib.data(), xlen - 1, (uint32_t)b.i, (uint32_t)b.j,
                                [&](uint32_t i) { return code(X[i]); }, [&](uint32_t j) { return code(Y[j]); }, ops.data(), h);
        // the 16-bit path in CIGAR form: every step ends on an aligned column; a jump over c rows / columns skips c - 1
        uint32_t ex, ey;
        const uint32_t tn = tb_walk(tb.data(), stride, (uint32_t)b.i, (uint32_t)b.j, tops.data(), &ex, &ey);
        std::vector<char> cols;  // walk order
        {
            uint32_t x = b.i, y = b.j;
            cols.push_back(X[x] == Y[y] ? '=' : 'X');
            for (uint32_t k = 0; k < tn; k++) {
                const uint32_t c = tops[k] & OP_COUNT_MASK;
                if ((tops[k] & ~OP_COUNT_MASK) == OP_DIAG) {
                    for (uint32_t s = 0; s < c; s++) { x--; y--; cols.push_back(X[x] == Y[y] ? '=' : 'X'); }
                } else if ((tops[k] & ~OP_COUNT_MASK) == OP_COL) {
                    for (uint32_t s = 1; s < c; s++) cols.push_back('D');
                    x -= c; y -= 1; cols.push_back(X[x] == Y[y] ? '=' : 'X');
                } else {
                    for (uint32_t s = 1; s < c; s++) cols.push_back('I');
                    y -= c; x -= 1; cols.push_back(X[x] == Y[y] ? '=' : 'X');
                }
            }
        }
        std::string want;
        for (size_t k = cols.size(); k > 0;) {
            size_t e = k; char c = cols[k - 1];
            while (k > 0 && cols[k - 1] == c) k--;
            want += std::to_string(e - k) + c;
        }
        // replay over the two reads
        int64_t score = 0; uint32_t x = h.db_start, y = h.q_start, mt = 0, mmc = 0, gaps = 0, ncols = 0, ids = 0;
        bool after_gap = false, first = true, ok_walk = true;
        for (uint32_t k = 0; k < nops; k++) {
            const uint32_t len = ops[k] >> 4, op = ops[k] & 15;
            if (op == CIGAR_I || op == CIGAR_D) {
                score += igap + (int64_t)len * egap; gaps += len; ncols += len; after_gap = true;
                if (op == CIGAR_I) y += len; else x += len;
                continue;
            }
            for (uint32_t s = 0; s < len; s++, x++, y++, ncols++) {
                const bool eq = X[x] == Y[y];
                if (eq != (op == CIGAR_EQ)) ok_walk = false;
                score += eq ? NW_POINT : -NW_POINT;
                if (eq) { mt++; if (!first && !after_gap) ids++; } else mmc++;
                first = after_gap = false;
            }
        }
        const bool ok = b.s == os && (uint32_t)b.i == obx && (uint32_t)b.j == oby && nw_stat_len(b.p) == olen &&
                        nw_stat_ids(b.p) == oid && ok_walk && cigar_text(ops.data(), nops) == want && score == b.s &&
                        x == h.db_end && y == h.q_end && h.db_end == obx + 1 && h.q_end == oby + 1 && h.db_start == ex &&
                        h.q_start == ey && (h.db_start == 0 || h.q_start == 0) && mt == h.matches && mmc == h.mismatches &&
                        gaps == h.gap_cols && ncols - 1 == olen && ids == oid && nops <= (uint32_t)(xlen + ylen);
        if (!ok) {
            bad++;
            if (bad < 5) printf("MISMATCH it=%d xlen=%d ylen=%d gaps %d %d: score %d/%d/%lld cell %d,%d/%u,%u len %u/%u ids %u/%u\n  got  %s\n  want %s\n",
                                it, xlen, ylen, igap, egap, b.s, os, (long long)score, b.i, b.j, obx, oby, ncols - 1, olen, ids, oid,
                                cigar_text(ops.data(), nops).c_str(), want.c_str());
        }
    }
    printf("%d cases, %d mismatches\n", n, bad);
    return bad != 0;
}
