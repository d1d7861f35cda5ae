// nw_core.cuh -- one wavefront step of the reference's full-matrix NW with
// lagged affine gaps (src/alignmentFunctions.c:389-489) plus forward-carried
// traceback statistics (length/identities of :493-560 and :254-258), written as
// a host/device function so the exact lane logic is unit-tested on the CPU
// (tests/emul/nw_emul.cpp, tb_emul.cpp) and executed unchanged by the CUDA
// kernel (nw.cuh).
//
// Geometry: X = database read (rows i), Y = query read (columns j).  A lane owns
// S consecutive columns j0..j0+S-1 of one row per step; lane l works on row
// i = t - l + 1 at step t (anti-diagonal wavefront over lane strips).  Cell
// (i,j) needs T[i-1][j-1], T[i][j-2], T[i-1][j-2], T[i-2][j-1] and the running
// maxima mf (per row) and mc[j-1] (per column), so everything a lane needs from
// its left neighbour was produced one step earlier (NwLink).
//
// Per-cell recurrence (names as in the reference):
//   if (j>1 && mf.score <= T[i][j-2]) mf = (T[i-1][j-2], y=j-2)              :434-438
//   D = T[i-1][j-1];  L = mf.score + iGap + (j-(mf.y+1))*eGap   (j>1)         :441-447
//   R = mc[j-1].score + iGap + (i-(mc[j-1].x+1))*eGap            (i>1)         :449-453
//   D>=L && D>=R -> D ; else R>L -> R ; else L ; then + (X[i]==Y[j] ? 4 : -4)  :440,457-472
//   if (i>1 && j>1 && T[i-2][j-1] > mc[j-1].score) mc[j-1] = (T[i-2][j-1], x=i-2)   :476-480
// The match score is added to all three candidates, so the choice is made on
// the values without it:  T = max3(D,L,R) + s,  diagonal <=> max3 == D,
// otherwise R <=> R > L.
//
// Statistics word of a cell p = (length << 16) | (8 * identities) of the cell's
// own traceback path: diagonal -> +1 column and +1 identity on match, i.e.
// p + 65540 + s with s = +-4;  jump to (px,py) -> + max(i-px, j-py) columns
// (src/alignmentFunctions.c:514-543).  length <= 6000 and 8*identities <= 24000
// keep both fields inside their 16 bits.
//
// Register layout: two row histories (T[i-1], T[i-2] and their statistics) that
// swap roles every step (the caller alternates them by step parity), so no value
// is ever moved between rows: the new row is written over the T[i-2] slots as
// they are consumed.
#pragma once
#include "common.cuh"

namespace imsame {

constexpr int NW_NEG = -(1 << 28);   // "-inf" that survives a handful of additions
constexpr int NW_POINT = 4;          // POINT, src/structs.h:13
constexpr int NW_STAT_LEN1 = 65536;  // one alignment column
constexpr int NW_STAT_DIAG = NW_STAT_LEN1 + NW_POINT;  // diagonal step: p + NW_STAT_DIAG + s  (s = +-4)

IMS_HD uint32_t nw_stat_len(int p) { return (uint32_t)p >> 16; }
IMS_HD uint32_t nw_stat_ids(int p) { return ((uint32_t)p & 0xFFFFu) >> 3; }

struct NwLink {
    int a, ap;          // T[i][j0-1] and its statistics
    int b, bp;          // T[i][j0-2] and its statistics
    int mfs, mfy, mfp;  // row maximum after cell (i, j0-1): score, column, statistics
};

struct NwBest {
    int s, i, j, p;  // score, row, column, statistics of the best border cell
};

// "last in row-major order among equal scores" (src/alignmentFunctions.c:483 uses >=)
IMS_HD bool best_better(const NwBest &c, const NwBest &b) {
    if (c.s != b.s) return c.s > b.s;
    if (c.i != b.i) return c.i > b.i;
    return c.j > b.j;
}

// one row of a lane's strip plus its two left halo columns
template <int S>
struct NwRow {
    int h[S + 1], p[S + 1];  // T[.][j0-1+k] and statistics, k = 0..S (k = 0: left halo column)
    int g, gp;               // T[.][j0-2]
};

template <int S>
struct NwLane {
    NwRow<S> r0, r1;             // row histories: at step t, r[t&1] is T[i-1] and r[~t&1] is T[i-2]
    int mcs[S], mcx[S], mcp[S];  // column maximum of column j0-1+k: score, row, statistics
    NwBest best;
};

IMS_HD int max3i(int a, int b, int c) {
#if defined(__CUDA_ARCH__)
    return __vimax3_s32(a, b, c);
#else
    const int m = a > b ? a : b;
    return m > c ? m : c;
#endif
}

// Row 0 (src/alignmentFunctions.c:404-413): T[0][j] = +-4, mc[j] = (T[0][j], x=0).
// ypk_halo: 2-bit codes of Y[j0-2], Y[j0-1], Y[j0] .. Y[j0+S-1] at bits 0,2,4,...
// first_lane: the lane that owns column 1 (its halo is column 0, which has no
// left neighbour and whose column maximum is never updated, guard j>1 at :476).
// t_first = step at which this lane processes row 1: row 0 goes into r[t_first & 1].
template <int S>
IMS_HD void nw_lane_init(NwLane<S> &L, uint32_t x0, uint64_t ypk_halo, bool first_lane, int t_first) {
    const bool odd = (t_first & 1) != 0;
#pragma unroll
    for (int k = 0; k <= S; k++) {
        const uint32_t y = (uint32_t)(ypk_halo >> (2 * (k + 1))) & 3u;
        const int row0 = (y == x0) ? NW_POINT : -NW_POINT;
        // the other history is "row -1": the first column-maximum test must fail (guard i>1 at :476)
        L.r0.h[k] = odd ? NW_NEG : row0;
        L.r1.h[k] = odd ? row0 : NW_NEG;
        L.r0.p[k] = 0;
        L.r1.p[k] = 0;
        if (k < S) {
            L.mcs[k] = row0;
            L.mcx[k] = 0;
            L.mcp[k] = 0;
        }
    }
    const uint32_t yg = (uint32_t)ypk_halo & 3u;
    const int g0 = first_lane ? NW_NEG : ((yg == x0) ? NW_POINT : -NW_POINT);
    L.r0.g = odd ? NW_NEG : g0;
    L.r1.g = odd ? g0 : NW_NEG;
    L.r0.gp = L.r1.gp = 0;
    L.best.s = NW_NEG * 2;
    L.best.i = L.best.j = L.best.p = 0;
}

// What the lane owning column 1 receives instead of a neighbour's link: column 0
// is T[i][0] = +-4 (:426); the row maximum starts as "-inf" so that L is -inf at
// j = 1 (:446) and the j = 2 test (:434, always true in the reference because
// mf.score == T[i][0]) always fires and installs (T[i-1][0], y = 0).
IMS_HD NwLink nw_first_link(uint32_t xi, uint32_t y0) {
    NwLink k;
    k.a = (xi == y0) ? NW_POINT : -NW_POINT;
    k.ap = 0;
    k.b = NW_NEG - 1;
    k.bp = 0;
    k.mfs = NW_NEG;
    k.mfy = 0;
    k.mfp = 0;
    return k;
}

// TB = 1: additionally store one back-pointer code per cell for the winners-only traceback
// (src/alignmentFunctions.c:459-471 xfrom/yfrom): 0 = diagonal, 0x8000|x = jump to the
// column maximum (x, j-1), 0x4000|y = jump to the row maximum (i-1, y).
constexpr uint16_t TB_DIAG = 0, TB_COL = 0x8000, TB_ROW = 0x4000, TB_MASK = 0x3FFF;
// TB = 2 (cigar.cuh): four bits per cell instead, the S cells of the strip in one 32-bit word (cell c at bits 4c):
// the choice (0 = diagonal, 1 = jump to the column maximum, 2 = jump to the row maximum) and whether the cell moved
// the row maximum to column j-2 (:434-438) or the maximum of column j-1 to row i-2 (:476-480).  The jump targets are
// where those bits were last set, so the walk finds them again without storing them.
constexpr uint32_t TBN_DIAG = 0, TBN_COL = 1, TBN_ROW = 2, TBN_DIR = 3, TBN_UP = 4, TBN_UC = 8;

// One row of the lane's strip.
//   P1 = T[i-1] (read only), P2 = T[i-2] on entry, T[i] on exit (written in place)
//   mm: bit 2c set <=> X[i] != Y[j0+c]
//   X1 = xlen-1, Y1 = ylen-1 (last row / column)
//   cl: slot of column Y1 inside a strip ((Y1 - 1 - jb) % S, the same for every lane);
//   owns_last: this lane's strip holds column Y1.
// Columns j > Y1 are padding: they only ever feed cells further right, never a real one.
//   tbrow: TB = 1: the row's S codes (uint16_t); TB = 2: the row's 32-bit word of 4-bit codes (S <= 8)
template <int S, int TB = 0>
IMS_HD void nw_row(NwLane<S> &L, const NwRow<S> &P1, NwRow<S> &P2, const NwLink &in, NwLink &out, int i, int j0,
                   uint32_t mm, int igap, int egap, int X1, int Y1, int cl, bool owns_last, bool first_lane,
                   void *tbrow = nullptr) {
    const int lb = igap - egap;                        // L = mfs + (j - mfy) * egap + lb
    const int rb = ((i == 1) ? NW_NEG : igap) - egap;  // no R candidate on row 1 (:449)
    int mfs = in.mfs, mfy = in.mfy, mfp = in.mfp;
    int nt = in.a, np = in.ap;   // value that becomes slot c of the new row: T[i][j0-1+c]
    int t2 = in.b;               // T[i][j-2]
    int r2 = P1.g, rp2 = P1.gp;  // T[i-1][j-2]
    uint32_t tbw[4] = {0u, 0u, 0u, 0u};  // TB = 1, S = 8: the row's codes, two per word
    uint32_t nib = 0u;                   // TB = 2: the row's 4-bit codes
#pragma unroll
    for (int c = 0; c < S; c++) {
        const int j = j0 + c;
        // consume T[i-2][j-1], then store T[i][j-1] in its place
        int o2 = P2.h[c];
        const int o2p = P2.p[c];
        if (c == 0) o2 = first_lane ? NW_NEG : o2;  // column 0's maximum is never updated (:476, j>1)
        P2.h[c] = nt;
        P2.p[c] = np;
        // row maximum: tests row i, copies row i-1 (:434-438)
        const bool up = mfs <= t2;
        mfs = up ? r2 : mfs;
        mfy = up ? j - 2 : mfy;
        mfp = up ? rp2 : mfp;
        const bool mis = ((mm >> (2 * c)) & 1u) != 0;
        const int s = mis ? -NW_POINT : NW_POINT;
        const int d = P1.h[c];
        const int dl = j - mfy;
        const int l = mfs + (dl * egap + lb);
        const int dr = i - L.mcx[c];
        const int r = L.mcs[c] + (dr * egap + rb);
        const int pd = P1.p[c] + s + NW_STAT_DIAG;
        const int pl = dl * NW_STAT_LEN1 + mfp;
        const int pr = dr * NW_STAT_LEN1 + L.mcp[c];
        const int m = max3i(d, l, r);
        const bool is_d = (m == d);
        const bool is_r = r > l;
        const int pj = is_r ? pr : pl;
        if (TB == 1) {
            const uint32_t code = is_d ? TB_DIAG : (is_r ? (uint32_t)(TB_COL | L.mcx[c]) : (uint32_t)(TB_ROW | mfy));
            // S = 8 (the only strip width the traceback launches): the row's eight codes leave as ONE 16-byte store
            // (tbrow is 16-byte aligned: strips start at multiples of 8 columns, rows at multiples of 256); as eight
            // 2-byte stores from 32 lanes on 32 different rows every store instruction touched 32 sectors
            if (S == 8) { if (c & 1) tbw[c >> 1] |= code << 16; else tbw[c >> 1] = code; }
            else static_cast<uint16_t *>(tbrow)[c] = (uint16_t)code;
        }
        // column maximum of column j-1 absorbs T[i-2][j-1], strictly greater only (:476-480)
        const bool uc = o2 > L.mcs[c];
        if (TB == 2)
            nib |= ((is_d ? TBN_DIAG : (is_r ? TBN_COL : TBN_ROW)) | (up ? TBN_UP : 0u) | (uc ? TBN_UC : 0u)) << (4 * c);
        L.mcs[c] = uc ? o2 : L.mcs[c];
        L.mcx[c] = uc ? i - 2 : L.mcx[c];
        L.mcp[c] = uc ? o2p : L.mcp[c];
        // next column
        t2 = nt;
        r2 = d;
        rp2 = P1.p[c];
        nt = m + s;
        np = is_d ? pd : pj;
    }
    if (TB == 1 && S == 8) {
#if defined(__CUDA_ARCH__)
        *reinterpret_cast<uint4 *>(tbrow) = make_uint4(tbw[0], tbw[1], tbw[2], tbw[3]);
#else
        for (int c = 0; c < 8; c++) static_cast<uint16_t *>(tbrow)[c] = (uint16_t)(tbw[c >> 1] >> (16 * (c & 1)));
#endif
    }
    if (TB == 2) *static_cast<uint32_t *>(tbrow) = nib;
    P2.h[S] = nt;
    P2.p[S] = np;
    P2.g = in.b;
    P2.gp = in.bp;
    // hand-over to the right neighbour: T[i][j0+S-1], T[i][j0+S-2]
    out.a = nt;
    out.ap = np;
    out.b = t2;
    out.bp = P2.p[S - 1];
    out.mfs = mfs;
    out.mfy = mfy;
    out.mfp = mfp;
    // best border cell (:481-484): every column of the last row, the last column of every row.
    // The new row sits in P2.h[1..S]; cl is warp-uniform, so this is one uniform switch per step.
    if (i == X1) {
#pragma unroll
        for (int c = 0; c < S; c++)
            if (j0 + c <= Y1 && P2.h[c + 1] >= L.best.s) {
                L.best.s = P2.h[c + 1]; L.best.i = i; L.best.j = j0 + c; L.best.p = P2.p[c + 1];
            }
    } else if (owns_last) {
        int lt = P2.h[S], lp = P2.p[S];
        switch (cl) {
#define IMS_CASE(C)                                        \
    case C:                                                \
        if (C < S) { lt = P2.h[(C < S ? C : 0) + 1]; lp = P2.p[(C < S ? C : 0) + 1]; } \
        break;
            IMS_CASE(0) IMS_CASE(1) IMS_CASE(2) IMS_CASE(3) IMS_CASE(4) IMS_CASE(5) IMS_CASE(6)
#undef IMS_CASE
            default: break;
        }
        if (lt >= L.best.s) { L.best.s = lt; L.best.i = i; L.best.j = Y1; L.best.p = lp; }
    }
}

}  // namespace imsame
