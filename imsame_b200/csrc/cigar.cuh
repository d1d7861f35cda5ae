// cigar.cuh -- K5: the alignment of every accepted hit as a CIGAR with exact coordinates
// (imsame_gpu_align_traceback).
//
// One warp per hit recomputes the pair's NW with the forward kernel's own row function (nw_core.cuh: nw_row, TB = 2)
// over the whole matrix -- the reference's NW has no band: its window is the database read x the query read -- and
// keeps 4 bits per cell: the choice made there, and whether the cell moved the row maximum or a column maximum.
// Lane 0 then walks back from the best border cell, which the same warp reduction as the forward kernel picks, to
// row 0 or column 0, and the warp leaves the path as run-length CIGAR operations.
//
// Tie-breaking is the forward kernel's, because the values and choices ARE the forward kernel's:
//   - a cell takes the diagonal if D >= L and D >= R, else the column jump (R) if R > L, else the row jump (L);
//   - the row maximum moves to T[i-1][j-2] when its score is <= T[i][j-2] (the latest column wins a tie), the
//     maximum of column j-1 moves to T[i-2][j-1] only when strictly greater (the earliest row wins);
//   - the best border cell (last row or last column) is the highest score, the last in row-major order on a tie.
// A CPU NW with these rules gives the same CIGAR; another optimal path can give another CIGAR of the same score.
//
// What the path means (it is what the score adds up):
//   - the start cell (x0, y0) on row 0 or column 0 is an aligned column: T[x0][y0] = +-4;
//   - a diagonal step to (i, j) aligns X[i] with Y[j] (+-4);
//   - a jump from the column maximum (x, j-1) to (i, j) skips X[x+1 .. i-1] (a deletion of g = i-x-1 >= 1
//     database bases: igap + g * egap) and aligns X[i] with Y[j] (+-4); a jump from the row maximum (i-1, y) skips
//     Y[y+1 .. j-1] (an insertion of g = j-y-1 >= 1 query bases) likewise.
// So score = 4 * (=) - 4 * (X) + sum over gap runs (igap + length * egap).  The record's length and identities
// (the reference's traceback text, src/alignmentFunctions.c:493-546) count the columns and the matches of that
// path without its start column, and without the matches of the aligned column that ends each gap (the reference
// prints such a jump as gap columns only): length = columns - 1.
#pragma once
#include "nw.cuh"

namespace imsame {

// BAM operation codes, op word = length << 4 | op
constexpr uint32_t CIGAR_I = 1, CIGAR_D = 2, CIGAR_EQ = 7, CIGAR_X = 8;

// == imsame_aln (include/imsame_gpu.h)
struct HitAln {
    int32_t score;
    uint32_t q_start, q_end, db_start, db_end;  // [start, end) inside the two reads
    uint32_t matches, mismatches, gap_cols;
};

constexpr int CG_S = 8;  // columns per lane: a row of a strip is one 32-bit word of 4-bit codes

// Code words of a hit: pass p (columns 256p+1 .. 256p+256) holds one word per (step, lane) in step order, so that
// the 32 lanes of a step store 128 contiguous bytes; lane l works on row i at step t = i - 1 + l.  Every pass but
// the last has 32 lanes and X1 + 31 steps.
IMS_HD uint64_t cg_words(uint32_t X1, uint32_t Y1) {
    const uint32_t passes = (Y1 + 32 * CG_S - 1) / (32 * CG_S), last = Y1 - (passes - 1) * 32 * CG_S;
    const uint32_t nl = (last + CG_S - 1) / CG_S;
    return ((uint64_t)(passes - 1) * (X1 + 31) + (X1 + nl - 1)) * 32;
}
IMS_HD uint32_t cg_code(const uint32_t *codes, uint32_t X1, uint32_t i, uint32_t j) {
    const uint32_t jj = j - 1, p = jj / (32 * CG_S), l = (jj % (32 * CG_S)) / CG_S, c = jj % CG_S;
    return (codes[((uint64_t)p * (X1 + 31) + (i - 1 + l)) * 32 + l] >> (4 * c)) & 15u;
}

// Walk from the best cell (bx, by) back to row 0 / column 0; xc(i), yc(j): 2-bit base codes.  Writes the ops in
// alignment order (at most xlen + ylen) and the coordinates and counts of h; returns the number of ops.
template <class XC, class YC>
IMS_HD uint32_t cg_walk(const uint32_t *codes, uint32_t X1, uint32_t bx, uint32_t by, XC xc, YC yc, uint32_t *ops,
                        HitAln &h) {
    uint32_t n = 0, op = 0, len = 0, x = bx, y = by;
    h.matches = h.mismatches = h.gap_cols = 0;
    auto put = [&](uint32_t o, uint32_t k) {
        if (len && o == op) { len += k; return; }
        if (len) ops[n++] = len << 4 | op;
        op = o;
        len = k;
    };
    auto column = [&](uint32_t i, uint32_t j) {
        const bool eq = xc(i) == yc(j);
        if (eq) h.matches++; else h.mismatches++;
        put(eq ? CIGAR_EQ : CIGAR_X, 1);
    };
    column(x, y);
    while (x > 0 && y > 0) {
        const uint32_t d = cg_code(codes, X1, x, y) & TBN_DIR;
        if (d == TBN_DIAG) {
            x--;
            y--;
        } else if (d == TBN_COL) {
            // the maximum of column y-1 that cell (x, y) saw: row u-2 of the latest row u < x that raised it, else row 0
            uint32_t u = x - 1;
            while (u >= 2 && !(cg_code(codes, X1, u, y) & TBN_UC)) u--;
            const uint32_t ux = u >= 2 ? u - 2 : 0;
            put(CIGAR_D, x - ux - 1);
            h.gap_cols += x - ux - 1;
            x = ux;
            y--;
        } else {
            // the row maximum that cell (x, y) saw: column v-2 of the latest column v <= y that raised it
            uint32_t v = y;
            while (v >= 2 && !(cg_code(codes, X1, x, v) & TBN_UP)) v--;
            const uint32_t uy = v >= 2 ? v - 2 : 0;
            put(CIGAR_I, y - uy - 1);
            h.gap_cols += y - uy - 1;
            x--;
            y = uy;
        }
        column(x, y);
    }
    if (len) ops[n++] = len << 4 | op;
    for (uint32_t a = 0, b = n - 1; a < b; a++, b--) {  // walk order -> alignment order
        const uint32_t t = ops[a];
        ops[a] = ops[b];
        ops[b] = t;
    }
    h.db_start = x;
    h.q_start = y;
    h.db_end = bx + 1;
    h.q_end = by + 1;
    return n;
}

#if defined(__CUDACC__)

struct CigarArgs {
    SeqMap db, q;      // hit h: database read h against query read h (PairBatch layout)
    uint32_t n;        // hits, sorted by cells, largest first
    uint32_t *work;    // atomic work-queue head, zeroed
    int igap, egap;
    NwLink *carry;     // 2 * MAX_READ links per warp of the grid (query reads of more than 257 bases), or null
    uint32_t *codes;   // hit h's code words start at codes + code_off[h] (cg_words)
    const uint64_t *code_off;
    uint32_t *ops;     // hit h's ops slice: ops + op_off[h], xlen + ylen words
    const uint64_t *op_off;
    uint32_t *n_ops;   // ops used per hit
    HitAln *aln;
    uint32_t *stats;   // forward (length << 16 | identities) per hit, for the caller's check against the records
};

__global__ void __launch_bounds__(NW_THREADS) cigar_kernel(CigarArgs a) {
    __shared__ uint8_t sx_all[NW_WARPS][NW_XBUF];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t *sx = sx_all[warp];
    NwLink *carry0 = a.carry ? a.carry + (size_t)(blockIdx.x * NW_WARPS + warp) * 2 * MAX_READ : nullptr;
    constexpr int S = CG_S;
    for (;;) {
        uint32_t idx = 0;
        if (lane == 0) idx = atomicAdd(a.work, 1u);
        idx = __shfl_sync(0xffffffffu, idx, 0);
        if (idx >= a.n) break;
        const uint32_t xs = read_start(a.db, idx), xlen = a.db.start[idx + 1] - xs;
        const uint32_t ys = read_start(a.q, idx), ylen = a.q.start[idx + 1] - ys;
        const int X1 = (int)xlen - 1, Y1 = (int)ylen - 1;
        uint32_t *codes = a.codes + a.code_off[idx];
        __syncwarp();
        for (uint32_t i = lane; i < xlen; i += 32) sx[i] = (uint8_t)base_at(a.db.pk, (uint64_t)xs + i);
        __syncwarp();
        const uint32_t x0 = sx[0];
        const uint32_t y0 = base_at(a.q.pk, ys);
        NwBest wbest;
        wbest.s = NW_NEG * 2; wbest.i = wbest.j = wbest.p = 0;
        int pass = 0;
        for (int jb = 0; jb < Y1; jb += 32 * S, pass++) {
            int nl = (Y1 - jb + S - 1) / S;
            nl = nl > 32 ? 32 : nl;
            const bool more = jb + 32 * S < Y1;
            const int j0 = jb + lane * S + 1;
            const bool first = (jb == 0) && (lane == 0);
            uint64_t halo;
            {
                const int64_t g = (int64_t)ys + j0 - 2;
                halo = g >= 0 ? fetch32(a.q.pk, (uint64_t)g) : (fetch32(a.q.pk, 0) << 2);
            }
            const uint32_t ycols = (uint32_t)(halo >> 4) & ((1u << (2 * S)) - 1u);
            NwLane<S> L;
            nw_lane_init<S>(L, x0, halo, first, lane);
            const int cl = (Y1 - 1 - jb) % S;
            const bool owns_last = (Y1 >= j0) && (Y1 < j0 + S);
            NwLink out;
            out.a = out.ap = out.b = out.bp = out.mfs = out.mfy = out.mfp = 0;
            const NwLink *cin = carry0 ? carry0 + (size_t)((pass + 1) & 1) * MAX_READ : nullptr;
            NwLink *cout = carry0 ? carry0 + (size_t)(pass & 1) * MAX_READ : nullptr;
            uint32_t *pcodes = codes + (uint64_t)pass * (uint64_t)(X1 + 31) * 32 + lane;
            const int steps = X1 + nl - 1;
#define IMS_CG_STEP(T_, PREV1, PREV2)                                                                      \
    {                                                                                                      \
        const int i = (T_) - lane + 1;                                                                     \
        NwLink in = shfl_up_link(out);                                                                     \
        const bool act = (lane < nl) && (i >= 1) && (i <= X1);                                             \
        if (act) {                                                                                         \
            const uint32_t xi = sx[i];                                                                     \
            if (lane == 0) in = (jb == 0) ? nw_first_link(xi, y0) : cin[i];                                \
            const uint32_t d_ = ycols ^ (xi * 0x55555555u);                                                \
            const uint32_t mm = (d_ | (d_ >> 1)) & 0x55555555u;                                            \
            nw_row<S, 2>(L, PREV1, PREV2, in, out, i, j0, mm, a.igap, a.egap, X1, Y1, cl, owns_last, first, \
                         pcodes + (uint64_t)(T_) * 32);                                                    \
            if (more && lane == 31) cout[i] = out;                                                         \
        }                                                                                                  \
    }
            for (int t = 0; t < steps; t += 2) {
                IMS_CG_STEP(t, L.r0, L.r1)
                if (t + 1 < steps) IMS_CG_STEP(t + 1, L.r1, L.r0)
            }
#undef IMS_CG_STEP
            NwBest b = L.best;
            if (lane >= nl) b.s = NW_NEG * 2;
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) {
                NwBest c;
                c.s = __shfl_xor_sync(0xffffffffu, b.s, o);
                c.i = __shfl_xor_sync(0xffffffffu, b.i, o);
                c.j = __shfl_xor_sync(0xffffffffu, b.j, o);
                c.p = __shfl_xor_sync(0xffffffffu, b.p, o);
                if (best_better(c, b)) b = c;
            }
            if (best_better(b, wbest)) wbest = b;
            __syncwarp();  // also orders the lanes' code stores before lane 0's walk (memory ordering of __syncwarp)
        }
        if (lane == 0) {
            HitAln h;
            const uint32_t qs = ys;
            const uint8_t *sxc = sx;
            const SeqMap q = a.q;
            a.n_ops[idx] = cg_walk(codes, (uint32_t)X1, (uint32_t)wbest.i, (uint32_t)wbest.j,
                                   [sxc](uint32_t i) { return (uint32_t)sxc[i]; },
                                   [q, qs](uint32_t j) { return base_at(q.pk, (uint64_t)qs + j); },
                                   a.ops + a.op_off[idx], h);
            h.score = wbest.s;
            a.aln[idx] = h;
            a.stats[idx] = nw_stat_len(wbest.p) << 16 | nw_stat_ids(wbest.p);
        }
        __syncwarp();
    }
}

#endif  // __CUDACC__

}  // namespace imsame
