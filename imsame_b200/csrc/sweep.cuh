// sweep.cuh -- several coverage/identity threshold sets in one run (imsame_gpu_align_sweep, capi_sweep.inc).
//
// Only the filter of the NW epilogue (src/alignmentFunctions.c:163) and the first-accepted selection after it
// (:172,189) depend on -coverage / -identity: word table, seed hits, e-value test, candidate pairs and the NW
// result (score, bx, by, length, identities) of every pair are the same for every set.  The NW kernels run
// unchanged with the intersection tables lmin_all = max_t lmin_t, imin_all = max_t imin_t and best = the run's
// prune key P[r]; these kernels apply each set's own tables to the NW statistics they leave in PairRes.stats and
// keep one key per set and read, best_t[t * nq + r].
//
// P[r] stays an upper bound of max_t best_t[r] (both only decrease, and P is only ever lowered to a key that
// every set has accepted or to that maximum), so every pruning test that reads P is exact for every set:
// a pair is skipped only when it cannot be earlier than the winner of any set, and a read leaves the late pass
// of a two-pass run only when every set has accepted it on an early word.
#pragma once
#include "scan.cuh"

namespace imsame {

constexpr int SWEEP_MAX = 16;                                 // IMSAME_SWEEP_MAX
constexpr uint32_t SWEEP_LSTRIDE = MAX_READ + 1;              // lmin_t[ylen], ylen in [0, MAX_READ]
constexpr uint32_t SWEEP_ISTRIDE = 2 * MAX_READ + 1;          // imin_t[len], len in [0, 2 MAX_READ]

struct SweepArgs {
    const PairRec *pairs;
    const PairRes *res;
    SeqMap db, q;
    const uint16_t *lmin, *imin;   // n_sets tables of SWEEP_LSTRIDE / SWEEP_ISTRIDE entries
    unsigned long long *best;      // n_sets x nq keys
    unsigned long long *payload;   // n_sets x nq payloads (sweep_select_kernel)
    unsigned long long *prune;     // P[r]: the key array every pruning test of the run reads
    uint32_t nq;
    int n_sets;
};

#if defined(__CUDACC__)

// the set-independent part of the filter: a pair the NW kernels aligned (pruned pairs and pairs with a read
// longer than MAX_READ carry stats == 0), with the read lengths of the generic kernel's `ok` (X1 >= 1, Y1 >= 1)
__device__ __forceinline__ bool sweep_pair_stats(const SweepArgs &a, const PairRec &pr, const PairRes &z, uint32_t &ylen,
                                                 uint32_t &len, uint32_t &id) {
    len = (z.stats >> 16) & 0x7FFFu;
    id = z.stats & 0xFFFFu;
    if (len == 0) return false;
    ylen = a.q.fixed_len ? a.q.fixed_len : a.q.start[pr.r + 1] - a.q.start[pr.r];
    const uint32_t xlen = a.db.fixed_len ? a.db.fixed_len : a.db.start[pr.s + 1] - a.db.start[pr.s];
    return xlen >= 2 && ylen >= 2 && xlen <= (uint32_t)MAX_READ && ylen <= (uint32_t)MAX_READ;
}
__device__ __forceinline__ bool sweep_passes(const SweepArgs &a, int t, uint32_t ylen, uint32_t len, uint32_t id) {
    return len >= a.lmin[(size_t)t * SWEEP_LSTRIDE + ylen] && id >= a.imin[(size_t)t * SWEEP_ISTRIDE + len];
}

// after the NW launches of one band of one (logical) segment: blockIdx.y + 1 = NW class, range = that class's
// launch range of the band (bin_offsets_kernel).  Each set takes its earliest accepted key; then P[r] is lowered
// to the largest of the read's set keys (values read here may be stale, i.e. higher: still a bound)
__global__ void sweep_accept_kernel(SweepArgs a, const uint32_t *launch_range, int band) {
    const int c = (int)blockIdx.y + 1;
    const uint32_t lo = launch_range[2 * (c * NW_BANDS + band)], hi = launch_range[2 * (c * NW_BANDS + band) + 1];
    for (uint32_t i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += gridDim.x * blockDim.x) {
        const PairRec pr = a.pairs[i];
        uint32_t ylen, len, id;
        if (!sweep_pair_stats(a, pr, a.res[i], ylen, len, id)) continue;
        bool any = false;
        for (int t = 0; t < a.n_sets; t++)
            if (sweep_passes(a, t, ylen, len, id)) {
                atomicMin(&a.best[(size_t)t * a.nq + pr.r], (unsigned long long)pr.key);
                any = true;
            }
        if (!any) continue;
        unsigned long long m = 0;
        for (int t = 0; t < a.n_sets; t++) {
            const unsigned long long b = *(volatile unsigned long long *)&a.best[(size_t)t * a.nq + pr.r];
            m = b > m ? b : m;
        }
        if (m != KEY_NONE) atomicMin(&a.prune[pr.r], m);
    }
}

// after the last band: the pair that owns a set's final key writes that set's payload (select_kernel's layout)
__global__ void sweep_select_kernel(SweepArgs a, uint32_t n, uint64_t seg_seq_base, unsigned long long *pairs_total) {
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(pairs_total, (unsigned long long)n);
    unsigned needed = 0;  // diagnostic (counters[7]), against set 0
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const PairRec pr = a.pairs[i];
        const PairRes z = a.res[i];
        needed += pr.key <= a.best[pr.r] ? 1u : 0u;
        uint32_t ylen, len, id;
        if (!sweep_pair_stats(a, pr, z, ylen, len, id)) continue;
        for (int t = 0; t < a.n_sets; t++) {
            const size_t at = (size_t)t * a.nq + pr.r;
            if (pr.key == a.best[at] && sweep_passes(a, t, ylen, len, id))
                a.payload[at] = ((unsigned long long)(seg_seq_base + pr.s) << 32) | (z.stats & 0x7FFFFFFFu);
        }
    }
    needed = __reduce_add_sync(0xffffffffu, needed);
    if ((threadIdx.x & 31) == 0 && needed) atomicAdd(pairs_total + 2, (unsigned long long)needed);
}

// readsize_kernel per set: flag[t] when a candidate with a read of more than MAX_READ bases is earlier in scan
// order than set t's final key
__global__ void sweep_readsize_kernel(SweepArgs a, uint32_t n, unsigned long long *flag) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const PairRec pr = a.pairs[i];
        const uint32_t ylen = a.q.fixed_len ? a.q.fixed_len : a.q.start[pr.r + 1] - a.q.start[pr.r];
        const uint32_t xlen = a.db.fixed_len ? a.db.fixed_len : a.db.start[pr.s + 1] - a.db.start[pr.s];
        if (xlen <= (uint32_t)MAX_READ && ylen <= (uint32_t)MAX_READ) continue;
        for (int t = 0; t < a.n_sets; t++)
            if (pr.key < a.best[(size_t)t * a.nq + pr.r]) flag[t] = 1ull;
    }
}

#endif  // __CUDACC__

}  // namespace imsame
