// kcache.cuh -- the pair-result cache of a seed-length sweep (imsame_gpu_align_kmers, capi_kmers.inc).
//
// The NW result of a candidate pair (src/alignmentFunctions.c:389-489 aligns the two WHOLE reads, wherever the seed
// was) depends on the two reads and the gap scores only, and the filter bit on the coverage / identity tables: none
// of them depends on k.  Seeds of different lengths keep finding the same (query read, database read) pairs, so the
// entries of a sweep after the first look every candidate up in a device hash table of the pairs the earlier entries
// aligned, keyed by (query read << 32 | database read of the shard), valued by the 32-bit PairRes.stats word.
//
// The NW kernels stay as they are.  A cached pair is hidden from them:
//   hide     (after the segment's scan)   original key and cached stats to a side array indexed like `pairs`,
//                                         pairs[i].key = KEY_NONE: both NW kernels skip it (key >= best[r]) and write
//                                         a zero result; where the cached filter bit is set, best[r] is lowered to the
//                                         key right away, as the NW epilogue would have done, so the bands prune as much
//                                         as in a separate run (the final key of a read is the smallest key of its
//                                         passing candidates whatever the order they are found in);
//   restore  (after the last band)        original key and cached stats back into pairs / res, where select_kernel
//                                         and readsize_kernel read them.
// After the entry, every pair the NW kernels aligned (a best cell on the last row or column: bx | by != 0; skipped
// pairs leave bx == by == 0) is inserted.
#pragma once
#include "nw.cuh"
#include "scan.cuh"

namespace imsame {

constexpr unsigned long long KC_EMPTY = ~0ull;  // never a key: query reads < 2^32 - 256, database reads < 2^31

struct KcSide {
    unsigned long long key;  // the pair's scan-order key while pairs[i].key is KEY_NONE
    uint32_t stats;          // its cached PairRes.stats
    uint32_t pad;
};

struct KcTable {
    unsigned long long *keys;  // KC_EMPTY = free slot
    uint32_t *vals;
    uint32_t mask;             // slots - 1 (a power of two; the host keeps the table at most half full)
};

#if defined(__CUDACC__)

__device__ __forceinline__ uint32_t kc_slot(unsigned long long key, uint32_t mask) {
    key ^= key >> 33;
    key *= 0xff51afd7ed558ccdull;
    key ^= key >> 33;
    return (uint32_t)key & mask;
}

__device__ __forceinline__ bool kc_find(const KcTable &t, unsigned long long key, uint32_t *val) {
    for (uint32_t h = kc_slot(key, t.mask);; h = (h + 1) & t.mask) {
        const unsigned long long k = t.keys[h];
        if (k == key) { *val = t.vals[h]; return true; }
        if (k == KC_EMPTY) return false;
    }
}

// a slot is reserved before it is taken: once `limit` (half the slots) are, the insertion stops and flags the overflow,
// so that every probe sequence ends at a free slot; the host doubles the table and runs the pass again
__device__ __forceinline__ void kc_insert(const KcTable &t, unsigned long long key, uint32_t val, unsigned long long *count,
                                          unsigned long long limit, unsigned long long *overflow) {
    uint32_t v;
    if (kc_find(t, key, &v)) return;  // (inserted by a pass that overflowed)
    if (atomicAdd(count, 1ull) >= limit) { *overflow = 1ull; return; }
    for (uint32_t h = kc_slot(key, t.mask);; h = (h + 1) & t.mask)
        if (atomicCAS(&t.keys[h], KC_EMPTY, key) == KC_EMPTY) { t.vals[h] = val; return; }
}

// pairs[0 .. n) of one logical segment (seg_seq_base: its first database read in the shard)
__global__ void kc_hide_kernel(PairRec *pairs, KcSide *side, uint32_t n, uint32_t seg_seq_base, KcTable t,
                               unsigned long long *best) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const PairRec pr = pairs[i];
        uint32_t v;
        if (!kc_find(t, ((unsigned long long)pr.r << 32) | (seg_seq_base + pr.s), &v)) continue;
        KcSide s;
        s.key = pr.key; s.stats = v; s.pad = 0;
        side[i] = s;
        pairs[i].key = KEY_NONE;
        if (v & 0x80000000u) atomicMin(&best[pr.r], pr.key);
    }
}

__global__ void kc_restore_kernel(PairRec *pairs, PairRes *res, const KcSide *side, uint32_t n) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        if (pairs[i].key != KEY_NONE) continue;
        const KcSide s = side[i];
        pairs[i].key = s.key;
        PairRes z;
        z.score = 0; z.bx = z.by = 0; z.stats = s.stats;  // (bx == by == 0: not inserted again)
        res[i] = z;
    }
}

__global__ void kc_insert_kernel(const PairRec *pairs, const PairRes *res, uint32_t n, uint32_t seg_seq_base, KcTable t,
                                 unsigned long long *count, unsigned long long limit, unsigned long long *overflow) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const PairRes z = res[i];
        if ((z.bx | z.by) == 0) continue;
        const PairRec pr = pairs[i];
        kc_insert(t, ((unsigned long long)pr.r << 32) | (seg_seq_base + pr.s), z.stats, count, limit, overflow);
    }
}

// growth: every entry of the old table into the new one
__global__ void kc_rehash_kernel(const unsigned long long *keys, const uint32_t *vals, uint32_t n_slots, KcTable t,
                                 unsigned long long *count, unsigned long long limit, unsigned long long *overflow) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_slots; i += gridDim.x * blockDim.x)
        if (keys[i] != KC_EMPTY) kc_insert(t, keys[i], vals[i], count, limit, overflow);
}

#endif  // __CUDACC__

}  // namespace imsame
