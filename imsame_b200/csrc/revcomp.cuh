// revcomp.cuh -- reverse complement of packed read sets: the per-word body of revcomp_kernel and the arithmetic that
// mirrors one database segment (capi_samples.inc: imsame_gpu_sample_revcomp, imsame_gpu_db_revcomp), shared by the
// kernels and their CPU emulation (tests/emul/revcomp_emul.cpp).
//
// revComp writes the records in reverse order and reverses each one (src/reverseComplement.c:56,71-112), which
// together is the whole concatenated array reversed and complemented.  A database shard is cut into segments at
// read boundaries (capi.cu: db_layout), so reverse segment j is the reverse complement of forward segment m-1-j and
// every segment is mirrored on its own.
#pragma once
#include "common.cuh"

namespace imsame {

// Word w of the reverse complement of a packed array of `total` bases: output base P = complement(input base
// total - 1 - P).  The 16 input bases total-16w-16 .. total-16w-1 as one word, its 2-bit groups reversed (bit
// reversal + swap inside each pair), high bit of every group flipped (A0 <-> T2, C1 <-> G3); bases past the end
// (and whole words past it: the zero padding) are 0.
IMS_HD uint32_t revcomp_word(const uint32_t *in, uint32_t total, uint32_t w) {
    const uint64_t first_out = (uint64_t)w * 16;  // output bases first_out .. first_out + 15
    if (first_out >= total) return 0;
    const uint32_t nb = total - first_out < 16 ? (uint32_t)(total - first_out) : 16u;  // valid bases in this word
    const int64_t lo = (int64_t)total - (int64_t)first_out - 16;                        // input index of the LAST output base
    uint32_t x = lo >= 0 ? fetch16(in, (uint64_t)lo) : (fetch16(in, 0) << (2 * (int)(-lo)));
    x = rev_bits32(x);
    x = ((x & 0xAAAAAAAAu) >> 1) | ((x & 0x55555555u) << 1);
    x ^= 0xAAAAAAAAu;
    return nb < 16 ? (x & ((1u << (2 * nb)) - 1u)) : x;
}

// Entry i of a mirrored ascending list of positions inside `total` bases: read offsets (n + 1 entries with the
// sentinel: start'[i] = total - start[n - i]) and word breaks (brk'[i] = total - brk[n_brk - 1 - i]) alike.
IMS_HD uint32_t mirror_entry(const uint32_t *in, uint32_t n_in, uint32_t total, uint32_t i) { return total - in[n_in - 1 - i]; }

// Word breaks kept after mirroring.  A break at a segment's first base sits at a read start (words never span
// reads, so it changes no word) and would mirror onto the segment's end, a position the loader never gives a break
// (db_layout keeps breaks < the segment's end): it is dropped.  Breaks are ascending, so it can only be the first
// one, and its mirror is the last entry of the mirrored list: the kept ones are the first n_brk - 1.
IMS_HD uint32_t mirror_n_brk(uint32_t n_brk, uint32_t first_brk) { return n_brk - (n_brk && first_brk == 0 ? 1u : 0u); }

// Where a segment [base, base + len) of a shard of `shard_len` positions (bases or reads) lies in the shard's
// reverse complement: pos_base' = shard_total - (pos_base + total), seq_base' = shard_nseqs - (seq_base + n).
IMS_HD uint64_t mirror_base(uint64_t shard_len, uint64_t base, uint64_t len) { return shard_len - (base + len); }

}  // namespace imsame
