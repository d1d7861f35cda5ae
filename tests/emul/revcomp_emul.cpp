// CPU emulation of the device reverse complement of a resident database (imsame_gpu_db_revcomp): the per-word body
// of revcomp_kernel and the segment mirror arithmetic (csrc/revcomp.cuh) applied to random multi-segment layouts,
// against a plain reverse complement of the concatenated reads laid out into segments by the rules of db_layout
// (capi.cu).  Fixed and ragged reads, totals that are no multiple of 16, one-read segments, word breaks at read and
// segment starts; and the mirror applied twice against the forward layout.
//   usage: revcomp_emul <n_cases> <seed>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>
#include "../../imsame_b200/csrc/revcomp.cuh"
using namespace imsame;

static uint64_t rng_state;
static uint64_t rnd() { uint64_t z = (rng_state += 0x9E3779B97F4A7C15ull); z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27)) * 0x94D049BB133111EBull; return z ^ (z >> 31); }
static const uint32_t PAD_WORDS = 16;

struct Seg {  // what capi.cu keeps per segment (host copies of the device arrays)
    uint64_t pos_base = 0, seq_base = 0;
    uint32_t n = 0, total = 0, fixed_len = 0, n_brk = 0;
    std::vector<uint32_t> pk, start, brk;
};

static std::vector<uint32_t> pack(const std::string &s) {  // pack_kernel: code = (ascii >> 1) & 3, 16 bases per word
    std::vector<uint32_t> pk((s.size() + 15) / 16 + PAD_WORDS, 0);
    for (size_t i = 0; i < s.size(); i++) pk[i / 16] |= (uint32_t)((s[i] >> 1) & 3) << (2 * (i % 16));
    return pk;
}

// db_layout: greedy whole reads up to seg_max bases per segment; breaks kept where base <= b < end
static std::vector<Seg> layout(const std::string &seq, const std::vector<uint64_t> &start, const std::vector<uint64_t> &brk,
                               uint32_t fixed, uint64_t seg_max) {
    const uint64_t n = start.size() - 1, total = seq.size();
    std::vector<Seg> segs;
    uint64_t r0 = 0, bi = 0;
    while (r0 < n) {
        const uint64_t base = start[r0];
        uint64_t r1;
        if (fixed) r1 = std::min<uint64_t>(n, r0 + std::max<uint64_t>(1, seg_max / fixed));
        else {
            r1 = r0 + 1;
            while (r1 < n && start[r1 + 1] - base <= seg_max) r1++;
        }
        const uint64_t end = r1 < n ? start[r1] : total;
        Seg s;
        s.pos_base = base; s.seq_base = r0; s.n = (uint32_t)(r1 - r0); s.total = (uint32_t)(end - base); s.fixed_len = fixed;
        s.pk = pack(seq.substr(base, end - base));
        if (!fixed)
            for (uint64_t r = r0; r <= r1; r++) s.start.push_back((uint32_t)((r < n ? start[r] : total) - base));
        while (bi < brk.size() && brk[bi] < end) {
            if (brk[bi] >= base) s.brk.push_back((uint32_t)(brk[bi] - base));
            bi++;
        }
        s.n_brk = (uint32_t)s.brk.size();
        segs.push_back(s);
        r0 = r1;
    }
    return segs;
}

// imsame_gpu_db_revcomp, one thread per element as the kernels run
static void mirror(std::vector<Seg> &segs, uint64_t shard_total, uint64_t shard_nseqs) {
    for (Seg &s : segs) {
        std::vector<uint32_t> out(s.pk.size());
        for (uint32_t w = 0; w < out.size(); w++) out[w] = revcomp_word(s.pk.data(), s.total, w);
        s.pk.swap(out);
        if (!s.fixed_len) {
            std::vector<uint32_t> st(s.n + 1);
            for (uint32_t i = 0; i <= s.n; i++) st[i] = mirror_entry(s.start.data(), s.n + 1, s.total, i);
            s.start.swap(st);
        }
        if (s.n_brk) {
            std::vector<uint32_t> b(s.n_brk);
            for (uint32_t i = 0; i < s.n_brk; i++) b[i] = mirror_entry(s.brk.data(), s.n_brk, s.total, i);
            const uint32_t kept = mirror_n_brk(s.n_brk, s.brk[0]);
            b.resize(kept);
            s.brk.swap(b);
            s.n_brk = kept;
        }
    }
    std::reverse(segs.begin(), segs.end());
    for (Seg &s : segs) {
        s.pos_base = mirror_base(shard_total, s.pos_base, s.total);
        s.seq_base = mirror_base(shard_nseqs, s.seq_base, s.n);
    }
}

static std::vector<uint32_t> without_zero(const std::vector<uint32_t> &v) {
    std::vector<uint32_t> o;
    for (uint32_t x : v) if (x) o.push_back(x);
    return o;
}

// same layout; breaks compared exactly, except that `got` may lack those at a segment's first base (a read start:
// they change no word; revcomp.cuh: mirror_n_brk drops the mirror image of one)
static bool same(const std::vector<Seg> &got, const std::vector<Seg> &want) {
    if (got.size() != want.size()) return false;
    for (size_t j = 0; j < got.size(); j++) {
        const Seg &a = got[j], &b = want[j];
        if (a.pos_base != b.pos_base || a.seq_base != b.seq_base || a.n != b.n || a.total != b.total || a.pk != b.pk) return false;
        if (!a.fixed_len && a.start != b.start) return false;
        if (without_zero(a.brk) != without_zero(b.brk) || a.brk.size() != a.n_brk) return false;
    }
    return true;
}

int main(int argc, char **argv) {
    const int n_cases = argc > 1 ? atoi(argv[1]) : 2000;
    rng_state = argc > 2 ? strtoull(argv[2], 0, 10) : 1;
    const char B[4] = {'A', 'C', 'G', 'T'};
    int bad = 0, multi = 0, one_read = 0, seg_start_brk = 0, not16 = 0;
    for (int it = 0; it < n_cases; it++) {
        const bool fixed = it % 3 == 0;
        const uint64_t n = 1 + rnd() % 60;
        const uint32_t L = 1 + rnd() % 40;
        std::vector<uint64_t> start(1, 0);
        for (uint64_t r = 0; r < n; r++) start.push_back(start.back() + (fixed ? L : 1 + rnd() % 70));
        const uint64_t total = start.back();
        std::string seq(total, 'A');
        for (auto &c : seq) c = B[rnd() & 3];
        const uint64_t seg_max = it % 7 == 0 ? 1 : 16 + rnd() % 400;  // 1: every segment holds one read
        // breaks: random positions, and some at read starts; the layout decides which are segment starts
        std::vector<uint64_t> brk;
        for (uint64_t p = 0; p < total; p++) {
            const bool at_read = std::binary_search(start.begin(), start.end() - 1, p);
            if (rnd() % (at_read ? 4 : 40) == 0) brk.push_back(p);
        }
        const std::vector<Seg> fwd = layout(seq, start, brk, fixed ? L : 0, seg_max);
        // the plain reverse complement: reads in reverse order, each reverse complemented; offsets and breaks mirrored
        std::string rseq(total, 'A');
        for (uint64_t i = 0; i < total; i++) {
            const char c = seq[total - 1 - i];
            rseq[i] = c == 'A' ? 'T' : c == 'C' ? 'G' : c == 'G' ? 'C' : 'A';
        }
        std::vector<uint64_t> rstart(n + 1), rbrk;
        for (uint64_t i = 0; i <= n; i++) rstart[i] = total - start[n - i];
        for (size_t i = brk.size(); i-- > 0;)
            if (brk[i] > 0) rbrk.push_back(total - brk[i]);  // (a break at base 0 would mirror onto the end: none there)
        // its segments are the forward ones mirrored: cut it where they end
        std::vector<Seg> want;
        {
            std::vector<uint64_t> cuts;  // reverse read index where each reverse segment starts
            for (size_t j = fwd.size(); j-- > 0;) cuts.push_back(n - (fwd[j].seq_base + fwd[j].n));
            for (size_t j = 0; j < cuts.size(); j++) {
                const uint64_t r0 = cuts[j], r1 = j + 1 < cuts.size() ? cuts[j + 1] : n;
                std::vector<uint64_t> st(rstart.begin() + r0, rstart.begin() + r1 + 1);
                for (auto &x : st) x -= rstart[r0];
                std::vector<uint64_t> bk;
                for (uint64_t b : rbrk)
                    if (b >= rstart[r0] && b < rstart[r1]) bk.push_back(b);
                std::vector<Seg> one = layout(rseq.substr(rstart[r0], rstart[r1] - rstart[r0]), st, {}, fixed ? L : 0, UINT64_MAX);
                Seg s = one[0];
                s.pos_base = rstart[r0]; s.seq_base = r0;
                for (uint64_t b : bk) s.brk.push_back((uint32_t)(b - rstart[r0]));
                s.n_brk = (uint32_t)s.brk.size();
                want.push_back(s);
            }
        }
        std::vector<Seg> got = fwd;
        mirror(got, total, n);
        bool ok = same(got, want);
        std::vector<Seg> back = got;  // involution
        mirror(back, total, n);
        ok = ok && same(back, fwd);
        multi += fwd.size() > 1;
        for (const Seg &s : fwd) {
            one_read += s.n == 1;
            seg_start_brk += s.n_brk && s.brk[0] == 0 && s.pos_base > 0;
            not16 += s.total % 16 != 0;
        }
        if (!ok) { bad++; if (bad < 5) printf("MISMATCH case %d: %s, %llu reads, %zu segments\n", it, fixed ? "fixed" : "ragged", (unsigned long long)n, fwd.size()); }
    }
    printf("%d layouts (%d multi-segment; %d one-read segments, %d breaks at a segment start, %d segment totals not a multiple of 16), %d mismatches\n",
           n_cases, multi, one_read, seg_start_brk, not16, bad);
    return bad != 0 || !multi || !one_read || !seg_start_brk || !not16;
}
