// capi.cu -- C ABI (include/imsame_gpu.h) over the sm_100a kernels.
// Host orchestration only: device memory, streams, launches, exact threshold
// tables.  There is no CPU implementation of the hot path in this library.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/imsame_gpu.h"
#include "../host/imsame_host.h"
#include "cigar.cuh"
#include "kcache.cuh"
#include "nw.cuh"
#include "nwp_launch.h"
#include "qtable.cuh"
#include "revcomp.cuh"
#include "scan.cuh"
#include "sweep.cuh"

using namespace imsame;

namespace {

constexpr uint64_t SEG_MAX_BASES = 1ull << 29;    // database segment size (positions stay uint32; bounds the pair table)
constexpr uint64_t STAGE_BYTES = 256ull << 20;    // ASCII staging buffer on the device
constexpr uint64_t PIN_BYTES = 32ull << 20;       // pinned bounce buffers for pageable host input (two of them)
constexpr uint32_t PAD_WORDS = 16;                // zero words after every packed array
constexpr uint32_t BINS_STRIDE = 7 * NW_NBINS + 8;

struct Seg {
    uint64_t pos_base = 0, seq_base = 0;  // offsets inside the shard handed to set_db
    uint32_t n = 0, total = 0, fixed_len = 0, n_brk = 0;
    uint32_t *pk = nullptr, *start = nullptr, *blk = nullptr, *brk = nullptr;
    cudaEvent_t ready = nullptr;  // bases uploaded and packed (recorded on the upload stream)
    bool wait_ready = false;      // the scan has to wait for `ready` (uploaded on another stream)
    bool borrowed = false;        // the buffers belong to an imsame_sample
};

enum Phase { PH_PACKQ, PH_K1, PH_PACKDB, PH_K2, PH_K2B, PH_K3, PH_SELECT, PH_H2D, PH_D2H, PH_COMM, PH_COUNT };

}  // namespace

struct imsame_ctx {
    int device = 0;
    int n_sm = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    // imsame_gpu_align uploads on a stream of its own, so that the database segments arrive and are packed while
    // the scan of the earlier ones runs (SURVEY 8(f) rank 2); everywhere else uploads share `stream`
    cudaStream_t copy_stream = nullptr;
    cudaStream_t up_stream = nullptr;  // the stream uploads currently go to (== stream outside imsame_gpu_align)
    cudaEvent_t q_ready = nullptr;     // query packed (recorded on up_stream)
    std::string cuda_err;

    // query
    uint32_t *q_pk = nullptr, *q_start = nullptr, *q_blk = nullptr;
    uint32_t nq = 0, q_total = 0, q_fixed = 0, q_maxlen = 0;
    uint32_t class_mask = 0;
    std::vector<uint32_t> q_start_host;
    uint32_t *off = nullptr, *cursor = nullptr, *tile_sums = nullptr;
    uint32_t *off_own = nullptr;  // the context's own offsets table (`off` may point into a resident sample instead)
    QEntry *qtab = nullptr;  // query word table entries, bucket by bucket (qtable.cuh)
    bool q_borrowed = false;  // the query buffers and its word table belong to an imsame_sample
    // "Early words first" (two-pass runs, see run_plan): the words that end inside the first early_bands k-mer-end
    // bands of their read have a table of their own (built once per query), the later words of the reads that are
    // still without an accepted hit after those bands a second one (built in the middle of every run)
    bool tab_full = false, tab_early = false;  // off/qtab resp. off_early/qtab_early hold this query's words
    uint32_t tab_early_split = 0;
    uint32_t *off_early = nullptr, *off_late = nullptr;
    QEntry *qtab_early = nullptr, *qtab_late = nullptr;
    uint64_t n_words_early = 0, n_words_late = 0;
    int passes_mode = 0;     // imsame_gpu_set_passes: 0 = decide per run, 1 = one pass, 2 = early words first
    int run_passes = 1;      // of the run in progress
    int run_early_bands = 0; // two passes: NW launches [0, run_early_bands) belong to the first
    uint64_t n_qwords = 0;
    uint64_t q_threads = 0;
    bool have_query = false;

    // database shard
    std::vector<Seg> segs;
    uint64_t db_total = 0, db_nseqs = 0;
    uint32_t db_maxlen = 0;
    bool have_db = false;
    bool db_rc = false;  // the resident database is the reverse complement of what was uploaded (imsame_gpu_db_revcomp)
    // the query and database of the last successful imsame_gpu_align (1) / imsame_gpu_align_sharded over this many
    // contexts, still resident, and the parameters this context ran it with (imsame_gpu_align_revcomp); 0 = none
    int last_align = 0;
    imsame_params align_params;

    // tables + work buffers
    uint16_t *d_nmin = nullptr, *d_lmin = nullptr, *d_imin = nullptr;
    uint32_t *d_lut = nullptr;
    unsigned long long *hkeys = nullptr, *hvals = nullptr;
    uint32_t hcap = 0;
    PairRec *pairs = nullptr;
    PairRes *res = nullptr;
    uint32_t *d_small = nullptr;  // [0] n_pairs, [1] work head
    unsigned long long *d_counters = nullptr;  // [0..3] scan counters, [4] cells, [5] pairs total, [6] pairs aligned, [7] pairs needed in hindsight
    int *d_overflow = nullptr;
    unsigned long long *keys = nullptr, *payload = nullptr, *pkey = nullptr;
    uint64_t keys_cap = 0;
    // state of a run in progress (run_begin .. run_end)
    unsigned long long *run_keys = nullptr, *run_payload = nullptr;
    imsame_params run_params;
    bool run_active = false;
    bool run_masked = false;   // the payloads of superseded keys have been dropped (run_mask)
    // threshold sweep (capi_sweep.inc): per-set keys and payloads (sweep_cap = sets x reads they hold), the
    // per-set filter tables (SWEEP_MAX of each) and read-size flags
    unsigned long long *sw_best = nullptr, *sw_payload = nullptr, *sw_flags = nullptr;
    uint64_t sweep_cap = 0;
    uint16_t *sw_lmin = nullptr, *sw_imin = nullptr;
    // communicator of a sharded database (capi_sharded.inc): NCCL over NVLink, one rank per GPU
    void *comm = nullptr;
    int comm_rank = 0, comm_size = 1;
    unsigned long long *comm_flag = nullptr;  // one device word for status / read-size reductions
    unsigned long long *comm_flag3 = nullptr; // three more: comm_status
    bool table_dirty = false;  // the pair table may hold entries of a run that failed before they were binned
    // (after the launch ranges: NBINS more work heads, for the second kernel of a mixed run)
    // per segment (stride BINS_STRIDE): [0,NBINS) counts | [NBINS, 3*NBINS+1) offsets + cursors |
    // NBINS work heads | 2*NBINS launch ranges
    uint32_t *d_bins = nullptr;
    uint32_t bins_segs = 0;
    uint64_t pairs_cap = 0;                       // capacity of pairs / res (all segments of a run)
    std::vector<uint64_t> seg_pair_base, seg_pair_count;
    NwLink *carry = nullptr;
    uint64_t carry_warps = 0;
    uint8_t *stage = nullptr;
    uint32_t *tb_pin = nullptr;            // pinned host buffer of imsame_gpu_traceback (ops, counts, cells), kept across calls
    uint64_t tb_pin_cap = 0;               // in 32-bit words
    uint8_t *pin[2] = {nullptr, nullptr};  // pinned bounce buffers (upload_pack), their copy-done events
    cudaEvent_t pin_ev[2] = {nullptr, nullptr};
    bool pin_busy[2] = {false, false};     // a copy out of the buffer has been enqueued (wait for pin_ev before refilling)
    int nw_grid[9] = {0};                 // by columns per lane (1..8)
    int cigar_grid = 0;                   // cigar_kernel (imsame_gpu_align_traceback)
    int nwp_grid[NW_CLASSES + 1] = {0};   // by NW class
    bool in_align = false;  // imsame_gpu_align: upload phases belong to the same stats
    int nw_mode = 0;  // 0: packed-word kernel where pw_eligible() holds, 1: generic kernel only
    int k = K;        // seed length (imsame_gpu_set_kmer); k_tables = the length off/cursor/tile_sums are sized for
    int k_tables = 0;
    int q_k = K;      // the seed length the resident query table was built with
    int scan_grid = 0;
    // test hook IMSAME_TEST_FAIL_ALLOC=N[,M] (read by imsame_gpu_create): device allocations N .. N+M-1 of this context fail
    uint64_t n_allocs = 0, fail_alloc_first = 0, fail_alloc_count = 0;

    // device blocks released by free_query / free_db, reused by the next set_query / set_db
    // (cudaFree + cudaMalloc of the ~3 GB of a cfg2 call cost several hundred ms per call)
    struct Block { void *p; size_t bytes; };
    std::vector<Block> live_blocks, free_blocks;

    // phase timing
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_used = 0;
    struct Span { int ph; cudaEvent_t a, b; };
    std::vector<Span> spans;
    uint64_t h2d_bytes = 0, d2h_bytes = 0;
    uint32_t launches = 0, k2_launches = 0, k3_launches = 0, k3_packed = 0;
};

namespace {

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            ctx->cuda_err = std::string(#call) + ": " + cudaGetErrorString(_e);                   \
            return _e == cudaErrorMemoryAllocation ? IMSAME_ENOMEM : IMSAME_ECUDA;                 \
        }                                                                                          \
    } while (0)

cudaEvent_t new_event(imsame_ctx *ctx) {
    if (ctx->ev_used == ctx->ev_pool.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        ctx->ev_pool.push_back(e);
    }
    return ctx->ev_pool[ctx->ev_used++];
}
struct PhaseScope {
    imsame_ctx *ctx;
    cudaStream_t stream;
    imsame_ctx::Span sp;
    PhaseScope(imsame_ctx *c, int ph, cudaStream_t on = nullptr) : ctx(c), stream(on ? on : c->stream) {
        sp.ph = ph;
        sp.a = new_event(c);
        sp.b = new_event(c);
        cudaEventRecord(sp.a, stream);
    }
    ~PhaseScope() {
        cudaEventRecord(sp.b, stream);
        ctx->spans.push_back(sp);
    }
};
void reset_timing(imsame_ctx *ctx) {
    ctx->ev_used = 0;
    ctx->spans.clear();
    ctx->h2d_bytes = ctx->d2h_bytes = 0;
    ctx->launches = ctx->k2_launches = ctx->k3_launches = ctx->k3_packed = 0;
}

// cudaMalloc of the context.  Under the test hook IMSAME_TEST_FAIL_ALLOC the chosen allocations ask for an impossible
// size instead: cudaMalloc fails and records the error as on a full device, and no memory outside the process is touched.
cudaError_t ctx_malloc(imsame_ctx *ctx, void **p, size_t bytes) {
    const uint64_t i = ++ctx->n_allocs;
    if (ctx->fail_alloc_first && i >= ctx->fail_alloc_first && i < ctx->fail_alloc_first + ctx->fail_alloc_count) {
        if (cudaMalloc(p, (size_t)1 << 50) == cudaSuccess) cudaFree(*p);
        *p = nullptr;
        return cudaErrorMemoryAllocation;
    }
    const cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) *p = nullptr;
    return e;
}

template <typename T>
int dev_alloc(imsame_ctx *ctx, T **p, uint64_t count) {
    const size_t bytes = (size_t)std::max<uint64_t>(count, 1) * sizeof(T);
    cudaError_t e = ctx_malloc(ctx, (void **)p, bytes);
    if (e == cudaErrorMemoryAllocation && !ctx->free_blocks.empty()) {  // give the recycled blocks back and retry
        cudaGetLastError();
        for (auto &b : ctx->free_blocks) cudaFree(b.p);
        ctx->free_blocks.clear();
        e = ctx_malloc(ctx, (void **)p, bytes);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();  // a failed cudaMalloc is not sticky: the next CK(cudaGetLastError()) must not report it again
        ctx->cuda_err = std::string("cudaMalloc: ") + cudaGetErrorString(e);
        return e == cudaErrorMemoryAllocation ? IMSAME_ENOMEM : IMSAME_ECUDA;
    }
    return IMSAME_OK;
}
template <typename T>
void dev_free(T *&p) {
    if (p) cudaFree(p);
    p = nullptr;
}

// recycled allocation: smallest released block of at least the size (and at most twice it), else cudaMalloc
template <typename T>
int pool_alloc(imsame_ctx *ctx, T **p, uint64_t count) {
    const size_t bytes = (size_t)std::max<uint64_t>(count, 1) * sizeof(T);
    int best = -1;
    for (size_t i = 0; i < ctx->free_blocks.size(); i++) {
        const size_t b = ctx->free_blocks[i].bytes;
        if (b >= bytes && b <= 2 * bytes + 4096 && (best < 0 || b < ctx->free_blocks[best].bytes)) best = (int)i;
    }
    if (best >= 0) {
        *p = (T *)ctx->free_blocks[best].p;
        ctx->live_blocks.push_back(ctx->free_blocks[best]);
        ctx->free_blocks.erase(ctx->free_blocks.begin() + best);
        return IMSAME_OK;
    }
    cudaError_t e = ctx_malloc(ctx, (void **)p, bytes);
    if (e == cudaErrorMemoryAllocation && !ctx->free_blocks.empty()) {  // give the cached blocks back and retry
        cudaGetLastError();
        for (auto &b : ctx->free_blocks) cudaFree(b.p);
        ctx->free_blocks.clear();
        e = ctx_malloc(ctx, (void **)p, bytes);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();  // (as in dev_alloc)
        ctx->cuda_err = std::string("cudaMalloc: ") + cudaGetErrorString(e);
        return e == cudaErrorMemoryAllocation ? IMSAME_ENOMEM : IMSAME_ECUDA;
    }
    ctx->live_blocks.push_back({(void *)*p, bytes});
    return IMSAME_OK;
}
template <typename T>
void pool_free(imsame_ctx *ctx, T *&p) {
    if (!p) return;
    for (size_t i = 0; i < ctx->live_blocks.size(); i++)
        if (ctx->live_blocks[i].p == (void *)p) {
            ctx->free_blocks.push_back(ctx->live_blocks[i]);
            ctx->live_blocks.erase(ctx->live_blocks.begin() + i);
            p = nullptr;
            return;
        }
    cudaFree(p);
    p = nullptr;
}
void pool_destroy(imsame_ctx *ctx) {
    for (auto &b : ctx->free_blocks) cudaFree(b.p);
    for (auto &b : ctx->live_blocks) cudaFree(b.p);
    ctx->free_blocks.clear();
    ctx->live_blocks.clear();
}

void free_query(imsame_ctx *ctx) {
    if (ctx->q_borrowed) {
        ctx->q_pk = ctx->q_start = ctx->q_blk = nullptr;
        ctx->qtab = nullptr;
        ctx->off = ctx->off_own;
        ctx->q_borrowed = false;
    } else {
        pool_free(ctx, ctx->q_pk); pool_free(ctx, ctx->q_start); pool_free(ctx, ctx->q_blk);
        pool_free(ctx, ctx->qtab);
    }
    pool_free(ctx, ctx->qtab_early); pool_free(ctx, ctx->qtab_late);
    ctx->tab_full = ctx->tab_early = false;
    ctx->have_query = false;
    ctx->last_align = 0;
}
void free_db(imsame_ctx *ctx) {
    for (Seg &s : ctx->segs) {
        if (!s.borrowed) { pool_free(ctx, s.pk); pool_free(ctx, s.start); pool_free(ctx, s.blk); pool_free(ctx, s.brk); }
        if (s.ready) cudaEventDestroy(s.ready);
    }
    ctx->segs.clear();
    ctx->have_db = false;
    ctx->db_rc = false;
    ctx->last_align = 0;
}

uint32_t uniform_len(const uint64_t *start, uint64_t n, uint64_t total) {
    if (n == 0) return 0;
    const uint64_t L = (n > 1 ? start[1] : total) - start[0];
    if (L == 0 || L > 0xFFFFFFFFull) return 0;
    for (uint64_t r = 0; r < n; r++) {
        const uint64_t e = (r + 1 < n) ? start[r + 1] : total;
        if (e - start[r] != L) return 0;
    }
    return (uint32_t)L;
}

// upload ASCII bases [0,n) in staged chunks and pack them into pk (device)
// copy with several host threads: one thread moves ~10 GB/s, the link to the GPU takes 50
static void par_memcpy(uint8_t *dst, const unsigned char *src, uint64_t n) {
    unsigned nt = std::thread::hardware_concurrency();
    nt = nt < 1 ? 1 : (nt > 8 ? 8 : nt);
    if (n < (4u << 20) || nt == 1) { memcpy(dst, src, n); return; }
    std::vector<std::thread> th;
    const uint64_t per = (n / nt + 63) & ~63ull;
    for (unsigned t = 1; t < nt; t++) {
        const uint64_t b = per * t, e = std::min<uint64_t>(n, b + per);
        if (b < e) th.emplace_back([=] { memcpy(dst + b, src + b, e - b); });
    }
    memcpy(dst, src, std::min<uint64_t>(per, n));
    for (auto &x : th) x.join();
}

// Pageable host input (the command line: buffers the FASTA loader malloc'ed) goes through two pinned bounce
// buffers filled by several host threads while the previous one is on its way to the device; a plain
// cudaMemcpyAsync from pageable memory is staged by the driver on one thread (~9 GB/s: 0.28 s for cfg2's
// database).  Pinned input (bench.py, imsame_gpu_host_alloc) is copied directly.
static bool host_is_pageable(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return a.type == cudaMemoryTypeUnregistered;
}

int upload_pack(imsame_ctx *ctx, const unsigned char *host, uint64_t n, uint32_t *pk, int ph_pack) {
    cudaStream_t up = ctx->up_stream ? ctx->up_stream : ctx->stream;
    if (!ctx->stage) { int rc = dev_alloc(ctx, &ctx->stage, STAGE_BYTES); if (rc) return rc; }
    if (n >= 2 * PIN_BYTES && host_is_pageable(host)) {
        for (int b = 0; b < 2; b++)
            if (!ctx->pin[b]) {
                if (cudaMallocHost((void **)&ctx->pin[b], PIN_BYTES) != cudaSuccess ||
                    cudaEventCreateWithFlags(&ctx->pin_ev[b], cudaEventDisableTiming) != cudaSuccess) {
                    cudaGetLastError();
                    if (ctx->pin[b]) { cudaFreeHost(ctx->pin[b]); ctx->pin[b] = nullptr; }
                    break;
                }
            }
        if (ctx->pin[0] && ctx->pin[1]) {
            uint64_t i = 0;
            for (uint64_t at = 0; at < n; at += PIN_BYTES, i++) {
                const int b = (int)(i & 1);
                const uint64_t len = std::min<uint64_t>(PIN_BYTES, n - at);
                // its previous content has left (also across calls: segments are uploaded back to back)
                if (ctx->pin_busy[b]) CK(cudaEventSynchronize(ctx->pin_ev[b]));
                par_memcpy(ctx->pin[b], host + at, len);
                {
                    PhaseScope ps(ctx, PH_H2D, up);
                    CK(cudaMemcpyAsync(ctx->stage, ctx->pin[b], len, cudaMemcpyHostToDevice, up));
                    CK(cudaEventRecord(ctx->pin_ev[b], up));
                    ctx->pin_busy[b] = true;
                    ctx->h2d_bytes += len;
                }
                {
                    PhaseScope ps(ctx, ph_pack, up);
                    const uint64_t words = (len + 15) / 16;
                    const int grid = (int)std::min<uint64_t>((words + 255) / 256, (uint64_t)ctx->n_sm * 16);
                    pack_kernel<<<grid, 256, 0, up>>>(ctx->stage, len, pk + at / 16);
                    ctx->launches++;
                }
            }
            CK(cudaGetLastError());
            return IMSAME_OK;
        }
    }
    for (uint64_t at = 0; at < n; at += STAGE_BYTES) {
        const uint64_t len = std::min<uint64_t>(STAGE_BYTES, n - at);
        {
            PhaseScope ps(ctx, PH_H2D, up);
            CK(cudaMemcpyAsync(ctx->stage, host + at, len, cudaMemcpyHostToDevice, up));
            ctx->h2d_bytes += len;
        }
        {
            PhaseScope ps(ctx, ph_pack, up);
            const uint64_t words = (len + 15) / 16;
            const int grid = (int)std::min<uint64_t>((words + 255) / 256, (uint64_t)ctx->n_sm * 16);
            pack_kernel<<<grid, 256, 0, up>>>(ctx->stage, len, pk + at / 16);
            ctx->launches++;
        }
    }
    CK(cudaGetLastError());
    return IMSAME_OK;
}

int upload_u32(imsame_ctx *ctx, uint32_t *dst, const uint32_t *src, uint64_t n) {
    PhaseScope ps(ctx, PH_H2D);
    CK(cudaMemcpyAsync(dst, src, n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    ctx->h2d_bytes += n * sizeof(uint32_t);
    return IMSAME_OK;
}

int ensure_work_buffers(imsame_ctx *ctx, uint32_t want_cap) {
    if (!ctx->d_lut) {  // (the last of them: a call that ran out of memory half way completes the set next time)
        int rc;
        if (!ctx->d_small && (rc = dev_alloc(ctx, &ctx->d_small, 4))) return rc;
        if (!ctx->d_counters && (rc = dev_alloc(ctx, &ctx->d_counters, 16))) return rc;
        if (!ctx->d_overflow && (rc = dev_alloc(ctx, &ctx->d_overflow, 1))) return rc;
        if (!ctx->d_nmin && (rc = dev_alloc(ctx, &ctx->d_nmin, EXT_MAX_READ + 1))) return rc;  // every read length the scan admits
        if (!ctx->d_lmin && (rc = dev_alloc(ctx, &ctx->d_lmin, IMSAME_MAX_READ_SIZE + 1))) return rc;
        if (!ctx->d_imin && (rc = dev_alloc(ctx, &ctx->d_imin, 2 * IMSAME_MAX_READ_SIZE + 1))) return rc;
        uint32_t *d_lut = nullptr;
        if ((rc = dev_alloc(ctx, &d_lut, EXT_LUT3_SIZE))) return rc;
        std::vector<uint32_t> lut(EXT_LUT3_SIZE);
        build_ext_lut3(lut.data());
        const cudaError_t e = cudaMemcpy(d_lut, lut.data(), EXT_LUT3_SIZE * sizeof(uint32_t), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            cudaFree(d_lut);
            ctx->cuda_err = std::string("cudaMemcpy: ") + cudaGetErrorString(e);
            return IMSAME_ECUDA;
        }
        ctx->d_lut = d_lut;
    }
    if (want_cap > ctx->hcap) {
        ctx->hcap = 0;  // a failed allocation below must not leave a stale capacity behind
        dev_free(ctx->hkeys); dev_free(ctx->hvals);
        int rc;
        if ((rc = dev_alloc(ctx, &ctx->hkeys, want_cap))) return rc;
        if ((rc = dev_alloc(ctx, &ctx->hvals, want_cap))) return rc;
        ctx->hcap = want_cap;
        CK(cudaMemsetAsync(ctx->hkeys, 0xFF, (size_t)want_cap * 8, ctx->stream));
        CK(cudaMemsetAsync(ctx->hvals, 0xFF, (size_t)want_cap * 8, ctx->stream));
    }
    return IMSAME_OK;
}

// the candidate list of a whole run (all segments) lives in pairs/res; grown geometrically, contents kept
int ensure_pairs(imsame_ctx *ctx, uint64_t need) {
    if (need <= ctx->pairs_cap) return IMSAME_OK;
    uint64_t cap = std::max<uint64_t>(ctx->pairs_cap, 1u << 20);
    while (cap < need) cap += cap / 2;
    PairRec *np = nullptr;
    PairRes *nr = nullptr;
    int rc;
    if ((rc = dev_alloc(ctx, &np, cap))) return rc;
    if ((rc = dev_alloc(ctx, &nr, cap))) { cudaFree(np); return rc; }
    if (ctx->pairs && ctx->pairs_cap) {
        CK(cudaMemcpyAsync(np, ctx->pairs, ctx->pairs_cap * sizeof(PairRec), cudaMemcpyDeviceToDevice, ctx->stream));
        // (a two-pass run grows the list during its second scan, when the NW results of the first pass are in place)
        CK(cudaMemcpyAsync(nr, ctx->res, ctx->pairs_cap * sizeof(PairRes), cudaMemcpyDeviceToDevice, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->copy_stream) CK(cudaStreamSynchronize(ctx->copy_stream));  // (segment-major experiment: NW launches may run there)
    dev_free(ctx->pairs); dev_free(ctx->res);
    ctx->pairs = np; ctx->res = nr; ctx->pairs_cap = cap;
    return IMSAME_OK;
}

template <int S, bool TB>
int launch_nw(imsame_ctx *ctx, NwArgs a) {
    if (!ctx->nw_grid[S]) {
        int per_sm = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, nw_kernel<S, false>, NW_THREADS, 0));
        ctx->nw_grid[S] = std::max(1, per_sm) * ctx->n_sm;
    }
    if (!a.s_class) a.s_class = S;
    nw_kernel<S, TB><<<ctx->nw_grid[S], NW_THREADS, 0, ctx->stream>>>(a);
    ctx->launches++;
    ctx->k3_launches++;
    CK(cudaGetLastError());
    return IMSAME_OK;
}

template <bool TB>
int launch_nw_class(imsame_ctx *ctx, NwArgs a, int c) {
    int rc = IMSAME_OK;
    {
        a.s_class = c;
        switch (nw_class_cols(c)) {  // columns per lane of the class (classes 9 and 10: two passes of 5)
            case 1: rc = launch_nw<1, TB>(ctx, a); break;
            case 2: rc = launch_nw<2, TB>(ctx, a); break;
            case 3: rc = launch_nw<3, TB>(ctx, a); break;
            case 4: rc = launch_nw<4, TB>(ctx, a); break;
            case 5: rc = launch_nw<5, TB>(ctx, a); break;
            case 6: rc = launch_nw<6, TB>(ctx, a); break;
            case 7: rc = launch_nw<7, TB>(ctx, a); break;
            default: rc = launch_nw<8, TB>(ctx, a); break;
        }
    }
    return rc;
}

// packed-word kernel (nwp.cuh) of NW class c; its ~150 instantiations live in their own translation unit
// (nwp_launch.cu) so that the two halves of the library compile side by side
int launch_nwp_class(imsame_ctx *ctx, NwArgs a, int c, uint32_t ymax) {
    c = c < 1 ? 1 : (c > NW_CLASSES ? NW_CLASSES : c);
    if (!ctx->nwp_grid[c]) {
        const int per_sm = nwp_blocks_per_sm(c);
        if (per_sm < 0) { ctx->cuda_err = "cudaOccupancyMaxActiveBlocksPerMultiprocessor(nwp_kernel)"; return IMSAME_ECUDA; }
        ctx->nwp_grid[c] = std::max(1, per_sm) * ctx->n_sm;
    }
    a.s_class = c;
    a.one = 1;
    nwp_launch(c, ctx->nwp_grid[c], ctx->stream, a, ymax);
    ctx->launches++;
    ctx->k3_launches++;
    ctx->k3_packed++;
    CK(cudaGetLastError());
    return IMSAME_OK;
}

bool use_packed(const imsame_ctx *ctx, uint32_t xmax, uint32_t ymax, int igap, int egap) {
    return ctx->nw_mode != 1 && pw_eligible(xmax, ymax, igap, egap, pw_bias(xmax, ymax, igap, egap));
}

// unsorted explicit pairs: every class kernel walks the whole list and skips the other classes
template <bool TB>
int launch_nw_classes(imsame_ctx *ctx, NwArgs a, uint32_t class_mask, uint32_t *work_heads /* >= 2 * (NW_CLASSES + 1) zeroed */,
                      bool packed = false, bool mixed = false, uint32_t ymax = IMSAME_MAX_READ_SIZE) {
    int rc = IMSAME_OK;
    a.check_class = 1;
    a.mixed = (mixed && !packed && !TB) ? 1 : 0;
    for (int c = 1; c <= NW_CLASSES && !rc; c++) {
        if (!(class_mask & (1u << c))) continue;
        a.work = work_heads + c;
        if ((packed || a.mixed) && !TB) rc = launch_nwp_class(ctx, a, c, ymax);
        if (!rc && (!packed || TB)) {
            if (a.mixed) a.work = work_heads + NW_CLASSES + 1 + c;
            rc = launch_nw_class<TB>(ctx, a, c);
        }
    }
    return rc;
}

int max_nw_grid(imsame_ctx *ctx) {
    int g = 0;
    for (int c = 1; c <= 8; c++) g = std::max(g, ctx->nw_grid[c]);
    for (int c = 1; c <= NW_CLASSES; c++) g = std::max(g, 2 * ctx->nwp_grid[c]);
    return g ? g : ctx->n_sm * 8;
}

int ensure_carry(imsame_ctx *ctx, uint32_t max_ylen) {
    if (max_ylen <= 256) return IMSAME_OK;  // Y1 <= 255: classes 1..8, one pass (nw_class_of)
    // the kernels with 5..8 columns per lane run multi-pass (nw_class_of: balanced passes)
    if (!ctx->nw_grid[5]) {
        int per_sm = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, nw_kernel<5, false>, NW_THREADS, 0));
        ctx->nw_grid[5] = std::max(1, per_sm) * ctx->n_sm;
    }
    if (!ctx->nw_grid[6]) {
        int per_sm = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, nw_kernel<6, false>, NW_THREADS, 0));
        ctx->nw_grid[6] = std::max(1, per_sm) * ctx->n_sm;
    }
    if (!ctx->nw_grid[7]) {
        int per_sm = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, nw_kernel<7, false>, NW_THREADS, 0));
        ctx->nw_grid[7] = std::max(1, per_sm) * ctx->n_sm;
    }
    if (!ctx->nw_grid[8]) {
        int per_sm = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, nw_kernel<8, false>, NW_THREADS, 0));
        ctx->nw_grid[8] = std::max(1, per_sm) * ctx->n_sm;
    }
    const uint64_t warps = (uint64_t)std::max(std::max(ctx->nw_grid[5], ctx->nw_grid[6]), std::max(ctx->nw_grid[7], ctx->nw_grid[8])) * NW_WARPS;
    if (warps > ctx->carry_warps) {
        dev_free(ctx->carry);
        ctx->carry_warps = 0;  // a failed allocation below must not leave a stale capacity behind
        int rc = dev_alloc(ctx, &ctx->carry, warps * 2 * MAX_READ);
        if (rc) return rc;
        ctx->carry_warps = warps;
    }
    return IMSAME_OK;
}

uint32_t class_mask_of(const uint64_t *start, uint64_t n, uint64_t total, uint32_t *maxlen) {
    uint32_t m = 0, mx = 0;
    for (uint64_t r = 0; r < n; r++) {
        const uint64_t e = (r + 1 < n) ? start[r + 1] : total;
        const uint32_t len = (uint32_t)(e - start[r]);
        mx = std::max(mx, len);
        m |= 1u << nw_class_of(len);
    }
    *maxlen = mx;
    return m;
}

void fill_stats(imsame_ctx *ctx, imsame_stats *st, const unsigned long long *cnt) {
    if (!st) return;
    float acc[PH_COUNT] = {0};
    float t_min = 0, t_max = 0;
    bool any = false;
    cudaEvent_t first = nullptr, last = nullptr;
    for (auto &sp : ctx->spans) {
        float ms = 0;
        cudaEventElapsedTime(&ms, sp.a, sp.b);
        acc[sp.ph] += ms;
        if (!any) { first = sp.a; any = true; }
        last = sp.b;
    }
    (void)t_min; (void)t_max;
    float total = 0;
    if (any) cudaEventElapsedTime(&total, first, last);
    st->ms_pack_query = acc[PH_PACKQ]; st->ms_k1 = acc[PH_K1]; st->ms_pack_db = acc[PH_PACKDB];
    st->ms_k2 = acc[PH_K2]; st->ms_k2b = acc[PH_K2B]; st->ms_k3 = acc[PH_K3]; st->ms_select = acc[PH_SELECT];
    st->ms_h2d = acc[PH_H2D]; st->ms_d2h = acc[PH_D2H]; st->ms_total = total; st->ms_comm = acc[PH_COMM];
    st->h2d_bytes = ctx->h2d_bytes; st->d2h_bytes = ctx->d2h_bytes;
    st->k2_launches = ctx->k2_launches; st->k3_launches = ctx->k3_launches; st->total_launches = ctx->launches;
    st->k3_packed_launches = ctx->k3_packed;
    st->n_query_kmers = ctx->run_passes == 2 ? ctx->n_words_early + ctx->n_words_late : ctx->n_qwords;
    st->scan_passes = (uint32_t)ctx->run_passes;
    if (cnt) {
        st->n_db_kmers = cnt[0]; st->n_hits = cnt[1]; st->n_evalue_pass = cnt[2];
        st->n_cells = cnt[4]; st->n_pairs = cnt[5]; st->n_pairs_dp = cnt[6]; st->n_accepted = cnt[7];
    }
}

}  // namespace

// K1 over the resident packed query (ctx->q_pk ...): histogram of the words, exclusive scan, scatter of the
// table entries.  part 0 = every word: off_dst / qtab_out: build into a resident sample's own offsets table and
// hand the entries (plain allocation) to the caller; nullptr: the context's own table and the recycled pool.
// part 1 / 2 = the early / the late words of a two-pass run (qtable.cuh: QTableArgs.part) into off_early /
// qtab_early resp. off_late / qtab_late.
static int build_query_table(imsame_ctx *ctx, uint32_t *off_dst, QEntry **qtab_out, int part = 0, uint32_t e_split = 0) {
    int rc;
    const uint32_t nq = ctx->nq, total = ctx->q_total;
    const uint64_t ncodes = ncodes_of(ctx->k);
    const uint32_t n_tiles = (uint32_t)((ncodes + SCAN_TILE - 1) / SCAN_TILE);
    if (ctx->k_tables != ctx->k) {
        dev_free(ctx->off_own); dev_free(ctx->cursor); dev_free(ctx->tile_sums); dev_free(ctx->off_early); dev_free(ctx->off_late);
        ctx->off_own = ctx->cursor = ctx->tile_sums = ctx->off_early = ctx->off_late = nullptr;
        ctx->k_tables = 0;
        if ((rc = dev_alloc(ctx, &ctx->off_own, (uint64_t)ncodes + 1))) return rc;
        if ((rc = dev_alloc(ctx, &ctx->cursor, (uint64_t)ncodes + 1))) return rc;
        if ((rc = dev_alloc(ctx, &ctx->tile_sums, (uint64_t)n_tiles + 1))) return rc;
        ctx->k_tables = ctx->k;
    }
    uint32_t *off = nullptr;
    QEntry **slot = nullptr;
    if (part == 0) {
        off = off_dst ? off_dst : ctx->off_own;
        ctx->off = off;
        slot = &ctx->qtab;
    } else {
        uint32_t **o = part == 1 ? &ctx->off_early : &ctx->off_late;
        if (!*o && (rc = dev_alloc(ctx, o, (uint64_t)ncodes + 1))) return rc;
        off = *o;
        slot = part == 1 ? &ctx->qtab_early : &ctx->qtab_late;
        pool_free(ctx, *slot);  // (the table of the previous run / query)
    }
    QTableArgs a;
    a.k = ctx->k;
    a.q.pk = ctx->q_pk; a.q.start = ctx->q_start; a.q.blk = ctx->q_blk; a.q.n = nq; a.q.total = total;
    a.q.fixed_len = ctx->q_fixed;
    a.n_threads = (uint32_t)std::min<uint64_t>(ctx->q_threads, 0xFFFFFFFFull);
    a.per = (uint32_t)(nq / ctx->q_threads);  // floorl(n_seqs / n_threads), src/IMSAME.c:414
    a.cnt = ctx->cursor;
    a.qtab = nullptr;
    a.part = part; a.e_split = e_split; a.best = ctx->run_keys;
    const int grid = (int)std::min<uint64_t>(((uint64_t)total + 255) / 256, (uint64_t)ctx->n_sm * 32);
    uint32_t n_words = 0;
    {
        PhaseScope ps(ctx, PH_K1);
        CK(cudaMemsetAsync(ctx->cursor, 0, ((size_t)ncodes + 1) * 4, ctx->stream));
        qtable_kernel<0><<<grid, 256, 0, ctx->stream>>>(a);
        scan_tiles_kernel<0><<<n_tiles, SCAN_THREADS, 0, ctx->stream>>>(ctx->cursor, ncodes, ctx->tile_sums, off);
        scan_sums_kernel<<<1, SCAN_THREADS, 0, ctx->stream>>>(ctx->tile_sums, n_tiles);
        scan_tiles_kernel<2><<<n_tiles, SCAN_THREADS, 0, ctx->stream>>>(ctx->cursor, ncodes, ctx->tile_sums, off);
        ctx->launches += 4;
        CK(cudaGetLastError());
    }
    CK(cudaMemcpyAsync(&n_words, off + ncodes, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (part == 0 && qtab_out) {
        if ((rc = dev_alloc(ctx, slot, (uint64_t)n_words + 1))) return rc;
        *qtab_out = *slot;
    } else if ((rc = pool_alloc(ctx, slot, (uint64_t)n_words + 1))) {
        return rc;
    }
    {
        PhaseScope ps(ctx, PH_K1);
        CK(cudaMemcpyAsync(ctx->cursor, off, ((size_t)ncodes + 1) * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        a.qtab = *slot;
        qtable_kernel<1><<<grid, 256, 0, ctx->stream>>>(a);
        ctx->launches++;
        CK(cudaGetLastError());
    }
    if (part == 0) { ctx->n_qwords = n_words; ctx->q_k = ctx->k; ctx->tab_full = true; }
    else if (part == 1) { ctx->n_words_early = n_words; ctx->q_k = ctx->k; ctx->tab_early = true; ctx->tab_early_split = e_split; }
    else ctx->n_words_late = n_words;
    return IMSAME_OK;
}

// ------------------------------------------------------------------------------------------
extern "C" {

const char *imsame_gpu_strerror(int code) {
    switch (code) {
        case IMSAME_OK: return "ok";
        case IMSAME_ENODEV: return "no usable sm_100 CUDA device";
        case IMSAME_ECUDA: return "CUDA runtime error";
        case IMSAME_EARG: return "bad argument";
        case IMSAME_ENOMEM: return "out of memory";
        case IMSAME_EREADSIZE: return "Read size reached for gapped alignment.";
        case IMSAME_ESTATE: return "call order violated";
        case IMSAME_ELIMIT: return "input exceeds an implementation limit";
        case IMSAME_EPEER: return "another database shard failed";
        case IMSAME_ENCCL: return "NCCL unavailable or failed";
        default: return "unknown error";
    }
}

const char *imsame_gpu_last_cuda_error(const imsame_ctx *ctx) { return ctx ? ctx->cuda_err.c_str() : ""; }

int imsame_gpu_mem_info(const imsame_ctx *ctx, uint64_t *free_bytes, uint64_t *total_bytes) {
    if (!ctx || !free_bytes || !total_bytes) return IMSAME_EARG;
    size_t f = 0, t = 0;
    if (cudaSetDevice(ctx->device) != cudaSuccess || cudaMemGetInfo(&f, &t) != cudaSuccess) {
        cudaGetLastError();
        return IMSAME_ECUDA;
    }
    *free_bytes = f;
    *total_bytes = t;
    return IMSAME_OK;
}

int imsame_gpu_create(imsame_ctx **out, int device) {
    if (!out) return IMSAME_EARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return IMSAME_ENODEV;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return IMSAME_ENODEV;
    if (prop.major != 10) return IMSAME_ENODEV;  // kernels are built for sm_100a only
    if (cudaSetDevice(device) != cudaSuccess) return IMSAME_ENODEV;
    imsame_ctx *ctx = new imsame_ctx();
    ctx->device = device;
    ctx->n_sm = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return IMSAME_ECUDA; }
    if (cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->q_ready, cudaEventDisableTiming) != cudaSuccess) { delete ctx; return IMSAME_ECUDA; }
    int per_sm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, scan_kernel<K>, SCAN_THREADS_K2, 0);
    if (const char *e = getenv("IMSAME_SCAN_BLOCKS_PER_SM")) per_sm = std::min(per_sm, std::max(1, atoi(e)));  // tuning knob
    ctx->scan_grid = std::max(1, per_sm) * ctx->n_sm;
    if (const char *e = getenv("IMSAME_TEST_FAIL_ALLOC")) {  // test hook: the error paths of running out of device memory
        unsigned long long first = 0, count = 1;
        if (sscanf(e, "%llu,%llu", &first, &count) >= 1) { ctx->fail_alloc_first = first; ctx->fail_alloc_count = count; }
    }
    *out = ctx;
    return IMSAME_OK;
}

void imsame_gpu_destroy(imsame_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    free_query(ctx);
    free_db(ctx);
    pool_destroy(ctx);
    dev_free(ctx->off_own); dev_free(ctx->cursor); dev_free(ctx->tile_sums); dev_free(ctx->off_early); dev_free(ctx->off_late);
    dev_free(ctx->d_nmin); dev_free(ctx->d_lmin); dev_free(ctx->d_imin); dev_free(ctx->d_lut);
    dev_free(ctx->hkeys); dev_free(ctx->hvals); dev_free(ctx->pairs); dev_free(ctx->res);
    dev_free(ctx->d_small); dev_free(ctx->d_counters); dev_free(ctx->d_overflow);
    dev_free(ctx->keys); dev_free(ctx->payload); dev_free(ctx->pkey); dev_free(ctx->d_bins); dev_free(ctx->carry); dev_free(ctx->stage);
    dev_free(ctx->sw_best); dev_free(ctx->sw_payload); dev_free(ctx->sw_flags); dev_free(ctx->sw_lmin); dev_free(ctx->sw_imin);
    if (ctx->tb_pin) cudaFreeHost(ctx->tb_pin);
    for (int b = 0; b < 2; b++) {
        if (ctx->pin[b]) cudaFreeHost(ctx->pin[b]);
        if (ctx->pin_ev[b]) cudaEventDestroy(ctx->pin_ev[b]);
    }
    imsame_gpu_comm_free(ctx);
    dev_free(ctx->comm_flag);
    for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
    if (ctx->q_ready) cudaEventDestroy(ctx->q_ready);
    delete ctx;
}

int imsame_gpu_set_stream(imsame_ctx *ctx, void *cuda_stream) {
    if (!ctx) return IMSAME_EARG;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    if (cuda_stream) {
        ctx->stream = (cudaStream_t)cuda_stream;
        ctx->own_stream = false;
    } else {
        CK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        ctx->own_stream = true;
    }
    return IMSAME_OK;
}

void *imsame_gpu_host_alloc(uint64_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
void imsame_gpu_host_free(void *p) {
    if (p) cudaFreeHost(p);
}
void imsame_gpu_free(void *p) { free(p); }

// ---- query: upload, pack, K1 ---------------------------------------------------------------
int imsame_gpu_set_query(imsame_ctx *ctx, const imsame_seqinfo *q, const imsame_params *p) {
    if (!ctx || !q || !p || !q->sequences || !q->start_pos || q->n_seqs == 0) return IMSAME_EARG;
    if (q->total_len >= 0xFFFFFF00ull || q->n_seqs >= 0xFFFFFF00ull) return IMSAME_ELIMIT;
    cudaSetDevice(ctx->device);
    free_query(ctx);
    const uint32_t nq = (uint32_t)q->n_seqs, total = (uint32_t)q->total_len;
    for (uint64_t r = 0; r < nq; r++) {
        const uint64_t e = (r + 1 < nq) ? q->start_pos[r + 1] : q->total_len;
        if (e <= q->start_pos[r]) return IMSAME_EARG;  // empty reads break the reference's scan too
    }
    ctx->nq = nq;
    ctx->q_total = total;
    ctx->q_fixed = uniform_len(q->start_pos, nq, q->total_len);
    ctx->class_mask = class_mask_of(q->start_pos, nq, q->total_len, &ctx->q_maxlen);
    if (ctx->q_maxlen > EXT_MAX_READ) return IMSAME_ELIMIT;  // walk state packs (score, step) in 15 + 16 bits
    ctx->q_start_host.resize((size_t)nq + 1);
    for (uint32_t r = 0; r < nq; r++) ctx->q_start_host[r] = (uint32_t)q->start_pos[r];
    ctx->q_start_host[nq] = total;
    ctx->q_threads = p->n_threads ? p->n_threads : 1;

    int rc;
    const uint64_t words = ((uint64_t)total + 15) / 16 + PAD_WORDS;
    if ((rc = pool_alloc(ctx, &ctx->q_pk, words))) return rc;
    {
        cudaStream_t up = ctx->up_stream ? ctx->up_stream : ctx->stream;
        CK(cudaMemsetAsync(ctx->q_pk, 0, words * 4, up));
        if ((rc = upload_pack(ctx, q->sequences, total, ctx->q_pk, PH_PACKQ))) return rc;
        if (up != ctx->stream) {  // the query table is built on the main stream
            CK(cudaEventRecord(ctx->q_ready, up));
            CK(cudaStreamWaitEvent(ctx->stream, ctx->q_ready, 0));
        }
    }
    if (!ctx->q_fixed) {
        if ((rc = pool_alloc(ctx, &ctx->q_start, (uint64_t)nq + 1))) return rc;
        if ((rc = upload_u32(ctx, ctx->q_start, ctx->q_start_host.data(), (uint64_t)nq + 1))) return rc;
        const uint64_t nblk = ((uint64_t)total + 63) / 64 + 1;
        if ((rc = pool_alloc(ctx, &ctx->q_blk, nblk))) return rc;
        PhaseScope ps(ctx, PH_K1);
        blk_kernel<<<std::min<uint32_t>((nq + 255) / 256, ctx->n_sm * 16), 256, 0, ctx->stream>>>(ctx->q_start, nq, ctx->q_blk);
        ctx->launches++;
    }
    // the word table(s) are built by the first run on this query, which knows whether it runs in one pass (every
    // word: build_query_table part 0) or early words first (run_plan)
    ctx->q_k = ctx->k;
    ctx->have_query = true;
    return IMSAME_OK;
}

// ---- database shard: upload + pack in segments of < 2^31 bases -------------------------------
}  // extern "C"

namespace {

// segment boundaries, device buffers and the small per-segment arrays (read offsets of ragged reads, word
// breaks); the bases themselves follow segment by segment (db_upload_seg)
int db_layout(imsame_ctx *ctx, const imsame_seqinfo *db) {
    if (!ctx || !db || !db->sequences || !db->start_pos || db->n_seqs == 0) return IMSAME_EARG;
    if (db->n_seqs >= 0xFFFFFF00ull) return IMSAME_ELIMIT;
    cudaSetDevice(ctx->device);
    free_db(ctx);
    ctx->db_total = db->total_len;
    ctx->db_nseqs = db->n_seqs;
    const uint32_t fixed = uniform_len(db->start_pos, db->n_seqs, db->total_len);
    uint32_t mx = 0;
    (void)class_mask_of(db->start_pos, db->n_seqs, db->total_len, &mx);
    ctx->db_maxlen = mx;
    if (mx > EXT_MAX_READ) return IMSAME_ELIMIT;
    uint64_t seg_max = SEG_MAX_BASES;
    if (const char *e = getenv("IMSAME_TEST_SEG_BASES"))  // test hook: several segments from a small database
        seg_max = std::min<uint64_t>(seg_max, std::max<uint64_t>(std::max<uint64_t>(mx, 1), strtoull(e, nullptr, 10)));
    std::vector<uint32_t> tmp;
    uint64_t r0 = 0, bi = 0;
    while (r0 < db->n_seqs) {
        // greedy: as many whole reads as fit
        const uint64_t base = db->start_pos[r0];
        uint64_t r1;
        if (fixed) {
            r1 = std::min<uint64_t>(db->n_seqs, r0 + seg_max / fixed);
        } else {
            uint64_t lo = r0 + 1, hi = db->n_seqs;  // largest r1 with start[r1] - base <= SEG_MAX
            while (lo < hi) {
                const uint64_t mid = (lo + hi + 1) / 2;
                const uint64_t e = mid < db->n_seqs ? db->start_pos[mid] : db->total_len;
                if (e - base <= seg_max) lo = mid; else hi = mid - 1;
            }
            r1 = lo;
        }
        const uint64_t end = r1 < db->n_seqs ? db->start_pos[r1] : db->total_len;
        if (end - base > 0xFFFFFF00ull) return IMSAME_ELIMIT;  // a single read larger than a segment
        Seg s;
        s.pos_base = base; s.seq_base = r0; s.n = (uint32_t)(r1 - r0); s.total = (uint32_t)(end - base);
        s.fixed_len = fixed;
        int rc;
        const uint64_t words = ((uint64_t)s.total + 15) / 16 + PAD_WORDS;
        if ((rc = pool_alloc(ctx, &s.pk, words))) return rc;
        if (cudaEventCreateWithFlags(&s.ready, cudaEventDisableTiming) != cudaSuccess) { pool_free(ctx, s.pk); return IMSAME_ECUDA; }
        ctx->segs.push_back(s);
        Seg &ss = ctx->segs.back();
        if (!fixed) {
            tmp.resize((size_t)s.n + 1);
            for (uint64_t r = r0; r < r1; r++) tmp[r - r0] = (uint32_t)(db->start_pos[r] - base);
            tmp[s.n] = s.total;
            if ((rc = pool_alloc(ctx, &ss.start, (uint64_t)s.n + 1))) return rc;
            if ((rc = upload_u32(ctx, ss.start, tmp.data(), (uint64_t)s.n + 1))) return rc;
            CK(cudaStreamSynchronize(ctx->stream));  // tmp is reused
            const uint64_t nblk = ((uint64_t)s.total + 63) / 64 + 1;
            if ((rc = pool_alloc(ctx, &ss.blk, nblk))) return rc;
            PhaseScope ps(ctx, PH_PACKDB);
            blk_kernel<<<std::min<uint32_t>((s.n + 255) / 256, ctx->n_sm * 16), 256, 0, ctx->stream>>>(ss.start, s.n, ss.blk);
            ctx->launches++;
        }
        // word breaks that fall inside this segment
        std::vector<uint32_t> brk;
        while (bi < db->n_breaks && db->break_pos[bi] < end) {
            if (db->break_pos[bi] >= base) brk.push_back((uint32_t)(db->break_pos[bi] - base));
            bi++;
        }
        if (!brk.empty()) {
            ss.n_brk = (uint32_t)brk.size();
            if ((rc = pool_alloc(ctx, &ss.brk, brk.size()))) return rc;
            if ((rc = upload_u32(ctx, ss.brk, brk.data(), brk.size()))) return rc;
            CK(cudaStreamSynchronize(ctx->stream));
        }
        r0 = r1;
    }
    ctx->have_db = true;
    return IMSAME_OK;
}

// bases of one segment: H2D (staged) + 2-bit packing on the upload stream
int db_upload_seg(imsame_ctx *ctx, const imsame_seqinfo *db, int seg) {
    Seg &s = ctx->segs[(size_t)seg];
    cudaStream_t up = ctx->up_stream ? ctx->up_stream : ctx->stream;
    const uint64_t words = ((uint64_t)s.total + 15) / 16 + PAD_WORDS;
    CK(cudaMemsetAsync(s.pk + words - PAD_WORDS - 1, 0, (PAD_WORDS + 1) * 4, up));
    int rc = upload_pack(ctx, db->sequences + s.pos_base, s.total, s.pk, PH_PACKDB);
    if (rc) return rc;
    s.wait_ready = up != ctx->stream;
    if (s.wait_ready) CK(cudaEventRecord(s.ready, up));
    return IMSAME_OK;
}

}  // namespace

extern "C" {

int imsame_gpu_set_db(imsame_ctx *ctx, const imsame_seqinfo *db) {
    int rc = db_layout(ctx, db);
    for (int seg = 0; seg < (int)ctx->segs.size() && !rc; seg++) rc = db_upload_seg(ctx, db, seg);
    if (rc) { if (ctx) ctx->have_db = false; return rc; }
    // the caller may refill or free its (pinned) host buffers as soon as this returns
    CK(cudaStreamSynchronize(ctx->up_stream ? ctx->up_stream : ctx->stream));
    return IMSAME_OK;
}

}  // extern "C"

// ---- K2 + K2b + K3 + selection over the resident shard ----------------------------------------
// Stepping form (used by multi-GPU callers to exchange the per-read keys between bands):
//   run_begin ; for seg: run_scan(seg) ; for band: run_band(seg, band) [; all-reduce(keys, MIN)] ;
//   run_select(seg) ; run_end.   imsame_gpu_run() is exactly that sequence without the exchange.
namespace {

SeqMap query_map(const imsame_ctx *ctx) {
    SeqMap qm;
    qm.pk = ctx->q_pk; qm.start = ctx->q_start; qm.blk = ctx->q_blk; qm.n = ctx->nq; qm.total = ctx->q_total;
    qm.fixed_len = ctx->q_fixed;
    return qm;
}
SeqMap seg_map(const Seg &s) {
    SeqMap dm;
    dm.pk = s.pk; dm.start = s.start; dm.blk = s.blk; dm.n = s.n; dm.total = s.total; dm.fixed_len = s.fixed_len;
    return dm;
}

}  // namespace

extern "C" int imsame_gpu_n_segments(const imsame_ctx *ctx) { return ctx ? (int)ctx->segs.size() : 0; }
extern "C" int imsame_gpu_n_bands(void) { return NW_BANDS; }

namespace {

constexpr int EARLY_BANDS = 6;         // of NW_BANDS = 32: the words that end inside the first 3/16 of their read
constexpr double TWO_PASS_HITS = 4e9;  // expected seed hits per GPU from which a run is made in two passes

inline uint32_t band_width_of(const imsame_ctx *ctx) { return (ctx->q_maxlen + 1 + NW_BANDS - 1) / NW_BANDS; }
// logical segments of a run: database segment (ls % nseg) scanned in pass (ls / nseg)
inline int n_lsegs(const imsame_ctx *ctx) { return (int)ctx->segs.size() * ctx->run_passes; }

// "Early words first".  The reference walks the words of a query read left to right and stops at the read's first
// accepted hit (src/alignmentFunctions.c:172,189).  The band-ordered NW launches already use that (a later candidate
// of an accepted read is pruned, not aligned), but the SCAN still extended every seed hit of every word: a read that
// is in the database is usually accepted on one of its first words (76 % of the accepted reads of a 2.5x-coverage
// database within the first 32 bases, 90 % within 64), and all the hits of its ~200 later words -- a third of the
// scan's work on config 2 -- are looked at for nothing.  A two-pass run scans the database with the table of the
// EARLY words only (k-mer end inside the first EARLY_BANDS bands of the read), aligns their bands, then builds the
// table of the LATE words of the reads that are still without an accepted hit and scans again.  Exact: a read
// accepted in the first pass has a key that every later word's key exceeds (make_key: k-mer end first), and a read
// that is not is scanned with all its words.  In a sharded run the keys are reduced between the passes, so a read
// accepted in ANY shard drops out of the second pass of every shard; the decision below only uses quantities
// that are the same on every rank.
void run_plan(imsame_ctx *ctx, const imsame_params *p, bool allow_two) {
    ctx->run_passes = 1;
    ctx->run_early_bands = 0;
    if (!allow_two || ctx->q_borrowed) return;  // a resident sample brings its table of every word along
    int mode = ctx->passes_mode;
    if (!mode)
        if (const char *e = getenv("IMSAME_PASSES")) mode = atoi(e);
    if (mode == 1) return;
    int nb = EARLY_BANDS;
    if (const char *e = getenv("IMSAME_EARLY_BANDS")) nb = atoi(e);  // tuning knob
    if (nb < 1 || nb >= NW_BANDS || (uint64_t)nb * band_width_of(ctx) <= (uint64_t)ctx->q_k) return;  // no early word at all
    if (mode != 2) {
        const double db_bases = ctx->comm_size > 1 ? (double)p->db_total_len_global / ctx->comm_size : (double)ctx->db_total;
        if ((double)ctx->q_total * db_bases / (double)ncodes_of(ctx->q_k) < TWO_PASS_HITS) return;
    }
    ctx->run_passes = 2;
    ctx->run_early_bands = nb;
}

}  // namespace

static int run_begin_impl(imsame_ctx *ctx, const imsame_params *p, uint64_t *d_keys, uint64_t *d_payload, bool allow_two);

// (the caller steps through scans and bands itself: one pass over the table of every word)
extern "C" int imsame_gpu_run_begin(imsame_ctx *ctx, const imsame_params *p, uint64_t *d_keys, uint64_t *d_payload) {
    return run_begin_impl(ctx, p, d_keys, d_payload, false);
}

static int run_begin_impl(imsame_ctx *ctx, const imsame_params *p, uint64_t *d_keys, uint64_t *d_payload, bool allow_two) {
    if (!ctx || !p) return IMSAME_EARG;
    if (!ctx->have_query || !ctx->have_db) return IMSAME_ESTATE;
    cudaSetDevice(ctx->device);
    if (!ctx->in_align) reset_timing(ctx);  // a run of its own: phase times and launch counts start here
    // field widths of the key (40-bit global position) and of the payload (read index << 32, reduced as int64)
    if (p->db_pos_base + ctx->db_total >= (1ull << KEY_POS_BITS) || p->db_seq_base + ctx->db_nseqs >= (1ull << 31))
        return IMSAME_ELIMIT;
    const uint32_t nq = ctx->nq;
    int rc;
    if (ctx->keys_cap < nq) {
        dev_free(ctx->keys); dev_free(ctx->payload); dev_free(ctx->pkey);
        ctx->keys_cap = 0;  // (as in ensure_work_buffers)
        if ((rc = dev_alloc(ctx, &ctx->keys, nq))) return rc;
        if ((rc = dev_alloc(ctx, &ctx->payload, nq))) return rc;
        if ((rc = dev_alloc(ctx, &ctx->pkey, nq))) return rc;
        ctx->keys_cap = nq;
    }
    run_plan(ctx, p, allow_two);
    // the table of the first (or only) pass; the k the query was set with decides, not a later set_kmer
    if (ctx->run_passes == 2) {
        const uint32_t split = (uint32_t)ctx->run_early_bands * band_width_of(ctx);
        if ((!ctx->tab_early || ctx->tab_early_split != split) && (rc = build_query_table(ctx, nullptr, nullptr, 1, split))) return rc;
    } else if (!ctx->q_borrowed && !ctx->tab_full) {
        if ((rc = build_query_table(ctx, nullptr, nullptr))) return rc;
    }
    const uint32_t nseg = (uint32_t)n_lsegs(ctx);
    if (ctx->bins_segs < nseg) {
        dev_free(ctx->d_bins);
        ctx->bins_segs = 0;
        if ((rc = dev_alloc(ctx, &ctx->d_bins, (uint64_t)nseg * BINS_STRIDE))) return rc;
        ctx->bins_segs = nseg;
    }
    ctx->seg_pair_base.assign(nseg, 0);
    ctx->seg_pair_count.assign(nseg, 0);
    if ((rc = ensure_pairs(ctx, 32ull * nq))) return rc;
    ctx->run_keys = d_keys ? (unsigned long long *)d_keys : ctx->keys;
    ctx->run_payload = d_payload ? (unsigned long long *)d_payload : ctx->payload;
    ctx->run_params = *p;

    // pair table: the reference semantics let ~0.2-0.4 % of random hits through the e-value test
    // (idents counts every match of the walk, src/alignmentFunctions.c:323,346), i.e. ~100 candidate
    // database reads per query read against a 10 M-read database; start at 64 slots per read per
    // segment and grow on overflow (run_scan)
    uint32_t cap = 1u << 20;
    while (cap < 64ull * nq && cap < (1u << 28)) cap <<= 1;
    if (const char *e = getenv("IMSAME_TEST_PAIR_SLOTS")) {  // test hook: start small so that the growth path runs
        cap = 1u << 8;
        while (cap < (uint32_t)atoi(e)) cap <<= 1;
    }
    cap = std::max(cap, ctx->hcap);
    if ((rc = ensure_carry(ctx, ctx->q_maxlen))) return rc;
    if ((rc = ensure_work_buffers(ctx, cap))) return rc;

    // exact threshold tables (host, long double) -> device
    const uint32_t nmin_len = std::max<uint32_t>(IMSAME_MAX_READ_SIZE, ctx->q_maxlen);
    std::vector<uint16_t> nmin((size_t)nmin_len + 1), lmin(IMSAME_MAX_READ_SIZE + 1), imin(2 * IMSAME_MAX_READ_SIZE + 1);
    const uint64_t db_total_global = p->db_total_len_global ? p->db_total_len_global : ctx->db_total;
    imsame_build_nmin_upto(p->min_e_value, db_total_global, nmin.data(), nmin_len);
    imsame_build_lmin(p->min_coverage, lmin.data());
    imsame_build_imin(p->min_identity, imin.data());
    CK(cudaMemcpyAsync(ctx->d_nmin, nmin.data(), nmin.size() * 2, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_lmin, lmin.data(), lmin.size() * 2, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_imin, imin.data(), imin.size() * 2, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(ctx->d_counters, 0, 16 * sizeof(unsigned long long), ctx->stream));
    if (ctx->table_dirty) {  // the previous run ended in an error between its scan and the binning: drop its entries
        CK(cudaMemsetAsync(ctx->hkeys, 0xFF, (size_t)ctx->hcap * 8, ctx->stream));
        CK(cudaMemsetAsync(ctx->hvals, 0xFF, (size_t)ctx->hcap * 8, ctx->stream));
        ctx->table_dirty = false;
    }
    {
        PhaseScope ps(ctx, PH_SELECT);
        const int g = std::min<int>((nq + 255) / 256, ctx->n_sm * 8);
        fill_u64_kernel<<<g, 256, 0, ctx->stream>>>(ctx->run_keys, KEY_NONE, nq);
        fill_u64_kernel<<<g, 256, 0, ctx->stream>>>(ctx->pkey, KEY_NONE, nq);
        ctx->launches += 2;
        CK(cudaMemsetAsync(ctx->run_payload, 0, (size_t)nq * 8, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));  // the host tables go out of scope
    ctx->run_active = true;
    ctx->run_masked = false;
    return IMSAME_OK;
}

// K2 for one (logical) segment, asynchronously: scan, extend, collect the candidates in the pair table
static int scan_launch(imsame_ctx *ctx, int seg) {
    const int n_db_segs = (int)ctx->segs.size();
    const bool late = seg >= n_db_segs;  // second pass of a two-pass run (run_plan)
    Seg &s = ctx->segs[(size_t)(seg % n_db_segs)];
    const imsame_params *p = &ctx->run_params;
    ctx->table_dirty = true;  // until bin_kernel<1> has emptied the table again (run_begin clears it otherwise)
    if (s.wait_ready) {       // the segment was uploaded on another stream (imsame_gpu_align)
        CK(cudaStreamWaitEvent(ctx->stream, s.ready, 0));
        s.wait_ready = false;
    }
    CK(cudaMemsetAsync(ctx->d_small, 0, 4 * sizeof(uint32_t), ctx->stream));
    CK(cudaMemsetAsync(ctx->d_overflow, 0, sizeof(int), ctx->stream));
    // counters of a failed attempt must not be kept: snapshot/restore is avoided by scanning into scratch
    CK(cudaMemsetAsync(ctx->d_counters + 8, 0, 4 * sizeof(unsigned long long), ctx->stream));
    PhaseScope ps(ctx, PH_K2);
    ScanArgs a;
    a.db = seg_map(s); a.q = query_map(ctx); a.brk = s.brk; a.n_brk = s.n_brk;
    if (ctx->run_passes == 2) { a.off = late ? ctx->off_late : ctx->off_early; a.qtab = late ? ctx->qtab_late : ctx->qtab_early; }
    else { a.off = ctx->off; a.qtab = ctx->qtab; }
    a.count_words = late ? 0 : 1;  // the database words are the same in both passes
    a.nmin = ctx->d_nmin; a.lut = ctx->d_lut; a.seg_pos_base = p->db_pos_base + s.pos_base;
    a.hkeys = ctx->hkeys; a.hvals = ctx->hvals; a.hmask = ctx->hcap - 1; a.best = ctx->run_keys;
    a.counters = ctx->d_counters + 8; a.overflow = ctx->d_overflow;
    a.k = ctx->q_k;
    if (ctx->q_k == K) scan_kernel<K><<<ctx->scan_grid, SCAN_THREADS_K2, 0, ctx->stream>>>(a);
    else scan_kernel<0><<<ctx->scan_grid, SCAN_THREADS_K2, 0, ctx->stream>>>(a);
    ctx->launches++; ctx->k2_launches++;
    CK(cudaGetLastError());
    return IMSAME_OK;
}

// wait for the scan of the segment (re-running it with a larger pair table if that overflowed), then K2b: sort
// the candidates into (class, band) bins
static int scan_finish(imsame_ctx *ctx, int seg) {
    const SeqMap qm = query_map(ctx);
    int rc;
    uint32_t *bins = ctx->d_bins + (size_t)seg * BINS_STRIDE;
    uint32_t *bin_count = bins, *bin_off = bins + NW_NBINS, *launch_range = bins + 4 * NW_NBINS + 4;
    uint64_t base = 0;
    for (int k = 0; k < seg; k++) base += ctx->seg_pair_count[k];
    if (base >= 0xFFFFFFFFull) return IMSAME_ELIMIT;
    BinArgs b;
    b.q = qm;
    b.band_width = (ctx->q_maxlen + 1 + NW_BANDS - 1) / NW_BANDS;
    b.bin_count = bin_count; b.bin_off = bin_off;
    uint32_t n_seg_pairs = 0;
    int g = 0;
    // ONE host synchronisation per segment: the counting pass over the pair table is queued behind the scan right
    // away (it only reads the table), and the overflow flag comes back together with the number of candidates
    for (int attempt = 0;; attempt++) {
        b.hkeys = ctx->hkeys; b.hvals = ctx->hvals; b.n_slots = ctx->hcap; b.pairs = ctx->pairs;
        g = (int)std::min<uint32_t>((ctx->hcap + BIN_THREADS * BIN_ITEMS - 1) / (BIN_THREADS * BIN_ITEMS), (uint32_t)ctx->n_sm * 8);
        {
            PhaseScope ps(ctx, PH_K2B);
            CK(cudaMemsetAsync(bins, 0, BINS_STRIDE * sizeof(uint32_t), ctx->stream));
            bin_kernel<0><<<g, BIN_THREADS, 0, ctx->stream>>>(b);
            bin_offsets_kernel<<<1, 32, 0, ctx->stream>>>(bin_count, bin_off, launch_range, ctx->d_small,
                                                        (uint32_t)max_nw_grid(ctx) * NW_WARPS * 8u, (uint32_t)base);
            ctx->launches += 2;
        }
        int overflow = 0;
        CK(cudaMemcpyAsync(&overflow, ctx->d_overflow, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(&n_seg_pairs, ctx->d_small, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (!overflow) break;
        if (ctx->hcap >= (1u << 30) || attempt == 7) return IMSAME_ELIMIT;
        if ((rc = ensure_work_buffers(ctx, ctx->hcap * 2))) return rc;  // reallocates + clears the table
        if ((rc = scan_launch(ctx, seg))) return rc;
    }
    if (base + n_seg_pairs >= 0xFFFFFFFFull) return IMSAME_ELIMIT;
    if ((rc = ensure_pairs(ctx, base + n_seg_pairs))) return rc;
    b.pairs = ctx->pairs;
    {
        PhaseScope ps(ctx, PH_K2B);
        add_counters_kernel<<<1, 32, 0, ctx->stream>>>(ctx->d_counters, ctx->d_counters + 8, 4);  // the attempt that counted
        bin_kernel<1><<<g, BIN_THREADS, 0, ctx->stream>>>(b);
        ctx->launches += 2;
    }
    ctx->seg_pair_base[seg] = base;
    ctx->seg_pair_count[seg] = n_seg_pairs;
    CK(cudaGetLastError());
    ctx->table_dirty = false;
    return IMSAME_OK;
}

extern "C" int imsame_gpu_run_scan(imsame_ctx *ctx, int seg) {
    if (!ctx || !ctx->run_active || seg < 0 || seg >= n_lsegs(ctx)) return IMSAME_ESTATE;
    cudaSetDevice(ctx->device);
    int rc = scan_launch(ctx, seg);
    return rc ? rc : scan_finish(ctx, seg);
}

// K3 for one band of one segment (every NW class present in the query)
extern "C" int imsame_gpu_run_band(imsame_ctx *ctx, int seg, int band) {
    if (!ctx || !ctx->run_active || seg < 0 || seg >= n_lsegs(ctx) || band < 0 || band >= NW_BANDS)
        return IMSAME_ESTATE;
    cudaSetDevice(ctx->device);
    const imsame_params *p = &ctx->run_params;
    const Seg &dbseg = ctx->segs[(size_t)seg % ctx->segs.size()];
    uint32_t *bins = ctx->d_bins + (size_t)seg * BINS_STRIDE;
    uint32_t *bin_work = bins + 3 * NW_NBINS + 4, *launch_range = bins + 4 * NW_NBINS + 4;
    PhaseScope ps(ctx, PH_K3);
    NwArgs a;
    a.db = seg_map(dbseg); a.q = query_map(ctx); a.pairs = ctx->pairs; a.res = ctx->res;
    a.igap = p->igap; a.egap = p->egap; a.lmin = ctx->d_lmin; a.imin = ctx->d_imin;
    a.best = ctx->run_keys; a.cells = ctx->d_counters + 4; a.carry = ctx->carry; a.s_class = 0;
    a.tb = nullptr; a.tb_off = nullptr; a.check_class = 0;
    int rc;
    const bool packed = use_packed(ctx, ctx->db_maxlen, ctx->q_maxlen, p->igap, p->egap);
    // some reads too long for packed words: the two kernels share every bin, pair by pair (NwArgs.mixed)
    const bool mixed = !packed && ctx->nw_mode != 1 && p->igap <= 0 && p->egap <= 0;
    uint32_t *bin_work2 = bins + 6 * NW_NBINS + 8;
    a.mixed = mixed ? 1 : 0;
    a.pw_bias = pw_bias(ctx->db_maxlen, ctx->q_maxlen, p->igap, p->egap);
    for (int c = 1; c <= NW_CLASSES; c++) {
        if (!(ctx->class_mask & (1u << c))) continue;
        const int bin = c * NW_BANDS + band;
        a.range = launch_range + 2 * bin;
        a.work = bin_work + bin;
        if (packed || mixed) { if ((rc = launch_nwp_class(ctx, a, c, ctx->q_maxlen))) return rc; }
        if (!packed) {
            if (mixed) a.work = bin_work2 + bin;
            if ((rc = launch_nw_class<false>(ctx, a, c))) return rc;
        }
    }
    return IMSAME_OK;
}

// record fields of the pairs of this segment that currently own their read's key
extern "C" int imsame_gpu_run_select(imsame_ctx *ctx, int seg) {
    if (!ctx || !ctx->run_active || seg < 0 || seg >= n_lsegs(ctx)) return IMSAME_ESTATE;
    cudaSetDevice(ctx->device);
    const Seg &dbseg = ctx->segs[(size_t)seg % ctx->segs.size()];
    PhaseScope ps(ctx, PH_SELECT);
    select_kernel<<<ctx->n_sm * 8, 256, 0, ctx->stream>>>(ctx->pairs + ctx->seg_pair_base[seg],
                                                        ctx->res + ctx->seg_pair_base[seg],
                                                        (uint32_t)ctx->seg_pair_count[seg], ctx->run_keys,
                                                        ctx->run_payload, ctx->pkey,
                                                        ctx->run_params.db_seq_base + dbseg.seq_base,
                                                        ctx->d_counters + 5);
    ctx->launches++;
    if (ctx->db_maxlen > IMSAME_MAX_READ_SIZE || ctx->q_maxlen > IMSAME_MAX_READ_SIZE) {
        // the keys are final here (all bands done, and exchanged between shards in a stepped run)
        readsize_kernel<<<ctx->n_sm * 8, 256, 0, ctx->stream>>>(ctx->pairs + ctx->seg_pair_base[seg],
                                                              (uint32_t)ctx->seg_pair_count[seg], seg_map(dbseg),
                                                              query_map(ctx), ctx->run_keys, ctx->d_counters + 12);
        ctx->launches++;
    }
    CK(cudaGetLastError());
    return IMSAME_OK;
}

// drop payloads that a later, smaller key (another segment or, after a reduction, another shard) superseded
static int run_mask(imsame_ctx *ctx) {
    if (ctx->run_masked) return IMSAME_OK;
    PhaseScope ps(ctx, PH_SELECT);
    mask_payload_kernel<<<ctx->n_sm * 4, 256, 0, ctx->stream>>>(ctx->run_keys, ctx->pkey, ctx->run_payload, ctx->nq);
    ctx->launches++;
    ctx->run_masked = true;
    CK(cudaGetLastError());
    return IMSAME_OK;
}

extern "C" int imsame_gpu_run_end(imsame_ctx *ctx, imsame_stats *st) {
    if (!ctx || !ctx->run_active) return IMSAME_ESTATE;
    cudaSetDevice(ctx->device);
    {
        int rc = run_mask(ctx);
        if (rc) return rc;
    }
    unsigned long long cnt[13] = {0};
    CK(cudaMemcpyAsync(cnt, ctx->d_counters, sizeof(cnt), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->run_active = false;
    // an over-long read reached NW before its query read was accepted (readsize_kernel, src/alignmentFunctions.c:155)
    if (cnt[12]) return IMSAME_EREADSIZE;
    fill_stats(ctx, st, cnt);
    if (getenv("IMSAME_TRACE"))
        fprintf(stderr, "[imsame] candidate pairs %llu, aligned %llu, not after their read's final hit in scan order %llu\n",
                cnt[5], cnt[6], cnt[7]);
    return IMSAME_OK;
}

// EXPERIMENT (IMSAME_SEGMENT_MAJOR = 1 | 2, measured in DESIGN.md 9.2, not the default): the NW launches of segment s
// run right after its scan -- 2: on the copy stream, i.e. concurrently with the scan of segment s + 1.  Segment-major
// order gives up the pruning across segments of the band-major order below; results are the same.  (The candidate
// buffers must have reached their final size: run once in the default order first.)
static int run_segment_major(imsame_ctx *ctx, imsame_stats *st, bool concurrent) {
    int rc;
    const int nseg = (int)ctx->segs.size();
    cudaEvent_t ev = nullptr;
    if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) return IMSAME_ECUDA;
    cudaStream_t main_stream = ctx->stream;
    for (int seg = 0; seg < nseg; seg++) {
        if ((rc = imsame_gpu_run_scan(ctx, seg))) break;
        if (concurrent) {
            cudaEventRecord(ev, main_stream);
            cudaStreamWaitEvent(ctx->copy_stream, ev, 0);
            ctx->stream = ctx->copy_stream;
        }
        for (int band = 0; band < NW_BANDS && !rc; band++) rc = imsame_gpu_run_band(ctx, seg, band);
        ctx->stream = main_stream;
        if (rc) break;
    }
    if (concurrent) {
        cudaEventRecord(ev, ctx->copy_stream);
        cudaStreamWaitEvent(main_stream, ev, 0);
    }
    cudaEventDestroy(ev);
    if (rc) return rc;
    for (int seg = 0; seg < nseg; seg++)
        if ((rc = imsame_gpu_run_select(ctx, seg))) return rc;
    return imsame_gpu_run_end(ctx, st);
}

// second pass of a two-pass run (run_plan), after the NW launches of the early bands: the table of the late words
// of the reads that have no accepted hit yet (their keys are in run_keys; reduced over the shards by then in a
// sharded run), and the scans of every database segment against it (logical segments nseg .. 2 nseg - 1)
static int late_pass_scans(imsame_ctx *ctx) {
    int rc;
    const int nseg = (int)ctx->segs.size();
    if ((rc = build_query_table(ctx, nullptr, nullptr, 2, (uint32_t)ctx->run_early_bands * band_width_of(ctx)))) return rc;
    for (int seg = 0; seg < nseg; seg++)
        if ((rc = imsame_gpu_run_scan(ctx, nseg + seg))) return rc;
    return IMSAME_OK;
}

// everything after the scans of the first (or only) pass: NW launches in ascending band order over ALL segments (an
// accepted early candidate prunes the read's later ones), in a two-pass run with the second scan after the early
// bands; the candidates of the first pass all lie in the early bands, those of the second pass in the later ones
// (bands merged into one launch for want of candidates start at launch 0: every launch is issued for them)
static int run_bands_and_finish(imsame_ctx *ctx, imsame_stats *st) {
    int rc;
    const int nseg = (int)ctx->segs.size();
    const bool two = ctx->run_passes == 2;
    for (int band = 0; band < (two ? ctx->run_early_bands : NW_BANDS); band++)
        for (int seg = 0; seg < nseg; seg++)
            if ((rc = imsame_gpu_run_band(ctx, seg, band))) return rc;
    if (two) {
        if ((rc = late_pass_scans(ctx))) return rc;
        for (int band = 0; band < NW_BANDS; band++)
            for (int seg = 0; seg < nseg; seg++)
                if ((rc = imsame_gpu_run_band(ctx, nseg + seg, band))) return rc;
    }
    for (int seg = 0; seg < n_lsegs(ctx); seg++)
        if ((rc = imsame_gpu_run_select(ctx, seg))) return rc;
    return imsame_gpu_run_end(ctx, st);
}

static int run_impl(imsame_ctx *ctx, const imsame_params *p, uint64_t *d_keys, uint64_t *d_payload,
                    imsame_stats *st) {
    int rc;
    const char *sm = getenv("IMSAME_SEGMENT_MAJOR");
    const bool segment_major = sm && atoi(sm) > 0 && !ctx->in_align;
    if ((rc = run_begin_impl(ctx, p, d_keys, d_payload, !segment_major))) return rc;
    const int nseg = (int)ctx->segs.size();
    if (segment_major) return run_segment_major(ctx, st, atoi(sm) == 2);
    for (int seg = 0; seg < nseg; seg++)
        if ((rc = imsame_gpu_run_scan(ctx, seg))) return rc;
    return run_bands_and_finish(ctx, st);
}

extern "C" {

int imsame_gpu_run(imsame_ctx *ctx, const imsame_params *p, uint64_t *d_keys, uint64_t *d_payload,
                   imsame_stats *st) {
    if (!ctx || !p) return IMSAME_EARG;
    return run_impl(ctx, p, d_keys, d_payload, st);
}

int imsame_gpu_set_kmer(imsame_ctx *ctx, int k) {
    if (!ctx || k < K_MIN || k > K_MAX) return IMSAME_EARG;
    if (ctx->run_active) return IMSAME_ESTATE;
    if (k != ctx->k) ctx->have_query = false;  // the resident word table belongs to the old length
    ctx->k = k;
    return IMSAME_OK;
}

int imsame_gpu_set_passes(imsame_ctx *ctx, int mode) {
    if (!ctx || mode < 0 || mode > 2) return IMSAME_EARG;
    if (ctx->run_active) return IMSAME_ESTATE;
    ctx->passes_mode = mode;
    return IMSAME_OK;
}

int imsame_gpu_set_nw_mode(imsame_ctx *ctx, int mode) {
    if (!ctx || mode < 0 || mode > 1) return IMSAME_EARG;
    ctx->nw_mode = mode;
    return IMSAME_OK;
}

int imsame_gpu_mask_payload(imsame_ctx *ctx, const uint64_t *reduced, const uint64_t *local, uint64_t *payload) {
    if (!ctx || !reduced || !local || !payload) return IMSAME_EARG;
    cudaSetDevice(ctx->device);
    mask_payload_kernel<<<ctx->n_sm * 4, 256, 0, ctx->stream>>>((const unsigned long long *)reduced,
                                                              (const unsigned long long *)local,
                                                              (unsigned long long *)payload, ctx->nq);
    ctx->launches++;
    CK(cudaGetLastError());
    return IMSAME_OK;
}

int imsame_gpu_fetch(imsame_ctx *ctx, const uint64_t *d_keys, const uint64_t *d_payload, imsame_best *out) {
    if (!ctx || !out) return IMSAME_EARG;
    if (!ctx->have_query) return IMSAME_ESTATE;
    cudaSetDevice(ctx->device);
    const uint64_t *k = d_keys ? d_keys : (const uint64_t *)ctx->keys;
    const uint64_t *pl = d_payload ? d_payload : (const uint64_t *)ctx->payload;
    if (!k || !pl) return IMSAME_ESTATE;
    const uint32_t nq = ctx->nq;
    std::vector<uint64_t> hk(nq), hp(nq);
    {
        PhaseScope ps(ctx, PH_D2H);
        CK(cudaMemcpyAsync(hk.data(), k, (size_t)nq * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(hp.data(), pl, (size_t)nq * 8, cudaMemcpyDeviceToHost, ctx->stream));
        ctx->d2h_bytes += (uint64_t)nq * 16;
    }
    CK(cudaStreamSynchronize(ctx->stream));
    for (uint32_t r = 0; r < nq; r++) {
        imsame_best b;
        memset(&b, 0, sizeof(b));
        if (hk[r] != KEY_NONE) {
            b.accepted = 1;
            b.qpos_end = (uint64_t)ctx->q_start_host[r] + key_erel(hk[r]) - 1;
            b.db_pos = key_dbpos(hk[r]);
            b.db_seq = hp[r] >> 32;
            b.length = (uint32_t)(hp[r] >> 16) & 0xFFFFu;
            b.identities = (uint32_t)hp[r] & 0xFFFFu;
        }
        out[r] = b;
    }
    return IMSAME_OK;
}

// One call = index build (src/IMSAME.c:232-281) + thread fan-out (:409-467).  The uploads run on a stream of
// their own, one database segment ahead of the scan: H2D + packing of segment s+1 overlap K2 of segment s
// (SURVEY 8(f) rank 2: the reference reads and indexes its whole database before the first alignment starts,
// src/IMSAME.c:196-289).
static int align_pipelined(imsame_ctx *ctx, const imsame_seqinfo *db, const imsame_seqinfo *query,
                           const imsame_params *p, imsame_stats *local) {
    int rc;
    if ((rc = imsame_gpu_set_query(ctx, query, p))) return rc;
    if ((rc = db_layout(ctx, db))) return rc;
    if ((rc = run_begin_impl(ctx, p, nullptr, nullptr, true))) return rc;
    const int nseg = (int)ctx->segs.size();
    if ((rc = db_upload_seg(ctx, db, 0))) return rc;
    for (int seg = 0; seg < nseg; seg++) {
        if ((rc = scan_launch(ctx, seg))) return rc;
        // issued while the scan runs; pageable input keeps the host busy here (pinned bounce buffers)
        if (seg + 1 < nseg && (rc = db_upload_seg(ctx, db, seg + 1))) return rc;
        if ((rc = scan_finish(ctx, seg))) return rc;
    }
    return run_bands_and_finish(ctx, local);
}

int imsame_gpu_align(imsame_ctx *ctx, const imsame_seqinfo *db, const imsame_seqinfo *query,
                     const imsame_params *p, imsame_best *out, imsame_stats *st) {
    if (!ctx || !db || !query || !p || !out) return IMSAME_EARG;
    cudaSetDevice(ctx->device);
    reset_timing(ctx);
    const bool trace = getenv("IMSAME_TRACE") != nullptr;
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t0 = now();
    imsame_stats local;
    memset(&local, 0, sizeof(local));
    ctx->in_align = true;
    ctx->up_stream = ctx->copy_stream;
    int rc = align_pipelined(ctx, db, query, p, &local);
    ctx->up_stream = nullptr;
    ctx->in_align = false;
    ctx->run_active = false;
    // nothing of the caller's buffers is in flight when this returns, whatever happened
    cudaStreamSynchronize(ctx->copy_stream);
    for (Seg &s : ctx->segs) s.wait_ready = false;
    if (rc) { ctx->have_db = false; return rc; }
    ctx->last_align = 1;
    ctx->align_params = *p;
    const double t3 = now();
    if ((rc = imsame_gpu_fetch(ctx, nullptr, nullptr, out))) return rc;
    if (trace) fprintf(stderr, "[imsame] host wall ms: upload + table + scan + NW %.1f  fetch %.1f\n", t3 - t0, now() - t3);
    uint64_t acc = 0;
    for (uint32_t r = 0; r < ctx->nq; r++) acc += out[r].accepted;
    if (st) {
        unsigned long long cnt[8];
        cudaMemcpy(cnt, ctx->d_counters, sizeof(cnt), cudaMemcpyDeviceToHost);
        fill_stats(ctx, st, cnt);
        st->n_accepted = acc;
    }
    return IMSAME_OK;
}


}  // extern "C"

// ---- explicit pairs: shared by imsame_gpu_nw_batch and imsame_gpu_traceback -------------------
namespace {

struct PairBatch {
    imsame_ctx *ctx;
    uint32_t n = 0, class_mask = 0, ymax = 0, xmax = 0;
    uint32_t *xpk = nullptr, *ypk = nullptr, *dxs = nullptr, *dys = nullptr, *dsmall = nullptr;
    PairRec *dp = nullptr;
    PairRes *dr = nullptr;
    uint16_t *dz = nullptr;
    unsigned long long *dcells = nullptr;
    std::vector<uint32_t> xs, ys;
    explicit PairBatch(imsame_ctx *c) : ctx(c) {}
    ~PairBatch() {  // blocks go back to the context's pool: the next batch / call reuses them
        pool_free(ctx, xpk); pool_free(ctx, ypk); pool_free(ctx, dxs); pool_free(ctx, dys); pool_free(ctx, dsmall);
        pool_free(ctx, dp); pool_free(ctx, dr); pool_free(ctx, dz); pool_free(ctx, dcells);
    }
    // X[i]/Y[i] ASCII reads -> packed device arrays + pair list (r = s = i)
    int upload(uint32_t n_pairs, const unsigned char *const *X, const uint32_t *xlen, const unsigned char *const *Y,
               const uint32_t *ylen) {
        n = n_pairs;
        xs.resize((size_t)n + 1);
        ys.resize((size_t)n + 1);
        uint64_t xt = 0, yt = 0;
        for (uint32_t i = 0; i < n; i++) {
            if (xlen[i] > IMSAME_MAX_READ_SIZE || ylen[i] > IMSAME_MAX_READ_SIZE) return IMSAME_EREADSIZE;
            if (xlen[i] == 0 || ylen[i] == 0) return IMSAME_EARG;
            xs[i] = (uint32_t)xt; ys[i] = (uint32_t)yt;
            xt += xlen[i]; yt += ylen[i];
            class_mask |= 1u << nw_class_of(ylen[i]);
            ymax = std::max(ymax, ylen[i]);
            xmax = std::max(xmax, xlen[i]);
        }
        if (xt >= 0xFFFFFF00ull || yt >= 0xFFFFFF00ull) return IMSAME_ELIMIT;
        xs[n] = (uint32_t)xt; ys[n] = (uint32_t)yt;
        std::vector<unsigned char> xa(xt), ya(yt);
        for (uint32_t i = 0; i < n; i++) {
            memcpy(xa.data() + xs[i], X[i], xlen[i]);
            memcpy(ya.data() + ys[i], Y[i], ylen[i]);
        }
        int rc;
        const uint64_t xw = (xt + 15) / 16 + PAD_WORDS, yw = (yt + 15) / 16 + PAD_WORDS;
        if ((rc = pool_alloc(ctx, &xpk, xw)) || (rc = pool_alloc(ctx, &ypk, yw)) ||
            (rc = pool_alloc(ctx, &dxs, (uint64_t)n + 1)) || (rc = pool_alloc(ctx, &dys, (uint64_t)n + 1)) ||
            (rc = pool_alloc(ctx, &dsmall, 32)) || (rc = pool_alloc(ctx, &dp, n)) || (rc = pool_alloc(ctx, &dr, n)) ||
            (rc = pool_alloc(ctx, &dz, 2 * IMSAME_MAX_READ_SIZE + 1)) || (rc = pool_alloc(ctx, &dcells, 4)))
            return rc;
        CK(cudaMemsetAsync(xpk, 0, xw * 4, ctx->stream));
        CK(cudaMemsetAsync(ypk, 0, yw * 4, ctx->stream));
        CK(cudaMemsetAsync(dz, 0, (2 * IMSAME_MAX_READ_SIZE + 1) * 2, ctx->stream));
        CK(cudaMemsetAsync(dcells, 0, 32, ctx->stream));
        if ((rc = upload_pack(ctx, xa.data(), xt, xpk, PH_PACKDB))) return rc;
        CK(cudaStreamSynchronize(ctx->stream));  // the staging buffer and xa are reused
        if ((rc = upload_pack(ctx, ya.data(), yt, ypk, PH_PACKQ))) return rc;
        std::vector<PairRec> hp(n);
        for (uint32_t i = 0; i < n; i++) { hp[i].r = i; hp[i].s = i; hp[i].key = 0; }
        uint32_t small[32] = {0};
        small[1] = n;  // range = [0, n); small[4..] = per-class work heads
        CK(cudaMemcpyAsync(dxs, xs.data(), ((size_t)n + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(dys, ys.data(), ((size_t)n + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(dp, hp.data(), (size_t)n * sizeof(PairRec), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(dsmall, small, sizeof(small), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));  // host vectors go out of scope
        return ensure_carry(ctx, ymax);
    }
    NwArgs args(int igap, int egap) const {
        NwArgs a;
        a.db.pk = xpk; a.db.start = dxs; a.db.blk = nullptr; a.db.n = n; a.db.total = xs[n]; a.db.fixed_len = 0;
        a.q.pk = ypk; a.q.start = dys; a.q.blk = nullptr; a.q.n = n; a.q.total = ys[n]; a.q.fixed_len = 0;
        a.pairs = dp; a.res = dr; a.range = dsmall; a.work = dsmall + 4; a.igap = igap; a.egap = egap;
        a.lmin = dz; a.imin = dz; a.best = nullptr; a.cells = dcells; a.carry = ctx->carry; a.s_class = 0;
        a.tb = nullptr; a.tb_off = nullptr;
        a.check_class = 1;
        a.mixed = 0;
        a.pw_bias = pw_bias(xmax, ymax, igap, egap);
        return a;
    }
};

}  // namespace

extern "C" {

// ---- NW on explicit pairs (src/alignmentFunctions.c:389-560 in isolation) -----------------------
int imsame_gpu_nw_batch(imsame_ctx *ctx, uint32_t n_pairs, const unsigned char *const *X, const uint32_t *xlen,
                        const unsigned char *const *Y, const uint32_t *ylen, int igap, int egap, int32_t *out5,
                        float *ms_kernel) {
    if (!ctx || !X || !Y || !xlen || !ylen || !out5) return IMSAME_EARG;
    if (n_pairs == 0) return IMSAME_OK;
    cudaSetDevice(ctx->device);
    PairBatch pb(ctx);
    int rc;
    if ((rc = pb.upload(n_pairs, X, xlen, Y, ylen))) return rc;
    NwArgs a = pb.args(igap, egap);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    cudaEventRecord(e0, ctx->stream);
    rc = launch_nw_classes<false>(ctx, a, pb.class_mask, pb.dsmall + 4, use_packed(ctx, pb.xmax, pb.ymax, igap, egap),
                                  ctx->nw_mode != 1 && igap <= 0 && egap <= 0, pb.ymax);
    cudaEventRecord(e1, ctx->stream);
    std::vector<PairRes> hr(n_pairs);
    if (!rc) {
        cudaError_t ce = cudaMemcpyAsync(hr.data(), pb.dr, (size_t)n_pairs * sizeof(PairRes), cudaMemcpyDeviceToHost, ctx->stream);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
        if (ce != cudaSuccess) { ctx->cuda_err = cudaGetErrorString(ce); rc = IMSAME_ECUDA; }
    }
    if (!rc && ms_kernel) cudaEventElapsedTime(ms_kernel, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (rc) return rc;
    for (uint32_t i = 0; i < n_pairs; i++) {
        out5[5 * i + 0] = hr[i].score;
        out5[5 * i + 1] = (int32_t)hr[i].bx;
        out5[5 * i + 2] = (int32_t)hr[i].by;
        out5[5 * i + 3] = (int32_t)((hr[i].stats & 0x7FFFFFFFu) >> 16);
        out5[5 * i + 4] = (int32_t)(hr[i].stats & 0xFFFFu);
    }
    return IMSAME_OK;
}

// ---- winners-only traceback (src/alignmentFunctions.c:493-546) ----------------------------------
int imsame_gpu_traceback(imsame_ctx *ctx, const imsame_seqinfo *db, const imsame_seqinfo *query,
                         const imsame_params *p, const imsame_best *best, uint64_t *ops_off, uint32_t **ops_out,
                         uint32_t *cell_xy) {
    if (!ctx || !db || !query || !p || !best || !ops_off || !ops_out || !cell_xy) return IMSAME_EARG;
    cudaSetDevice(ctx->device);
    const uint64_t nq = query->n_seqs;
    constexpr uint64_t TB_BUDGET = 3ull << 30;  // bytes of back-pointer codes per batch
    std::vector<uint32_t> all_ops;
    std::vector<uint64_t> winners;
    for (uint64_t r = 0; r < nq; r++) {
        ops_off[r] = 0;
        cell_xy[4 * r] = cell_xy[4 * r + 1] = cell_xy[4 * r + 2] = cell_xy[4 * r + 3] = 0;
        if (best[r].accepted) {
            if (best[r].db_seq < p->db_seq_base || best[r].db_seq - p->db_seq_base >= db->n_seqs) return IMSAME_EARG;
            winners.push_back(r);
        }
    }
    std::vector<uint64_t> n_ops_of(nq, 0);
    const bool trace = getenv("IMSAME_TRACE") != nullptr;
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double t_prep = 0, t_upload = 0, t_gpu = 0, t_merge = 0;
    // everything that comes back goes through ONE pinned buffer kept in the context (a cudaMallocHost per call
    // cost more than the kernels of a 100 k-read comparison)
    auto pinned = [&](uint64_t words) -> uint32_t * {
        if (words > ctx->tb_pin_cap) {
            if (ctx->tb_pin) cudaFreeHost(ctx->tb_pin);
            ctx->tb_pin = nullptr; ctx->tb_pin_cap = 0;
            const uint64_t cap = words + words / 4 + 1024;
            if (cudaMallocHost((void **)&ctx->tb_pin, (size_t)cap * 4) != cudaSuccess) { cudaGetLastError(); ctx->tb_pin = nullptr; return nullptr; }
            ctx->tb_pin_cap = cap;
        }
        return ctx->tb_pin;
    };
    size_t w0 = 0;
    while (w0 < winners.size()) {
        double t0 = now();
        // batch: as many winners as fit the table budget
        std::vector<const unsigned char *> X, Y;
        std::vector<uint32_t> xl, yl, strides;
        std::vector<uint64_t> tb_off, op_off;
        uint64_t tb_elems = 0, op_elems = 0;
        size_t w1 = w0;
        {
            const size_t guess = std::min<size_t>(winners.size() - w0, 1u << 20);
            X.reserve(guess); Y.reserve(guess); xl.reserve(guess); yl.reserve(guess); strides.reserve(guess);
            tb_off.reserve(guess); op_off.reserve(guess);
        }
        while (w1 < winners.size()) {
            const uint64_t r = winners[w1], s = best[r].db_seq - p->db_seq_base;
            const uint64_t xe = s + 1 < db->n_seqs ? db->start_pos[s + 1] : db->total_len;
            const uint64_t ye = r + 1 < nq ? query->start_pos[r + 1] : query->total_len;
            const uint32_t xlen = (uint32_t)(xe - db->start_pos[s]), ylen = (uint32_t)(ye - query->start_pos[r]);
            if (xlen > IMSAME_MAX_READ_SIZE || ylen > IMSAME_MAX_READ_SIZE) return IMSAME_EREADSIZE;
            const uint32_t stride = tb_stride(ylen, 8);  // every pair runs in the 8-columns-per-lane kernel (16-byte code stores)
            const uint64_t need = (uint64_t)(xlen > 1 ? xlen - 1 : 1) * stride;
            if (w1 > w0 && (tb_elems + need) * 2 > TB_BUDGET) break;
            X.push_back(db->sequences + db->start_pos[s]);
            Y.push_back(query->sequences + query->start_pos[r]);
            xl.push_back(xlen); yl.push_back(ylen); strides.push_back(stride);
            tb_off.push_back(tb_elems); op_off.push_back(op_elems);
            tb_elems += need;
            op_elems += (uint64_t)xlen + ylen + 2;
            w1++;
        }
        const uint32_t nb = (uint32_t)(w1 - w0);
        t_prep += now() - t0; t0 = now();
        PairBatch pb(ctx);
        int rc;
        if ((rc = pb.upload(nb, X.data(), xl.data(), Y.data(), yl.data()))) return rc;
        t_upload += now() - t0; t0 = now();
        uint16_t *d_tb = nullptr;
        uint64_t *d_tboff = nullptr, *d_opoff = nullptr;
        uint32_t *d_str = nullptr, *d_ops = nullptr, *d_nops = nullptr, *d_end = nullptr, *d_coff = nullptr, *d_tiles = nullptr,
                 *d_cops = nullptr;
        const uint32_t n_tiles = (nb + SCAN_TILE - 1) / SCAN_TILE;
        // recycled blocks (pool): a cudaMalloc + cudaFree of the 3 GB table per batch cost 0.1 - 3 s each
        auto cleanup = [&]() {
            pool_free(ctx, d_tb); pool_free(ctx, d_tboff); pool_free(ctx, d_opoff); pool_free(ctx, d_str); pool_free(ctx, d_ops);
            pool_free(ctx, d_nops); pool_free(ctx, d_end); pool_free(ctx, d_coff); pool_free(ctx, d_tiles); pool_free(ctx, d_cops);
        };
        if ((rc = pool_alloc(ctx, &d_tb, tb_elems)) || (rc = pool_alloc(ctx, &d_tboff, nb)) || (rc = pool_alloc(ctx, &d_opoff, nb)) ||
            (rc = pool_alloc(ctx, &d_str, nb)) || (rc = pool_alloc(ctx, &d_ops, op_elems)) || (rc = pool_alloc(ctx, &d_nops, nb)) ||
            (rc = pool_alloc(ctx, &d_end, 2ull * nb)) || (rc = pool_alloc(ctx, &d_coff, (uint64_t)nb + 1)) ||
            (rc = pool_alloc(ctx, &d_tiles, (uint64_t)n_tiles + 1))) { cleanup(); return rc; }
        {
            cudaError_t up = cudaMemcpyAsync(d_tboff, tb_off.data(), (size_t)nb * 8, cudaMemcpyHostToDevice, ctx->stream);
            if (up == cudaSuccess) up = cudaMemcpyAsync(d_opoff, op_off.data(), (size_t)nb * 8, cudaMemcpyHostToDevice, ctx->stream);
            if (up == cudaSuccess) up = cudaMemcpyAsync(d_str, strides.data(), (size_t)nb * 4, cudaMemcpyHostToDevice, ctx->stream);
            if (up != cudaSuccess) {
                ctx->cuda_err = std::string("imsame_gpu_traceback: cudaMemcpyAsync: ") + cudaGetErrorString(up);
                cleanup();
                return IMSAME_ECUDA;
            }
        }
        NwArgs a = pb.args(p->igap, p->egap);
        a.tb = d_tb;
        a.tb_off = d_tboff;
        a.check_class = 0;
        a.work = pb.dsmall + 4;
        rc = launch_nw<8, true>(ctx, a);
        if (!rc) {
            tb_walk_kernel<<<std::min<uint32_t>((nb + 127) / 128, (uint32_t)ctx->n_sm * 8), 128, 0, ctx->stream>>>(
                pb.dr, d_tb, d_tboff, d_str, nb, d_ops, d_opoff, d_nops, d_end);
            // compact offsets of the ops actually used = exclusive scan of n_ops
            scan_tiles_kernel<0><<<n_tiles, SCAN_THREADS, 0, ctx->stream>>>(d_nops, nb, d_tiles, d_coff);
            scan_sums_kernel<<<1, SCAN_THREADS, 0, ctx->stream>>>(d_tiles, n_tiles);
            scan_tiles_kernel<2><<<n_tiles, SCAN_THREADS, 0, ctx->stream>>>(d_nops, nb, d_tiles, d_coff);
            ctx->launches += 4;
        }
        // pinned layout: [compact offsets nb + 1 | n_ops nb | end cells 2 nb | PairRes 4 nb | compact ops ...]
        const uint64_t fixed_words = (uint64_t)nb + 1 + nb + 2ull * nb + 4ull * nb;
        cudaError_t ce = cudaGetLastError();
        uint32_t *h = (!rc && ce == cudaSuccess) ? pinned(fixed_words + op_elems / 8 + 1024) : nullptr;
        if (!rc && ce == cudaSuccess && !h) { cleanup(); return IMSAME_ENOMEM; }
        uint32_t *h_coff = h, *h_nops = h ? h + nb + 1 : nullptr, *h_end = h ? h_nops + nb : nullptr;
        PairRes *h_res = h ? reinterpret_cast<PairRes *>(h_end + 2ull * nb) : nullptr;
        static_assert(sizeof(PairRes) == 16, "PairRes is copied as four words");
        if (!rc && ce == cudaSuccess) ce = cudaMemcpyAsync(h_coff, d_coff, ((size_t)nb + 1) * 4, cudaMemcpyDeviceToHost, ctx->stream);
        if (!rc && ce == cudaSuccess) ce = cudaMemcpyAsync(h_nops, d_nops, (size_t)nb * 4, cudaMemcpyDeviceToHost, ctx->stream);
        if (!rc && ce == cudaSuccess) ce = cudaMemcpyAsync(h_end, d_end, (size_t)nb * 8, cudaMemcpyDeviceToHost, ctx->stream);
        if (!rc && ce == cudaSuccess) ce = cudaMemcpyAsync(h_res, pb.dr, (size_t)nb * sizeof(PairRes), cudaMemcpyDeviceToHost, ctx->stream);
        if (!rc && ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
        if (!rc && ce == cudaSuccess) {
            const uint64_t total_ops = h_coff[nb];
            if ((rc = pool_alloc(ctx, &d_cops, total_ops + 1))) { cleanup(); return rc; }
            compact_ops_kernel<<<std::min<uint32_t>((nb + 7) / 8, (uint32_t)ctx->n_sm * 8), 256, 0, ctx->stream>>>(
                d_ops, d_opoff, d_nops, d_coff, nb, d_cops);
            ctx->launches++;
            ce = cudaGetLastError();
            // the fixed part is consumed before the buffer may move
            for (uint32_t i = 0; i < nb; i++) {
                const uint64_t r = winners[w0 + i];
                n_ops_of[r] = h_nops[i];
                cell_xy[4 * r] = h_res[i].bx; cell_xy[4 * r + 1] = h_res[i].by;
                cell_xy[4 * r + 2] = h_end[2 * i]; cell_xy[4 * r + 3] = h_end[2 * i + 1];
            }
            uint32_t *h_ops = pinned(total_ops + 16);
            if (!h_ops) { cleanup(); return IMSAME_ENOMEM; }
            if (ce == cudaSuccess && total_ops) ce = cudaMemcpyAsync(h_ops, d_cops, total_ops * 4, cudaMemcpyDeviceToHost, ctx->stream);
            if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
            t_gpu += now() - t0; t0 = now();
            if (ce == cudaSuccess) all_ops.insert(all_ops.end(), h_ops, h_ops + total_ops);  // batch order = ascending read order
            t_merge += now() - t0;
        }
        cleanup();
        if (rc) return rc;
        if (ce != cudaSuccess) { ctx->cuda_err = cudaGetErrorString(ce); return IMSAME_ECUDA; }
        w0 = w1;
    }
    if (trace)
        fprintf(stderr, "[imsame] traceback of %zu winners: lists %.1f ms, upload + pack %.1f ms, NW + walk + D2H %.1f ms, merge %.1f ms\n",
                winners.size(), t_prep, t_upload, t_gpu, t_merge);
    // winners were visited in ascending read order, so first_op is already monotone
    uint64_t at = 0;
    for (uint64_t r = 0; r < nq; r++) { ops_off[r] = at; at += n_ops_of[r]; }
    ops_off[nq] = at;
    uint32_t *out = (uint32_t *)malloc(std::max<size_t>(all_ops.size(), 1) * sizeof(uint32_t));
    if (!out) return IMSAME_ENOMEM;
    memcpy(out, all_ops.data(), all_ops.size() * sizeof(uint32_t));
    *ops_out = out;
    return IMSAME_OK;
}

}  // extern "C"

#include "capi_sharded.inc"
#include "capi_samples.inc"
#include "capi_sweep.inc"
#include "capi_cigar.inc"
#include "capi_kmers.inc"
