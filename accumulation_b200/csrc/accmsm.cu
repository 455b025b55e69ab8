// Host side of libaccmsm.so: context, HBM-resident commitment keys, kernel orchestration and the C-ABI
// declared in include/accmsm.h.  No CPU arithmetic path exists here: every group / field operation is a
// CUDA kernel from msm.cuh / vec.cuh, and every entry point fails with ACCMSM_E_CUDA without a device.
#include <algorithm>
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/accmsm.h"
#include "msm.cuh"
#include "sort.cuh"
#include "vec.cuh"
#include "ipa.cuh"
#include "wire.cuh"
#include "hostfp.hpp"

using namespace accmsm;

namespace {

enum Stage { ST_H2D = 0, ST_DIGITS, ST_SCAN, ST_SCATTER, ST_ACCUMULATE, ST_FIXUP, ST_REDUCE, ST_FINISH, ST_D2H, ST_VEC, ST_VEC_D2H, ST_COUNT };
const char *STAGE_NAMES[ST_COUNT] = {"h2d", "digits", "scan", "scatter", "accumulate", "fixup", "bucket_reduce", "finish", "d2h",
                                     "vec_kernel", "vec_d2h"};

struct Bases {
    int curve = 0;
    size_t n = 0;
    affine_t *d_xy = nullptr;
    uint8_t *d_inf = nullptr;   // nullptr when no base is the identity
    // optional window table (accmsm_precompute_bases): d_table[w * n + i] = 2^(pre_c * w) * base_i
    affine_t *d_table = nullptr;
    uint32_t pre_c = 0, pre_nwin = 0;
};

template <class T> struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;   // elements
    cudaError_t ensure(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = n + n / 8 + 64;
        cudaError_t e = cudaMalloc(&p, want * sizeof(T));
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

}  // namespace

struct IpaSession;
void ipa_session_free(IpaSession *s);
struct CsrSet;
void csr_set_free(CsrSet *c);
struct HpSession;
void hp_session_free(accmsm_ctx *ctx, HpSession *s);

struct GroupWorker;
struct GroupKey;
struct GroupCsr;

struct accmsm_ctx {
    // ---- device group (accmsm_init_multi, multi_api.inc): a group ctx owns one child ctx per device, one host thread
    //      per child, and no CUDA state of its own; every entry point below dispatches on !kids.empty()
    std::vector<accmsm_ctx *> kids;
    std::vector<GroupWorker *> workers;
    std::unordered_map<uint64_t, GroupKey *> gkeys;
    std::unordered_map<uint64_t, GroupCsr *> gcsrs;
    std::unordered_map<uint64_t, struct GroupIpaSession *> gsessions;   // IpaPC::open sessions sharded across the children
    std::unordered_map<uint64_t, struct GroupHpSession *> ghp_sessions; // hp-as prover sessions over the children's columns
    std::vector<char> peer_ok;                           // child g can store straight into child 0's memory
    std::vector<char> peer_read;                         // [i * children + j]: child i's kernels can read child j's memory
    void *d_gather = nullptr;                            // on child 0's device: partial sums of all children, rank-major
    size_t min_shard = size_t(1) << 16;                  // keys are cut into shards of at least this many points
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    std::mutex mu;
    std::string last_error;
    std::unordered_map<uint64_t, Bases> bases;
    std::unordered_map<uint64_t, struct IpaSession *> ipa_sessions;
    std::vector<struct IpaSession *> ipa_free;
    std::unordered_map<uint64_t, struct CsrSet *> csr_sets;
    std::unordered_map<uint64_t, HpSession *> hp_sessions;  // ASForHadamardProducts::prove sessions (fused_api.inc)
    std::vector<std::pair<void *, size_t>> vec_cache;   // recycled scratch blocks of the field-vector entry points
    uint64_t next_handle = 1;
    int window_bits = 0;
    uint64_t launches = 0;
    int acc_ctas_per_sm[2] = {0, 0};

    // MSM workspace
    DevBuf<uint32_t> digits, hist, offsets, cursor, entries, cta_ids, tile_sums, tile_offs;
    DevBuf<xyzz_t> buckets, red_sum[2], red_wsum[2], cta_parts, partial;
    DevBuf<uint8_t> scalars, misc;
    DevBuf<uint2> sort_pairs;                                   // sort.cuh: (key low bits, entry) pairs in partition order
    DevBuf<uint32_t> sort_tile_count, sort_part_count, sort_part_offs;
    int segments_override = 0;                                  // development knob (ACCMSM_SEGMENTS): point segments of a large host-scalar MSM (1 = no pipelining)
    int seg0_pct = 25;                                          // share of the first of two segments (ACCMSM_SEG0_PCT)
    std::vector<int> seg_pcts;                                  // development knob (ACCMSM_SEG_PCTS="12,60"): cumulative segment boundaries in percent
    bool no_coop_precompute = false;                            // development knob (ACCMSM_NO_COOP_PRECOMPUTE)
    bool trace = false;                                         // development knob ACCMSM_TRACE: timeline of the segments of a pipelined host-scalar MSM on stderr
    std::vector<std::pair<std::string, cudaEvent_t>> trace_ev;
    std::vector<double> trace_host_us;                          // host clock at every trace point (when the launch was ENQUEUED)
    int sort_lb_override = 0;                                   // development knob (ACCMSM_SORT_LB), 0 = automatic; -1 = first-version sort
    DevBuf<uint8_t> oneshot_inf, ipa_tabs;      // ipa_tabs: half tables of h(X)'s coefficients (ipa_half_tables)
    bool no_ipa_tabs = false;                   // development knob (ACCMSM_NO_IPA_TABS)
    bool no_coop_finish = false;                // development knob (ACCMSM_NO_COOP_FINISH)
    DevBuf<affine_t> oneshot_xy, pair_pts[2];   // pair_pts / pair_off: ping-pong lists of the batch-affine rounds
    DevBuf<uint32_t> pair_off[2];
    DevBuf<uint8_t> pair_pref, pair_kinds, pair_tfac, pair_ctot, pair_cfac;
    int affine_rounds_override = -1;            // development knob (ACCMSM_AFFINE_ROUNDS), -1 = automatic
    DevBuf<xyzz_t> fold_partial;                // IpaPC::open folded-key materialisation (ipa.cuh)
    DevBuf<uint32_t> fold_flag;
    int ipa_fold_rounds = 5, ipa_fold_min_log = 11;   // accmsm_set_ipa_fold (2^18 -> 2^13 -> 2^8, 2^20 -> 2^15 -> 2^10: profiles/r02v_fold_policy.txt)
    int fk_small_c = 0;                               // development knob ACCMSM_FK_C: window bits of a materialised key of <= 2^13 points (0 = the rule of registered keys; 10 / 11 / 12 measured slower, profiles/r02w_fk_window.txt)
    // Results that go back to the caller leave the device UN-NORMALISED (XYZZ, 128 B each) and are converted to affine by the
    // host thread that receives them (hostfp.hpp: one inversion for all results of a call)
    xyzz_t *d_out_raw = nullptr;
    int out_curve = 0;           // curve of the sums in d_out_raw (set by msm_reduce / the combine entry points)
    uint64_t *h_out = nullptr;   // pinned: MAX_JOBS x 16 u64 raw results + 64 u64 of small extras
    void *h_stage = nullptr;     // pinned staging for pageable host sources (upload())
    size_t stage_cap = 0;
    cudaEvent_t stage_done = nullptr;
    bool stage_busy = false;
    std::vector<cudaEvent_t> chunk_events;   // download() / chunked upload: one per 4 MiB chunk
    cudaStream_t copy_stream = nullptr;      // chunked upload of large scalar vectors (msm_host_scalars)
    // Side stream for launches that are off the critical path of a pass: the gated fallback sort of a long pass (its kernels
    // return at once unless the radix sort stood down) runs beside the radix sort's write / bucket passes, and the fix-up
    // of a point segment beside the sort of the next one.  aux_fork orders it after the launching stream, aux_join back.
    cudaStream_t aux_stream = nullptr;
    cudaEvent_t aux_fork = nullptr, aux_join = nullptr;
    bool aux_dirty = false;                  // work enqueued on aux_stream that the launching stream has not waited for yet
    bool no_aux = false;                     // development knob (ACCMSM_NO_AUX): everything on the launching stream
    cudaEvent_t ev[ST_COUNT + 1];
    bool ev_valid[ST_COUNT + 1];
    float timings[ST_COUNT];
    // One workspace per ctx, but `*_dev` entry points may only ENQUEUE on a caller stream: ws_done is recorded after
    // every enqueue that touches the workspace and every later user on a different stream waits on it first.
    cudaEvent_t ws_done = nullptr;
    cudaStream_t ws_stream = nullptr;
    bool ws_pending = false;
    // small host arguments (challenges, xi, randomizers: <= 1 KiB) are copied into a ring of page-locked slots before
    // the async H2D, so a caller that passes page-locked memory may reuse its buffer as soon as the call returns
    static constexpr int ARG_SLOTS = 16;
    static constexpr size_t ARG_SLOT_BYTES = 1024;
    uint8_t *h_args = nullptr;
    cudaEvent_t arg_done[ARG_SLOTS] = {nullptr};
    bool arg_used[ARG_SLOTS] = {false};
    int arg_next = 0;
};

namespace {

#define CU(ctx, call)                                                                          \
    do {                                                                                       \
        cudaError_t _e = (call);                                                               \
        if (_e != cudaSuccess) {                                                               \
            (ctx)->last_error = std::string(#call) + ": " + cudaGetErrorString(_e);            \
            return _e == cudaErrorMemoryAllocation ? ACCMSM_E_NOMEM : ACCMSM_E_CUDA;           \
        }                                                                                      \
    } while (0)

int fail_arg(accmsm_ctx *ctx, const char *msg) {
    if (ctx) ctx->last_error = msg;
    return ACCMSM_E_ARG;
}

void mark(accmsm_ctx *ctx, int idx, cudaStream_t st) {
    cudaEventRecord(ctx->ev[idx], st);
    ctx->ev_valid[idx] = true;
}
void clear_marks(accmsm_ctx *ctx) {
    for (int i = 0; i <= ST_COUNT; i++) ctx->ev_valid[i] = false;
    for (int i = 0; i < ST_COUNT; i++) ctx->timings[i] = 0.f;
}
// timings[i] = elapsed between mark i and the next valid mark
void collect_timings(accmsm_ctx *ctx) {
    int prev = -1;
    for (int i = 0; i <= ST_COUNT; i++) {
        if (!ctx->ev_valid[i]) continue;
        if (prev >= 0) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, ctx->ev[prev], ctx->ev[i]) == cudaSuccess) ctx->timings[prev] = ms;
            else (void)cudaGetLastError();   // not ready yet: leave the slot, clear the non-sticky error
        }
        prev = i;
    }
    if (ctx->trace && !ctx->trace_ev.empty()) {      // ACCMSM_TRACE: timeline of the segments of a pipelined host-scalar MSM
        size_t ti = 0;
        for (auto &le : ctx->trace_ev) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, ctx->trace_ev[0].second, le.second) != cudaSuccess) (void)cudaGetLastError();
            const double host_ms = ti < ctx->trace_host_us.size() ? (ctx->trace_host_us[ti] - ctx->trace_host_us[0]) / 1e3 : 0.0;
            ti++;
            fprintf(stderr, "[accmsm trace] %8.3f ms (enqueued by the host at %7.3f ms)  %s\n", ms, host_ms, le.first.c_str());
            if (&le != &ctx->trace_ev[0]) cudaEventDestroy(le.second);
        }
        cudaEventDestroy(ctx->trace_ev[0].second);
        ctx->trace_ev.clear();
        ctx->trace_host_us.clear();
    }
}

void trace_point(accmsm_ctx *ctx, cudaStream_t st, const std::string &label) {
    if (!ctx->trace) return;
    cudaEvent_t ev; cudaEventCreate(&ev); cudaEventRecord(ev, st);
    ctx->trace_ev.push_back({label, ev});
    ctx->trace_host_us.push_back(std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count());
}

// side stream (see accmsm_ctx::aux_stream): aux_begin makes it wait for everything enqueued on `st` so far and returns it
// (or `st` itself when the side stream is unavailable / switched off); aux_sync makes `st` wait for everything enqueued on it
cudaStream_t aux_begin(accmsm_ctx *ctx, cudaStream_t st) {
    if (ctx->no_aux) return st;
    if (!ctx->aux_stream) {
        if (cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->aux_fork, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->aux_join, cudaEventDisableTiming) != cudaSuccess) {
            (void)cudaGetLastError(); ctx->no_aux = true; return st;
        }
    }
    if (cudaEventRecord(ctx->aux_fork, st) != cudaSuccess || cudaStreamWaitEvent(ctx->aux_stream, ctx->aux_fork, 0) != cudaSuccess) {
        (void)cudaGetLastError(); return st;
    }
    ctx->aux_dirty = true;
    return ctx->aux_stream;
}
int aux_sync(accmsm_ctx *ctx, cudaStream_t st) {
    if (!ctx->aux_dirty) return ACCMSM_OK;
    CU(ctx, cudaEventRecord(ctx->aux_join, ctx->aux_stream));
    CU(ctx, cudaStreamWaitEvent(st, ctx->aux_join, 0));
    ctx->aux_dirty = false;
    return ACCMSM_OK;
}

// workspace ordering across streams (see accmsm_ctx::ws_done)
int ws_acquire(accmsm_ctx *ctx, cudaStream_t st) {
    if (ctx->ws_pending && ctx->ws_stream != st) CU(ctx, cudaStreamWaitEvent(st, ctx->ws_done, 0));
    ctx->ws_stream = st;
    return ACCMSM_OK;
}
int ws_release(accmsm_ctx *ctx, cudaStream_t st) {
    CU(ctx, cudaEventRecord(ctx->ws_done, st));
    ctx->ws_stream = st; ctx->ws_pending = true;
    return ACCMSM_OK;
}
// async H2D of a small host argument through a ctx-owned page-locked slot (the caller's buffer is free on return)
int upload_small(accmsm_ctx *ctx, void *d_dst, const void *h_src, size_t bytes, cudaStream_t st) {
    if (!bytes) return ACCMSM_OK;
    if (bytes > accmsm_ctx::ARG_SLOT_BYTES) { CU(ctx, cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, st)); CU(ctx, cudaStreamSynchronize(st)); return ACCMSM_OK; }
    const int slot = ctx->arg_next;
    ctx->arg_next = (slot + 1) % accmsm_ctx::ARG_SLOTS;
    if (ctx->arg_used[slot]) CU(ctx, cudaEventSynchronize(ctx->arg_done[slot]));
    uint8_t *h = ctx->h_args + (size_t)slot * accmsm_ctx::ARG_SLOT_BYTES;
    memcpy(h, h_src, bytes);
    CU(ctx, cudaMemcpyAsync(d_dst, h, bytes, cudaMemcpyHostToDevice, st));
    CU(ctx, cudaEventRecord(ctx->arg_done[slot], st));
    ctx->arg_used[slot] = true;
    return ACCMSM_OK;
}

constexpr size_t PRECOMPUTE_COOP_MAX = 1u << 12;    // keys up to this many points build their window table with k_precompute_coop (one group per SM: 0.93 -> 0.65 ms; no gain once two groups share an SM)
uint32_t pick_window_bits(const accmsm_ctx *ctx, size_t n) {
    if (ctx->window_bits >= 2 && ctx->window_bits <= 16) return (uint32_t)ctx->window_bits;
    uint32_t lg = 0;
    while ((size_t(1) << (lg + 1)) <= n) lg++;
    int c = (int)lg - 3;
    return (uint32_t)std::min(16, std::max(4, c));
}

// The window table is used whenever the key has one (unless an explicit window override asks for something else),
// also for MSMs much shorter than the key: a short MSM is bound by the latency of its tail, and the table path has no
// Horner over windows (~256 dependent doublings, ~0.9 ms), only a reduction over mostly empty buckets.
// Builds (or rebuilds) the window table of a key: table[w * n + i] = 2^(c w) * base_i.  Caller holds ctx->mu.
// `storage` (optional): a caller-owned buffer of *storage_cap records that is grown when too small and then holds the
// table -- the IPA open sessions recycle theirs, because cudaMalloc / cudaFree in the middle of an opening stall.
int precompute_table(accmsm_ctx *ctx, Bases &B, int window_bits, affine_t **storage = nullptr, size_t *storage_cap = nullptr) {
    if (!storage) {
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        if (B.d_table) { cudaFree(B.d_table); B.d_table = nullptr; B.pre_c = B.pre_nwin = 0; }
    }
    if (B.n == 0) return ACCMSM_OK;
    // auto: measured best per key size (profiles/r01l_window_rule.txt).  Scalars are < 2^254, so what counts is
    // ceil(254 / c) non-empty windows and the bucket count 2^(c-1) of the single bucket set: c = 17 has 15 working
    // windows (the 16th covers bit 255 only) over 2^16 buckets and wins from 2^15 to 2^19 points; c = 20 (13 windows,
    // 2^19 buckets) from 2^20 on, where the insertions dominate the reduction.
    uint32_t lg = 0;
    while ((size_t(1) << (lg + 1)) <= B.n) lg++;
    uint32_t c = window_bits ? (uint32_t)window_bits : lg >= 20 ? 20u : lg >= 15 ? 17u : lg >= 13 ? 15u : 10u;
    uint32_t nwin = (256 + c - 1) / c;
    if ((size_t)nwin * B.n >= (size_t(1) << 31)) return fail_arg(ctx, "precompute_bases: windows * n must be < 2^31");
    affine_t *table = nullptr;
    const size_t records = (size_t)nwin * B.n;
    if (storage) {
        if (*storage_cap < records) {
            if (*storage) cudaFree(*storage);
            *storage = nullptr; *storage_cap = 0;
            CU(ctx, cudaMalloc(storage, records * sizeof(affine_t)));
            *storage_cap = records;
        }
        table = *storage;
    } else {
        CU(ctx, cudaMalloc(&table, records * sizeof(affine_t)));
    }
    if (B.n <= PRECOMPUTE_COOP_MAX && !ctx->no_coop_precompute) {      // short key: latency-bound, one cooperative group per 32 bases
        uint32_t groups = (uint32_t)((B.n + 31) / 32);
        if (B.curve == 0) k_precompute_coop<0><<<groups, 128, 0, ctx->stream>>>(B.d_xy, (uint32_t)B.n, c, nwin, table);
        else k_precompute_coop<1><<<groups, 128, 0, ctx->stream>>>(B.d_xy, (uint32_t)B.n, c, nwin, table);
    } else {
        uint32_t blocks = (uint32_t)((B.n + 127) / 128);
        if (B.curve == 0) k_precompute<0><<<blocks, 128, 0, ctx->stream>>>(B.d_xy, (uint32_t)B.n, c, nwin, table);
        else k_precompute<1><<<blocks, 128, 0, ctx->stream>>>(B.d_xy, (uint32_t)B.n, c, nwin, table);
    }
    ctx->launches++;
    if (!storage) {      // sessions stay asynchronous: the table is consumed on the same stream
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) { cudaFree(table); CU(ctx, e); }
    }
    B.d_table = table; B.pre_c = c; B.pre_nwin = nwin;
    return ACCMSM_OK;
}

bool use_table(const accmsm_ctx *ctx, const Bases &B, size_t n) {
    (void)n;
    if (!B.d_table) return false;
    return !ctx->window_bits || (uint32_t)ctx->window_bits == B.pre_c;
}

constexpr uint32_t ACC_WARP_MAX_KEYS = 8192;        // warp-per-bucket accumulation up to this many buckets ...
constexpr size_t ACC_WARP_MAX_ENTRIES = 1u << 17;   // ... and bucket insertions (measured: 0.106 vs 0.221 ms at 2^12 points, c = 10; one CTA per bucket loses beyond 8192 buckets)

#ifndef RED_L0_BLK
#define RED_L0_BLK 32     // threads per row / column sum of the first reduction level (one warp: 16-32 serial adds + 5 shuffle steps; measured best of 32/64/128/256)
#endif

struct MsmJobs {
    uint32_t njobs = 1;
    size_t offset[MAX_JOBS] = {0};     // first base of every job inside the key
    uint32_t tail_base = NONE_ID;      // index of the hiding generator when the last pair of every job is (H, r)
    uint32_t map_log_h = NONE_ID;      // IPA round index map (msm.cuh), NONE_ID = identity
    MsmJobs() {}
    explicit MsmJobs(size_t off) { offset[0] = off; }
};

MsmShape make_shape(const accmsm_ctx *ctx, const Bases &B, const MsmJobs &jobs, size_t n, size_t n_for_c) {
    MsmShape sh;
    sh.n = (uint32_t)n;
    sh.njobs = jobs.njobs;
    sh.tail_base = jobs.tail_base;
    sh.map_log_h = jobs.map_log_h;
    for (int j = 0; j < MAX_JOBS; j++) sh.job_off[j] = j < (int)jobs.njobs ? (uint32_t)jobs.offset[j] : 0u;
    if (use_table(ctx, B, n)) {
        sh.c = B.pre_c;
        sh.nwin = B.pre_nwin;
        sh.nb = 1u << (sh.c - 1);
        sh.sets_per_job = 1;
        sh.hist_stride = 0;
        sh.ent_stride = (uint32_t)B.n;
    } else {
        sh.c = pick_window_bits(ctx, n_for_c);
        sh.nwin = (256 + sh.c - 1) / sh.c;
        sh.nb = 1u << (sh.c - 1);
        sh.sets_per_job = sh.nwin;
        sh.hist_stride = sh.nb;
        sh.ent_stride = 0;
    }
    sh.nkeys = sh.njobs * sh.sets_per_job * sh.nb;
    return sh;
}

// How many batch-affine halving rounds precede the XYZZ accumulation (0 = none).
int affine_rounds(const accmsm_ctx *ctx, const MsmShape &sh, size_t n_entries) {
    if (ctx->affine_rounds_override >= 0) return ctx->affine_rounds_override;
    return 0;
}

// exclusive scan of counts[0..nkeys) into offsets[0..nkeys] (+ optional copy into cursor)
int launch_scan(accmsm_ctx *ctx, const uint32_t *counts, uint32_t nkeys, uint32_t *offsets, uint32_t *cursor, cudaStream_t st,
                SortGate gate = SortGate{nullptr, 0}) {
    uint32_t ntiles = (nkeys + SCAN_TILE - 1) / SCAN_TILE;
    if (ntiles <= SCAN_ONE_CTA_TILES) {
        k_scan<<<1, 1024, 0, st>>>(counts, nkeys, offsets, cursor, gate);
        ctx->launches++;
    } else {
        CU(ctx, ctx->tile_sums.ensure(ntiles));
        CU(ctx, ctx->tile_offs.ensure(ntiles + 1));
        k_scan_tile_sums<<<ntiles, 1024, 0, st>>>(counts, nkeys, ctx->tile_sums.p, gate);
        k_scan<<<1, 1024, 0, st>>>(ctx->tile_sums.p, ntiles, ctx->tile_offs.p, nullptr, gate);
        k_scan_tiles<<<ntiles, 1024, 0, st>>>(counts, nkeys, ctx->tile_offs.p, offsets, cursor, gate);
        ctx->launches += 3;
    }
    return ACCMSM_OK;
}

constexpr size_t SORT_SMEM_OPT_IN = 220 * 1024;      // dynamic shared memory the sort kernels may use (227 KB per CTA minus their static part)
// both tile passes: the count pass asks for 2 nparts words, more than the 48 KB default once nparts > 6144
template <class Src> bool sort_opt_in() {
    return cudaFuncSetAttribute(k_sort_tiles<Src, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SORT_SMEM_OPT_IN) == cudaSuccess &&
           cudaFuncSetAttribute(k_sort_tiles<Src, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SORT_SMEM_OPT_IN) == cudaSuccess;
}

// ---- the MSM pipeline in two stages ---------------------------------------------------------------------------------
// msm_accumulate: sort the (bucket, point) pairs of `n` (base, scalar) pairs and accumulate them into ctx->buckets.
//                 into = false: every non-empty bucket is overwritten (empty ones are never read: the reduction tests
//                 the offsets); into = true: the sums are ADDED to zero-initialised buckets -- several point segments of
//                 one MSM then share the bucket set (msm_host_scalars pipelines their uploads).
// msm_reduce:     bucket reduction, (plain key: Horner over windows), extra partials, normalisation / raw partial.
// n_for_c: the length that picks the window size of a plain key (all segments of one MSM must agree on it).
template <int CURVE, class Src>
int msm_accumulate(accmsm_ctx *ctx, const Bases &B, const MsmJobs &jobs, size_t n, size_t n_for_c, const Src &src, bool into,
                   cudaStream_t st, MsmShape *sh_out, bool fixup_aside = false) {
    MsmShape sh = make_shape(ctx, B, jobs, n, n_for_c);
    *sh_out = sh;
    const bool tabled = sh.ent_stride != 0;
    const affine_t *points = tabled ? B.d_table : B.d_xy;
    const size_t n_entries = (size_t)sh.n * sh.nwin * sh.njobs;
    if (n_entries >= (size_t(1) << 31)) return fail_arg(ctx, "msm: jobs * windows * n must be < 2^31");
    CU(ctx, ctx->entries.ensure(n_entries));
    CU(ctx, ctx->hist.ensure(sh.nkeys));          // also scratch of the batch-affine rounds
    CU(ctx, ctx->offsets.ensure(sh.nkeys + 1));
    CU(ctx, ctx->buckets.ensure(sh.nkeys));
    { int wrc = ws_acquire(ctx, st); if (wrc) return wrc; }

    // Sort of the (bucket key, table index | sign) pairs.  Long passes: two-level radix sort staged through shared memory
    // (sort.cuh: digits never touch HBM, no global atomics), with the first-version counting sort gated behind it for skewed
    // inputs.  Short passes: the counting sort alone (3 launches; with a few thousand pairs nothing is bandwidth-bound).
    const bool radix = ctx->sort_lb_override >= 0 && n_entries >= (size_t(1) << 17) && sh.nkeys >= 1024u;
    SortGate fallback{nullptr, 0};
    cudaStream_t fb = st;                // stream of the first-version sort: `st`, or the side stream behind a radix sort
    if (radix) {
        SortPlan pl;
        pl.lb = ctx->sort_lb_override > 0 ? (uint32_t)ctx->sort_lb_override : 9;      // measured: 9 beats 10 and 11 at 2^19 buckets
        pl.lb = std::min(SORT_MAX_LB, std::max(9u, pl.lb));
        while (((sh.nkeys + (1u << pl.lb) - 1) >> pl.lb) > SORT_MAX_PARTS && pl.lb < SORT_MAX_LB) pl.lb++;
        pl.nparts = (sh.nkeys + (1u << pl.lb) - 1) >> pl.lb;
        if (pl.nparts > SORT_MAX_PARTS) return fail_arg(ctx, "msm: too many bucket sets in one pass");
        pl.tiles_per_job = (sh.n + SORT_TILE - 1) / SORT_TILE;
        pl.ntiles = pl.tiles_per_job * sh.njobs;
        // shared-memory staging: a tile's pairs (write pass), a partition's entries (bucket pass, 1.25 x the mean size)
        pl.stage_pairs = (uint32_t)SORT_TILE * sh.nwin <= SORT_STAGE_MAX ? (uint32_t)SORT_TILE * sh.nwin : 0u;
        pl.bucket_cap = (uint32_t)std::min<size_t>(49152, std::max<size_t>(4096, n_entries / pl.nparts * 5 / 4 + 1024));
        CU(ctx, ctx->sort_tile_count.ensure((size_t)2 * pl.ntiles * pl.nparts));
        CU(ctx, ctx->sort_part_count.ensure(pl.nparts + 1));
        CU(ctx, ctx->sort_part_offs.ensure(pl.nparts + 1));
        CU(ctx, ctx->sort_pairs.ensure(n_entries));
        uint32_t *tile_count = ctx->sort_tile_count.p, *tile_hist = tile_count + (size_t)pl.ntiles * pl.nparts;
        uint32_t *max_part = ctx->sort_part_count.p + pl.nparts;
        // skew: one partition holds more than 4 x its share (and more than a CTA streams in ~50 us)
        const SortGate gate{max_part, (uint32_t)std::min<size_t>(0x7fffffffu, std::max<size_t>(65536, 4 * n_entries / pl.nparts))};
        fallback = gate;
        const size_t smem0 = (size_t)2 * pl.nparts * sizeof(uint32_t);
        const size_t smem1 = smem0 + (size_t)pl.stage_pairs * sizeof(uint2);
        const size_t smem2 = ((size_t(1) << pl.lb) + pl.bucket_cap) * sizeof(uint32_t);
        if (smem1 > SORT_SMEM_OPT_IN || smem2 > SORT_SMEM_OPT_IN) return fail_arg(ctx, "msm: sort staging exceeds shared memory");
        mark(ctx, ST_DIGITS, st);
        trace_point(ctx, st, "  sort begins");
        CU(ctx, cudaMemsetAsync(max_part, 0, sizeof(uint32_t), st));
        k_sort_tiles<Src, false><<<pl.ntiles, SORT_THREADS, smem0, st>>>(src, sh, B.d_inf, pl, 0u, pl.tiles_per_job, tile_count, tile_hist, nullptr, nullptr, gate);
        CU(ctx, cudaGetLastError());      // a refused count launch leaves tile_count unwritten: nothing below may read it
        mark(ctx, ST_SCAN, st);
        k_sort_tile_scan<<<(pl.nparts + TS_PARTS - 1) / TS_PARTS, TS_PARTS * TS_SEGS, 0, st>>>(tile_count, pl.ntiles, pl.nparts, ctx->sort_part_count.p, max_part);
        ctx->launches += 2;
        { int src2 = launch_scan(ctx, ctx->sort_part_count.p, pl.nparts, ctx->sort_part_offs.p, nullptr, st); if (src2) return src2; }
        // the gate word is final: the fallback chain below goes to the side stream, next to the write / bucket passes
        fb = aux_begin(ctx, st);
        mark(ctx, ST_SCATTER, st);
        trace_point(ctx, st, "  counted + scanned");
        k_sort_tiles<Src, true><<<pl.ntiles, SORT_THREADS, smem1, st>>>(src, sh, B.d_inf, pl, 0u, pl.tiles_per_job, tile_count, tile_hist, ctx->sort_part_offs.p, ctx->sort_pairs.p, gate);
        k_sort_buckets<<<pl.nparts, SORT_BUCKET_THREADS, smem2, st>>>(ctx->sort_pairs.p, ctx->sort_part_offs.p, pl.lb, sh.nkeys, pl.bucket_cap, ctx->offsets.p, ctx->entries.p, gate);
        ctx->launches += 2;
        trace_point(ctx, st, "  radix sort done");
    }
    {
        // first-version counting sort: the only sort of a short pass; behind the gate of a long one (its kernels return at
        // once unless the radix sort stood down)
        CU(ctx, ctx->digits.ensure(n_entries));
        CU(ctx, ctx->cursor.ensure(sh.nkeys));
        if (!radix) mark(ctx, ST_DIGITS, st);
        CU(ctx, cudaMemsetAsync(ctx->hist.p, 0, sh.nkeys * sizeof(uint32_t), fb));
        // behind the gate: a small grid (grid-stride loops), so standing down costs next to nothing
        dim3 blocks(radix ? std::min<uint32_t>((sh.n + 255) / 256, (uint32_t)ctx->sm_count * 8) : (sh.n + 255) / 256, sh.njobs);
        k_digits<Src><<<blocks, 256, 0, fb>>>(src, sh, B.d_inf, ctx->digits.p, ctx->hist.p, 0u, sh.n, fallback);
        if (!radix) mark(ctx, ST_SCAN, st);
        { int src2 = launch_scan(ctx, ctx->hist.p, sh.nkeys, ctx->offsets.p, ctx->cursor.p, fb, fallback); if (src2) return src2; }
        if (!radix) mark(ctx, ST_SCATTER, st);
        k_scatter<<<blocks, 256, 0, fb>>>(sh, ctx->digits.p, ctx->cursor.p, ctx->entries.p, fallback);
        ctx->launches += 2;
    }
    { int arc = aux_sync(ctx, st); if (arc) return arc; }      // fallback chain (and an earlier segment's fix-up) before the buckets are touched
    mark(ctx, ST_ACCUMULATE, st);
    trace_point(ctx, st, "  gated fallback sort passed");
    if (!into && sh.nkeys <= ACC_WARP_MAX_KEYS && n_entries <= ACC_WARP_MAX_ENTRIES) {
        // short MSM: one group of four replica warps per bucket, no slice merging (k_accumulate_warp_coop in msm.cuh)
        k_accumulate_warp_coop<CURVE><<<sh.nkeys, 128, 0, st>>>(ctx->offsets.p, sh.nkeys, ctx->entries.p, points, ctx->buckets.p);
        ctx->launches++;
        mark(ctx, ST_FIXUP, st);
    } else {
        // grid: a whole number of resident waves, shrunk for small inputs so every thread still gets a
        // few entries (upper bound n * nwin; the real count is only known on the device)
        // optional batch-affine pre-reduction (msm.cuh): `rounds` halvings of every bucket's list in affine coordinates
        const uint32_t *acc_offsets = ctx->offsets.p, *acc_entries = ctx->entries.p;
        const affine_t *acc_points = points;
        size_t acc_bound = n_entries;
        int rounds = into ? 0 : affine_rounds(ctx, sh, n_entries);
        for (int r = 0; r < rounds; r++) {
            const size_t out_bound = (acc_bound + sh.nkeys) / 2 + 1;
            CU(ctx, ctx->pair_off[r & 1].ensure(sh.nkeys + 1));
            CU(ctx, ctx->pair_pts[r & 1].ensure(out_bound));
            k_pair_counts<<<(sh.nkeys + 255) / 256, 256, 0, st>>>(acc_offsets, sh.nkeys, ctx->hist.p);
            ctx->launches++;
            { int src2 = launch_scan(ctx, ctx->hist.p, sh.nkeys, ctx->pair_off[r & 1].p, nullptr, st); if (src2) return src2; }
            uint32_t pgrid = (uint32_t)((out_bound + (size_t)PAIR_THREADS * PAIR_B - 1) / ((size_t)PAIR_THREADS * PAIR_B));
            CU(ctx, ctx->pair_pref.ensure(out_bound * 32));
            CU(ctx, ctx->pair_kinds.ensure(out_bound));
            CU(ctx, ctx->pair_tfac.ensure((size_t)pgrid * PAIR_THREADS * 32));
            CU(ctx, ctx->pair_ctot.ensure((size_t)pgrid * 32));
            CU(ctx, ctx->pair_cfac.ensure((size_t)pgrid * 32));
            const uint32_t *oin = acc_offsets, *oout = ctx->pair_off[r & 1].p;
            affine_t *pout = ctx->pair_pts[r & 1].p;
            if (r == 0) {
                k_pair_fwd<CURVE, true><<<pgrid, PAIR_THREADS, 0, st>>>(oin, oout, sh.nkeys, ctx->entries.p, points, ctx->pair_pref.p, ctx->pair_kinds.p, ctx->pair_tfac.p, ctx->pair_ctot.p);
                k_pair_mid<CURVE><<<1, PAIR_MID_THREADS, 0, st>>>(oout, sh.nkeys, ctx->pair_ctot.p, ctx->pair_cfac.p);
                k_pair_bwd<CURVE, true><<<pgrid, PAIR_THREADS, 0, st>>>(oin, oout, sh.nkeys, ctx->entries.p, points, ctx->pair_pref.p, ctx->pair_kinds.p, ctx->pair_tfac.p, ctx->pair_cfac.p, pout);
            } else {
                k_pair_fwd<CURVE, false><<<pgrid, PAIR_THREADS, 0, st>>>(oin, oout, sh.nkeys, nullptr, acc_points, ctx->pair_pref.p, ctx->pair_kinds.p, ctx->pair_tfac.p, ctx->pair_ctot.p);
                k_pair_mid<CURVE><<<1, PAIR_MID_THREADS, 0, st>>>(oout, sh.nkeys, ctx->pair_ctot.p, ctx->pair_cfac.p);
                k_pair_bwd<CURVE, false><<<pgrid, PAIR_THREADS, 0, st>>>(oin, oout, sh.nkeys, nullptr, acc_points, ctx->pair_pref.p, ctx->pair_kinds.p, ctx->pair_tfac.p, ctx->pair_cfac.p, pout);
            }
            ctx->launches += 3;
            acc_offsets = ctx->pair_off[r & 1].p; acc_entries = nullptr; acc_points = ctx->pair_pts[r & 1].p; acc_bound = out_bound;
        }
        int per_sm = ctx->acc_ctas_per_sm[CURVE];
        uint32_t gmax = (uint32_t)(ctx->sm_count * per_sm);
        uint32_t want = (uint32_t)((acc_bound + (size_t)ACC_THREADS * 8 - 1) / ((size_t)ACC_THREADS * 8));
        uint32_t grid = std::max(1u, std::min(gmax, want));
        CU(ctx, ctx->cta_ids.ensure(2 * grid));
        CU(ctx, ctx->cta_parts.ensure(2 * grid));
        size_t smem = 2 * ACC_THREADS * (sizeof(xyzz_t) + sizeof(uint32_t));
        if (into) k_accumulate<CURVE, true><<<grid, ACC_THREADS, smem, st>>>(acc_offsets, sh.nkeys, acc_entries, acc_points, ctx->buckets.p,
                                                                              ctx->cta_ids.p, ctx->cta_parts.p);
        else k_accumulate<CURVE, false><<<grid, ACC_THREADS, smem, st>>>(acc_offsets, sh.nkeys, acc_entries, acc_points, ctx->buckets.p,
                                                                          ctx->cta_ids.p, ctx->cta_parts.p);
        mark(ctx, ST_FIXUP, st);
        trace_point(ctx, st, "  k_accumulate done");
        uint32_t ns = 2 * grid;
        // k_fixup merges the 2 boundary slots of every accumulate CTA in ONE CTA's shared memory: the grid above is capped in
        // accmsm_init (acc_ctas_per_sm) so that they fit; a part with more SMs than that cap assumes must fail loudly, not overflow
        if (ns > (uint32_t)(FIX_THREADS * FIX_PER_T)) return fail_arg(ctx, "msm: accumulate grid exceeds the fix-up kernel's slots");
        size_t smem2 = ns * (sizeof(xyzz_t) + sizeof(uint32_t));
        // fixup_aside: more point segments follow (msm_host_scalars) -- the fix-up runs beside the sort of the next segment
        // and is waited for before that segment's accumulation touches the buckets (aux_sync above)
        cudaStream_t fx = fixup_aside ? aux_begin(ctx, st) : st;
        k_fixup<CURVE><<<1, FIX_THREADS, smem2, fx>>>(ctx->cta_ids.p, ctx->cta_parts.p, ns, ctx->buckets.p);
        ctx->launches += 2;
    }
    return ACCMSM_OK;
}

// use_offsets = false: every bucket holds a valid (possibly identity) point and the emptiness test on the offsets of the
// last accumulated segment must not be used
template <int CURVE>
int msm_reduce(accmsm_ctx *ctx, const MsmShape &sh, bool use_offsets, const xyzz_t *d_extra, uint32_t n_extra, xyzz_t *d_partial,
               bool normalise, cudaStream_t st, xyzz_t *d_out_raw) {
    if (!d_out_raw) d_out_raw = ctx->d_out_raw;
    ctx->out_curve = CURVE;
    const uint32_t nsets = sh.njobs * sh.sets_per_job;          // bucket sets to reduce
    const uint32_t *offs = use_offsets ? ctx->offsets.p : nullptr;
    { int arc = aux_sync(ctx, st); if (arc) return arc; }
    mark(ctx, ST_REDUCE, st);
    const xyzz_t *window_sums = nullptr;
    {
        // depth-optimised reduction (msm.cuh): rows / columns of the bucket index, twice, then 32-item weighted sums
        const uint32_t m = sh.c - 1, N0 = sh.nb;
        const uint32_t C0 = N0 > 1024 ? 1u << (m / 2) : 0, R0 = N0 > 1024 ? N0 / C0 : 0;
        CU(ctx, ctx->red_sum[0].ensure((size_t)nsets * (R0 + C0) + 1));
        CU(ctx, ctx->red_wsum[0].ensure((size_t)nsets * 128));
        CU(ctx, ctx->red_wsum[1].ensure(nsets));
        xyzz_t *scratch = ctx->red_sum[0].p, *leaf = ctx->red_wsum[0].p, *sums = ctx->red_wsum[1].p;
        CU(ctx, cudaMemsetAsync(leaf, 0, (size_t)nsets * 128 * sizeof(xyzz_t), st));   // all-zero = identity (ZZ == 0)
        int nlevels;
        SumTasks t1; memset(&t1, 0, sizeof t1);
        if (N0 > 1024) {
            SumTasks t0; memset(&t0, 0, sizeof t0);
            // R_hi = sum_lo B[hi][lo] (R0 outputs of C0 items), C_lo = sum_hi B[hi][lo] (C0 outputs of R0 items).  With plain
            // warps the column sums are the longer chains (R0 = 2 C0 for an odd number of index bits: 32 + 5 dependent additions
            // against 16 + 5): they are cut in two halves of the rows -- outputs interleaved, element 2 lo + h -- so that every warp of
            // the level has the same depth, and the next level adds the two halves on the fly (SumTask::pair).
            const bool split = (R0 + C0) * nsets > 320u && R0 > C0;
            const uint32_t CW = split ? 2 * C0 : C0;          // column-sum array: [2 lo + h] when split
            CU(ctx, ctx->red_sum[0].ensure((size_t)nsets * (R0 + CW) + 1));
            scratch = ctx->red_sum[0].p;
            t0.t[0] = SumTask{0, 0, R0, C0, C0, 1, 1, 0};
            if (split) {
                t0.ntasks = 3;
                t0.t[1] = SumTask{0, R0, C0, R0 / 2, 1, C0, 2, 0};
                t0.t[2] = SumTask{(R0 / 2) * C0, R0 + 1, C0, R0 / 2, 1, C0, 2, 0};
            } else {
                t0.ntasks = 2;
                t0.t[1] = SumTask{0, R0, C0, R0, 1, C0, 1, 0};
            }
            const uint32_t nout0 = R0 + (split ? 2 * C0 : C0);
            // first level: cooperative groups while the grid is small enough to be latency-bound (measured: 0.132 vs 0.147 ms
            // with 256 outputs, 0.202 vs 0.175 ms with 512), plain warps when it is throughput-bound (2^19 buckets)
            if (!split && (R0 + C0) * nsets <= 320u)
                k_sums_coop<CURVE><<<dim3(nout0, nsets), 128, 0, st>>>(ctx->buckets.p, N0, offs, scratch, R0 + CW, t0);
            else
                k_sums<CURVE, RED_L0_BLK><<<dim3(nout0, nsets), RED_L0_BLK, 0, st>>>(ctx->buckets.p, N0, offs, scratch, R0 + CW, t0);
            t1.ntasks = 4;
            const uint32_t pw = split ? 2u : 1u, pr = split ? 1u : 0u;
            t1.t[0] = SumTask{0, 0, R0 / 32, 32, 32, 1, 1, 0};            t1.t[1] = SumTask{0, 32, 32, R0 / 32, 1, 32, 1, 0};
            t1.t[2] = SumTask{R0, 64, C0 / 32, 32, 32 * pw, pw, 1, pr};   t1.t[3] = SumTask{R0, 96, 32, C0 / 32, pw, 32 * pw, 1, pr};
            k_sums_coop<CURVE><<<dim3(R0 / 32 + C0 / 32 + 64, nsets), 128, 0, st>>>(scratch, R0 + CW, nullptr, leaf, 128, t1);
            ctx->launches += 2;
            nlevels = 2;
        } else if (N0 > 32) {
            t1.ntasks = 2;
            t1.t[0] = SumTask{0, 0, N0 / 32, 32, 32, 1, 1, 0};     t1.t[1] = SumTask{0, 32, 32, N0 / 32, 1, 32, 1, 0};
            k_sums_coop<CURVE><<<dim3(N0 / 32 + 32, nsets), 128, 0, st>>>(ctx->buckets.p, N0, offs, leaf, 128, t1);
            ctx->launches++;
            nlevels = 1;
        } else {
            t1.ntasks = 1;
            t1.t[0] = SumTask{0, 0, N0, 1, 1, 1, 1, 0};
            k_sums_coop<CURVE><<<dim3(N0, nsets), 128, 0, st>>>(ctx->buckets.p, N0, offs, leaf, 128, t1);
            ctx->launches++;
            nlevels = 0;
        }
        uint32_t s0 = 0;
        while (C0 && (1u << s0) < C0) s0++;
        CU(ctx, ctx->red_sum[1].ensure((size_t)nsets * 5));
        const uint32_t narr = nlevels == 2 ? 4 : nlevels == 1 ? 2 : 1;
        k_leaf_scan_coop<CURVE><<<dim3(narr, nsets), 128, 0, st>>>(leaf, 128, ctx->red_sum[1].p);
        k_leaf_combine_coop<CURVE><<<nsets, 256, 0, st>>>(ctx->red_sum[1].p, nlevels, s0, sums);
        ctx->launches += 2;
        window_sums = sums;
    }
    mark(ctx, ST_FINISH, st);
    if (sh.sets_per_job > 1 && !ctx->no_coop_finish)      // plain key: Horner over the windows by a cooperative group
        k_finish_coop<CURVE><<<sh.njobs, 128, 0, st>>>(window_sums, sh.sets_per_job, sh.c, d_extra, n_extra, d_partial, normalise ? d_out_raw : nullptr);
    else
        k_finish<CURVE><<<sh.njobs, 32, 0, st>>>(window_sums, sh.sets_per_job, sh.c, d_extra, n_extra, d_partial, normalise ? d_out_raw : nullptr);
    ctx->launches++;
    CU(ctx, cudaGetLastError());
    return ws_release(ctx, st);
}

// The whole pipeline over one segment.  Leaves the per-window sums combined into either a device partial (d_partial) or the
// un-normalised result in ctx->d_out_raw (or d_out_raw), which the host fetches and converts to affine.
template <int CURVE, class Src>
int run_msm(accmsm_ctx *ctx, const Bases &B, const MsmJobs &jobs, size_t n, const Src &src,
            const xyzz_t *d_extra, uint32_t n_extra, xyzz_t *d_partial, bool normalise, cudaStream_t st,
            xyzz_t *d_out_raw = nullptr) {
    MsmShape sh;
    int rc = msm_accumulate<CURVE>(ctx, B, jobs, n, n, src, false, st, &sh);
    if (rc) return rc;
    return msm_reduce<CURVE>(ctx, sh, true, d_extra, n_extra, d_partial, normalise, st, d_out_raw);
}

// run_msm over scalar vectors resident in HBM (one pointer per job), dispatched on the key's curve
int msm_mem(accmsm_ctx *ctx, const Bases &B, const MsmJobs &jobs, size_t n, const uint8_t *const *d_scalars, int mont,
            const xyzz_t *d_extra, uint32_t n_extra, xyzz_t *d_partial, bool normalise, cudaStream_t st,
            xyzz_t *d_out_raw = nullptr) {
    if (B.curve == 0) {
        MemScalars<1> src; src.montgomery = mont;
        for (uint32_t j = 0; j < MAX_JOBS; j++) src.ptr[j] = j < jobs.njobs ? d_scalars[j] : nullptr;
        return run_msm<0>(ctx, B, jobs, n, src, d_extra, n_extra, d_partial, normalise, st, d_out_raw);
    }
    MemScalars<0> src; src.montgomery = mont;
    for (uint32_t j = 0; j < MAX_JOBS; j++) src.ptr[j] = j < jobs.njobs ? d_scalars[j] : nullptr;
    return run_msm<1>(ctx, B, jobs, n, src, d_extra, n_extra, d_partial, normalise, st, d_out_raw);
}
int msm_mem1(accmsm_ctx *ctx, const Bases &B, size_t offset, size_t n, const uint8_t *d_scalars, int mont,
             const xyzz_t *d_extra, uint32_t n_extra, xyzz_t *d_partial, bool normalise, cudaStream_t st) {
    return msm_mem(ctx, B, MsmJobs(offset), n, &d_scalars, mont, d_extra, n_extra, d_partial, normalise, st, nullptr);
}

// Host -> device copy of a scalar / vector buffer.  Page-locked sources go straight to the DMA engine.  Pageable ones
// (a Rust Vec, a numpy array) would be staged by the driver on one thread at ~16 GB/s; here they are copied into a
// page-locked staging buffer by several threads, chunk by chunk, and every chunk's DMA overlaps the next chunk's memcpy.
int upload(accmsm_ctx *ctx, void *d_dst, const void *h_src, size_t bytes, cudaStream_t st) {
    if (!bytes) return ACCMSM_OK;
    constexpr size_t CHUNK = 4u << 20;
    bool pageable = false;
    if (bytes >= 2 * CHUNK) {
        cudaPointerAttributes attr;
        cudaError_t e = cudaPointerGetAttributes(&attr, h_src);
        if (e != cudaSuccess) { (void)cudaGetLastError(); pageable = true; }
        else pageable = attr.type == cudaMemoryTypeUnregistered;
    }
    if (!pageable) { CU(ctx, cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, st)); return ACCMSM_OK; }
    // one staging buffer: wait until the DMA of the previous upload has drained it
    if (ctx->stage_busy) { CU(ctx, cudaEventSynchronize(ctx->stage_done)); ctx->stage_busy = false; }
    if (ctx->stage_cap < bytes) {
        if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
        ctx->h_stage = nullptr; ctx->stage_cap = 0;
        CU(ctx, cudaMallocHost(&ctx->h_stage, bytes + bytes / 8));
        ctx->stage_cap = bytes + bytes / 8;
    }
    const char *src = (const char *)h_src;
    char *stage = (char *)ctx->h_stage;
    for (size_t off = 0; off < bytes; off += CHUNK) {
        const size_t len = std::min(CHUNK, bytes - off);
        const int parts = 4;
#pragma omp parallel for num_threads(parts) schedule(static)
        for (int p = 0; p < parts; p++) {
            size_t lo = len * p / parts, hi = len * (p + 1) / parts;
            memcpy(stage + off + lo, src + off + lo, hi - lo);
        }
        CU(ctx, cudaMemcpyAsync((char *)d_dst + off, stage + off, len, cudaMemcpyHostToDevice, st));
    }
    CU(ctx, cudaEventRecord(ctx->stage_done, st));
    ctx->stage_busy = true;
    return ACCMSM_OK;
}

// Device -> host copy of a result vector, the mirror image of upload(): for a large pageable destination every chunk is
// DMA'd into the page-locked staging buffer and copied out by several threads while the next chunks are in flight.
// Blocks until the data is in h_dst when it takes the staged path; otherwise only enqueues.
int download(accmsm_ctx *ctx, void *h_dst, const void *d_src, size_t bytes, cudaStream_t st) {
    if (!bytes) return ACCMSM_OK;
    constexpr size_t CHUNK = 4u << 20;
    bool pageable = false;
    if (bytes >= 2 * CHUNK) {
        cudaPointerAttributes attr;
        cudaError_t e = cudaPointerGetAttributes(&attr, h_dst);
        if (e != cudaSuccess) { (void)cudaGetLastError(); pageable = true; }
        else pageable = attr.type == cudaMemoryTypeUnregistered;
    }
    if (!pageable) { CU(ctx, cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, st)); return ACCMSM_OK; }
    if (ctx->stage_busy) { CU(ctx, cudaEventSynchronize(ctx->stage_done)); ctx->stage_busy = false; }
    if (ctx->stage_cap < bytes) {
        if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
        ctx->h_stage = nullptr; ctx->stage_cap = 0;
        CU(ctx, cudaMallocHost(&ctx->h_stage, bytes + bytes / 8));
        ctx->stage_cap = bytes + bytes / 8;
    }
    const size_t nchunks = (bytes + CHUNK - 1) / CHUNK;
    while (ctx->chunk_events.size() < nchunks) {
        cudaEvent_t ev;
        CU(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        ctx->chunk_events.push_back(ev);
    }
    char *dst = (char *)h_dst;
    const char *stage = (const char *)ctx->h_stage;
    for (size_t k = 0; k < nchunks; k++) {
        const size_t off = k * CHUNK, len = std::min(CHUNK, bytes - off);
        CU(ctx, cudaMemcpyAsync((char *)ctx->h_stage + off, (const char *)d_src + off, len, cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaEventRecord(ctx->chunk_events[k], st));
    }
    for (size_t k = 0; k < nchunks; k++) {
        const size_t off = k * CHUNK, len = std::min(CHUNK, bytes - off);
        CU(ctx, cudaEventSynchronize(ctx->chunk_events[k]));
        const int parts = 4;
#pragma omp parallel for num_threads(parts) schedule(static)
        for (int p = 0; p < parts; p++) {
            size_t lo = len * p / parts, hi = len * (p + 1) / parts;
            memcpy(dst + off + lo, stage + off + lo, hi - lo);
        }
    }
    return ACCMSM_OK;
}

// k un-normalised results (XYZZ in device memory) -> host, affine conversion on the host (hostfp.hpp, one inversion)
int fetch_points(accmsm_ctx *ctx, int curve, const xyzz_t *d_raw, size_t k, uint64_t *out_xy, uint8_t *out_inf, cudaStream_t st) {
    if (k > MAX_JOBS) return fail_arg(ctx, "fetch_points: too many results");
    CU(ctx, cudaMemcpyAsync(ctx->h_out, d_raw, k * sizeof(xyzz_t), cudaMemcpyDeviceToHost, st));
    CU(ctx, cudaStreamSynchronize(st));
    hostfp::xyzz_to_affine(curve == 0 ? 0 : 1, ctx->h_out, k, out_xy, out_inf);
    return ACCMSM_OK;
}
// the single result of the last pass -> host
int fetch_affine(accmsm_ctx *ctx, uint64_t out_xy[8], uint8_t *out_inf, cudaStream_t st) {
    mark(ctx, ST_D2H, st);
    CU(ctx, cudaMemcpyAsync(ctx->h_out, ctx->d_out_raw, sizeof(xyzz_t), cudaMemcpyDeviceToHost, st));
    mark(ctx, ST_COUNT, st);
    CU(ctx, cudaStreamSynchronize(st));
    hostfp::xyzz_to_affine(ctx->out_curve == 0 ? 0 : 1, ctx->h_out, 1, out_xy, out_inf);
    collect_timings(ctx);
    return ACCMSM_OK;
}

int write_identity(accmsm_ctx *ctx, int curve, uint64_t out_xy[8], uint8_t *out_inf) {
    (void)ctx;
    static const uint64_t R_P[4] = {0x34786d38fffffffdULL, 0x992c350be41914adULL, 0xffffffffffffffffULL, 0x3fffffffffffffffULL};
    static const uint64_t R_Q[4] = {0x5b2b3e9cfffffffdULL, 0x992c350be3420567ULL, 0xffffffffffffffffULL, 0x3fffffffffffffffULL};
    memset(out_xy, 0, 32);
    memcpy(out_xy + 4, curve == 0 ? R_P : R_Q, 32);
    *out_inf = 1;
    return ACCMSM_OK;
}

const Bases *find_bases(accmsm_ctx *ctx, uint64_t handle) {
    auto it = ctx->bases.find(handle);
    if (it == ctx->bases.end()) { ctx->last_error = "unknown bases handle"; return nullptr; }
    return &it->second;
}

// MSM of host scalars, one vector: uploads and enqueues on the ctx stream.  d_extra/n_extra: XYZZ partials added before
// normalisation.  d_partial (nullable): where the un-normalised sum goes (DEVICE memory, possibly a peer GPU's);
// normalise: the result goes to ctx->d_out_raw (XYZZ; fetch_affine converts it on the host).  The caller fetches / synchronises.
//
// Large vectors (>= 16 MiB) hide the PCIe transfer behind the arithmetic: the points are cut into two segments of 1/4 and
// 3/4 of the vector, the upload runs on a copy stream in 4 MiB chunks, and the second segment travels while the first one is
// sorted and accumulated; both segments add into ONE zero-initialised bucket set (k_accumulate `into` mode: no extra
// additions), then one reduction; the fix-up of the first segment runs on the side stream beside the sort of the second.
// The split balances "work on segment 0" against "upload of the rest" (0.15 + 2.3 f ms against 0.63 (1 - f) ms on a PCIe 5
// x16 link: f ~ 0.17; 12 % leaves the GPU waiting for data, 37 % exposes more of the first upload -- profiles/r02i_*,
// r02z_e2e_aux.txt; slower uploads, e.g. eight GPUs sharing one host, favour the larger first segment).  Every segment
// pays ~0.15 ms of fixed cost (sort launches, slice merge), so two segments beat three.  Pageable sources are staged chunk
// by chunk into page-locked memory by 4 threads on the way.
int msm_host_scalars(accmsm_ctx *ctx, const Bases &B, size_t offset, size_t n, const uint64_t *scalars, int mont,
                     const xyzz_t *d_extra, uint32_t n_extra, xyzz_t *d_partial, bool normalise) {
    cudaStream_t st = ctx->stream;
    CU(ctx, ctx->scalars.ensure(n * 32));
    mark(ctx, ST_H2D, st);
    constexpr size_t CHUNK = 4u << 20;
    const size_t bytes = n * 32;
    if (bytes < 4 * CHUNK || ctx->segments_override == 1) {
        { int urc = upload(ctx, ctx->scalars.p, scalars, bytes, st); if (urc) return urc; }
        return msm_mem1(ctx, B, offset, n, ctx->scalars.p, mont, d_extra, n_extra, d_partial, normalise, st);
    }
    if (!ctx->copy_stream) CU(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    const uint32_t nchunks = (uint32_t)((bytes + CHUNK - 1) / CHUNK), chunk_elems = (uint32_t)(CHUNK / 32);
    while (ctx->chunk_events.size() < nchunks) {
        cudaEvent_t ev;
        CU(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        ctx->chunk_events.push_back(ev);
    }
    cudaPointerAttributes attr;
    cudaError_t pe = cudaPointerGetAttributes(&attr, scalars);
    const bool pageable = pe != cudaSuccess || attr.type == cudaMemoryTypeUnregistered;
    if (pe != cudaSuccess) (void)cudaGetLastError();
    if (pageable) {
        if (ctx->stage_busy) { CU(ctx, cudaEventSynchronize(ctx->stage_done)); ctx->stage_busy = false; }
        if (ctx->stage_cap < bytes) {
            if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
            ctx->h_stage = nullptr; ctx->stage_cap = 0;
            CU(ctx, cudaMallocHost(&ctx->h_stage, bytes + bytes / 8));
            ctx->stage_cap = bytes + bytes / 8;
        }
    }
    const char *src = (const char *)scalars;
    char *stage = (char *)ctx->h_stage;
    // the copy stream must not overwrite scalars an earlier call on this ctx is still reading
    { int wrc = ws_acquire(ctx, st); if (wrc) return wrc; }
    CU(ctx, cudaEventRecord(ctx->stage_done, st));
    CU(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->stage_done, 0));
    auto feed = [&](uint32_t c) -> int {
        const size_t off = (size_t)c * CHUNK, len = std::min(CHUNK, bytes - off);
        const char *from = src + off;
        if (pageable) {
            const int parts = 4;
#pragma omp parallel for num_threads(parts) schedule(static)
            for (int p = 0; p < parts; p++) {
                size_t lo = len * p / parts, hi = len * (p + 1) / parts;
                memcpy(stage + off + lo, src + off + lo, hi - lo);
            }
            from = stage + off;
        }
        CU(ctx, cudaMemcpyAsync(ctx->scalars.p + off, from, len, cudaMemcpyHostToDevice, ctx->copy_stream));
        CU(ctx, cudaEventRecord(ctx->chunk_events[c], ctx->copy_stream));
        return ACCMSM_OK;
    };
    // segment boundaries on chunk boundaries
    const int nseg = ctx->segments_override > 1 ? ctx->segments_override : 2;
    std::vector<uint32_t> seg_end;       // in chunks
    if (!ctx->seg_pcts.empty()) { for (int pc : ctx->seg_pcts) seg_end.push_back(std::max(1u, (nchunks * (uint32_t)pc + 50) / 100)); seg_end.push_back(nchunks); }
    else if (nseg == 2) { seg_end.push_back(std::max(1u, (nchunks * (uint32_t)ctx->seg0_pct + 50) / 100)); seg_end.push_back(nchunks); }
    else for (int g = 1; g <= nseg; g++) seg_end.push_back(std::max<uint32_t>(g, (uint32_t)((uint64_t)nchunks * g / nseg)));
    seg_end.back() = nchunks;
    MsmShape sh;
    {   // all segments add into one bucket set: zero = identity
        const MsmShape s0 = make_shape(ctx, B, MsmJobs(offset), n, n);
        CU(ctx, ctx->buckets.ensure(s0.nkeys));
        CU(ctx, cudaMemsetAsync(ctx->buckets.p, 0, (size_t)s0.nkeys * sizeof(xyzz_t), st));
    }
    auto tr = [&](const std::string &label) { trace_point(ctx, st, label); };
    tr("start");
    uint32_t c0 = 0;
    for (size_t g = 0; g < seg_end.size(); g++) {
        const uint32_t c1 = std::min(seg_end[g], nchunks);
        if (c1 <= c0) continue;
        for (uint32_t c = c0; c < c1; c++) { int frc = feed(c); if (frc) return frc; }
        CU(ctx, cudaStreamWaitEvent(st, ctx->chunk_events[c1 - 1], 0));
        tr("seg" + std::to_string(g) + " arrived (chunks " + std::to_string(c0) + ".." + std::to_string(c1) + ")");
        const size_t e0 = (size_t)c0 * chunk_elems, e1 = std::min<size_t>(n, (size_t)c1 * chunk_elems);
        const uint8_t *ptr = ctx->scalars.p + e0 * 32;
        int rc;
        if (B.curve == 0) { MemScalars<1> ms; ms.montgomery = mont; for (uint32_t j = 0; j < MAX_JOBS; j++) ms.ptr[j] = j ? nullptr : ptr;
                            rc = msm_accumulate<0>(ctx, B, MsmJobs(offset + e0), e1 - e0, n, ms, true, st, &sh, c1 < nchunks); }
        else { MemScalars<0> ms; ms.montgomery = mont; for (uint32_t j = 0; j < MAX_JOBS; j++) ms.ptr[j] = j ? nullptr : ptr;
               rc = msm_accumulate<1>(ctx, B, MsmJobs(offset + e0), e1 - e0, n, ms, true, st, &sh, c1 < nchunks); }
        if (rc) return rc;
        tr("seg" + std::to_string(g) + " accumulated");
        c0 = c1;
    }
    if (pageable) { CU(ctx, cudaEventRecord(ctx->stage_done, ctx->copy_stream)); ctx->stage_busy = true; }
    const int rrc = B.curve == 0 ? msm_reduce<0>(ctx, sh, false, d_extra, n_extra, d_partial, normalise, st, nullptr)
                                 : msm_reduce<1>(ctx, sh, false, d_extra, n_extra, d_partial, normalise, st, nullptr);
    tr("reduced");
    return rrc;
}

// identity partial(s) into d_out[0..k)
template <int CURVE> void launch_identity_partials(accmsm_ctx *ctx, xyzz_t *d_out, uint32_t k, cudaStream_t st) {
    k_finish<CURVE><<<k, 32, 0, st>>>(nullptr, 0, 1, nullptr, 0, d_out, nullptr);
    ctx->launches++;
}
int launch_identity_partials(accmsm_ctx *ctx, int curve, xyzz_t *d_out, uint32_t k, cudaStream_t st) {
    if (curve == 0) launch_identity_partials<0>(ctx, d_out, k, st); else launch_identity_partials<1>(ctx, d_out, k, st);
    CU(ctx, cudaGetLastError());
    return ACCMSM_OK;
}

// k scalar vectors from the host (k x n x 32 B) against bases [offset, offset + n), optional last pair
// (base tail_index, tail[j]) per vector, as ONE pass per MAX_JOBS vectors; un-normalised sums -> d_partials[0..k)
// and/or affine images -> host.  Enqueues on the ctx stream and synchronises.
int msm_rows_host(accmsm_ctx *ctx, const Bases &B, size_t offset, size_t n, size_t k, const uint64_t *scalars, int mont,
                  size_t tail_index, const uint64_t *tail_scalars, xyzz_t *d_partials, uint64_t *out_xy, uint8_t *out_inf) {
    cudaStream_t st = ctx->stream;
    const bool tail = tail_scalars != nullptr;
    const size_t n_eff = n + (tail ? 1 : 0), row = n_eff * 32;
    clear_marks(ctx);
    if (n_eff == 0) {
        if (d_partials) { int rc = launch_identity_partials(ctx, B.curve, d_partials, (uint32_t)k, st); if (rc) return rc; }
        if (out_xy) for (size_t j = 0; j < k; j++) write_identity(ctx, B.curve, out_xy + 8 * j, out_inf + j);
        CU(ctx, cudaStreamSynchronize(st));
        return ACCMSM_OK;
    }
    CU(ctx, ctx->scalars.ensure(k * row));
    mark(ctx, ST_H2D, st);
    if (!tail) { int urc = upload(ctx, ctx->scalars.p, scalars, k * row, st); if (urc) return urc; }
    else for (size_t j = 0; j < k; j++) {
        if (n) { int urc = upload(ctx, ctx->scalars.p + j * row, scalars + j * n * 4, n * 32, st); if (urc) return urc; }
        { int urc = upload_small(ctx, ctx->scalars.p + j * row + n * 32, tail_scalars + 4 * j, 32, st); if (urc) return urc; }
    }
    for (size_t j0 = 0; j0 < k; j0 += MAX_JOBS) {
        MsmJobs jobs;
        jobs.njobs = (uint32_t)std::min<size_t>(MAX_JOBS, k - j0);
        if (tail) jobs.tail_base = (uint32_t)tail_index;
        const uint8_t *ptrs[MAX_JOBS];
        for (uint32_t j = 0; j < jobs.njobs; j++) { jobs.offset[j] = offset; ptrs[j] = ctx->scalars.p + (j0 + j) * row; }
        int rc = msm_mem(ctx, B, jobs, n_eff, ptrs, mont, nullptr, 0, d_partials ? d_partials + j0 : nullptr, out_xy != nullptr, st);
        if (rc) return rc;
        if (out_xy) {
            mark(ctx, ST_D2H, st);
            CU(ctx, cudaMemcpyAsync(ctx->h_out, ctx->d_out_raw, jobs.njobs * sizeof(xyzz_t), cudaMemcpyDeviceToHost, st));
            mark(ctx, ST_COUNT, st);
            CU(ctx, cudaStreamSynchronize(st));
            hostfp::xyzz_to_affine(B.curve == 0 ? 0 : 1, ctx->h_out, jobs.njobs, out_xy + 8 * j0, out_inf + j0);
        }
    }
    if (!out_xy) { mark(ctx, ST_COUNT, st); CU(ctx, cudaStreamSynchronize(st)); }
    collect_timings(ctx);
    return ACCMSM_OK;
}

}  // namespace

// ---- device-group layer (multi_api.inc): the same entry points over a key sharded by point range across GPUs
int group_destroy(accmsm_ctx *g);
int group_register_bases(accmsm_ctx *g, int curve, const uint64_t *xy, const uint8_t *infinity, size_t n, uint64_t seed,
                         uint64_t first_index, bool synthetic, uint64_t *handle);
int group_release_bases(accmsm_ctx *g, uint64_t handle);
int group_serialize_bases(accmsm_ctx *g, uint64_t handle, size_t offset, size_t n, uint8_t *out);
int group_precompute(accmsm_ctx *g, uint64_t handle, int window_bits);
int group_download_bases(accmsm_ctx *g, uint64_t handle, size_t offset, size_t n, uint64_t *xy_out);
int group_msm_rows(accmsm_ctx *g, uint64_t handle, size_t offset, size_t n, size_t k, const uint64_t *scalars, int mont,
                   bool has_tail, size_t tail_index, const uint64_t *tail_scalars, uint64_t *out_xy, uint8_t *out_inf);
int group_ipa_final_key(accmsm_ctx *g, uint64_t handle, const uint64_t *challenges_mont, int k, uint64_t out_xy[8], uint8_t *out_inf);
int group_hp_decide(accmsm_ctx *g, uint64_t handle, const uint64_t *a_mont, const uint64_t *b_mont, size_t n, size_t hiding_index,
                    const uint64_t *randomness_mont, uint64_t *xy, uint8_t *inf);
int group_hp_product_poly_comm(accmsm_ctx *g, uint64_t handle, const uint64_t *const *a_vecs, const size_t *a_lens,
                               const uint64_t *const *b_vecs, const size_t *b_lens, int n_in, const uint64_t *mu, size_t len,
                               const uint64_t *hiding_a, size_t n_ha, const uint64_t *hiding_b, size_t n_hb, uint64_t *out_low_xy,
                               uint8_t *out_low_inf, uint64_t *out_high_xy, uint8_t *out_high_inf, uint64_t *out_tvecs);
int group_register_csr(accmsm_ctx *g, int field, int n_mats, const uint32_t *const *row_ptr, const uint32_t *const *cols,
                       const uint64_t *const *coeffs_mont, size_t n_rows, uint64_t *handle);
int group_release_csr(accmsm_ctx *g, uint64_t handle);
template <class F>
int group_csr_pass(accmsm_ctx *g, const std::string &what, uint64_t key_handle, uint64_t csr_handle, size_t n_z, size_t n_hp,
                   size_t hiding_index, const uint64_t *tails_mont, size_t m, size_t n_vecs, uint64_t *const *out_vecs, uint64_t *out_xy,
                   uint8_t *out_inf, F run);
int group_open_key(accmsm_ctx *g, uint64_t handle, uint64_t *kid0_handle);     // full key on child 0 for IpaPC::open sessions
// hp-as prover sessions: every child holds the columns of its key shard
int group_hp_prove_begin(accmsm_ctx *g, uint64_t key_handle, const uint64_t *const *a_vecs, const size_t *a_lens,
                         const uint64_t *const *b_vecs, const size_t *b_lens, int n, size_t len, const uint64_t *hiding_a,
                         const uint64_t *hiding_b, size_t hiding_index, const uint64_t *rand_mont, uint64_t *comm_xy, uint8_t *comm_inf,
                         uint64_t *session);
int group_hp_prove_ppc(accmsm_ctx *g, uint64_t session, const uint64_t *mu_mont, size_t n_mu, uint64_t *low_xy, uint8_t *low_inf,
                       uint64_t *high_xy, uint8_t *high_inf);
int group_hp_prove_finish(accmsm_ctx *g, uint64_t session, const uint64_t nu_mont[4], uint64_t *a_star, uint64_t *b_star, size_t capacity,
                          size_t *out_len, bool nark_as = false, const uint64_t *beta_mont = nullptr, size_t n_beta = 0,
                          uint64_t *w_star = nullptr);
int group_hp_prove_abort(accmsm_ctx *g, uint64_t session);
// ASForR1CSNark::prove sessions: an hp session per child over its rows of the key and the matrices
int group_nark_as_prove_begin(accmsm_ctx *g, uint64_t key_handle, uint64_t csr_handle, int n_fresh, const uint64_t *const *inputs,
                              size_t n_input, const uint64_t *const *witnesses, size_t n_witness, int n_acc, const uint64_t *const *acc_w,
                              const uint64_t *const *acc_a, const size_t *acc_a_lens, const uint64_t *const *acc_b, const size_t *acc_b_lens,
                              const uint64_t *r_input, const uint64_t *r_witness, const uint64_t *hiding_a, const uint64_t *hiding_b,
                              size_t hiding_index, const uint64_t *tails_mont, uint64_t *comm_xy, uint8_t *comm_inf, uint64_t *session);
// IpaPC::open sessions sharded cyclically across the children of a group (multi_api.inc).  GROUP_IPA_UNSHARDED: the
// opening is too small to shard / the id is not a sharded session, and child 0 serves the call as before.
constexpr int GROUP_IPA_UNSHARDED = 1;
int group_ipa_begin(accmsm_ctx *g, uint64_t handle, const uint64_t *coeffs_mont, size_t n_coeffs, int k, const uint64_t point_mont[4],
                    const uint64_t h_prime_xy[8], const uint64_t *challenges_mont, int m, const uint64_t *alphas_mont,
                    const uint64_t *random_poly_mont, size_t n_random, uint64_t *session, uint64_t *eval_out);
int group_ipa_use_hiding_generator(accmsm_ctx *g, uint64_t session, size_t h_index, const uint64_t xi0_mont[4]);
int group_ipa_round(accmsm_ctx *g, uint64_t session, const uint64_t *xi_mont, uint64_t l_xy[8], uint8_t *l_inf, uint64_t r_xy[8],
                    uint8_t *r_inf, int *done);
int group_ipa_fold(accmsm_ctx *g, uint64_t session, const uint64_t xi_mont[4], const uint64_t xi_inv_mont[4]);
int group_ipa_finish(accmsm_ctx *g, uint64_t session, uint64_t final_key_xy[8], uint64_t c_mont[4]);
int group_ipa_hide(accmsm_ctx *g, uint64_t session, const uint64_t *hiding_mont, size_t n_hiding, size_t s_index,
                   const uint64_t rho_mont[4], uint64_t comm_xy[8], uint8_t *comm_inf);
int group_ipa_hiding_challenge(accmsm_ctx *g, uint64_t session, const uint64_t alpha_mont[4]);
inline bool is_group(const accmsm_ctx *ctx) { return ctx && !ctx->kids.empty(); }
// the result of a call a group forwarded to child 0, with child 0's error message
inline int group_fwd0(accmsm_ctx *g, int rc) { if (rc) g->last_error = g->kids[0]->last_error; return rc; }
// fn(child 0, handle of the whole key on child 0), forwarded: IpaPC::open sessions too small to shard
template <class F> int group_fwd0_open_key(accmsm_ctx *g, uint64_t handle, F fn) {
    uint64_t h0 = 0;
    { std::lock_guard<std::mutex> lock(g->mu); int rc = group_open_key(g, handle, &h0); if (rc) return rc; }
    return group_fwd0(g, fn(g->kids[0], h0));
}
#define GROUP_NO_DEV(ctx, name) do { if (is_group(ctx)) return fail_arg(ctx, name ": device-pointer entry points need a single-device ctx (accmsm_device_ctx)"); } while (0)

// =====================================================================================================
// C-ABI
// =====================================================================================================
extern "C" {

const char *accmsm_strerror(int code) {
    switch (code) {
        case ACCMSM_OK: return "ok";
        case ACCMSM_E_CUDA: return "CUDA runtime error";
        case ACCMSM_E_ARG: return "invalid argument";
        case ACCMSM_E_HANDLE: return "unknown bases handle";
        case ACCMSM_E_NOMEM: return "out of device or pinned memory";
        default: return "unknown error";
    }
}

const char *accmsm_last_error(accmsm_ctx *ctx) { return ctx ? ctx->last_error.c_str() : "null ctx"; }

const char *accmsm_stage_name(int stage) { return stage >= 0 && stage < ST_COUNT ? STAGE_NAMES[stage] : ""; }

int accmsm_init(accmsm_ctx **out, int device) {
    if (!out) return ACCMSM_E_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0 || device < 0 || device >= count) return ACCMSM_E_CUDA;
    if (cudaSetDevice(device) != cudaSuccess) return ACCMSM_E_CUDA;
    accmsm_ctx *ctx = new accmsm_ctx();
    ctx->device = device;
    if (const char *e = getenv("ACCMSM_AFFINE_ROUNDS")) ctx->affine_rounds_override = atoi(e);
    if (const char *e = getenv("ACCMSM_SORT_LB")) ctx->sort_lb_override = atoi(e);
    if (const char *e = getenv("ACCMSM_SEGMENTS")) ctx->segments_override = atoi(e);
    if (const char *e = getenv("ACCMSM_SEG0_PCT")) ctx->seg0_pct = std::min(90, std::max(1, atoi(e)));
    if (const char *e = getenv("ACCMSM_SEG_PCTS")) { for (const char *q = e; *q;) { ctx->seg_pcts.push_back(atoi(q)); while (*q && *q != ',') q++; if (*q) q++; } }
    if (const char *e = getenv("ACCMSM_TRACE")) ctx->trace = atoi(e) != 0;
    if (const char *e = getenv("ACCMSM_NO_AUX")) ctx->no_aux = atoi(e) != 0;
    if (const char *e = getenv("ACCMSM_NO_IPA_TABS")) ctx->no_ipa_tabs = atoi(e) != 0;
    if (const char *e = getenv("ACCMSM_NO_COOP_FINISH")) ctx->no_coop_finish = atoi(e) != 0;
    if (const char *e = getenv("ACCMSM_NO_COOP_PRECOMPUTE")) ctx->no_coop_precompute = atoi(e) != 0;
    if (const char *e = getenv("ACCMSM_FK_C")) ctx->fk_small_c = atoi(e);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete ctx; return ACCMSM_E_CUDA; }
    ctx->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return ACCMSM_E_CUDA; }
    for (int i = 0; i <= ST_COUNT; i++) { cudaEventCreate(&ctx->ev[i]); ctx->ev_valid[i] = false; }
    cudaEventCreateWithFlags(&ctx->stage_done, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&ctx->ws_done, cudaEventDisableTiming);
    for (int i = 0; i < accmsm_ctx::ARG_SLOTS; i++) cudaEventCreateWithFlags(&ctx->arg_done[i], cudaEventDisableTiming);
    bool ok = cudaMallocHost(&ctx->h_args, accmsm_ctx::ARG_SLOTS * accmsm_ctx::ARG_SLOT_BYTES) == cudaSuccess && cudaMalloc(&ctx->d_out_raw, MAX_JOBS * sizeof(xyzz_t)) == cudaSuccess &&
              cudaMallocHost(&ctx->h_out, (MAX_JOBS * 16 + 64) * sizeof(uint64_t)) == cudaSuccess;
    // shared-memory opt-in and resident CTAs per SM for the accumulate kernels
    size_t smem = 2 * ACC_THREADS * (sizeof(xyzz_t) + sizeof(uint32_t));
    size_t smem_fix = (size_t)FIX_THREADS * FIX_PER_T * (sizeof(xyzz_t) + sizeof(uint32_t));
    ok = ok && cudaFuncSetAttribute(k_accumulate<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(k_accumulate<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(k_accumulate<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(k_accumulate<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess;
    // the sort kernels opt in ONCE to the most dynamic shared memory they can ever ask for: the attribute is per function
    // and device, not per ctx, and the ctxs of a device group launch concurrently from several threads
    ok = ok && sort_opt_in<MemScalars<0>>() && sort_opt_in<MemScalars<1>>() && sort_opt_in<IpaScalars<0>>() && sort_opt_in<IpaScalars<1>>() &&
         sort_opt_in<IpaRoundScalars<0>>() && sort_opt_in<IpaRoundScalars<1>>() &&
         cudaFuncSetAttribute(k_sort_buckets, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SORT_SMEM_OPT_IN) == cudaSuccess;
    {   // k_tvecs: 2 n_in TVEC_THREADS field elements, n_in <= VEC_MAX_INPUTS
        const int tv = 2 * VEC_MAX_INPUTS * TVEC_THREADS * (int)sizeof(fe_t);
        ok = ok && cudaFuncSetAttribute(k_tvecs<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, tv) == cudaSuccess &&
             cudaFuncSetAttribute(k_tvecs<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, tv) == cudaSuccess;
    }
    ok = ok && cudaFuncSetAttribute(k_fixup<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::min<size_t>(smem_fix, 227 * 1024)) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(k_fixup<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::min<size_t>(smem_fix, 227 * 1024)) == cudaSuccess;
    if (ok) {
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->acc_ctas_per_sm[0], k_accumulate<0, false>, ACC_THREADS, smem);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->acc_ctas_per_sm[1], k_accumulate<1, false>, ACC_THREADS, smem);
        for (int c = 0; c < 2; c++) {
            if (ctx->acc_ctas_per_sm[c] < 1) ctx->acc_ctas_per_sm[c] = 1;
            // k_fixup holds 2 slots per accumulate CTA: at most FIX_THREADS * FIX_PER_T slots
            int cap = (FIX_THREADS * FIX_PER_T / 2) / ctx->sm_count;
            if (ctx->acc_ctas_per_sm[c] > cap) ctx->acc_ctas_per_sm[c] = std::max(1, cap);
        }
    }
    if (!ok) {
        ctx->last_error = cudaGetErrorString(cudaGetLastError());
        accmsm_destroy(ctx);
        return ACCMSM_E_CUDA;
    }
    *out = ctx;
    return ACCMSM_OK;
}

void accmsm_destroy(accmsm_ctx *ctx) {
    if (!ctx) return;
    if (is_group(ctx)) { group_destroy(ctx); return; }
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (auto &kv : ctx->bases) {
        cudaFree(kv.second.d_xy);
        if (kv.second.d_inf) cudaFree(kv.second.d_inf);
        if (kv.second.d_table) cudaFree(kv.second.d_table);
    }
    for (auto &kv : ctx->ipa_sessions) ipa_session_free(kv.second);
    for (auto *fs : ctx->ipa_free) ipa_session_free(fs);
    for (auto &kv : ctx->csr_sets) csr_set_free(kv.second);
    for (auto &kv : ctx->hp_sessions) hp_session_free(ctx, kv.second);     // before the cache their blocks return to
    for (auto &b : ctx->vec_cache) cudaFree(b.first);
    ctx->digits.release(); ctx->hist.release(); ctx->offsets.release(); ctx->cursor.release(); ctx->entries.release();
    ctx->cta_ids.release(); ctx->tile_sums.release(); ctx->tile_offs.release(); ctx->buckets.release(); ctx->cta_parts.release(); ctx->partial.release();
    ctx->scalars.release(); ctx->misc.release(); ctx->oneshot_xy.release(); ctx->oneshot_inf.release(); ctx->ipa_tabs.release();
    ctx->sort_pairs.release(); ctx->sort_tile_count.release(); ctx->sort_part_count.release(); ctx->sort_part_offs.release();
    for (int i = 0; i < 2; i++) { ctx->pair_pts[i].release(); ctx->pair_off[i].release(); }
    ctx->fold_partial.release(); ctx->fold_flag.release();
    ctx->pair_pref.release(); ctx->pair_kinds.release(); ctx->pair_tfac.release(); ctx->pair_ctot.release(); ctx->pair_cfac.release();
    for (int i = 0; i < 2; i++) { ctx->red_sum[i].release(); ctx->red_wsum[i].release(); }
    if (ctx->d_out_raw) cudaFree(ctx->d_out_raw);
    if (ctx->h_out) cudaFreeHost(ctx->h_out);
    if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
    if (ctx->stage_done) cudaEventDestroy(ctx->stage_done);
    if (ctx->ws_done) cudaEventDestroy(ctx->ws_done);
    for (int i = 0; i < accmsm_ctx::ARG_SLOTS; i++) if (ctx->arg_done[i]) cudaEventDestroy(ctx->arg_done[i]);
    if (ctx->h_args) cudaFreeHost(ctx->h_args);
    for (cudaEvent_t ev : ctx->chunk_events) cudaEventDestroy(ev);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
    if (ctx->aux_fork) cudaEventDestroy(ctx->aux_fork);
    if (ctx->aux_join) cudaEventDestroy(ctx->aux_join);
    for (int i = 0; i <= ST_COUNT; i++) cudaEventDestroy(ctx->ev[i]);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

// Page-locked host memory for scalar / vector buffers: H2D from pinned memory runs at the PCIe rate (~53 GB/s
// measured), from pageable memory at ~16 GB/s (2 ms instead of 0.6 ms for 2^20 scalars).
void *accmsm_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaMallocHost(&p, std::max<size_t>(bytes, 1)) != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }
    return p;
}
void accmsm_host_free(void *p) { if (p) cudaFreeHost(p); }

int accmsm_set_window_bits(accmsm_ctx *ctx, int c) {
    if (!ctx || c < 0 || c > 16 || c == 1) return fail_arg(ctx, "window bits must be 0 (auto) or 2..16");
    for (accmsm_ctx *kid : ctx->kids) kid->window_bits = c;
    ctx->window_bits = c;
    return ACCMSM_OK;
}

int accmsm_set_ipa_fold(accmsm_ctx *ctx, int rounds, int min_log_n) {
    if (!ctx || rounds < 0 || rounds > 10 || min_log_n < 0 || min_log_n > 31)
        return fail_arg(ctx, "set_ipa_fold: rounds must be 0 (never) or 1..10, min_log_n 0..31");
    for (accmsm_ctx *kid : ctx->kids) accmsm_set_ipa_fold(kid, rounds, min_log_n);
    std::lock_guard<std::mutex> lock(ctx->mu);
    ctx->ipa_fold_rounds = rounds; ctx->ipa_fold_min_log = min_log_n;
    return ACCMSM_OK;
}

uint64_t accmsm_kernel_launches(accmsm_ctx *ctx) {
    if (!ctx) return 0;
    uint64_t total = ctx->launches;
    for (accmsm_ctx *kid : ctx->kids) total += kid->launches;
    return total;
}

int accmsm_last_timings(accmsm_ctx *ctx, float *ms_out, int max_stages) {
    if (!ctx || !ms_out) return ACCMSM_E_ARG;
    int k = std::min<int>(max_stages, ST_COUNT);
    if (is_group(ctx)) {        // per stage: the slowest child (the children run concurrently)
        for (int i = 0; i < k; i++) ms_out[i] = 0.f;
        float tmp[ST_COUNT];
        for (accmsm_ctx *kid : ctx->kids) {
            accmsm_last_timings(kid, tmp, k);
            for (int i = 0; i < k; i++) ms_out[i] = std::max(ms_out[i], tmp[i]);
        }
        return k;
    }
    // calls that only enqueued on a caller stream are collected here, once the caller has synchronised
    std::lock_guard<std::mutex> lock(ctx->mu);
    collect_timings(ctx);
    for (int i = 0; i < k; i++) ms_out[i] = ctx->timings[i];
    return k;
}

int accmsm_register_bases(accmsm_ctx *ctx, int curve, const uint64_t *xy, const uint8_t *infinity, size_t n,
                          uint64_t *handle) {
    if (!ctx || !handle || (curve != 0 && curve != 1) || (n && !xy)) return fail_arg(ctx, "register_bases: bad argument");
    if (is_group(ctx)) return group_register_bases(ctx, curve, xy, infinity, n, 0, 0, false, handle);
    if (n >= (size_t(1) << 31)) return fail_arg(ctx, "register_bases: n must be < 2^31");
    std::lock_guard<std::mutex> lock(ctx->mu);
    CU(ctx, cudaSetDevice(ctx->device));
    Bases B;
    B.curve = curve; B.n = n;
    CU(ctx, cudaMalloc(&B.d_xy, std::max<size_t>(n, 1) * sizeof(affine_t)));
    if (n) { int urc = upload(ctx, B.d_xy, xy, n * sizeof(affine_t), ctx->stream); if (urc) { cudaFree(B.d_xy); return urc; } }
    bool any_inf = false;
    if (infinity) for (size_t i = 0; i < n && !any_inf; i++) any_inf = infinity[i] != 0;
    if (any_inf) {
        CU(ctx, cudaMalloc(&B.d_inf, n));
        CU(ctx, cudaMemcpyAsync(B.d_inf, infinity, n, cudaMemcpyHostToDevice, ctx->stream));
    }
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    *handle = ctx->next_handle++;
    ctx->bases[*handle] = B;
    return ACCMSM_OK;
}

int accmsm_register_synthetic_bases(accmsm_ctx *ctx, int curve, uint64_t seed, uint64_t first_index, size_t n,
                                    uint64_t *handle) {
    if (!ctx || !handle || (curve != 0 && curve != 1)) return fail_arg(ctx, "register_synthetic_bases: bad argument");
    if (is_group(ctx)) return group_register_bases(ctx, curve, nullptr, nullptr, n, seed, first_index, true, handle);
    if (n >= (size_t(1) << 31)) return fail_arg(ctx, "register_synthetic_bases: n must be < 2^31");
    std::lock_guard<std::mutex> lock(ctx->mu);
    CU(ctx, cudaSetDevice(ctx->device));
    Bases B;
    B.curve = curve; B.n = n;
    CU(ctx, cudaMalloc(&B.d_xy, std::max<size_t>(n, 1) * sizeof(affine_t)));
    if (n) {
        uint32_t blocks = (uint32_t)((n + 127) / 128);
        if (curve == 0) k_synth_points<0><<<blocks, 128, 0, ctx->stream>>>(seed, first_index, (uint32_t)n, B.d_xy);
        else k_synth_points<1><<<blocks, 128, 0, ctx->stream>>>(seed, first_index, (uint32_t)n, B.d_xy);
        ctx->launches++;
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) { cudaFree(B.d_xy); CU(ctx, e); }
    }
    *handle = ctx->next_handle++;
    ctx->bases[*handle] = B;
    return ACCMSM_OK;
}

int accmsm_precompute_bases(accmsm_ctx *ctx, uint64_t handle, int window_bits) {
    if (!ctx || window_bits < 0 || (window_bits && (window_bits < 4 || window_bits > 21)))
        return fail_arg(ctx, "precompute_bases: window bits must be 0 (auto) or 4..21");
    if (is_group(ctx)) return group_precompute(ctx, handle, window_bits);
    std::lock_guard<std::mutex> lock(ctx->mu);
    auto it = ctx->bases.find(handle);
    if (it == ctx->bases.end()) { ctx->last_error = "unknown bases handle"; return ACCMSM_E_HANDLE; }
    CU(ctx, cudaSetDevice(ctx->device));
    return precompute_table(ctx, it->second, window_bits);
}

int accmsm_download_bases(accmsm_ctx *ctx, uint64_t handle, size_t offset, size_t n, uint64_t *xy_out) {
    if (!ctx || (n && !xy_out)) return fail_arg(ctx, "download_bases: bad argument");
    if (is_group(ctx)) return group_download_bases(ctx, handle, offset, n, xy_out);
    std::lock_guard<std::mutex> lock(ctx->mu);
    const Bases *B = find_bases(ctx, handle);
    if (!B) return ACCMSM_E_HANDLE;
    if (offset > B->n || n > B->n - offset) return fail_arg(ctx, "download_bases: range exceeds registered bases");
    CU(ctx, cudaSetDevice(ctx->device));
    if (n) { int drc = download(ctx, xy_out, B->d_xy + offset, n * sizeof(affine_t), ctx->stream); if (drc) return drc; }
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return ACCMSM_OK;
}

int accmsm_release_bases(accmsm_ctx *ctx, uint64_t handle) {
    if (!ctx) return ACCMSM_E_ARG;
    if (is_group(ctx)) return group_release_bases(ctx, handle);
    std::lock_guard<std::mutex> lock(ctx->mu);
    auto it = ctx->bases.find(handle);
    if (it == ctx->bases.end()) { ctx->last_error = "unknown bases handle"; return ACCMSM_E_HANDLE; }
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaFree(it->second.d_xy);
    if (it->second.d_inf) cudaFree(it->second.d_inf);
    if (it->second.d_table) cudaFree(it->second.d_table);
    ctx->bases.erase(it);
    return ACCMSM_OK;
}

int accmsm_msm(accmsm_ctx *ctx, uint64_t handle, size_t offset, size_t n, const uint64_t *scalars,
               int scalars_montgomery, uint64_t out_xy[8], uint8_t *out_inf) {
    if (!ctx || !out_xy || !out_inf || (n && !scalars)) return fail_arg(ctx, "msm: bad argument");
    if (is_group(ctx)) return group_msm_rows(ctx, handle, offset, n, 1, scalars, scalars_montgomery, false, 0, nullptr, out_xy, out_inf);
    std::lock_guard<std::mutex> lock(ctx->mu);
    const Bases *B = find_bases(ctx, handle);
    if (!B) return ACCMSM_E_HANDLE;
    if (offset > B->n || n > B->n - offset) return fail_arg(ctx, "msm: range exceeds registered bases");
    if (n == 0) return write_identity(ctx, B->curve, out_xy, out_inf);
    CU(ctx, cudaSetDevice(ctx->device));
    int rc = msm_host_scalars(ctx, *B, offset, n, scalars, scalars_montgomery, nullptr, 0, nullptr, true);
    if (rc) return rc;
    return fetch_affine(ctx, out_xy, out_inf, ctx->stream);
}

// VariableBaseMSM::multi_scalar_mul(&bases, &scalars) for bases that are not a registered key (the literal ark-ec
// signature; in the reference: the O(log D) / O(n_inputs) linear combinations of commitments, e.g.
// src/hp_as/mod.rs:391-406, src/ipa_pc_as/mod.rs:322-343).  Bases go up with the call and are dropped after it.
int accmsm_msm_oneshot(accmsm_ctx *ctx, int curve, const uint64_t *bases_xy, const uint8_t *infinity, const uint64_t *scalars,
                       int scalars_montgomery, size_t n, uint64_t out_xy[8], uint8_t *out_inf) {
    if (!ctx || !out_xy || !out_inf || (curve != 0 && curve != 1) || (n && (!bases_xy || !scalars)) || n >= (size_t(1) << 31))
        return fail_arg(ctx, "msm_oneshot: bad argument");
    if (is_group(ctx)) return accmsm_msm_oneshot(ctx->kids[0], curve, bases_xy, infinity, scalars, scalars_montgomery, n, out_xy, out_inf);
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (n == 0) return write_identity(ctx, curve, out_xy, out_inf);
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    clear_marks(ctx);
    CU(ctx, ctx->scalars.ensure(n * 32));
    CU(ctx, ctx->oneshot_xy.ensure(n));
    mark(ctx, ST_H2D, st);
    CU(ctx, cudaMemcpyAsync(ctx->oneshot_xy.p, bases_xy, n * sizeof(affine_t), cudaMemcpyHostToDevice, st));
    CU(ctx, cudaMemcpyAsync(ctx->scalars.p, scalars, n * 32, cudaMemcpyHostToDevice, st));
    Bases B;
    B.curve = curve; B.n = n; B.d_xy = ctx->oneshot_xy.p;
    bool any_inf = false;
    if (infinity) for (size_t i = 0; i < n && !any_inf; i++) any_inf = infinity[i] != 0;
    if (any_inf) {
        CU(ctx, ctx->misc.ensure(std::max<size_t>(n, 64 * 32)));
        CU(ctx, cudaMemcpyAsync(ctx->misc.p, infinity, n, cudaMemcpyHostToDevice, st));
        B.d_inf = ctx->misc.p;
    }
    int rc = msm_mem1(ctx, B, 0, n, ctx->scalars.p, scalars_montgomery, nullptr, 0, nullptr, true, st);
    if (rc) return rc;
    return fetch_affine(ctx, out_xy, out_inf, st);
}

// m independent one-shot MSMs of the same length n, each over its OWN bases (bases_xy: m x n x 8 u64, scalars: m x n x 4 u64,
// infinity: m x n bytes or NULL): the succinct-check group equations of all inputs and accumulators of one
// AtomicASForInnerProductArgPC::prove / verify (src/ipa_pc_as/mod.rs:198-205 is called once per input, :262-270 / :625-640
// loop over them; 2k + 3 terms each).  Up to MAX_JOBS of them share one pass of the pipeline, so the latency-bound tail of a
// short MSM (bucket reduction, Horner over the windows) is paid once per pass, not once per equation.
int accmsm_msm_oneshot_batch(accmsm_ctx *ctx, int curve, const uint64_t *bases_xy, const uint8_t *infinity, const uint64_t *scalars,
                             int scalars_montgomery, size_t n, size_t m, uint64_t *out_xy, uint8_t *out_inf) {
    if (!ctx || (m && (!out_xy || !out_inf)) || (curve != 0 && curve != 1) || (n && m && (!bases_xy || !scalars)) ||
        n >= (size_t(1) << 31) || m >= (size_t(1) << 20) || n * m >= (size_t(1) << 31))
        return fail_arg(ctx, "msm_oneshot_batch: bad argument");
    if (is_group(ctx)) return accmsm_msm_oneshot_batch(ctx->kids[0], curve, bases_xy, infinity, scalars, scalars_montgomery, n, m, out_xy, out_inf);
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (m == 0) return ACCMSM_OK;
    if (n == 0) { for (size_t j = 0; j < m; j++) write_identity(ctx, curve, out_xy + 8 * j, out_inf + j); return ACCMSM_OK; }
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    clear_marks(ctx);
    CU(ctx, ctx->scalars.ensure(m * n * 32));
    CU(ctx, ctx->oneshot_xy.ensure(m * n));
    mark(ctx, ST_H2D, st);
    { int urc = upload(ctx, ctx->oneshot_xy.p, bases_xy, m * n * sizeof(affine_t), st); if (urc) return urc; }
    { int urc = upload(ctx, ctx->scalars.p, scalars, m * n * 32, st); if (urc) return urc; }
    Bases B;
    B.curve = curve; B.n = m * n; B.d_xy = ctx->oneshot_xy.p;
    bool any_inf = false;
    if (infinity) for (size_t i = 0; i < m * n && !any_inf; i++) any_inf = infinity[i] != 0;
    if (any_inf) {
        CU(ctx, ctx->oneshot_inf.ensure(m * n));
        { int urc = upload(ctx, ctx->oneshot_inf.p, infinity, m * n, st); if (urc) return urc; }
        B.d_inf = ctx->oneshot_inf.p;
    }
    for (size_t j0 = 0; j0 < m; j0 += MAX_JOBS) {
        MsmJobs jobs;
        jobs.njobs = (uint32_t)std::min<size_t>(MAX_JOBS, m - j0);
        const uint8_t *ptrs[MAX_JOBS];
        for (uint32_t j = 0; j < jobs.njobs; j++) { jobs.offset[j] = (j0 + j) * n; ptrs[j] = ctx->scalars.p + (j0 + j) * n * 32; }
        int rc = msm_mem(ctx, B, jobs, n, ptrs, scalars_montgomery, nullptr, 0, nullptr, true, st);
        if (rc) return rc;
        mark(ctx, ST_D2H, st);
        rc = fetch_points(ctx, curve, ctx->d_out_raw, jobs.njobs, out_xy + 8 * j0, out_inf + j0, st);
        if (rc) return rc;
    }
    mark(ctx, ST_COUNT, st);
    collect_timings(ctx);
    return ACCMSM_OK;
}

int accmsm_msm_batch(accmsm_ctx *ctx, uint64_t handle, size_t offset, size_t n, size_t k, const uint64_t *scalars,
                     int scalars_montgomery, uint64_t *out_xy, uint8_t *out_inf) {
    if (!ctx || (k && (!out_xy || !out_inf)) || (n && k && !scalars)) return fail_arg(ctx, "msm_batch: bad argument");
    if (is_group(ctx)) return group_msm_rows(ctx, handle, offset, n, k, scalars, scalars_montgomery, false, 0, nullptr, out_xy, out_inf);
    std::lock_guard<std::mutex> lock(ctx->mu);
    const Bases *B = find_bases(ctx, handle);
    if (!B) return ACCMSM_E_HANDLE;
    if (offset > B->n || n > B->n - offset) return fail_arg(ctx, "msm_batch: range exceeds registered bases");
    if (n == 0) { for (size_t j = 0; j < k; j++) write_identity(ctx, B->curve, out_xy + 8 * j, out_inf + j); return ACCMSM_OK; }
    CU(ctx, cudaSetDevice(ctx->device));
    // all k scalar vectors go up in one copy; groups of MAX_JOBS share one pass of the pipeline (one sort,
    // one accumulation over all their bucket sets, one reduction, one finish launch)
    return msm_rows_host(ctx, *B, offset, n, k, scalars, scalars_montgomery, 0, nullptr, nullptr, out_xy, out_inf);
}

int accmsm_commit(accmsm_ctx *ctx, uint64_t handle, size_t n, const uint64_t *elems_mont, size_t hiding_index,
                  const uint64_t *randomizer_mont, uint64_t out_xy[8], uint8_t *out_inf) {
    if (!ctx || !out_xy || !out_inf || (n && !elems_mont)) return fail_arg(ctx, "commit: bad argument");
    if (!randomizer_mont) return accmsm_msm(ctx, handle, 0, n, elems_mont, 1, out_xy, out_inf);
    if (is_group(ctx)) return group_msm_rows(ctx, handle, 0, n, 1, elems_mont, 1, true, hiding_index, randomizer_mont, out_xy, out_inf);
    std::lock_guard<std::mutex> lock(ctx->mu);
    const Bases *B = find_bases(ctx, handle);
    if (!B) return ACCMSM_E_HANDLE;
    if (n > B->n || hiding_index >= B->n) return fail_arg(ctx, "commit: range exceeds registered bases");
    CU(ctx, cudaSetDevice(ctx->device));
    // one pass over n + 1 pairs: the elements against the generators, then (hiding generator, randomizer)
    return msm_rows_host(ctx, *B, 0, n, 1, elems_mont, 1, hiding_index, randomizer_mont, nullptr, out_xy, out_inf);
}

int accmsm_msm_dev(accmsm_ctx *ctx, uint64_t handle, size_t offset, size_t n, const void *d_scalars,
                   int scalars_montgomery, uint64_t out_xy[8], uint8_t *out_inf, void *stream) {
    if (!ctx || !out_xy || !out_inf || (n && !d_scalars)) return fail_arg(ctx, "msm_dev: bad argument");
    GROUP_NO_DEV(ctx, "msm_dev");
    std::lock_guard<std::mutex> lock(ctx->mu);
    const Bases *B = find_bases(ctx, handle);
    if (!B) return ACCMSM_E_HANDLE;
    if (offset > B->n || n > B->n - offset) return fail_arg(ctx, "msm_dev: range exceeds registered bases");
    if (n == 0) return write_identity(ctx, B->curve, out_xy, out_inf);
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
    clear_marks(ctx);
    int rc = msm_mem1(ctx, *B, offset, n, (const uint8_t *)d_scalars, scalars_montgomery, nullptr, 0, nullptr, true, st);
    if (rc) return rc;
    return fetch_affine(ctx, out_xy, out_inf, st);
}

int accmsm_msm_partial_dev(accmsm_ctx *ctx, uint64_t handle, size_t offset, size_t n, const void *d_scalars,
                           int scalars_montgomery, void *d_out_partial, void *stream) {
    if (!ctx || !d_out_partial || (n && !d_scalars)) return fail_arg(ctx, "msm_partial_dev: bad argument");
    GROUP_NO_DEV(ctx, "msm_partial_dev");
    std::lock_guard<std::mutex> lock(ctx->mu);
    const Bases *B = find_bases(ctx, handle);
    if (!B) return ACCMSM_E_HANDLE;
    if (offset > B->n || n > B->n - offset) return fail_arg(ctx, "msm_partial_dev: range exceeds registered bases");
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
    clear_marks(ctx);
    int rc;
    if (n == 0) {
        { int wrc = ws_acquire(ctx, st); if (wrc) return wrc; }
        if (B->curve == 0) k_finish<0><<<1, 32, 0, st>>>(nullptr, 0, 1, nullptr, 0, (xyzz_t *)d_out_partial, nullptr);
        else k_finish<1><<<1, 32, 0, st>>>(nullptr, 0, 1, nullptr, 0, (xyzz_t *)d_out_partial, nullptr);
        ctx->launches++;
        rc = ws_release(ctx, st);
    } else {
        rc = msm_mem1(ctx, *B, offset, n, (const uint8_t *)d_scalars, scalars_montgomery, nullptr, 0, (xyzz_t *)d_out_partial, false, st);
    }
    if (rc) return rc;
    mark(ctx, ST_COUNT, st);
    if (!stream) { CU(ctx, cudaStreamSynchronize(st)); collect_timings(ctx); }
    return ACCMSM_OK;
}

// k scalar vectors from HOST memory against bases [offset, offset + n); optional last pair (base tail_index,
// tail_scalars[j]) per vector; the k un-normalised sums go to d_out_partials (DEVICE memory, k x 16 u64, possibly a peer
// GPU's).  One GPU's share of msm / msm_batch / commit when the key is sharded by point range.  Blocking.
int accmsm_msm_partial(accmsm_ctx *ctx, uint64_t handle, size_t offset, size_t n, size_t k, const uint64_t *scalars,
                       int scalars_montgomery, size_t tail_index, const uint64_t *tail_scalars, void *d_out_partials) {
    if (!ctx || is_group(ctx) || !d_out_partials || k == 0 || (n && !scalars)) return fail_arg(ctx, "msm_partial: bad argument");
    std::lock_guard<std::mutex> lock(ctx->mu);
    const Bases *B = find_bases(ctx, handle);
    if (!B) return ACCMSM_E_HANDLE;
    if (offset > B->n || n > B->n - offset || (tail_scalars && tail_index >= B->n)) return fail_arg(ctx, "msm_partial: range exceeds registered bases");
    CU(ctx, cudaSetDevice(ctx->device));
    if (k == 1 && !tail_scalars && n) {       // the single-vector path overlaps the digit kernel with a chunked upload
        clear_marks(ctx);
        int rc = msm_host_scalars(ctx, *B, offset, n, scalars, scalars_montgomery, nullptr, 0, (xyzz_t *)d_out_partials, false);
        if (rc) return rc;
        mark(ctx, ST_COUNT, ctx->stream);
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        collect_timings(ctx);
        return ACCMSM_OK;
    }
    return msm_rows_host(ctx, *B, offset, n, k, scalars, scalars_montgomery, tail_index, tail_scalars, (xyzz_t *)d_out_partials, nullptr, nullptr);
}

int accmsm_combine_partials_dev(accmsm_ctx *ctx, int curve, const void *d_partials, size_t k, uint64_t out_xy[8],
                                uint8_t *out_inf, void *stream) {
    if (!ctx || !out_xy || !out_inf || (k && !d_partials) || (curve != 0 && curve != 1)) return fail_arg(ctx, "combine_partials: bad argument");
    GROUP_NO_DEV(ctx, "combine_partials_dev");
    std::lock_guard<std::mutex> lock(ctx->mu);
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
    // stage marks of a preceding accmsm_*_partial_dev on the same stream are kept (bench.py reads them)
    { int wrc = ws_acquire(ctx, st); if (wrc) return wrc; }
    mark(ctx, ST_FINISH, st);
    if (curve == 0) k_finish<0><<<1, 32, 0, st>>>(nullptr, 0, 1, (const xyzz_t *)d_partials, (uint32_t)k, nullptr, ctx->d_out_raw);
    else k_finish<1><<<1, 32, 0, st>>>(nullptr, 0, 1, (const xyzz_t *)d_partials, (uint32_t)k, nullptr, ctx->d_out_raw);
    ctx->out_curve = curve;
    ctx->launches++;
    return fetch_affine(ctx, out_xy, out_inf, st);
}

int accmsm_combine_partials_batch_dev(accmsm_ctx *ctx, int curve, const void *d_partials, size_t k, size_t m, uint64_t *out_xy,
                                      uint8_t *out_inf, void *stream) {
    if (!ctx || !out_xy || !out_inf || !d_partials || k == 0 || m == 0 || m > MAX_JOBS || (curve != 0 && curve != 1))
        return fail_arg(ctx, "combine_partials_batch: bad argument");
    GROUP_NO_DEV(ctx, "combine_partials_batch_dev");
    std::lock_guard<std::mutex> lock(ctx->mu);
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
    { int wrc = ws_acquire(ctx, st); if (wrc) return wrc; }
    if (curve == 0) k_combine_batch<0><<<(uint32_t)m, 32, 0, st>>>((const xyzz_t *)d_partials, (uint32_t)k, (uint32_t)m, ctx->d_out_raw);
    else k_combine_batch<1><<<(uint32_t)m, 32, 0, st>>>((const xyzz_t *)d_partials, (uint32_t)k, (uint32_t)m, ctx->d_out_raw);
    ctx->out_curve = curve;
    ctx->launches++;
    return fetch_points(ctx, curve, ctx->d_out_raw, m, out_xy, out_inf, st);
}

// Half tables of h(X)'s coefficients for IpaScalars (msm.cuh), built on `st` into ctx->ipa_tabs: worth it once the MSM has
// more coefficients than the tables have entries.  *lo / *hi stay NULL otherwise (the per-bit loop is used).
static int ipa_half_tables(accmsm_ctx *ctx, int sfield, const uint8_t *d_challenges, int k, size_t n, cudaStream_t st,
                           const uint8_t **lo, const uint8_t **hi) {
    *lo = *hi = nullptr;
    if (k < 8 || k > 30 || ctx->no_ipa_tabs) return ACCMSM_OK;
    const uint32_t kl = (uint32_t)k / 2u, entries = (1u << kl) + (1u << ((uint32_t)k - kl));
    if (n < 4 * (size_t)entries) return ACCMSM_OK;
    // the tables are workspace: an earlier call left in flight on another stream may still be reading them
    { int wrc = ws_acquire(ctx, st); if (wrc) return wrc; }
    CU(ctx, ctx->ipa_tabs.ensure((size_t)entries * 32));
    if (sfield == 0) k_ipa_half_tables<0><<<(entries + 255) / 256, 256, 0, st>>>(d_challenges, k, ctx->ipa_tabs.p);
    else k_ipa_half_tables<1><<<(entries + 255) / 256, 256, 0, st>>>(d_challenges, k, ctx->ipa_tabs.p);
    ctx->launches++;
    *lo = ctx->ipa_tabs.p;
    *hi = ctx->ipa_tabs.p + ((size_t)1 << kl) * 32;
    return ACCMSM_OK;
}

static int ipa_run(accmsm_ctx *ctx, const Bases &B, const uint64_t *challenges_mont, int k, size_t coeff_offset, size_t n,
                   xyzz_t *d_partial, bool normalise, cudaStream_t st) {
    CU(ctx, ctx->misc.ensure(64 * 32));
    { int wrc = ws_acquire(ctx, st); if (wrc) return wrc; }
    if (k) { int urc = upload_small(ctx, ctx->misc.p, challenges_mont, (size_t)k * 32, st); if (urc) return urc; }
    const uint8_t *lo = nullptr, *hi = nullptr;
    { int trc = ipa_half_tables(ctx, B.curve == 0 ? 1 : 0, ctx->misc.p, k, n, st, &lo, &hi); if (trc) return trc; }
    if (B.curve == 0) { IpaScalars<1> src{ctx->misc.p, k, (uint32_t)coeff_offset, lo, hi}; return run_msm<0>(ctx, B, MsmJobs(0), n, src, nullptr, 0, d_partial, normalise, st); }
    IpaScalars<0> src{ctx->misc.p, k, (uint32_t)coeff_offset, lo, hi};
    return run_msm<1>(ctx, B, MsmJobs(0), n, src, nullptr, 0, d_partial, normalise, st);
}

int accmsm_ipa_final_key(accmsm_ctx *ctx, uint64_t handle, const uint64_t *challenges_mont, int k, uint64_t out_xy[8],
                         uint8_t *out_inf) {
    if (!ctx || !out_xy || !out_inf || (k && !challenges_mont) || k < 0 || k > 30) return fail_arg(ctx, "ipa_final_key: bad argument");
    if (is_group(ctx)) return group_ipa_final_key(ctx, handle, challenges_mont, k, out_xy, out_inf);
    std::lock_guard<std::mutex> lock(ctx->mu);
    const Bases *B = find_bases(ctx, handle);
    if (!B) return ACCMSM_E_HANDLE;
    size_t n = size_t(1) << k;
    if (n > B->n) return fail_arg(ctx, "ipa_final_key: key shorter than 2^k");
    CU(ctx, cudaSetDevice(ctx->device));
    clear_marks(ctx);
    mark(ctx, ST_H2D, ctx->stream);
    int rc = ipa_run(ctx, *B, challenges_mont, k, 0, n, nullptr, true, ctx->stream);
    if (rc) return rc;
    return fetch_affine(ctx, out_xy, out_inf, ctx->stream);
}

int accmsm_ipa_check_final_key(accmsm_ctx *ctx, uint64_t handle, const uint64_t *challenges_mont, int k,
                               const uint64_t expected_xy[8], uint8_t expected_inf, int *accept, uint64_t out_xy[8],
                               uint8_t *out_inf) {
    if (!accept || !expected_xy) return fail_arg(ctx, "ipa_check_final_key: bad argument");
    uint64_t xy[8]; uint8_t inf = 0;
    int rc = accmsm_ipa_final_key(ctx, handle, challenges_mont, k, xy, &inf);
    if (rc) return rc;
    // affine equality exactly as GroupAffine's PartialEq: both identity, or same (x, y)
    *accept = (inf || expected_inf) ? (inf != 0) == (expected_inf != 0) : memcmp(xy, expected_xy, 64) == 0;
    if (out_xy) memcpy(out_xy, xy, 64);
    if (out_inf) *out_inf = inf;
    return ACCMSM_OK;
}

int accmsm_ipa_final_key_partial_dev(accmsm_ctx *ctx, uint64_t handle, const uint64_t *challenges_mont, int k,
                                     size_t coeff_offset, size_t n, void *d_out_partial, void *stream) {
    if (!ctx || !d_out_partial || (k && !challenges_mont) || k < 0 || k > 30) return fail_arg(ctx, "ipa_final_key_partial_dev: bad argument");
    GROUP_NO_DEV(ctx, "ipa_final_key_partial_dev");
    std::lock_guard<std::mutex> lock(ctx->mu);
    const Bases *B = find_bases(ctx, handle);
    if (!B) return ACCMSM_E_HANDLE;
    if (n == 0 || n > B->n || coeff_offset + n > (size_t(1) << k)) return fail_arg(ctx, "ipa_final_key_partial_dev: bad range");
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
    clear_marks(ctx);
    int rc = ipa_run(ctx, *B, challenges_mont, k, coeff_offset, n, (xyzz_t *)d_out_partial, false, st);
    if (rc) return rc;
    mark(ctx, ST_COUNT, st);
    if (!stream) { CU(ctx, cudaStreamSynchronize(st)); collect_timings(ctx); }
    return ACCMSM_OK;
}

}  // extern "C"

#include "vec_api.inc"
#include "ipa_api.inc"
#include "fused_api.inc"
#include "wire_api.inc"
#include "multi_api.inc"
