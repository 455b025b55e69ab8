// Pippenger variable-base MSM for sm_100a (K2 of SURVEY.md 2b).  Replaces
// ark_ec::msm::VariableBaseMSM::multi_scalar_mul (ark-ec 0.2.0, SURVEY.md App. A.1) as reached from
// PedersenCommitment::commit / IpaPC::cm_commit (reference call sites: src/hp_as/mod.rs:196,197,214,377,
// 910-918; src/r1cs_nark_as/r1cs_nark/mod.rs:216-261,375-407; src/ipa_pc_as/mod.rs:155,454-462,836-845).
//
// Two key layouts: a plain key (per-window bucket sets, Horner over windows at the end) and a key with a window table
// table[w][i] = 2^(c w) P_i built once at registration (k_precompute): all windows then share ONE bucket set, so there
// is one bucket reduction and no window doublings.  Up to MAX_JOBS MSMs of equal length share one pass ("jobs").
//
// Pipeline (all on one stream, no host round trips):
//   k_digits      scalar source (HBM scalars, h(X) coefficients or IPA round scalars generated in registers) ->
//                 (optional from-Montgomery) -> signed radix-2^c digits, histogram of bucket keys (atomics
//                 aggregated per warp with match_any)
//   k_scan*       exclusive prefix sum of the histogram -> bucket offsets + scatter cursors (tiled beyond 32 K keys)
//   k_scatter     counting-sort scatter of (table index | sign) into bucket order
//   k_accumulate  perfectly balanced segmented accumulation: every thread sums an equal-length slice of
//                 the sorted entry list with XYZZ mixed additions; runs that straddle thread / CTA
//                 boundaries are merged by a segmented scan in shared memory (hot buckets are
//                 tree-reduced, never serialised: constant scalar vectors cost the same as random ones)
//   k_fixup       merges the two boundary partials of every CTA
//   k_accumulate_warp_coop   short MSMs instead: four replica warps per bucket (coop.cuh), no merging
//   k_sums /      bucket reduction sum_b b*B_b organised for depth: row / column sums of the bucket index (twice),
//   k_leaf_*_coop then four 32-item weighted sums; latency-bound levels run as cooperative groups (coop.cuh)
//   k_finish      (plain key: Horner combine of the window sums, c doublings per window), extra partials,
//                 normalisation with a binary-GCD inversion
#pragma once
#include <cuda_runtime.h>
#include "ec.cuh"

namespace accmsm {

constexpr uint32_t NONE_ID = 0xffffffffu;
constexpr int ACC_THREADS = 256;       // threads per accumulate CTA
constexpr int FIX_THREADS = 512;       // k_fixup: one CTA, FIX_PER_T slots per thread (<= 1536 slots fit in 227 KB)
constexpr int FIX_PER_T = 3;
static_assert((size_t)FIX_THREADS * FIX_PER_T * (sizeof(uint32_t) + 128) <= 227 * 1024, "k_fixup slots must fit in one CTA's shared memory");
constexpr int MAX_WINDOWS = 64;
constexpr int MAX_JOBS = 8;            // MSMs that share one pass of the pipeline (same key, same length)

struct MsmShape {
    uint32_t n;        // number of (base, scalar) pairs
    uint32_t c;        // window bits
    uint32_t nwin;     // number of signed windows = ceil(256 / c)
    uint32_t nb;       // buckets per window = 2^(c-1)
    uint32_t nkeys;    // bucket sets * nb
    // Two sort layouts.  Plain key: every window has its own bucket set (hist_stride = nb) and an entry is the
    // point index.  Precomputed key (table[w][i] = 2^(c w) P_i): all windows share ONE bucket set
    // (hist_stride = 0) and an entry indexes the table: w * ent_stride + ent_offset + i.
    uint32_t hist_stride;
    uint32_t ent_stride;
    // Batch: njobs MSMs of the same length over (possibly different) ranges of one key go through the
    // pipeline together -- hp_as::decide commits a, b, a o b (src/hp_as/mod.rs:910-918), the NARK commits
    // z_A, z_B, z_C (src/r1cs_nark_as/r1cs_nark/mod.rs:216-218), an IPA round its (l, r) pair.  Job j owns
    // bucket sets [j * sets_per_job, (j + 1) * sets_per_job) and reads bases job_off[j] + i.
    uint32_t njobs;
    uint32_t sets_per_job;   // nwin (plain key) or 1 (window table)
    uint32_t job_off[MAX_JOBS];
    // Optional hiding term: when tail_base != NONE_ID the last of the n pairs of every job is
    // (base tail_base, randomizer) -- PedersenCommitment::commit(ck, elems, Some(r)) = MSM + r * hiding_generator
    // in the same pass (SURVEY.md App. A.2).
    uint32_t tail_base;
    // Optional index map (IPA opening rounds over the unfolded key): pair i of a job addresses base
    // job_off + ((i >> map_log_h) << (map_log_h + 1)) + (i & (2^map_log_h - 1)), i.e. the lower (job_off = 0) or upper
    // (job_off = 2^map_log_h) half of every block of 2^(map_log_h + 1) consecutive bases.  NONE_ID = identity map.
    uint32_t map_log_h;
};
ACC_D uint32_t msm_base_index(const MsmShape &sh, uint32_t job, uint32_t i) {
    if (sh.tail_base != NONE_ID && i == sh.n - 1) return sh.tail_base;
    if (sh.map_log_h != NONE_ID) return sh.job_off[job] + ((i >> sh.map_log_h) << (sh.map_log_h + 1)) + (i & ((1u << sh.map_log_h) - 1u));
    return sh.job_off[job] + i;
}

// ------------------------------------------------------------------------------------------------
// vectorised loads / stores (128-bit, coalesced when consecutive threads touch consecutive records)
// ------------------------------------------------------------------------------------------------
ACC_D fe_t load_fe(const void *p) {
    const uint4 *q = reinterpret_cast<const uint4 *>(p);
    uint4 a = q[0], b = q[1];
    fe_t r;
    r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w; r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
    return r;
}
ACC_D fe_t load_fe_nc(const void *p) {   // read-only path for data that is streamed once
    const uint4 *q = reinterpret_cast<const uint4 *>(p);
    uint4 a = __ldg(q), b = __ldg(q + 1);
    fe_t r;
    r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w; r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
    return r;
}
ACC_D void store_fe(void *p, const fe_t &r) {
    uint4 *q = reinterpret_cast<uint4 *>(p);
    q[0] = make_uint4(r.l[0], r.l[1], r.l[2], r.l[3]);
    q[1] = make_uint4(r.l[4], r.l[5], r.l[6], r.l[7]);
}
ACC_D affine_t load_affine(const affine_t *p) {
    affine_t r;
    r.x = load_fe_nc(&p->x); r.y = load_fe_nc(&p->y);
    return r;
}
ACC_D xyzz_t load_xyzz(const xyzz_t *p) {
    xyzz_t r;
    r.x = load_fe(&p->x); r.y = load_fe(&p->y); r.zz = load_fe(&p->zz); r.zzz = load_fe(&p->zzz);
    return r;
}
ACC_D void store_xyzz(xyzz_t *p, const xyzz_t &r) {
    store_fe(&p->x, r.x); store_fe(&p->y, r.y); store_fe(&p->zz, r.zz); store_fe(&p->zzz, r.zzz);
}

// ------------------------------------------------------------------------------------------------
// scalar sources for k_digits
// ------------------------------------------------------------------------------------------------
// Scalars resident in HBM: n x 32 B, either the Fp256 Montgomery image (what PedersenCommitment::commit
// receives; into_repr() is done here) or canonical BigInteger256 (what VariableBaseMSM receives).
template <int SFIELD> struct MemScalars {
    const uint8_t *ptr[MAX_JOBS];
    int montgomery;
    ACC_D fe_t canonical(uint32_t job, uint32_t i) const {
        fe_t s = load_fe_nc(ptr[job] + (size_t)i * 32);
        if (montgomery) s = Fp<SFIELD>::from_mont(s);
        return s;
    }
};
// K3: coefficients of the IPA succinct-check polynomial h(X) = prod_{i=1..k} (1 + xi_i X^(2^(k-i)))
// generated on the fly (never materialised in HBM): coeff[j] = prod_{i : bit (k-i) of j set} xi_i
// (ark-poly-commit SuccinctCheckPolynomial::compute_coeffs, SURVEY.md App. A.3; reference call sites
// src/ipa_pc_as/mod.rs:400 and :836 via IpaPC::check).  `offset` lets a GPU own a slice of the key.
template <int SFIELD> struct IpaScalars {
    const uint8_t *challenges;  // k x 32 B Montgomery, xi_1 first
    int k;
    uint32_t offset;
    // Optional half tables (k_ipa_half_tables): lo[t] = coefficient of the index whose low kl = k / 2 bits are t, hi[t] the same
    // for the high k - kl bits, so coeff[j] = hi[j >> kl] * lo[j & (2^kl - 1)] -- ONE product per coefficient instead of one
    // per set bit (and, across a warp, one per bit position: k warp-level products).  The digit kernels call canonical() in
    // both sort passes: at k = 20 that loop was 0.2 ms of a 3.3 ms decide tail.
    const uint8_t *lo_tab = nullptr, *hi_tab = nullptr;
    ACC_D fe_t coeff_mont(uint32_t i) const {
        uint32_t j = i + offset;
        if (lo_tab) {
            const uint32_t kl = (uint32_t)k / 2u;
            return Fp<SFIELD>::mul(load_fe(hi_tab + (size_t)(j >> kl) * 32), load_fe(lo_tab + (size_t)(j & ((1u << kl) - 1u)) * 32));
        }
        fe_t acc = Fp<SFIELD>::one();
        for (int b = 0; b < k; b++) {          // bit b of j <-> challenge index k - b  (1-based)
            if ((j >> b) & 1u) acc = Fp<SFIELD>::mul(acc, load_fe(challenges + (size_t)(k - 1 - b) * 32));
        }
        return acc;
    }
    ACC_D fe_t canonical(uint32_t, uint32_t i) const { return Fp<SFIELD>::from_mont(coeff_mont(i)); }
};
// tab[0 .. 2^kl) = lo table, tab[2^kl .. 2^kl + 2^(k - kl)) = hi table (Montgomery), kl = k / 2
template <int SFIELD>
__global__ void __launch_bounds__(256) k_ipa_half_tables(const uint8_t *__restrict__ challenges, int k, uint8_t *__restrict__ tab) {
    const uint32_t kl = (uint32_t)k / 2u, kh = (uint32_t)k - kl, nlo = 1u << kl, nhi = 1u << kh;
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nlo + nhi) return;
    const bool is_hi = t >= nlo;
    const uint32_t v = is_hi ? t - nlo : t, b0 = is_hi ? kl : 0u, nb = is_hi ? kh : kl;
    fe_t acc = Fp<SFIELD>::one();
    for (uint32_t b = 0; b < nb; b++) {
        if ((v >> b) & 1u) acc = Fp<SFIELD>::mul(acc, load_fe(challenges + (size_t)(k - 1 - (int)(b0 + b)) * 32));
    }
    store_fe(tab + (size_t)t * 32, acc);
}

// Scalars of one IPA opening round expressed over the UNFOLDED commitment key (SURVEY.md App. A.2).  After j folds the
// key is G^(j)[i] = sum_u C_j(u) G[u n_j + i] with C_j(u) = prod_{m <= j : bit (j - m) of u} xi_m (the h(X) coefficient
// of the top j index bits), so with h = n_j / 2
//     l = <a_R, G^(j)_L> = sum_{u, i' < h} a[h + i'] C_j(u) G[u n_j + i']          (job 0)
//     r = <a_L, G^(j)_R> = sum_{u, i' < h} a[i']     C_j(u) G[u n_j + h + i']      (job 1)
// are MSMs over the registered key (window table, no Horner over windows) and the key is never folded.
template <int SFIELD> struct IpaRoundScalars {
    const uint8_t *a;           // current coefficient vector, 2h Montgomery elements
    const uint8_t *challenges;  // xi_1 .. xi_j, Montgomery
    int j;
    uint32_t log_h;
    const uint8_t *tail;        // nullable: 2 canonical scalars, the last pair (hiding generator) of job 0 / job 1
    uint32_t n_pairs;
    ACC_D fe_t canonical(uint32_t job, uint32_t i) const {
        using F = Fp<SFIELD>;
        if (tail && i == n_pairs - 1) return load_fe(tail + (size_t)job * 32);
        const uint32_t h = 1u << log_h, ip = i & (h - 1u), u = i >> log_h;
        fe_t acc = load_fe(a + (size_t)((job == 0 ? h : 0u) + ip) * 32);
        for (int m = 1; m <= j; m++) {
            if ((u >> (j - m)) & 1u) acc = F::mul(acc, load_fe(challenges + (size_t)(m - 1) * 32));
        }
        return F::from_mont(acc);
    }
};

// The first-version sort kernels below double as the fallback of the shared-memory radix sort (sort.cuh) for skewed
// scalar distributions: with a gate they run only when the largest partition the radix sort counted exceeds `thr`
// (decided on the device, no host round trip); max_part == nullptr: always run.
struct SortGate {
    const uint32_t *max_part;
    uint32_t thr;
};
ACC_D bool gate_closed(const SortGate &g) { return g.max_part && *g.max_part <= g.thr; }

// bits [pos, pos + c) of a 256-bit little-endian integer, c <= 24
ACC_D uint32_t extract_bits(const uint32_t *s, uint32_t pos, uint32_t c) {
    uint32_t limb = pos >> 5, off = pos & 31;
    uint32_t lo = limb < 8 ? s[limb] : 0u;
    uint32_t hi = limb + 1 < 8 ? s[limb + 1] : 0u;
    uint64_t v = ((uint64_t)hi << 32) | lo;
    return (uint32_t)(v >> off) & ((1u << c) - 1u);
}

// ------------------------------------------------------------------------------------------------
// k_digits: one thread per scalar.  digits[w * n + i] = 0 for a zero digit, else |d| | (d < 0) << 31.
// ------------------------------------------------------------------------------------------------
template <class Src>
__global__ void __launch_bounds__(256) k_digits(Src src, MsmShape sh, const uint8_t *__restrict__ base_is_identity,
                                                 uint32_t *__restrict__ digits, uint32_t *__restrict__ hist,
                                                 uint32_t i0, uint32_t i1, SortGate gate) {
    if (gate_closed(gate)) return;
    // scalars [i0, i1) of every job; grid-stride, so a gated launch can use a small grid that costs nothing when it stands down
    const uint32_t job = blockIdx.y;
    digits += (size_t)job * sh.nwin * sh.n;
    hist += (size_t)job * sh.sets_per_job * sh.nb;
    for (uint32_t i = i0 + blockIdx.x * blockDim.x + threadIdx.x; i < i1; i += gridDim.x * blockDim.x) {
    fe_t s = src.canonical(job, i);
    if (base_is_identity && base_is_identity[msm_base_index(sh, job, i)]) s = Fp<0>::zero();   // identity bases contribute nothing
    const uint32_t half = 1u << (sh.c - 1);
    const unsigned am = __activemask();            // lanes with i < n (the others have returned)
    const uint32_t lane = threadIdx.x & 31;
    uint32_t carry = 0;
    for (uint32_t w = 0; w < sh.nwin; w++) {
        uint32_t raw = extract_bits(s.l, w * sh.c, sh.c) + carry;
        uint32_t enc = 0;
        if (raw > half) {             // negative digit raw - 2^c, borrow one from the next window
            uint32_t mag = (1u << sh.c) - raw;
            carry = 1;
            enc = mag ? (mag | 0x80000000u) : 0u;   // raw == 2^c -> digit 0 with carry
        } else {
            carry = 0;
            enc = raw;
        }
        digits[(size_t)w * sh.n + i] = enc;
        uint32_t mag = enc & 0x7fffffffu;
        // Histogram update, aggregated per warp: lanes that land in the same bucket (constant scalar vectors -- the
        // reference's own fixtures, src/hp_as/mod.rs:991 -- or the short top window, where all n digits fall into a
        // handful of buckets) send ONE atomic with their count instead of serialising on one L2 address.
        const uint32_t key = mag ? w * sh.hist_stride + mag - 1 : NONE_ID;
        const unsigned peers = __match_any_sync(am, key);      // lanes of this warp that hit the same bucket
        if (mag && lane == (uint32_t)(__ffs(peers) - 1)) atomicAdd(&hist[key], (uint32_t)__popc(peers));
    }
    }
}

// ------------------------------------------------------------------------------------------------
// Exclusive scan of hist[0..nkeys) into offsets[0..nkeys] and cursor[0..nkeys).  Tiles of 4096 keys
// (1024 threads x one 128-bit load).  Up to SCAN_ONE_CTA_TILES tiles a single CTA walks them serially
// (k_scan); beyond that: k_scan_tile_sums -> k_scan over the tile sums -> k_scan_tiles.
// ------------------------------------------------------------------------------------------------
constexpr uint32_t SCAN_TILE = 4096;
constexpr uint32_t SCAN_ONE_CTA_TILES = 8;

// exclusive scan of one tile starting at `carry`; returns the tile total (valid in every thread)
ACC_D uint32_t scan_tile(const uint32_t *__restrict__ hist, uint32_t nkeys, uint32_t base, uint32_t carry,
                         uint32_t *__restrict__ offsets, uint32_t *__restrict__ cursor, uint32_t *warp_sums,
                         uint32_t *total_s) {
    const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    uint32_t k0 = base + tid * 4;
    uint32_t v[4];
    if (k0 + 3 < nkeys) {
        uint4 q = *reinterpret_cast<const uint4 *>(hist + k0);
        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
    } else {
#pragma unroll
        for (int j = 0; j < 4; j++) v[j] = (k0 + j < nkeys) ? hist[k0 + j] : 0u;
    }
    uint32_t tsum = v[0] + v[1] + v[2] + v[3];
    uint32_t incl = tsum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
    }
    if (lane == 31) warp_sums[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        uint32_t ws = warp_sums[lane];
        uint32_t wi = ws;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t o = __shfl_up_sync(0xffffffffu, wi, d);
            if (lane >= d) wi += o;
        }
        warp_sums[lane] = wi - ws;  // exclusive prefix of warp sums
        if (lane == 31) *total_s = wi;
    }
    __syncthreads();
    uint32_t excl = carry + warp_sums[wid] + incl - tsum;
    if (offsets) {
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (k0 + j < nkeys) { offsets[k0 + j] = excl; if (cursor) cursor[k0 + j] = excl; }
            excl += v[j];
        }
    }
    uint32_t total = *total_s;
    __syncthreads();
    return total;
}

__global__ void __launch_bounds__(1024) k_scan(const uint32_t *__restrict__ hist, uint32_t nkeys,
                                                uint32_t *__restrict__ offsets, uint32_t *__restrict__ cursor, SortGate gate) {
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t total_s;
    if (gate_closed(gate)) return;
    uint32_t carry = 0;
    for (uint32_t base = 0; base < nkeys; base += SCAN_TILE)
        carry += scan_tile(hist, nkeys, base, carry, offsets, cursor, warp_sums, &total_s);
    if (threadIdx.x == 0) offsets[nkeys] = carry;
}
__global__ void __launch_bounds__(1024) k_scan_tile_sums(const uint32_t *__restrict__ hist, uint32_t nkeys,
                                                          uint32_t *__restrict__ tile_sums, SortGate gate) {
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t total_s;
    if (gate_closed(gate)) return;
    uint32_t total = scan_tile(hist, nkeys, blockIdx.x * SCAN_TILE, 0, nullptr, nullptr, warp_sums, &total_s);
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}
// tile_offs = exclusive scan of the tile sums (ntiles + 1 entries, the last one is the grand total)
__global__ void __launch_bounds__(1024) k_scan_tiles(const uint32_t *__restrict__ hist, uint32_t nkeys,
                                                      const uint32_t *__restrict__ tile_offs, uint32_t *__restrict__ offsets,
                                                      uint32_t *__restrict__ cursor, SortGate gate) {
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t total_s;
    if (gate_closed(gate)) return;
    scan_tile(hist, nkeys, blockIdx.x * SCAN_TILE, tile_offs[blockIdx.x], offsets, cursor, warp_sums, &total_s);
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) offsets[nkeys] = tile_offs[gridDim.x];
}

// ------------------------------------------------------------------------------------------------
// k_scatter: entries[cursor[key]++] = point index | sign
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_scatter(MsmShape sh, const uint32_t *__restrict__ digits,
                                                  uint32_t *__restrict__ cursor, uint32_t *__restrict__ entries, SortGate gate) {
    if (gate_closed(gate)) return;
    const uint32_t job = blockIdx.y;
    digits += (size_t)job * sh.nwin * sh.n;
    cursor += (size_t)job * sh.sets_per_job * sh.nb;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < sh.n; i += gridDim.x * blockDim.x) {
    const uint32_t base_index = msm_base_index(sh, job, i);
    const unsigned am = __activemask();
    const uint32_t lane = threadIdx.x & 31;
    for (uint32_t w = 0; w < sh.nwin; w++) {
        uint32_t enc = digits[(size_t)w * sh.n + i];
        uint32_t mag = enc & 0x7fffffffu;
        const uint32_t key = mag ? w * sh.hist_stride + mag - 1 : NONE_ID;
        const unsigned peers = __match_any_sync(am, key);      // one atomic reserves the range of all lanes in a bucket
        const uint32_t lead = __ffs(peers) - 1;
        uint32_t pos = 0;
        if (mag && lane == lead) pos = atomicAdd(&cursor[key], (uint32_t)__popc(peers));
        pos = __shfl_sync(am, pos, lead) + __popc(peers & ((1u << lane) - 1u));
        if (mag) entries[pos] = (w * sh.ent_stride + base_index) | (enc & 0x80000000u);
    }
    }
}

ACC_D xyzz_t shfl_down_xyzz(const xyzz_t &p, int d) {
    xyzz_t r;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        r.x.l[i] = __shfl_down_sync(0xffffffffu, p.x.l[i], d);
        r.y.l[i] = __shfl_down_sync(0xffffffffu, p.y.l[i], d);
        r.zz.l[i] = __shfl_down_sync(0xffffffffu, p.zz.l[i], d);
        r.zzz.l[i] = __shfl_down_sync(0xffffffffu, p.zzz.l[i], d);
    }
    return r;
}

}  // namespace accmsm
#include "coop.cuh"   // needs load_fe / store_fe above
namespace accmsm {

// ------------------------------------------------------------------------------------------------
// segmented inclusive scan of (id, point) slots in shared memory; slots with equal ids are contiguous.
// After it, the last slot of every id-group holds the group's sum.  NS <= 2 * blockDim.x * SLOTS_PER_T.
// ------------------------------------------------------------------------------------------------
template <int CURVE, int PER_T, template <int> class FT = Fp>
ACC_D void seg_scan(xyzz_t *pt, const uint32_t *id, uint32_t ns) {
    using Cv = Curve<CURVE, FT>;
    // Hillis-Steele in place.  A step reads slot i - d and writes slot i; the slots are swept in PER_T
    // phases from the top stripe down, so a phase only ever reads slots that this step has not written
    // yet (writes of a phase land in its own stripe, reads come from it or from lower stripes) and one
    // point per thread is live at a time.
    for (uint32_t d = 1; d < ns; d <<= 1) {
        // equal ids are contiguous: if no slot has a partner at distance d, none has one further away
        bool any = false;
#pragma unroll 1
        for (int r = 0; r < PER_T; r++) {
            uint32_t i = threadIdx.x + r * blockDim.x;
            any |= i < ns && i >= d && id[i] != NONE_ID && id[i] == id[i - d];
        }
        if (!__syncthreads_or(any)) break;
#pragma unroll 1
        for (int r = PER_T - 1; r >= 0; r--) {
            uint32_t i = threadIdx.x + r * blockDim.x;
            bool doit = i < ns && i >= d && id[i] != NONE_ID && id[i] == id[i - d];
            xyzz_t mine;
            if (doit) { mine = pt[i]; xyzz_t other = pt[i - d]; Cv::add(mine, other); }
            __syncthreads();
            if (doit) pt[i] = mine;
            __syncthreads();
        }
    }
}

// The identity cannot be an affine record; it is stored as x = 2^256 - 1 (not a canonical field element), y = 0.
ACC_D bool affine_is_identity_marker(const fe_t &x) {
    uint32_t d = 0xffffffffu;
#pragma unroll
    for (int i = 0; i < 8; i++) d &= x.l[i];
    return d == 0xffffffffu;
}
ACC_D affine_t affine_identity_marker() {
    affine_t r;
#pragma unroll
    for (int i = 0; i < 8; i++) { r.x.l[i] = 0xffffffffu; r.y.l[i] = 0u; }
    return r;
}
// ------------------------------------------------------------------------------------------------
// k_accumulate
// ------------------------------------------------------------------------------------------------
template <int CURVE, bool INTO>
__global__ void __launch_bounds__(ACC_THREADS, 2)
k_accumulate(const uint32_t *__restrict__ offsets, uint32_t nkeys, const uint32_t *__restrict__ entries,
             const affine_t *__restrict__ bases, xyzz_t *__restrict__ buckets,
             uint32_t *__restrict__ cta_ids, xyzz_t *__restrict__ cta_parts) {
    constexpr bool into = INTO;
    // INTO: the buckets already hold the sums of earlier point segments of the same MSM (zero-initialised = identity;
    // msm_host_scalars pipelines the upload of one segment behind the accumulation of the previous one): the run that
    // STARTS a bucket continues from the stored value, so merging segments costs one 128-byte load per bucket, no additions
    using Cv = Curve<CURVE>;
    extern __shared__ uint4 smem_raw[];
    xyzz_t *slot_pt = reinterpret_cast<xyzz_t *>(smem_raw);
    uint32_t *slot_id = reinterpret_cast<uint32_t *>(slot_pt + 2 * ACC_THREADS);

    const uint32_t M = offsets[nkeys];
    const uint32_t T = gridDim.x * blockDim.x;
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t L = (M + T - 1) / T;
    const uint64_t s64 = (uint64_t)t * L;
    const uint32_t s = s64 < M ? (uint32_t)s64 : M;
    const uint32_t e = (s64 + L < M) ? (uint32_t)(s64 + L) : M;

    // slot 2t = the first run of the slice (may continue the previous thread's last run), slot 2t + 1 = the
    // last run (may continue into the next thread's slice); written straight to shared memory so that only
    // one accumulator lives in registers
    uint32_t head_id = NONE_ID, tail_id = NONE_ID;
    slot_pt[2 * threadIdx.x + 1] = Cv::identity();
    if (s >= e) slot_pt[2 * threadIdx.x] = Cv::identity();

    if (s < e) {
        // bucket containing entry s: first k with offsets[k + 1] > s
        uint32_t lo = 0, hi = nkeys - 1;
        while (lo < hi) {
            uint32_t mid = (lo + hi) >> 1;
            if (offsets[mid + 1] > s) hi = mid; else lo = mid + 1;
        }
        // One flat loop over the slice: every lane of a warp executes exactly L iterations and spends them
        // in the mixed add; a bucket boundary only costs the (cheap, divergent) flush of the finished run.
        uint32_t k = lo, bend = offsets[k + 1];
        bool first_run = true;
        xyzz_t acc = (into && s == offsets[k]) ? load_xyzz(buckets + k) : Cv::identity();
        // entries == nullptr: "direct" list (after batch-affine rounds, below): entry p IS point p of `bases`, no sign,
        // and x = 2^256 - 1 marks the identity
        uint32_t ent = entries ? entries[s] : s;
        affine_t pt = load_affine(bases + (ent & 0x7fffffffu));
#pragma unroll 1
        for (uint32_t p = s; p < e; p++) {
            if (p == bend) {                       // the run of bucket k ended with entry p - 1
                if (first_run) { slot_pt[2 * threadIdx.x] = acc; head_id = k; first_run = false; }
                else store_xyzz(buckets + k, acc);  // a run strictly inside this slice is complete
                acc = Cv::identity();
                k++; bend = offsets[k + 1];
                if (bend == p) {                   // empty buckets ahead: binary search for the bucket holding entry p
                    uint32_t blo = k + 1, bhi = nkeys - 1;   // (a linear walk over 2^19 empty buckets is what makes
                    while (blo < bhi) {                      //  constant scalar vectors slow otherwise)
                        uint32_t mid = (blo + bhi) >> 1;
                        if (offsets[mid + 1] > p) bhi = mid; else blo = mid + 1;
                    }
                    k = blo; bend = offsets[k + 1];
                }
                if (into) acc = load_xyzz(buckets + k);      // entry p is the first of bucket k
            }
            const uint32_t cur_sign = ent >> 31;
            affine_t cur = pt;
            if (p + 1 < e) {                       // software prefetch of the next point (a gather from HBM / L2)
                ent = entries ? entries[p + 1] : p + 1;
                pt = load_affine(bases + (ent & 0x7fffffffu));
            }
            if (cur_sign) cur.y = Cv::F::neg(cur.y);
            if (entries || !affine_is_identity_marker(cur.x)) Cv::madd(acc, cur);
        }
        if (first_run) { slot_pt[2 * threadIdx.x] = acc; head_id = k; tail_id = k; }   // equal ids stay contiguous
        else { slot_pt[2 * threadIdx.x + 1] = acc; tail_id = k; }
    }
    slot_id[2 * threadIdx.x] = head_id;
    slot_id[2 * threadIdx.x + 1] = tail_id;
    __syncthreads();
    const uint32_t ns = 2 * ACC_THREADS;
    seg_scan<CURVE, 2>(slot_pt, slot_id, ns);

    // ids of the first slot and of the last slot that holds work
    const uint32_t first_id = slot_id[0];
    __shared__ uint32_t last_id_s;
    if (threadIdx.x == 0) last_id_s = NONE_ID;
    __syncthreads();
    for (int r = 0; r < 2; r++) {
        uint32_t i = threadIdx.x + r * blockDim.x;
        bool valid = slot_id[i] != NONE_ID;
        bool next_valid = (i + 1 < ns) && slot_id[i + 1] != NONE_ID;
        if (valid && !next_valid) last_id_s = slot_id[i];
    }
    __syncthreads();
    const uint32_t last_id = last_id_s;
    if (threadIdx.x == 0) {
        cta_ids[2 * blockIdx.x] = first_id;
        cta_ids[2 * blockIdx.x + 1] = last_id;
        if (first_id == last_id) store_xyzz(cta_parts + 2 * blockIdx.x + 1, Cv::identity());
    }
    for (int r = 0; r < 2; r++) {
        uint32_t i = threadIdx.x + r * blockDim.x;
        uint32_t id = slot_id[i];
        if (id == NONE_ID) continue;
        bool group_end = (i + 1 == ns) || slot_id[i + 1] != id;
        if (!group_end) continue;
        if (id == first_id) store_xyzz(cta_parts + 2 * blockIdx.x, slot_pt[i]);
        else if (id == last_id) store_xyzz(cta_parts + 2 * blockIdx.x + 1, slot_pt[i]);
        else store_xyzz(buckets + id, slot_pt[i]);
    }
}

// k_accumulate_warp_coop: one GROUP of four replica warps (coop.cuh, included further down) per bucket, for short MSMs
// (a few thousand buckets).  Lane j folds entries j, j + 32, ... of its bucket, then the 32 partials are summed by a
// shuffle tree; every addition is a cooperative one.  The balanced kernel above needs a segmented scan (4-5 dependent
// point additions) plus k_fixup to merge slices; here nothing is merged across warps, which wins while the whole problem
// is bound by latency, not throughput (0.106 vs 0.221 ms at 2^12 points).
template <int CURVE>
__global__ void __launch_bounds__(128) k_accumulate_warp_coop(const uint32_t *__restrict__ offsets, uint32_t nkeys,
                                                               const uint32_t *__restrict__ entries,
                                                               const affine_t *__restrict__ bases, xyzz_t *__restrict__ buckets);

// ------------------------------------------------------------------------------------------------
// Batch-affine pre-reduction (SURVEY.md App. D.5(ii)).  One round halves the points of every bucket: neighbours
// (2j, 2j + 1) of the bucket's list are added in AFFINE coordinates,
//     lambda = (y1 - y0) / (x1 - x0),  x3 = lambda^2 - x0 - x1,  y3 = lambda (x0 - x3) - y0        (5M + 1S + 1 inversion)
// and ALL divisions of a round share ONE inversion (Montgomery's trick across the whole grid): k_pair_fwd computes the
// denominators and per-thread prefix products and scans the thread totals over the CTA, k_pair_mid scans the CTA totals
// and inverts the grid total once (binary GCD), k_pair_bwd back-substitutes and forms the sums.  That is ~6 products
// per addition instead of the 10 of the XYZZ mixed add.  After a few rounds the shortened lists go through
// k_accumulate in "direct" mode.  Exceptional pairs are peeled: x0 == x1 with y0 == y1 is a doubling
// (lambda = 3 x0^2 / 2 y0), with y0 == -y1 the sum is the identity (stored as a marker, skipped downstream); an odd
// last element or an identity partner passes through.  Results are the same affine points any other addition law gives.
// ------------------------------------------------------------------------------------------------
constexpr int PAIR_THREADS = 256;
constexpr int PAIR_B = 32;              // output slots per thread
constexpr int PAIR_MID_THREADS = 1024;

__global__ void __launch_bounds__(256) k_pair_counts(const uint32_t *__restrict__ offsets, uint32_t nkeys,
                                                      uint32_t *__restrict__ counts) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < nkeys) counts[k] = (offsets[k + 1] - offsets[k] + 1u) >> 1;
}

// x / y of input i of a pair round: the FIRST round reads the window table through the sorted entry list (index | sign)
template <bool FIRST>
ACC_D fe_t pair_load_x(const uint32_t *__restrict__ entries, const affine_t *__restrict__ pts, uint32_t i) {
    return load_fe_nc(&pts[FIRST ? (entries[i] & 0x7fffffffu) : i].x);
}
template <int CURVE, bool FIRST>
ACC_D fe_t pair_load_y(const uint32_t *__restrict__ entries, const affine_t *__restrict__ pts, uint32_t i) {
    using F = typename Curve<CURVE>::F;
    if (FIRST) {
        uint32_t ent = entries[i];
        fe_t y = load_fe_nc(&pts[ent & 0x7fffffffu].y);
        return (ent >> 31) ? F::neg(y) : y;
    }
    return load_fe_nc(&pts[i].y);
}
enum : uint8_t { PAIR_PASS0 = 0, PAIR_PASS1 = 1, PAIR_ADD = 2, PAIR_DBL = 3, PAIR_IDENT = 4 };

// walks the output slots [s0, s1) of one thread forwards: bucket k of slot s without a linear walk over empty buckets
struct PairWalk {
    uint32_t k, bend;
    ACC_D void init(const uint32_t *__restrict__ off_out, uint32_t nkeys, uint32_t s) {
        uint32_t lo = 0, hi = nkeys - 1;
        while (lo < hi) {
            uint32_t mid = (lo + hi) >> 1;
            if (off_out[mid + 1] > s) hi = mid; else lo = mid + 1;
        }
        k = lo; bend = off_out[k + 1];
    }
    ACC_D void advance_to(const uint32_t *__restrict__ off_out, uint32_t nkeys, uint32_t s) {
        if (s != bend) return;
        k++; bend = off_out[k + 1];
        if (bend == s) init(off_out, nkeys, s);
    }
};

// forward pass: denominators, per-thread prefix products (to HBM), pair kinds; product scans over the CTA; the thread's
// share of the inverse (everything but the grid-wide inverse) and the CTA total go to HBM
template <int CURVE, bool FIRST>
__global__ void __launch_bounds__(PAIR_THREADS) k_pair_fwd(const uint32_t *__restrict__ off_in, const uint32_t *__restrict__ off_out,
                                                           uint32_t nkeys, const uint32_t *__restrict__ entries,
                                                           const affine_t *__restrict__ pts_in, uint8_t *__restrict__ pref,
                                                           uint8_t *__restrict__ kinds, uint8_t *__restrict__ thread_factor,
                                                           uint8_t *__restrict__ cta_total) {
    using F = typename Curve<CURVE>::F;
    __shared__ fe_t sh_pre[PAIR_THREADS];
    __shared__ fe_t sh_suf[PAIR_THREADS];
    const uint32_t M_out = off_out[nkeys];
    if ((uint64_t)blockIdx.x * PAIR_THREADS * PAIR_B >= M_out) return;      // whole CTA beyond the list (grid is an upper bound)
    const uint32_t t = blockIdx.x * PAIR_THREADS + threadIdx.x;
    const uint64_t s64 = (uint64_t)t * PAIR_B;
    const uint32_t s0 = s64 < M_out ? (uint32_t)s64 : M_out;
    const uint32_t s1 = (s64 + PAIR_B < M_out) ? (uint32_t)(s64 + PAIR_B) : M_out;
    fe_t run = F::one();
    if (s0 < s1) {
        PairWalk w; w.init(off_out, nkeys, s0);
#pragma unroll 1
        for (uint32_t s = s0; s < s1; s++) {
            w.advance_to(off_out, nkeys, s);
            const uint32_t i0 = off_in[w.k] + 2 * (s - off_out[w.k]);
            const bool has_pair = i0 + 1 < off_in[w.k + 1];
            uint8_t kind = PAIR_PASS0;
            fe_t den = F::one();
            if (has_pair) {
                const fe_t x0 = pair_load_x<FIRST>(entries, pts_in, i0), x1 = pair_load_x<FIRST>(entries, pts_in, i0 + 1);
                if (!FIRST && affine_is_identity_marker(x1)) kind = PAIR_PASS0;
                else if (!FIRST && affine_is_identity_marker(x0)) kind = PAIR_PASS1;
                else {
                    den = F::sub(x1, x0);
                    kind = PAIR_ADD;
                    if (F::is_zero(den)) {           // same x: doubling or cancellation
                        const fe_t y0 = pair_load_y<CURVE, FIRST>(entries, pts_in, i0), y1 = pair_load_y<CURVE, FIRST>(entries, pts_in, i0 + 1);
                        if (F::eq(y0, y1) && !F::is_zero(y0)) { den = F::dbl(y0); kind = PAIR_DBL; }
                        else { den = F::one(); kind = PAIR_IDENT; }
                    }
                }
            }
            store_fe(pref + (size_t)s * 32, run);
            kinds[s] = kind;
            run = F::mul(run, den);
        }
    }
    sh_pre[threadIdx.x] = run;
    sh_suf[threadIdx.x] = run;
    __syncthreads();
#pragma unroll 1
    for (int d = 1; d < PAIR_THREADS; d <<= 1) {
        fe_t a, b;
        const bool up = (int)threadIdx.x >= d, dn = (int)threadIdx.x + d < PAIR_THREADS;
        if (up) a = F::mul(sh_pre[threadIdx.x], sh_pre[threadIdx.x - d]);
        if (dn) b = F::mul(sh_suf[threadIdx.x], sh_suf[threadIdx.x + d]);
        __syncthreads();
        if (up) sh_pre[threadIdx.x] = a;
        if (dn) sh_suf[threadIdx.x] = b;
        __syncthreads();
    }
    // 1 / (own total) = 1 / (CTA total) * (product of the other threads' totals)
    fe_t f = F::one();
    if (threadIdx.x > 0) f = sh_pre[threadIdx.x - 1];
    if (threadIdx.x + 1 < PAIR_THREADS) f = F::mul(f, sh_suf[threadIdx.x + 1]);
    store_fe(thread_factor + (size_t)t * 32, f);
    if (threadIdx.x == 0) store_fe(cta_total + (size_t)blockIdx.x * 32, sh_pre[PAIR_THREADS - 1]);
}

// middle pass, one CTA: cta_factor[c] = 1 / (total of CTA c) = 1 / (grid total) * (product of all other CTA totals);
// ONE inversion for the whole round
template <int CURVE>
__global__ void __launch_bounds__(PAIR_MID_THREADS) k_pair_mid(const uint32_t *__restrict__ off_out, uint32_t nkeys,
                                                               const uint8_t *__restrict__ cta_total, uint8_t *__restrict__ cta_factor) {
    using F = typename Curve<CURVE>::F;
    __shared__ fe_t sh[PAIR_MID_THREADS];
    __shared__ fe_t carry_s;
    const uint32_t M_out = off_out[nkeys];
    const uint32_t ncta = (uint32_t)(((uint64_t)M_out + PAIR_THREADS * PAIR_B - 1) / ((uint64_t)PAIR_THREADS * PAIR_B));
    if (ncta == 0) return;
    const uint32_t nchunks = (ncta + PAIR_MID_THREADS - 1) / PAIR_MID_THREADS;
    // forward: cta_factor[c] = product of totals before c
    if (threadIdx.x == 0) carry_s = F::one();
    __syncthreads();
    for (uint32_t ch = 0; ch < nchunks; ch++) {
        const uint32_t c = ch * PAIR_MID_THREADS + threadIdx.x;
        fe_t v = c < ncta ? load_fe(cta_total + (size_t)c * 32) : F::one();
        sh[threadIdx.x] = v;
        __syncthreads();
        for (int d = 1; d < PAIR_MID_THREADS; d <<= 1) {
            fe_t a;
            const bool up = (int)threadIdx.x >= d;
            if (up) a = F::mul(sh[threadIdx.x], sh[threadIdx.x - d]);
            __syncthreads();
            if (up) sh[threadIdx.x] = a;
            __syncthreads();
        }
        const fe_t carry = carry_s;
        fe_t excl = threadIdx.x > 0 ? F::mul(carry, sh[threadIdx.x - 1]) : carry;
        if (c < ncta) store_fe(cta_factor + (size_t)c * 32, excl);
        __syncthreads();
        if (threadIdx.x == PAIR_MID_THREADS - 1) carry_s = F::mul(carry, sh[threadIdx.x]);
        __syncthreads();
    }
    // grid total and its inverse
    __shared__ fe_t inv_s;
    if (threadIdx.x == 0) inv_s = F::inv_gcd(carry_s);
    __syncthreads();
    // backward: multiply in the product of totals after c, then the inverse
    if (threadIdx.x == 0) carry_s = inv_s;          // carry = inv * (product of totals after the current chunk)
    __syncthreads();
    for (uint32_t chi = nchunks; chi-- > 0;) {
        const uint32_t c = chi * PAIR_MID_THREADS + threadIdx.x;
        fe_t v = c < ncta ? load_fe(cta_total + (size_t)c * 32) : F::one();
        sh[threadIdx.x] = v;
        __syncthreads();
        for (int d = 1; d < PAIR_MID_THREADS; d <<= 1) {       // inclusive suffix products
            fe_t a;
            const bool dn = (int)threadIdx.x + d < PAIR_MID_THREADS;
            if (dn) a = F::mul(sh[threadIdx.x], sh[threadIdx.x + d]);
            __syncthreads();
            if (dn) sh[threadIdx.x] = a;
            __syncthreads();
        }
        const fe_t carry = carry_s;
        fe_t after = threadIdx.x + 1 < PAIR_MID_THREADS ? F::mul(carry, sh[threadIdx.x + 1]) : carry;
        if (c < ncta) store_fe(cta_factor + (size_t)c * 32, F::mul(load_fe(cta_factor + (size_t)c * 32), after));
        __syncthreads();
        if (threadIdx.x == 0) carry_s = F::mul(carry, sh[0]);
        __syncthreads();
    }
}

// backward pass: back-substitution of the shared inverse, slopes, sums
template <int CURVE, bool FIRST>
__global__ void __launch_bounds__(PAIR_THREADS) k_pair_bwd(const uint32_t *__restrict__ off_in, const uint32_t *__restrict__ off_out,
                                                           uint32_t nkeys, const uint32_t *__restrict__ entries,
                                                           const affine_t *__restrict__ pts_in, const uint8_t *__restrict__ pref,
                                                           const uint8_t *__restrict__ kinds, const uint8_t *__restrict__ thread_factor,
                                                           const uint8_t *__restrict__ cta_factor, affine_t *__restrict__ pts_out) {
    using F = typename Curve<CURVE>::F;
    const uint32_t M_out = off_out[nkeys];
    const uint32_t t = blockIdx.x * PAIR_THREADS + threadIdx.x;
    const uint64_t s64 = (uint64_t)t * PAIR_B;
    if (s64 >= M_out) return;
    const uint32_t s0 = (uint32_t)s64;
    const uint32_t s1 = (s64 + PAIR_B < M_out) ? (uint32_t)(s64 + PAIR_B) : M_out;
    fe_t rinv = F::mul(load_fe(cta_factor + (size_t)blockIdx.x * 32), load_fe(thread_factor + (size_t)t * 32));
    // bucket of the last slot, then walk backwards
    uint32_t k, bstart;
    {
        PairWalk w; w.init(off_out, nkeys, s1 - 1);
        k = w.k; bstart = off_out[k];
    }
#pragma unroll 1
    for (uint32_t s = s1; s-- > s0;) {
        if (s < bstart) {
            k--; bstart = off_out[k];
            if (s < bstart) { PairWalk w; w.init(off_out, nkeys, s); k = w.k; bstart = off_out[k]; }
        }
        const uint32_t i0 = off_in[k] + 2 * (s - bstart);
        const uint8_t kind = kinds[s];
        affine_t r;
        if (kind == PAIR_PASS0 || kind == PAIR_PASS1) {
            const uint32_t i = kind == PAIR_PASS0 ? i0 : i0 + 1;
            r.x = pair_load_x<FIRST>(entries, pts_in, i);
            r.y = pair_load_y<CURVE, FIRST>(entries, pts_in, i);
        } else if (kind == PAIR_IDENT) {
            r = affine_identity_marker();
        } else {
            const fe_t x0 = pair_load_x<FIRST>(entries, pts_in, i0), y0 = pair_load_y<CURVE, FIRST>(entries, pts_in, i0);
            const fe_t x1 = pair_load_x<FIRST>(entries, pts_in, i0 + 1);
            fe_t den, num;
            if (kind == PAIR_ADD) { den = F::sub(x1, x0); num = F::sub(pair_load_y<CURVE, FIRST>(entries, pts_in, i0 + 1), y0); }
            else { den = F::dbl(y0); fe_t xx = F::sqr(x0); num = F::add(F::dbl(xx), xx); }
            const fe_t dinv = F::mul(rinv, load_fe(pref + (size_t)s * 32));
            rinv = F::mul(rinv, den);
            const fe_t lam = F::mul(num, dinv);
            r.x = F::sub(F::sub(F::sqr(lam), x0), x1);
            r.y = F::sub(F::mul(lam, F::sub(x0, r.x)), y0);
        }
        store_fe(&pts_out[s].x, r.x); store_fe(&pts_out[s].y, r.y);
    }
}

// k_fixup: one CTA merges the 2 * G boundary partials left by k_accumulate and writes the buckets.
template <int CURVE>
__global__ void __launch_bounds__(FIX_THREADS) k_fixup(const uint32_t *__restrict__ cta_ids,
                                                 const xyzz_t *__restrict__ cta_parts, uint32_t ns,
                                                 xyzz_t *__restrict__ buckets) {
    extern __shared__ uint4 smem_raw[];
    xyzz_t *slot_pt = reinterpret_cast<xyzz_t *>(smem_raw);
    uint32_t *slot_id = reinterpret_cast<uint32_t *>(slot_pt + ns);
    for (uint32_t i = threadIdx.x; i < ns; i += blockDim.x) {
        slot_id[i] = cta_ids[i];
        slot_pt[i] = load_xyzz(cta_parts + i);
    }
    __syncthreads();
    seg_scan<CURVE, FIX_PER_T, FpCall>(slot_pt, slot_id, ns);      // one pass over ~600 slots: latency-bound, keep the code small
    for (uint32_t i = threadIdx.x; i < ns; i += blockDim.x) {
        uint32_t id = slot_id[i];
        if (id == NONE_ID) continue;
        bool group_end = (i + 1 == ns) || slot_id[i + 1] != id;
        if (group_end) store_xyzz(buckets + id, slot_pt[i]);
    }
}

// ------------------------------------------------------------------------------------------------
// bucket reduction  S = sum_{k < nb} (k + 1) * B_k  per bucket set, as  W + T  with  W = sum k B_k,  T = sum B_k.
//
// The tail of the MSM is bound by the latency of dependent point additions (one warp needs ~10k cycles per XYZZ
// add, tools/latbench.cu), so the reduction is organised for depth, not for work: the bucket index is split
// k = hi * C + lo and
//     W = C * sum_hi hi * R_hi + sum_lo lo * C_lo,      R_hi = sum_lo B[hi][lo],   C_lo = sum_hi B[hi][lo]
// turns one weighted sum over R * C items into plain (tree) sums plus two weighted sums over R and C items.
// Applied twice (nb <= 2^20 -> <= 1024 -> <= 32) the weighted sums left are over <= 32 items: one warp each.
// k_sums / k_sums_coop do every plain-sum level (tasks describe rows / columns), k_leaf_scan_coop the four 32-item
// weighted sums and k_leaf_combine_coop the recombination.  Depth for 2^19 buckets: ~12 + 5 + 10 additions + 15 doublings, instead of ~90.
// ------------------------------------------------------------------------------------------------

struct SumTask {
    uint32_t in_off;      // first item of the task inside the set's input array
    uint32_t out_off;     // first output inside the set's output array
    uint32_t n_out;       // outputs
    uint32_t len;         // items per output
    uint32_t stride_out;  // input step between consecutive outputs
    uint32_t stride_len;  // input step between consecutive items of one output
    uint32_t out_stride;  // output step between consecutive outputs (0 = 1)
    uint32_t pair;        // 1: every item is the sum of two adjacent elements (the two halves of a split column sum)
};
struct SumTasks {
    SumTask t[4];
    uint32_t ntasks;
};

// out[set][task.out_off + o] = sum_{j < len} in[set][task.in_off + o * stride_out + j * stride_len]
// One CTA of BLK threads per output.  offsets != nullptr: `in` are buckets and empty ones (never written) are skipped.
template <int CURVE, int BLK>
__global__ void __launch_bounds__(BLK) k_sums(const xyzz_t *__restrict__ in, uint32_t in_set_stride,
                                              const uint32_t *__restrict__ offsets, xyzz_t *__restrict__ out,
                                              uint32_t out_set_stride, SumTasks tasks) {
    using Cv = Curve<CURVE, FpCall>;
    __shared__ xyzz_t part[BLK / 32];
    uint32_t o = blockIdx.x, ti = 0;
    while (ti + 1 < tasks.ntasks && o >= tasks.t[ti].n_out) { o -= tasks.t[ti].n_out; ti++; }
    const SumTask tk = tasks.t[ti];
    const uint32_t set = blockIdx.y;
    const xyzz_t *src = in + (size_t)set * in_set_stride;
    const uint32_t *offs = offsets ? offsets + (size_t)set * in_set_stride : nullptr;
    xyzz_t acc = Cv::identity();
    for (uint32_t j = threadIdx.x; j < tk.len; j += BLK) {
        uint32_t idx = tk.in_off + o * tk.stride_out + j * tk.stride_len;
        if (!offs || offs[idx + 1] != offs[idx]) { xyzz_t b = load_xyzz(src + idx); Cv::add(acc, b); }
        if (tk.pair) { xyzz_t b = load_xyzz(src + idx + 1); Cv::add(acc, b); }
    }
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t live = tk.len < BLK ? tk.len : BLK;       // threads that may hold something
#pragma unroll 1
    for (int d = 16; d >= 1; d >>= 1) {
        if ((uint32_t)d < live) {                            // uniform across the CTA
            xyzz_t other = shfl_down_xyzz(acc, d);
            if (lane < (uint32_t)d) Cv::add(acc, other);
        }
    }
    if (BLK > 32) {
        if (lane == 0) part[wid] = acc;
        __syncthreads();
        if (wid == 0) {
            acc = lane < BLK / 32 && lane * 32 < live ? part[lane] : Cv::identity();
#pragma unroll 1
            for (int d = BLK / 64; d >= 1; d >>= 1) {
                if ((uint32_t)d * 32 < live) {
                    xyzz_t other = shfl_down_xyzz(acc, d);
                    if (lane < (uint32_t)d) Cv::add(acc, other);
                }
            }
        }
    }
    if (threadIdx.x == 0) store_xyzz(out + (size_t)set * out_set_stride + tk.out_off + o * (tk.out_stride ? tk.out_stride : 1u), acc);
}

// Leaf of the reduction per bucket set: leaf[set][a][j], a < 4, j < 32.  W_a = sum_j j * leaf[a][j] (suffix scan, then a
// sum over the lanes >= 1), T_a = sum_j leaf[a][j], and
//   nlevels == 2:  S = 2^s0 * (2^5 * W_0 + W_1) + (2^5 * W_2 + W_3) + T_0
//   nlevels == 1:  S = 2^5 * W_0 + W_1 + T_0            nlevels == 0:  S = W_0 + T_0
// (k_leaf_scan_coop / k_leaf_combine_coop below.)

template <int CURVE>
__global__ void __launch_bounds__(128) k_accumulate_warp_coop(const uint32_t *__restrict__ offsets, uint32_t nkeys,
                                                               const uint32_t *__restrict__ entries,
                                                               const affine_t *__restrict__ bases, xyzz_t *__restrict__ buckets) {
    using Cv = Curve<CURVE, FpCall>;
    using Co = Coop<CURVE>;
    __shared__ CoopScratch scratch;
    const uint32_t k = blockIdx.x, lane = threadIdx.x & 31;
    CoopCtx c{&scratch, threadIdx.x >> 5, lane, 1, 0};
    const uint32_t b0 = offsets[k], b1 = offsets[k + 1];
    if (b0 == b1) return;                      // empty bucket (CTA-uniform): never read by the reduction
    xyzz_t acc = Cv::identity();
#pragma unroll 1
    for (uint32_t p0 = b0; p0 < b1; p0 += 32) {
        const uint32_t p = p0 + lane;
        xyzz_t q = Cv::identity();
        if (p < b1) {
            uint32_t ent = entries[p];
            affine_t pt = load_affine(bases + (ent & 0x7fffffffu));
            if (ent >> 31) pt.y = Cv::F::neg(pt.y);
            q = Cv::from_affine(pt);
        }
        if (p0 == b0) acc = q; else Co::add(c, acc, q);
    }
    const uint32_t m = b1 - b0;
#pragma unroll 1
    for (int d = 16; d >= 1; d >>= 1) {
        if ((uint32_t)d < m) {
            xyzz_t other = shfl_down_xyzz(acc, d), t = acc;
            if (lane >= (uint32_t)d) other = Cv::identity();
            Co::add(c, t, other);
            if (lane < (uint32_t)d) acc = t;
        }
    }
    if (threadIdx.x == 0) store_xyzz(buckets + k, acc);
}

// Cooperative versions (coop.cuh: four replica warps per warp of points, ~3x lower latency per point operation).
// k_sums_coop: one group (128 threads) per output.
template <int CURVE>
__global__ void __launch_bounds__(128) k_sums_coop(const xyzz_t *__restrict__ in, uint32_t in_set_stride,
                                                    const uint32_t *__restrict__ offsets, xyzz_t *__restrict__ out,
                                                    uint32_t out_set_stride, SumTasks tasks) {
    using Cv = Curve<CURVE, FpCall>;
    using Co = Coop<CURVE>;
    __shared__ CoopScratch scratch;
    uint32_t o = blockIdx.x, ti = 0;
    while (ti + 1 < tasks.ntasks && o >= tasks.t[ti].n_out) { o -= tasks.t[ti].n_out; ti++; }
    const SumTask tk = tasks.t[ti];
    const uint32_t set = blockIdx.y, lane = threadIdx.x & 31;
    CoopCtx c{&scratch, threadIdx.x >> 5, lane, 1, 0};
    const xyzz_t *src = in + (size_t)set * in_set_stride;
    const uint32_t *offs = offsets ? offsets + (size_t)set * in_set_stride : nullptr;
    xyzz_t acc = Cv::identity();
#pragma unroll 1
    for (uint32_t j0 = 0; j0 < tk.len; j0 += 32) {
        const uint32_t j = j0 + lane;
        xyzz_t b = Cv::identity(), b2 = Cv::identity();
        if (j < tk.len) {
            uint32_t idx = tk.in_off + o * tk.stride_out + j * tk.stride_len;
            if (!offs || offs[idx + 1] != offs[idx]) b = load_xyzz(src + idx);
            if (tk.pair) b2 = load_xyzz(src + idx + 1);
        }
        if (j0 == 0) acc = b; else Co::add(c, acc, b);
        if (tk.pair) Co::add(c, acc, b2);          // uniform across the group
    }
    const uint32_t live = tk.len < 32 ? tk.len : 32;
#pragma unroll 1
    for (int d = 16; d >= 1; d >>= 1) {
        if ((uint32_t)d < live) {
            xyzz_t other = shfl_down_xyzz(acc, d), t = acc;
            if (lane >= (uint32_t)d) other = Cv::identity();     // idle lanes must not wander into the P == Q path
            Co::add(c, t, other);
            if (lane < (uint32_t)d) acc = t;
        }
    }
    if (threadIdx.x == 0) store_xyzz(out + (size_t)set * out_set_stride + tk.out_off + o * (tk.out_stride ? tk.out_stride : 1u), acc);
}

// The leaf in cooperative form, two launches so that every group is its own CTA (a 16-warp CTA would be capped at 128
// registers per thread and spill the points): k_leaf_scan_coop, grid (arrays, sets): W_a = sum_j j * leaf[a][j] and, for
// a == 0, T_0 = sum_j leaf[0][j] -> ws[set][0..3], ws[set][4]; k_leaf_combine_coop, grid sets x 2 groups: the recombination
// (formulas above).
template <int CURVE>
__global__ void __launch_bounds__(128) k_leaf_scan_coop(const xyzz_t *__restrict__ leaf, uint32_t leaf_set_stride,
                                                         xyzz_t *__restrict__ ws) {
    using Cv = Curve<CURVE, FpCall>;
    using Co = Coop<CURVE>;
    __shared__ CoopScratch scratch;
    const uint32_t a = blockIdx.x, set = blockIdx.y, lane = threadIdx.x & 31;
    CoopCtx c{&scratch, threadIdx.x >> 5, lane, 1, 0};
    xyzz_t run = load_xyzz(leaf + (size_t)set * leaf_set_stride + a * 32 + lane);
#pragma unroll 1
    for (int d = 1; d < 32; d <<= 1) {            // suffix scan: run_j = sum_{i >= j} item_i
        xyzz_t o = shfl_down_xyzz(run, d), t = run;
        if (lane + d >= 32) o = Cv::identity();   // idle lanes must not wander into the P == Q path
        Co::add(c, t, o);
        if (lane + d < 32) run = t;
    }
    if (a == 0 && threadIdx.x == 0) store_xyzz(ws + (size_t)set * 5 + 4, run);
    xyzz_t jr = lane >= 1 ? run : Cv::identity();   // sum_j j * item_j = sum_{j >= 1} run_j
#pragma unroll 1
    for (int d = 16; d >= 1; d >>= 1) {
        xyzz_t o = shfl_down_xyzz(jr, d), t = jr;
        if (lane >= (uint32_t)d) o = Cv::identity();
        Co::add(c, t, o);
        if (lane < (uint32_t)d) jr = t;
    }
    if (threadIdx.x == 0) store_xyzz(ws + (size_t)set * 5 + a, jr);
}
//   nlevels == 2:  S = 2^s0 * (2^5 * W_0 + W_1) + (2^5 * W_2 + W_3) + T_0
//   nlevels == 1:  S = 2^5 * W_0 + W_1 + T_0            nlevels == 0:  S = W_0 + T_0
template <int CURVE>
__global__ void __launch_bounds__(256) k_leaf_combine_coop(const xyzz_t *__restrict__ ws, int nlevels, uint32_t s0,
                                                            xyzz_t *__restrict__ out) {
    using Co = Coop<CURVE>;
    __shared__ CoopScratch scratch[2];
    __shared__ xyzz_t H[2];
    const uint32_t set = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = warp >> 2;
    CoopCtx c{&scratch[g], warp & 3u, lane, 1 + g, 0};
    const xyzz_t *w = ws + (size_t)set * 5;
    if (nlevels >= 1 && (g == 0 || nlevels == 2)) {      // the two 2^5 recombinations, one group each
        xyzz_t hi = load_xyzz(w + 2 * g);
#pragma unroll 1
        for (int b = 0; b < 5; b++) hi = Co::dbl(c, hi);
        xyzz_t lo = load_xyzz(w + 2 * g + 1);
        Co::add(c, hi, lo);
        if (c.role == 0 && lane == 0) H[g] = hi;
    }
    __syncthreads();
    if (g == 0) {
        xyzz_t acc = nlevels >= 1 ? H[0] : load_xyzz(w);
        if (nlevels == 2) {
#pragma unroll 1
            for (uint32_t b = 0; b < s0; b++) acc = Co::dbl(c, acc);
            xyzz_t lo = H[1];
            Co::add(c, acc, lo);
        }
        xyzz_t t = load_xyzz(w + 4);
        Co::add(c, acc, t);
        if (threadIdx.x == 0) store_xyzz(out + set, acc);
    }
}

// k_finish (one CTA per job): out = sum_w 2^(c w) S_w (+ optional extra partials), left as an un-normalised XYZZ sum.
template <int CURVE>
__global__ void k_finish(const xyzz_t *__restrict__ window_sums, uint32_t nwin, uint32_t c,
                         const xyzz_t *__restrict__ extra, uint32_t n_extra,
                         xyzz_t *__restrict__ out_partial, xyzz_t *__restrict__ out_raw) {
    using Cv = Curve<CURVE>;      // loops over one dbl / one sqr-mul body: already instruction-cache friendly
    if (threadIdx.x != 0) return;
    const uint32_t job = blockIdx.x;
    window_sums += (size_t)job * nwin;
    xyzz_t acc = Cv::identity();
    for (int w = (int)nwin - 1; w >= 0; w--) {
        if (!Cv::is_identity(acc)) for (uint32_t b = 0; b < c; b++) acc = Cv::dbl(acc);
        xyzz_t s = load_xyzz(window_sums + w);
        Cv::add(acc, s);
    }
    for (uint32_t i = 0; i < n_extra; i++) { xyzz_t s = load_xyzz(extra + (size_t)job * n_extra + i); Cv::add(acc, s); }
    // out_partial: a share for a later combine (possibly a peer GPU's memory); out_raw: the result the host fetches and converts
    // to affine itself (hostfp.hpp) -- the single inversion of an MSM does not run on one GPU thread any more
    if (out_partial) store_xyzz(out_partial + job, acc);
    if (out_raw) store_xyzz(out_raw + job, acc);
}

// k_finish for PLAIN keys (no window table): the Horner over the windows is ~256 dependent doublings -- 0.8 ms on one thread,
// the whole latency of a one-shot MSM (succinct-check equations, short commitment combinations).  One cooperative group
// (coop.cuh) per job runs every doubling in 3 product phases and every addition in 4; all lanes carry the same point.
template <int CURVE>
__global__ void __launch_bounds__(128) k_finish_coop(const xyzz_t *__restrict__ window_sums, uint32_t nwin, uint32_t c,
                                                      const xyzz_t *__restrict__ extra, uint32_t n_extra,
                                                      xyzz_t *__restrict__ out_partial, xyzz_t *__restrict__ out_raw) {
    using Cv = Curve<CURVE, FpCall>;
    using Co = Coop<CURVE>;
    __shared__ CoopScratch scratch;
    CoopCtx cc{&scratch, threadIdx.x >> 5, threadIdx.x & 31, 1, 0};
    const uint32_t job = blockIdx.x;
    window_sums += (size_t)job * nwin;
    xyzz_t acc = Cv::identity();
#pragma unroll 1
    for (int w = (int)nwin - 1; w >= 0; w--) {
        if (!Cv::is_identity(acc)) {                 // uniform across the group: every lane holds the same point
#pragma unroll 1
            for (uint32_t b = 0; b < c; b++) acc = Co::dbl(cc, acc);
        }
        xyzz_t s = load_xyzz(window_sums + w);
        Co::add(cc, acc, s);
    }
#pragma unroll 1
    for (uint32_t i = 0; i < n_extra; i++) { xyzz_t s = load_xyzz(extra + (size_t)job * n_extra + i); Co::add(cc, acc, s); }
    if (threadIdx.x == 0) {
        if (out_partial) store_xyzz(out_partial + job, acc);
        if (out_raw) store_xyzz(out_raw + job, acc);
    }
}

// out[j] = sum_r partials[r * m + j], j < m: the G-way add after an all-gather of m shares per rank (rank-major, as the
// gather leaves them).  One CTA per output, one thread (G <= 16 additions); the host normalises.
template <int CURVE>
__global__ void k_combine_batch(const xyzz_t *__restrict__ partials, uint32_t k, uint32_t m, xyzz_t *__restrict__ out_raw) {
    using Cv = Curve<CURVE>;
    if (threadIdx.x != 0) return;
    const uint32_t j = blockIdx.x;
    xyzz_t acc = Cv::identity();
    for (uint32_t r = 0; r < k; r++) { xyzz_t s = load_xyzz(partials + (size_t)r * m + j); Cv::add(acc, s); }
    store_xyzz(out_raw + j, acc);
}

// ------------------------------------------------------------------------------------------------
// k_precompute: table[w * n + i] = 2^(c w) * P_i in affine form, w < nwin.  One thread per base walks the
// doubling chain in XYZZ, keeps the nwin - 1 intermediate points in local memory and normalises them with
// ONE inversion (Montgomery batch inversion over its own chain).  Run once per registered key: commitment
// keys are fixed for the life of a prover (trim / index time), so the MSM then needs a single bucket set,
// one bucket reduction and no window doublings.
// ------------------------------------------------------------------------------------------------
constexpr int MAX_PRE_WINDOWS = 64;   // c >= 4
template <int CURVE>
__global__ void __launch_bounds__(128) k_precompute(const affine_t *__restrict__ bases, uint32_t n, uint32_t c,
                                                     uint32_t nwin, affine_t *__restrict__ table) {
    using Cv = Curve<CURVE>;
    using F = typename Cv::F;
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    affine_t p = load_affine(bases + i);
    store_fe(&table[i].x, p.x); store_fe(&table[i].y, p.y);
    xyzz_t pts[MAX_PRE_WINDOWS];
    fe_t pref[MAX_PRE_WINDOWS];
    xyzz_t cur = Cv::from_affine(p);
    fe_t run = F::one();
#pragma unroll 1
    for (uint32_t w = 1; w < nwin; w++) {
#pragma unroll 1
        for (uint32_t b = 0; b < c; b++) cur = Cv::dbl(cur);
        pts[w] = cur;
        pref[w] = run;
        run = F::mul(run, cur.zzz);
    }
    fe_t inv = F::inv(run);
#pragma unroll 1
    for (uint32_t w = nwin - 1; w >= 1; w--) {
        fe_t t = F::mul(inv, pref[w]);            // ZZZ_w^-1
        inv = F::mul(inv, pts[w].zzz);
        fe_t zt = F::mul(pts[w].zz, t);           // ZZ^-1 = (ZZ t)^2 since ZZ^3 = ZZZ^2
        affine_t *dst = table + (size_t)w * n + i;
        store_fe(&dst->x, F::mul(pts[w].x, F::sqr(zt)));
        store_fe(&dst->y, F::mul(pts[w].y, t));
    }
}

// k_precompute_coop: the same table for SHORT keys, where the launch above is bound by the latency of one thread's chain
// (255 doublings x 9 products + a Fermat inversion, ~0.9 ms whatever the key length): one cooperative group (coop.cuh: four
// replica warps on the four sub-partitions of an SM) per 32 bases runs every doubling in 3 product phases, the inversion
// is the binary-GCD one (divergent, but nothing else competes for the SM), and the back-substitution of the windows is
// dealt round-robin to the four replicas (every replica walks the running inverse, each converts its own windows).
// Used by the folded keys an IpaPC::open session materialises (ipa_api.inc) and for registered keys up to 2^12 points
// (PRECOMPUTE_COOP_MAX, accmsm.cu).
template <int CURVE>
__global__ void __launch_bounds__(128) k_precompute_coop(const affine_t *__restrict__ bases, uint32_t n, uint32_t c,
                                                          uint32_t nwin, affine_t *__restrict__ table) {
    using Cv = Curve<CURVE, FpCall>;
    using F = typename Cv::F;
    using Co = Coop<CURVE>;
    __shared__ CoopScratch scratch;
    const uint32_t lane = threadIdx.x & 31, role = threadIdx.x >> 5;
    CoopCtx cc{&scratch, role, lane, 1, 0};
    const uint32_t i = blockIdx.x * 32 + lane;
    const bool live = i < n;                       // idle lanes of the last group walk a copy of base n - 1 (no stores)
    affine_t p = load_affine(bases + (live ? i : n - 1));
    if (live && role == 0) { store_fe(&table[i].x, p.x); store_fe(&table[i].y, p.y); }
    xyzz_t pts[MAX_PRE_WINDOWS];
    fe_t pref[MAX_PRE_WINDOWS];
    xyzz_t cur = Cv::from_affine(p);
    fe_t run = F::one();
#pragma unroll 1
    for (uint32_t w = 1; w < nwin; w++) {
#pragma unroll 1
        for (uint32_t b = 0; b < c; b++) cur = Co::dbl(cc, cur);
        pts[w] = cur;
        pref[w] = run;
        run = F::mul(run, cur.zzz);
    }
    fe_t inv = F::inv_gcd(run);
#pragma unroll 1
    for (uint32_t w = nwin - 1; w >= 1; w--) {
        if ((w & 3u) == role) {
            fe_t t = F::mul(inv, pref[w]);            // ZZZ_w^-1
            fe_t zt = F::mul(pts[w].zz, t);           // ZZ^-1 = (ZZ t)^2 since ZZ^3 = ZZZ^2
            if (live) {
                affine_t *dst = table + (size_t)w * n + i;
                store_fe(&dst->x, F::mul(pts[w].x, F::sqr(zt)));
                store_fe(&dst->y, F::mul(pts[w].y, t));
            }
        }
        inv = F::mul(inv, pts[w].zzz);
    }
}

// ------------------------------------------------------------------------------------------------
// k_synth_points: seeded synthetic commitment key for benchmarks / tests (SURVEY.md 8d): base i is
// s_i * G with G = (-1, 2) and s_i a 254-bit SplitMix64 value of (seed, global index), so any shard of
// the key can be generated independently on its own GPU without a host round trip.
// ------------------------------------------------------------------------------------------------
ACC_D uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}
template <int CURVE>
__global__ void __launch_bounds__(128) k_synth_points(uint64_t seed, uint64_t first_index, uint32_t n,
                                                       affine_t *__restrict__ out) {
    using Cv = Curve<CURVE>;
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t idx = first_index + i;
    uint32_t s[8];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        uint64_t v = splitmix64(seed ^ splitmix64(idx * 4 + j));
        s[2 * j] = (uint32_t)v; s[2 * j + 1] = (uint32_t)(v >> 32);
    }
    s[7] &= 0x3fffffffu;    // < 2^254 < group order
    s[0] |= 1u;             // never zero
    affine_t g;
    g.x = Cv::F::neg(Cv::F::one());
    g.y = Cv::F::dbl(Cv::F::one());
    xyzz_t acc = Cv::identity();
#pragma unroll 1
    for (int b = 253; b >= 0; b--) {
        acc = Cv::dbl(acc);
        if ((s[b >> 5] >> (b & 31)) & 1u) Cv::madd(acc, g);
    }
    affine_t a; uint32_t inf;
    Cv::to_affine(acc, a, inf);
    store_fe(&out[i].x, a.x); store_fe(&out[i].y, a.y);
}

}  // namespace accmsm
