// Device side of IpaPC::open (ark-poly-commit ipa_pc, SURVEY.md App. A.2; reference call sites
// src/ipa_pc_as/mod.rs:454-462 (AS prove), :525-534 (index: default proof), examples/scaling-pc.rs:72-81).
// The opening state -- coefficient vector and z-vector (1, z, z^2, ...) -- stays resident in HBM across the log2(D)
// rounds; per round only the two points (l, r) go to the host sponge and one challenge comes back.
//   round:  l = cm_commit(key_l, coeffs_r) + <coeffs_r, z_l> h'     r = cm_commit(key_r, coeffs_l) + <coeffs_l, z_r> h'
//   fold:   coeffs_l += xi^-1 coeffs_r ;  z_l += xi z_r ;  key_l += xi key_r
// The key is never folded explicitly: the folded key of round j is a fixed linear combination of the registered key
// (coefficients = products of the challenges so far), so every round's (l, r) is an MSM over the REGISTERED key with
// scalars generated on the fly (IpaRoundScalars in msm.cuh) -- the window table applies, there is no Horner over
// windows and no per-round scalar multiplication of n/2 generators; final_comm_key is one more such MSM.
#pragma once
#include "vec.cuh"

namespace accmsm {

// z_vec[i] = scale * z^(offset + (i << log_stride)) by square-and-multiply on the index (one thread per element).
// offset < 2^log_stride; (0, 0, nullptr) gives the plain power vector.  The strided form is the z-vector of ONE cyclic
// shard (index mod 2^log_stride == offset) of a multi-GPU opening; `scale` carries the factor the z-vector has picked
// up in rounds that were folded elsewhere.
template <int FIELD>
__global__ void __launch_bounds__(256) k_powers(const uint8_t *__restrict__ z_ptr, uint32_t n, uint8_t *__restrict__ out,
                                                 uint32_t log_stride, uint32_t offset, const uint8_t *__restrict__ scale) {
    using F = Fp<FIELD>;
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe_t zc = load_fe(z_ptr), pw = scale ? load_fe(scale) : F::one();
    for (uint32_t b = 0; b < log_stride; b++) {
        if ((offset >> b) & 1u) pw = F::mul(pw, zc);
        zc = F::sqr(zc);
    }
    for (uint32_t e = i; e; e >>= 1) {
        if (e & 1u) pw = F::mul(pw, zc);
        zc = F::sqr(zc);
    }
    store_fe(out + (size_t)i * 32, pw);
}

// blockIdx.y = 0: <coeffs[h..2h), z[0..h)>   blockIdx.y = 1: <coeffs[0..h), z[h..2h)>; per-block partial sums
template <int FIELD>
__global__ void __launch_bounds__(256) k_ipa_inner_partial(const uint8_t *__restrict__ coeffs, const uint8_t *__restrict__ z,
                                                            uint32_t h, uint8_t *__restrict__ partials) {
    using F = Fp<FIELD>;
    __shared__ fe_t sh[256];
    const uint8_t *a = blockIdx.y == 0 ? coeffs + (size_t)h * 32 : coeffs;
    const uint8_t *b = blockIdx.y == 0 ? z : z + (size_t)h * 32;
    fe_t acc = F::zero();
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < h; i += gridDim.x * blockDim.x)
        acc = F::add(acc, F::mul(load_fe_nc(a + (size_t)i * 32), load_fe_nc(b + (size_t)i * 32)));
    fe_t s = block_sum<FIELD>(acc, sh);
    if (threadIdx.x == 0) store_fe(partials + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 32, s);
}
// grid = 2 blocks: out[y] = canonical(scale * sum of partials[y][0..nparts)), scale = 1 when nullptr  -- canonical
// because it feeds either the byte loop of k_ipa_hp_mul or the digit decomposition of the MSM
template <int FIELD>
__global__ void __launch_bounds__(256) k_ipa_inner_final(const uint8_t *__restrict__ partials, uint32_t nparts,
                                                          const uint8_t *__restrict__ scale, uint8_t *__restrict__ out_canon) {
    using F = Fp<FIELD>;
    __shared__ fe_t sh[256];
    fe_t acc = F::zero();
    for (uint32_t i = threadIdx.x; i < nparts; i += blockDim.x)
        acc = F::add(acc, load_fe(partials + ((size_t)blockIdx.x * nparts + i) * 32));
    fe_t s = block_sum<FIELD>(acc, sh);
    if (threadIdx.x == 0) {
        if (scale) s = F::mul(s, load_fe(scale));
        store_fe(out_canon + (size_t)blockIdx.x * 32, F::from_mont(s));
    }
}

// hp_table[j] = 2^(8 j) h' (XYZZ), j < 32, once per opening session: a chain of 248 dependent doublings, run by one
// cooperative group (coop.cuh: 3 product phases per doubling instead of 9 serial products; 128 threads)
template <int CURVE>
__global__ void __launch_bounds__(128) k_ipa_hp_table(const affine_t *__restrict__ hp, xyzz_t *__restrict__ table) {
    using Cv = Curve<CURVE, FpCall>;
    using Co = Coop<CURVE>;
    __shared__ CoopScratch scratch;
    CoopCtx c{&scratch, threadIdx.x >> 5, threadIdx.x & 31u, 1, 0};
    xyzz_t cur = Cv::from_affine(load_affine(hp));
#pragma unroll 1
    for (int j = 0; j < 32; j++) {
        if (threadIdx.x == 0) store_xyzz(table + j, cur);
        if (j < 31) {
#pragma unroll 1
            for (int b = 0; b < 8; b++) cur = Co::dbl(c, cur);
        }
    }
}
// out[y] = ip[y] * h' for y = 0, 1 (one cooperative group each, 256 threads): lane j multiplies byte j of the scalar into
// 2^(8j) h', then the 32 partial points are summed by a shuffle tree.
template <int CURVE>
__global__ void __launch_bounds__(256) k_ipa_hp_mul(const xyzz_t *__restrict__ table, const uint8_t *__restrict__ ip_canon,
                                                     xyzz_t *__restrict__ out) {
    using Cv = Curve<CURVE, FpCall>;
    using Co = Coop<CURVE>;
    __shared__ CoopScratch scratch[2];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31, y = warp >> 2;
    CoopCtx c{&scratch[y], warp & 3u, lane, 1 + y, 0};
    const uint32_t byte = ip_canon[y * 32 + lane];
    const xyzz_t base = load_xyzz(table + lane);
    xyzz_t acc = Cv::identity();
#pragma unroll 1
    for (int b = 7; b >= 0; b--) {
        acc = Co::dbl(c, acc);
        xyzz_t q = ((byte >> b) & 1u) ? base : Cv::identity();
        Co::add(c, acc, q);
    }
#pragma unroll 1
    for (int d = 16; d >= 1; d >>= 1) {
        xyzz_t o = shfl_down_xyzz(acc, d), t = acc;
        if (lane >= (uint32_t)d) o = Cv::identity();
        Co::add(c, t, o);
        if (lane < (uint32_t)d) acc = t;
    }
    if ((warp & 3u) == 0 && lane == 0) store_xyzz(out + y, acc);
}

// coeffs[i] += xi_inv * coeffs[i + h] ;  z[i] += xi * z[i + h].  The challenge and its inverse travel as kernel
// arguments (no H2D copy from caller memory that could still be in flight when the caller reuses its buffer); thread 0
// also records xi as challenge `round` of the session.
template <int FIELD>
__global__ void __launch_bounds__(256) k_ipa_fold_scalars(uint8_t *__restrict__ coeffs, uint8_t *__restrict__ z, uint32_t h,
                                                           fe_t x, fe_t xinv, uint8_t *__restrict__ challenge_slot) {
    using F = Fp<FIELD>;
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0 && challenge_slot) store_fe(challenge_slot, x);
    if (i >= h) return;
    uint8_t *c0 = coeffs + (size_t)i * 32, *z0 = z + (size_t)i * 32;
    store_fe(c0, F::add(load_fe(c0), F::mul(xinv, load_fe(coeffs + (size_t)(i + h) * 32))));
    store_fe(z0, F::add(load_fe(z0), F::mul(x, load_fe(z + (size_t)(i + h) * 32))));
}

// zk opening: hiding[0] -= e, so that the hiding polynomial vanishes at the point (one thread)
template <int FIELD>
__global__ void k_ipa_hide_adjust(uint8_t *__restrict__ hiding, const uint8_t *__restrict__ e) {
    store_fe(hiding, Fp<FIELD>::sub(load_fe(hiding), load_fe(e)));
}
// zk opening: coeffs[i] += alpha * hiding[i] once alpha is squeezed from (C, z, v, hiding_comm); alpha travels as a kernel
// argument like the round challenges
template <int FIELD>
__global__ void __launch_bounds__(256) k_ipa_hide_fold(uint8_t *__restrict__ coeffs, const uint8_t *__restrict__ hiding,
                                                        uint32_t n, fe_t alpha) {
    using F = Fp<FIELD>;
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t *c = coeffs + (size_t)i * 32;
    store_fe(c, F::add(load_fe(c), F::mul(alpha, load_fe(hiding + (size_t)i * 32))));
}


// ------------------------------------------------------------------------------------------------
// Folded-key materialisation.  The unfolded rounds above cost one MSM over ALL n0 / 2 pairs per job in every round,
// although the folded key of round j has only n0 / 2^j points.  After J rounds the folded key
//     FK[p] = sum_{u < 2^J} C(u) * G[u * m + p],   p < m = n / 2^J,   C(u) = prod_{r <= J : bit (J - r) of u} xi_r
// is materialised once and the session continues on it as on a freshly registered key (window table included).
// All m outputs share the 2^J scalars C(u), so nothing is sorted per point: the scalars are cut into signed
// sub-digits of `cs` bits INSIDE each window of the current key's table (table[w] = 2^(c w) G supplies the window
// weight; G = ceil(c / cs) Horner groups supply the sub-digit weight), one tiny counting sort orders the
// (u, w) pairs of every group by digit magnitude (k_fold_digits, one CTA), and k_fold_accumulate gives one thread
// per (output, group, window slice) the classical running-sum walk  sum_d d * B_d  over that shared list: every lane
// of a warp follows the same list, the loads table[w][u * m + p] are coalesced across p and there is no divergence.
// k_fold_combine adds the slices, runs the Horner recombination over the groups and normalises.
// Cost: n * nwin * G mixed additions (52 per key point for c = 20, J = 5) against J more unfolded rounds saved per
// J rounds that follow.
// ------------------------------------------------------------------------------------------------
struct FoldShape {
    uint32_t J;         // rounds folded at once; 2^J blocks of the current key are combined
    uint32_t m;         // points of the folded key
    uint32_t stride;    // points per window of the current key's table
    uint32_t c, nwin;   // radix and windows of that table
    uint32_t cs, G;     // sub-digit bits and sub-digits per table window
    uint32_t WS;        // window slices: slice ws takes the windows w with w % WS == ws
    uint32_t nbk;       // 2^(cs - 1): largest digit magnitude
};
constexpr uint32_t FOLD_MAX_KEYS = 8192;      // G * WS * (nbk + 1) list heads, held in shared memory by k_fold_digits
constexpr int FOLD_THREADS = 128;
ACC_D uint32_t fold_list(const FoldShape &f, uint32_t g, uint32_t ws, uint32_t d) { return (g * f.WS + ws) * (f.nbk + 1) + d; }
ACC_D uint32_t fold_width(const FoldShape &f, uint32_t g) { return f.c - g * f.cs < f.cs ? f.c - g * f.cs : f.cs; }

// One CTA.  entries[offsets[list] .. offsets[list + 1]) = (sign << 31 | w << 16 | u) of the pairs whose sub-digit g of
// window w has magnitude d, list = fold_list(g, w % WS, d).  digits = scratch of 2^J * nwin * G words.
template <int SFIELD>
__global__ void __launch_bounds__(256) k_fold_digits(const uint8_t *__restrict__ challenges, FoldShape f,
                                                      uint32_t *__restrict__ digits, uint32_t *__restrict__ offsets,
                                                      uint32_t *__restrict__ entries) {
    using F = Fp<SFIELD>;
    __shared__ uint32_t heads[FOLD_MAX_KEYS + 1];
    __shared__ uint32_t chunk_sum[256];
    const uint32_t T = 1u << f.J, nlists = f.G * f.WS * (f.nbk + 1), tid = threadIdx.x;
    for (uint32_t k = tid; k <= nlists; k += 256) heads[k] = 0;
    __syncthreads();
    for (uint32_t u = tid; u < T; u += 256) {
        fe_t acc = F::one();
        for (uint32_t r = 1; r <= f.J; r++)
            if ((u >> (f.J - r)) & 1u) acc = F::mul(acc, load_fe(challenges + (size_t)(r - 1) * 32));
        const fe_t s = F::from_mont(acc);
        uint32_t carry = 0;
        for (uint32_t w = 0; w < f.nwin; w++) {
            for (uint32_t g = 0; g < f.G; g++) {
                const uint32_t width = fold_width(f, g), half = 1u << (width - 1);
                const uint32_t raw = extract_bits(s.l, w * f.c + g * f.cs, width) + carry;
                uint32_t enc;
                if (raw > half) { uint32_t mag = (1u << width) - raw; carry = 1; enc = mag ? (mag | 0x80000000u) : 0u; }
                else { carry = 0; enc = raw; }
                digits[(size_t)(w * f.G + g) * T + u] = enc;
                if (enc & 0x7fffffffu) atomicAdd(&heads[fold_list(f, g, w % f.WS, enc & 0x7fffffffu)], 1u);
            }
        }
    }
    __syncthreads();
    // exclusive scan of the list lengths: contiguous chunk per thread, 256-wide scan of the chunk sums
    const uint32_t per = (nlists + 1 + 255) / 256, k0 = tid * per, k1 = k0 + per < nlists + 1 ? k0 + per : nlists + 1;
    uint32_t sum = 0;
    for (uint32_t k = k0; k < k1; k++) sum += heads[k];
    chunk_sum[tid] = sum;
    __syncthreads();
    for (uint32_t d = 1; d < 256; d <<= 1) {
        uint32_t v = tid >= d ? chunk_sum[tid - d] : 0u;
        __syncthreads();
        chunk_sum[tid] += v;
        __syncthreads();
    }
    uint32_t run = chunk_sum[tid] - sum;
    for (uint32_t k = k0; k < k1; k++) { uint32_t h = heads[k]; heads[k] = run; offsets[k] = run; run += h; }
    __syncthreads();
    for (uint32_t idx = tid; idx < T * f.nwin * f.G; idx += 256) {
        const uint32_t u = idx % T, wg = idx / T, w = wg / f.G, g = wg % f.G;
        const uint32_t enc = digits[idx], mag = enc & 0x7fffffffu;
        if (!mag) continue;
        const uint32_t pos = atomicAdd(&heads[fold_list(f, g, w % f.WS, mag)], 1u);
        entries[pos] = (enc & 0x80000000u) | (w << 16) | u;
    }
}

// grid (ceil(m / FOLD_THREADS), G * WS): partial[(g * WS + ws) * m + p] = sum_d d * B_d over the list of (g, ws),
// B_d = sum of +-table[w][base + u * m + p] over the list entries of magnitude d
// MINB = resident CTAs per SM the compiler must allow: 4 (128 registers, a few spills) pays when the grid fills the machine
// (9.2 -> 8.5 ms at 2^20), 3 (168 registers, no spills) is faster for the smaller grids (2.67 vs 2.80 ms at 2^18)
template <int CURVE, int MINB>
__global__ void __launch_bounds__(FOLD_THREADS, MINB) k_fold_accumulate(const affine_t *__restrict__ table, FoldShape f,
                                                                   const uint32_t *__restrict__ offsets,
                                                                   const uint32_t *__restrict__ entries,
                                                                   xyzz_t *__restrict__ partial) {
    using Cv = Curve<CURVE>;
    const uint32_t p = blockIdx.x * FOLD_THREADS + threadIdx.x;
    if (p >= f.m) return;
    const uint32_t gw = blockIdx.y, g = gw / f.WS;
    const uint32_t *off = offsets + (size_t)gw * (f.nbk + 1);
    xyzz_t running = Cv::identity(), total = Cv::identity();
#pragma unroll 1
    for (uint32_t d = 1u << (fold_width(f, g) - 1); d >= 1; d--) {
        const uint32_t e1 = __ldg(off + d + 1);
#pragma unroll 1
        for (uint32_t e = __ldg(off + d); e < e1; e++) {
            const uint32_t ent = __ldg(entries + e);
            const uint32_t w = (ent >> 16) & 0x7fffu, u = ent & 0xffffu;
            affine_t pt = load_affine(table + (size_t)w * f.stride + (size_t)u * f.m + p);
            if (ent >> 31) pt.y = Cv::F::neg(pt.y);
            Cv::madd(running, pt);
        }
        Cv::add(total, running);
    }
    store_xyzz(partial + (size_t)gw * f.m + p, total);
}

// one thread per output: FK[p] = sum_g 2^(cs g) sum_ws partial[g][ws][p], normalised; an identity result (possible
// only for keys with a linear relation the challenges hit) is counted in *n_identity and the fold is abandoned
template <int CURVE>
__global__ void __launch_bounds__(FOLD_THREADS) k_fold_combine(const xyzz_t *__restrict__ partial, FoldShape f,
                                                                affine_t *__restrict__ out, uint32_t *__restrict__ n_identity) {
    using Cv = Curve<CURVE, FpCall>;
    const uint32_t p = blockIdx.x * FOLD_THREADS + threadIdx.x;
    if (p >= f.m) return;
    xyzz_t acc = Cv::identity();
#pragma unroll 1
    for (int g = (int)f.G - 1; g >= 0; g--) {
        if (!Cv::is_identity(acc)) {
#pragma unroll 1
            for (uint32_t b = 0; b < f.cs; b++) acc = Cv::dbl(acc);
        }
#pragma unroll 1
        for (uint32_t ws = 0; ws < f.WS; ws++) {
            xyzz_t t = load_xyzz(partial + (size_t)((uint32_t)g * f.WS + ws) * f.m + p);
            Cv::add(acc, t);
        }
    }
    affine_t a; uint32_t inf;
    Cv::template to_affine<true>(acc, a, inf);
    if (inf) atomicAdd(n_identity, 1u);
    store_fe(&out[p].x, a.x); store_fe(&out[p].y, a.y);
}

// Cyclic key layout of one shard of a multi-GPU opening: out[t] = key[offset + (t << log_stride)], read from the
// contiguous point ranges [start[s], start[s] + count[s]) that hold the key (peer pointers over NVLink, or a local copy
// of one range).  Indices that fall in none of the given ranges are left untouched, so one launch per copied range
// fills the layout piece by piece.
constexpr int CYCLIC_MAX_SRC = 16;
struct CyclicSrc {
    const affine_t *xy[CYCLIC_MAX_SRC];
    uint64_t start[CYCLIC_MAX_SRC], count[CYCLIC_MAX_SRC];
    int n_src;
};
__global__ void __launch_bounds__(256) k_cyclic_gather(CyclicSrc src, uint64_t offset, uint32_t log_stride, uint64_t n_out,
                                                        affine_t *__restrict__ out) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_out) return;
    const uint64_t i = offset + (t << log_stride);
    for (int s = 0; s < src.n_src; s++) {
        if (i < src.start[s] || i - src.start[s] >= src.count[s]) continue;
        const uint4 *p = reinterpret_cast<const uint4 *>(src.xy[s] + (i - src.start[s]));
        uint4 *o = reinterpret_cast<uint4 *>(out + t);
        const uint4 a = p[0], b = p[1], c = p[2], d = p[3];
        o[0] = a; o[1] = b; o[2] = c; o[3] = d;
        return;
    }
}

}  // namespace accmsm
