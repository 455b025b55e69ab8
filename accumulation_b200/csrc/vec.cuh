// Field-vector kernels around the MSM (K3 materialised, K4, K5 of SURVEY.md 2b).  All are HBM-streaming
// kernels: one 255-bit Montgomery product per 32-byte element read, 128-bit coalesced loads/stores.
// They restate, on the device, loops that the reference runs serially on one core:
//   compute_hp / scale_vector / combine_vectors / compute_t_vecs   src/hp_as/mod.rs:278-349,482-512
//   combine_succinct_check_polynomials, evaluate                   src/ipa_pc_as/mod.rs:391-404,439
//   matrix_vec_mul / inner_prod                                    src/r1cs_nark_as/r1cs_nark/mod.rs:443-462
#pragma once
#include "msm.cuh"

namespace accmsm {

constexpr int VEC_MAX_INPUTS = 16;
struct VecPtrs {
    const uint8_t *ptr[VEC_MAX_INPUTS];
    uint32_t len[VEC_MAX_INPUTS];
};

// h(X) coefficients via two half tables: coeff[j] = hi[j >> L] * lo[j & (2^L - 1)], where lo / hi hold the products
// of the challenges selected by the low L / high k - L index bits.  One product per coefficient instead of ~k/2
// (the element-wise kernel is then bound by its 32-byte store, not by the multiplier); the tables (<= 2 x 2^11 entries
// per polynomial) stay in L1/L2.  alphas (nullable) are folded into the hi tables: hi_i *= alpha_i.
// Cyclic shard form (log_shards > 0): the tables cover only coefficients shard_index + 2^log_shards t, t < 2^(k -
// log_shards), indexed by t.  The low log_shards index bits are then fixed, so the product of their challenges is one
// constant per polynomial, folded into the hi tables like alpha.  (0, 0) is the whole polynomial.
template <int FIELD>
__global__ void __launch_bounds__(256) k_coeff_tables(const uint8_t *__restrict__ challenges, int m, int k, int L,
                                                       const uint8_t *__restrict__ alphas, uint8_t *__restrict__ lo,
                                                       uint8_t *__restrict__ hi, uint32_t log_shards, uint32_t shard_index) {
    using F = Fp<FIELD>;
    const int kl = k - (int)log_shards;
    const uint32_t n_lo = 1u << L, n_hi = 1u << (kl - L), per = n_lo + n_hi;
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= per * (uint32_t)m) return;
    const uint32_t i = t / per, e = t % per;
    const uint8_t *ch = challenges + (size_t)i * k * 32;
    const bool is_lo = e < n_lo;
    const uint32_t idx = is_lo ? e : e - n_lo;
    const int b0 = (int)log_shards + (is_lo ? 0 : L), nb = is_lo ? L : kl - L;
    fe_t acc = (!is_lo && alphas) ? load_fe(alphas + (size_t)i * 32) : F::one();
    if (!is_lo) {
        for (uint32_t b = 0; b < log_shards; b++)
            if ((shard_index >> b) & 1u) acc = F::mul(acc, load_fe(ch + (size_t)(k - 1 - (int)b) * 32));
    }
    for (int b = 0; b < nb; b++) {             // index bit b0 + b  <->  challenge k - 1 - (b0 + b)
        if ((idx >> b) & 1u) acc = F::mul(acc, load_fe(ch + (size_t)(k - 1 - (b0 + b)) * 32));
    }
    store_fe((is_lo ? lo + (size_t)i * n_lo * 32 : hi + (size_t)i * n_hi * 32) + (size_t)idx * 32, acc);
}
// out[j] = random_poly[j] (j < n_random) + sum_i hi_i[j >> L] * lo_i[j & mask]
template <int FIELD>
__global__ void __launch_bounds__(256) k_coeffs_from_tables(const uint8_t *__restrict__ lo, const uint8_t *__restrict__ hi, int m,
                                                             int k, int L, const uint8_t *__restrict__ random_poly,
                                                             uint32_t n_random, uint8_t *__restrict__ out) {
    using F = Fp<FIELD>;
    uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= (1u << k)) return;
    const uint32_t n_lo = 1u << L, n_hi = 1u << (k - L), jl = j & (n_lo - 1u), jh = j >> L;
    fe_t acc = F::mul(load_fe(hi + (size_t)jh * 32), load_fe(lo + (size_t)jl * 32));
    for (int i = 1; i < m; i++)
        acc = F::add(acc, F::mul(load_fe(hi + ((size_t)i * n_hi + jh) * 32), load_fe(lo + ((size_t)i * n_lo + jl) * 32)));
    if (random_poly && j < n_random) acc = F::add(acc, load_fe_nc(random_poly + (size_t)j * 32));
    store_fe(out + (size_t)j * 32, acc);
}

// block-wide sum of one field element per thread (blockDim.x == 256); result valid in thread 0
template <int FIELD> ACC_D fe_t block_sum(fe_t v, fe_t *sh) {
    using F = Fp<FIELD>;
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int d = 128; d >= 1; d >>= 1) {
        if ((int)threadIdx.x < d) sh[threadIdx.x] = F::add(sh[threadIdx.x], sh[threadIdx.x + d]);
        __syncthreads();
    }
    return sh[0];
}

// polynomial evaluation: thread t folds `chunk` coefficients by Horner and scales by z^(t*chunk); chunk = 16 up to 2^20
// coefficients (more threads: latency), 64 beyond (fewer products per coefficient: throughput)
inline uint32_t poly_chunk(size_t n) { return n > (size_t(1) << 20) ? 64u : 16u; }
template <int FIELD>
__global__ void __launch_bounds__(256) k_poly_eval_partial(const uint8_t *__restrict__ coeffs, uint32_t n,
                                                            const uint8_t *__restrict__ z_ptr, uint8_t *__restrict__ partials,
                                                            uint32_t chunk) {
    using F = Fp<FIELD>;
    __shared__ fe_t sh[256];
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    fe_t z = load_fe(z_ptr);
    fe_t term = F::zero();
    uint32_t lo = t * chunk;
    if (lo < n) {
        uint32_t hi = lo + chunk < n ? lo + chunk : n;
        fe_t acc = F::zero();
        for (uint32_t j = hi; j-- > lo;) acc = F::add(F::mul(acc, z), load_fe_nc(coeffs + (size_t)j * 32));
        // z^(t * chunk): zc = z^chunk, then square-and-multiply on t
        fe_t zc = z;
#pragma unroll 1
        for (uint32_t i = 1; i < chunk; i <<= 1) zc = F::sqr(zc);
        fe_t pw = F::one();
        for (uint32_t e = t; e; e >>= 1) {
            if (e & 1u) pw = F::mul(pw, zc);
            zc = F::sqr(zc);
        }
        term = F::mul(acc, pw);
    }
    fe_t s = block_sum<FIELD>(term, sh);
    if (threadIdx.x == 0) store_fe(partials + (size_t)blockIdx.x * 32, s);
}
template <int FIELD>
__global__ void __launch_bounds__(256) k_field_sum(const uint8_t *__restrict__ in, uint32_t n, uint8_t *__restrict__ out) {
    using F = Fp<FIELD>;
    __shared__ fe_t sh[256];
    fe_t acc = F::zero();
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) acc = F::add(acc, load_fe(in + (size_t)i * 32));
    fe_t s = block_sum<FIELD>(acc, sh);
    if (threadIdx.x == 0) store_fe(out, s);
}

template <int FIELD>
__global__ void __launch_bounds__(256) k_hadamard(const uint8_t *__restrict__ a, const uint8_t *__restrict__ b, uint32_t n,
                                                   uint8_t *__restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    store_fe(out + (size_t)i * 32, Fp<FIELD>::mul(load_fe_nc(a + (size_t)i * 32), load_fe_nc(b + (size_t)i * 32)));
}
template <int FIELD>
__global__ void __launch_bounds__(256) k_scale(const uint8_t *__restrict__ v, uint32_t n, const uint8_t *__restrict__ c,
                                                uint8_t *__restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    store_fe(out + (size_t)i * 32, Fp<FIELD>::mul(load_fe_nc(v + (size_t)i * 32), load_fe(c)));
}
// out[li] = h * hiding[li] + sum_ni ch[ni] * vecs[ni][li]   (ragged inputs: missing elements are skipped; h = *hiding_ch, or 1
// when hiding_ch is null)
template <int FIELD>
__global__ void __launch_bounds__(256) k_lincomb(VecPtrs vecs, int m, const uint8_t *__restrict__ ch,
                                                  const uint8_t *__restrict__ hiding, uint32_t n_hiding, uint32_t out_len,
                                                  uint8_t *__restrict__ out, const uint8_t *__restrict__ hiding_ch) {
    using F = Fp<FIELD>;
    uint32_t li = blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= out_len) return;
    fe_t acc = F::zero();
    if (hiding && li < n_hiding) {
        acc = load_fe_nc(hiding + (size_t)li * 32);
        if (hiding_ch) acc = F::mul(acc, load_fe(hiding_ch));
    }
    for (int ni = 0; ni < m; ni++) {
        if (li < vecs.len[ni]) acc = F::add(acc, F::mul(load_fe(ch + (size_t)ni * 32), load_fe_nc(vecs.ptr[ni] + (size_t)li * 32)));
    }
    store_fe(out + (size_t)li * 32, acc);
}

// t-vectors: per position li, T[k] = sum_{i+j=k} A[i] * B'[j] with A[i] = mu_i a_i[li] (+ mu_n ha[li] for i = 0),
// B'[j] = b_{n-1-j}[li] (+ mu_1 hb[li] for j = 0).  A and B' are staged in shared memory ([limb-row][thread]).
constexpr int TVEC_THREADS = 64;
template <int FIELD>
__global__ void __launch_bounds__(TVEC_THREADS) k_tvecs(VecPtrs a, VecPtrs b, int n, const uint8_t *__restrict__ mu, uint32_t len,
                                                         const uint8_t *__restrict__ ha, uint32_t n_ha,
                                                         const uint8_t *__restrict__ hb, uint32_t n_hb,
                                                         uint8_t *__restrict__ out) {
    using F = Fp<FIELD>;
    extern __shared__ uint4 smem_raw[];
    fe_t *A = reinterpret_cast<fe_t *>(smem_raw);                 // [n][TVEC_THREADS]
    fe_t *Bp = A + (size_t)n * TVEC_THREADS;                        // [n][TVEC_THREADS]
    uint32_t li = blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= len) return;
    for (int i = 0; i < n; i++) {
        fe_t av = li < a.len[i] ? F::mul(load_fe(mu + (size_t)i * 32), load_fe_nc(a.ptr[i] + (size_t)li * 32)) : F::zero();
        if (i == 0 && ha && li < n_ha) av = F::add(av, F::mul(load_fe_nc(ha + (size_t)li * 32), load_fe(mu + (size_t)n * 32)));
        A[i * TVEC_THREADS + threadIdx.x] = av;
        int src = n - 1 - i;   // B'[i] = b_{n-1-i}
        fe_t bv = li < b.len[src] ? load_fe_nc(b.ptr[src] + (size_t)li * 32) : F::zero();
        if (i == 0 && hb && li < n_hb) bv = F::add(bv, F::mul(load_fe_nc(hb + (size_t)li * 32), load_fe(mu + 32)));
        Bp[i * TVEC_THREADS + threadIdx.x] = bv;
    }
    for (int k = 0; k < 2 * n - 1; k++) {
        fe_t acc = F::zero();
        int i0 = k - (n - 1) > 0 ? k - (n - 1) : 0, i1 = k < n - 1 ? k : n - 1;
        for (int i = i0; i <= i1; i++) acc = F::add(acc, F::mul(A[i * TVEC_THREADS + threadIdx.x], Bp[(k - i) * TVEC_THREADS + threadIdx.x]));
        store_fe(out + ((size_t)k * len + li) * 32, acc);
    }
}

// zk hiding rows of ASForHadamardProducts::prove (src/hp_as/mod.rs:179-230), straight into the first three rows of a pass's
// scalar buffer (out + j * row_stride): ha, hb, and cross = ha o b_0 + a_{n-1} o hb, the hiding part of the middle t-vector
// (SURVEY.md App. C.3: T[n-1] carries mu_n (ha o b_0 + a_{n-1} o hb) for n >= 2).  b_0 and a_{n-1} are ragged (zero beyond their
// lengths); ha and hb have len elements.
template <int FIELD>
__global__ void __launch_bounds__(256) k_hp_hiding_rows(const uint8_t *__restrict__ ha, const uint8_t *__restrict__ hb,
                                                         const uint8_t *__restrict__ b_first, uint32_t n_b_first,
                                                         const uint8_t *__restrict__ a_last, uint32_t n_a_last, uint32_t len,
                                                         uint8_t *__restrict__ out, size_t row_stride) {
    using F = Fp<FIELD>;
    uint32_t li = blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= len) return;
    const size_t o = (size_t)li * 32;
    const fe_t h_a = load_fe_nc(ha + o), h_b = load_fe_nc(hb + o);
    fe_t cross = F::zero();
    if (li < n_b_first) cross = F::mul(h_a, load_fe_nc(b_first + o));
    if (li < n_a_last) cross = F::add(cross, F::mul(load_fe_nc(a_last + o), h_b));
    store_fe(out + o, h_a);
    store_fe(out + row_stride + o, h_b);
    store_fe(out + 2 * row_stride + o, cross);
}

// CSR sparse mat-vec, up to 3 matrices over the same z = input || witness; one thread per (matrix, row)
struct CsrMats {
    const uint32_t *row_ptr[3];
    const uint32_t *cols[3];
    const uint8_t *coeffs[3];
    uint8_t *out[3];
};
template <int FIELD>
__global__ void __launch_bounds__(256) k_csr_matvec(CsrMats mats, uint32_t n_rows, const uint8_t *__restrict__ input,
                                                     uint32_t n_input, const uint8_t *__restrict__ witness) {
    using F = Fp<FIELD>;
    uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    int mi = blockIdx.y;
    if (r >= n_rows) return;
    const fe_t one = F::one();
    fe_t acc = F::zero();
    uint32_t e0 = mats.row_ptr[mi][r], e1 = mats.row_ptr[mi][r + 1];
    for (uint32_t e = e0; e < e1; e++) {
        uint32_t col = mats.cols[mi][e];
        fe_t z = col < n_input ? load_fe(input + (size_t)col * 32) : load_fe(witness + (size_t)(col - n_input) * 32);
        fe_t cf = load_fe_nc(mats.coeffs[mi] + (size_t)e * 32);
        acc = F::add(acc, F::eq(cf, one) ? z : F::mul(z, cf));   // coeff.is_one() fast path (:459)
    }
    store_fe(mats.out[mi] + (size_t)r * 32, acc);
}

// R1CSNark rows (src/r1cs_nark_as/r1cs_nark/mod.rs:183-261 prove, :335-419 verify; the AS decider
// src/r1cs_nark_as/mod.rs:1031-1112): one thread per constraint row walks row r of A, B and C once.  Every (col, coeff) is
// loaded once and feeds the z-sum over input || witness and, when proving, the r-sum over 0 || r (input columns add nothing
// to it).  The products are formed in registers and every result goes straight to row j of the pass's scalar rows
// (out + j * row_stride):
//   NARK_PROVE:  z_A, z_B, z_C, r_A, r_B, r_C, cross = z_A r_B + z_B r_A, rr = r_A r_B
//   NARK_VERIFY: t_A, t_B, t_C, t_A t_B
//   NARK_DECIDE: t_A, t_B, t_C, a*, b*, a* b*.  The host has uploaded a*[0, n_a) into row 3 and b*[0, n_b) into row 4; the
//                thread reads its entry there (zero at or beyond the length, and stores that zero), so every scalar of the
//                six rows is written before the pass reads it.
enum NarkMode : int { NARK_PROVE, NARK_VERIFY, NARK_DECIDE };
template <int FIELD, int MODE>
__global__ void __launch_bounds__(256) k_nark_rows(CsrMats mats, uint32_t n_rows, const uint8_t *__restrict__ input, uint32_t n_input,
                                                    const uint8_t *__restrict__ witness, const uint8_t *__restrict__ rvec,
                                                    uint8_t *__restrict__ out, size_t row_stride, uint32_t n_a, uint32_t n_b) {
    using F = Fp<FIELD>;
    constexpr bool ZK = MODE == NARK_PROVE;
    uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const fe_t one = F::one();
    fe_t za = F::zero(), zb = F::zero(), ra = F::zero(), rb = F::zero();
#pragma unroll
    for (int mi = 0; mi < 3; mi++) {
        fe_t zs = F::zero(), rs = F::zero();
        const uint32_t e0 = mats.row_ptr[mi][r], e1 = mats.row_ptr[mi][r + 1];
        for (uint32_t e = e0; e < e1; e++) {
            const uint32_t col = mats.cols[mi][e];
            const fe_t cf = load_fe_nc(mats.coeffs[mi] + (size_t)e * 32);
            const bool unit = F::eq(cf, one);          // coeff.is_one() fast path (:459)
            if (col < n_input) {
                const fe_t z = load_fe(input + (size_t)col * 32);
                zs = F::add(zs, unit ? z : F::mul(z, cf));
            } else {
                const size_t w = (size_t)(col - n_input) * 32;
                const fe_t z = load_fe(witness + w);
                zs = F::add(zs, unit ? z : F::mul(z, cf));
                if (ZK) {
                    const fe_t rv = load_fe(rvec + w);
                    rs = F::add(rs, unit ? rv : F::mul(rv, cf));
                }
            }
        }
        store_fe(out + (size_t)mi * row_stride + (size_t)r * 32, zs);
        if (ZK) store_fe(out + (size_t)(3 + mi) * row_stride + (size_t)r * 32, rs);
        if (mi == 0) { za = zs; ra = rs; }
        if (mi == 1) { zb = zs; rb = rs; }
    }
    if (ZK) {
        store_fe(out + (size_t)6 * row_stride + (size_t)r * 32, F::add(F::mul(za, rb), F::mul(zb, ra)));
        store_fe(out + (size_t)7 * row_stride + (size_t)r * 32, F::mul(ra, rb));
    } else if (MODE == NARK_VERIFY) {
        store_fe(out + (size_t)3 * row_stride + (size_t)r * 32, F::mul(za, zb));
    } else {
        uint8_t *pa = out + (size_t)3 * row_stride + (size_t)r * 32, *pb = out + (size_t)4 * row_stride + (size_t)r * 32;
        fe_t a = F::zero(), b = F::zero();
        if (r < n_a) a = load_fe(pa); else store_fe(pa, a);
        if (r < n_b) b = load_fe(pb); else store_fe(pb, b);
        store_fe(out + (size_t)5 * row_stride + (size_t)r * 32, F::mul(a, b));
    }
}

}  // namespace accmsm
