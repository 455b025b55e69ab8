// Host-side 255-bit Montgomery arithmetic on 4 x 64-bit limbs (same memory image as fe_t / ark-ff Fp256), used by the
// library's HOST code for the O(1) field work that sits on a latency-critical path:
//   * the affine conversion of the one (or few) XYZZ sums an entry point returns to the caller -- the device leaves the
//     un-normalised sum, the host thread that receives it does the single inversion (a host core inverts in ~10 us what
//     one GPU thread needs ~50 us for, and nothing else on the device can proceed meanwhile);
//   * the inverse of a round challenge of IpaPC::open (upstream computes `round_challenge.inverse()` on the host too).
// This is not a CPU path of the product: no MSM, vector kernel or point addition runs here.
#pragma once
#include <cstdint>
#include <cstring>

namespace accmsm {
namespace hostfp {

typedef unsigned __int128 u128;

struct Modulus {
    uint64_t m[4];     // modulus, little-endian limbs
    uint64_t ninv;     // -m^-1 mod 2^64
    uint64_t one[4];   // R mod m (Montgomery image of 1)
};

// FIELD 0 = Fp (Pallas base / Vesta scalar), FIELD 1 = Fq (Pallas scalar / Vesta base); SURVEY.md App. B
inline const Modulus &modulus(int field) {
    static const Modulus M[2] = {
        {{0x992d30ed00000001ULL, 0x224698fc094cf91bULL, 0x0ULL, 0x4000000000000000ULL}, 0x992d30ecffffffffULL,
         {0x34786d38fffffffdULL, 0x992c350be41914adULL, 0xffffffffffffffffULL, 0x3fffffffffffffffULL}},
        {{0x8c46eb2100000001ULL, 0x224698fc0994a8ddULL, 0x0ULL, 0x4000000000000000ULL}, 0x8c46eb20ffffffffULL,
         {0x5b2b3e9cfffffffdULL, 0x992c350be3420567ULL, 0xffffffffffffffffULL, 0x3fffffffffffffffULL}},
    };
    return M[field];
}

inline bool is_zero(const uint64_t a[4]) { return (a[0] | a[1] | a[2] | a[3]) == 0; }

// r = a b R^-1 mod m (CIOS); inputs < m, output < m.  r may alias a or b.
inline void mul(const Modulus &M, const uint64_t a[4], const uint64_t b[4], uint64_t r[4]) {
    uint64_t t[6] = {0, 0, 0, 0, 0, 0};
    for (int i = 0; i < 4; i++) {
        u128 c = 0;
        for (int j = 0; j < 4; j++) {
            c += (u128)a[j] * b[i] + t[j];
            t[j] = (uint64_t)c;
            c >>= 64;
        }
        c += t[4];
        t[4] = (uint64_t)c;
        t[5] = (uint64_t)(c >> 64);
        const uint64_t q = t[0] * M.ninv;
        c = (u128)q * M.m[0] + t[0];
        c >>= 64;
        for (int j = 1; j < 4; j++) {
            c += (u128)q * M.m[j] + t[j];
            t[j - 1] = (uint64_t)c;
            c >>= 64;
        }
        c += t[4];
        t[3] = (uint64_t)c;
        t[4] = t[5] + (uint64_t)(c >> 64);
    }
    // conditional subtraction (t < 2 m)
    uint64_t d[4];
    u128 br = 0;
    for (int j = 0; j < 4; j++) {
        u128 x = (u128)t[j] - M.m[j] - (uint64_t)br;
        d[j] = (uint64_t)x;
        br = (x >> 64) & 1;
    }
    const bool ge = t[4] != 0 || br == 0;
    for (int j = 0; j < 4; j++) r[j] = ge ? d[j] : t[j];
}

// r = a + b mod m; inputs < m, output < m (m < 2^255: the sum does not carry out of 256 bits).  r may alias a or b.
inline void add(const Modulus &M, const uint64_t a[4], const uint64_t b[4], uint64_t r[4]) {
    uint64_t s[4], d[4];
    u128 c = 0;
    for (int j = 0; j < 4; j++) { c += (u128)a[j] + b[j]; s[j] = (uint64_t)c; c >>= 64; }
    u128 br = 0;
    for (int j = 0; j < 4; j++) {
        u128 x = (u128)s[j] - M.m[j] - (uint64_t)br;
        d[j] = (uint64_t)x;
        br = (x >> 64) & 1;
    }
    for (int j = 0; j < 4; j++) r[j] = br ? s[j] : d[j];
}

// a^(m - 2) in the Montgomery domain: maps the image a R to a^-1 R; inv(0) = 0.  4-bit fixed windows: 252 squarings + ~70 products.
inline void inv(const Modulus &M, const uint64_t a[4], uint64_t r[4]) {
    uint64_t e[4] = {M.m[0] - 2, M.m[1], M.m[2], M.m[3]};     // m[0] ends in ...01: no borrow
    uint64_t tab[16][4];
    memcpy(tab[0], M.one, 32);
    memcpy(tab[1], a, 32);
    for (int i = 2; i < 16; i++) mul(M, tab[i - 1], a, tab[i]);
    uint64_t acc[4];
    memcpy(acc, M.one, 32);
    bool started = false;
    for (int nib = 63; nib >= 0; nib--) {
        const unsigned w = (unsigned)((e[nib / 16] >> (4 * (nib % 16))) & 0xf);
        if (started) for (int s = 0; s < 4; s++) mul(M, acc, acc, acc);
        if (w) { mul(M, acc, tab[w], acc); started = true; }
    }
    memcpy(r, acc, 32);
}

// XYZZ (X, Y, ZZ, ZZZ; 16 u64) -> affine (x = X / ZZ, y = Y / ZZZ) + infinity flag, for k points with ONE inversion
// (Montgomery's trick over the ZZZ's).  The identity (ZZ == 0) comes back as ark's (0, 1, true).  Same field elements as
// Curve::to_affine on the device: x = X (ZZ / ZZZ)^2, y = Y / ZZZ.
inline void xyzz_to_affine(int field, const uint64_t *raw, size_t k, uint64_t *out_xy, uint8_t *out_inf) {
    const Modulus &M = modulus(field);
    constexpr size_t MAXK = 64;
    uint64_t pref[MAXK][4];
    uint64_t run[4];
    for (size_t base = 0; base < k; base += MAXK) {
        const size_t kk = k - base < MAXK ? k - base : MAXK;
        memcpy(run, M.one, 32);
        for (size_t i = 0; i < kk; i++) {
            const uint64_t *p = raw + 16 * (base + i);
            memcpy(pref[i], run, 32);
            if (!is_zero(p + 8)) mul(M, run, p + 12, run);
        }
        uint64_t invrun[4];
        inv(M, run, invrun);
        for (size_t i = kk; i-- > 0;) {
            const uint64_t *p = raw + 16 * (base + i);
            uint64_t *o = out_xy + 8 * (base + i);
            if (is_zero(p + 8)) {
                memset(o, 0, 32); memcpy(o + 4, M.one, 32); out_inf[base + i] = 1;
                continue;
            }
            uint64_t t[4], zt[4];
            mul(M, invrun, pref[i], t);          // 1 / ZZZ_i
            mul(M, invrun, p + 12, invrun);      // drop ZZZ_i from the running inverse
            mul(M, p + 8, t, zt);                // ZZ / ZZZ = 1 / Z
            mul(M, zt, zt, zt);                  // 1 / ZZ
            mul(M, p, zt, o);
            mul(M, p + 4, t, o + 4);
            out_inf[base + i] = 0;
        }
    }
}

}  // namespace hostfp
}  // namespace accmsm
