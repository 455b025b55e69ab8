// C++ harness of the zero-knowledge IpaPC opening through accumulation_b200/host/ark_mirror.hpp (InnerProductArgPC::open_zk):
// a zk proof passes the succinct-check group equation with C' = C + alpha hiding_comm - (r + alpha rho) s and the decider's
// final-key check, a corrupted rand or hiding_comm is rejected, and the order errors of the session are reported.  Runs on a
// single-device ctx, or on a device group with ACCMSM_TEST_DEVICES="0,0".  Expected values come from the CPU oracle.
#include <cstdio>
#include <cstdlib>
#include <string>
#include "../../accumulation_b200/host/ark_mirror.hpp"
#include "../../oracle/oracle.h"

using namespace accmsm_host;
static int failures = 0;
#define CHECK(name, cond) do { bool ok_ = (cond); std::printf("%s %s\n", ok_ ? "PASS" : "FAIL", name); if (!ok_) failures++; } while (0)

static std::vector<Fe> gen_scalars(int field, uint64_t seed, size_t n) {
    std::vector<Fe> v(n);
    if (n) oracle_gen_scalars(field, seed, n, 1, v[0].data());
    return v;
}
static std::vector<Affine> gen_points(int curve, uint64_t seed, size_t n) {
    std::vector<uint64_t> xy(n * 8);
    oracle_gen_points(curve, seed, n, xy.data());
    std::vector<Affine> out(n);
    for (size_t i = 0; i < n; i++) out[i] = affine_from(xy.data() + 8 * i, 0);
    return out;
}
static std::vector<uint64_t> flat(const std::vector<Affine> &p) {
    std::vector<uint64_t> xy(p.size() * 8);
    for (size_t i = 0; i < p.size(); i++) affine_to(p[i], xy.data() + 8 * i);
    return xy;
}
static Affine oracle_commit_(int curve, const std::vector<Affine> &gens, const std::vector<Fe> &elems, const Affine *h = nullptr, const Fe *r = nullptr) {
    auto xy = flat(gens); uint64_t hx[8]; if (h) affine_to(*h, hx);
    uint64_t out[8]; uint8_t inf = 0;
    oracle_commit(curve, xy.data(), gens.size(), elems.empty() ? nullptr : elems[0].data(), elems.size(), h ? hx : nullptr, r ? r->data() : nullptr, out, &inf);
    return affine_from(out, inf);
}

int main() {
    std::shared_ptr<Context> ctx;
    try {
        const char *devs = getenv("ACCMSM_TEST_DEVICES");
        if (devs && *devs) {
            std::vector<int> d;
            for (const char *p = devs; *p;) { d.push_back(atoi(p)); while (*p && *p != ',') p++; if (*p == ',') p++; }
            ctx = std::make_shared<Context>(d, 16);
            printf("device group of %d\n", accmsm_device_count(ctx->raw()));
        } else ctx = std::make_shared<Context>(0);
    }
    catch (const AccmsmError &e) { std::printf("NO_GPU %s\n", e.what()); return 3; }   // no CPU fallback: refuse to run

    for (int curve = 0; curve < 2; curve++) {
        const int sf = scalar_field(curve);
        std::string tag = curve == 0 ? "pallas " : "vesta ";
        const int k = 8; const size_t D = size_t(1) << k;
        auto pts = gen_points(curve, 500 + curve, D + 1);
        std::vector<Affine> key(pts.begin(), pts.begin() + D);
        Affine hgen = pts[D];
        auto coeffs = gen_scalars(sf, 9, D);
        Fe z = gen_scalars(sf, 10, 1)[0];
        auto squeeze = [&](const Affine &l, const Affine &r) {
            Fe xi = gen_scalars(sf, l.x[0] ^ (r.x[1] << 1) ^ 0x5eed, 1)[0], inv;
            oracle_fe_inv(sf, xi.data(), inv.data(), 1);
            return std::make_pair(xi, inv);
        };
        {   // zk opening (MakeZK::Enabled): C = commit(P, s, r); C' = C + alpha hiding_comm - (r + alpha rho) s passes succinct_check
            Affine sgen = gen_points(curve, 520 + curve, 1)[0];
            CommitterKey zk_ck(ctx, curve, key, hgen, true, sgen);
            auto hiding = gen_scalars(sf, 16, D - 3);
            Fe rho = gen_scalars(sf, 17, 1)[0], rr = gen_scalars(sf, 18, 1)[0], xi0 = gen_scalars(sf, 15, 1)[0], zero{};
            auto alpha_of = [&](const Affine &hc) { return gen_scalars(sf, hc.x[0] ^ 0xa1fa, 1)[0]; };
            IpaProofCore zp = InnerProductArgPC::open_zk(zk_ck, coeffs, k, z, hiding, rho, alpha_of, [&](const Affine &, const Fe &) { return xi0; },
                                                         [&](const Affine &l, const Affine &r) { return squeeze(l, r).first; });
            Fe t, rand;
            oracle_fe_mul(sf, zp.hiding_alpha.data(), rho.data(), t.data(), 1);
            oracle_fe_add(sf, rr.data(), t.data(), rand.data(), 1);
            const Affine C = oracle_commit_(curve, key, coeffs, &sgen, &rr);
            auto mul = [&](const Affine &p, const Fe &mont) {
                Fe canon; oracle_fe_from_mont(sf, mont.data(), canon.data(), 1);
                uint64_t xy[8], o[8]; uint8_t oi = 0; affine_to(p, xy);
                oracle_point_mul(curve, xy, p.infinity, canon.data(), o, &oi);
                return affine_from(o, oi);
            };
            auto add = [&](const Affine &a, const Affine &b) {
                uint64_t ax[8], bx[8], o[8]; uint8_t oi = 0; affine_to(a, ax); affine_to(b, bx);
                oracle_point_add(curve, ax, a.infinity, bx, b.infinity, o, &oi);
                return affine_from(o, oi);
            };
            auto c_prime = [&](const Affine &hc, const Fe &rnd) { Fe neg; oracle_fe_sub(sf, zero.data(), rnd.data(), neg.data(), 1); return add(add(C, mul(hc, zp.hiding_alpha)), mul(sgen, neg)); };
            const Affine hprime = mul(hgen, xi0);
            Fe vz; oracle_poly_evaluate(sf, coeffs[0].data(), D, z.data(), vz.data());      // the hiding polynomial vanishes at z
            auto succinct = [&](const Affine &cp) {
                auto zlx = flat(zp.l_vec), zrx = flat(zp.r_vec), zcx = flat({cp}), zhx = flat({hprime}), zfx = flat({zp.final_comm_key});
                return oracle_ipa_succinct_check(curve, zcx.data(), cp.infinity, z.data(), vz.data(), zlx.data(), zrx.data(), k, zp.round_challenges[0].data(),
                                                 zhx.data(), zfx.data(), zp.c.data()) == 1;
            };
            CHECK((tag + "ipa zk open: C' from hiding_comm and rand passes succinct_check").c_str(), succinct(c_prime(*zp.hiding_comm, rand)));
            Fe bad_rand = rand; bad_rand[0] ^= 1;
            CHECK((tag + "ipa zk open: a corrupted rand is rejected").c_str(), !succinct(c_prime(*zp.hiding_comm, bad_rand)));
            CHECK((tag + "ipa zk open: a corrupted hiding_comm is rejected").c_str(), !succinct(c_prime(hgen, rand)));
            CHECK((tag + "ipa zk open: check_final_key accepts").c_str(),
                  InnerProductArgPC::check_final_key(zk_ck, SuccinctCheckPolynomial{zp.round_challenges}, zp.final_comm_key));
            // order errors: ACCMSM_E_ARG
            accmsm_ctx *c = ctx->raw();
            uint64_t sess = 0, hc[8], l[8], r[8], fk[8]; uint8_t hi = 0, li = 0, ri = 0; Fe cc;
            ctx->check(accmsm_ipa_open_begin(c, zk_ck.handle(), coeffs[0].data(), D, k, z.data(), nullptr, &sess), "ipa_open_begin");
            bool ok = accmsm_ipa_open_hiding_challenge(c, sess, rho.data()) == ACCMSM_E_ARG;                         // no hide yet
            ok = ok && accmsm_ipa_open_hide(c, sess, hiding[0].data(), D + 1, *zk_ck.s_index(), rho.data(), hc, &hi) == ACCMSM_E_ARG;  // > 2^k
            ok = ok && accmsm_ipa_open_hide(c, sess, hiding[0].data(), hiding.size(), *zk_ck.s_index(), rho.data(), hc, &hi) == ACCMSM_OK;
            ok = ok && accmsm_ipa_open_hide(c, sess, hiding[0].data(), hiding.size(), *zk_ck.s_index(), rho.data(), hc, &hi) == ACCMSM_E_ARG;  // twice
            ok = ok && accmsm_ipa_open_use_hiding_generator(c, sess, zk_ck.hiding_index(), xi0.data()) == ACCMSM_OK;
            ok = ok && accmsm_ipa_open_round(c, sess, l, &li, r, &ri) == ACCMSM_E_ARG;                                 // alpha not applied
            ok = ok && accmsm_ipa_open_hiding_challenge(c, sess, rho.data()) == ACCMSM_OK;
            ok = ok && accmsm_ipa_open_hiding_challenge(c, sess, rho.data()) == ACCMSM_E_ARG;                         // twice
            ok = ok && accmsm_ipa_open_round(c, sess, l, &li, r, &ri) == ACCMSM_OK;
            ok = ok && accmsm_ipa_open_hide(c, sess, hiding[0].data(), hiding.size(), *zk_ck.s_index(), rho.data(), hc, &hi) == ACCMSM_E_ARG;  // after a round
            ok = ok && accmsm_ipa_open_finish(c, sess, fk, cc.data()) == ACCMSM_E_ARG;                                // rounds left: released
            CHECK((tag + "ipa zk open: order errors are reported").c_str(), ok);
        }
    }
    std::printf("%d failure(s)\n", failures);
    return failures ? 1 : 0;
}
