// C++ harness of the R1CS NARK prove (zk) and verify through accumulation_b200/host/ark_mirror.hpp
// (r1cs_nark::IndexMatrices::{prove_zk, verify}): the zk first message equals the oracle's 8 commitments, the proof (w' and
// the sigmas formed on the host, the left-hand sides from one batched MSM) verifies and a corrupted w' is rejected, the
// non-zk proof verifies, and a prove without blinders is refused.  Runs on a single-device ctx, or on a device group with
// ACCMSM_TEST_DEVICES="0,0".  Expected values come from the CPU oracle.
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
static std::vector<Fe> matvec(int field, const r1cs_nark::Matrix &m, const std::vector<Fe> &x, const std::vector<Fe> &w) {
    r1cs_nark::Csr c = r1cs_nark::to_csr(m);
    std::vector<Fe> out(m.size());
    oracle_csr_matvec(field, c.row_ptr.data(), c.cols.data(), c.coeffs.data(), m.size(), x[0].data(), x.size(), w.empty() ? nullptr : w[0].data(),
                      w.size(), out[0].data());
    return out;
}
static std::vector<Fe> fe_op(void (*op)(int, const uint64_t *, const uint64_t *, uint64_t *, size_t), int field, const std::vector<Fe> &a,
                             const std::vector<Fe> &b) {
    std::vector<Fe> out(a.size());
    op(field, a[0].data(), b[0].data(), out[0].data(), a.size());
    return out;
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
        const std::string tag = curve == 0 ? "pallas " : "vesta ";
        // a satisfying system: A, B over input || free witness, C row i = 1 * out_i with out_i = (A z)_i (B z)_i
        const size_t M = 700, n_in = 3, n_free = 200, n_wit = n_free + M;
        Fe one{}; { uint64_t c1[4] = {1, 0, 0, 0}; oracle_fe_to_mont(sf, c1, one.data(), 1); }
        auto cf = gen_scalars(sf, 40 + curve, 4 * M);
        uint64_t lcg = 0x9E3779B97F4A7C15ull;
        r1cs_nark::Matrix A(M), B(M), Cm(M);
        for (size_t i = 0; i < M; i++) {
            for (int e = 0; e < 2; e++) {
                lcg = lcg * 6364136223846793005ull + 1442695040888963407ull; A[i].push_back({e ? cf[4 * i] : one, (size_t)(lcg >> 33) % (n_in + n_free)});
                lcg = lcg * 6364136223846793005ull + 1442695040888963407ull; B[i].push_back({cf[4 * i + 1 + e], (size_t)(lcg >> 33) % (n_in + n_free)});
            }
            Cm[i].push_back({one, n_in + n_free + i});
        }
        auto input = gen_scalars(sf, 50 + curve, n_in);
        input[0] = one;
        auto witness = gen_scalars(sf, 51 + curve, n_free);
        witness.resize(n_wit);
        auto out = fe_op(oracle_hadamard, sf, matvec(sf, A, input, witness), matvec(sf, B, input, witness));
        std::copy(out.begin(), out.end(), witness.begin() + n_free);

        auto pts = gen_points(curve, 530 + curve, M + 1);
        std::vector<Affine> gens(pts.begin(), pts.begin() + M);
        CommitterKey ck(ctx, curve, gens, pts[M], true);
        r1cs_nark::IndexMatrices idx(ck, A, B, Cm);
        auto r = gen_scalars(sf, 60 + curve, n_wit);
        auto bl = gen_scalars(sf, 61 + curve, 8);
        std::array<Fe, 8> blinders; std::copy(bl.begin(), bl.end(), blinders.begin());

        // oracle first message
        std::vector<Fe> zero_in(n_in);
        std::vector<std::vector<Fe>> vecs;
        for (auto *m : {&A, &B, &Cm}) vecs.push_back(matvec(sf, *m, input, witness));
        for (auto *m : {&A, &B, &Cm}) vecs.push_back(matvec(sf, *m, zero_in, r));
        vecs.push_back(fe_op(oracle_fe_add, sf, fe_op(oracle_hadamard, sf, vecs[0], vecs[4]), fe_op(oracle_hadamard, sf, vecs[1], vecs[3])));
        vecs.push_back(fe_op(oracle_hadamard, sf, vecs[3], vecs[4]));
        std::vector<uint64_t> gxy(M * 8), hxy(8);
        for (size_t i = 0; i < M; i++) affine_to(gens[i], gxy.data() + 8 * i);
        affine_to(pts[M], hxy.data());
        bool same = true;
        const std::vector<Affine> first = idx.prove_zk(input, witness, r, blinders);
        for (int j = 0; j < 8; j++) {
            uint64_t o[8]; uint8_t oi = 0;
            oracle_commit(curve, gxy.data(), M, vecs[j][0].data(), M, hxy.data(), bl[j].data(), o, &oi);
            same = same && first[j] == affine_from(o, oi);
        }
        CHECK((tag + "nark prove_zk: the 8 commitments equal the oracle's").c_str(), same);

        // second message: gamma from the first, w' = w + gamma r on the device, the sigmas on the host
        const Fe gamma = gen_scalars(sf, first[0].x[0] ^ first[7].x[1] ^ 0x9a33a, 1)[0];
        std::vector<Fe> ch{gamma};
        auto w_prime = ASForHadamardProducts::combine_vectors(*ctx, sf, {&r}, ch, &witness);
        auto gm = [&](const Fe &a, const Fe &b) { Fe o; oracle_fe_mul(sf, a.data(), b.data(), o.data(), 1); return o; };
        auto ad = [&](const Fe &a, const Fe &b) { Fe o; oracle_fe_add(sf, a.data(), b.data(), o.data(), 1); return o; };
        const Fe g2 = gm(gamma, gamma);
        std::array<Fe, 4> sig = {ad(bl[0], gm(gamma, bl[3])), ad(bl[1], gm(gamma, bl[4])), ad(bl[2], gm(gamma, bl[5])),
                                 ad(ad(bl[2], gm(gamma, bl[6])), gm(g2, bl[7]))};
        // left-hand sides: one batched MSM of 4 equations x 3 terms (canonical scalars; (identity, 0) pads the 2-term ones)
        Fe gc, g2c, c1{}, c0{};
        oracle_fe_from_mont(sf, gamma.data(), gc.data(), 1); oracle_fe_from_mont(sf, g2.data(), g2c.data(), 1); c1[0] = 1;
        Affine ident = first[0]; ident.infinity = true;
        std::vector<std::vector<Affine>> eb;
        std::vector<std::vector<Fe>> es;
        for (int i = 0; i < 3; i++) { eb.push_back({first[i], first[3 + i], ident}); es.push_back({c1, gc, c0}); }
        eb.push_back({first[2], first[6], first[7]}); es.push_back({c1, gc, g2c});
        auto lhs = VariableBaseMSM::multi_scalar_mul_batch(*ctx, curve, eb, es);
        std::array<Affine, 4> expected = {lhs[0], lhs[1], lhs[2], lhs[3]};
        std::vector<std::vector<Fe>> t;
        CHECK((tag + "nark verify: the zk proof is accepted").c_str(), idx.verify(input, w_prime, expected, sig, &t));
        bool t_ok = t.size() == 3;
        for (int m = 0; m < 3 && t_ok; m++) t_ok = t[m] == matvec(sf, *std::array<const r1cs_nark::Matrix *, 3>{&A, &B, &Cm}[m], input, w_prime);
        CHECK((tag + "nark verify: t_A, t_B, t_C equal the oracle's").c_str(), t_ok);
        auto bad = w_prime; bad[5][1] ^= 1;
        CHECK((tag + "nark verify: a corrupted w' is rejected").c_str(), !idx.verify(input, bad, expected, sig));

        // without zk: matvec_commit's three commitments, w itself
        auto plain = idx.matvec_commit(input, witness);
        std::array<Affine, 4> exp0 = {plain.second[0], plain.second[1], plain.second[2], plain.second[2]};
        CHECK((tag + "nark verify: the non-zk proof is accepted").c_str(), idx.verify(input, witness, exp0) && !idx.verify(input, w_prime, exp0));

        // argument errors: no blinders (ACCMSM_E_ARG), an unknown csr handle (ACCMSM_E_HANDLE)
        uint64_t xy[64]; uint8_t inf[8];
        const bool refused =
            accmsm_nark_prove_zk(ctx->raw(), ck.handle(), idx.handle(), input[0].data(), n_in, witness[0].data(), n_wit, r[0].data(),
                                 ck.hiding_index(), nullptr, nullptr, xy, inf) == ACCMSM_E_ARG &&
            accmsm_nark_prove_zk(ctx->raw(), ck.handle(), 0xFFFFFFFFull, input[0].data(), n_in, witness[0].data(), n_wit, r[0].data(),
                                 ck.hiding_index(), bl[0].data(), nullptr, xy, inf) == ACCMSM_E_HANDLE;
        CHECK((tag + "nark prove_zk: missing blinders and an unknown csr handle are refused").c_str(), refused);
    }
    std::printf("%d failure(s)\n", failures);
    return failures ? 1 : 0;
}
