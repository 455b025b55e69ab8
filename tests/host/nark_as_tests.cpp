// C++ harness of the R1CS NARK accumulation decider through accumulation_b200/host/ark_mirror.hpp (r1cs_nark_as::decide):
// an accumulator whose six commitments come from the CPU oracle is accepted with and without randomness, a corrupted w*, a
// swapped C1* / C2* and an r1cs_input of the wrong length are rejected, and hp vectors longer than the rows and an unknown
// csr handle are refused.  Runs on a single-device ctx, or on a device group with ACCMSM_TEST_DEVICES="0,0".
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
static std::vector<Fe> matvec(int field, const r1cs_nark::Matrix &m, const std::vector<Fe> &x, const std::vector<Fe> &w) {
    r1cs_nark::Csr c = r1cs_nark::to_csr(m);
    std::vector<Fe> out(m.size());
    oracle_csr_matvec(field, c.row_ptr.data(), c.cols.data(), c.coeffs.data(), m.size(), x[0].data(), x.size(), w.empty() ? nullptr : w[0].data(),
                      w.size(), out[0].data());
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
        const size_t M = 900, n_in = 4, n_wit = 300;
        auto cf = gen_scalars(sf, 70 + curve, 3 * M);
        uint64_t lcg = 0x2545F4914F6CDD1Dull;
        r1cs_nark::Matrix A(M), B(M), Cm(M);
        for (size_t i = 0; i < M; i++) {
            r1cs_nark::Matrix *mats[3] = {&A, &B, &Cm};
            for (int m = 0; m < 3; m++) for (int e = 0; e < 2; e++) {
                lcg = lcg * 6364136223846793005ull + 1442695040888963407ull;
                (*mats[m])[i].push_back({cf[3 * i + m], (size_t)(lcg >> 33) % (n_in + n_wit)});
            }
        }
        auto x = gen_scalars(sf, 80 + curve, n_in);
        auto w = gen_scalars(sf, 81 + curve, n_wit);
        auto a = gen_scalars(sf, 82 + curve, M), b = gen_scalars(sf, 83 + curve, M - 100);
        auto sg = gen_scalars(sf, 84 + curve, 3), hr = gen_scalars(sf, 85 + curve, 3);

        std::vector<uint64_t> pxy((M + 1) * 8);
        oracle_gen_points(curve, 630 + curve, M + 1, pxy.data());
        std::vector<Affine> gens(M);
        for (size_t i = 0; i < M; i++) gens[i] = affine_from(pxy.data() + 8 * i, 0);
        CommitterKey ck(ctx, curve, gens, affine_from(pxy.data() + 8 * M, 0), true);
        r1cs_nark::IndexMatrices idx(ck, A, B, Cm, n_in);

        // the six commitments from the oracle: Commit(t_M, sigma_M), Commit(a, r1), Commit(b, r2), Commit(a o b, r3)
        std::vector<std::vector<Fe>> vecs;
        for (auto *m : {&A, &B, &Cm}) vecs.push_back(matvec(sf, *m, x, w));
        std::vector<Fe> prod(b.size());
        oracle_hadamard(sf, a[0].data(), b[0].data(), prod[0].data(), b.size());
        vecs.push_back(a); vecs.push_back(b); vecs.push_back(prod);
        auto commit = [&](int j, bool hiding) {
            uint64_t o[8]; uint8_t oi = 0;
            const Fe &r = j < 3 ? sg[j] : hr[j - 3];
            oracle_commit(curve, pxy.data(), vecs[j].size(), vecs[j][0].data(), vecs[j].size(), hiding ? pxy.data() + 8 * M : nullptr,
                          hiding ? r.data() : nullptr, o, &oi);
            return affine_from(o, oi);
        };
        auto records = [&](bool hiding, r1cs_nark_as::AccumulatorInstance *inst, r1cs_nark_as::AccumulatorWitness *wit) {
            inst->r1cs_input = x;
            inst->comm_a = commit(0, hiding); inst->comm_b = commit(1, hiding); inst->comm_c = commit(2, hiding);
            inst->hp_instance = {commit(3, hiding), commit(4, hiding), commit(5, hiding)};
            wit->r1cs_blinded_witness = w;
            wit->hp_witness.a_vec = a; wit->hp_witness.b_vec = b;
            if (hiding) {
                wit->hp_witness.randomness = ASForHadamardProducts::Randomness{hr[0], hr[1], hr[2]};
                wit->randomness = r1cs_nark_as::AccumulatorWitnessRandomness{sg[0], sg[1], sg[2]};
            }
        };
        r1cs_nark_as::AccumulatorInstance inst; r1cs_nark_as::AccumulatorWitness wit;
        records(true, &inst, &wit);
        CHECK((tag + "nark_as decide: the zk accumulator is accepted").c_str(), r1cs_nark_as::decide(idx, inst, wit));
        auto bad_w = wit; bad_w.r1cs_blinded_witness[7][2] ^= 1;
        CHECK((tag + "nark_as decide: a corrupted w* is rejected").c_str(), !r1cs_nark_as::decide(idx, inst, bad_w));
        auto swapped = inst; std::swap(swapped.hp_instance.comm_1, swapped.hp_instance.comm_2);
        CHECK((tag + "nark_as decide: C1* swapped with C2* is rejected").c_str(), !r1cs_nark_as::decide(idx, swapped, wit));
        auto short_x = inst; short_x.r1cs_input.pop_back();
        CHECK((tag + "nark_as decide: an r1cs_input of the wrong length is rejected").c_str(), !r1cs_nark_as::decide(idx, short_x, wit));
        r1cs_nark_as::AccumulatorInstance inst0; r1cs_nark_as::AccumulatorWitness wit0;
        records(false, &inst0, &wit0);
        CHECK((tag + "nark_as decide: the accumulator without randomness is accepted").c_str(),
              r1cs_nark_as::decide(idx, inst0, wit0) && !r1cs_nark_as::decide(idx, inst0, wit));

        // argument errors: hp vectors longer than the rows (ACCMSM_E_ARG), an unknown csr handle (ACCMSM_E_HANDLE)
        uint64_t exp[48] = {0}; uint8_t einf[6] = {0}; int acc = 0;
        auto longer = gen_scalars(sf, 86 + curve, M + 1);
        const bool refused =
            accmsm_nark_as_decide(ctx->raw(), ck.handle(), idx.handle(), x[0].data(), n_in, w[0].data(), n_wit, longer[0].data(), M + 1,
                                  b[0].data(), b.size(), ck.hiding_index(), nullptr, nullptr, exp, einf, &acc, nullptr, nullptr) == ACCMSM_E_ARG &&
            accmsm_nark_as_decide(ctx->raw(), ck.handle(), 0xFFFFFFFFull, x[0].data(), n_in, w[0].data(), n_wit, a[0].data(), M,
                                  b[0].data(), b.size(), ck.hiding_index(), sg[0].data(), hr[0].data(), exp, einf, &acc, nullptr, nullptr) == ACCMSM_E_HANDLE;
        CHECK((tag + "nark_as decide: hp vectors longer than the rows and an unknown csr handle are refused").c_str(), refused);
    }
    std::printf("%d failure(s)\n", failures);
    return failures ? 1 : 0;
}
