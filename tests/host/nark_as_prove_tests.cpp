// C++ harness of the R1CS NARK accumulation prover through accumulation_b200/host/ark_mirror.hpp (r1cs_nark_as::prove): NARK
// proofs of a satisfying system are accumulated with and without zero knowledge, and the new accumulator of one prove is an
// old accumulator of the next; r1cs_nark_as::decide accepts both, and rejects a corrupted w* and the accumulator of a corrupted
// proof.  A beta_of that returns the wrong number of challenges is refused.  Runs on a single-device ctx, or on a device group
// with ACCMSM_TEST_DEVICES="0,0".
#include <cstdio>
#include <cstdlib>
#include <string>
#include "../../accumulation_b200/host/ark_mirror.hpp"
#include "../../oracle/oracle.h"

using namespace accmsm_host;
using HP = ASForHadamardProducts;
static int failures = 0;
#define CHECK(name, cond) do { bool ok_ = (cond); std::printf("%s %s\n", ok_ ? "PASS" : "FAIL", name); if (!ok_) failures++; } while (0)

static std::vector<Fe> gen_scalars(int field, uint64_t seed, size_t n) {
    std::vector<Fe> v(n);
    if (n) oracle_gen_scalars(field, seed, n, 1, v[0].data());
    return v;
}
// stand-in sponge: a small deterministic mix of the absorbed points into 128-bit challenges (Montgomery images < the modulus)
static Fe squeeze(uint64_t tag, const std::vector<Affine> &pts, uint64_t salt) {
    uint64_t h = 0x9E3779B97F4A7C15ull ^ tag ^ (salt * 0xBF58476D1CE4E5B9ull);
    for (const auto &p : pts) for (int i = 0; i < 4; i++) { h = (h ^ p.x[i] ^ (p.y[i] << 1) ^ p.infinity) * 0x94D049BB133111EBull; h ^= h >> 31; }
    return Fe{h | 1, h * 0x2545F4914F6CDD1Dull, 0, 0};
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
        const accmsm::hostfp::Modulus &Mod = accmsm::hostfp::modulus(sf);
        const Fe one{Mod.one[0], Mod.one[1], Mod.one[2], Mod.one[3]};
        const std::string tag = curve == 0 ? "pallas " : "vesta ";
        // a satisfying system: A, B random over input || free witness, C row i = out_i = (A z)_i (B z)_i placed after the free witness
        const size_t M = 1200 + 31 * curve, n_in = 3, n_free = 400;
        auto cf = gen_scalars(sf, 90 + curve, 4 * M);
        uint64_t lcg = 0x2545F4914F6CDD1Dull;
        r1cs_nark::Matrix A(M), B(M), Cm(M);
        for (size_t i = 0; i < M; i++) {
            for (int e = 0; e < 2; e++) {
                lcg = lcg * 6364136223846793005ull + 1442695040888963407ull;
                A[i].push_back({cf[4 * i + e], (size_t)(lcg >> 33) % (n_in + n_free)});
                lcg = lcg * 6364136223846793005ull + 1442695040888963407ull;
                B[i].push_back({cf[4 * i + 2 + e], (size_t)(lcg >> 33) % (n_in + n_free)});
            }
            Cm[i].push_back({one, n_in + n_free + i});
        }
        auto x = gen_scalars(sf, 91 + curve, n_in);
        x[0] = one;
        auto w = gen_scalars(sf, 92 + curve, n_free);
        w.resize(n_free + M);
        const auto za = matvec(sf, A, x, w), zb = matvec(sf, B, x, w);
        for (size_t i = 0; i < M; i++) w[n_free + i] = HP::mul(Mod, za[i], zb[i]);

        std::vector<uint64_t> pxy((M + 1) * 8);
        oracle_gen_points(curve, 650 + curve, M + 1, pxy.data());
        std::vector<Affine> gens(M);
        for (size_t i = 0; i < M; i++) gens[i] = affine_from(pxy.data() + 8 * i, 0);
        CommitterKey ck(ctx, curve, gens, affine_from(pxy.data() + 8 * M, 0), true);
        r1cs_nark::IndexMatrices idx(ck, A, B, Cm, n_in);

        r1cs_nark_as::GammaOf gamma_of = [](const std::vector<Affine> &first) { return squeeze(3, first, 0); };
        for (bool zk : {true, false}) {
            const std::string t = tag + (zk ? "zk " : "plain ");
            uint64_t seed = 1000 + 100 * curve + (zk ? 50 : 0);
            // a NARK proof of (x, wit): the zk first message from the device, w' = w + gamma r, the sigmas on the host
            auto proof_of = [&](const std::vector<Fe> &wit) {
                r1cs_nark_as::FreshInput in;
                in.r1cs_input = x;
                if (!zk) { in.first_msg = idx.matvec_commit(x, wit).second; in.blinded_witness = wit; return in; }
                auto r = gen_scalars(sf, seed++, wit.size()), bl = gen_scalars(sf, seed++, 8);
                std::array<Fe, 8> b8; for (int j = 0; j < 8; j++) b8[j] = bl[j];
                in.first_msg = idx.prove_zk(x, wit, r, b8);
                const Fe g = gamma_of(in.first_msg);
                in.blinded_witness = HP::combine_vectors(*ctx, sf, {&r}, {g}, &wit);
                std::array<Fe, 4> s;
                for (int j = 0; j < 3; j++) s[j] = HP::add(Mod, b8[j], HP::mul(Mod, g, b8[3 + j]));
                s[3] = HP::add(Mod, HP::add(Mod, b8[2], HP::mul(Mod, g, b8[6])), HP::mul(Mod, HP::mul(Mod, g, g), b8[7]));
                in.sigmas = s;
                return in;
            };
            auto randomness = [&]() {
                std::optional<r1cs_nark_as::ProverRandomness> z;
                if (!zk) return z;
                auto sr = gen_scalars(sf, seed++, 3), hr = gen_scalars(sf, seed++, 3);
                z = r1cs_nark_as::ProverRandomness{gen_scalars(sf, seed, n_in), gen_scalars(sf, seed + 1, w.size()), {sr[0], sr[1], sr[2]},
                                                   HP::HidingVecs{gen_scalars(sf, seed + 2, M), gen_scalars(sf, seed + 3, M), {hr[0], hr[1], hr[2]}}};
                seed += 4;
                return z;
            };
            auto sponge = [&](size_t n, size_t extra) {
                HP::MuOf mu_of = [n](const std::optional<std::array<Affine, 3>> &hc) {
                    std::vector<Affine> pts; if (hc) pts.assign(hc->begin(), hc->end());
                    std::vector<Fe> mu;
                    for (size_t i = 1; i < n; i++) mu.push_back(squeeze(1, pts, i));
                    return mu;
                };
                HP::NuOf nu_of = [](const std::vector<Affine> &lo, const std::vector<Affine> &hi) {
                    std::vector<Affine> pts(lo); pts.insert(pts.end(), hi.begin(), hi.end());
                    return squeeze(2, pts, 0);
                };
                r1cs_nark_as::BetaOf beta_of = [n, extra](const HP::InputInstance &hp, const std::optional<std::array<Affine, 3>> &cr) {
                    std::vector<Affine> pts{hp.comm_1, hp.comm_2, hp.comm_3}; if (cr) pts.insert(pts.end(), cr->begin(), cr->end());
                    std::vector<Fe> beta;
                    for (size_t i = 1; i < n + extra; i++) beta.push_back(squeeze(4, pts, i));
                    return beta;
                };
                return std::make_tuple(mu_of, nu_of, beta_of);
            };
            const size_t zx = zk ? 1 : 0;
            // two fresh inputs -> acc1; one fresh input + acc1 -> acc2
            auto [mu2, nu2, beta2] = sponge(2, zx);
            auto out1 = r1cs_nark_as::prove(idx, {proof_of(w), proof_of(w)}, {}, gamma_of, mu2, nu2, beta2, randomness());
            CHECK((t + "two fresh proofs: the new accumulator is accepted").c_str(),
                  r1cs_nark_as::decide(idx, out1.instance, out1.witness) && out1.witness.randomness.has_value() == zk &&
                  out1.proof.randomness_comms.has_value() == zk);
            auto out2 = r1cs_nark_as::prove(idx, {proof_of(w)}, {{out1.instance, out1.witness}}, gamma_of, mu2, nu2, beta2, randomness());
            CHECK((t + "a fresh proof and an old accumulator: the new accumulator is accepted").c_str(),
                  r1cs_nark_as::decide(idx, out2.instance, out2.witness));
            auto bad = out2.witness; bad.r1cs_blinded_witness[9][1] ^= 1;
            CHECK((t + "a corrupted w* is rejected").c_str(), !r1cs_nark_as::decide(idx, out2.instance, bad));
            auto bad_in = proof_of(w); bad_in.blinded_witness[5][0] ^= 1;
            auto out3 = r1cs_nark_as::prove(idx, {bad_in}, {{out1.instance, out1.witness}}, gamma_of, mu2, nu2, beta2, randomness());
            CHECK((t + "the accumulator of a corrupted proof is rejected").c_str(), !r1cs_nark_as::decide(idx, out3.instance, out3.witness));
            auto [mu_, nu_, short_beta] = sponge(2, zx == 1 ? 0 : 1);       // one beta too few with zk, one too many without
            bool refused = false;
            try { r1cs_nark_as::prove(idx, {proof_of(w)}, {{out1.instance, out1.witness}}, gamma_of, mu_, nu_, short_beta, randomness()); }
            catch (const AccmsmError &) { refused = true; }
            auto out4 = r1cs_nark_as::prove(idx, {proof_of(w)}, {{out2.instance, out2.witness}}, gamma_of, mu2, nu2, beta2, randomness());
            CHECK((t + "a wrong beta count is refused and the ctx still proves").c_str(), refused && r1cs_nark_as::decide(idx, out4.instance, out4.witness));
        }
    }
    std::printf("%d failure(s)\n", failures);
    return failures ? 1 : 0;
}
