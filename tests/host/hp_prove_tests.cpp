// C++ harness of the Hadamard-product accumulation prover through accumulation_b200/host/ark_mirror.hpp
// (ASForHadamardProducts::prove / verify / decide): inputs whose instances come from the CPU oracle are accumulated with and
// without zero knowledge, the new accumulator passes verify and decide, and a corrupted a*, a challenge the verifier does not
// share, swapped low / high commitments and a corrupted input are rejected.  Runs on a single-device ctx, or on a device group
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
        const size_t L = 1500 + 77 * curve;
        std::vector<uint64_t> pxy((L + 1) * 8);
        oracle_gen_points(curve, 640 + curve, L + 1, pxy.data());
        std::vector<Affine> gens(L);
        for (size_t i = 0; i < L; i++) gens[i] = affine_from(pxy.data() + 8 * i, 0);
        CommitterKey ck(ctx, curve, gens, affine_from(pxy.data() + 8 * L, 0), true);
        auto commit = [&](const std::vector<Fe> &v, const Fe *r) {
            uint64_t o[8]; uint8_t oi = 0;
            oracle_commit(curve, pxy.data(), v.size(), v.empty() ? nullptr : v[0].data(), v.size(), r ? pxy.data() + 8 * L : nullptr,
                          r ? r->data() : nullptr, o, &oi);
            return affine_from(o, oi);
        };
        for (bool zk : {true, false}) {
            const std::string t = tag + (zk ? "zk " : "plain ");
            const size_t n = 3;
            std::vector<HP::InputWitness> wits;
            std::vector<HP::InputInstance> insts;
            for (size_t i = 0; i < n; i++) {
                HP::InputWitness w;
                w.a_vec = gen_scalars(sf, 700 + 10 * i + curve, L - 40 * i);
                w.b_vec = gen_scalars(sf, 701 + 10 * i + curve, i == 0 ? L : L - 13 * i);
                std::vector<Fe> prod(std::min(w.a_vec.size(), w.b_vec.size()));
                oracle_hadamard(sf, w.a_vec[0].data(), w.b_vec[0].data(), prod[0].data(), prod.size());
                if (zk) { auto r = gen_scalars(sf, 702 + 10 * i + curve, 3); w.randomness = HP::Randomness{r[0], r[1], r[2]}; }
                const HP::Randomness *r = w.randomness ? &*w.randomness : nullptr;
                insts.push_back({commit(w.a_vec, r ? &r->rand_1 : nullptr), commit(w.b_vec, r ? &r->rand_2 : nullptr), commit(prod, r ? &r->rand_3 : nullptr)});
                wits.push_back(w);
            }
            std::optional<HP::HidingVecs> hz;
            if (zk) { auto r = gen_scalars(sf, 790 + curve, 3); hz = HP::HidingVecs{gen_scalars(sf, 791 + curve, L), gen_scalars(sf, 792 + curve, L), {r[0], r[1], r[2]}}; }
            HP::MuOf mu_of = [&](const std::optional<std::array<Affine, 3>> &hc) {
                std::vector<Affine> pts; if (hc) pts.assign(hc->begin(), hc->end());
                std::vector<Fe> mu;
                for (size_t i = 1; i < n; i++) mu.push_back(squeeze(1, pts, i));
                return mu;
            };
            HP::NuOf nu_of = [&](const std::vector<Affine> &lo, const std::vector<Affine> &hi) {
                std::vector<Affine> pts(lo); pts.insert(pts.end(), hi.begin(), hi.end());
                return squeeze(2, pts, 0);
            };
            HP::ProveOutput out = HP::prove(ck, wits, insts, mu_of, nu_of, hz);
            CHECK((t + "prove -> verify accepts").c_str(), HP::verify(ck, insts, out.instance, out.proof, mu_of, nu_of));
            CHECK((t + "prove -> decide accepts").c_str(), HP::decide(ck, out.instance, out.witness) && out.witness.randomness.has_value() == zk);
            auto bad = out.witness; bad.a_vec[5][1] ^= 1;
            CHECK((t + "a corrupted a* is rejected").c_str(), !HP::decide(ck, out.instance, bad));
            HP::NuOf other_nu = [&](const std::vector<Affine> &lo, const std::vector<Affine> &hi) { Fe v = nu_of(lo, hi); v[0] ^= 4; return v; };
            CHECK((t + "a nu the verifier does not share is rejected").c_str(), !HP::verify(ck, insts, out.instance, out.proof, mu_of, other_nu));
            auto swapped = out.proof; std::swap(swapped.low, swapped.high);
            CHECK((t + "low / high swapped is rejected").c_str(), !HP::verify(ck, insts, out.instance, swapped, mu_of, nu_of));
            auto bad_in = wits; bad_in[1].b_vec[3][0] ^= 1;
            HP::ProveOutput out2 = HP::prove(ck, bad_in, insts, mu_of, nu_of, hz);
            CHECK((t + "a corrupted input is rejected").c_str(),
                  !(HP::verify(ck, insts, out2.instance, out2.proof, mu_of, nu_of) && HP::decide(ck, out2.instance, out2.witness)));
        }
    }
    std::printf("%d failure(s)\n", failures);
    return failures ? 1 : 0;
}
