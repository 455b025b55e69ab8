// C++ host side above the C-ABI (include/accmsm.h): a mirror of the interface through which
// arkworks-rs/accumulation reaches its hot path, with the reference's names, argument meaning and error
// behaviour, so that compiled callers (and the Rust `[patch]` of ark-poly-commit, INTEGRATION.md) have a
// one-to-one template.  The reference is Rust; this image has no cargo, hence C++ (DESIGN.md 1).
//
//   reference (ark-poly-commit / ark-accumulation)                     here
//   trivial_pc::CommitterKey{generators, hiding_generator}             accmsm_host::CommitterKey
//   trivial_pc::PedersenCommitment::commit(ck, elems, randomizer)      PedersenCommitment::commit
//   ipa_pc::InnerProductArgPC::cm_commit / check (final key) / open    InnerProductArgPC::{cm_commit, check_final_key, open}
//   ipa_pc::SuccinctCheckPolynomial(Vec<F>)::compute_coeffs            SuccinctCheckPolynomial::compute_coeffs
//   hp_as: compute_hp, compute_t_vecs, combine_vectors, scale_vector,  ASForHadamardProducts::...
//          compute_product_poly_comm, prove, verify, decide   (src/hp_as/mod.rs:278-512, 646-925)
//   r1cs_nark: Matrix<F> = Vec<Vec<(F, usize)>>, matrix_vec_mul,       r1cs_nark::{Matrix, matrix_vec_mul, IndexMatrices}
//              R1CSNark::prove (zk first message) / verify             IndexMatrices::{matvec_commit, prove_zk, verify}
//                                        (src/r1cs_nark_as/r1cs_nark/mod.rs:183-419, 443-462)
//   r1cs_nark_as: AccumulatorInstance, AccumulatorWitness, decide       r1cs_nark_as::{AccumulatorInstance, AccumulatorWitness, decide}
//                                        (src/r1cs_nark_as/data_structures.rs:156-227, src/r1cs_nark_as/mod.rs:1031-1112)
// Every call computes on the GPU; there is no CPU path.  ark's commit is infallible -> failures throw AccmsmError
// (the Rust wrapper panics / maps to PCError at the same places).
#pragma once
#include <array>
#include <cstdint>
#include <cstring>
#include <functional>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../../include/accmsm.h"
#include "../csrc/hostfp.hpp"

namespace accmsm_host {

using Fe = std::array<uint64_t, 4>;          // Fp256 Montgomery image, little-endian limbs (ark-ff memory image)
struct Affine {                               // ark_ec::short_weierstrass_jacobian::GroupAffine
    Fe x{}, y{};
    bool infinity = false;
    bool operator==(const Affine &o) const {  // GroupAffine's PartialEq
        if (infinity || o.infinity) return infinity == o.infinity;
        return x == o.x && y == o.y;
    }
    bool operator!=(const Affine &o) const { return !(*this == o); }
};
enum Curve { PALLAS = 0, VESTA = 1 };
inline int scalar_field(int curve) { return curve == PALLAS ? 1 : 0; }

struct AccmsmError : std::runtime_error { using std::runtime_error::runtime_error; };

class Context {
public:
    explicit Context(int device = 0) {
        int rc = accmsm_init(&ctx_, device);
        if (rc) throw AccmsmError(std::string("accmsm_init: ") + accmsm_strerror(rc) + " (a CUDA device is required; there is no CPU path)");
    }
    // a group of GPUs behind the same calls (accmsm_init_multi): keys are sharded by point range inside the library
    explicit Context(const std::vector<int> &devices, size_t min_shard = size_t(1) << 16) {
        int rc = accmsm_init_multi(&ctx_, devices.data(), (int)devices.size());
        if (rc) throw AccmsmError(std::string("accmsm_init_multi: ") + accmsm_strerror(rc) + " (a CUDA device is required; there is no CPU path)");
        accmsm_set_min_shard(ctx_, min_shard);
    }
    ~Context() { accmsm_destroy(ctx_); }
    Context(const Context &) = delete;
    Context &operator=(const Context &) = delete;
    accmsm_ctx *raw() const { return ctx_; }
    void check(int rc, const char *what) const {
        if (rc) throw AccmsmError(std::string(what) + ": " + accmsm_strerror(rc) + " (" + accmsm_last_error(ctx_) + ")");
    }
private:
    accmsm_ctx *ctx_ = nullptr;
};

// trivial_pc::CommitterKey / the comm_key part of ipa_pc::CommitterKey.  The hiding generator is registered as
// the base after the last generator, so commit(elems, Some(r)) is one pass of the device MSM.
class CommitterKey {
public:
    // s (ipa_pc::CommitterKey::s, needs the hiding generator h): registered after h, so a zk opening's hiding_comm is one pass
    CommitterKey(std::shared_ptr<Context> ctx, int curve, const std::vector<Affine> &generators,
                 const std::optional<Affine> &hiding_generator = std::nullopt, bool precompute = true,
                 const std::optional<Affine> &s = std::nullopt)
        : ctx_(std::move(ctx)), curve_(curve), n_(generators.size()), has_hiding_(hiding_generator.has_value()), has_s_(s.has_value()) {
        if (s && !hiding_generator) throw AccmsmError("CommitterKey: s follows the hiding generator h; pass both");
        std::vector<uint64_t> xy;
        std::vector<uint8_t> inf;
        xy.reserve((n_ + 1) * 8);
        auto push = [&](const Affine &g) {
            xy.insert(xy.end(), g.x.begin(), g.x.end());
            xy.insert(xy.end(), g.y.begin(), g.y.end());
            inf.push_back(g.infinity ? 1 : 0);
        };
        for (const auto &g : generators) push(g);
        if (hiding_generator) push(*hiding_generator);
        if (s) push(*s);
        ctx_->check(accmsm_register_bases(ctx_->raw(), curve, xy.data(), inf.data(), inf.size(), &handle_), "register_bases");
        if (precompute) ctx_->check(accmsm_precompute_bases(ctx_->raw(), handle_, 0), "precompute_bases");
    }
    ~CommitterKey() { accmsm_release_bases(ctx_->raw(), handle_); }
    CommitterKey(const CommitterKey &) = delete;
    CommitterKey &operator=(const CommitterKey &) = delete;
    size_t supported_num_elems() const { return n_; }          // src/hp_as/mod.rs:129,681
    int curve() const { return curve_; }
    uint64_t handle() const { return handle_; }
    size_t hiding_index() const { return n_; }
    bool has_hiding() const { return has_hiding_; }
    std::optional<size_t> s_index() const { return has_s_ ? std::optional<size_t>(n_ + 1) : std::nullopt; }
    const std::shared_ptr<Context> &ctx() const { return ctx_; }
private:
    std::shared_ptr<Context> ctx_;
    int curve_;
    size_t n_;
    bool has_hiding_, has_s_;
    uint64_t handle_ = 0;
};

inline Affine affine_from(const uint64_t xy[8], uint8_t inf) {
    Affine a;
    std::memcpy(a.x.data(), xy, 32); std::memcpy(a.y.data(), xy + 4, 32);
    a.infinity = inf != 0;
    return a;
}
inline void affine_to(const Affine &a, uint64_t xy[8]) { std::memcpy(xy, a.x.data(), 32); std::memcpy(xy + 4, a.y.data(), 32); }

struct PedersenCommitment {
    // PedersenCommitment::commit(ck, elems, randomizer) -> G  (src/hp_as/mod.rs:196; ark-ec truncates to min(len))
    static Affine commit(const CommitterKey &ck, const std::vector<Fe> &elems, const std::optional<Fe> &randomizer = std::nullopt) {
        if (randomizer && !ck.has_hiding()) throw AccmsmError("commit: the key has no hiding generator");
        size_t n = std::min(elems.size(), ck.supported_num_elems());
        uint64_t xy[8]; uint8_t inf = 0;
        ck.ctx()->check(accmsm_commit(ck.ctx()->raw(), ck.handle(), n, n ? elems[0].data() : nullptr, ck.hiding_index(),
                                      randomizer ? randomizer->data() : nullptr, xy, &inf), "commit");
        return affine_from(xy, inf);
    }
    // several vectors of equal length over one key in shared passes (hp_as::decide, NARK prove)
    static std::vector<Affine> commit_batch(const CommitterKey &ck, const std::vector<std::vector<Fe>> &vecs) {
        std::vector<Affine> out;
        if (vecs.empty()) return out;
        size_t n = std::min(vecs[0].size(), ck.supported_num_elems());
        std::vector<uint64_t> flat(vecs.size() * n * 4), xy(vecs.size() * 8);
        std::vector<uint8_t> inf(vecs.size());
        for (size_t j = 0; j < vecs.size(); j++) {
            if (vecs[j].size() < n) throw AccmsmError("commit_batch: vectors of different length");
            if (n) std::memcpy(flat.data() + j * n * 4, vecs[j][0].data(), n * 32);
        }
        ck.ctx()->check(accmsm_msm_batch(ck.ctx()->raw(), ck.handle(), 0, n, vecs.size(), flat.data(), 1, xy.data(), inf.data()), "msm_batch");
        for (size_t j = 0; j < vecs.size(); j++) out.push_back(affine_from(xy.data() + 8 * j, inf[j]));
        return out;
    }
};

// ipa_pc::SuccinctCheckPolynomial(pub Vec<F>)  (src/ipa_pc_as/mod.rs:245,400,418)
struct SuccinctCheckPolynomial {
    std::vector<Fe> challenges;   // .0, xi_1 first
    std::vector<Fe> compute_coeffs(const Context &ctx, int field) const {
        std::vector<Fe> out(size_t(1) << challenges.size());
        ctx.check(accmsm_compute_coeffs(ctx.raw(), field, challenges.empty() ? nullptr : challenges[0].data(), (int)challenges.size(),
                                        out[0].data()), "compute_coeffs");
        return out;
    }
};

struct IpaProofCore {             // the fields of ipa_pc::Proof produced by the opening loop
    std::vector<Affine> l_vec, r_vec;
    Affine final_comm_key;
    Fe c{};
    std::vector<Fe> round_challenges;
    std::optional<Affine> hiding_comm;   // zk opening: the proof's hiding_comm, and the alpha squeezed from it (rand = r + alpha rho
    Fe hiding_alpha{};                   // and C' = C + alpha hiding_comm - rand s stay with the caller, as upstream)
};

struct InnerProductArgPC {
    static Affine cm_commit(const CommitterKey &comm_key, const std::vector<Fe> &scalars, const std::optional<Fe> &randomizer = std::nullopt) {
        return PedersenCommitment::commit(comm_key, scalars, randomizer);
    }
    // tail of check_individual_opening_challenges (AS decide, src/ipa_pc_as/mod.rs:836-845):
    // final_key = cm_commit(vk.comm_key, h.compute_coeffs());  Ok(final_key == proof.final_comm_key)
    static bool check_final_key(const CommitterKey &vk, const SuccinctCheckPolynomial &h, const Affine &final_comm_key) {
        uint64_t exp[8], xy[8]; uint8_t inf = 0; int accept = 0;
        affine_to(final_comm_key, exp);
        vk.ctx()->check(accmsm_ipa_check_final_key(vk.ctx()->raw(), vk.handle(), h.challenges.empty() ? nullptr : h.challenges[0].data(),
                                                   (int)h.challenges.size(), exp, final_comm_key.infinity, &accept, xy, &inf), "ipa_check_final_key");
        return accept != 0;
    }
    // the opening loop of open_individual_opening_challenges (src/ipa_pc_as/mod.rs:454-462); the caller is the host
    // transcript: round_challenge(l, r) -> (xi, xi^-1)
    // h' = xi_0 * h: pass the point h_prime, or (faster) xi_0 when h is the hiding generator registered with `ck`
    static IpaProofCore open(const CommitterKey &ck, const std::vector<Fe> &combined_coeffs, int log_d, const Fe &point,
                             const Affine &h_prime, const std::function<std::pair<Fe, Fe>(const Affine &, const Affine &)> &round_challenge,
                             const std::optional<Fe> &xi0 = std::nullopt) {
        uint64_t hp[8]; affine_to(h_prime, hp);
        uint64_t sess = 0;
        if (xi0 && !ck.has_hiding()) throw AccmsmError("open: the key has no hiding generator");
        ck.ctx()->check(accmsm_ipa_open_begin(ck.ctx()->raw(), ck.handle(), combined_coeffs.empty() ? nullptr : combined_coeffs[0].data(),
                                              combined_coeffs.size(), log_d, point.data(), xi0 ? nullptr : hp, &sess), "ipa_open_begin");
        if (xi0) ck.ctx()->check(accmsm_ipa_open_use_hiding_generator(ck.ctx()->raw(), sess, ck.hiding_index(), xi0->data()), "ipa_open_use_hiding_generator");
        IpaProofCore p;
        for (int r = 0; r < log_d; r++) {
            uint64_t l[8], rr[8]; uint8_t li = 0, ri = 0;
            ck.ctx()->check(accmsm_ipa_open_round(ck.ctx()->raw(), sess, l, &li, rr, &ri), "ipa_open_round");
            p.l_vec.push_back(affine_from(l, li)); p.r_vec.push_back(affine_from(rr, ri));
            auto xi = round_challenge(p.l_vec.back(), p.r_vec.back());
            ck.ctx()->check(accmsm_ipa_open_fold(ck.ctx()->raw(), sess, xi.first.data(), xi.second.data()), "ipa_open_fold");
            p.round_challenges.push_back(xi.first);
        }
        uint64_t fk[8];
        ck.ctx()->check(accmsm_ipa_open_finish(ck.ctx()->raw(), sess, fk, p.c.data()), "ipa_open_finish");
        p.final_comm_key = affine_from(fk, 0);
        return p;
    }
    // The same loop with ONE library call per round (accmsm_ipa_open_fold_round: fold with the challenge squeezed from the
    // previous (l, r) -- its inverse is computed inside the library, on the host, like upstream's round_challenge.inverse() --
    // and run the next round): what the patched open_individual_opening_challenges uses.  round_challenge(l, r) -> xi.
    static IpaProofCore open_one_call_per_round(const CommitterKey &ck, const std::vector<Fe> &combined_coeffs, int log_d, const Fe &point,
                                                const Affine &h_prime, const std::function<Fe(const Affine &, const Affine &)> &round_challenge,
                                                const std::optional<Fe> &xi0 = std::nullopt) {
        uint64_t hp[8]; affine_to(h_prime, hp);
        uint64_t sess = 0;
        if (xi0 && !ck.has_hiding()) throw AccmsmError("open: the key has no hiding generator");
        ck.ctx()->check(accmsm_ipa_open_begin(ck.ctx()->raw(), ck.handle(), combined_coeffs.empty() ? nullptr : combined_coeffs[0].data(),
                                              combined_coeffs.size(), log_d, point.data(), xi0 ? nullptr : hp, &sess), "ipa_open_begin");
        if (xi0) ck.ctx()->check(accmsm_ipa_open_use_hiding_generator(ck.ctx()->raw(), sess, ck.hiding_index(), xi0->data()), "ipa_open_use_hiding_generator");
        IpaProofCore p;
        uint64_t l[8], rr[8]; uint8_t li = 0, ri = 0; int done = log_d == 0;
        if (!done) ck.ctx()->check(accmsm_ipa_open_round(ck.ctx()->raw(), sess, l, &li, rr, &ri), "ipa_open_round");
        while (!done) {
            p.l_vec.push_back(affine_from(l, li)); p.r_vec.push_back(affine_from(rr, ri));
            Fe xi = round_challenge(p.l_vec.back(), p.r_vec.back());
            p.round_challenges.push_back(xi);
            ck.ctx()->check(accmsm_ipa_open_fold_round(ck.ctx()->raw(), sess, xi.data(), l, &li, rr, &ri, &done), "ipa_open_fold_round");
        }
        uint64_t fk[8];
        ck.ctx()->check(accmsm_ipa_open_finish(ck.ctx()->raw(), sess, fk, p.c.data()), "ipa_open_finish");
        p.final_comm_key = affine_from(fk, 0);
        return p;
    }
    // zk form (MakeZK::Enabled): before the first round the random polynomial `hiding` (<= 2^log_d coefficients from the caller's
    // rng) is shifted on the device to vanish at the point and committed with (s, rho); alpha_of(hiding_comm) is the host sponge
    // over (C, z, v, hiding_comm); xi0_of(hiding_comm, alpha) returns xi_0, which the caller squeezes from C'.  h' = xi_0 * h.
    static IpaProofCore open_zk(const CommitterKey &ck, const std::vector<Fe> &combined_coeffs, int log_d, const Fe &point,
                                const std::vector<Fe> &hiding, const Fe &rho, const std::function<Fe(const Affine &)> &alpha_of,
                                const std::function<Fe(const Affine &, const Fe &)> &xi0_of,
                                const std::function<Fe(const Affine &, const Affine &)> &round_challenge) {
        if (!ck.s_index()) throw AccmsmError("open_zk: the key has no s (CommitterKey(.., s))");
        uint64_t sess = 0;
        accmsm_ctx *c = ck.ctx()->raw();
        ck.ctx()->check(accmsm_ipa_open_begin(c, ck.handle(), combined_coeffs.empty() ? nullptr : combined_coeffs[0].data(),
                                              combined_coeffs.size(), log_d, point.data(), nullptr, &sess), "ipa_open_begin");
        IpaProofCore p;
        uint64_t fk[8], xy[8]; uint8_t inf = 0;
        try {
            ck.ctx()->check(accmsm_ipa_open_hide(c, sess, hiding.empty() ? nullptr : hiding[0].data(), hiding.size(), *ck.s_index(), rho.data(),
                                                 xy, &inf), "ipa_open_hide");
            p.hiding_comm = affine_from(xy, inf);
            p.hiding_alpha = alpha_of(*p.hiding_comm);
            ck.ctx()->check(accmsm_ipa_open_hiding_challenge(c, sess, p.hiding_alpha.data()), "ipa_open_hiding_challenge");
            const Fe xi0 = xi0_of(*p.hiding_comm, p.hiding_alpha);
            ck.ctx()->check(accmsm_ipa_open_use_hiding_generator(c, sess, ck.hiding_index(), xi0.data()), "ipa_open_use_hiding_generator");
        } catch (...) {
            accmsm_ipa_open_finish(c, sess, fk, p.c.data());      // releases the session
            throw;
        }
        uint64_t l[8], rr[8]; uint8_t li = 0, ri = 0; int done = log_d == 0;
        if (!done) ck.ctx()->check(accmsm_ipa_open_round(c, sess, l, &li, rr, &ri), "ipa_open_round");
        while (!done) {
            p.l_vec.push_back(affine_from(l, li)); p.r_vec.push_back(affine_from(rr, ri));
            Fe xi = round_challenge(p.l_vec.back(), p.r_vec.back());
            p.round_challenges.push_back(xi);
            ck.ctx()->check(accmsm_ipa_open_fold_round(c, sess, xi.data(), l, &li, rr, &ri, &done), "ipa_open_fold_round");
        }
        ck.ctx()->check(accmsm_ipa_open_finish(c, sess, fk, p.c.data()), "ipa_open_finish");
        p.final_comm_key = affine_from(fk, 0);
        return p;
    }
};

// ark_ec::msm::VariableBaseMSM::multi_scalar_mul(&bases, &scalars).into_affine() on bases that are NOT a registered key: the short
// linear combinations of commitments (src/hp_as/mod.rs:391-406, src/ipa_pc_as/mod.rs:322-343) and the 2k + 3 term group equation of
// IpaPC::succinct_check (:198-205).  Scalars are BigInteger256 images (canonical, `into_repr()` done by the caller, as upstream).
struct VariableBaseMSM {
    static Affine multi_scalar_mul(const Context &ctx, int curve, const std::vector<Affine> &bases, const std::vector<Fe> &scalars_canonical) {
        const size_t n = std::min(bases.size(), scalars_canonical.size());      // ark-ec truncates to the shorter slice
        std::vector<uint64_t> xy(n * 8); std::vector<uint8_t> inf(n);
        for (size_t i = 0; i < n; i++) { affine_to(bases[i], xy.data() + 8 * i); inf[i] = bases[i].infinity; }
        uint64_t out[8]; uint8_t oi = 0;
        ctx.check(accmsm_msm_oneshot(ctx.raw(), curve, xy.data(), inf.data(), n ? scalars_canonical[0].data() : nullptr, 0, n, out, &oi), "msm_oneshot");
        return affine_from(out, oi);
    }
    // m such MSMs of equal length in shared passes (the succinct checks of all inputs and accumulators of one prove / verify)
    static std::vector<Affine> multi_scalar_mul_batch(const Context &ctx, int curve, const std::vector<std::vector<Affine>> &bases,
                                                      const std::vector<std::vector<Fe>> &scalars_canonical) {
        const size_t m = std::min(bases.size(), scalars_canonical.size());
        size_t n = m ? SIZE_MAX : 0;
        for (size_t j = 0; j < m; j++) n = std::min(n, std::min(bases[j].size(), scalars_canonical[j].size()));
        std::vector<uint64_t> xy(m * n * 8), sc(m * n * 4); std::vector<uint8_t> inf(m * n);
        for (size_t j = 0; j < m; j++) for (size_t i = 0; i < n; i++) {
            affine_to(bases[j][i], xy.data() + 8 * (j * n + i)); inf[j * n + i] = bases[j][i].infinity;
            std::copy(scalars_canonical[j][i].begin(), scalars_canonical[j][i].end(), sc.begin() + 4 * (j * n + i));
        }
        std::vector<uint64_t> out(m * 8); std::vector<uint8_t> oi(m);
        ctx.check(accmsm_msm_oneshot_batch(ctx.raw(), curve, xy.data(), inf.data(), sc.data(), 0, n, m, out.data(), oi.data()), "msm_oneshot_batch");
        std::vector<Affine> res(m);
        for (size_t j = 0; j < m; j++) res[j] = affine_from(out.data() + 8 * j, oi[j]);
        return res;
    }
};

struct ASForHadamardProducts {
    struct InputInstance { Affine comm_1, comm_2, comm_3; };                       // src/hp_as/data_structures.rs:14-23
    struct Randomness { Fe rand_1, rand_2, rand_3; };
    struct InputWitness { std::vector<Fe> a_vec, b_vec; std::optional<Randomness> randomness; };   // :54-63

    static std::vector<Fe> compute_hp(const Context &ctx, int field, const std::vector<Fe> &a, const std::vector<Fe> &b) {   // :278-285
        size_t n = std::min(a.size(), b.size());
        std::vector<Fe> out(n);
        if (n) ctx.check(accmsm_vec_hadamard(ctx.raw(), field, a[0].data(), b[0].data(), n, out[0].data()), "vec_hadamard");
        return out;
    }
    static std::vector<Fe> scale_vector(const Context &ctx, int field, const std::vector<Fe> &v, const Fe &coeff) {          // :482-489
        std::vector<Fe> out(v.size());
        if (!v.empty()) ctx.check(accmsm_vec_scale(ctx.raw(), field, v[0].data(), v.size(), coeff.data(), out[0].data()), "vec_scale");
        return out;
    }
    static std::vector<Fe> combine_vectors(const Context &ctx, int field, const std::vector<const std::vector<Fe> *> &vectors,
                                           const std::vector<Fe> &challenges, const std::vector<Fe> *hiding_vec = nullptr) { // :492-512
        std::vector<const uint64_t *> ptrs; std::vector<size_t> lens; size_t cap = hiding_vec ? hiding_vec->size() : 0;
        for (auto *v : vectors) { ptrs.push_back(v->empty() ? nullptr : (*v)[0].data()); lens.push_back(v->size()); cap = std::max(cap, v->size()); }
        std::vector<Fe> out(cap);
        size_t olen = 0;
        ctx.check(accmsm_vec_lincomb(ctx.raw(), field, ptrs.data(), lens.data(), (int)vectors.size(), challenges.empty() ? nullptr : challenges[0].data(),
                                     hiding_vec && !hiding_vec->empty() ? (*hiding_vec)[0].data() : nullptr, hiding_vec ? hiding_vec->size() : 0,
                                     cap ? out[0].data() : nullptr, cap, &olen), "vec_lincomb");
        out.resize(olen);
        return out;
    }
    // decide (:894-925): one fused device call
    static bool decide(const CommitterKey &ck, const InputInstance &instance, const InputWitness &witness) {
        size_t n = std::min({witness.a_vec.size(), witness.b_vec.size(), ck.supported_num_elems()});
        uint64_t exp[24]; uint8_t einf[3] = {instance.comm_1.infinity, instance.comm_2.infinity, instance.comm_3.infinity};
        affine_to(instance.comm_1, exp); affine_to(instance.comm_2, exp + 8); affine_to(instance.comm_3, exp + 16);
        uint64_t r[12];
        if (witness.randomness) {
            if (!ck.has_hiding()) throw AccmsmError("decide: the key has no hiding generator");
            std::memcpy(r, witness.randomness->rand_1.data(), 32); std::memcpy(r + 4, witness.randomness->rand_2.data(), 32);
            std::memcpy(r + 8, witness.randomness->rand_3.data(), 32);
        }
        int accept = 0;
        ck.ctx()->check(accmsm_hp_decide(ck.ctx()->raw(), ck.handle(), n ? witness.a_vec[0].data() : nullptr, n ? witness.b_vec[0].data() : nullptr, n,
                                         ck.hiding_index(), witness.randomness ? r : nullptr, exp, einf, &accept, nullptr, nullptr), "hp_decide");
        return accept != 0;
    }

    // prove (:646-813) over the already padded pairs, inputs first, then old accumulators (the placeholder padding of :676-710
    // stays with the caller).  The sponge is the callables: mu_of(hiding_comms) -> mu_1 .. mu_{n-1}, nu_of(low, high) -> nu.
    // One device session (accmsm_hp_prove_*) forms the hiding commitments, the product-polynomial commitments and a*, b*; the
    // randomness (App. C.5) is host arithmetic and the new instance (C.6) one 3-equation batched MSM, as upstream.
    struct Proof { std::optional<std::array<Affine, 3>> hiding_comms; std::vector<Affine> low, high; };   // src/hp_as/data_structures.rs
    struct HidingVecs { std::vector<Fe> a_vec, b_vec; Randomness randomness; };                           // hp_vec_len elements each
    using MuOf = std::function<std::vector<Fe>(const std::optional<std::array<Affine, 3>> &)>;
    using NuOf = std::function<Fe(const std::vector<Affine> &, const std::vector<Affine> &)>;
    struct ProveOutput { InputInstance instance; InputWitness witness; Proof proof; };
    static ProveOutput prove(const CommitterKey &ck, const std::vector<InputWitness> &witnesses, const std::vector<InputInstance> &instances,
                             const MuOf &mu_of, const NuOf &nu_of, const std::optional<HidingVecs> &zk = std::nullopt) {
        const size_t n = witnesses.size(), L = ck.supported_num_elems();
        const accmsm::hostfp::Modulus &M = accmsm::hostfp::modulus(scalar_field(ck.curve()));
        if (zk && !ck.has_hiding()) throw AccmsmError("prove: the key has no hiding generator");
        if (instances.size() != n) throw AccmsmError("prove: one instance per witness");
        std::vector<const uint64_t *> ap, bp; std::vector<size_t> al, bl;
        for (const auto &w : witnesses) {
            al.push_back(std::min(w.a_vec.size(), L)); ap.push_back(al.back() ? w.a_vec[0].data() : nullptr);
            bl.push_back(std::min(w.b_vec.size(), L)); bp.push_back(bl.back() ? w.b_vec[0].data() : nullptr);
        }
        accmsm_ctx *c = ck.ctx()->raw();
        uint64_t hr[12], hxy[24], sess = 0; uint8_t hinf[3] = {0, 0, 0};
        std::vector<Fe> ha, hb;
        if (zk) {
            ha = zk->a_vec; hb = zk->b_vec;
            ha.resize(L); hb.resize(L);        // hp_vec_len elements (zero padded)
            std::memcpy(hr, zk->randomness.rand_1.data(), 32); std::memcpy(hr + 4, zk->randomness.rand_2.data(), 32);
            std::memcpy(hr + 8, zk->randomness.rand_3.data(), 32);
        }
        const std::vector<Fe> zero(1);
        ck.ctx()->check(accmsm_hp_prove_begin(c, ck.handle(), ap.data(), al.data(), bp.data(), bl.data(), (int)n, L,
                                              zk ? (L ? ha[0].data() : zero[0].data()) : nullptr, zk ? (L ? hb[0].data() : zero[0].data()) : nullptr,
                                              ck.hiding_index(), zk ? hr : nullptr, hxy, hinf, &sess), "hp_prove_begin");
        ProveOutput out;
        std::vector<Fe> mu(1, Fe{M.one[0], M.one[1], M.one[2], M.one[3]});
        try {
            if (zk) out.proof.hiding_comms = std::array<Affine, 3>{affine_from(hxy, hinf[0]), affine_from(hxy + 8, hinf[1]), affine_from(hxy + 16, hinf[2])};
            const std::vector<Fe> mus = mu_of(out.proof.hiding_comms);
            if (mus.size() + 1 != n) throw AccmsmError("prove: mu_of must return n - 1 challenges");
            mu.insert(mu.end(), mus.begin(), mus.end());
            if (zk) { Fe mn; accmsm::hostfp::mul(M, mu[1].data(), mu[n - 1].data(), mn.data()); mu.push_back(mn); }
            std::vector<uint64_t> lo(8 * n), hi(8 * n); std::vector<uint8_t> li(n), hinf2(n);
            ck.ctx()->check(accmsm_hp_prove_product_poly_comm(c, sess, mu[0].data(), mu.size(), lo.data(), li.data(), hi.data(), hinf2.data()),
                            "hp_prove_product_poly_comm");
            for (size_t j = 0; j + 1 < n; j++) { out.proof.low.push_back(affine_from(&lo[8 * j], li[j])); out.proof.high.push_back(affine_from(&hi[8 * j], hinf2[j])); }
        } catch (...) {
            accmsm_hp_prove_abort(c, sess);
            throw;
        }
        const Fe nu = nu_of(out.proof.low, out.proof.high);
        std::vector<Fe> a_star(L), b_star(L);
        size_t olen[2] = {0, 0};
        ck.ctx()->check(accmsm_hp_prove_finish(c, sess, nu.data(), L ? a_star[0].data() : nullptr, L ? b_star[0].data() : nullptr, L, olen),
                        "hp_prove_finish");
        a_star.resize(olen[0]); b_star.resize(olen[1]);
        out.witness.a_vec = std::move(a_star); out.witness.b_vec = std::move(b_star);
        const std::vector<Fe> nus = powers(M, nu, 2 * n - 1);
        if (zk) {       // App. C.5; absent randomness entries add nothing
            Fe r1 = mul(M, mu[n], zk->randomness.rand_1), r2 = mul(M, mu[1], zk->randomness.rand_2), r3 = mul(M, mu[n], zk->randomness.rand_3);
            for (size_t i = 0; i < n; i++) {
                if (const auto &r = witnesses[i].randomness) {
                    r1 = add(M, r1, mul(M, mul(M, mu[i], nus[i]), r->rand_1));
                    r3 = add(M, r3, mul(M, mu[i], r->rand_3));
                }
                if (const auto &r = witnesses[n - 1 - i].randomness) r2 = add(M, r2, mul(M, nus[i], r->rand_2));
            }
            out.witness.randomness = Randomness{r1, r2, mul(M, r3, nus[n - 1])};
        }
        out.instance = combined_commitments(ck, instances, out.proof, mu, nu);
        return out;
    }
    // verify (:815-892): mu and nu from the same sponge, C1*, C2*, C3* recomputed from the old instances and the proof; accept iff
    // they equal new_instance.  A proof whose shape does not fit n is rejected.
    static bool verify(const CommitterKey &ck, const std::vector<InputInstance> &instances, const InputInstance &new_instance, const Proof &proof,
                       const MuOf &mu_of, const NuOf &nu_of) {
        const size_t n = instances.size();
        const accmsm::hostfp::Modulus &M = accmsm::hostfp::modulus(scalar_field(ck.curve()));
        if (n < 1 || proof.low.size() != n - 1 || proof.high.size() != n - 1) return false;
        std::vector<Fe> mu(1, Fe{M.one[0], M.one[1], M.one[2], M.one[3]});
        const std::vector<Fe> mus = mu_of(proof.hiding_comms);
        if (mus.size() + 1 != n) return false;
        mu.insert(mu.end(), mus.begin(), mus.end());
        if (proof.hiding_comms) { if (n < 2) return false; mu.push_back(mul(M, mu[1], mu[n - 1])); }
        const InputInstance got = combined_commitments(ck, instances, proof, mu, nu_of(proof.low, proof.high));
        return got.comm_1 == new_instance.comm_1 && got.comm_2 == new_instance.comm_2 && got.comm_3 == new_instance.comm_3;
    }
    // compute_combined_hp_commitments (:409-479, App. C.6): C1* = [mu_n H1] + sum_i mu_i nu^i C1_i, C2* = [mu_1 H2] + sum_j nu^j C2_{n-1-j},
    // C3* = sum_j nu^j low_j + sum_j nu^(n+j) high_j + nu^(n-1) ([mu_n H3] + sum_i mu_i C3_i), one batched MSM of 3 equations
    static InputInstance combined_commitments(const CommitterKey &ck, const std::vector<InputInstance> &instances, const Proof &proof,
                                              const std::vector<Fe> &mu, const Fe &nu) {
        const size_t n = instances.size();
        const accmsm::hostfp::Modulus &M = accmsm::hostfp::modulus(scalar_field(ck.curve()));
        const std::vector<Fe> nus = powers(M, nu, 2 * n - 1);
        std::vector<std::vector<Affine>> pts(3);
        std::vector<std::vector<Fe>> sc(3);
        auto term = [&](int e, const Affine &p, const Fe &s) { pts[e].push_back(p); sc[e].push_back(canonical(M, s)); };
        for (size_t i = 0; i < n; i++) {
            term(0, instances[i].comm_1, mul(M, mu[i], nus[i]));
            term(1, instances[n - 1 - i].comm_2, nus[i]);
            term(2, instances[i].comm_3, mul(M, mu[i], nus[n - 1]));
        }
        for (size_t j = 0; j + 1 < n; j++) { term(2, proof.low[j], nus[j]); term(2, proof.high[j], nus[n + j]); }
        if (proof.hiding_comms) {
            term(0, (*proof.hiding_comms)[0], mu[n]);
            term(1, (*proof.hiding_comms)[1], mu[1]);
            term(2, (*proof.hiding_comms)[2], mul(M, mu[n], nus[n - 1]));
        }
        size_t width = 0;
        for (const auto &e : pts) width = std::max(width, e.size());
        for (int e = 0; e < 3; e++) while (pts[e].size() < width) {     // (a point flagged as the identity, 0)
            Affine p = pts[e][0]; p.infinity = true;
            pts[e].push_back(p); sc[e].push_back(Fe{});
        }
        const std::vector<Affine> r = VariableBaseMSM::multi_scalar_mul_batch(*ck.ctx(), ck.curve(), pts, sc);
        return InputInstance{r[0], r[1], r[2]};
    }
private:
    static Fe mul(const accmsm::hostfp::Modulus &M, const Fe &a, const Fe &b) { Fe r; accmsm::hostfp::mul(M, a.data(), b.data(), r.data()); return r; }
    static Fe add(const accmsm::hostfp::Modulus &M, const Fe &a, const Fe &b) { Fe r; accmsm::hostfp::add(M, a.data(), b.data(), r.data()); return r; }
    static Fe canonical(const accmsm::hostfp::Modulus &M, const Fe &a) { const Fe one{1, 0, 0, 0}; return mul(M, a, one); }   // a R * 1 * R^-1
    static std::vector<Fe> powers(const accmsm::hostfp::Modulus &M, const Fe &x, size_t k) {
        std::vector<Fe> p(k);
        if (k) p[0] = Fe{M.one[0], M.one[1], M.one[2], M.one[3]};
        for (size_t j = 1; j < k; j++) p[j] = mul(M, p[j - 1], x);
        return p;
    }
};

namespace r1cs_nark {
// ark_relations::r1cs::Matrix<F> = Vec<Vec<(F, usize)>>  (src/r1cs_nark_as/r1cs_nark/data_structures.rs:17-29)
using Matrix = std::vector<std::vector<std::pair<Fe, size_t>>>;

struct Csr { std::vector<uint32_t> row_ptr, cols; std::vector<uint64_t> coeffs; };
inline Csr to_csr(const Matrix &m) {
    Csr c; c.row_ptr.push_back(0);
    for (const auto &row : m) {
        for (const auto &e : row) { c.cols.push_back((uint32_t)e.second); c.coeffs.insert(c.coeffs.end(), e.first.begin(), e.first.end()); }
        c.row_ptr.push_back((uint32_t)c.cols.size());
    }
    return c;
}
// matrix_vec_mul(matrix, input, witness) for A, B, C at once (src/r1cs_nark_as/r1cs_nark/mod.rs:443-447)
inline std::vector<std::vector<Fe>> matrix_vec_mul(const Context &ctx, int field, const std::vector<const Matrix *> &mats,
                                                   const std::vector<Fe> &input, const std::vector<Fe> &witness) {
    std::vector<Csr> csr; for (auto *m : mats) csr.push_back(to_csr(*m));
    size_t n_rows = mats.empty() ? 0 : mats[0]->size();
    std::vector<std::vector<Fe>> out(mats.size(), std::vector<Fe>(n_rows));
    std::vector<const uint32_t *> rp, cl; std::vector<const uint64_t *> cf; std::vector<uint64_t *> op;
    for (size_t i = 0; i < mats.size(); i++) { rp.push_back(csr[i].row_ptr.data()); cl.push_back(csr[i].cols.data()); cf.push_back(csr[i].coeffs.data()); op.push_back(n_rows ? out[i][0].data() : nullptr); }
    if (n_rows) ctx.check(accmsm_csr_matvec(ctx.raw(), field, (int)mats.size(), rp.data(), cl.data(), cf.data(), n_rows, input.empty() ? nullptr : input[0].data(),
                                            input.size(), witness.empty() ? nullptr : witness[0].data(), witness.size(), op.data()), "csr_matvec");
    return out;
}
// IndexProverKey{a, b, c, ck} with the matrices resident on the device (registered at index time)
class IndexMatrices {
public:
    // num_instance_variables: the index's input length (IndexInfo), which r1cs_nark_as::decide checks r1cs_input against
    IndexMatrices(const CommitterKey &ck, const Matrix &a, const Matrix &b, const Matrix &c,
                  std::optional<size_t> num_instance_variables = std::nullopt)
        : ck_(ck), n_rows_(a.size()), num_instance_variables_(num_instance_variables) {
        Csr ca = to_csr(a), cb = to_csr(b), cc = to_csr(c);
        const uint32_t *rp[3] = {ca.row_ptr.data(), cb.row_ptr.data(), cc.row_ptr.data()};
        const uint32_t *cl[3] = {ca.cols.data(), cb.cols.data(), cc.cols.data()};
        const uint64_t *cf[3] = {ca.coeffs.data(), cb.coeffs.data(), cc.coeffs.data()};
        ck.ctx()->check(accmsm_register_csr(ck.ctx()->raw(), scalar_field(ck.curve()), 3, rp, cl, cf, n_rows_, &handle_), "register_csr");
    }
    ~IndexMatrices() { accmsm_release_csr(ck_.ctx()->raw(), handle_); }
    uint64_t handle() const { return handle_; }
    const CommitterKey &ck() const { return ck_; }
    std::optional<size_t> num_instance_variables() const { return num_instance_variables_; }
    // z_M = M (input || witness), comm_M = Commit(z_M, blinder_M)   (prove :183-185 + :216-218; decide src/r1cs_nark_as/mod.rs:1052-1097)
    std::pair<std::vector<std::vector<Fe>>, std::vector<Affine>> matvec_commit(const std::vector<Fe> &input, const std::vector<Fe> &witness,
                                                                              const std::optional<std::array<Fe, 3>> &blinders = std::nullopt) const {
        std::vector<std::vector<Fe>> vecs(3, std::vector<Fe>(n_rows_));
        uint64_t *op[3] = {vecs[0][0].data(), vecs[1][0].data(), vecs[2][0].data()};
        uint64_t xy[24]; uint8_t inf[3]; uint64_t bl[12];
        if (blinders) for (int m = 0; m < 3; m++) std::memcpy(bl + 4 * m, (*blinders)[m].data(), 32);
        ck_.ctx()->check(accmsm_csr_matvec_commit(ck_.ctx()->raw(), ck_.handle(), handle_, input.empty() ? nullptr : input[0].data(), input.size(),
                                                  witness.empty() ? nullptr : witness[0].data(), witness.size(), ck_.hiding_index(),
                                                  blinders ? bl : nullptr, op, xy, inf), "csr_matvec_commit");
        std::vector<Affine> comms;
        for (int m = 0; m < 3; m++) comms.push_back(affine_from(xy + 8 * m, inf[m]));
        return {vecs, comms};
    }
    // zk prove first message (prove :183-261): Commit(z_M, blinder_M), Commit(r_M, rblinder_M), Commit(cross, blinder_1),
    // Commit(rr, blinder_2) with z_M = M (input || witness), r_M = M (0 || r), in ONE library call (one vector launch, one
    // pass).  blinders and the result in the order A, B, C, rA, rB, rC, 1, 2.  The caller squeezes gamma from the result,
    // forms w' = w + gamma r (ASForHadamardProducts::combine_vectors) and the sigmas, as upstream.
    std::vector<Affine> prove_zk(const std::vector<Fe> &input, const std::vector<Fe> &witness, const std::vector<Fe> &r,
                                 const std::array<Fe, 8> &blinders) const {
        if (!ck_.has_hiding()) throw AccmsmError("prove_zk: the key has no hiding generator");
        if (r.size() != witness.size()) throw AccmsmError("prove_zk: r must be as long as the witness");
        uint64_t xy[64]; uint8_t inf[8];
        ck_.ctx()->check(accmsm_nark_prove_zk(ck_.ctx()->raw(), ck_.handle(), handle_, input.empty() ? nullptr : input[0].data(), input.size(),
                                              witness.empty() ? nullptr : witness[0].data(), witness.size(), r.empty() ? nullptr : r[0].data(),
                                              ck_.hiding_index(), blinders[0].data(), nullptr, xy, inf), "nark_prove_zk");
        std::vector<Affine> first;
        for (int j = 0; j < 8; j++) first.push_back(affine_from(xy + 8 * j, inf[j]));
        return first;
    }
    // verify (:335-419): accept iff Commit(t_M, sigma_M) == expected[M] and Commit(t_A o t_B, sigma_o) == expected[3], with
    // t_M = M (input || blinded_witness), in ONE library call.  expected: comm_M + gamma comm_rM and comm_C + gamma comm_1 +
    // gamma^2 comm_2, or without zk (sigmas = nullopt) comm_A, comm_B, comm_C, comm_C.  t_vecs (nullable) receives t_A, t_B, t_C.
    bool verify(const std::vector<Fe> &input, const std::vector<Fe> &blinded_witness, const std::array<Affine, 4> &expected,
                const std::optional<std::array<Fe, 4>> &sigmas = std::nullopt, std::vector<std::vector<Fe>> *t_vecs = nullptr) const {
        uint64_t exp[32]; uint8_t einf[4];
        for (int j = 0; j < 4; j++) { affine_to(expected[j], exp + 8 * j); einf[j] = expected[j].infinity; }
        uint64_t *op[3] = {nullptr, nullptr, nullptr};
        if (t_vecs) {
            t_vecs->assign(3, std::vector<Fe>(n_rows_));
            if (n_rows_) for (int m = 0; m < 3; m++) op[m] = (*t_vecs)[m][0].data();
        }
        int accept = 0;
        ck_.ctx()->check(accmsm_nark_verify(ck_.ctx()->raw(), ck_.handle(), handle_, input.empty() ? nullptr : input[0].data(), input.size(),
                                            blinded_witness.empty() ? nullptr : blinded_witness[0].data(), blinded_witness.size(),
                                            ck_.hiding_index(), sigmas ? (*sigmas)[0].data() : nullptr, exp, einf, &accept, nullptr, nullptr,
                                            t_vecs ? op : nullptr), "nark_verify");
        return accept != 0;
    }
private:
    const CommitterKey &ck_;
    size_t n_rows_;
    std::optional<size_t> num_instance_variables_;
    uint64_t handle_ = 0;
};
}  // namespace r1cs_nark

namespace r1cs_nark_as {
// src/r1cs_nark_as/data_structures.rs:156-171, :218-227
struct AccumulatorInstance {
    std::vector<Fe> r1cs_input;
    Affine comm_a, comm_b, comm_c;
    ASForHadamardProducts::InputInstance hp_instance;
};
struct AccumulatorWitnessRandomness { Fe sigma_a, sigma_b, sigma_c; };
struct AccumulatorWitness {
    std::vector<Fe> r1cs_blinded_witness;
    ASForHadamardProducts::InputWitness hp_witness;
    std::optional<AccumulatorWitnessRandomness> randomness;
};
// ASForR1CSNark::decide (src/r1cs_nark_as/mod.rs:1031-1112): t_M = M (r1cs_input || r1cs_blinded_witness); accept iff
// Commit(t_M, sigma_M) == comm_M for M = A, B, C and hp_as::decide(ck, hp_instance, hp_witness), in ONE library call (one
// vector launch, the six commitments in one pass).  An r1cs_input whose length differs from the index's is rejected here.
inline bool decide(const r1cs_nark::IndexMatrices &index, const AccumulatorInstance &instance, const AccumulatorWitness &witness) {
    const CommitterKey &ck = index.ck();
    if (index.num_instance_variables() && instance.r1cs_input.size() != *index.num_instance_variables()) return false;
    const auto &hw = witness.hp_witness;
    if ((witness.randomness || hw.randomness) && !ck.has_hiding()) throw AccmsmError("decide: the key has no hiding generator");
    const Affine *pts[6] = {&instance.comm_a, &instance.comm_b, &instance.comm_c, &instance.hp_instance.comm_1,
                            &instance.hp_instance.comm_2, &instance.hp_instance.comm_3};
    uint64_t exp[48]; uint8_t einf[6];
    for (int j = 0; j < 6; j++) { affine_to(*pts[j], exp + 8 * j); einf[j] = pts[j]->infinity; }
    uint64_t sig[12], hr[12];
    if (witness.randomness) {
        std::memcpy(sig, witness.randomness->sigma_a.data(), 32); std::memcpy(sig + 4, witness.randomness->sigma_b.data(), 32);
        std::memcpy(sig + 8, witness.randomness->sigma_c.data(), 32);
    }
    if (hw.randomness) {
        std::memcpy(hr, hw.randomness->rand_1.data(), 32); std::memcpy(hr + 4, hw.randomness->rand_2.data(), 32);
        std::memcpy(hr + 8, hw.randomness->rand_3.data(), 32);
    }
    const auto &x = instance.r1cs_input, &w = witness.r1cs_blinded_witness;
    int accept = 0;
    ck.ctx()->check(accmsm_nark_as_decide(ck.ctx()->raw(), ck.handle(), index.handle(), x.empty() ? nullptr : x[0].data(), x.size(),
                                          w.empty() ? nullptr : w[0].data(), w.size(), hw.a_vec.empty() ? nullptr : hw.a_vec[0].data(),
                                          hw.a_vec.size(), hw.b_vec.empty() ? nullptr : hw.b_vec[0].data(), hw.b_vec.size(),
                                          ck.hiding_index(), witness.randomness ? sig : nullptr, hw.randomness ? hr : nullptr, exp, einf,
                                          &accept, nullptr, nullptr), "nark_as_decide");
    return accept != 0;
}
}  // namespace r1cs_nark_as

}  // namespace accmsm_host
