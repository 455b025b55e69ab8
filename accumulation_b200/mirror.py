"""Reference-named harness mirror of the calls that reach the hot path (SURVEY.md 8a/8b).

Same names, argument meaning and accept/reject behaviour as the reference's call sites, so the parity
tests read like the reference's own; everything computes on the GPU through the C-ABI.  The C++ twin of
this file, used by the Rust-side integration, is `accumulation_b200/host/ark_mirror.hpp`.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, List, Optional, Sequence

import numpy as np


@dataclass
class CommitterKey:
    """trivial_pc::CommitterKey{generators, hiding_generator} / ipa_pc::CommitterKey{comm_key, h, s}.

    The hiding generator is registered as the base after the last generator so that
    `commit(elems, randomizer)` is a single device MSM (SURVEY.md App. A.2); IpaPC's s, when given, follows it
    (generators || h || s), so a zk opening's hiding_comm is one device MSM too."""
    bases: "object"          # accumulation_b200.Bases: generators || hiding_generator [|| s]
    num_generators: int
    s_index: Optional[int] = None

    @staticmethod
    def new(ctx, curve: int, generators_xy, hiding_generator_xy=None, precompute: bool = False, s_xy=None) -> "CommitterKey":
        """precompute: also build the window table (once per key; trim / index time in the reference)"""
        gens = np.ascontiguousarray(generators_xy, dtype=np.uint64).reshape(-1, 8)
        if s_xy is not None and hiding_generator_xy is None:
            raise ValueError("CommitterKey.new: s follows the hiding generator h; pass both")
        extra = [np.ascontiguousarray(p, dtype=np.uint64).reshape(1, 8) for p in (hiding_generator_xy, s_xy) if p is not None]
        allb = np.concatenate([gens] + extra) if extra else gens
        bases = ctx.register_bases(curve, allb)
        if precompute:
            bases.precompute()
        return CommitterKey(bases, gens.shape[0], None if s_xy is None else gens.shape[0] + 1)

    def supported_num_elems(self) -> int:   # src/hp_as/mod.rs:129,681
        return self.num_generators

    @property
    def curve(self) -> int:
        return self.bases.curve


class PedersenCommitment:
    """ark_poly_commit::trivial_pc::PedersenCommitment (call sites: src/hp_as/mod.rs:196,197,214,377,910-918;
    src/r1cs_nark_as/r1cs_nark/mod.rs:216-261,375-407; src/r1cs_nark_as/mod.rs:394-410,1081-1097)."""

    @staticmethod
    def commit(ck: CommitterKey, elems, randomizer=None):
        """-> (xy[8], infinity).  ark-ec truncates to min(len(generators), len(elems))."""
        el = np.ascontiguousarray(elems, dtype=np.uint64).reshape(-1, 4)[: ck.num_generators]
        ctx = ck.bases.ctx
        if randomizer is None:
            return ctx.msm(ck.bases, el, montgomery=True)
        return ctx.commit(ck.bases, el, hiding_index=ck.num_generators, randomizer_mont=randomizer)


class SuccinctCheckPolynomial:
    """ark_poly_commit::ipa_pc::SuccinctCheckPolynomial(pub Vec<F>) (src/ipa_pc_as/mod.rs:245,400,418)."""

    def __init__(self, ctx, field: int, challenges):
        self.ctx, self.field = ctx, field
        self.challenges = np.ascontiguousarray(challenges, dtype=np.uint64).reshape(-1, 4)

    def compute_coeffs(self):
        return self.ctx.compute_coeffs(self.field, self.challenges)


_MODULI = (0x40000000000000000000000000000000224698FC094CF91B992D30ED00000001,   # Fp: Pallas base / Vesta scalar
           0x40000000000000000000000000000000224698FC0994A8DD8C46EB2100000001)   # Fq: Pallas scalar / Vesta base


def _fe_to_int(field: int, mont) -> int:
    """host-side scalar helper (one element per IPA round, like ark-ff on the Rust host): Montgomery limbs -> int"""
    m = _MODULI[field]
    v = sum(int(x) << (64 * i) for i, x in enumerate(np.asarray(mont, dtype=np.uint64).reshape(4)))
    return v * pow(1 << 256, -1, m) % m


def _int_to_fe(field: int, v: int) -> np.ndarray:
    m = _MODULI[field]
    w = (v % m) * (1 << 256) % m
    return np.array([(w >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(4)], dtype=np.uint64)


def _canon(values) -> np.ndarray:
    """canonical integers -> (n, 4) limbs"""
    return np.array([[(v >> (64 * j)) & 0xFFFFFFFFFFFFFFFF for j in range(4)] for v in values], dtype=np.uint64).reshape(-1, 4)


def _canon_mont(field: int, values) -> np.ndarray:
    """integers -> (n, 4) Montgomery limbs"""
    return np.array([_int_to_fe(field, v) for v in values], dtype=np.uint64).reshape(-1, 4)


def _same_affine(a, b) -> bool:
    """GroupAffine PartialEq on (xy, inf) pairs: both identity, or the same (x, y)"""
    if int(a[1]) or int(b[1]):
        return bool(int(a[1])) == bool(int(b[1]))
    return np.array_equal(np.asarray(a[0], dtype=np.uint64), np.asarray(b[0], dtype=np.uint64))


@dataclass
class ZkHiding:
    """What a zk opening (MakeZK::Enabled) adds to InnerProductArgPC.open: the random hiding polynomial (<= 2^k
    coefficients from the caller's rng), its randomiser rho, the commitment C = (xy, inf) being opened with its randomness
    r, and `alpha(hiding_comm) -> alpha`, the host sponge over (C, z, v, hiding_comm).  Montgomery limbs throughout."""
    coeffs: "object"
    rand: "object"
    comm: tuple
    comm_rand: "object"
    alpha: Callable


class InnerProductArgPC:
    """The parts of ark_poly_commit::ipa_pc::InnerProductArgPC that run the MSM."""

    @staticmethod
    def open(ck: CommitterKey, combined_coeffs, point, h_prime_xy, round_challenge, log_d: Optional[int] = None, xi0=None,
             hiding: Optional["ZkHiding"] = None):
        """Core of open_individual_opening_challenges (SURVEY.md App. A.2; src/ipa_pc_as/mod.rs:454-462) after the
        host has combined the polynomials and derived h' = xi_0 * h (pass either the point h_prime_xy, or xi0 when h is the
        hiding generator of `ck`: faster, no separate scalar multiplication).  `round_challenge(prev_xi, l, r) -> xi` is the
        host sponge (Montgomery limbs in and out; prev_xi is None in the first round).
        hiding (MakeZK::Enabled, needs ck.s_index): before the first round the random polynomial is shifted to vanish at
        the point and committed, alpha is squeezed from hiding_comm, P += alpha hiding' on the device and
        C' = C + alpha hiding_comm - rand s with rand = r + alpha rho; xi0 (or h_prime_xy) may then be a callable of C'.
        Returns (l_vec, r_vec, final_comm_key_xy, c, challenges), plus (hiding_comm, rand) when hiding is given."""
        from . import scalar_field
        ctx = ck.bases.ctx
        field = scalar_field(ck.curve)
        cf = np.ascontiguousarray(combined_coeffs, dtype=np.uint64).reshape(-1, 4)
        k = log_d if log_d is not None else max(cf.shape[0] - 1, 0).bit_length()
        hiding_comm = rand = None
        if hiding is not None:
            if ck.s_index is None:
                raise ValueError("InnerProductArgPC.open: a zk opening needs a key registered with s (CommitterKey.new(.., s_xy=))")
            hp_now = None if callable(h_prime_xy) else h_prime_xy
            sess = ctx.ipa_open_begin(ck.bases, cf, k, point, hp_now)
            try:
                hiding_comm = ctx.ipa_open_hide(sess, hiding.coeffs, ck.s_index, hiding.rand)
                alpha = np.ascontiguousarray(hiding.alpha(hiding_comm), dtype=np.uint64).reshape(4)
                ctx.ipa_open_hiding_challenge(sess, alpha)
                rand = _int_to_fe(field, _fe_to_int(field, hiding.comm_rand) + _fe_to_int(field, alpha) * _fe_to_int(field, hiding.rand))
                c_prime = InnerProductArgPC.hiding_commitment(ck, hiding.comm, hiding_comm, alpha, rand)
                if callable(xi0):
                    xi0 = xi0(c_prime)
                if callable(h_prime_xy):
                    raise ValueError("InnerProductArgPC.open: h' derived from C' goes in as xi0 (h' = xi_0 * h)")
                if xi0 is not None:
                    ctx.ipa_open_use_hiding_generator(sess, ck.num_generators, xi0)
            except Exception:
                InnerProductArgPC._release(ctx, sess)
                raise
        elif xi0 is not None:      # h' = xi_0 * (hiding generator registered after the generators): no point needed
            sess = ctx.ipa_open_begin(ck.bases, cf, k, point, None)
            ctx.ipa_open_use_hiding_generator(sess, ck.num_generators, xi0)
        else:
            sess = ctx.ipa_open_begin(ck.bases, cf, k, point, h_prime_xy)
        l_vec, r_vec, challenges, xi = [], [], [], None
        lr = ctx.ipa_open_round(sess) if k else None
        while lr is not None:                      # one library call per round: fold (xi^-1 inside) + next round
            l, r = lr
            xi = np.ascontiguousarray(round_challenge(xi, l, r), dtype=np.uint64).reshape(4)
            l_vec.append(l); r_vec.append(r); challenges.append(xi)
            lr = ctx.ipa_open_fold_round(sess, xi)
        final_key, c = ctx.ipa_open_finish(sess)
        if hiding is not None:
            return l_vec, r_vec, final_key, c, challenges, hiding_comm, rand
        return l_vec, r_vec, final_key, c, challenges

    @staticmethod
    def _release(ctx, sess):
        try:
            ctx.ipa_open_finish(sess)       # finishing a session with rounds left releases it
        except Exception:
            pass

    @staticmethod
    def hiding_commitment(ck: CommitterKey, comm, hiding_comm, alpha, rand):
        """C' = C + alpha hiding_comm - rand s, the commitment a zk opening proves against (upstream computes it on the
        host before squeezing xi_0; here one 3-term device MSM) -> (xy, inf)"""
        from . import scalar_field
        f = scalar_field(ck.curve)
        m = _MODULI[f]
        s_xy = ck.bases.ctx.download_bases(ck.bases, ck.s_index, 1).reshape(8)
        pts = np.array([np.asarray(comm[0], dtype=np.uint64), np.asarray(hiding_comm[0], dtype=np.uint64), s_xy])
        inf = np.array([int(comm[1]), int(hiding_comm[1]), 0], dtype=np.uint8)
        sc = _canon([1, _fe_to_int(f, alpha), (-_fe_to_int(f, rand)) % m])
        return ck.bases.ctx.msm_oneshot(ck.curve, pts, sc, montgomery=False, infinity=inf)

    @staticmethod
    def cm_commit(comm_key: CommitterKey, scalars, hiding_generator_index: Optional[int] = None, randomizer=None):
        if randomizer is None:
            return PedersenCommitment.commit(comm_key, scalars)
        el = np.ascontiguousarray(scalars, dtype=np.uint64).reshape(-1, 4)[: comm_key.num_generators]
        idx = comm_key.num_generators if hiding_generator_index is None else hiding_generator_index
        return comm_key.bases.ctx.commit(comm_key.bases, el, hiding_index=idx, randomizer_mont=randomizer)

    @staticmethod
    def succinct_check_equation(ctx, curve: int, comm, point, value, l_vec, r_vec, round_challenges, h_prime_xy, final_comm_key_xy, c,
                                hiding=None) -> bool:
        """Group equation of IpaPC::succinct_check (SURVEY.md App. A.2; src/ipa_pc_as/mod.rs:198-205) with the transcript
        values supplied by the host:  C + v h' + sum_i (xi_i^-1 l_i + xi_i r_i) == c final_comm_key + (h(z) c) h'.
        One 2k + 3 term MSM over unregistered points (accmsm_msm_oneshot) whose result must be the identity; the O(k)
        scalar preparation (inverses, h(z)) is host arithmetic like in the reference.  comm = (xy, inf).
        hiding = (hiding_comm, alpha, rand, s_xy) of a zk proof: C becomes C' = C + alpha hiding_comm - rand s, two more
        terms (2k + 5)."""
        bases, inf, sc = InnerProductArgPC.succinct_check_terms(curve, comm, point, value, l_vec, r_vec, round_challenges, h_prime_xy,
                                                                final_comm_key_xy, c, hiding)
        _, res_inf = ctx.msm_oneshot(curve, bases, sc, montgomery=False, infinity=inf)
        return bool(res_inf)

    @staticmethod
    def succinct_check_terms(curve: int, comm, point, value, l_vec, r_vec, round_challenges, h_prime_xy, final_comm_key_xy, c,
                             hiding=None):
        """(bases (2k + 3, 8), infinity flags, canonical scalars (2k + 3, 4)) of the equation above; 2k + 5 with hiding"""
        from . import scalar_field
        f = scalar_field(curve)
        m = _MODULI[f]
        xis = [_fe_to_int(f, x) for x in np.asarray(round_challenges, dtype=np.uint64).reshape(-1, 4)]
        k = len(xis)
        z, v, cc = _fe_to_int(f, point), _fe_to_int(f, value), _fe_to_int(f, c)
        hz = 1
        for i, xi in enumerate(xis, start=1):
            hz = hz * (1 + xi * pow(z, 1 << (k - i), m)) % m
        bases = [np.asarray(comm[0], dtype=np.uint64)] + [np.asarray(p[0], dtype=np.uint64) for p in l_vec] + \
                [np.asarray(p[0], dtype=np.uint64) for p in r_vec] + [np.asarray(h_prime_xy, dtype=np.uint64), np.asarray(final_comm_key_xy, dtype=np.uint64)]
        inf = [int(comm[1])] + [int(p[1]) for p in l_vec] + [int(p[1]) for p in r_vec] + [0, 0]
        scal = [1] + [pow(xi, -1, m) for xi in xis] + xis + [(v - hz * cc) % m, (-cc) % m]
        if hiding is not None:
            hiding_comm, alpha, rand, s_xy = hiding
            bases += [np.asarray(hiding_comm[0], dtype=np.uint64), np.asarray(s_xy, dtype=np.uint64).reshape(8)]
            inf += [int(hiding_comm[1]), 0]
            scal += [_fe_to_int(f, alpha), (-_fe_to_int(f, rand)) % m]
        return np.array(bases), np.array(inf, dtype=np.uint8), _canon(scal)

    @staticmethod
    def succinct_check_equations(ctx, curve: int, instances) -> list:
        """The equations of ALL inputs and accumulators of one prove / verify (the loops at src/ipa_pc_as/mod.rs:262-270 and
        :625-640 call succinct_check once per instance) as ONE batched call (accmsm_msm_oneshot_batch): `instances` is a list
        of argument tuples of succinct_check_equation (without ctx and curve), all of the same degree.  zk instances (with
        the hiding tuple) and others mix: the others are padded with two (identity, 0) terms."""
        terms = [InnerProductArgPC.succinct_check_terms(curve, *inst) for inst in instances]
        if not terms:
            return []
        width = max(t[0].shape[0] for t in terms)
        padded = []
        for b, i, sc in terms:
            pad = width - b.shape[0]
            if pad:
                b = np.concatenate([b, np.repeat(b[:1], pad, axis=0)])
                i = np.concatenate([i, np.ones(pad, dtype=np.uint8)])
                sc = np.concatenate([sc, np.zeros((pad, 4), dtype=np.uint64)])
            padded.append((b, i, sc))
        _, inf = ctx.msm_oneshot_batch(curve, np.stack([t[0] for t in padded]), np.stack([t[2] for t in padded]), montgomery=False,
                                       infinity=np.stack([t[1] for t in padded]))
        return [bool(x) for x in inf]

    @staticmethod
    def check_final_key(vk: CommitterKey, check_poly_challenges, final_comm_key_xy, final_comm_key_inf: int = 0) -> bool:
        """Tail of check_individual_opening_challenges (reached from decide, src/ipa_pc_as/mod.rs:836-845):
        final_key = cm_commit(vk.comm_key, h.compute_coeffs()); accept iff final_key == proof.final_comm_key."""
        ok, _, _ = vk.bases.ctx.ipa_check_final_key(vk.bases, check_poly_challenges, final_comm_key_xy, final_comm_key_inf)
        return ok


def matrix_vec_mul(ctx, field: int, matrices, inp, wit):
    """r1cs_nark::matrix_vec_mul for A, B, C in one launch (src/r1cs_nark_as/r1cs_nark/mod.rs:443-447)."""
    return ctx.csr_matvec(field, matrices, inp, wit)


class ASForHadamardProducts:
    """Vector / commitment steps of src/hp_as/mod.rs that sit on the hot path."""

    @staticmethod
    def compute_hp(ctx, field, a_vec, b_vec):                       # :278-285
        return ctx.hadamard(field, a_vec, b_vec)

    @staticmethod
    def compute_t_vecs(ctx, field, a_vecs, b_vecs, mu_challenges, hp_vec_len, hiding_vecs=None):   # :288-349
        ha, hb = hiding_vecs if hiding_vecs is not None else (None, None)
        return ctx.tvecs(field, a_vecs, b_vecs, mu_challenges, hp_vec_len, ha, hb)

    @staticmethod
    def combine_vectors(ctx, field, vectors, challenges, hiding_vecs=None):   # :492-512
        return ctx.lincomb(field, vectors, challenges, hiding_vecs)

    @staticmethod
    def scale_vector(ctx, field, vector, coeff):                    # :482-489
        return ctx.scale(field, vector, coeff)

    @staticmethod
    def compute_product_poly_comm(ck: CommitterKey, t_vecs) -> tuple:   # :354-388
        """(low, high): commitments to every t-vector except the middle one, without randomiser."""
        n2 = len(t_vecs)
        mid = (n2 - 1) // 2
        low = [PedersenCommitment.commit(ck, t_vecs[i]) for i in range(mid)]
        high = [PedersenCommitment.commit(ck, t_vecs[i]) for i in range(mid + 1, n2)]
        return low, high

    @staticmethod
    def compute_t_vecs_and_product_poly_comm(ck: CommitterKey, a_vecs, b_vecs, mu_challenges, hp_vec_len, hiding_vecs=None):
        """compute_t_vecs (:288-349) feeding compute_product_poly_comm (:354-388) without the t-vectors leaving HBM.
        -> (low, high) lists of (xy, inf)"""
        ha, hb = hiding_vecs if hiding_vecs is not None else (None, None)
        (low, linf), (high, hinf), _ = ck.bases.ctx.hp_product_poly_comm(ck.bases, a_vecs, b_vecs, mu_challenges, hp_vec_len, ha, hb)
        return [(low[i], int(linf[i])) for i in range(low.shape[0])], [(high[i], int(hinf[i])) for i in range(high.shape[0])]

    @staticmethod
    def decide(ck: CommitterKey, instance, witness) -> bool:        # :894-925
        """instance = (comm_1, comm_2, comm_3) as (xy, inf) pairs; witness = (a_vec, b_vec, randomness|None),
        randomness = (rand_1, rand_2, rand_3).  One fused device call: Hadamard product + the three commitments in a
        shared pass of the MSM pipeline + the comparison."""
        a_vec, b_vec, rand = witness
        a = np.ascontiguousarray(a_vec, dtype=np.uint64).reshape(-1, 4)[: ck.num_generators]
        b = np.ascontiguousarray(b_vec, dtype=np.uint64).reshape(-1, 4)[: ck.num_generators]
        exp_xy = np.array([np.asarray(c[0], dtype=np.uint64) for c in instance])
        exp_inf = np.array([int(c[1]) for c in instance], dtype=np.uint8)
        r = None if rand is None else np.array([np.asarray(x, dtype=np.uint64) for x in rand])
        ok, _, _ = ck.bases.ctx.hp_decide(ck.bases, a, b, exp_xy, exp_inf, hiding_index=ck.num_generators, randomness=r)
        return ok

    @staticmethod
    def prove(ck: CommitterKey, witnesses, instances, mu_fn: Callable, nu_fn: Callable, zk=None):   # :646-813
        """ASForHadamardProducts::prove over the already padded pairs, inputs first, then old accumulators (the placeholder
        padding of :676-710 stays with the caller).  witnesses: [(a, b, (r1, r2, r3) | None)], instances: [(C1, C2, C3)] with
        (xy, inf) points.  zk = (ha, hb, (hr1, hr2, hr3)) from the caller's rng (ha, hb of hp_vec_len = ck.num_generators
        elements).  The sponge is the callables: mu_fn(hiding_comms | None) -> mu_1 .. mu_{n-1} and nu_fn(low, high) -> nu
        (Montgomery limbs).  One device session (begin, product_poly_comm, finish) forms the hiding commitments, the
        product-polynomial commitments and a*, b*; the randomness (App. C.5) is host arithmetic and the new instance (C.6) one
        3-equation msm_oneshot_batch.  -> (new instance (C1*, C2*, C3*), new witness (a*, b*, rand* | None),
        proof (hiding_comms | None, low, high))"""
        from . import scalar_field
        ctx, f = ck.bases.ctx, scalar_field(ck.curve)
        m, L, n = _MODULI[f], ck.num_generators, len(witnesses)
        a = [np.ascontiguousarray(w[0], dtype=np.uint64).reshape(-1, 4)[:L] for w in witnesses]
        b = [np.ascontiguousarray(w[1], dtype=np.uint64).reshape(-1, 4)[:L] for w in witnesses]
        ha, hb, hr = (None, None, None) if zk is None else zk
        sess, hc = ctx.hp_prove_begin(ck.bases, a, b, L, ha, hb, hiding_index=ck.num_generators, hiding_rand=None if hr is None else np.array(hr))
        try:
            hiding_comms = None if hc is None else [(hc[0][j], int(hc[1][j])) for j in range(3)]
            mus = [_fe_to_int(f, x) for x in np.asarray(mu_fn(hiding_comms), dtype=np.uint64).reshape(-1, 4)]
            mu = [1] + mus + ([mus[0] * mus[-1] % m] if zk is not None else [])
            (lo, linf), (hi, hinf) = ctx.hp_prove_product_poly_comm(sess, n, _canon_mont(f, mu))
            low = [(lo[j], int(linf[j])) for j in range(n - 1)]
            high = [(hi[j], int(hinf[j])) for j in range(n - 1)]
            nu = np.ascontiguousarray(nu_fn(low, high), dtype=np.uint64).reshape(4)
        except Exception:
            try:
                ctx.hp_prove_abort(sess)
            except Exception:
                pass
            raise
        a_star, b_star = ctx.hp_prove_finish(sess, nu, L)
        v = _fe_to_int(f, nu)
        nus = [pow(v, j, m) for j in range(2 * n - 1)]
        rand = None
        if zk is not None:
            hrs = [_fe_to_int(f, x) for x in hr]
            rs = [None if w[2] is None else [_fe_to_int(f, x) for x in w[2]] for w in witnesses]
            mu_n = mu[n]
            r1 = (mu_n * hrs[0] + sum(mu[i] * nus[i] * rs[i][0] for i in range(n) if rs[i] is not None)) % m
            r2 = (mu[1] * hrs[1] + sum(nus[j] * rs[n - 1 - j][1] for j in range(n) if rs[n - 1 - j] is not None)) % m
            r3 = (mu_n * hrs[2] + sum(mu[i] * rs[i][2] for i in range(n) if rs[i] is not None)) * nus[n - 1] % m
            rand = [_int_to_fe(f, r) for r in (r1, r2, r3)]
        new_instance = ASForHadamardProducts.combined_commitments(ck, instances, hiding_comms, low, high, mu, v)
        return new_instance, (a_star, b_star, rand), (hiding_comms, low, high)

    @staticmethod
    def combined_commitments(ck: CommitterKey, instances, hiding_comms, low, high, mu, nu: int):    # :409-479 (App. C.6)
        """C1* = [mu_n H1] + sum_i mu_i nu^i C1_i,  C2* = [mu_1 H2] + sum_j nu^j C2_{n-1-j},
        C3* = sum_j nu^j low_j + sum_j nu^(n+j) high_j + nu^(n-1) ([mu_n H3] + sum_i mu_i C3_i), as ONE msm_oneshot_batch of
        3 equations padded with (identity, 0) terms.  mu: integers (n, n + 1 with hiding entries), nu: an integer."""
        from . import scalar_field
        m = _MODULI[scalar_field(ck.curve)]
        n = len(instances)
        nus = [pow(nu, j, m) for j in range(2 * n - 1)]
        e1 = [(instances[i][0], mu[i] * nus[i]) for i in range(n)]
        e2 = [(instances[n - 1 - j][1], nus[j]) for j in range(n)]
        e3 = [(low[j], nus[j]) for j in range(n - 1)] + [(high[j], nus[n + j]) for j in range(n - 1)]
        e3 += [(instances[i][2], mu[i] * nus[n - 1]) for i in range(n)]
        if hiding_comms is not None:
            e1.append((hiding_comms[0], mu[n]))
            e2.append((hiding_comms[1], mu[1]))
            e3.append((hiding_comms[2], mu[n] * nus[n - 1]))
        eqs = [e1, e2, e3]
        width = max(len(e) for e in eqs)
        eqs = [e + [((e[0][0][0], 1), 0)] * (width - len(e)) for e in eqs]     # (a point flagged as the identity, 0)
        pts = np.array([[np.asarray(p[0], dtype=np.uint64) for p, _ in e] for e in eqs])
        infs = np.array([[int(p[1]) for p, _ in e] for e in eqs], dtype=np.uint8)
        sc = np.stack([_canon([s % m for _, s in e]) for e in eqs])
        xy, inf = ck.bases.ctx.msm_oneshot_batch(ck.curve, pts, sc, montgomery=False, infinity=infs)
        return tuple((xy[j], int(inf[j])) for j in range(3))

    @staticmethod
    def verify(ck: CommitterKey, instances, new_instance, proof, mu_fn: Callable, nu_fn: Callable) -> bool:   # :815-892
        """The verifier's O(n) recomputation: mu and nu from the same sponge callables as prove, then C1*, C2*, C3* from the
        old instances and the proof (one msm_oneshot_batch), accept iff they equal new_instance.  A proof whose shape does not
        fit n (low / high of n - 1 points each) is rejected."""
        from . import scalar_field
        f = scalar_field(ck.curve)
        m, n = _MODULI[f], len(instances)
        hiding_comms, low, high = proof
        if n < 1 or len(low) != n - 1 or len(high) != n - 1 or (hiding_comms is not None and len(hiding_comms) != 3):
            return False
        mus = [_fe_to_int(f, x) for x in np.asarray(mu_fn(hiding_comms), dtype=np.uint64).reshape(-1, 4)]
        if len(mus) != n - 1:
            return False
        mu = [1] + mus + ([mus[0] * mus[-1] % m] if hiding_comms is not None else [])
        nu = _fe_to_int(f, nu_fn(low, high))
        got = ASForHadamardProducts.combined_commitments(ck, instances, hiding_comms, low, high, mu, nu)
        return all(_same_affine(g, e) for g, e in zip(got, new_instance))


@dataclass
class NarkProof:
    """r1cs_nark::Proof (src/r1cs_nark_as/r1cs_nark/data_structures.rs): first_msg = [comm_a, comm_b, comm_c] without zk, or
    [comm_a, comm_b, comm_c, comm_r_a, comm_r_b, comm_r_c, comm_1, comm_2] with it, as (xy, inf); blinded_witness = w (no zk)
    or w' = w + gamma r; sigmas = (sigma_a, sigma_b, sigma_c, sigma_o) as (4, 4) Montgomery limbs, None without zk."""
    first_msg: list
    blinded_witness: "object"
    sigmas: "object" = None


class R1CSNark:
    """The mat-vec + commitment steps of src/r1cs_nark_as/r1cs_nark/mod.rs (prove :183-316, verify :335-419) and of
    ASForR1CSNark::decide (src/r1cs_nark_as/mod.rs:1052-1097) with the index matrices registered once."""

    def __init__(self, ck: CommitterKey, matrices, num_instance_variables: Optional[int] = None):
        """num_instance_variables: the index's input length (IndexInfo), which ASForR1CSNark.decide checks r1cs_input against"""
        from . import scalar_field
        self.ck = ck
        self.num_instance_variables = num_instance_variables
        self.n_mats = len(matrices)
        self.n_rows = int(np.asarray(matrices[0][0]).size - 1)
        self.csr = ck.bases.ctx.register_csr(scalar_field(ck.curve), matrices)

    def matvec_commit(self, inp, wit, blinders=None):
        """-> ([M (input || witness)], [(comm_xy, inf)])"""
        vecs, xy, inf = self.ck.bases.ctx.csr_matvec_commit(self.ck.bases, self.csr, self.n_mats, self.n_rows, inp, wit,
                                                             hiding_index=self.ck.num_generators, blinders=blinders)
        return vecs, [(xy[i], int(inf[i])) for i in range(self.n_mats)]

    def prove(self, inp, wit, gamma_fn: Callable, zk=None) -> NarkProof:
        """R1CSNark::prove (:183-316).  zk = (r, blinders): the random witness-length vector and the 8 blinders in the order
        A, B, C, rA, rB, rC, 1, 2 (the caller's rng); gamma_fn(first_msg) -> gamma is the host sponge over the first message.
        Without zk: one matvec_commit.  With zk: one nark_prove_zk call (one vector launch + one 8-job pass), then
        w' = w + gamma r on the device and the sigmas on the host."""
        from . import scalar_field
        if zk is None:
            _, comms = self.matvec_commit(inp, wit)
            return NarkProof(comms, np.ascontiguousarray(wit, dtype=np.uint64).reshape(-1, 4), None)
        ctx, f = self.ck.bases.ctx, scalar_field(self.ck.curve)
        r, blinders = zk
        _, xy, inf = ctx.nark_prove_zk(self.ck.bases, self.csr, self.n_rows, inp, wit, r, blinders, hiding_index=self.ck.num_generators,
                                       want_vecs=False)
        first = [(xy[i], int(inf[i])) for i in range(8)]
        gamma = np.ascontiguousarray(gamma_fn(first), dtype=np.uint64).reshape(4)
        w = np.ascontiguousarray(wit, dtype=np.uint64).reshape(-1, 4)
        w_prime = ctx.lincomb(f, [r], gamma.reshape(1, 4), hiding=w) if w.shape[0] else w
        m, g = _MODULI[f], _fe_to_int(f, gamma)
        b = [_fe_to_int(f, x) for x in np.asarray(blinders, dtype=np.uint64).reshape(8, 4)]
        sig = [b[i] + g * b[3 + i] for i in range(3)] + [b[2] + g * b[6] + g * g % m * b[7]]
        return NarkProof(first, w_prime, np.array([_int_to_fe(f, s) for s in sig]))

    def verify(self, inp, proof: NarkProof, gamma=None) -> bool:
        """R1CSNark::verify (:335-419).  With zk the four left-hand sides comm_M + gamma comm_rM and comm_C + gamma comm_1 +
        gamma^2 comm_2 come from ONE msm_oneshot_batch (4 equations x 3 terms, the 2-term ones padded with (identity, 0));
        then one nark_verify call: t_M = M (input || w'), the 4 commitments in one pass, and the comparison."""
        from . import scalar_field
        ctx, f = self.ck.bases.ctx, scalar_field(self.ck.curve)
        fm = proof.first_msg
        if proof.sigmas is None:
            lhs = [fm[0], fm[1], fm[2], fm[2]]
        else:
            m, g = _MODULI[f], _fe_to_int(f, gamma)
            eqs = [[(fm[i], 1), (fm[3 + i], g), (fm[i], None)] for i in range(3)] + [[(fm[2], 1), (fm[6], g), (fm[7], g * g % m)]]
            pts = np.array([[np.asarray(p[0], dtype=np.uint64) for p, _ in eq] for eq in eqs])
            infs = np.array([[1 if s is None else int(p[1]) for p, s in eq] for eq in eqs], dtype=np.uint8)
            sc = np.stack([_canon([0 if s is None else s for _, s in eq]) for eq in eqs])
            xy, inf = ctx.msm_oneshot_batch(self.ck.curve, pts, sc, montgomery=False, infinity=infs)
            lhs = [(xy[i], int(inf[i])) for i in range(4)]
        ok, _, _, _ = ctx.nark_verify(self.ck.bases, self.csr, self.n_rows, inp, proof.blinded_witness,
                                      np.array([np.asarray(p[0], dtype=np.uint64) for p in lhs]), [p[1] for p in lhs],
                                      hiding_index=self.ck.num_generators, sigmas=proof.sigmas)
        return ok

    def release(self):
        self.ck.bases.ctx.release_csr(self.csr)


@dataclass
class AccumulatorInstance:
    """r1cs_nark_as::AccumulatorInstance (src/r1cs_nark_as/data_structures.rs:156-171): comm_a, comm_b, comm_c and the
    hp_instance (comm_1, comm_2, comm_3) as (xy, inf)."""
    r1cs_input: "object"
    comm_a: tuple
    comm_b: tuple
    comm_c: tuple
    hp_instance: tuple


@dataclass
class AccumulatorWitness:
    """r1cs_nark_as::AccumulatorWitness (src/r1cs_nark_as/data_structures.rs:218-227): hp_witness = (a_vec, b_vec,
    randomness | None) as in ASForHadamardProducts.decide; randomness = (sigma_a, sigma_b, sigma_c) or None."""
    r1cs_blinded_witness: "object"
    hp_witness: tuple
    randomness: "object" = None


class ASForR1CSNark:
    """The decider of src/r1cs_nark_as/mod.rs (:1031-1112) over an R1CSNark index (matrices registered once)."""

    @staticmethod
    def decide(nark: R1CSNark, instance: AccumulatorInstance, witness: AccumulatorWitness) -> bool:
        """t_M = M (r1cs_input || r1cs_blinded_witness); accept iff Commit(t_M, sigma_M) == comm_M for M = A, B, C and the hp
        decider accepts (a*, b*, randomness) against hp_instance.  One nark_as_decide call: one vector launch, the six
        commitments in one 6-job pass, the comparison.  An r1cs_input whose length differs from the index's is rejected on
        the host."""
        x = np.ascontiguousarray(instance.r1cs_input, dtype=np.uint64).reshape(-1, 4)
        if nark.num_instance_variables is not None and x.shape[0] != nark.num_instance_variables:
            return False
        a_vec, b_vec, hp_rand = witness.hp_witness
        pts = [instance.comm_a, instance.comm_b, instance.comm_c, *instance.hp_instance]
        exp_xy = np.array([np.asarray(p[0], dtype=np.uint64) for p in pts])
        exp_inf = np.array([int(p[1]) for p in pts], dtype=np.uint8)
        sig = None if witness.randomness is None else np.array([np.asarray(v, dtype=np.uint64) for v in witness.randomness])
        hr = None if hp_rand is None else np.array([np.asarray(v, dtype=np.uint64) for v in hp_rand])
        ok, _, _ = nark.ck.bases.ctx.nark_as_decide(nark.ck.bases, nark.csr, x, witness.r1cs_blinded_witness, a_vec, b_vec, exp_xy, exp_inf,
                                                     hiding_index=nark.ck.num_generators, sigmas=sig, hp_randomness=hr)
        return ok
