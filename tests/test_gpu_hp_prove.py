"""The prover of the Hadamard-product accumulation scheme, ASForHadamardProducts::prove (src/hp_as/mod.rs:646-813), as a device
session: accmsm_hp_prove_begin (the pairs uploaded once; with zk one kernel and one 3-job pass for the hiding commitments),
accmsm_hp_prove_product_poly_comm (k_tvecs and the 2n - 2 commitments) and accmsm_hp_prove_finish (a*, b*).

The oracle side is restated here from SURVEY App. C.1-C.7 over the oracle primitives (tvecs, combine_vectors, scale, hadamard,
commit, point_mul, point_add).  The unmarked tests check that restatement without a GPU: its accumulator is accepted by the
restated verify and decide, and every corruption is rejected.  The gpu tests compare every output of the session bit for bit
with it, on both curves, on one context and on device groups."""
import ctypes as C
import hashlib

import numpy as np
import pytest

import accumulation_b200 as ab
from oracle import cref
from tests.util import same_point
from tests.test_gpu_msm_dispatch import passes, plan, table_window_bits

E_ARG, E_HANDLE = -2, -3
MODULI = (0x40000000000000000000000000000000224698FC094CF91B992D30ED00000001,
          0x40000000000000000000000000000000224698FC0994A8DD8C46EB2100000001)
IDENTITY = (np.zeros(8, np.uint64), 1)


# ---- helpers --------------------------------------------------------------------------------------------------------------
def to_mont(f, xs):
    m = MODULI[f]
    return cref.ints_to_arr([(x % m) * (1 << 256) % m for x in xs]).reshape(-1, 4)


def from_mont(f, arr):
    m = MODULI[f]
    return [x * pow(1 << 256, -1, m) % m for x in cref.arr_to_ints(arr)]


def _digest(tag, points):
    h = hashlib.sha256(tag)
    for p in points or []:
        h.update(np.asarray(p[0], np.uint64).tobytes()); h.update(bytes([int(p[1])]))
    return h


def mu_stand_in(f, n):
    """host sponge stand-in: mu_1 .. mu_{n-1} as 128-bit values derived from the hiding commitments (or from nothing)"""
    def fn(hiding_comms):
        h = _digest(b"mu", hiding_comms)
        out = []
        for i in range(n - 1):
            h.update(bytes([i]))
            out.append(int.from_bytes(h.digest()[:16], "little") | 1)
        return to_mont(f, out)
    return fn


def nu_stand_in(f):
    def fn(low, high):
        return to_mont(f, [int.from_bytes(_digest(b"nu", list(low) + list(high)).digest()[:16], "little") | 1]).reshape(4)
    return fn


def mu_list(f, mus, zk):
    m = MODULI[f]
    mus = from_mont(f, mus)
    return [1] + mus + ([mus[0] * mus[-1] % m] if zk else [])


def _pm(curve, p, s):
    return cref.point_mul(curve, p[0], p[1], cref.from_int(s))


def _psum(curve, terms):
    acc = IDENTITY
    for p, s in terms:
        q = _pm(curve, p, s)
        acc = cref.point_add(curve, acc[0], acc[1], q[0], q[1])
    return acc


def _flip(a, i, j):
    b = np.array(a, dtype=np.uint64, copy=True)
    b[i, j] ^= np.uint64(1)
    return b


# ---- oracle restatement (SURVEY App. C.1-C.7) -------------------------------------------------------------------------------
def oracle_commit(curve, gens, h, v, r=None):
    v = np.asarray(v, np.uint64).reshape(-1, 4)
    return cref.commit(curve, gens[: v.shape[0]], v) if r is None else cref.commit(curve, gens[: v.shape[0]], v, h, r)


def oracle_hiding_comms(curve, gens, h, a, b, zk):
    """Commit(ha, r1), Commit(hb, r2), Commit(ha o b_0 + a_{n-1} o hb, r3): the hiding part of the middle t-vector (C.3)"""
    f = cref.scalar_field(curve)
    ha, hb, hr = zk
    k0, k1 = min(ha.shape[0], b[0].shape[0]), min(a[-1].shape[0], hb.shape[0])
    one = to_mont(f, [1, 1])
    cross = cref.combine_vectors(f, [cref.hadamard(f, ha[:k0], b[0][:k0]), cref.hadamard(f, a[-1][:k1], hb[:k1])], one)
    return [oracle_commit(curve, gens, h, ha, hr[0]), oracle_commit(curve, gens, h, hb, hr[1]), oracle_commit(curve, gens, h, cross, hr[2])]


def oracle_combined(curve, insts, hiding_comms, low, high, mu, nu):
    """C1*, C2*, C3* (C.6)"""
    m = MODULI[cref.scalar_field(curve)]
    n = len(insts)
    nus = [pow(nu, j, m) for j in range(2 * n - 1)]
    e1 = [(insts[i][0], mu[i] * nus[i] % m) for i in range(n)]
    e2 = [(insts[n - 1 - j][1], nus[j]) for j in range(n)]
    e3 = [(low[j], nus[j]) for j in range(n - 1)] + [(high[j], nus[n + j]) for j in range(n - 1)]
    e3 += [(insts[i][2], mu[i] * nus[n - 1] % m) for i in range(n)]
    if hiding_comms is not None:
        e1.append((hiding_comms[0], mu[n])); e2.append((hiding_comms[1], mu[1])); e3.append((hiding_comms[2], mu[n] * nus[n - 1] % m))
    return [_psum(curve, e) for e in (e1, e2, e3)]


def oracle_prove(curve, gens, h, L, wits, insts, mu, nu, zk=None, zk_comm=None):
    """ASForHadamardProducts::prove with fixed challenges (mu: ints with mu_0 = 1 (and mu_n), nu: int) -> (hiding comms, low,
    high, a*, b*, rand*, new instance).  zk_comm (default zk): the hiding vectors the hiding commitments are formed from."""
    f = cref.scalar_field(curve)
    m = MODULI[f]
    n = len(wits)
    a, b = [w[0] for w in wits], [w[1] for w in wits]
    hc = None if zk is None else oracle_hiding_comms(curve, gens, h, a, b, zk if zk_comm is None else zk_comm)
    ha, hb, hr = (None, None, None) if zk is None else zk
    t = cref.tvecs(f, a, b, to_mont(f, mu), L, ha, hb)
    low = [oracle_commit(curve, gens, h, t[j]) for j in range(n - 1)]
    high = [oracle_commit(curve, gens, h, t[n + j]) for j in range(n - 1)]
    nus = [pow(nu, j, m) for j in range(2 * n - 1)]
    a_star = cref.combine_vectors(f, a, to_mont(f, [mu[i] * nus[i] for i in range(n)]), None if zk is None else cref.scale(f, ha, to_mont(f, [mu[n]])))
    b_star = cref.combine_vectors(f, b[::-1], to_mont(f, nus[:n]), None if zk is None else cref.scale(f, hb, to_mont(f, [mu[1]])))
    rand = None
    if zk is not None:
        hrs = from_mont(f, hr)
        rs = [None if w[2] is None else from_mont(f, w[2]) for w in wits]
        r1 = mu[n] * hrs[0] + sum(mu[i] * nus[i] * rs[i][0] for i in range(n) if rs[i] is not None)
        r2 = mu[1] * hrs[1] + sum(nus[j] * rs[n - 1 - j][1] for j in range(n) if rs[n - 1 - j] is not None)
        r3 = (mu[n] * hrs[2] + sum(mu[i] * rs[i][2] for i in range(n) if rs[i] is not None)) * nus[n - 1]
        rand = to_mont(f, [r1, r2, r3])
    return hc, low, high, a_star, b_star, rand, oracle_combined(curve, insts, hc, low, high, mu, nu)


def oracle_decide(curve, gens, h, inst, a, b, rand):
    """C.7"""
    f = cref.scalar_field(curve)
    k = min(a.shape[0], b.shape[0])
    prod = cref.hadamard(f, a[:k], b[:k]) if k else np.zeros((0, 4), np.uint64)
    got = [oracle_commit(curve, gens, h, v, None if rand is None else rand[j]) for j, v in enumerate((a, b, prod))]
    return all(same_point(g, e) for g, e in zip(got, inst))


def oracle_verify(curve, insts, new_inst, proof, mu, nu):
    hc, low, high = proof
    got = oracle_combined(curve, insts, hc, low, high, mu, nu)
    return all(same_point(g, e) for g, e in zip(got, new_inst))


def make_inputs(curve, gens, h, n, lens, seed, zk, L):
    """n pairs with ragged lengths (lens: [(|a_i|, |b_i|)]) and their instances; with zk every pair has randomness and the hiding
    vectors have L elements"""
    f = cref.scalar_field(curve)
    wits, insts = [], []
    for i in range(n):
        la, lb = lens[i]
        a, b = cref.gen_scalars(f, seed + 3 * i, la, True), cref.gen_scalars(f, seed + 3 * i + 1, lb, True)
        r = cref.gen_scalars(f, seed + 3 * i + 2, 3, True) if zk else None
        k = min(la, lb)
        prod = cref.hadamard(f, a[:k], b[:k]) if k else np.zeros((0, 4), np.uint64)
        insts.append([oracle_commit(curve, gens, h, v, None if r is None else r[j]) for j, v in enumerate((a, b, prod))])
        wits.append((a, b, r))
    hz = (cref.gen_scalars(f, seed + 900, L, True), cref.gen_scalars(f, seed + 901, L, True), cref.gen_scalars(f, seed + 902, 3, True)) if zk else None
    return wits, insts, hz


# ---- CPU: the restatement itself --------------------------------------------------------------------------------------------
def _cpu_case(curve, n, zk, L=24):
    f = cref.scalar_field(curve)
    pts = cref.gen_points(curve, 0x6A00 + curve, L + 1)
    gens, h = pts[:L], pts[L]
    lens = [(L - (i % 3), L - 2 * (i % 2)) for i in range(n)]
    wits, insts, hz = make_inputs(curve, gens, h, n, lens, 0x6A10 + 17 * n, zk, L)
    return f, gens, h, L, wits, insts, hz


@pytest.mark.parametrize("curve,n,zk", [(0, 2, True), (1, 3, True), (0, 3, False), (1, 1, False)])
def test_oracle_accumulator_is_accepted_and_every_corruption_rejected(curve, n, zk):
    f, gens, h, L, wits, insts, hz = _cpu_case(curve, n, zk)
    m = MODULI[f]

    def run(wits_p=wits, zk_p=hz, mu_p=None, nu_p=None, rand_fix=None):
        """prove with the given (possibly corrupted) pieces; the verifier re-derives mu and nu from the transcript"""
        hc = None if hz is None else oracle_hiding_comms(curve, gens, h, [w[0] for w in wits], [w[1] for w in wits], hz)
        mu = mu_list(f, mu_stand_in(f, n)(hc), zk)
        t = cref.tvecs(f, [w[0] for w in wits_p], [w[1] for w in wits_p], to_mont(f, mu_p or mu), L,
                       *(None, None) if zk_p is None else zk_p[:2])
        low = [oracle_commit(curve, gens, h, t[j]) for j in range(n - 1)]
        high = [oracle_commit(curve, gens, h, t[n + j]) for j in range(n - 1)]
        nu = from_mont(f, nu_stand_in(f)(low, high))[0]
        out = oracle_prove(curve, gens, h, L, wits_p, insts, mu_p or mu, nu if nu_p is None else nu_p, zk_p, zk_comm=hz)
        hc2, low2, high2, a_s, b_s, rand, new = out
        if rand_fix is not None:
            rand = rand_fix(rand)
        proof = (hc2, low2, high2)
        return oracle_verify(curve, insts, new, proof, mu, nu) and oracle_decide(curve, gens, h, new, a_s, b_s, rand), (insts, new, proof, mu, nu)

    ok, (_, new, proof, mu, nu) = run()
    assert ok
    # the product-polynomial commitments swapped are rejected by verify
    if n > 1:
        assert not oracle_verify(curve, insts, new, (proof[0], proof[2], proof[1]), mu, nu)
    cases = []
    for i in range(n):
        for side in (0, 1):
            w = [list(x) for x in wits]
            w[i][side] = _flip(w[i][side], 1, side + 1)
            cases.append((f"{'ab'[side]}_{i}", dict(wits_p=[tuple(x) for x in w])))
    for i in range(1, n):
        cases.append((f"mu_{i}", dict(mu_p=[x if j != i else (x + 1) % m for j, x in enumerate(mu)])))
    if n > 1:         # with n = 1, a* = a_0 and b* = b_0 whatever nu is
        cases.append(("nu", dict(nu_p=(nu + 1) % m)))
    if zk:
        for j in range(2):
            z = list(hz); z[j] = _flip(z[j], 3, 0)
            cases.append((f"h{'ab'[j]}", dict(zk_p=tuple(z))))
        for j in range(3):
            z = list(hz); z[2] = _flip(z[2], j, 1)
            cases.append((f"hr{j + 1}", dict(zk_p=tuple(z))))
            for i in range(n):
                w = [list(x) for x in wits]
                w[i][2] = _flip(w[i][2], j, 0)
                cases.append((f"r{j + 1}_{i}", dict(wits_p=[tuple(x) for x in w])))
    for name, kw in cases:
        assert not run(**kw)[0], name


# ---- GPU: the session against the restatement -----------------------------------------------------------------------------
def _ptrs(vecs):
    arr = (C.c_void_p * max(len(vecs), 1))()
    for i, v in enumerate(vecs):
        arr[i] = v.ctypes.data if v.size else None
    return arr


def session_on(c, B, wits, L, hz, hiding_index, count=None):
    """the three steps on context c with the stand-in sponge -> (hiding comms, low, high, a*, b*, mu, nu).  count = (table_c,)
    asserts the launch count of every step"""
    f = cref.scalar_field(B.curve)
    n = len(wits)
    a, b = [w[0] for w in wits], [w[1] for w in wits]
    before = c.kernel_launches()
    sess, hc = c.hp_prove_begin(B, a, b, L, *(None, None) if hz is None else hz[:2], hiding_index=hiding_index,
                                hiding_rand=None if hz is None else hz[2])
    if count is not None:
        tc = count[0]
        assert c.kernel_launches() - before == (0 if hz is None else (1 if L else 0) + plan(L + 1, 3, table_c=tc).launches)
    hcl = None if hc is None else [(hc[0][j], int(hc[1][j])) for j in range(3)]
    mu = mu_list(f, mu_stand_in(f, n)(hcl), hz is not None)
    before = c.kernel_launches()
    (lo, linf), (hi, hinf) = c.hp_prove_product_poly_comm(sess, n, to_mont(f, mu))
    if count is not None:
        assert c.kernel_launches() - before == ((1 + sum(p.launches for p in passes(L, 2 * n - 2, table_c=count[0]))) if L else 0)
    low = [(lo[j], int(linf[j])) for j in range(n - 1)]
    high = [(hi[j], int(hinf[j])) for j in range(n - 1)]
    nu_m = nu_stand_in(f)(low, high)
    before = c.kernel_launches()
    a_s, b_s = c.hp_prove_finish(sess, nu_m, L)
    if count is not None:
        assert c.kernel_launches() - before == int(a_s.shape[0] > 0) + int(b_s.shape[0] > 0)
    return hcl, low, high, a_s, b_s, mu, from_mont(f, nu_m)[0]


def check_session(c, curve, B, pts, n_gens, wits, insts, hz, L, count=None):
    """every output of the session bit for bit against the restatement; returns them"""
    gens, h = pts[:n_gens], pts[n_gens]
    hc, low, high, a_s, b_s, mu, nu = session_on(c, B, wits, L, hz, n_gens, count)
    ohc, olow, ohigh, oa, ob, orand, onew = oracle_prove(curve, gens, h, L, wits, insts, mu, nu, hz)
    if hz is None:
        assert hc is None
    else:
        for j in range(3):
            assert same_point(hc[j], ohc[j]), ("hiding", j)
    for j in range(len(wits) - 1):
        assert same_point(low[j], olow[j]), ("low", j)
        assert same_point(high[j], ohigh[j]), ("high", j)
    assert np.array_equal(a_s, oa) and np.array_equal(b_s, ob)
    assert oracle_decide(curve, gens, h, onew, a_s, b_s, orand)
    return hc, low, high, a_s, b_s


# (curve, n, L, key generators, table bits | None, zk, ragged)
PARITY_CASES = [
    (0, 2, 1 << 16, 1 << 16, "auto", True, False),
    (0, 2, 1 << 16, 1 << 16, "auto", False, False),
    (1, 3, 1 << 16, 1 << 16, "auto", True, True),
    (0, 6, 1 << 16, 1 << 16, "auto", True, True),
    (1, 6, 1 << 16, 1 << 16, "auto", False, False),
    (0, 1, 1 << 16, 1 << 16, "auto", False, False),
    (0, 2, 1 << 20, 1 << 20, 20, True, False),             # the 3-job and 2-job passes over a c = 20 table at full size
    (1, 3, 3000, 5000, None, True, True),                   # Vesta, key longer than len
    (1, 1, 3000, 5000, None, False, True),
    (0, 3, 0, 64, None, True, False),                       # len = 0: the hiding comms are r_j H
    (1, 2, 0, 64, None, False, False),
]


def _lens(n, L, ragged):
    return [(max(L - 37 * i - 5, 0), max(L - 11 * (n - i), 0)) if ragged else (L, L) for i in range(n)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", PARITY_CASES, ids=[f"{'pallas' if c[0] == 0 else 'vesta'}-n{c[1]}-{c[2]}-{'zk' if c[5] else 'plain'}"
                                                     f"{'-ragged' if c[6] else ''}" for c in PARITY_CASES])
def test_session_matches_the_oracle(ctx, case):
    curve, n, L, n_gens, table, zk, ragged = case
    pts = cref.gen_points(curve, 0x6B00 + curve, n_gens + 1)
    B = ctx.register_bases(curve, pts)
    table_c = None
    if table is not None:
        B.precompute(0 if table == "auto" else table)
        table_c = table_window_bits(n_gens + 1, 0 if table == "auto" else table)
    try:
        wits, insts, hz = make_inputs(curve, pts[:n_gens], pts[n_gens], n, _lens(n, L, ragged), 0x6B10 + n, zk, L)
        check_session(ctx, curve, B, pts, n_gens, wits, insts, hz, L, count=(table_c,))
    finally:
        B.release()


def _mirror_case(c, curve, n, L, zk, seed):
    pts = cref.gen_points(curve, seed, L + 1)
    ck = ab.CommitterKey.new(c, curve, pts[:L], pts[L], precompute=True)
    # ragged, but a* and b* of the same length: the mirror's decide commits both over min(|a*|, |b*|)
    lens = [(L, L)] + _lens(n, L, True)[1:]
    wits, insts, hz = make_inputs(curve, pts[:L], pts[L], n, lens, seed + 1, zk, L)
    return pts, ck, wits, insts, hz


@pytest.mark.gpu
@pytest.mark.parametrize("curve,n,zk", [(0, 2, True), (1, 3, True), (0, 6, True), (1, 2, False), (0, 1, False)])
def test_mirror_prove_verify_decide(ctx, curve, n, zk):
    """mirror.ASForHadamardProducts.prove -> verify -> decide accepts, and every corruption is rejected by one of them"""
    f = cref.scalar_field(curve)
    m = MODULI[f]
    L = 2000 + 111 * curve
    pts, ck, wits, insts, hz = _mirror_case(ctx, curve, n, L, zk, 0x6C00 + curve)
    HP = ab.ASForHadamardProducts
    mu_fn, nu_fn = mu_stand_in(f, n), nu_stand_in(f)
    try:
        new, (a_s, b_s, rand), proof = HP.prove(ck, wits, insts, mu_fn, nu_fn, zk=hz)
        assert HP.verify(ck, insts, new, proof, mu_fn, nu_fn)
        assert HP.decide(ck, new, (a_s, b_s, rand))
        # the same as the restatement
        mu = mu_list(f, mu_fn(proof[0]), zk)
        nu = from_mont(f, nu_fn(proof[1], proof[2]))[0]
        _, _, _, oa, ob, orand, onew = oracle_prove(curve, pts[:L], pts[L], L, wits, insts, mu, nu, hz)
        assert np.array_equal(a_s, oa) and np.array_equal(b_s, ob) and all(same_point(x, y) for x, y in zip(new, onew))
        assert (rand is None) == (orand is None) and (rand is None or np.array_equal(np.array(rand), orand))

        def rejected(wits_p=wits, mu_p=mu_fn, nu_p=nu_fn, post=None):
            nw, (pa, pb, pr), pf = HP.prove(ck, wits_p, insts, mu_p, nu_p, zk=hz)
            if post is not None:
                nw, pa, pb, pr, pf = post(nw, pa, pb, pr, pf)
            return not (HP.verify(ck, insts, nw, pf, mu_fn, nu_fn) and HP.decide(ck, nw, (pa, pb, pr)))

        for i in range(n):
            for side in (0, 1):
                w = [list(x) for x in wits]
                w[i][side] = _flip(w[i][side], 0, 1)
                assert rejected(wits_p=[tuple(x) for x in w]), (side, i)
        for i in range(n - 1):
            def bad_mu(hc, i=i):
                v = np.array(mu_fn(hc), dtype=np.uint64).reshape(-1, 4)
                return to_mont(f, [x + (j == i) for j, x in enumerate(from_mont(f, v))])
            assert rejected(mu_p=bad_mu), ("mu", i + 1)
        if n > 1:
            assert rejected(nu_p=lambda lo, hi: to_mont(f, [from_mont(f, nu_fn(lo, hi))[0] + 1]).reshape(4)), "nu"
            assert rejected(post=lambda nw, pa, pb, pr, pf: (nw, pa, pb, pr, (pf[0], pf[2], pf[1]))), "low/high swapped"
        assert rejected(post=lambda nw, pa, pb, pr, pf: (nw, _flip(pa, 0, 0), pb, pr, pf)), "a*"
        assert rejected(post=lambda nw, pa, pb, pr, pf: (nw, pa, _flip(pb, 1, 0), pr, pf)), "b*"
        if zk:
            for j in range(3):
                w = [list(x) for x in wits]
                w[n - 1][2] = _flip(w[n - 1][2], j, 0)
                assert rejected(wits_p=[tuple(x) for x in w]), ("r", j)
                assert rejected(post=lambda nw, pa, pb, pr, pf, j=j: (nw, pa, pb, [_flip(np.array(pr), j, 0)[j] if k == j else pr[k]
                                                                               for k in range(3)], pf)), ("r*", j)
                # hiding comm j replaced by the next one in the proof
                assert rejected(post=lambda nw, pa, pb, pr, pf, j=j: (nw, pa, pb, pr, ([pf[0][(k + 1) % 3] if k == j else pf[0][k]
                                                                                          for k in range(3)], pf[1], pf[2]))), ("hiding comm", j)
    finally:
        ck.bases.release()


def _group_scenarios(c1, cg, curve, n_gens, seed):
    """zk and plain, n = 2, 3, 6, ragged lengths ending inside different shards: the group gives the single context's outputs
    bit for bit, and both the oracle's"""
    L = 3000
    pts = cref.gen_points(curve, seed, n_gens + 1)
    B1, Bg = c1.register_bases(curve, pts), cg.register_bases(curve, pts)
    try:
        for n, zk in [(2, True), (3, False), (6, True), (1, False)]:
            wits, insts, hz = make_inputs(curve, pts[:n_gens], pts[n_gens], n, _lens(n, L, True), seed + n, zk, L)
            r1 = check_session(c1, curve, B1, pts, n_gens, wits, insts, hz, L)
            rg = check_session(cg, curve, Bg, pts, n_gens, wits, insts, hz, L)
            for x, y in zip(r1, rg):
                if isinstance(x, np.ndarray):
                    assert np.array_equal(x, y), (n, zk)
                elif x is not None:
                    assert all(np.array_equal(p[0], q[0]) and p[1] == q[1] for p, q in zip(x, y)), (n, zk)
        # len = 0 with zk: the hiding comms are r_j H, from the child that owns H alone
        wits, insts, hz = make_inputs(curve, pts[:n_gens], pts[n_gens], 2, [(0, 0), (0, 0)], seed + 50, True, 0)
        h1 = check_session(c1, curve, B1, pts, n_gens, wits, insts, hz, 0)[0]
        hg = check_session(cg, curve, Bg, pts, n_gens, wits, insts, hz, 0)[0]
        assert all(np.array_equal(p[0], q[0]) and p[1] == q[1] for p, q in zip(h1, hg))
    finally:
        B1.release(); Bg.release()


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0]])
@pytest.mark.parametrize("long_key", [False, True])
def test_group_is_bit_identical(ctx, devices, long_key):
    """columns cut along the key's point ranges; with a key four times longer than len every column sits on child 0 and the
    last child owns only the hiding generator"""
    curve = 1 if long_key else 0
    g = ab.Context(devices=devices, min_shard=16)
    try:
        _group_scenarios(ctx, g, curve, 12000 if long_key else 3000, 0x6D00 + curve)
    finally:
        g.close()


@pytest.fixture(scope="module")
def no_peer_group():
    with pytest.MonkeyPatch.context() as mp:
        mp.setenv("ACCMSM_NO_PEER", "1")
        c = ab.Context(devices=[0, 0, 0], min_shard=16)
    yield c
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("long_key", [False, True])
def test_group_without_peer_access_is_bit_identical(ctx, no_peer_group, long_key):
    curve = 0 if long_key else 1
    _group_scenarios(ctx, no_peer_group, curve, 12000 if long_key else 3000, 0x6D40 + curve)


@pytest.mark.gpu
def test_calls_between_the_steps_and_two_live_sessions(ctx):
    """an msm and an hp_decide (both through the ctx's scalar buffer) between every two steps, and two sessions interleaved"""
    curve, L = 0, 5000
    f = cref.scalar_field(curve)
    pts = cref.gen_points(curve, 0x6E00, L + 1)
    B = ctx.register_bases(curve, pts)
    other_pts = cref.gen_points(curve, 0x6E01, 2 * L)
    other = ctx.register_bases(curve, other_pts)
    try:
        w1, i1, z1 = make_inputs(curve, pts[:L], pts[L], 3, _lens(3, L, True), 0x6E10, True, L)
        w2, i2, z2 = make_inputs(curve, pts[:L], pts[L], 2, _lens(2, L, False), 0x6E20, True, L)
        big = cref.gen_scalars(f, 0x6E30, 2 * L, True)
        exp_msm = cref.commit(curve, other_pts, big)

        def noise():
            assert same_point(ctx.msm(other, big), exp_msm)
            ok, _, _ = ctx.hp_decide(other, big, big[::-1].copy(), np.zeros((3, 8), np.uint64), np.zeros(3, np.uint8), hiding_index=0,
                                     randomness=cref.gen_scalars(f, 1, 3, True))
            assert not ok

        states = {}
        for k, (w, z) in enumerate(((w1, z1), (w2, z2))):
            sess, hc = ctx.hp_prove_begin(B, [x[0] for x in w], [x[1] for x in w], L, z[0], z[1], hiding_index=L, hiding_rand=z[2])
            states[k] = (sess, [(hc[0][j], int(hc[1][j])) for j in range(3)], w, z)
            noise()
        got = {}
        for k in (1, 0):
            sess, hc, w, z = states[k]
            n = len(w)
            mu = mu_list(f, mu_stand_in(f, n)(hc), True)
            (lo, linf), (hi, hinf) = ctx.hp_prove_product_poly_comm(sess, n, to_mont(f, mu))
            noise()
            got[k] = (hc, [(lo[j], int(linf[j])) for j in range(n - 1)], [(hi[j], int(hinf[j])) for j in range(n - 1)], mu)
        for k in (0, 1):
            sess, _, w, z = states[k]
            hc, low, high, mu = got[k]
            nu_m = nu_stand_in(f)(low, high)
            a_s, b_s = ctx.hp_prove_finish(sess, nu_m, L)
            noise()
            ins = i1 if k == 0 else i2
            ohc, olow, ohigh, oa, ob, _, _ = oracle_prove(curve, pts[:L], pts[L], L, w, ins, mu, from_mont(f, nu_m)[0], z)
            assert all(same_point(x, y) for x, y in zip(hc + low + high, ohc + olow + ohigh)), k
            assert np.array_equal(a_s, oa) and np.array_equal(b_s, ob), k
    finally:
        B.release(); other.release()


def _rc_begin(c, key, a, b, n, L, ha=None, hb=None, hiding=0, hr=None, out=True, sess=True):
    p = lambda v: None if v is None else v.ctypes.data_as(C.c_void_p)
    al = np.array([v.shape[0] for v in a], dtype=np.uint64)
    bl = np.array([v.shape[0] for v in b], dtype=np.uint64)
    xy, inf, s = np.zeros((3, 8), np.uint64), np.zeros(3, np.uint8), C.c_uint64(0)
    rc = c._lib.accmsm_hp_prove_begin(c._h, C.c_uint64(key), _ptrs(a), p(al), _ptrs(b), p(bl), C.c_int(n), C.c_size_t(L), p(ha), p(hb),
                                      C.c_size_t(hiding), p(hr), p(xy) if out else None, p(inf) if out else None,
                                      C.byref(s) if sess else None)
    return rc, int(s.value)


def _rc_ppc(c, sess, mu, n_out):
    p = lambda v: v.ctypes.data_as(C.c_void_p)
    lo, hi = np.zeros((max(n_out, 1), 8), np.uint64), np.zeros((max(n_out, 1), 8), np.uint64)
    li, hf = np.zeros(max(n_out, 1), np.uint8), np.zeros(max(n_out, 1), np.uint8)
    return c._lib.accmsm_hp_prove_product_poly_comm(c._h, C.c_uint64(sess), p(mu), C.c_size_t(mu.shape[0]), p(lo), p(li), p(hi), p(hf))


def _rc_finish(c, sess, nu, cap):
    a, b = np.zeros((max(cap, 1), 4), np.uint64), np.zeros((max(cap, 1), 4), np.uint64)
    ol = (C.c_size_t * 2)()
    rc = c._lib.accmsm_hp_prove_finish(c._h, C.c_uint64(sess), nu.ctypes.data_as(C.c_void_p), a.ctypes.data_as(C.c_void_p),
                                       b.ctypes.data_as(C.c_void_p), C.c_size_t(cap), ol)
    return rc, (ol[0], ol[1])


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_argument_order_and_handle_errors(ctx, devices):
    c = ctx if devices is None else ab.Context(devices=devices, min_shard=16)
    curve, L = 0, 64
    f = cref.scalar_field(curve)
    pts = cref.gen_points(curve, 0x6F00, L + 1)
    B = c.register_bases(curve, pts)
    try:
        wits, insts, hz = make_inputs(curve, pts[:L], pts[L], 3, _lens(3, L, True), 0x6F10, True, L)
        a, b = [w[0] for w in wits], [w[1] for w in wits]
        ha, hb, hr = hz
        kw = dict(key=B.handle, a=a, b=b, n=3, L=L, ha=ha, hb=hb, hiding=L, hr=hr)
        rc = lambda **o: _rc_begin(c, **{**kw, **o})
        # begin: counts, one-sided hiding, hiding with n = 1, vectors longer than len, ranges beyond the key, null pointers
        assert rc(n=0)[0] == E_ARG and rc(a=a * 6, b=b * 6, n=18)[0] == E_ARG
        assert rc(hb=None)[0] == E_ARG and rc(ha=None)[0] == E_ARG
        assert rc(a=a[:1], b=b[:1], n=1)[0] == E_ARG
        assert rc(L=40)[0] == E_ARG and rc(L=L + 2)[0] == E_ARG and rc(hiding=L + 1)[0] == E_ARG
        assert rc(hr=None)[0] == E_ARG and rc(out=False)[0] == E_ARG and rc(sess=False)[0] == E_ARG
        assert rc(key=987654)[0] == E_HANDLE
        # a session that survives its argument errors
        r0, s = rc()
        assert r0 == 0
        mu = to_mont(f, mu_list(f, mu_stand_in(f, 3)(None), True))
        nu = to_mont(f, [12345]).reshape(4)
        assert _rc_finish(c, 987654, nu, L)[0] == E_HANDLE
        assert _rc_ppc(c, 987654, mu, 2) == E_HANDLE
        assert _rc_ppc(c, s, mu[:3], 2) == E_ARG and _rc_ppc(c, s, np.concatenate([mu, mu[:1]]), 2) == E_ARG   # wrong mu count
        assert _rc_ppc(c, s, mu, 2) == 0
        assert _rc_ppc(c, s, mu, 2) == E_ARG                            # twice
        assert _rc_finish(c, s, nu, L - 1) == (E_ARG, (L, L))           # too small: released anyway
        assert _rc_ppc(c, s, mu, 2) == E_HANDLE and _rc_finish(c, s, nu, L)[0] == E_HANDLE
        # finish before product_poly_comm: E_ARG, released
        r0, s = rc()
        assert r0 == 0 and _rc_finish(c, s, nu, L)[0] == E_ARG and c._lib.accmsm_hp_prove_abort(c._h, C.c_uint64(s)) == E_HANDLE
        # abort
        r0, s = rc(ha=None, hb=None, hr=None)
        assert r0 == 0 and c._lib.accmsm_hp_prove_abort(c._h, C.c_uint64(s)) == 0
        assert _rc_ppc(c, s, mu[:3], 2) == E_HANDLE and c._lib.accmsm_hp_prove_abort(c._h, C.c_uint64(s)) == E_HANDLE
        # the context still works
        check_session(c, curve, B, pts, L, wits, insts, hz, L)
    finally:
        B.release()
        if c is not ctx:
            c.close()


@pytest.mark.gpu
def test_prove_cycles_leave_device_memory_where_it_was(ctx):
    import torch
    curve, n, L = 0, 3, 1 << 15
    f = cref.scalar_field(curve)
    pts, ck, wits, insts, hz = _mirror_case(ctx, curve, n, L, True, 0x6F40)
    HP = ab.ASForHadamardProducts
    try:
        mu_fn, nu_fn = mu_stand_in(f, n), nu_stand_in(f)
        first = HP.prove(ck, wits, insts, mu_fn, nu_fn, zk=hz)
        torch.cuda.synchronize(0)
        free0 = torch.cuda.mem_get_info(0)[0]
        for _ in range(20):
            new, wit, proof = HP.prove(ck, wits, insts, mu_fn, nu_fn, zk=hz)
        torch.cuda.synchronize(0)
        free1 = torch.cuda.mem_get_info(0)[0]
        assert free0 - free1 <= (8 << 20), (free0, free1)
        assert np.array_equal(wit[0], first[1][0]) and HP.decide(ck, new, wit)
    finally:
        ck.bases.release()
