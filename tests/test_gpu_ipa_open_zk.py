"""GPU tests of the zero-knowledge IpaPC opening (MakeZK::Enabled): accmsm_ipa_open_hide / accmsm_ipa_open_hiding_challenge.

Before its first round upstream's open_individual_opening_challenges draws a random polynomial, shifts it to vanish at
the point (hiding[0] -= hiding(z)), commits to it as hiding_comm = cm_commit(key, hiding', s, rho), squeezes alpha from
hiding_comm and opens P' = P + alpha hiding'; the verifier rebuilds C' = C + alpha hiding_comm - (r + alpha rho) s.
The oracle here is composed from existing reference primitives: poly_evaluate, commit, combine_vectors and the
round-by-round opening.  Every hiding_comm, (l, r), final key and c is bit-exact with it, on the single-device ctx and on
virtual (and, with >= 2 GPUs, real) device groups."""
import ctypes as C
import hashlib

import numpy as np
import pytest

import accumulation_b200 as ab
from accumulation_b200.mirror import _MODULI, _fe_to_int, _int_to_fe
from oracle import cref
from tests.test_gpu_ipa_open import oracle_open, sponge_stand_in
from tests.util import same_point

pytestmark = pytest.mark.gpu

E_ARG, E_HANDLE = -2, -3


def _device_lists():
    lists = [[0, 0], [0, 0, 0], [0, 0, 0, 0]]
    try:
        import torch
        if torch.cuda.device_count() >= 2:
            lists.append(list(range(min(torch.cuda.device_count(), 8))))
    except Exception:
        pass
    return lists


@pytest.fixture(scope="module", params=_device_lists(), ids=lambda d: "dev" + "".join(map(str, d)))
def gctx(request):
    """min_shard = 0: every opening of 2^k >= 2 coefficients is sharded over the largest power of two <= children"""
    c = ab.Context(devices=request.param, min_shard=0)
    yield c
    c.close()


def alpha_of(sf):
    """host stand-in for the sponge over (C, z, v, hiding_comm)"""
    def alpha(hiding_comm):
        h = hashlib.blake2s(b"zk-alpha")
        h.update(np.asarray(hiding_comm[0], dtype=np.uint64).tobytes()); h.update(bytes([int(hiding_comm[1])]))
        return _int_to_fe(sf, int.from_bytes(h.digest()[:16], "little") | 1)
    return alpha


class Case:
    """one zk opening: key = generators || h || s, P = the combined succinct-check polynomial, its commitment C with
    randomness r, the hiding polynomial and rho"""

    def __init__(self, curve, k, n_hiding=None, seed=900):
        self.curve, self.k, self.n = curve, k, 1 << k
        sf = self.sf = cref.scalar_field(curve)
        n = self.n
        pts = cref.gen_points(curve, seed + k, n + 2)
        self.key, self.h, self.s = pts[:n], pts[n], pts[n + 1]
        self.all = pts
        m = 2
        self.chm = cref.gen_scalars(sf, seed + 1, m * k, True).reshape(m, k, 4)
        self.al = cref.gen_scalars(sf, seed + 2, m, True)
        self.rp = cref.gen_scalars(sf, seed + 3, min(3, n), True)      # the random linear polynomial fits 2^k (k = 1: 2)
        self.P = cref.combine_check_polys(sf, self.chm, self.al, self.rp)
        self.z = cref.gen_scalars(sf, seed + 4, 1, True).reshape(4)
        self.xi0 = cref.gen_scalars(sf, seed + 5, 1, True).reshape(4)
        self.hp, inf = cref.point_mul(curve, self.h, 0, cref.from_mont(sf, self.xi0.reshape(1, 4)).reshape(4))
        assert inf == 0
        self.hiding = cref.gen_scalars(sf, seed + 6, n if n_hiding is None else n_hiding, True)
        self.rho = cref.gen_scalars(sf, seed + 7, 1, True).reshape(4)
        self.r = cref.gen_scalars(sf, seed + 8, 1, True).reshape(4)
        self.C = cref.commit(curve, self.key, self.P, self.s, self.r)
        self.squeeze = sponge_stand_in(sf)
        self.alpha_fn = alpha_of(sf)
        self._oracle = None

    def oracle(self):
        """-> dict of the oracle's hiding', hiding_comm, alpha, P', rand, C' and the proof"""
        if self._oracle is None:
            sf, n = self.sf, self.n
            hid = np.zeros((n, 4), np.uint64)
            hid[: self.hiding.shape[0]] = self.hiding
            e = cref.poly_evaluate(sf, hid, self.z)
            hid[0] = cref.fe_sub(sf, hid[0], e)
            hc = cref.commit(self.curve, self.key, hid, self.s, self.rho)
            alpha = self.alpha_fn(hc)
            P2 = cref.combine_vectors(sf, [self.P, hid], np.stack([_int_to_fe(sf, 1), alpha]))
            rand = _int_to_fe(sf, _fe_to_int(sf, self.r) + _fe_to_int(sf, alpha) * _fe_to_int(sf, self.rho))
            m = _MODULI[sf]
            t1 = cref.point_mul(self.curve, hc[0], hc[1], cref.from_mont(sf, alpha.reshape(1, 4)).reshape(4))
            t2 = cref.point_mul(self.curve, self.s, 0, cref.from_mont(sf, _int_to_fe(sf, m - _fe_to_int(sf, rand)).reshape(1, 4)).reshape(4))
            cp = cref.point_add(self.curve, *cref.point_add(self.curve, self.C[0], self.C[1], *t1), *t2)
            proof = oracle_open(self.curve, self.key, P2, self.z, self.hp, self.squeeze)
            self._oracle = dict(hiding=hid, hc=hc, alpha=alpha, P2=P2, rand=rand, C2=cp, proof=proof)
        return self._oracle


def run_zk(c, B, case, combined, by_index, n_hiding=None):
    """begin / begin_combined -> hide -> alpha -> hiding_challenge -> (xi_0 by index) -> rounds -> finish"""
    if combined:
        sess, ev = c.ipa_open_begin_combined(B, case.chm, case.al, case.z, None if by_index else case.hp, case.rp)
    else:
        sess, ev = c.ipa_open_begin(B, case.P, case.k, case.z, None if by_index else case.hp), None
    hc = c.ipa_open_hide(sess, case.hiding, case.n + 1, case.rho)
    alpha = case.alpha_fn(hc)
    c.ipa_open_hiding_challenge(sess, alpha)
    if by_index:
        c.ipa_open_use_hiding_generator(sess, case.n, case.xi0)
    l_vec, r_vec, chs, xi = [], [], [], None
    lr = c.ipa_open_round(sess) if case.k else None
    while lr is not None:
        l, r = lr
        xi = np.ascontiguousarray(case.squeeze(xi, l, r), dtype=np.uint64).reshape(4)
        l_vec.append(l); r_vec.append(r); chs.append(xi)
        lr = c.ipa_open_fold_round(sess, xi)
    fk, cc = c.ipa_open_finish(sess)
    return dict(hc=hc, alpha=alpha, ev=ev, proof=(l_vec, r_vec, fk, cc, chs))


def same_proof(a, b):
    return (len(a[0]) == len(b[0]) and all(same_point(x, y) for x, y in zip(a[0] + a[1], b[0] + b[1]))
            and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3]) and all(np.array_equal(x, y) for x, y in zip(a[4], b[4])))


def assert_matches_oracle(case, got):
    o = case.oracle()
    assert same_point(got["hc"], o["hc"])
    assert np.array_equal(got["alpha"], o["alpha"])
    el, er, efk, ec, echs = o["proof"]
    gl, gr, gfk, gc, gchs = got["proof"]
    assert len(gl) == case.k
    assert all(same_point(x, y) for x, y in zip(gl + gr, el + er))
    assert all(np.array_equal(x, y) for x, y in zip(gchs, echs))
    assert np.array_equal(gfk, efk) and np.array_equal(gc, ec)
    if got["ev"] is not None:      # the hiding polynomial vanishes at z: P'(z) = P(z)
        assert np.array_equal(got["ev"], cref.poly_evaluate(case.sf, o["P2"], case.z).reshape(4))


_CASES = {}


def case_for(curve, k, n_hiding):
    key = (curve, k, n_hiding)
    if key not in _CASES:
        _CASES[key] = Case(curve, k, n_hiding)
    return _CASES[key]


@pytest.mark.parametrize("curve", [0, 1])
@pytest.mark.parametrize("k,n_hiding,precompute,fold", [
    (1, None, False, False), (5, 3, True, False), (10, None, False, False), (10, None, True, False),
    (13, None, True, True), (13, None, False, False)])
def test_zk_open_parity(ctx, curve, k, n_hiding, precompute, fold):
    """begin and begin_combined, h' as a point and by index: hiding_comm, every (l, r), the final key and c equal the
    oracle; C' equals the plain commitment to P' (which ties rand to the commitment); the 2k + 5 term succinct-check
    equation and check_final_key accept"""
    case = case_for(curve, k, n_hiding)
    ck = ab.CommitterKey.new(ctx, curve, case.key, case.h, precompute=precompute, s_xy=case.s)
    assert ck.s_index == case.n + 1
    if fold:
        ctx.set_ipa_fold(5, 11)       # 2^13 -> 2^8 on a materialised key (needs the window table)
    else:
        ctx.set_ipa_fold(0, 11)
    try:
        runs = [run_zk(ctx, ck.bases, case, combined, by_index) for combined in (False, True) for by_index in (False, True)]
    finally:
        ctx.set_ipa_fold()
    o = case.oracle()
    for got in runs:
        assert_matches_oracle(case, got)
    got = runs[-1]
    l_vec, r_vec, fk, c, chs = got["proof"]
    # C' from the library's hiding_comm and rand equals the non-hiding commitment to P'
    c2 = ab.InnerProductArgPC.hiding_commitment(ck, case.C, got["hc"], got["alpha"], o["rand"])
    assert same_point(c2, cref.commit(curve, case.key, o["P2"]))
    assert same_point(c2, o["C2"])
    v = cref.poly_evaluate(case.sf, case.P, case.z).reshape(4)
    assert cref.ipa_succinct_check(curve, c2, case.z, v, np.array([p[0] for p in l_vec]), np.array([p[0] for p in r_vec]),
                                   np.array(chs), case.hp, fk, c)
    hid = (got["hc"], got["alpha"], o["rand"], case.s)
    args = (case.C, case.z, v, l_vec, r_vec, np.array(chs), case.hp, fk, c)
    assert ab.InnerProductArgPC.succinct_check_equation(ctx, curve, *args, hid)
    assert ab.InnerProductArgPC.check_final_key(ck, np.array(chs), fk, 0)
    ck.bases.release()


@pytest.mark.parametrize("curve", [0, 1])
def test_zk_succinct_check_rejects_and_mixed_batch(ctx, curve):
    """a flipped rand, hiding_comm or alpha is rejected; a mixed zk / non-zk batch is one call with the expected verdicts"""
    case = case_for(curve, 5, 3)
    o = case.oracle()
    sf, m = case.sf, _MODULI[case.sf]
    l_vec, r_vec, fk, c, chs = o["proof"]
    v = cref.poly_evaluate(sf, case.P, case.z).reshape(4)
    args = (case.C, case.z, v, l_vec, r_vec, np.array(chs), case.hp, fk, c)
    good = (o["hc"], o["alpha"], o["rand"], case.s)
    bump = lambda x: _int_to_fe(sf, (_fe_to_int(sf, x) + 1) % m)
    bad_rand = (o["hc"], o["alpha"], bump(o["rand"]), case.s)
    bad_hc = ((case.key[0], 0), o["alpha"], o["rand"], case.s)
    bad_alpha = (o["hc"], bump(o["alpha"]), o["rand"], case.s)
    eq = ab.InnerProductArgPC.succinct_check_equation
    assert eq(ctx, curve, *args, good)
    for bad in (bad_rand, bad_hc, bad_alpha):
        assert not eq(ctx, curve, *args, bad)
    assert not eq(ctx, curve, *args)                     # C itself is not what the zk proof opens
    plain = (o["C2"],) + args[1:]                        # ... C' is, as a non-hiding instance
    assert eq(ctx, curve, *plain)
    batch = [args + (good,), plain, args + (bad_rand,), args, plain + (None,), args + (bad_alpha,)]
    assert ab.InnerProductArgPC.succinct_check_equations(ctx, curve, batch) == [True, True, False, False, True, False]


@pytest.mark.parametrize("curve", [0, 1])
def test_zk_open_mirror(ctx, curve):
    """InnerProductArgPC.open with ZkHiding, xi_0 squeezed from C' (a callable): the oracle's proof for that xi_0"""
    case = case_for(curve, 10, None)
    ck = ab.CommitterKey.new(ctx, curve, case.key, case.h, s_xy=case.s)
    seen = {}

    def xi0_of(c_prime):
        seen["C2"] = c_prime
        return case.xi0
    hz = ab.ZkHiding(coeffs=case.hiding, rand=case.rho, comm=case.C, comm_rand=case.r, alpha=case.alpha_fn)
    l_vec, r_vec, fk, c, chs, hc, rand = ab.InnerProductArgPC.open(ck, case.P, case.z, None, case.squeeze, log_d=case.k, xi0=xi0_of,
                                                                   hiding=hz)
    o = case.oracle()
    assert same_point(hc, o["hc"]) and np.array_equal(rand, o["rand"])
    assert same_point(seen["C2"], o["C2"])
    assert_matches_oracle(case, dict(hc=hc, alpha=o["alpha"], ev=None, proof=(l_vec, r_vec, fk, c, chs)))
    ck.bases.release()


def _G(gctx, k):
    G = 1
    while 2 * G <= gctx.device_count() and 2 * G <= (1 << k):
        G *= 2
    return G


def _launches(gctx):
    return [gctx.device_ctx(i).kernel_launches() for i in range(gctx.device_count())]


@pytest.mark.parametrize("curve", [0, 1])
@pytest.mark.parametrize("k,n_hiding,precompute", [(1, None, False), (5, 3, True), (10, None, True), (13, None, False)])
def test_zk_group_parity(ctx, gctx, curve, k, n_hiding, precompute):
    """sharded over the children (child c commits hiding[c::G] over key[c::G]; (s, rho) rides on child s_index mod G) and
    unsharded (min_shard above 2^k / 2: child 0): the same hiding_comm and proof as the single-device ctx and the oracle"""
    case = case_for(curve, k, n_hiding)
    B = gctx.register_bases(curve, case.all)
    Bs = ctx.register_bases(curve, case.all)
    if precompute:
        B.precompute(); Bs.precompute()
    try:
        G = _G(gctx, k)
        for combined, by_index in ((False, False), (True, True), (True, False)):
            before = _launches(gctx)
            got = run_zk(gctx, B, case, combined, by_index)
            after = _launches(gctx)
            assert all(after[i] > before[i] for i in range(G)), (before, after)
            one = run_zk(ctx, Bs, case, combined, by_index)
            assert same_point(got["hc"], one["hc"]) and same_proof(got["proof"], one["proof"])
            assert_matches_oracle(case, got)
            if combined:
                assert np.array_equal(got["ev"], one["ev"])
        gctx.set_min_shard(case.n // 2 + 1)
        try:
            before = _launches(gctx)
            got = run_zk(gctx, B, case, True, True)
            after = _launches(gctx)
        finally:
            gctx.set_min_shard(0)
        assert after[0] > before[0] and after[1:] == before[1:]
        assert_matches_oracle(case, got)
        fk, chs = got["proof"][2], got["proof"][4]
        assert ab.InnerProductArgPC.check_final_key(ab.CommitterKey(B, case.n), np.array(chs), fk, 0)
    finally:
        B.release(); Bs.release()


def _hide_rc(c, sess, coeffs, s_index, rho):
    cf = np.ascontiguousarray(coeffs, dtype=np.uint64).reshape(-1, 4)
    out, inf = np.empty(8, np.uint64), C.c_uint8(0)
    return c._lib.accmsm_ipa_open_hide(c._h, C.c_uint64(sess), cf.ctypes.data_as(C.c_void_p) if cf.shape[0] else None,
                                       C.c_size_t(cf.shape[0]), C.c_size_t(s_index), np.ascontiguousarray(rho).ctypes.data_as(C.c_void_p),
                                       out.ctypes.data_as(C.c_void_p), C.byref(inf))


def _challenge_rc(c, sess, alpha):
    return c._lib.accmsm_ipa_open_hiding_challenge(c._h, C.c_uint64(sess), np.ascontiguousarray(alpha).ctypes.data_as(C.c_void_p))


def _round_rc(c, sess):
    l, r, li, ri = np.empty(8, np.uint64), np.empty(8, np.uint64), C.c_uint8(0), C.c_uint8(0)
    return c._lib.accmsm_ipa_open_round(c._h, C.c_uint64(sess), l.ctypes.data_as(C.c_void_p), C.byref(li),
                                        r.ctypes.data_as(C.c_void_p), C.byref(ri))


def _order_errors(c, B, case):
    """every order / argument error is ACCMSM_E_ARG; a session refused a round before its hiding challenge still gives the
    oracle's proof once the challenge is applied"""
    alpha = case.alpha_fn(case.oracle()["hc"])
    # hiding_challenge without hide
    sess = c.ipa_open_begin(B, case.P, case.k, case.z, case.hp)
    assert _challenge_rc(c, sess, alpha) == E_ARG
    # too long a hiding polynomial, s beyond the key
    assert _hide_rc(c, sess, np.zeros((case.n + 1, 4), np.uint64), case.n + 1, case.rho) == E_ARG
    assert _hide_rc(c, sess, case.hiding, case.n + 2, case.rho) == E_ARG
    # hide, then hide again; round before the challenge; challenge twice
    assert _hide_rc(c, sess, case.hiding, case.n + 1, case.rho) == 0
    assert _hide_rc(c, sess, case.hiding, case.n + 1, case.rho) == E_ARG
    assert _round_rc(c, sess) == E_ARG
    assert _challenge_rc(c, sess, alpha) == 0
    assert _challenge_rc(c, sess, alpha) == E_ARG
    l_vec, r_vec, chs, xi = [], [], [], None
    lr = c.ipa_open_round(sess)
    # hide after the first round
    assert _hide_rc(c, sess, case.hiding, case.n + 1, case.rho) == E_ARG
    while lr is not None:
        l, r = lr
        xi = np.ascontiguousarray(case.squeeze(xi, l, r), dtype=np.uint64).reshape(4)
        l_vec.append(l); r_vec.append(r); chs.append(xi)
        lr = c.ipa_open_fold_round(sess, xi)
    fk, cc = c.ipa_open_finish(sess)
    el, er, efk, ec, _ = case.oracle()["proof"]
    assert all(same_point(x, y) for x, y in zip(l_vec + r_vec, el + er))
    assert np.array_equal(fk, efk) and np.array_equal(cc, ec)


def test_zk_errors(ctx):
    case = case_for(0, 5, 3)
    B = ctx.register_bases(0, case.all)
    try:
        _order_errors(ctx, B, case)
        # a session begun as one cyclic shard (log_shards > 0) cannot be hidden
        sess = ctx.ipa_open_begin_shard(B, case.P[::2], case.k - 1, case.z, case.hp, 0, 1)
        assert _hide_rc(ctx, sess, case.hiding[::2], case.n + 1, case.rho) == E_ARG
        fk, c = np.empty(8, np.uint64), np.empty(4, np.uint64)
        ctx._lib.accmsm_ipa_open_finish(ctx._h, C.c_uint64(sess), fk.ctypes.data_as(C.c_void_p), c.ctypes.data_as(C.c_void_p))
    finally:
        B.release()


def test_zk_group_errors(gctx):
    case = case_for(0, 5, 3)
    B = gctx.register_bases(0, case.all)
    try:
        _order_errors(gctx, B, case)
        gctx.set_min_shard(case.n)           # unsharded: forwarded to child 0
        try:
            _order_errors(gctx, B, case)
        finally:
            gctx.set_min_shard(0)
    finally:
        B.release()


def test_zk_open_repeatable_and_no_leak(ctx, gctx):
    """repeated hide / finish cycles give the same bits and do not grow device memory"""
    import torch
    case = case_for(1, 13, None)
    ck = ab.CommitterKey.new(ctx, 1, case.key, case.h, precompute=True, s_xy=case.s)
    B = gctx.register_bases(1, case.all)
    B.precompute()
    try:
        first = run_zk(ctx, ck.bases, case, True, True)
        gfirst = run_zk(gctx, B, case, True, True)
        assert same_proof(first["proof"], gfirst["proof"])
        torch.cuda.synchronize(0)
        free0 = torch.cuda.mem_get_info(0)[0]
        for _ in range(3):
            assert same_proof(run_zk(ctx, ck.bases, case, True, True)["proof"], first["proof"])
            assert same_proof(run_zk(gctx, B, case, True, True)["proof"], first["proof"])
        torch.cuda.synchronize(0)
        free1 = torch.cuda.mem_get_info(0)[0]
        assert free0 - free1 <= (8 << 20), (free0, free1)
    finally:
        ck.bases.release(); B.release()
