"""GPU tests of IpaPC::open sessions sharded across the children of a device group (accmsm_init_multi; multi_api.inc).
The plain session calls (accmsm_ipa_open_begin / _begin_combined / _round / _fold / _fold_round / _finish) on a group
ctx run the opening cyclically sharded over G = 2^g children whenever 2^k / G >= min_shard: child c holds key[c::G] and
coeffs[c::G] for the first k - g rounds, child 0 runs the last g rounds over the children's (final key, coefficient)
pairs.  Every (l, r), the final key and c are bit-exact with the oracle's round-by-round opening and with the
single-device ctx.

On a single-GPU box the groups list device 0 several times (virtual groups: every path of the group layer runs, only
the NVLink hop is local); with >= 2 GPUs a real group over every device is added."""
import ctypes as C

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


def _G(gctx, k):
    G = 1
    while 2 * G <= gctx.device_count() and 2 * G <= (1 << k):
        G *= 2
    return G


def _inv(sf, xi):
    return _int_to_fe(sf, pow(_fe_to_int(sf, xi), -1, _MODULI[sf]))


def _drive(c, sess, k, squeeze, sf, separate=False):
    """the prover's loop: fold_round per round, or round + fold as two calls"""
    l_vec, r_vec, chs, xi = [], [], [], None
    lr = c.ipa_open_round(sess) if k else None
    while lr is not None:
        l, r = lr
        xi = np.ascontiguousarray(squeeze(xi, l, r), dtype=np.uint64).reshape(4)
        l_vec.append(l); r_vec.append(r); chs.append(xi)
        if separate:
            c.ipa_open_fold(sess, xi, _inv(sf, xi))
            lr = c.ipa_open_round(sess) if len(l_vec) < k else None
        else:
            lr = c.ipa_open_fold_round(sess, xi)
    fk, cc = c.ipa_open_finish(sess)
    return l_vec, r_vec, fk, cc, chs


def _same_proof(a, b):
    return (len(a[0]) == len(b[0]) and all(same_point(x, y) for x, y in zip(a[0] + a[1], b[0] + b[1]))
            and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3]) and all(np.array_equal(x, y) for x, y in zip(a[4], b[4])))


def _launches(gctx):
    return [gctx.device_ctx(i).kernel_launches() for i in range(gctx.device_count())]


_ORACLE = {}


def _oracle(curve, key, coeffs, z, hp, squeeze, tag):
    if tag not in _ORACLE:
        _ORACLE[tag] = oracle_open(curve, key, coeffs, z, hp, squeeze)
    return _ORACLE[tag]


@pytest.mark.parametrize("curve", [0, 1])
@pytest.mark.parametrize("kcase,precompute,long_key,short_coeffs", [
    ("logG", False, False, False), ("logG+1", False, True, False), (6, True, False, True),
    (10, False, True, False), (10, True, False, True), (13, True, True, True)])
def test_group_open_parity(ctx, gctx, curve, kcase, precompute, long_key, short_coeffs):
    G0 = _G(gctx, 20)
    k = {"logG": G0.bit_length() - 1, "logG+1": G0.bit_length()}.get(kcase, kcase)
    G = _G(gctx, k)
    assert G >= 2
    sf = cref.scalar_field(curve)
    n = 1 << k
    extra = 5 if long_key else 0
    pts = cref.gen_points(curve, 700 + k, n + extra + 1)
    key, hp = pts[:n + extra], pts[n + extra]
    n_coeffs = n - 3 if short_coeffs else n          # not a multiple of G
    coeffs = cref.gen_scalars(sf, 701 + k, n_coeffs, True)
    padded = np.concatenate([coeffs, np.zeros((n - n_coeffs, 4), np.uint64)])
    z = cref.gen_scalars(sf, 702, 1, True).reshape(4)
    squeeze = sponge_stand_in(sf)
    B = gctx.register_bases(curve, key)
    Bs = ctx.register_bases(curve, key)
    if precompute:
        B.precompute(); Bs.precompute()
    try:
        before = _launches(gctx)
        got = _drive(gctx, gctx.ipa_open_begin(B, coeffs, k, z, hp), k, squeeze, sf)
        after = _launches(gctx)
        assert all(after[i] > before[i] for i in range(G)), (before, after)     # every child of the G ran kernels
        one = _drive(ctx, ctx.ipa_open_begin(Bs, coeffs, k, z, hp), k, squeeze, sf)
        el, er, efk, ec, echs = _oracle(curve, key[:n], padded, z, hp, squeeze, ("parity", curve, k, short_coeffs, long_key))
        assert len(got[0]) == k
        assert all(same_point(x, y) for x, y in zip(got[0] + got[1], el + er))
        assert all(np.array_equal(x, y) for x, y in zip(got[4], echs))
        assert np.array_equal(got[2], efk) and np.array_equal(got[3], ec)
        assert _same_proof(got, one)
        ck = ab.CommitterKey(B, n + extra)
        assert ab.InnerProductArgPC.check_final_key(ck, np.array(got[4]), got[2], 0)
        bad = got[2].copy(); bad[3] ^= np.uint64(2)
        assert not ab.InnerProductArgPC.check_final_key(ck, np.array(got[4]), bad, 0)
    finally:
        B.release(); Bs.release()


@pytest.mark.parametrize("curve", [0, 1])
def test_group_open_hiding_generator_by_index(gctx, curve):
    """h' = xi_0 * key[h_index] given by (index, xi_0): the same proof as with the point; indices in the last and the
    first shard; rounds driven as fold_round and as round + fold"""
    sf = cref.scalar_field(curve)
    k = 7
    n = 1 << k
    pts = cref.gen_points(curve, 720, n + 1)                 # generators || hiding generator (the last shard holds it)
    coeffs = cref.gen_scalars(sf, 721, n, True)
    z = cref.gen_scalars(sf, 722, 1, True).reshape(4)
    xi0 = cref.gen_scalars(sf, 723, 1, True).reshape(4)
    squeeze = sponge_stand_in(sf)
    B = gctx.register_bases(curve, pts)
    B.precompute()
    try:
        for h_index in (n, 1):
            hp, hp_inf = cref.point_mul(curve, pts[h_index], 0, cref.from_mont(sf, xi0.reshape(1, 4)).reshape(4))
            assert hp_inf == 0
            el, er, efk, ec, _ = _oracle(curve, pts[:n], coeffs, z, hp, squeeze, ("hiding", curve, h_index))
            for separate in (False, True):
                by_point = _drive(gctx, gctx.ipa_open_begin(B, coeffs, k, z, hp), k, squeeze, sf, separate)
                sess = gctx.ipa_open_begin(B, coeffs, k, z, None)
                gctx.ipa_open_use_hiding_generator(sess, h_index, xi0)
                by_index = _drive(gctx, sess, k, squeeze, sf, separate)
                assert _same_proof(by_point, by_index)
                assert all(same_point(x, y) for x, y in zip(by_index[0] + by_index[1], el + er))
                assert np.array_equal(by_index[2], efk) and np.array_equal(by_index[3], ec)
        # after the first round the hiding generator can no longer be switched
        sess = gctx.ipa_open_begin(B, coeffs, k, z, None)
        gctx.ipa_open_use_hiding_generator(sess, n, xi0)
        gctx.ipa_open_round(sess)
        with pytest.raises(ab.AccmsmError):
            gctx.ipa_open_use_hiding_generator(sess, n, xi0)
        with pytest.raises(ab.AccmsmError):
            gctx.ipa_open_finish(sess)
    finally:
        B.release()


@pytest.mark.parametrize("curve", [0, 1])
@pytest.mark.parametrize("rounds,min_log,k", [(1, 2, 10), (5, 11, 13)])
def test_group_open_fold_policy(gctx, curve, rounds, min_log, k):
    """accmsm_set_ipa_fold applies per child (the children materialise their folded key shards): results unchanged"""
    sf = cref.scalar_field(curve)
    n = 1 << k
    pts = cref.gen_points(curve, 700 + k, n + 1)
    key, hp = pts[:n], pts[n]
    coeffs = cref.gen_scalars(sf, 701 + k, n, True)
    z = cref.gen_scalars(sf, 702, 1, True).reshape(4)
    squeeze = sponge_stand_in(sf)
    B = gctx.register_bases(curve, key)
    B.precompute()
    gctx.set_ipa_fold(rounds, min_log)
    try:
        got = _drive(gctx, gctx.ipa_open_begin(B, coeffs, k, z, hp), k, squeeze, sf)
    finally:
        gctx.set_ipa_fold()
        B.release()
    el, er, efk, ec, _ = _oracle(curve, key, coeffs, z, hp, squeeze, ("parity", curve, k, False, False))
    assert all(same_point(x, y) for x, y in zip(got[0] + got[1], el + er))
    assert np.array_equal(got[2], efk) and np.array_equal(got[3], ec)


@pytest.mark.parametrize("curve,k,m,n_random", [(0, 8, 2, 2), (1, 6, 3, 5), (0, 2, 2, 3)])
def test_group_open_combined(ctx, gctx, curve, k, m, n_random):
    """begin_combined: every child builds and evaluates its cyclic slice of [random poly] + sum_j alpha_j h_j(X);
    eval_out and the proof equal the single-device ctx's and the oracle's"""
    sf = cref.scalar_field(curve)
    n = 1 << k
    pts = cref.gen_points(curve, 740 + k, n + 1)
    key, hp = pts[:n], pts[n]
    chm = cref.gen_scalars(sf, 741, m * k, True).reshape(m, k, 4)
    al = cref.gen_scalars(sf, 742, m, True)
    rp = cref.gen_scalars(sf, 743, n_random, True)
    z = cref.gen_scalars(sf, 744, 1, True).reshape(4)
    squeeze = sponge_stand_in(sf)
    combined = cref.combine_check_polys(sf, chm, al, rp)
    B = gctx.register_bases(curve, key)
    Bs = ctx.register_bases(curve, key)
    try:
        sess, ev = gctx.ipa_open_begin_combined(B, chm, al, z, hp, rp)
        assert np.array_equal(ev, cref.poly_evaluate(sf, combined, z).reshape(4))
        got = _drive(gctx, sess, k, squeeze, sf, separate=True)
        s1, ev1 = ctx.ipa_open_begin_combined(Bs, chm, al, z, hp, rp)
        assert np.array_equal(ev, ev1)
        assert _same_proof(got, _drive(ctx, s1, k, squeeze, sf, separate=True))
        el, er, efk, ec, _ = oracle_open(curve, key, combined, z, hp, squeeze)
        assert all(same_point(x, y) for x, y in zip(got[0] + got[1], el + er))
        assert np.array_equal(got[2], efk) and np.array_equal(got[3], ec)
        assert ab.InnerProductArgPC.check_final_key(ab.CommitterKey(B, n), np.array(got[4]), got[2], 0)
    finally:
        B.release(); Bs.release()


def test_group_open_min_shard_keeps_small_openings_on_child_0(gctx):
    """with min_shard above 2^k / 2 the opening runs on child 0 only; the result is the same"""
    curve, k = 0, 8
    sf = cref.scalar_field(curve)
    n = 1 << k
    pts = cref.gen_points(curve, 700 + k, n + 1)
    key, hp = pts[:n], pts[n]
    coeffs = cref.gen_scalars(sf, 701 + k, n, True)
    z = cref.gen_scalars(sf, 702, 1, True).reshape(4)
    squeeze = sponge_stand_in(sf)
    gctx.set_min_shard(n // 2 + 1)
    try:
        B = gctx.register_bases(curve, key)
        before = _launches(gctx)
        got = _drive(gctx, gctx.ipa_open_begin(B, coeffs, k, z, hp), k, squeeze, sf)
        after = _launches(gctx)
        B.release()
    finally:
        gctx.set_min_shard(0)
    assert after[0] > before[0] and after[1:] == before[1:]
    el, er, efk, ec, _ = _oracle(curve, key, coeffs, z, hp, squeeze, ("parity", curve, k, False, False))
    assert all(same_point(x, y) for x, y in zip(got[0] + got[1], el + er))
    assert np.array_equal(got[2], efk) and np.array_equal(got[3], ec)


def test_group_open_interleaved_sessions(gctx):
    """two sharded sessions, and a sharded one with a child-0 one (min_shard = 32: 2^8 is sharded, 2^5 is not),
    advanced round by round in turn"""
    curve = 1
    sf = cref.scalar_field(curve)
    squeeze = sponge_stand_in(sf)
    z = cref.gen_scalars(sf, 760, 1, True).reshape(4)
    cases = []
    for k, seed in ((8, 761), (9, 762), (5, 763)):
        n = 1 << k
        pts = cref.gen_points(curve, seed, n + 1)
        coeffs = cref.gen_scalars(sf, seed + 1, n, True)
        cases.append((k, pts[:n], pts[n], coeffs))
    gctx.set_min_shard(32)
    bases = []
    try:
        for pair in ((0, 1), (0, 2)):
            sess = {}
            for i in pair:
                k, key, hp, coeffs = cases[i]
                bases.append(gctx.register_bases(curve, key))
                sess[i] = [gctx.ipa_open_begin(bases[-1], coeffs, k, z, hp), [], [], [], None, None]
            for i in pair:
                sess[i][5] = gctx.ipa_open_round(sess[i][0])
            while any(s[5] is not None for s in sess.values()):
                for i in pair:
                    s = sess[i]
                    if s[5] is None:
                        continue
                    l, r = s[5]
                    s[4] = np.ascontiguousarray(squeeze(s[4], l, r), dtype=np.uint64).reshape(4)
                    s[1].append(l); s[2].append(r); s[3].append(s[4])
                    s[5] = gctx.ipa_open_fold_round(s[0], s[4])
            for i in pair:
                k, key, hp, coeffs = cases[i]
                fk, c = gctx.ipa_open_finish(sess[i][0])
                el, er, efk, ec, _ = _oracle(curve, key, coeffs, z, hp, squeeze, ("interleave", i))
                assert len(sess[i][1]) == k
                assert all(same_point(x, y) for x, y in zip(sess[i][1] + sess[i][2], el + er))
                assert np.array_equal(fk, efk) and np.array_equal(c, ec)
    finally:
        gctx.set_min_shard(0)
        for b in bases:
            b.release()


def test_group_open_errors(gctx):
    """finish with rounds left: ACCMSM_E_ARG and the session is gone (ACCMSM_E_HANDLE); a zero challenge is refused
    without harming the session; a fresh session works afterwards"""
    curve, k = 0, 6
    sf = cref.scalar_field(curve)
    n = 1 << k
    pts = cref.gen_points(curve, 700 + k, n + 1)
    key, hp = pts[:n], pts[n]
    coeffs = cref.gen_scalars(sf, 701 + k, n, True)
    z = cref.gen_scalars(sf, 702, 1, True).reshape(4)
    squeeze = sponge_stand_in(sf)
    lib, h = gctx._lib, gctx._h
    fk, c = np.empty(8, np.uint64), np.empty(4, np.uint64)
    fkp, cp = fk.ctypes.data_as(C.POINTER(C.c_uint64)), c.ctypes.data_as(C.POINTER(C.c_uint64))
    B = gctx.register_bases(curve, key)
    try:
        for rounds_done in (0, 2, k - 1):
            sess = gctx.ipa_open_begin(B, coeffs, k, z, hp)
            lr, xi = gctx.ipa_open_round(sess), None
            for _ in range(rounds_done):
                xi = squeeze(xi, *lr)
                lr = gctx.ipa_open_fold_round(sess, xi)
            assert lib.accmsm_ipa_open_finish(h, C.c_uint64(sess), fkp, cp) == E_ARG
            assert lib.accmsm_ipa_open_finish(h, C.c_uint64(sess), fkp, cp) == E_HANDLE
        sess = gctx.ipa_open_begin(B, coeffs, k, z, hp)
        l_vec, r_vec, chs, xi = [], [], [], None
        lr = gctx.ipa_open_round(sess)
        with pytest.raises(ab.AccmsmError):
            gctx.ipa_open_fold_round(sess, np.zeros(4, np.uint64))
        while lr is not None:
            l, r = lr
            xi = np.ascontiguousarray(squeeze(xi, l, r), dtype=np.uint64).reshape(4)
            l_vec.append(l); r_vec.append(r); chs.append(xi)
            lr = gctx.ipa_open_fold_round(sess, xi)
        fk2, c2 = gctx.ipa_open_finish(sess)
        el, er, efk, ec, _ = _oracle(curve, key, coeffs, z, hp, squeeze, ("parity", curve, k, False, False))
        assert all(same_point(x, y) for x, y in zip(l_vec + r_vec, el + er))
        assert np.array_equal(fk2, efk) and np.array_equal(c2, ec)
    finally:
        B.release()


def test_group_open_repeatable_and_no_leak(gctx):
    """repeat openings give the same bits; register -> open -> release cycles (cyclic layouts with window tables, the
    tail key) return their device memory"""
    import torch
    curve, k = 0, 14
    sf = cref.scalar_field(curve)
    n = 1 << k
    pts = cref.gen_points(curve, 780, n + 1)
    key, hp = pts[:n], pts[n]
    coeffs = cref.gen_scalars(sf, 781, n, True)
    z = cref.gen_scalars(sf, 782, 1, True).reshape(4)
    squeeze = sponge_stand_in(sf)

    def cycle():
        B = gctx.register_bases(curve, key)
        B.precompute()
        try:
            return _drive(gctx, gctx.ipa_open_begin(B, coeffs, k, z, hp), k, squeeze, sf)
        finally:
            B.release()

    first = cycle()
    cycle()
    torch.cuda.synchronize(0)
    free0 = torch.cuda.mem_get_info(0)[0]
    for _ in range(3):
        assert _same_proof(cycle(), first)
    torch.cuda.synchronize(0)
    free1 = torch.cuda.mem_get_info(0)[0]
    assert free0 - free1 <= (8 << 20), (free0, free1)
