"""The decider of the R1CS NARK accumulation scheme, ASForR1CSNark::decide (src/r1cs_nark_as/mod.rs:1031-1112), on the device:
one vector launch (k_nark_rows in decide mode) and one 6-job pass of the MSM pipeline (accmsm_nark_as_decide).

The oracle side is restated here from SURVEY App. C.10 and C.7 over the oracle primitives (csr_matvec, hadamard, commit):
t_M = M (x* || w*); accept iff Commit(t_M, sigma_M*) == comm_M* for M = A, B, C, Commit(a*, r1*) == C1*, Commit(b*, r2*) == C2*
and Commit(a* o b*, r3*) == C3*, the product over min(|a*|, |b*|).  The unmarked tests check that restatement without a GPU;
the gpu tests compare all six commitments bit for bit with it, on both curves, on one context and on device groups."""
import ctypes as C

import numpy as np
import pytest

import accumulation_b200 as ab
from oracle import cref
from tests.util import same_point
from tests.test_gpu_msm_dispatch import plan, table_window_bits
from tests.test_gpu_nark import (_system, gamma_stand_in, oracle_lhs, oracle_nark_prove, oracle_nark_verify, satisfying_system,
                                 zk_randomness)

E_ARG, E_HANDLE = -2, -3


# ---- oracle restatement (SURVEY App. C.10, C.7) ---------------------------------------------------------------------------
def oracle_decide_rhs(curve, mats, gens, h, x, w, a, b, sigmas=None, hp_rand=None):
    """the six right-hand commitments: Commit(t_M, sigma_M) for M = A, B, C, Commit(a, r1), Commit(b, r2), Commit(a o b, r3)"""
    f = cref.scalar_field(curve)
    x, w = np.asarray(x, np.uint64).reshape(-1, 4), np.asarray(w, np.uint64).reshape(-1, 4)
    a, b = np.asarray(a, np.uint64).reshape(-1, 4), np.asarray(b, np.uint64).reshape(-1, 4)
    t = [cref.csr_matvec(f, *m, x, w) for m in mats]
    k = min(a.shape[0], b.shape[0])
    prod = cref.hadamard(f, a[:k], b[:k]) if k else np.zeros((0, 4), np.uint64)
    vecs = t + [a, b, prod]
    rand = [None if sigmas is None else sigmas[j] for j in range(3)] + [None if hp_rand is None else hp_rand[j] for j in range(3)]
    return [cref.commit(curve, gens[:v.shape[0]], v) if r is None else cref.commit(curve, gens[:v.shape[0]], v, h, r)
            for v, r in zip(vecs, rand)]


def oracle_decide(curve, mats, gens, h, x, w, a, b, expected, sigmas=None, hp_rand=None):
    """ASForR1CSNark::decide -> (accept, the six right-hand commitments); expected = comm_A*, comm_B*, comm_C*, C1*, C2*, C3*"""
    rhs = oracle_decide_rhs(curve, mats, gens, h, x, w, a, b, sigmas, hp_rand)
    return all(same_point(e, r) for e, r in zip(expected, rhs)), rhs


def accumulator_from_zk_proof(curve, mats, gens, h, x, wit, r, bl):
    """the accumulator formed from one verified zk NARK proof: (x, w', sigma_A, sigma_B, sigma_C) against comm_M + gamma comm_rM,
    and the hp part (t_A, t_B; sigma_A, sigma_B, sigma_o) against (comm_A + gamma comm_rA, comm_B + gamma comm_rB,
    comm_C + gamma comm_1 + gamma^2 comm_2) -> (w', sigmas, a, b, hp_rand, expected)"""
    f = cref.scalar_field(curve)
    _, first, gamma, wp, sig = oracle_nark_prove(curve, mats, gens, h, x, wit, gamma_stand_in(f), (r, bl))
    lhs = oracle_lhs(curve, first, gamma)
    t = [cref.csr_matvec(f, *m, x, wp) for m in mats]
    return wp, sig[:3], t[0], t[1], np.stack([sig[0], sig[1], sig[3]]), [lhs[0], lhs[1], lhs[2], lhs[0], lhs[1], lhs[3]]


def _hp_vectors(field, n_a, n_b, seed):
    return cref.gen_scalars(field, seed, n_a, True), cref.gen_scalars(field, seed + 1, n_b, True)


def _randomness(field, mode, seed):
    """mode: 'zk' (sigma* and hp randomness), 'plain' (neither), 'sigma' (sigma* only), 'hp' (hp randomness only)"""
    sig = cref.gen_scalars(field, seed, 3, True) if mode in ("zk", "sigma") else None
    hpr = cref.gen_scalars(field, seed + 1, 3, True) if mode in ("zk", "hp") else None
    return sig, hpr


def _flip(a, i, j):
    b = np.array(a, dtype=np.uint64, copy=True)
    b[i, j] ^= np.uint64(1)
    return b


def corruptions(x, w, a, b, sig, hpr, expected):
    """(name, w, a, b, sigmas, hp_rand, expected) each of which must be rejected: one limb of w*, a*, b*, every sigma and r_i,
    every expected point, and C1* swapped with C2*"""
    out = [("w", _flip(w, 1, 0), a, b, sig, hpr, expected), ("a", w, _flip(a, 2, 1), b, sig, hpr, expected),
           ("b", w, a, _flip(b, 0, 3), sig, hpr, expected)]
    for j in range(3):
        if sig is not None:
            out.append((f"sigma{j}", w, a, b, _flip(sig, j, 0), hpr, expected))
        if hpr is not None:
            out.append((f"r{j + 1}", w, a, b, sig, _flip(hpr, j, 2), expected))
    for j in range(6):
        e = list(expected)
        e[j] = (_flip(np.asarray(e[j][0]).reshape(1, 8), 0, 0).reshape(8), e[j][1])
        out.append((f"expected{j}", w, a, b, sig, hpr, e))
    e = list(expected)
    e[3], e[4] = e[4], e[3]
    out.append(("swap C1 C2", w, a, b, sig, hpr, e))
    return out


# ---- CPU: the restatement itself ------------------------------------------------------------------------------------------
def _cpu_case(curve, M=24, seed=7):
    f = cref.scalar_field(curve)
    mats, x, w = satisfying_system(f, M, 3, 5, seed)
    pts = cref.gen_points(curve, 0x5A00 + curve, M + 1)
    return f, mats, x, w, pts[:M], pts[M]


@pytest.mark.parametrize("curve", [0, 1])
def test_oracle_accumulator_accepts_and_corruptions_reject(curve):
    f, mats, x, w, gens, h = _cpu_case(curve)
    M = gens.shape[0]
    a, b = _hp_vectors(f, M, M - 5, 0x5A10)
    sig, hpr = _randomness(f, "zk", 0x5A20)
    expected = oracle_decide_rhs(curve, mats, gens, h, x, w, a, b, sig, hpr)
    assert oracle_decide(curve, mats, gens, h, x, w, a, b, expected, sig, hpr)[0]
    cases = corruptions(x, w, a, b, sig, hpr, expected)
    assert len(cases) == 3 + 6 + 6 + 1
    for name, cw, ca, cb, cs, ch, ce in cases:
        assert not oracle_decide(curve, mats, gens, h, x, cw, ca, cb, ce, cs, ch)[0], name


@pytest.mark.parametrize("curve", [0, 1])
def test_oracle_accumulator_of_one_zk_proof_is_accepted(curve):
    """accepted by construction from the NARK verify equations"""
    f, mats, x, wit, gens, h = _cpu_case(curve, M=20, seed=11)
    r, bl = zk_randomness(f, wit.shape[0], 0x5A30)
    wp, sig, a, b, hpr, expected = accumulator_from_zk_proof(curve, mats, gens, h, x, wit, r, bl)
    _, first, gamma, _, sig4 = oracle_nark_prove(curve, mats, gens, h, x, wit, gamma_stand_in(f), (r, bl))
    assert oracle_nark_verify(curve, mats, gens, h, x, first, gamma, wp, sig4)[0]
    assert oracle_decide(curve, mats, gens, h, x, wp, a, b, expected, sig, hpr)[0]
    assert not oracle_decide(curve, mats, gens, h, x, wit, a, b, expected, sig, hpr)[0]      # w instead of w'


# ---- GPU ------------------------------------------------------------------------------------------------------------------
def _exp_arrays(expected):
    return np.array([np.asarray(p[0], np.uint64) for p in expected]), np.array([int(p[1]) for p in expected], np.uint8)


def decide_on(c, B, csr, x, w, a, b, expected, n_gens, sig, hpr):
    exy, einf = _exp_arrays(expected)
    return c.nark_as_decide(B, csr, x, w, a, b, exy, einf, hiding_index=n_gens, sigmas=sig, hp_randomness=hpr)


def check_decide(c, curve, mats, x, w, a, b, pts, n_gens, B, table_c, sig, hpr, count_launches=True, expected=None):
    """nark_as_decide on context c against the restatement: the six commitments bit for bit, accept equal to the oracle's,
    one vector launch + one 6-job pass.  expected: None = the restatement's own commitments (an accepted accumulator)"""
    M = np.asarray(mats[0][0]).size - 1
    gens, h = pts[:n_gens], pts[n_gens]
    rhs = oracle_decide_rhs(curve, mats, gens, h, x, w, a, b, sig, hpr)
    expected = rhs if expected is None else expected
    ok_o = all(same_point(e, r) for e, r in zip(expected, rhs))
    csr = c.register_csr(cref.scalar_field(curve), mats)
    try:
        before = c.kernel_launches()
        ok, xy, inf = decide_on(c, B, csr, x, w, a, b, expected, n_gens, sig, hpr)
        if count_launches:
            n_eff = M + (0 if sig is None and hpr is None else 1)
            assert c.kernel_launches() - before == (1 if M else 0) + (plan(n_eff, 6, table_c=table_c).launches if n_eff else 0)
        assert ok == ok_o
        for j in range(6):
            assert same_point((xy[j], inf[j]), rhs[j]), ("comm", j)
        return ok, (xy, inf)
    finally:
        c.release_csr(csr)


# (system, curve, M, key generators, table bits or None, randomness, n_a, n_b)
PARITY_CASES = [
    ("scaling", 0, 1 << 16, 1 << 16, "auto", "zk", None, None),
    ("dense", 1, 1 << 16, 1 << 16, None, "zk", None, None),
    ("scaling", 0, 1 << 20, 1 << 20, 20, "zk", None, None),       # the 6-job shape at full size over a c = 20 table
    ("satisfying", 1, 3000, 5000, None, "zk", None, None),        # Vesta, key longer than n_rows
    ("satisfying", 1, 3000, 5000, None, "plain", None, None),
    ("satisfying", 0, 3000, 3000, "auto", "sigma", None, None),
    ("satisfying", 0, 3000, 3000, "auto", "hp", None, None),
    ("satisfying", 1, 3000, 3000, None, "zk", 3000, 2222),        # n_a != n_b
    ("satisfying", 0, 3000, 3000, None, "zk", 0, 1717),           # n_a = 0
    ("satisfying", 1, 1, 1, None, "zk", None, None),
    ("no_witness", 0, 40, 64, "auto", "zk", None, None),          # n_witness = 0
    ("no_witness", 1, 40, 64, None, "plain", 17, 40),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", PARITY_CASES, ids=[f"{c[0]}-{'pallas' if c[1] == 0 else 'vesta'}-{c[2]}-{c[5]}-{c[6]}-{c[7]}"
                                                     for c in PARITY_CASES])
def test_decide_matches_the_oracle(ctx, case):
    name, curve, M, n_gens, table, mode, n_a, n_b = case
    f = cref.scalar_field(curve)
    mats, x, w = _system((name, curve, M))
    pts = cref.gen_points(curve, 0x5B00 + curve, n_gens + 1)
    B = ctx.register_bases(curve, pts)
    table_c = None
    if table is not None:
        B.precompute(0 if table == "auto" else table)
        table_c = table_window_bits(n_gens + 1, 0 if table == "auto" else table)
    try:
        a, b = _hp_vectors(f, M if n_a is None else n_a, M if n_b is None else n_b, 0x5B10)
        sig, hpr = _randomness(f, mode, 0x5B20)
        ok, _ = check_decide(ctx, curve, mats, x, w, a, b, pts, n_gens, B, table_c, sig, hpr)
        assert ok
    finally:
        B.release()


@pytest.mark.gpu
@pytest.mark.parametrize("curve", [0, 1])
def test_every_corruption_is_rejected_on_the_device(ctx, curve):
    f = cref.scalar_field(curve)
    M = 700
    mats, x, w = satisfying_system(f, M, 3, 200, 0x5C00 + curve)
    pts = cref.gen_points(curve, 0x5C10 + curve, M + 1)
    B = ctx.register_bases(curve, pts)
    B.precompute()
    csr = ctx.register_csr(f, mats)
    try:
        a, b = _hp_vectors(f, M, M - 50, 0x5C20)
        sig, hpr = _randomness(f, "zk", 0x5C30)
        expected = oracle_decide_rhs(curve, mats, pts[:M], pts[M], x, w, a, b, sig, hpr)
        assert decide_on(ctx, B, csr, x, w, a, b, expected, M, sig, hpr)[0]
        for name, cw, ca, cb, cs, ch, ce in corruptions(x, w, a, b, sig, hpr, expected):
            ok, xy, inf = decide_on(ctx, B, csr, x, cw, ca, cb, ce, M, cs, ch)
            assert not ok, name
            rhs = oracle_decide_rhs(curve, mats, pts[:M], pts[M], x, cw, ca, cb, cs, ch)
            assert all(same_point((xy[j], inf[j]), rhs[j]) for j in range(6)), name
        # the accumulator of one zk NARK proof is accepted on the device as well
        r, bl = zk_randomness(f, w.shape[0], 0x5C40)
        wp, zs, za, zb, zh, ze = accumulator_from_zk_proof(curve, mats, pts[:M], pts[M], x, w, r, bl)
        assert decide_on(ctx, B, csr, x, wp, za, zb, ze, M, zs, zh)[0]
    finally:
        ctx.release_csr(csr); B.release()


def _small_key(c, curve, n_gens, seed=0x5D00, precompute=True):
    pts = cref.gen_points(curve, seed + curve, n_gens + 1)
    return pts, ab.CommitterKey.new(c, curve, pts[:n_gens], pts[n_gens], precompute=precompute)


def _records(x, w, a, b, sig, hpr, expected):
    inst = ab.AccumulatorInstance(x, expected[0], expected[1], expected[2], tuple(expected[3:]))
    wit = ab.AccumulatorWitness(w, (a, b, None if hpr is None else list(hpr)), None if sig is None else list(sig))
    return inst, wit


@pytest.mark.gpu
@pytest.mark.parametrize("curve", [0, 1])
def test_mirror_end_to_end(ctx, curve):
    """ASForR1CSNark.decide: the restatement's accumulator and the accumulator of a device zk NARK proof are accepted, each
    corruption and an r1cs_input of the wrong length are rejected, and the non-zk accumulator decides the same way"""
    f = cref.scalar_field(curve)
    M = 1500 + 37 * curve
    n_in = 5
    mats, x, w = satisfying_system(f, M, n_in, 700, 0x5D10 + curve)
    pts, ck = _small_key(ctx, curve, M)
    nark = ab.R1CSNark(ck, mats, num_instance_variables=n_in)
    try:
        a, b = _hp_vectors(f, M, M, 0x5D20)
        sig, hpr = _randomness(f, "zk", 0x5D30)
        expected = oracle_decide_rhs(curve, mats, pts[:M], pts[M], x, w, a, b, sig, hpr)
        assert ab.ASForR1CSNark.decide(nark, *_records(x, w, a, b, sig, hpr, expected))
        for name, cw, ca, cb, cs, ch, ce in corruptions(x, w, a, b, sig, hpr, expected):
            assert not ab.ASForR1CSNark.decide(nark, *_records(x, cw, ca, cb, cs, ch, ce)), name
        assert not ab.ASForR1CSNark.decide(nark, *_records(x[:-1], np.concatenate([x[-1:], w]), a, b, sig, hpr, expected))
        # the accumulator of a device zk proof: x, w', sigma_A..C; hp part (t_A, t_B; sigma_A, sigma_B, sigma_o)
        gam = gamma_stand_in(f)
        r, bl = zk_randomness(f, w.shape[0], 0x5D40)
        proof = nark.prove(x, w, gam, zk=(r, bl))
        gamma = gam(proof.first_msg)
        assert nark.verify(x, proof, gamma)
        lhs = oracle_lhs(curve, proof.first_msg, gamma)
        t = [cref.csr_matvec(f, *m, x, proof.blinded_witness) for m in mats]
        s = proof.sigmas
        inst, wit = _records(x, proof.blinded_witness, t[0], t[1], s[:3], np.stack([s[0], s[1], s[3]]),
                             [lhs[0], lhs[1], lhs[2], lhs[0], lhs[1], lhs[3]])
        assert ab.ASForR1CSNark.decide(nark, inst, wit)
        # without randomness
        e0 = oracle_decide_rhs(curve, mats, pts[:M], pts[M], x, w, a, b)
        assert ab.ASForR1CSNark.decide(nark, *_records(x, w, a, b, None, None, e0))
        assert not ab.ASForR1CSNark.decide(nark, *_records(x, _flip(w, 4, 0), a, b, None, None, e0))
    finally:
        nark.release(); ck.bases.release()


def _group_scenarios(c1, cg, curve, n_gens, M, seed):
    """zk, plain and one-sided randomness with n_a, n_b ending inside different shards: the group gives the single-device
    ctx's points bit for bit, and both the oracle's"""
    f = cref.scalar_field(curve)
    mats, x, w = satisfying_system(f, M, 4, 900, seed)
    pts = cref.gen_points(curve, seed + 1, n_gens + 1)
    B1, Bg = c1.register_bases(curve, pts), cg.register_bases(curve, pts)
    try:
        for mode, n_a, n_b in [("zk", M, M), ("plain", M // 2 + 3, M - 1), ("sigma", 0, M // 3), ("hp", M - 7, M // 2)]:
            a, b = _hp_vectors(f, n_a, n_b, seed + 2)
            sig, hpr = _randomness(f, mode, seed + 3)
            ok1, r1 = check_decide(c1, curve, mats, x, w, a, b, pts, n_gens, B1, None, sig, hpr)
            okg, rg = check_decide(cg, curve, mats, x, w, a, b, pts, n_gens, Bg, None, sig, hpr, count_launches=False)
            assert ok1 and okg, mode
            assert np.array_equal(r1[0], rg[0]) and np.array_equal(r1[1], rg[1]), mode
        # a corruption is rejected on the group too
        a, b = _hp_vectors(f, M, M, seed + 2)
        sig, hpr = _randomness(f, "zk", seed + 3)
        expected = oracle_decide_rhs(curve, mats, pts[:n_gens], pts[n_gens], x, w, a, b, sig, hpr)
        ok, _ = check_decide(cg, curve, mats, x, w, _flip(a, M - 1, 0), b, pts, n_gens, Bg, None, sig, hpr, count_launches=False,
                             expected=expected)
        assert not ok
    finally:
        B1.release(); Bg.release()


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0]])
@pytest.mark.parametrize("long_key", [False, True])
def test_group_is_bit_identical(ctx, devices, long_key):
    """rows cut along the key's point ranges; with a key four times longer than n_rows the rows sit on child 0 and the last
    child owns only the hiding generator"""
    curve = 1 if long_key else 0
    M = 3000
    g = ab.Context(devices=devices, min_shard=16)
    try:
        _group_scenarios(ctx, g, curve, 4 * M if long_key else M, M, 0x5E00 + curve)
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
    M = 3000
    _group_scenarios(ctx, no_peer_group, curve, 4 * M if long_key else M, M, 0x5E40 + curve)


def _decide_rc(c, key, csr, x, n_x, w, n_w, a, n_a, b, n_b, hiding, sig, hpr, exp=True, acc=True):
    e, ei = np.zeros((6, 8), np.uint64), np.zeros(6, np.uint8)
    res = C.c_int(0)
    p = lambda v: None if v is None else v.ctypes.data_as(C.c_void_p)
    return c._lib.accmsm_nark_as_decide(c._h, C.c_uint64(key), C.c_uint64(csr), p(x), C.c_size_t(n_x), p(w), C.c_size_t(n_w), p(a),
                                        C.c_size_t(n_a), p(b), C.c_size_t(n_b), C.c_size_t(hiding), p(sig), p(hpr),
                                        p(e) if exp else None, p(ei) if exp else None, C.byref(res) if acc else None, None, None)


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_argument_errors(ctx, devices):
    c = ctx if devices is None else ab.Context(devices=devices, min_shard=16)
    curve = 0
    f = cref.scalar_field(curve)
    M = 64
    mats, x, w = satisfying_system(f, M, 3, 20, 0x5F00)
    n_x, n_w = x.shape[0], w.shape[0]
    pts = cref.gen_points(curve, 0x5F10, M + 1)
    B = c.register_bases(curve, pts)
    short = c.register_bases(curve, pts[: M // 2])
    csr = c.register_csr(f, mats)
    csr2 = c.register_csr(f, mats[:2])
    other = c.register_csr(1 - f, mats)
    a, b = _hp_vectors(f, M + 1, M + 1, 0x5F20)
    sig, hpr = _randomness(f, "zk", 0x5F30)
    try:
        rc = lambda **kw: _decide_rc(c, **{**dict(key=B.handle, csr=csr, x=x, n_x=n_x, w=w, n_w=n_w, a=a, n_a=M, b=b, n_b=M, hiding=M,
                                                  sig=sig, hpr=hpr), **kw})
        assert rc() == 0
        assert rc(sig=None) == 0 and rc(hpr=None) == 0 and rc(sig=None, hpr=None) == 0
        # hp vectors longer than the rows
        assert rc(n_a=M + 1) == E_ARG and rc(n_b=M + 1) == E_ARG and rc(n_a=M + 1, sig=None, hpr=None) == E_ARG
        # not 3 matrices, the other field, rows or hiding index beyond the key
        assert rc(csr=csr2) == E_ARG and rc(csr=other) == E_ARG
        assert rc(key=short.handle, hiding=M // 2 - 1) == E_ARG and rc(hiding=M + 1) == E_ARG
        # a column beyond input || witness
        assert rc(n_w=n_w - 1) == E_ARG and rc(n_w=n_w - 1, sig=None, hpr=None) == E_ARG
        # null pointers
        assert rc(x=None) == E_ARG and rc(w=None) == E_ARG and rc(a=None) == E_ARG and rc(b=None) == E_ARG
        assert rc(exp=False) == E_ARG and rc(acc=False) == E_ARG
        assert rc(a=None, n_a=0, b=None, n_b=0) == 0
        # unknown handles
        assert rc(key=987654) == E_HANDLE and rc(csr=987654) == E_HANDLE
        # the context still works
        assert rc() == 0
    finally:
        for h in (csr, csr2, other):
            c.release_csr(h)
        B.release(); short.release()
        if c is not ctx:
            c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_no_rows_leaves_the_tail_terms(ctx, devices):
    """n_rows = 0 (so n_a = n_b = 0): the six results are sigma_M H and r_i H, or identities without randomness"""
    c = ctx if devices is None else ab.Context(devices=devices, min_shard=16)
    curve = 1
    f = cref.scalar_field(curve)
    mats = [(np.zeros(1, np.uint32), np.zeros(0, np.uint32), np.zeros((0, 4), np.uint64))] * 3
    pts = cref.gen_points(curve, 0x5F40, 9)
    B = c.register_bases(curve, pts)
    try:
        x = cref.gen_scalars(f, 3, 2, True)
        none = np.zeros((0, 4), np.uint64)
        for mode in ("zk", "sigma", "hp", "plain"):
            sig, hpr = _randomness(f, mode, 0x5F50)
            ok, _ = check_decide(c, curve, mats, x, none, none, none, pts, 8, B, None, sig, hpr, count_launches=devices is None)
            assert ok, mode
    finally:
        B.release()
        if c is not ctx:
            c.close()


@pytest.mark.gpu
def test_cycles_leave_device_memory_where_it_was(ctx):
    import torch
    curve = 0
    f = cref.scalar_field(curve)
    M = 1 << 14
    mats, x, w = satisfying_system(f, M, 4, 4000, 0x5F60)
    pts, ck = _small_key(ctx, curve, M)
    nark = ab.R1CSNark(ck, mats, num_instance_variables=4)
    try:
        a, b = _hp_vectors(f, M, M, 0x5F70)
        sig, hpr = _randomness(f, "zk", 0x5F80)
        expected = oracle_decide_rhs(curve, mats, pts[:M], pts[M], x, w, a, b, sig, hpr)
        inst, wit = _records(x, w, a, b, sig, hpr, expected)
        assert ab.ASForR1CSNark.decide(nark, inst, wit)
        torch.cuda.synchronize(0)
        free0 = torch.cuda.mem_get_info(0)[0]
        for _ in range(20):
            assert ab.ASForR1CSNark.decide(nark, inst, wit)
        torch.cuda.synchronize(0)
        free1 = torch.cuda.mem_get_info(0)[0]
        assert free0 - free1 <= (8 << 20), (free0, free1)
    finally:
        nark.release(); ck.bases.release()
