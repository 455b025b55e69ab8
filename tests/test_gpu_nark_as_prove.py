"""The prover of the R1CS NARK accumulation scheme, ASForR1CSNark::prove (src/r1cs_nark_as/mod.rs:713-926), as a device session:
accmsm_nark_as_prove_begin (one row-kernel launch writes the fresh inputs' mat-vecs into the hp pair buffers; with zk also
M (r_x || r_w), the hp hiding rows and one 6-job pass), accmsm_hp_prove_product_poly_comm on the same session, and
accmsm_nark_as_prove_finish (a*, b* and w*: three k_lincomb launches).

The oracle side is restated here from SURVEY App. C.12 over the oracle primitives, reusing the restated NARK prover
(tests/test_gpu_nark.py), the restated hp prover (tests/test_gpu_hp_prove.py) and the restated decider
(tests/test_gpu_nark_as.py).  The unmarked tests check that restatement without a GPU: the decider accepts its new accumulator
and rejects every corruption of it.  The gpu tests compare every output of the session and of mirror.ASForR1CSNark.prove bit for
bit with it, on both curves, on one context and on device groups."""
import ctypes as C

import numpy as np
import pytest

import accumulation_b200 as ab
from oracle import cref
from tests.util import same_point
from tests.test_gpu_msm_dispatch import plan, table_window_bits
from tests.test_gpu_hp_prove import (MODULI, _digest, _psum, from_mont, mu_list, mu_stand_in, nu_stand_in, oracle_commit,
                                     oracle_prove, to_mont)
from tests.test_gpu_nark import _system, gamma_stand_in, oracle_lhs, oracle_nark_prove, satisfying_system, zk_randomness
from tests.test_gpu_nark_as import corruptions, oracle_decide

E_ARG, E_HANDLE = -2, -3


# ---- oracle restatement (SURVEY App. C.12) ----------------------------------------------------------------------------------
def beta_stand_in(f, k):
    """host sponge stand-in: beta_1 .. beta_{k-1} from the new hp instance and the randomness commitments"""
    def fn(hp_inst, comm_r):
        h = _digest(b"beta", list(hp_inst) + list(comm_r or []))
        out = []
        for i in range(k - 1):
            h.update(bytes([i]))
            out.append(int.from_bytes(h.digest()[:16], "little") | 1)
        return to_mont(f, out)
    return fn


def oracle_as_prove(curve, mats, gens, h, fresh, accs, zk=None, fixed=None):
    """ASForR1CSNark::prove.  fresh: [(x, first_msg, gamma, w', sigmas4 | None)]; accs: [(x, w, a, b, sigma | None, hp_rand |
    None, expected6)] (the shape of corruptions()); zk = (r_x, r_w, sigma_r, ha, hb, hr).  Challenges: the stand-ins over this
    transcript, or fixed = (mu, nu, beta) as ints.  -> (begin points (6) | None, low, high, new accumulator in the shape of accs,
    (mu, nu, beta))"""
    f = cref.scalar_field(curve)
    m = MODULI[f]
    L = np.asarray(mats[0][0]).size - 1
    comm_r = None
    if zk is not None:
        r_x, r_w, sig_r, ha, hb, hr = zk
        comm_r = [oracle_commit(curve, gens, h, cref.csr_matvec(f, *mt, r_x, r_w), sig_r[j]) for j, mt in enumerate(mats)]
    blinded = [oracle_lhs(curve, first, gamma) for _, first, gamma, _, _ in fresh]
    wits = [(cref.csr_matvec(f, *mats[0], x, wp), cref.csr_matvec(f, *mats[1], x, wp), None if s is None else np.stack([s[0], s[1], s[3]]))
            for x, _, _, wp, s in fresh] + [(a, b, hpr) for _, _, a, b, _, hpr, _ in accs]
    insts = [(bl[0], bl[1], bl[3]) for bl in blinded] + [tuple(e[3:]) for *_, e in accs]
    hpzk = None if zk is None else (ha, hb, hr)
    n = len(wits)
    if fixed is None:
        mu = mu_list(f, mu_stand_in(f, n)(oracle_prove(curve, gens, h, L, wits, insts, [1] * (n + 1), 1, hpzk)[0]), zk is not None)
        _, low, high, *_ = oracle_prove(curve, gens, h, L, wits, insts, mu, 1, hpzk)
        nu = from_mont(f, nu_stand_in(f)(low, high))[0]
    else:
        mu, nu, beta = fixed
    hc, low, high, a_s, b_s, rand, hp_new = oracle_prove(curve, gens, h, L, wits, insts, mu, nu, hpzk)
    if fixed is None:
        beta = [1] + from_mont(f, beta_stand_in(f, n + (zk is not None))(hp_new, comm_r))
    xs = [x for x, *_ in fresh] + [a[0] for a in accs] + ([r_x] if zk is not None else [])
    ws = [wp for _, _, _, wp, _ in fresh] + [a[1] for a in accs] + ([r_w] if zk is not None else [])
    bm = to_mont(f, beta)
    x_star, w_star = cref.combine_vectors(f, xs, bm), cref.combine_vectors(f, ws, bm)
    comms = [bl[:3] for bl in blinded] + [a[6][:3] for a in accs] + ([comm_r] if zk is not None else [])
    comm_star = [_psum(curve, [(c[j], beta[k]) for k, c in enumerate(comms)]) for j in range(3)]
    sigs = [None if s is None else from_mont(f, s[:3]) for *_, s in fresh] + [None if a[4] is None else from_mont(f, a[4]) for a in accs]
    sigs += [from_mont(f, sig_r)] if zk is not None else []
    sig_star = None
    if any(s is not None for s in sigs):
        sig_star = to_mont(f, [sum(beta[k] * s[j] for k, s in enumerate(sigs) if s is not None) % m for j in range(3)])
    acc = (x_star, w_star, a_s, b_s, sig_star, rand, comm_star + list(hp_new))
    return (None if zk is None else list(hc) + comm_r), low, high, acc, (mu, nu, beta)


def fresh_input(curve, mats, gens, h, x, w, zk, seed):
    """one fresh input from the restated NARK prover -> (x, first_msg, gamma, w', sigmas | None)"""
    f = cref.scalar_field(curve)
    _, first, gamma, wp, sig = oracle_nark_prove(curve, mats, gens, h, x, w, gamma_stand_in(f),
                                                 zk_randomness(f, w.shape[0], seed) if zk else None)
    return x, first, gamma, wp, sig


def synthetic_fresh(curve, n_rows, n_x, n_w, zk, seed):
    """a fresh input whose first message is arbitrary points: the session does not check the NARK proof, so this exercises it
    at full size without forming eight commitments per input on the host"""
    f = cref.scalar_field(curve)
    first = [(p, 0) for p in cref.gen_points(curve, seed, 8 if zk else 3)]
    return (cref.gen_scalars(f, seed + 1, n_x, True), first, gamma_stand_in(f)(first) if zk else None,
            cref.gen_scalars(f, seed + 2, n_w, True), cref.gen_scalars(f, seed + 3, 4, True) if zk else None)


def synthetic_acc(curve, n_x, n_w, la, lb, zk, seed):
    """an old accumulator with arbitrary commitments (the prover combines them without checking them)"""
    f = cref.scalar_field(curve)
    pts = cref.gen_points(curve, seed, 6)
    return (cref.gen_scalars(f, seed + 1, n_x, True), cref.gen_scalars(f, seed + 2, n_w, True), cref.gen_scalars(f, seed + 3, la, True),
            cref.gen_scalars(f, seed + 4, lb, True), cref.gen_scalars(f, seed + 5, 3, True) if zk else None,
            cref.gen_scalars(f, seed + 6, 3, True) if zk else None, [(p, 0) for p in pts])


def prover_zk(f, n_x, n_w, n_rows, seed):
    return (cref.gen_scalars(f, seed, n_x, True), cref.gen_scalars(f, seed + 1, n_w, True), cref.gen_scalars(f, seed + 2, 3, True),
            cref.gen_scalars(f, seed + 3, n_rows, True), cref.gen_scalars(f, seed + 4, n_rows, True), cref.gen_scalars(f, seed + 5, 3, True))


def accepted(curve, mats, gens, h, acc):
    x, w, a, b, sig, hpr, e = acc
    return oracle_decide(curve, mats, gens, h, x, w, a, b, e, sig, hpr)[0]


# ---- CPU: the restatement itself --------------------------------------------------------------------------------------------
def _cpu_accs(curve, mats, gens, h, x, w, n_a, zk, seed):
    """n_a valid accumulators, each the new accumulator of a (2, 0) prove"""
    f = cref.scalar_field(curve)
    out = []
    for j in range(n_a):
        fr = [fresh_input(curve, mats, gens, h, x, w, zk, seed + 10 * j + i) for i in range(2)]
        z = prover_zk(f, x.shape[0], w.shape[0], gens.shape[0], seed + 10 * j + 5) if zk else None
        out.append(oracle_as_prove(curve, mats, gens, h, fr, [], z)[3])
    return out


@pytest.mark.parametrize("shape", [(1, 0), (2, 0), (1, 2), (0, 2), (3, 1)])
@pytest.mark.parametrize("zk", [False, True])
def test_oracle_accumulator_accepts_and_corruptions_reject(shape, zk):
    n_f, n_a = shape
    if zk and n_f + n_a < 2:
        pytest.skip("zero knowledge needs two hp inputs (the caller pads, src/hp_as/mod.rs:676-710)")
    curve = (n_f + n_a) % 2
    f = cref.scalar_field(curve)
    M = 20
    mats, x, w = satisfying_system(f, M, 3, 5, 0x7A00 + 7 * n_f + n_a)
    pts = cref.gen_points(curve, 0x7A10 + curve, M + 1)
    gens, h = pts[:M], pts[M]
    accs = _cpu_accs(curve, mats, gens, h, x, w, n_a, zk, 0x7A20)
    assert all(accepted(curve, mats, gens, h, a) for a in accs)
    fr = [fresh_input(curve, mats, gens, h, x, w, zk, 0x7A40 + i) for i in range(n_f)]
    z = prover_zk(f, x.shape[0], w.shape[0], M, 0x7A60) if zk else None
    new = oracle_as_prove(curve, mats, gens, h, fr, accs, z)[3]
    assert accepted(curve, mats, gens, h, new)
    x_s, w_s, a_s, b_s, sig, hpr, e = new
    assert (sig is None) == (not zk) and (hpr is None) == (not zk)
    for name, cw, ca, cb, cs, ch, ce in corruptions(x_s, w_s, a_s, b_s, sig, hpr, e):
        assert not oracle_decide(curve, mats, gens, h, x_s, cw, ca, cb, ce, cs, ch)[0], name


# ---- GPU: the session against the restatement -------------------------------------------------------------------------------
def _records(acc):
    x, w, a, b, sig, hpr, e = acc
    return (ab.AccumulatorInstance(x, e[0], e[1], e[2], tuple(e[3:])),
            ab.AccumulatorWitness(w, (a, b, None if hpr is None else list(hpr)), None if sig is None else list(sig)))


def _from_records(inst, wit):
    a, b, hpr = wit.hp_witness
    return (np.asarray(inst.r1cs_input), np.asarray(wit.r1cs_blinded_witness), a, b,
            None if wit.randomness is None else np.array(wit.randomness), None if hpr is None else np.array(hpr),
            [inst.comm_a, inst.comm_b, inst.comm_c] + list(inst.hp_instance))


def _proof(fr):
    x, first, gamma, wp, sig = fr
    return x, ab.NarkProof(first, wp, sig)


def session_on(c, B, csr, fresh, accs, zk, n_rows, hiding_index, table_c=None, count=False):
    """begin, product_poly_comm and finish on context c with the stand-in sponge over the device transcript -> (begin points,
    low, high, a*, b*, w*, (mu, nu, beta)).  The oracle's hp instance for beta comes from the device's challenges, so a wrong
    device output shows up as a mismatch, not as a different transcript."""
    f = cref.scalar_field(B.curve)
    n = len(fresh) + len(accs)
    n_w = (fresh[0][3] if fresh else accs[0][1]).shape[0]
    before = c.kernel_launches()
    sess, pts = c.nark_as_prove_begin(B, csr, [fr[0] for fr in fresh], [fr[3] for fr in fresh], [a[1] for a in accs], [a[2] for a in accs],
                                      [a[3] for a in accs], zk=None if zk is None else (zk[0], zk[1], zk[3], zk[4], np.concatenate([zk[2], zk[5]])),
                                      hiding_index=hiding_index, n_input=(fresh[0][0] if fresh else accs[0][0]).shape[0])
    if count:
        exp = (plan(n_rows + 1, 6, table_c=table_c).launches + (2 if n_rows else 0)) if zk is not None else int(bool(n_rows and fresh))
        assert c.kernel_launches() - before == exp
    begin = None if pts is None else [(pts[0][j], int(pts[1][j])) for j in range(6)]
    mu = mu_list(f, mu_stand_in(f, n)(None if begin is None else begin[:3]), zk is not None)
    (lo, linf), (hi, hinf) = c.hp_prove_product_poly_comm(sess, n, to_mont(f, mu))
    low = [(lo[j], int(linf[j])) for j in range(n - 1)]
    high = [(hi[j], int(hinf[j])) for j in range(n - 1)]
    nu = from_mont(f, nu_stand_in(f)(low, high))[0]
    return sess, begin, low, high, mu, nu


def check_session(c, curve, B, csr, pts, n_gens, mats, fresh, accs, zk, table_c=None, count=False):
    """every output of the session bit for bit against the restatement -> (begin points, low, high, a*, b*, w*)"""
    f = cref.scalar_field(curve)
    gens, h = pts[:n_gens], pts[n_gens]
    n_rows = np.asarray(mats[0][0]).size - 1
    n = len(fresh) + len(accs)
    sess, begin, low, high, mu, nu = session_on(c, B, csr, fresh, accs, zk, n_rows, n_gens, table_c, count)
    # the restatement's hp instance with the device's challenges gives beta
    _, _, _, _, _, _, hp_new = oracle_prove(curve, gens, h, n_rows, *_hp_args(curve, mats, fresh, accs, zk), mu, nu,
                                            None if zk is None else (zk[3], zk[4], zk[5]))
    comm_r = None if begin is None else begin[3:]
    beta = [1] + from_mont(f, beta_stand_in(f, n + (zk is not None))(hp_new, comm_r))
    n_w = (fresh[0][3] if fresh else accs[0][1]).shape[0]
    before = c.kernel_launches()
    a_s, b_s, w_s = c.nark_as_prove_finish(sess, to_mont(f, [nu]).reshape(4), to_mont(f, beta), n_rows, n_w)
    if count:
        assert c.kernel_launches() - before == int(a_s.shape[0] > 0) + int(b_s.shape[0] > 0) + int(n_w > 0)
    ob, olow, ohigh, oacc, _ = oracle_as_prove(curve, mats, gens, h, fresh, accs, zk, fixed=(mu, nu, beta))
    assert (begin is None) == (ob is None)
    for j in range(6 if begin is not None else 0):
        assert same_point(begin[j], ob[j]), ("begin", j)
    for j in range(n - 1):
        assert same_point(low[j], olow[j]) and same_point(high[j], ohigh[j]), ("low/high", j)
    assert np.array_equal(a_s, oacc[2]) and np.array_equal(b_s, oacc[3]) and np.array_equal(w_s, oacc[1])
    return begin, low, high, a_s, b_s, w_s


def _hp_args(curve, mats, fresh, accs, zk):
    f = cref.scalar_field(curve)
    wits = [(cref.csr_matvec(f, *mats[0], x, wp), cref.csr_matvec(f, *mats[1], x, wp), None if s is None else np.stack([s[0], s[1], s[3]]))
            for x, _, _, wp, s in fresh] + [(a, b, hpr) for _, _, a, b, _, hpr, _ in accs]
    insts = [(bl[0], bl[1], bl[3]) for bl in (oracle_lhs(curve, first, g) for _, first, g, _, _ in fresh)] + [tuple(e[3:]) for *_, e in accs]
    return wits, insts


# (system, curve, M, key generators, table bits | None, zk, n_fresh, n_acc, ragged accumulator pairs)
PARITY_CASES = [
    ("scaling", 0, 1 << 16, 1 << 16, "auto", True, 1, 2, False),
    ("scaling", 0, 1 << 16, 1 << 16, "auto", False, 1, 2, False),
    ("dense", 1, 1 << 16, 1 << 16, None, True, 2, 1, False),
    ("scaling", 0, 1 << 20, 1 << 20, 20, True, 1, 2, False),     # the 6-job pass at full size over a c = 20 table
    ("satisfying", 1, 3000, 5000, None, True, 2, 1, False),       # Vesta, key longer than n_rows
    ("satisfying", 0, 3000, 3000, "auto", True, 1, 3, True),      # ragged accumulator pairs
    ("satisfying", 1, 3000, 3000, None, False, 0, 2, True),       # no fresh input: begin launches nothing
    ("satisfying", 0, 3000, 3000, None, False, 3, 0, False),
    ("no_witness", 0, 40, 64, "auto", True, 1, 1, False),         # n_witness = 0
    ("no_witness", 1, 40, 64, None, False, 2, 0, False),
]


def _case_inputs(curve, mats, x, w, n_f, n_a, zk, ragged, seed):
    f = cref.scalar_field(curve)
    M = np.asarray(mats[0][0]).size - 1
    fresh = [synthetic_fresh(curve, M, x.shape[0], w.shape[0], zk, seed + 10 * i) for i in range(n_f)]
    accs = [synthetic_acc(curve, x.shape[0], w.shape[0], max(M - 37 * j - 5, 0) if ragged else M, max(M - 11 * (j + 1), 0) if ragged else M,
                          zk, seed + 100 + 10 * j) for j in range(n_a)]
    z = prover_zk(f, x.shape[0], w.shape[0], M, seed + 500) if zk else None
    return fresh, accs, z


@pytest.mark.gpu
@pytest.mark.parametrize("case", PARITY_CASES, ids=[f"{c[0]}-{'pallas' if c[1] == 0 else 'vesta'}-{c[2]}-{'zk' if c[5] else 'plain'}-"
                                                     f"f{c[6]}a{c[7]}{'-ragged' if c[8] else ''}" for c in PARITY_CASES])
def test_session_matches_the_oracle(ctx, case):
    name, curve, M, n_gens, table, zk, n_f, n_a, ragged = case
    f = cref.scalar_field(curve)
    mats, x, w = _system((name, curve, M))
    pts = cref.gen_points(curve, 0x7B00 + curve, n_gens + 1)
    B = ctx.register_bases(curve, pts)
    table_c = None
    if table is not None:
        B.precompute(0 if table == "auto" else table)
        table_c = table_window_bits(n_gens + 1, 0 if table == "auto" else table)
    csr = ctx.register_csr(f, mats)
    try:
        fresh, accs, z = _case_inputs(curve, mats, x, w, n_f, n_a, zk, ragged, 0x7B10)
        check_session(ctx, curve, B, csr, pts, n_gens, mats, fresh, accs, z, table_c, count=True)
    finally:
        ctx.release_csr(csr); B.release()


def _beta_fn(f, n, zk):
    return beta_stand_in(f, n + (1 if zk else 0))


def mirror_prove(nark, curve, fresh, accs, zk):
    f = cref.scalar_field(curve)
    n = len(fresh) + len(accs)
    return ab.ASForR1CSNark.prove(nark, [_proof(fr) for fr in fresh], [_records(a) for a in accs], gamma_stand_in(f), mu_stand_in(f, n),
                                  nu_stand_in(f), _beta_fn(f, n, zk is not None), zk=zk)


@pytest.mark.gpu
@pytest.mark.parametrize("curve,zk", [(0, True), (1, True), (0, False), (1, False)])
def test_chained_accumulation_is_decided_on_the_device(ctx, curve, zk):
    """the new accumulator of one prove is an old accumulator of the next, three times (the shape of the reference's ASTests);
    mirror.ASForR1CSNark.prove gives the restatement's accumulator bit for bit and the device decider accepts each one"""
    f = cref.scalar_field(curve)
    M = 1500 + 37 * curve
    mats, x, w = satisfying_system(f, M, 5, 600, 0x7C00 + curve)
    pts = cref.gen_points(curve, 0x7C10 + curve, M + 1)
    gens, h = pts[:M], pts[M]
    ck = ab.CommitterKey.new(ctx, curve, gens, h, precompute=True)
    nark = ab.R1CSNark(ck, mats, num_instance_variables=5)
    try:
        accs = []
        for step in range(3):
            fresh = [fresh_input(curve, mats, gens, h, x, w, zk, 0x7C20 + 10 * step + i) for i in range(1 if step else 2)]
            z = prover_zk(f, x.shape[0], w.shape[0], M, 0x7C40 + step) if zk else None
            inst, wit, proof = mirror_prove(nark, curve, fresh, accs, z)
            _, _, _, oacc, _ = oracle_as_prove(curve, mats, gens, h, fresh, accs, z)
            got = _from_records(inst, wit)
            for j in range(4):
                assert np.array_equal(got[j], oacc[j]), (step, j)
            for j in (4, 5):
                assert (got[j] is None) == (oacc[j] is None) and (got[j] is None or np.array_equal(got[j], oacc[j])), (step, j)
            assert all(same_point(p, q) for p, q in zip(got[6], oacc[6])), step
            assert accepted(curve, mats, gens, h, oacc)
            assert ab.ASForR1CSNark.decide(nark, inst, wit), step
            accs = accs[1:] + [oacc] if len(accs) == 2 else accs + [oacc]
    finally:
        nark.release(); ck.bases.release()


def _group_scenarios(c1, cg, curve, n_gens, M, seed):
    """zk and plain, fresh and accumulator pairs, ragged lengths ending inside different shards: the group gives the single
    context's outputs bit for bit, and both the oracle's"""
    f = cref.scalar_field(curve)
    mats, x, w = satisfying_system(f, M, 4, 900, seed)
    pts = cref.gen_points(curve, seed + 1, n_gens + 1)
    B1, Bg = c1.register_bases(curve, pts), cg.register_bases(curve, pts)
    csr1, csrg = c1.register_csr(f, mats), cg.register_csr(f, mats)
    try:
        for zk, n_f, n_a in [(True, 1, 2), (False, 2, 1), (True, 0, 2), (False, 0, 2), (True, 3, 0)]:
            fresh, accs, z = _case_inputs(curve, mats, x, w, n_f, n_a, zk, True, seed + 7 * n_f + n_a)
            r1 = check_session(c1, curve, B1, csr1, pts, n_gens, mats, fresh, accs, z)
            rg = check_session(cg, curve, Bg, csrg, pts, n_gens, mats, fresh, accs, z)
            for p, q in zip(r1, rg):
                if isinstance(p, np.ndarray):
                    assert np.array_equal(p, q), (zk, n_f, n_a)
                elif p is not None:
                    assert all(np.array_equal(u[0], v[0]) and u[1] == v[1] for u, v in zip(p, q)), (zk, n_f, n_a)
    finally:
        c1.release_csr(csr1); cg.release_csr(csrg); B1.release(); Bg.release()


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0]])
@pytest.mark.parametrize("long_key", [False, True])
def test_group_is_bit_identical(ctx, devices, long_key):
    """rows cut along the key's point ranges; with a key four times longer than n_rows every row sits on child 0 and the last
    child owns only the hiding generator"""
    curve = 1 if long_key else 0
    M = 3000
    g = ab.Context(devices=devices, min_shard=16)
    try:
        _group_scenarios(ctx, g, curve, 4 * M if long_key else M, M, 0x7D00 + curve)
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
    _group_scenarios(ctx, no_peer_group, curve, 4 * M if long_key else M, M, 0x7D40 + curve)


@pytest.mark.gpu
def test_hp_and_nark_as_sessions_live_at_once(ctx):
    """a plain hp session and a NARK-AS session interleaved, with an msm and a NARK decide between the steps"""
    from tests.test_gpu_hp_prove import _lens, make_inputs, oracle_prove as hp_oracle
    curve, M = 0, 3000
    f = cref.scalar_field(curve)
    mats, x, w = satisfying_system(f, M, 4, 900, 0x7E00)
    pts = cref.gen_points(curve, 0x7E01, M + 1)
    B = ctx.register_bases(curve, pts)
    csr = ctx.register_csr(f, mats)
    other_pts = cref.gen_points(curve, 0x7E02, 2 * M)
    other = ctx.register_bases(curve, other_pts)
    try:
        big = cref.gen_scalars(f, 0x7E03, 2 * M, True)
        exp_msm = cref.commit(curve, other_pts, big)

        def noise():
            assert same_point(ctx.msm(other, big), exp_msm)
            ok, _, _ = ctx.nark_as_decide(B, csr, x, w, big[:M], big[:M], np.zeros((6, 8), np.uint64), np.zeros(6, np.uint8), hiding_index=M)
            assert not ok

        hw, hi_, hz = make_inputs(curve, pts[:M], pts[M], 3, _lens(3, M, True), 0x7E10, True, M)
        fresh, accs, z = _case_inputs(curve, mats, x, w, 1, 2, True, True, 0x7E20)
        hs, hc = ctx.hp_prove_begin(B, [v[0] for v in hw], [v[1] for v in hw], M, hz[0], hz[1], hiding_index=M, hiding_rand=hz[2])
        noise()
        ns, begin, low, high, mu, nu = session_on(ctx, B, csr, fresh, accs, z, M, M)
        noise()
        hcl = [(hc[0][j], int(hc[1][j])) for j in range(3)]
        hmu = mu_list(f, mu_stand_in(f, 3)(hcl), True)
        (lo, linf), (hi, hinf) = ctx.hp_prove_product_poly_comm(hs, 3, to_mont(f, hmu))
        noise()
        hlow, hhigh = [(lo[j], int(linf[j])) for j in range(2)], [(hi[j], int(hinf[j])) for j in range(2)]
        hnu = nu_stand_in(f)(hlow, hhigh)
        # finish of the other kind is refused and releases the session: so finish each with its own call
        _, _, _, _, _, _, hp_new = oracle_prove(curve, pts[:M], pts[M], M, *_hp_args(curve, mats, fresh, accs, z), mu, nu, (z[3], z[4], z[5]))
        beta = [1] + from_mont(f, beta_stand_in(f, 4)(hp_new, begin[3:]))
        a_s, b_s, w_s = ctx.nark_as_prove_finish(ns, to_mont(f, [nu]).reshape(4), to_mont(f, beta), M, w.shape[0])
        noise()
        ha_s, hb_s = ctx.hp_prove_finish(hs, hnu, M)
        _, _, _, oacc, _ = oracle_as_prove(curve, mats, pts[:M], pts[M], fresh, accs, z, fixed=(mu, nu, beta))
        assert np.array_equal(a_s, oacc[2]) and np.array_equal(b_s, oacc[3]) and np.array_equal(w_s, oacc[1])
        _, _, _, oa, ob, _, _ = hp_oracle(curve, pts[:M], pts[M], M, hw, hi_, hmu, from_mont(f, hnu)[0], hz)
        assert np.array_equal(ha_s, oa) and np.array_equal(hb_s, ob)
    finally:
        ctx.release_csr(csr); B.release(); other.release()


def _ptrs(vecs):
    arr = (C.c_void_p * max(len(vecs), 1))()
    for i, v in enumerate(vecs):
        arr[i] = v.ctypes.data if v.size else None
    return arr


def _rc_begin(c, key, csr, xs, n_x, ws, n_w, aw, aa, bb, rx=None, rw=None, ha=None, hb=None, hiding=0, rand=None, sess=True):
    p = lambda v: None if v is None else v.ctypes.data_as(C.c_void_p)
    al = np.array([v.shape[0] for v in aa] or [0], dtype=np.uint64)
    bl = np.array([v.shape[0] for v in bb] or [0], dtype=np.uint64)
    xy, inf, s = np.zeros((6, 8), np.uint64), np.zeros(6, np.uint8), C.c_uint64(0)
    rc = c._lib.accmsm_nark_as_prove_begin(c._h, C.c_uint64(key), C.c_uint64(csr), C.c_int(len(xs)), _ptrs(xs), C.c_size_t(n_x), _ptrs(ws),
                                           C.c_size_t(n_w), C.c_int(len(aa)), _ptrs(aw), _ptrs(aa), p(al), _ptrs(bb), p(bl), p(rx), p(rw),
                                           p(ha), p(hb), C.c_size_t(hiding), p(rand), p(xy), p(inf), C.byref(s) if sess else None)
    return rc, int(s.value)


def _rc_ppc(c, sess, mu):
    p = lambda v: v.ctypes.data_as(C.c_void_p)
    k = max(mu.shape[0], 1)
    lo, hi, li, hf = np.zeros((k, 8), np.uint64), np.zeros((k, 8), np.uint64), np.zeros(k, np.uint8), np.zeros(k, np.uint8)
    return c._lib.accmsm_hp_prove_product_poly_comm(c._h, C.c_uint64(sess), p(mu), C.c_size_t(mu.shape[0]), p(lo), p(li), p(hi), p(hf))


def _rc_finish(c, sess, nu, beta, cap, n_w, hp=False):
    a, b, w = np.zeros((max(cap, 1), 4), np.uint64), np.zeros((max(cap, 1), 4), np.uint64), np.zeros((max(n_w, 1), 4), np.uint64)
    ol = (C.c_size_t * 2)()
    p = lambda v: v.ctypes.data_as(C.c_void_p)
    if hp:
        return c._lib.accmsm_hp_prove_finish(c._h, C.c_uint64(sess), p(nu), p(a), p(b), C.c_size_t(cap), ol)
    return c._lib.accmsm_nark_as_prove_finish(c._h, C.c_uint64(sess), p(nu), p(beta), C.c_size_t(beta.shape[0]), p(a), p(b), C.c_size_t(cap),
                                              ol, p(w))


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_argument_errors(ctx, devices):
    c = ctx if devices is None else ab.Context(devices=devices, min_shard=16)
    curve = 0
    f = cref.scalar_field(curve)
    M = 64
    mats, x, w = satisfying_system(f, M, 3, 20, 0x7F00)
    n_x, n_w = x.shape[0], w.shape[0]
    pts = cref.gen_points(curve, 0x7F10, M + 1)
    B = c.register_bases(curve, pts)
    short = c.register_bases(curve, pts[: M // 2])
    csr, csr2 = c.register_csr(f, mats), c.register_csr(f, mats[:2])
    fresh, accs, z = _case_inputs(curve, mats, x, w, 1, 2, True, True, 0x7F20)
    rx, rw, sr, ha, hb, hr = z
    rand = np.concatenate([sr, hr])
    xs, ws = [fresh[0][0]], [fresh[0][3]]
    aw, aa, bb = [a[1] for a in accs], [a[2] for a in accs], [a[3] for a in accs]
    hs_pts = cref.gen_points(curve, 0x7F30, M + 1)
    Bh = c.register_bases(curve, hs_pts)
    try:
        kw = dict(key=B.handle, csr=csr, xs=xs, n_x=n_x, ws=ws, n_w=n_w, aw=aw, aa=aa, bb=bb, rx=rx, rw=rw, ha=ha, hb=hb, hiding=M, rand=rand)
        rc = lambda **o: _rc_begin(c, **{**kw, **o})
        nozk = dict(rx=None, rw=None, ha=None, hb=None, rand=None)
        # not 3 matrices; n_fresh + n_acc outside 1..16; zk with one hp input; zk half given
        assert rc(csr=csr2)[0] == E_ARG
        assert rc(xs=[], ws=[], aw=[], aa=[], bb=[], **nozk)[0] == E_ARG
        assert rc(aw=aw * 8, aa=aa * 8, bb=bb * 8)[0] == E_ARG
        assert rc(aw=[], aa=[], bb=[])[0] == E_ARG and rc(aw=[], aa=[], bb=[], **nozk)[0] == 0
        for k in nozk:
            assert rc(**{k: None})[0] == E_ARG, k
        # an accumulator pair longer than the rows, rows or hiding index beyond the key, a column beyond input || witness
        long = cref.gen_scalars(f, 1, M + 1, True)
        assert rc(aa=[long, aa[1]])[0] == E_ARG and rc(bb=[bb[0], long], **nozk)[0] == E_ARG
        assert rc(key=short.handle, hiding=M // 2 - 1)[0] == E_ARG and rc(hiding=M + 1)[0] == E_ARG
        assert rc(n_w=n_w - 1)[0] == E_ARG and rc(n_w=n_w - 1, **nozk)[0] == E_ARG
        assert rc(sess=False)[0] == E_ARG
        assert rc(key=987654)[0] == E_HANDLE and rc(csr=987654)[0] == E_HANDLE
        mu = to_mont(f, mu_list(f, mu_stand_in(f, 3)(None), True))
        nu = to_mont(f, [12345]).reshape(4)
        beta = to_mont(f, [1, 5, 7, 9])
        # finish before product_poly_comm; wrong n_beta; each finish on the other kind of session: E_ARG, released
        r0, s = rc()
        assert r0 == 0 and _rc_finish(c, s, nu, beta, M, n_w) == E_ARG and _rc_ppc(c, s, mu) == E_HANDLE
        r0, s = rc()
        assert r0 == 0 and _rc_ppc(c, s, mu) == 0
        assert _rc_finish(c, s, nu, beta[:3], M, n_w) == E_ARG and _rc_finish(c, s, nu, beta, M, n_w) == E_HANDLE
        r0, s = rc()
        assert r0 == 0 and _rc_ppc(c, s, mu) == 0
        assert _rc_finish(c, s, nu, beta, M, n_w, hp=True) == E_ARG and c._lib.accmsm_hp_prove_abort(c._h, C.c_uint64(s)) == E_HANDLE
        from tests.test_gpu_hp_prove import _rc_begin as hp_begin
        r0, s = hp_begin(c, B.handle, aa, bb, 2, M)
        assert r0 == 0 and _rc_ppc(c, s, mu[:2]) == 0
        assert _rc_finish(c, s, nu, beta[:2], M, n_w) == E_ARG and _rc_ppc(c, s, mu[:2]) == E_HANDLE
        # an unknown session; abort of a NARK-AS session
        assert _rc_finish(c, 987654, nu, beta, M, n_w) == E_HANDLE
        r0, s = rc()
        assert r0 == 0 and c._lib.accmsm_hp_prove_abort(c._h, C.c_uint64(s)) == 0 and _rc_ppc(c, s, mu) == E_HANDLE
        # the context still works
        check_session(c, curve, B, csr, pts, M, mats, fresh, accs, z)
    finally:
        c.release_csr(csr); c.release_csr(csr2)
        B.release(); short.release(); Bh.release()
        if c is not ctx:
            c.close()


@pytest.mark.gpu
def test_prove_cycles_leave_device_memory_where_it_was(ctx):
    import torch
    curve = 0
    f = cref.scalar_field(curve)
    M = 1 << 14
    mats, x, w = satisfying_system(f, M, 4, 4000, 0x7F60)
    pts = cref.gen_points(curve, 0x7F61, M + 1)
    ck = ab.CommitterKey.new(ctx, curve, pts[:M], pts[M], precompute=True)
    nark = ab.R1CSNark(ck, mats, num_instance_variables=4)
    try:
        fresh, accs, z = _case_inputs(curve, mats, x, w, 1, 2, True, False, 0x7F70)
        first = mirror_prove(nark, curve, fresh, accs, z)
        torch.cuda.synchronize(0)
        free0 = torch.cuda.mem_get_info(0)[0]
        for _ in range(20):
            inst, wit, _ = mirror_prove(nark, curve, fresh, accs, z)
        torch.cuda.synchronize(0)
        free1 = torch.cuda.mem_get_info(0)[0]
        assert free0 - free1 <= (8 << 20), (free0, free1)
        assert np.array_equal(wit.r1cs_blinded_witness, first[1].r1cs_blinded_witness)
    finally:
        nark.release(); ck.bases.release()
