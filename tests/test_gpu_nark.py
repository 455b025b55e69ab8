"""The R1CS NARK prove (zk) and verify of src/r1cs_nark_as/r1cs_nark/mod.rs (:183-316, :335-419) on the device: one vector
launch (k_nark_rows) and one pass of the MSM pipeline per call (accmsm_nark_prove_zk: 8 commitments; accmsm_nark_verify: 4).

The oracle side is restated here from the reference over the oracle primitives (csr_matvec, hadamard, fe_*, commit,
point_mul, point_add).  The unmarked tests check that restatement on small seeded systems without a GPU; the gpu tests
compare every vector and commitment of both calls bit for bit with it, on both curves, on one context and on device groups."""
import ctypes as C
import hashlib

import numpy as np
import pytest

import accumulation_b200 as ab
from oracle import cref
from tests.util import fe_ints, same_point
from tests.test_gpu_fused import scaling_nark_matrices
from tests.test_gpu_msm_dispatch import plan, table_window_bits

E_ARG, E_HANDLE = -2, -3
_Q0 = 0x40000000000000000000000000000000224698FC094CF91B992D30ED00000001
_Q1 = 0x40000000000000000000000000000000224698FC0994A8DD8C46EB2100000001   # scalar moduli: Fp, Fq


# ---- oracle restatement (SURVEY App. C.9) -------------------------------------------------------------------------------
def _gamma_canon(field, gamma_mont):
    return cref.from_mont(field, np.asarray(gamma_mont, dtype=np.uint64).reshape(1, 4)).reshape(4)


def _scalar(field, gamma_mont, n):
    return np.repeat(np.asarray(gamma_mont, dtype=np.uint64).reshape(1, 4), n, axis=0)


def oracle_nark_prove(curve, mats, gens, h, inp, wit, gamma_fn, zk=None):
    """R1CSNark::prove -> (vectors, first_msg, gamma, w', sigmas); zk = (r, blinders[8]: A, B, C, rA, rB, rC, 1, 2)"""
    f = cref.scalar_field(curve)
    inp, wit = np.asarray(inp, np.uint64).reshape(-1, 4), np.asarray(wit, np.uint64).reshape(-1, 4)
    n_rows = np.asarray(mats[0][0]).size - 1
    g = gens[:n_rows]
    z = [cref.csr_matvec(f, *m, inp, wit) for m in mats]                              # z_M = M (x || w)
    if zk is None:
        return z, [cref.commit(curve, g, v) for v in z], None, wit, None
    r, bl = np.asarray(zk[0], np.uint64).reshape(-1, 4), np.asarray(zk[1], np.uint64).reshape(8, 4)
    rv = [cref.csr_matvec(f, *m, np.zeros_like(inp), r) for m in mats]                # r_M = M (0 || r)
    cross = cref.fe_add(f, cref.hadamard(f, z[0], rv[1]), cref.hadamard(f, z[1], rv[0]))
    rr = cref.hadamard(f, rv[0], rv[1])
    vecs = z + rv + [cross, rr]
    first = [cref.commit(curve, g, v, h, bl[j]) for j, v in enumerate(vecs)]
    gamma = np.asarray(gamma_fn(first), np.uint64).reshape(4)
    w_prime = cref.fe_add(f, wit, cref.fe_mul(f, _scalar(f, gamma, wit.shape[0]), r)) if wit.shape[0] else wit
    gm = gamma.reshape(1, 4)
    sig = [cref.fe_add(f, bl[i:i + 1], cref.fe_mul(f, gm, bl[3 + i:4 + i])) for i in range(3)]
    sig.append(cref.fe_add(f, cref.fe_add(f, bl[2:3], cref.fe_mul(f, gm, bl[6:7])), cref.fe_mul(f, cref.fe_mul(f, gm, gm), bl[7:8])))
    return vecs, first, gamma, w_prime, np.concatenate(sig)


def oracle_lhs(curve, first, gamma_mont):
    """comm_M + gamma comm_rM (M = A, B, C) and comm_C + gamma comm_1 + gamma^2 comm_2; without zk comm_A, comm_B, comm_C, comm_C"""
    if len(first) == 3:
        return [first[0], first[1], first[2], first[2]]
    f = cref.scalar_field(curve)
    g = _gamma_canon(f, gamma_mont)
    g2 = cref.from_int(cref.to_int(g) ** 2 % [_Q0, _Q1][f])

    def axpy(p, q, s):
        return cref.point_add(curve, p[0], p[1], *cref.point_mul(curve, q[0], q[1], s))
    lhs = [axpy(first[i], first[3 + i], g) for i in range(3)]
    lhs.append(axpy(axpy(first[2], first[6], g), first[7], g2))
    return lhs


def oracle_nark_verify(curve, mats, gens, h, inp, first, gamma, w_prime, sigmas):
    """R1CSNark::verify -> (accept, [t_A, t_B, t_C], the 4 right-hand commitments)"""
    f = cref.scalar_field(curve)
    n_rows = np.asarray(mats[0][0]).size - 1
    g = gens[:n_rows]
    t = [cref.csr_matvec(f, *m, inp, w_prime) for m in mats]                          # t_M = M (x || w')
    prod = cref.hadamard(f, t[0], t[1])
    if sigmas is None:
        rhs = [cref.commit(curve, g, v) for v in t + [prod]]
    else:
        rhs = [cref.commit(curve, g, v, h, sigmas[j]) for j, v in enumerate(t + [prod])]
    lhs = oracle_lhs(curve, first, gamma)
    return all(same_point(a, b) for a, b in zip(lhs, rhs)), t, rhs


def gamma_stand_in(field):
    """host stand-in for the sponge over the first message"""
    def fn(first):
        hsh = hashlib.sha256(b"".join(np.asarray(p[0], np.uint64).tobytes() + bytes([int(p[1])]) for p in first)).digest()
        v = int.from_bytes(hsh, "little") % [_Q0, _Q1][field]
        return cref.to_mont(field, cref.from_int(v).reshape(1, 4)).reshape(4)
    return fn


# ---- systems --------------------------------------------------------------------------------------------------------------
def satisfying_system(field, M, n_in, n_free, seed, nnz=3):
    """A, B: nnz random entries per row over input || free witness; C row i = 1 * out_i, with out_i = (A z)_i (B z)_i placed
    after the free witness -> (mats, input, witness)"""
    rng = np.random.default_rng(seed)
    one = cref.to_mont(field, cref.from_int(1).reshape(1, 4))
    n_src = n_in + n_free
    mats = []
    for mi in range(2):
        row_ptr = np.arange(M + 1, dtype=np.uint32) * nnz
        cols = rng.integers(0, n_src, M * nnz).astype(np.uint32)
        coeffs = cref.gen_scalars(field, seed + mi, M * nnz, True)
        coeffs[::3] = one
        mats.append((row_ptr, cols, coeffs))
    mats.append((np.arange(M + 1, dtype=np.uint32), (n_src + np.arange(M)).astype(np.uint32), np.repeat(one, M, axis=0)))
    inp = cref.gen_scalars(field, seed + 10, n_in, True)
    inp[0] = one[0]
    free = cref.gen_scalars(field, seed + 11, n_free, True)
    part = np.concatenate([free, np.zeros((M, 4), np.uint64)])
    out = cref.hadamard(field, cref.csr_matvec(field, *mats[0], inp, part), cref.csr_matvec(field, *mats[1], inp, part))
    return mats, inp, np.concatenate([free, out])


def scaling_system(field, M, seed):
    """the scaling-nark circuit (tests/test_gpu_fused.py) with a satisfying witness a, b, a b, a b, ..."""
    mats, n_in, n_wit = scaling_nark_matrices(field, M)
    inp = cref.gen_scalars(field, seed, n_in, True)
    ab_ = cref.gen_scalars(field, seed + 1, 2, True)
    wit = np.concatenate([ab_, np.repeat(cref.hadamard(field, ab_[:1], ab_[1:]), n_wit - 2, axis=0)])
    return mats, inp, wit


def zk_randomness(field, n_wit, seed):
    return cref.gen_scalars(field, seed, n_wit, True), cref.gen_scalars(field, seed + 1, 8, True)


# ---- CPU: the restatement itself ------------------------------------------------------------------------------------------
def _cpu_case(curve, M=24, seed=5):
    f = cref.scalar_field(curve)
    mats, inp, wit = satisfying_system(f, M, 3, 5, seed)
    pts = cref.gen_points(curve, 0x4E00 + curve, M + 1)
    r, bl = zk_randomness(f, wit.shape[0], seed + 20)
    vecs, first, gamma, wp, sig = oracle_nark_prove(curve, mats, pts[:M], pts[M], inp, wit, gamma_stand_in(f), (r, bl))
    return f, mats, inp, wit, pts, r, vecs, first, gamma, wp, sig


@pytest.mark.parametrize("curve", [0, 1])
def test_oracle_proof_verifies_and_corruptions_reject(curve):
    f, mats, inp, wit, pts, r, vecs, first, gamma, wp, sig = _cpu_case(curve)
    M = pts.shape[0] - 1
    verify = lambda fm, g, w, s: oracle_nark_verify(curve, mats, pts[:M], pts[M], inp, fm, g, w, s)[0]
    assert verify(first, gamma, wp, sig)
    wb = wp.copy(); wb[1, 0] ^= np.uint64(1)
    assert not verify(first, gamma, wb, sig)
    sb = sig.copy(); sb[3, 2] ^= np.uint64(1)
    assert not verify(first, gamma, wp, sb)
    gb = gamma.copy(); gb[0] ^= np.uint64(1)
    assert not verify(first, gb, wp, sig)
    swapped = first[:6] + [first[7], first[6]]
    assert not verify(swapped, gamma, wp, sig)
    # non-zk: the commitments of z_M alone and w itself
    _, first0, _, w0, _ = oracle_nark_prove(curve, mats, pts[:M], pts[M], inp, wit, gamma_stand_in(f))
    assert verify(first0, None, w0, None)
    wb = wit.copy(); wb[0, 1] ^= np.uint64(1)
    assert not verify(first0, None, wb, None)


def test_oracle_r_vectors_are_the_matrices_times_zero_input_and_r():
    """r_M = M (0 || r): recomputed here with python ints from the CSR arrays"""
    f, mats, inp, wit, pts, r, vecs, *_ = _cpu_case(1, M=17, seed=9)
    q = [_Q0, _Q1][f]
    n_in = inp.shape[0]
    rs = fe_ints(f, r)
    for mi, (rp, cols, cf) in enumerate(mats):
        cfs = fe_ints(f, cf)
        exp = [sum(cfs[e] * rs[cols[e] - n_in] for e in range(rp[i], rp[i + 1]) if cols[e] >= n_in) % q for i in range(rp.size - 1)]
        assert fe_ints(f, vecs[3 + mi]) == exp, mi
        assert np.array_equal(vecs[3 + mi], cref.csr_matvec(f, rp, cols, cf, np.zeros_like(inp), r))


# ---- GPU ------------------------------------------------------------------------------------------------------------------
def _first_points(xy, inf):
    return [(xy[i], int(inf[i])) for i in range(xy.shape[0])]


def check_calls(c, curve, mats, inp, wit, key_pts, n_gens, bases, table_c, r, bl, count_launches=True):
    """nark_prove_zk and nark_verify on context c against the oracle: 8 vectors + 8 commitments, 3 vectors + 4 commitments,
    accept equal to the oracle's; one vector launch + one pass each"""
    f = cref.scalar_field(curve)
    M = np.asarray(mats[0][0]).size - 1
    gens, h = key_pts[:n_gens], key_pts[n_gens]
    csr = c.register_csr(f, mats)
    try:
        gam = gamma_stand_in(f)
        evecs, efirst, egamma, ewp, esig = oracle_nark_prove(curve, mats, gens, h, inp, wit, gam, (r, bl))
        before = c.kernel_launches()
        vecs, xy, inf = c.nark_prove_zk(bases, csr, M, inp, wit, r, bl, hiding_index=n_gens)
        if count_launches:
            assert c.kernel_launches() - before == (1 + plan(M + 1, 8, table_c=table_c).launches if M else 0)
        for j in range(8):
            assert np.array_equal(vecs[j], evecs[j]), ("vec", j)
            assert same_point((xy[j], inf[j]), efirst[j]), ("comm", j)
        ok_o, et, erhs = oracle_nark_verify(curve, mats, gens, h, inp, efirst, egamma, ewp, esig)
        lhs = oracle_lhs(curve, efirst, egamma)
        before = c.kernel_launches()
        ok, tv, vxy, vinf = c.nark_verify(bases, csr, M, inp, ewp, np.array([p[0] for p in lhs]), [p[1] for p in lhs],
                                          hiding_index=n_gens, sigmas=esig, want_vecs=True)
        if count_launches:
            assert c.kernel_launches() - before == (1 + plan(M + 1, 4, table_c=table_c).launches if M else 0)
        assert ok == ok_o
        for j in range(3):
            assert np.array_equal(tv[j], et[j]), ("t", j)
        for j in range(4):
            assert same_point((vxy[j], vinf[j]), erhs[j]), ("rhs", j)
        return ok, (vecs, xy, inf, tv, vxy, vinf)
    finally:
        c.release_csr(csr)


def _system(case):
    name, curve, M = case
    f = cref.scalar_field(curve)
    if name == "scaling":
        mats, inp, wit = scaling_system(f, M, 0x4E10)
    elif name == "dense":
        mats, n_in, n_wit = scaling_nark_matrices(f, M, dense=True, seed=7)
        inp, wit = cref.gen_scalars(f, 0x4E11, n_in, True), cref.gen_scalars(f, 0x4E12, n_wit, True)
    elif name == "no_witness":         # every column an input: n_witness = 0
        mats, inp, wit = satisfying_system(f, M, 6, 0, 0x4E13)
        inp = np.concatenate([inp, wit]); wit = np.zeros((0, 4), np.uint64)
    else:
        mats, inp, wit = satisfying_system(f, M, 4, max(M // 3, 1), 0x4E14)
    return mats, inp, wit


# (system, curve, M, key generators, table bits or None)
PARITY_CASES = [
    ("scaling", 0, 1 << 16, 1 << 16, "auto"),     # six constant jobs ending in 0 with two uniform ones in one 8-job pass
    ("dense", 1, 1 << 16, 1 << 16, None),
    ("scaling", 1, 1 << 20, 1 << 20, 20),         # the 8-job shape over a c = 20 table
    ("satisfying", 1, 3000, 5000, None),          # Vesta, key longer than M
    ("satisfying", 0, 1, 1, None),
    ("no_witness", 0, 40, 64, "auto"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", PARITY_CASES, ids=[f"{c[0]}-{'pallas' if c[1] == 0 else 'vesta'}-{c[2]}" for c in PARITY_CASES])
def test_nark_prove_and_verify_match_the_oracle(ctx, case):
    name, curve, M, n_gens, table = case
    f = cref.scalar_field(curve)
    mats, inp, wit = _system((name, curve, M))
    pts = cref.gen_points(curve, 0x4E20 + curve, n_gens + 1)
    B = ctx.register_bases(curve, pts)
    table_c = None
    if table is not None:
        B.precompute(0 if table == "auto" else table)
        table_c = table_window_bits(n_gens + 1, 0 if table == "auto" else table)
    try:
        r, bl = zk_randomness(f, wit.shape[0], 0x4E30)
        ok, _ = check_calls(ctx, curve, mats, inp, wit, pts, n_gens, B, table_c, r, bl)
        assert ok == (name != "dense")
    finally:
        B.release()


def _small_key(c, curve, n_gens, seed=0x4E40, precompute=False):
    pts = cref.gen_points(curve, seed + curve, n_gens + 1)
    return pts, ab.CommitterKey.new(c, curve, pts[:n_gens], pts[n_gens], precompute=precompute)


@pytest.mark.gpu
@pytest.mark.parametrize("curve", [0, 1])
def test_mirror_end_to_end(ctx, curve):
    """R1CSNark.prove / verify: a device proof verifies on the device and in the oracle, an oracle proof on the device, each
    corruption is rejected, and the non-zk forms accept and reject the same way"""
    f = cref.scalar_field(curve)
    M = 1500 + 37 * curve
    mats, inp, wit = satisfying_system(f, M, 5, 700, 0x4E50 + curve)
    pts, ck = _small_key(ctx, curve, M, precompute=True)
    nark = ab.R1CSNark(ck, mats)
    try:
        gam = gamma_stand_in(f)
        r, bl = zk_randomness(f, wit.shape[0], 0x4E60)
        proof = nark.prove(inp, wit, gam, zk=(r, bl))
        gamma = gam(proof.first_msg)
        assert nark.verify(inp, proof, gamma)
        assert oracle_nark_verify(curve, mats, pts[:M], pts[M], inp, proof.first_msg, gamma, proof.blinded_witness, proof.sigmas)[0]
        _, efirst, egamma, ewp, esig = oracle_nark_prove(curve, mats, pts[:M], pts[M], inp, wit, gam, (r, bl))
        assert all(same_point(a, b) for a, b in zip(proof.first_msg, efirst))
        assert np.array_equal(proof.blinded_witness, ewp) and np.array_equal(proof.sigmas, esig)
        assert nark.verify(inp, ab.NarkProof(efirst, ewp, esig), egamma)
        wb = proof.blinded_witness.copy(); wb[3, 1] ^= np.uint64(1)
        assert not nark.verify(inp, ab.NarkProof(proof.first_msg, wb, proof.sigmas), gamma)
        sb = proof.sigmas.copy(); sb[3, 0] ^= np.uint64(1)
        assert not nark.verify(inp, ab.NarkProof(proof.first_msg, proof.blinded_witness, sb), gamma)
        gb = gamma.copy(); gb[2] ^= np.uint64(1)
        assert not nark.verify(inp, proof, gb)
        swapped = proof.first_msg[:6] + [proof.first_msg[7], proof.first_msg[6]]
        assert not nark.verify(inp, ab.NarkProof(swapped, proof.blinded_witness, proof.sigmas), gamma)
        # without zk
        p0 = nark.prove(inp, wit, gam)
        assert p0.sigmas is None and len(p0.first_msg) == 3
        assert nark.verify(inp, p0)
        assert oracle_nark_verify(curve, mats, pts[:M], pts[M], inp, p0.first_msg, None, p0.blinded_witness, None)[0]
        wb = wit.copy(); wb[2, 0] ^= np.uint64(1)
        assert not nark.verify(inp, ab.NarkProof(p0.first_msg, wb, None))
        assert not nark.verify(inp, ab.NarkProof([p0.first_msg[1], p0.first_msg[0], p0.first_msg[2]], wit, None))
    finally:
        nark.release(); ck.bases.release()


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0]])
@pytest.mark.parametrize("long_key", [False, True])
def test_group_is_bit_identical(ctx, devices, long_key):
    """rows cut along the key's point ranges; with a key four times longer than M the rows sit on child 0 and the last child
    owns only the hiding generator"""
    curve = 1 if long_key else 0
    f = cref.scalar_field(curve)
    M = 3000
    n_gens = 4 * M if long_key else M
    mats, inp, wit = satisfying_system(f, M, 4, 900, 0x4E70)
    pts = cref.gen_points(curve, 0x4E80 + curve, n_gens + 1)
    r, bl = zk_randomness(f, wit.shape[0], 0x4E90)
    g = ab.Context(devices=devices, min_shard=16)
    B1 = ctx.register_bases(curve, pts)
    Bg = g.register_bases(curve, pts)
    try:
        ok1, res1 = check_calls(ctx, curve, mats, inp, wit, pts, n_gens, B1, None, r, bl)
        okg, resg = check_calls(g, curve, mats, inp, wit, pts, n_gens, Bg, None, r, bl, count_launches=False)
        assert ok1 and okg
        for a, b in zip(res1, resg):
            if isinstance(a, list):
                assert all(np.array_equal(x, y) for x, y in zip(a, b))
            else:
                assert np.array_equal(a, b)
        # verify without zk on the group as well
        csr = g.register_csr(f, mats)
        try:
            _, efirst, _, _, _ = oracle_nark_prove(curve, mats, pts[:n_gens], pts[n_gens], inp, wit, None)
            lhs = oracle_lhs(curve, efirst, None)
            ok, _, _, _ = g.nark_verify(Bg, csr, M, inp, wit, np.array([p[0] for p in lhs]), [p[1] for p in lhs], hiding_index=n_gens)
            assert ok
        finally:
            g.release_csr(csr)
    finally:
        B1.release(); Bg.release(); g.close()


def _prove_rc(c, key, csr, inp, n_in, wit, n_wit, r, hiding, bl):
    xy, inf = np.empty((8, 8), np.uint64), np.empty(8, np.uint8)
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    return c._lib.accmsm_nark_prove_zk(c._h, C.c_uint64(key), C.c_uint64(csr), p(inp), C.c_size_t(n_in), p(wit), C.c_size_t(n_wit), p(r),
                                       C.c_size_t(hiding), p(bl), None, p(xy), p(inf))


def _verify_rc(c, key, csr, inp, n_in, wit, n_wit, hiding, sig, exp=True, acc=True):
    e, ei = np.zeros((4, 8), np.uint64), np.zeros(4, np.uint8)
    a = C.c_int(0)
    p = lambda x: None if x is None else x.ctypes.data_as(C.c_void_p)
    return c._lib.accmsm_nark_verify(c._h, C.c_uint64(key), C.c_uint64(csr), p(inp), C.c_size_t(n_in), p(wit), C.c_size_t(n_wit),
                                     C.c_size_t(hiding), p(sig), p(e) if exp else None, p(ei) if exp else None,
                                     C.byref(a) if acc else None, None, None, None)


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_argument_errors(ctx, devices):
    c = ctx if devices is None else ab.Context(devices=devices, min_shard=16)
    curve = 0
    f = cref.scalar_field(curve)
    M = 64
    mats, inp, wit = satisfying_system(f, M, 3, 20, 0x4EA0)
    n_in, n_wit = inp.shape[0], wit.shape[0]
    pts = cref.gen_points(curve, 0x4EB0, M + 1)
    B = c.register_bases(curve, pts)
    short = c.register_bases(curve, pts[: M // 2])
    csr = c.register_csr(f, mats)
    csr2 = c.register_csr(f, mats[:2])
    other = c.register_csr(1 - f, mats)
    r, bl = zk_randomness(f, n_wit, 0x4EC0)
    sig = bl[:4].copy()
    try:
        assert _prove_rc(c, B.handle, csr, inp, n_in, wit, n_wit, r, M, bl) == 0
        assert _verify_rc(c, B.handle, csr, inp, n_in, wit, n_wit, M, sig) == 0
        for args in [(B.handle, csr2, M, bl), (B.handle, csr, M, None), (B.handle, other, M, bl), (short.handle, csr, M // 2 - 1, bl),
                     (B.handle, csr, M + 1, bl)]:
            key, cs, hid, b = args
            assert _prove_rc(c, key, cs, inp, n_in, wit, n_wit, r, hid, b) == E_ARG, args
            if b is not None:
                assert _verify_rc(c, key, cs, inp, n_in, wit, n_wit, hid, sig) == E_ARG, args
        # a column beyond input || witness
        assert _prove_rc(c, B.handle, csr, inp, n_in, wit, n_wit - 1, r, M, bl) == E_ARG
        assert _verify_rc(c, B.handle, csr, inp, n_in, wit, n_wit - 1, M, sig) == E_ARG
        assert _verify_rc(c, B.handle, csr, inp, n_in, wit, n_wit - 1, M, None) == E_ARG
        # null pointers
        assert _prove_rc(c, B.handle, csr, None, n_in, wit, n_wit, r, M, bl) == E_ARG
        assert _prove_rc(c, B.handle, csr, inp, n_in, None, n_wit, r, M, bl) == E_ARG
        assert _prove_rc(c, B.handle, csr, inp, n_in, wit, n_wit, None, M, bl) == E_ARG
        assert _verify_rc(c, B.handle, csr, None, n_in, wit, n_wit, M, sig) == E_ARG
        assert _verify_rc(c, B.handle, csr, inp, n_in, None, n_wit, M, sig) == E_ARG
        assert _verify_rc(c, B.handle, csr, inp, n_in, wit, n_wit, M, sig, exp=False) == E_ARG
        assert _verify_rc(c, B.handle, csr, inp, n_in, wit, n_wit, M, sig, acc=False) == E_ARG
        # unknown handles
        assert _prove_rc(c, 987654, csr, inp, n_in, wit, n_wit, r, M, bl) == E_HANDLE
        assert _prove_rc(c, B.handle, 987654, inp, n_in, wit, n_wit, r, M, bl) == E_HANDLE
        assert _verify_rc(c, 987654, csr, inp, n_in, wit, n_wit, M, sig) == E_HANDLE
        assert _verify_rc(c, B.handle, 987654, inp, n_in, wit, n_wit, M, sig) == E_HANDLE
        # the context still works
        assert _prove_rc(c, B.handle, csr, inp, n_in, wit, n_wit, r, M, bl) == 0
    finally:
        for h in (csr, csr2, other):
            c.release_csr(h)
        B.release(); short.release()
        if c is not ctx:
            c.close()


@pytest.mark.gpu
def test_no_rows_gives_the_blinder_terms(ctx):
    """n_rows = 0: prove gives blinder_j H, verify sigma_j H, and the identity without sigmas (as csr_matvec_commit)"""
    curve = 1
    f = cref.scalar_field(curve)
    mats = [(np.zeros(1, np.uint32), np.zeros(0, np.uint32), np.zeros((0, 4), np.uint64))] * 3
    pts = cref.gen_points(curve, 0x4ED0, 9)
    B = ctx.register_bases(curve, pts)
    csr = ctx.register_csr(f, mats)
    try:
        inp = cref.gen_scalars(f, 1, 2, True)
        bl = cref.gen_scalars(f, 2, 8, True)
        _, xy, inf = ctx.nark_prove_zk(B, csr, 0, inp, np.zeros((0, 4), np.uint64), np.zeros((0, 4), np.uint64), bl, hiding_index=8)
        for j in range(8):
            assert same_point((xy[j], inf[j]), cref.commit(curve, pts[:0], np.zeros((0, 4), np.uint64), pts[8], bl[j]))
        ident = np.zeros((4, 8), np.uint64)
        ok, _, vxy, vinf = ctx.nark_verify(B, csr, 0, inp, np.zeros((0, 4), np.uint64), ident, [1] * 4, hiding_index=8)
        assert ok and all(vinf)
    finally:
        ctx.release_csr(csr); B.release()


@pytest.mark.gpu
def test_cycles_leave_device_memory_where_it_was(ctx):
    import torch
    curve = 0
    f = cref.scalar_field(curve)
    M = 1 << 14
    mats, inp, wit = satisfying_system(f, M, 4, 4000, 0x4EE0)
    pts, ck = _small_key(ctx, curve, M, precompute=True)
    nark = ab.R1CSNark(ck, mats)
    try:
        gam = gamma_stand_in(f)
        r, bl = zk_randomness(f, wit.shape[0], 0x4EF0)
        first = nark.prove(inp, wit, gam, zk=(r, bl))
        assert nark.verify(inp, first, gam(first.first_msg))
        torch.cuda.synchronize(0)
        free0 = torch.cuda.mem_get_info(0)[0]
        for _ in range(20):
            p = nark.prove(inp, wit, gam, zk=(r, bl))
            assert all(same_point(a, b) for a, b in zip(p.first_msg, first.first_msg))
            assert nark.verify(inp, p, gam(p.first_msg))
        torch.cuda.synchronize(0)
        free1 = torch.cuda.mem_get_info(0)[0]
        assert free0 - free1 <= (8 << 20), (free0, free1)
    finally:
        nark.release(); ck.bases.release()
