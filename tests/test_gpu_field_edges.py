"""The device build of the field and group arithmetic at the edges of the field, through the library's own kernels.

tests/test_host_limbs.py feeds edge values to the HOST build of fp.cuh / ec.cuh (emulated carry flag).  The device build
has the real add.cc / addc.cc / mad*.cc / add.cc.u64 chains, FpCall's out-of-line product and the cooperative group law of
coop.cuh, and the other GPU tests feed it seeded random elements: a carry that only ripples through a run of 0xffffffff
or 0 limbs turns up about once in 2^32 random operands.  Here the edge values reach the device through entry points that
already exist, each chosen for the primitive it runs, and every result is compared bit for bit with the C oracle
(oracle/cref.py) or with Python integers (oracle/pyref.py).

The edge sets are built and checked on the CPU (the test_edge_* tests and the window-table threshold); every other test
is marked gpu."""
import os
import re
from functools import lru_cache

import numpy as np
import pytest

import accumulation_b200 as ab
from accumulation_b200 import wire
from oracle import cref, pyref
from tests.util import same_point

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = pyref.R_MONT
MODULI = (pyref.P_PALLAS_BASE, pyref.Q_PALLAS_SCALAR)     # field ids: 0 = Fp, 1 = Fq; the base field id of a curve is its id
PALLAS, VESTA = pyref.PALLAS, pyref.VESTA
FIELDS = pytest.mark.parametrize("field", [0, 1])
CURVES = pytest.mark.parametrize("curve", [PALLAS, VESTA])

# ---- edge sets ---------------------------------------------------------------------------------------------------------
# Edge points whose x integer, or whose x Montgomery image, is one of the six values nearest 0 or p that give a point
# (searched in the order 1, -1, 2, -2, ..., negative = p - d; x = p - 1 is the generator's and is skipped)
X_INTEGERS = {PALLAS: (1, -2, 3, 4, -4, 5), VESTA: (1, -2, 3, -3, 5, -6)}
X_IMAGES = {PALLAS: (1, -1, 2, 3, -3, 4), VESTA: (-1, 2, 3, -3, 4, -4)}
# Points next to the PositiveY boundary: y = (p - 1) / 2 - d and -y = (p + 1) / 2 + d agree above their low limb, so only
# the low limb decides which root the flag names.  The first d is the nearest y for which y^2 - 5 is a cube; the second is
# the nearest after it for which Fp::sqrt(y^2) returns the other root, so the flag must flip the root in both directions.
# x is a cube root of y^2 - 5 (a general cube root, such as sympy's nthroot_mod, takes minutes here, so they are kept and
# checked instead).
Y_HALF = {PALLAS: ((5, 0x2801CF79D30B618A2BBA96B4C822F34BEE2C7B2711A458BA080DB6B86A73590C),
                   (11, 0x137858148C955F30A65369F01574D5F0C81F458E0AAA56DE3C37C313B5D5BB38)),
          VESTA: ((1, 0x3D8D6363F4BC4EBAA84CB6BFE2FF15DAD0C13DB41CFDDEE99C4F04AA70FB48D7),
                  (5, 0x1FFB3A4A30D290A73DE412776935A60BE3E324F3509711FC96CBD034192F30F5))}
# The window tables are checked on two keys, one on each side of PRECOMPUTE_COOP_MAX (accmsm.cu): the edge key itself runs
# k_precompute_coop (FpCall, coop doubling, binary-GCD inversion), the edge key padded with seeded points to TABLE_KEY_N
# runs k_precompute (inline Fp, Fermat inversion).
TABLE_KEY_N = 4097


@lru_cache(maxsize=None)
def image_edges(field):
    """Montgomery images at the edges of the field (the kernels see images, so the edges are images)"""
    m = MODULI[field]
    one = R % m
    return (0, 1, 2, (1 << 32) - 1, 1 << 32, (1 << 224) - 1, (1 << 254) - 1, m >> 1, (m + 1) // 2, m - (1 << 32), m - 2, m - 1,
            one, one - 1, one & ~(0xFFFFFFFF << 128), R * R % m, R ** 3 % m, (1 << 255) % m)


def edges(field):
    return cref.ints_to_arr(image_edges(field))


def img(field, x):
    """Montgomery image of the integer x"""
    m = MODULI[field]
    return x % m * R % m


def img_arr(field, xs):
    return cref.ints_to_arr([img(field, x) for x in xs])


def root_of_unity(field):
    """5^T with p - 1 = 2^32 T: a primitive 2^32-th root of unity (Fp::root_of_unity)"""
    m = MODULI[field]
    return pow(5, (m - 1) >> 32, m)


def is_x_on_curve(curve, x):
    m = MODULI[curve]
    return pyref.sqrt_mod((x ** 3 + 5) % m, m) is not None


@lru_cache(maxsize=None)
def edge_points(curve):
    """canonical (x, y) of G, 2G, 3G, the x-integer, x-image and y-near-half points, each followed by its negation"""
    m = MODULI[curve]
    rinv = pow(R, -1, m)

    def lift(x):
        return (x, pyref.sqrt_mod((x ** 3 + 5) % m, m))
    g = pyref.generator(curve)
    base = [g, pyref.add(g, g, curve), pyref.mul(3, g, curve)]
    base += [lift(x % m) for x in X_INTEGERS[curve]]
    base += [lift(v % m * rinv % m) for v in X_IMAGES[curve]]
    base += [(x, (m - 1) // 2 - d) for d, x in Y_HALF[curve]]
    return tuple(q for P in base for q in (P, pyref.neg(P, curve)))


def points_image(curve, pts):
    return cref.ints_to_arr([img(curve, c) for P in pts for c in P]).reshape(-1, 8)


def edge_key(curve):
    """every edge point twice, then its negation: buckets, folds and table chains meet equal and opposite edge points"""
    pts = edge_points(curve)
    return points_image(curve, [q for P in pts for q in (P, P, pyref.neg(P, curve))])


def edge_scalars(curve):
    """canonical scalars at the edges of the scalar field"""
    r = pyref.scalar_modulus(curve)
    return (0, 1, 2, r - 1, r - 2, (r - 1) // 2, (r + 1) // 2, 1 << 253, (1 << 254) - 1, r - (1 << 64))


def tiled(a, n):
    return np.ascontiguousarray(np.resize(np.asarray(a, np.uint64), (n, a.shape[1])))


def coop_max():
    src = open(os.path.join(ROOT, "accumulation_b200", "csrc", "accmsm.cu")).read()
    mt = re.search(r"constexpr size_t PRECOMPUTE_COOP_MAX = 1u << (\d+);", src)
    assert mt and "B.n <= PRECOMPUTE_COOP_MAX" in src
    return 1 << int(mt.group(1))


# ---- 1. the edge sets, on the CPU --------------------------------------------------------------------------------------
@FIELDS
def test_edge_images_are_canonical(field):
    m = MODULI[field]
    vals = image_edges(field)
    assert len(set(vals)) == len(vals) and all(0 <= v < m for v in vals)
    # Fp::one() (fp.cuh) is R mod m; one - 1 and one with limb 4 cleared each differ from it in a single 32-bit limb
    one = cref.to_int(cref.to_mont(field, cref.ints_to_arr([1]))[0])
    assert vals[12] == one

    def limbs_differing(a, b):
        return [i for i in range(8) if (a >> (32 * i)) & 0xFFFFFFFF != (b >> (32 * i)) & 0xFFFFFFFF]
    assert limbs_differing(vals[13], one) == [0] and limbs_differing(vals[14], one) == [4]
    w = root_of_unity(field)
    assert pow(w, 1 << 31, m) == m - 1


@CURVES
def test_edge_points_are_on_the_curve(curve):
    m = MODULI[curve]
    assert not is_x_on_curve(curve, 0)                               # x = 0: 5 is not a square; the decompression test relies on it
    rinv = pow(R, -1, m)

    def nearest_ends(x_of, skip):
        found = [v for d in range(1, 40) for v in (d, -d) if v != skip and is_x_on_curve(curve, x_of(v))]
        return tuple(found[:6])
    assert nearest_ends(lambda v: v % m, -1) == X_INTEGERS[curve]
    assert nearest_ends(lambda v: v % m * rinv % m, None) == X_IMAGES[curve]
    (d1, _), (d2, _) = Y_HALF[curve]

    def sqrt_returns_larger(y):                                      # wire._sqrt takes the steps of Fp::sqrt
        r = wire._sqrt(curve, y * y % m)
        return r > m - r
    cubes = [e for e in range(d2 + 1) if pow((((m - 1) // 2 - e) ** 2 - 5) % m, (m - 1) // 3, m) == 1]
    assert cubes[0] == d1 and cubes[-1] == d2
    first = sqrt_returns_larger((m - 1) // 2 - d1)
    assert [sqrt_returns_larger((m - 1) // 2 - e) != first for e in cubes] == [False] * (len(cubes) - 1) + [True]
    for d, _ in Y_HALF[curve]:
        y = (m - 1) // 2 - d
        assert y >> 32 == (m - y) >> 32
    pts = edge_points(curve)
    assert len(set(pts)) == len(pts) == 34
    assert all(pyref.on_curve(P, curve) for P in pts)
    xy = points_image(curve, pts)
    assert all(cref.on_curve(curve, row) for row in xy)
    assert cref.to_int(xy[0, :4]) == img(curve, m - 1) and cref.to_int(xy[0, 4:]) == img(curve, 2)     # G = (-1, 2)
    near_half = [P for P in pts if abs(P[1] - (m - 1) // 2) <= d2 + 1]
    assert [P[1] > m - P[1] for P in near_half] == [False, True, False, True]     # both sides of the PositiveY flag


@CURVES
def test_edge_scalars_in_both_forms(curve):
    r = pyref.scalar_modulus(curve)
    sf = cref.scalar_field(curve)
    canon = cref.ints_to_arr(edge_scalars(curve))
    assert all(0 <= s < r for s in edge_scalars(curve))
    mont = cref.to_mont(sf, canon)
    assert np.array_equal(cref.from_mont(sf, mont), canon)
    assert [cref.to_int(v) for v in mont] == [img(sf, s) for s in edge_scalars(curve)]


def test_table_keys_sit_on_either_side_of_the_coop_threshold():
    """precompute_table picks k_precompute_coop up to PRECOMPUTE_COOP_MAX points and k_precompute above; both count as one
    launch, so the key sizes of test_window_table_entries are pinned to the constant here"""
    n = len(edge_key(PALLAS))
    assert n == len(edge_key(VESTA)) == 102
    assert n <= coop_max() < TABLE_KEY_N


# ---- 2. field arithmetic through the vector kernels --------------------------------------------------------------------
def cross(field):
    e = edges(field)
    return np.repeat(e, len(e), axis=0), np.tile(e, (len(e), 1))


@pytest.mark.gpu
@FIELDS
@pytest.mark.parametrize("n", [324, 65537])
def test_fp_mul_hadamard(ctx, field, n):
    """Fp::mul in k_hadamard: every pair of edge images (18 x 18 = 324), also repeated over 257 blocks"""
    a, b = (tiled(v, n) for v in cross(field))
    assert np.array_equal(ctx.hadamard(field, a, b), cref.hadamard(field, a, b))


@pytest.mark.gpu
@FIELDS
def test_fp_mul_broadcast_scale(ctx, field):
    """Fp::mul in k_scale: every edge image as the coefficient over the whole edge set"""
    e = edges(field)
    for c in e:
        assert np.array_equal(ctx.scale(field, e, c), cref.scale(field, e, c))


@pytest.mark.gpu
@FIELDS
def test_fp_add_reduce_once_lincomb(ctx, field):
    """Fp::add + reduce_once in k_lincomb with unit challenges: sums that land on exactly m are stored as 0"""
    m = MODULI[field]
    one = img_arr(field, [1])
    a, b = cross(field)
    ones2 = np.repeat(one, 2, axis=0)
    assert np.array_equal(ctx.lincomb(field, [a, b], ones2), cref.combine_vectors(field, [a, b], ones2))
    vals = image_edges(field)
    neg = cref.ints_to_arr([(m - v) % m for v in vals])
    assert not ctx.lincomb(field, [edges(field), neg], ones2).any()             # (a, m - a) -> 0, not m
    top = cref.ints_to_arr([m - 1] * 1000)
    ones16 = np.repeat(one, 16, axis=0)
    got = ctx.lincomb(field, [top] * 16, ones16)                                  # VEC_MAX_INPUTS inputs of m - 1
    assert np.array_equal(got, cref.combine_vectors(field, [top] * 16, ones16))
    assert np.array_equal(got, np.repeat(cref.ints_to_arr([m - 16]), 1000, axis=0))
    rows = [tiled(np.roll(edges(field), i, axis=0), 300 - 7 * i) for i in range(16)]
    ch = tiled(edges(field), 16)
    assert np.array_equal(ctx.lincomb(field, rows, ch), cref.combine_vectors(field, rows, ch))
    hid = tiled(np.roll(edges(field), 5, axis=0), 333)                           # hiding_ch absent: h = 1
    got = ctx.lincomb(field, rows, ones16, hid)
    assert got.shape[0] == 333 and np.array_equal(got, cref.combine_vectors(field, rows, ones16, hid))


@pytest.mark.gpu
@FIELDS
@pytest.mark.parametrize("n", [1, 16, 17, 4096, (1 << 20) + 1])
def test_fp_sqr_block_sum_poly_evaluate(ctx, field, n):
    """Fp::sqr (powers of z), block_sum and k_field_sum in k_poly_eval_partial: edge coefficients at edge points.  2^20 + 1
    coefficients take the chunk = 64 branch (poly_chunk, vec.cuh); z = one gives the field sum of the edge addends"""
    m = MODULI[field]
    cf = tiled(edges(field), n)
    one = R % m
    zs = [0, one, m - one, img(field, root_of_unity(field))] + list(image_edges(field))
    for z in cref.ints_to_arr(zs):
        assert np.array_equal(ctx.poly_evaluate(field, cf, z), cref.poly_evaluate(field, cf, z).reshape(4)), cref.to_int(z)
    vals = image_edges(field)                                                   # the image of a sum is the sum of the images
    total = (n // len(vals) * sum(vals) + sum(vals[: n % len(vals)])) % m
    assert cref.to_int(ctx.poly_evaluate(field, cf, cref.ints_to_arr([one])[0])) == total


@pytest.mark.gpu
@FIELDS
@pytest.mark.parametrize("k", [1, 6, 11])
def test_challenge_products_coeff_tables(ctx, field, k):
    """products of challenges in k_coeff_tables / k_coeffs_from_tables: all one (every coefficient is one), all -one (+-one
    by the parity of the index), edge challenges, edge alphas and an edge random polynomial"""
    m = MODULI[field]
    one = R % m
    ch_one = cref.ints_to_arr([one] * k)
    got = ctx.compute_coeffs(field, ch_one)
    assert np.array_equal(got, cref.ints_to_arr([one] * (1 << k)))
    ch_neg = cref.ints_to_arr([m - one] * k)
    got = ctx.compute_coeffs(field, ch_neg)
    assert np.array_equal(got, cref.ints_to_arr([m - one if bin(j).count("1") & 1 else one for j in range(1 << k)]))
    e = edges(field)
    for shift in (0, 7, 12):
        ch = tiled(np.roll(e, -shift, axis=0), k)
        assert np.array_equal(ctx.compute_coeffs(field, ch), cref.compute_coeffs(field, ch))
    chm = np.stack([ch_one, ch_neg, tiled(np.roll(e, -3, axis=0), k), tiled(np.roll(e, -9, axis=0), k)])
    alphas = tiled(np.roll(e, -10, axis=0), 4)                                   # m - 2, m - 1, one, one - 1
    rp = tiled(e, min(len(e), 1 << k))
    assert np.array_equal(ctx.combine_check_polys(field, chm, alphas, rp), cref.combine_check_polys(field, chm, alphas, rp))
    assert np.array_equal(ctx.combine_check_polys(field, chm, alphas), cref.combine_check_polys(field, chm, alphas))


@pytest.mark.gpu
@FIELDS
@pytest.mark.parametrize("n_in,zk", [(2, False), (2, True), (16, False), (16, True)])
def test_convolution_tvecs(ctx, field, n_in, zk):
    """Fp::mul / Fp::add of the convolution in k_tvecs: mu = one and edge mu, a and b from the edge set; n_in = 16 is the
    shared-memory opt-in at its limit (accmsm.cu)"""
    L = 1000
    e = edges(field)
    a = [tiled(np.roll(e, i, axis=0), L - 3 * i) for i in range(n_in)]
    b = [tiled(np.roll(e, -5 * i, axis=0), L - i) for i in range(n_in)]
    ha = tiled(np.roll(e, 2, axis=0), L) if zk else None
    hb = tiled(np.roll(e, 9, axis=0), L - 1) if zk else None
    for mu in (tiled(img_arr(field, [1]), n_in + 1), tiled(np.roll(e, -4, axis=0), n_in + 1)):
        got = ctx.tvecs(field, a, b, mu, L, ha, hb)
        assert np.array_equal(got, np.asarray(cref.tvecs(field, a, b, mu, L, ha, hb)).reshape(got.shape))


@pytest.mark.gpu
@FIELDS
def test_eq_one_fast_path_csr_matvec(ctx, field):
    """F::eq(cf, one) in k_csr_matvec: a coefficient of exactly one passes z through, one - 1 and one with limb 4 cleared
    (each differs from one in one limb) and zero must multiply; columns n_input - 1 and n_input sit on the input / witness
    boundary; z is the edge set"""
    m = MODULI[field]
    one = R % m
    z = edges(field)
    n_in = 5
    inp, wit = z[:n_in], z[n_in:]
    cf_vals = [one, one - 1, one & ~(0xFFFFFFFF << 128), 0] + list(image_edges(field))
    cols_b = [n_in - 1, n_in, 0, len(z) - 1]
    n_rows = len(cf_vals) * len(cols_b)

    def csr(rows):
        rp = np.cumsum([0] + [len(r) for r in rows]).astype(np.uint32)
        cols = np.array([c for r in rows for _, c in r], np.uint32)
        return rp, cols, cref.ints_to_arr([v for r in rows for v, _ in r])
    single = [[(cf_vals[r // len(cols_b)], cols_b[r % len(cols_b)])] for r in range(n_rows)]
    full = [[(cf_vals[(r + j) % len(cf_vals)], j) for j in range(len(z))] for r in range(n_rows)]
    pairs = [[] if r % 5 == 0 else [(cf_vals[r % len(cf_vals)], n_in - 1), (cf_vals[7 * r % len(cf_vals)], n_in)] for r in range(n_rows)]
    mats = [csr(single), csr(full), csr(pairs)]
    outs = ab.matrix_vec_mul(ctx, field, mats, inp, wit)
    for (rp, cl, cf), o in zip(mats, outs):
        assert np.array_equal(o, cref.csr_matvec(field, rp, cl, cf, inp, wit))
    vals = image_edges(field)
    for r in range(4 * len(cols_b)):                                            # the four near-one coefficients, one column each
        zv = vals[cols_b[r % len(cols_b)]]
        want = zv if r < len(cols_b) else (cf_vals[r // len(cols_b)] * zv * pow(R, -1, m)) % m
        assert cref.to_int(outs[0][r]) == want


# ---- 3. square roots and encodings -------------------------------------------------------------------------------------
@pytest.mark.gpu
@CURVES
def test_sqrt_and_encodings_wire_round_trip(ctx, curve):
    """Fp::sqrt, to_mont / from_mont, neg and lt in k_wire_decompress / k_wire_compress on every edge point; the four points
    next to (p - 1) / 2 pin the root choice from the PositiveY flag whichever root Fp::sqrt returns"""
    xy = points_image(curve, edge_points(curve))
    data = wire.key_to_compressed(curve, xy)
    B = ctx.register_bases_compressed(curve, data)
    try:
        assert np.array_equal(ctx.download_bases(B), xy)
        assert ctx.serialize_bases(B) == data
    finally:
        B.release()


@pytest.mark.gpu
@CURVES
def test_invalid_x_fails_decompress(ctx, curve):
    """x = 0 (x^3 + 5 = 5 is not a square), x = p, p + 1 and 2^256 - 1 (not canonical), neither flag set: an error return"""
    m = MODULI[curve]
    good = wire.key_to_compressed(curve, points_image(curve, edge_points(curve)))
    for x in (0, m, m + 1, (1 << 256) - 1):
        rec = x.to_bytes(32, "little") + b"\x00"
        with pytest.raises(ab.AccmsmError):
            ctx.register_bases_compressed(curve, rec)
        data = bytearray(good)
        data[33 * 5:33 * 6] = rec
        with pytest.raises(ab.AccmsmError):
            ctx.register_bases_compressed(curve, bytes(data))


# ---- 4. group law on edge points ---------------------------------------------------------------------------------------
def scalar_sets(curve, n):
    """-> [(scalars, montgomery)]: edge scalars canonical and as images, seeded random images, all one"""
    sf = cref.scalar_field(curve)
    canon = tiled(cref.ints_to_arr(edge_scalars(curve)), n)
    return [(canon, False), (cref.to_mont(sf, canon), True), (cref.gen_scalars(sf, 900 + curve, n, True), True),
            (tiled(img_arr(sf, [1]), n), True)]


def oracle_msm(curve, key, sc, mont):
    return cref.commit(curve, key, sc) if mont else cref.msm_ark(curve, key, sc)


@pytest.mark.gpu
@CURVES
def test_group_law_plain_msm(ctx, curve):
    """madd / add / dbl of ec.cuh on a plain key of edge points, equal and opposite ones in the same buckets"""
    key = edge_key(curve)
    B = ctx.register_bases(curve, key)
    try:
        for sc, mont in scalar_sets(curve, len(key)):
            assert same_point(ctx.msm(B, sc, montgomery=mont), oracle_msm(curve, key, sc, mont))
    finally:
        B.release()


_TABLE_CACHE = {}


def expected_table(curve, c):
    """[w, i] -> 2^(c w) * key_i from the oracle, w < ceil(256 / c)"""
    if (curve, c) not in _TABLE_CACHE:
        key = edge_key(curve)
        nwin = -(-256 // c)
        step = cref.from_int(1 << c)
        out = np.empty((nwin, len(key), 8), np.uint64)
        for i, P in enumerate(key):
            cur = P
            for w in range(nwin):
                out[w, i] = cur
                cur, inf = cref.point_mul(curve, cur, 0, step)
                assert not inf
        _TABLE_CACHE[(curve, c)] = out
    return _TABLE_CACHE[(curve, c)]


@pytest.mark.gpu
@CURVES
@pytest.mark.parametrize("c", [8, 13])
@pytest.mark.parametrize("builder", ["coop", "plain"])
def test_window_table_entries(ctx, curve, c, builder):
    """k_precompute_coop (edge key, <= PRECOMPUTE_COOP_MAX points) and k_precompute (padded to TABLE_KEY_N points): after
    precompute(c), the one-hot scalar 2^(c w) on base i returns table entry w of base i alone"""
    assert not int(os.environ.get("ACCMSM_NO_COOP_PRECOMPUTE", "0"))        # the knob would move every key off the coop builder
    edge = edge_key(curve)
    n = len(edge)
    key = edge if builder == "coop" else np.concatenate([edge, cref.gen_points(curve, 910 + curve, TABLE_KEY_N - n)])
    assert (len(key) <= coop_max()) == (builder == "coop")
    nwin = -(-256 // c)
    sc = np.zeros((nwin, n, n, 4), np.uint64)
    for w in range(nwin):
        sc[w, np.arange(n), np.arange(n)] = cref.from_int(1 << (c * w))
    ctx.set_window_bits(0)                                                   # auto: the MSM uses the key's table
    B = ctx.register_bases(curve, key).precompute(c)
    try:
        xy, inf = ctx.msm_batch(B, sc.reshape(nwin * n, n, 4), montgomery=False)
    finally:
        B.release()
    assert not inf.any()
    exp = expected_table(curve, c)
    bad = [(w, i) for w in range(nwin) for i in range(n) if not np.array_equal(xy[w * n + i], exp[w, i])]
    assert not bad, bad[:10]


@pytest.mark.gpu
@CURVES
def test_unregistered_bases_oneshot(ctx, curve):
    """msm_oneshot and msm_oneshot_batch (bases that are not a registered key) on the edge points"""
    key = edge_key(curve)
    sets = scalar_sets(curve, len(key))
    for sc, mont in sets:
        assert same_point(ctx.msm_oneshot(curve, key, sc, montgomery=mont), oracle_msm(curve, key, sc, mont))
    mont_sets = [sc for sc, mont in sets if mont]
    xy, inf = ctx.msm_oneshot_batch(curve, np.stack([key] * len(mont_sets)), np.stack(mont_sets))
    for j, sc in enumerate(mont_sets):
        assert same_point((xy[j], inf[j]), cref.commit(curve, key, sc))


@pytest.mark.gpu
@CURVES
@pytest.mark.parametrize("k", [5, 8])
def test_ipa_final_key_unit_challenges(ctx, curve, k):
    """h(X) of challenges +-one (every coefficient +-one, every scalar extreme) over edge points: ipa_final_key and
    ipa_check_final_key against the oracle's fold.  k = 8 on 256 points takes the half-table path (ipa_half_tables)"""
    sf = cref.scalar_field(curve)
    q = pyref.scalar_modulus(curve)
    edge = edge_key(curve)
    key = edge if (1 << k) <= len(edge) else np.concatenate([edge, cref.gen_points(curve, 920 + curve, (1 << k) - len(edge))])
    one = R % q
    B = ctx.register_bases(curve, key)
    try:
        folds = []
        for signs in ([1] * k, [-1] * k, [(-1) ** i for i in range(k)]):
            ch = cref.ints_to_arr([one if s > 0 else q - one for s in signs])
            exp = cref.ipa_fold_key(curve, key[: 1 << k], ch)
            assert same_point(ctx.ipa_final_key(B, ch), exp)
            ok, out, inf = ctx.ipa_check_final_key(B, ch, exp[0], exp[1])
            assert ok and same_point((out, inf), exp)
            folds.append(exp)
        assert not same_point(folds[0], folds[1])
        assert not ctx.ipa_check_final_key(B, ch, folds[0][0], folds[0][1])[0]      # the last challenges against the first fold
    finally:
        B.release()
