"""Every branch of the IpaPC::open session, each case known to run the branch it is named for.

An opening session (accumulation_b200/csrc/ipa_api.inc, ipa.cuh) makes host-side decisions the proof must not depend on:
when to materialise the folded key (the fold policy of accmsm_set_ipa_fold), the shape of that materialisation (sub-digit
width, Horner groups, window slices, the MINB variant of k_fold_accumulate, the bail when the list heads do not fit), the
window bits of the new key's table, how many grid-stride passes the inner products make, whether the finish builds the
half tables of h(X), and how many coefficients one thread evaluates.  The session model below restates those decisions in
Python, citing the C++ line of each rule, and predicts the kernel launches of every session call.  Every GPU case asserts
those counts, so a case that silently ran the unfolded path (the materialisation bails without an error by design) fails.

The unmarked tests run without a GPU: the case table reaches every branch, the model reproduces the materialisation
shapes of the production degrees, and the signed sub-digits of k_fold_digits recompose the challenge products.  The GPU
tests compare every l and r, every challenge, the final key and c bit for bit with the oracle."""
from dataclasses import dataclass, field
from typing import Optional

import numpy as np
import pytest

import accumulation_b200 as ab
from oracle import cref, pyref
from tests.test_gpu_ipa_open import oracle_open, sponge_stand_in
from tests.test_gpu_msm_dispatch import plan, table_window_bits
from tests.util import fe_ints, same_point

# ---- constants of the session (ipa_api.inc, ipa.cuh, vec.cuh, accmsm.cu) --------------------------------------------------
IPA_IP_BLOCKS = 128             # ipa_api.inc:48
IP_THREADS = 256                # ipa_api.inc:524: k_ipa_inner_partial<<<grid, 256>>>
FOLD_MAX_KEYS = 8192            # ipa.cuh:173
FOLD_FILL = 50000               # ipa_api.inc:143: threads that fill the machine
FOLD_MINB4_WORK = 100000        # ipa_api.inc:169
FK_SMALL_MAX = (1 << 13) + 1    # ipa_api.inc:183
DEFAULT_POLICY = (5, 11)        # accmsm.cu:123


def poly_chunk(n):
    """coefficients per thread of k_poly_eval_partial (vec.cuh:79)"""
    return 64 if n > 1 << 20 else 16


def inner_product_passes(h):
    """(nparts, grid-stride passes of the busiest thread) of k_ipa_inner_partial over h products (ipa_api.inc:518, ipa.cuh:47)"""
    nparts = min(IPA_IP_BLOCKS, (h + 255) // 256)
    return nparts, -(-h // (nparts * IP_THREADS))


def half_tables(kk, n, no_ipa_tabs=False):
    """launches of ipa_half_tables: 1 when the MSM has at least 4x as many coefficients as the tables have entries
    (accmsm.cu:1520-1522), else 0 and the per-bit coefficient loop runs"""
    if kk < 8 or kk > 30 or no_ipa_tabs:
        return 0
    kl = kk // 2
    return 1 if n >= 4 * ((1 << kl) + (1 << (kk - kl))) else 0


def fk_table_bits(nk_n, fk_small_c=0):
    """window bits of a materialised key of nk_n points: ACCMSM_FK_C for short keys, else the key-size rule
    (ipa_api.inc:183, accmsm.cu:298)"""
    if nk_n <= FK_SMALL_MAX and 4 <= fk_small_c <= 20:
        return fk_small_c
    return table_window_bits(nk_n)


@dataclass
class FoldShape:
    round: int
    J: int
    m: int
    c: int
    nwin: int
    G: int
    cs: int
    widths: list
    WS: int
    nbk: int
    nlists: int
    minb: int
    outcome: str = ""           # "materialised", "bail" (nlists > FOLD_MAX_KEYS) or "identity"
    new_c: Optional[int] = None


def fold_shape(rnd, J, key_n, c):
    """FoldShape of ipa_materialise_key (ipa_api.inc:136-146) and the k_fold_accumulate variant (:169)"""
    nwin = -(-256 // c)
    m = key_n >> J
    G = max(1, (c + J // 2) // J)
    cs = -(-c // G)
    G = -(-c // cs)
    nbk = 1 << (cs - 1)
    want = (FOLD_FILL + m * G // 2) // (m * G)
    WS = min(4, nwin, max(1, want))
    widths = [min(cs, c - g * cs) for g in range(G)]          # fold_width (ipa.cuh:176)
    return FoldShape(rnd, J, m, c, nwin, G, cs, widths, WS, nbk, G * WS * (nbk + 1), 4 if m * G * WS >= FOLD_MINB4_WORK else 3)


@dataclass
class SessionModel:
    calls: list = field(default_factory=list)       # (kind, launches) of every session call in order
    folds: list = field(default_factory=list)       # FoldShape of every attempted materialisation that reached the shape
    ip_passes: set = field(default_factory=set)
    finish_tabs: int = 0


def model_session(k, rounds, min_log, table_c, indexed, fk_small_c=0, no_ipa_tabs=False, identity_rounds=()):
    """Launches of begin, every round, every fold and the finish of a 2^k opening.  table_c: window bits of the registered
    key's table (None: no table).  identity_rounds: rounds whose folded key holds an identity (the fold is abandoned)."""
    sm = SessionModel()
    n = 1 << k
    s_n, key_n, base, c, rnd = n, n, 0, table_c, 0
    sm.calls.append(("begin", 1 if indexed else 2))            # k_powers (+ k_ipa_hp_table for a point h', ipa_api.inc:107)

    def round_call():
        sm.ip_passes.add(inner_product_passes(s_n // 2)[1])
        n_pairs = key_n // 2 + (1 if indexed else 0)         # ipa_api.inc:545
        # inner products, their sum (+ k_ipa_hp_mul for a point h', :532), then one 2-job pass over the current key
        sm.calls.append(("round", (2 if indexed else 3) + plan(n_pairs, 2, table_c=c).launches))

    if k:
        round_call()
    while s_n > 1:
        s_n //= 2
        rnd += 1
        launches = 1                                           # k_ipa_fold_scalars (:615)
        # the policy fires on round - base_round == rounds only (:619-620): after a fallback it never fires again
        if rounds > 0 and rnd - base == rounds and s_n >= 2 and key_n >= 1 << min_log:
            J = rnd - base
            if c is not None and 1 <= J <= 10 and key_n >> J >= 1:        # :132
                f = fold_shape(rnd, J, key_n, c)
                if f.nlists > FOLD_MAX_KEYS:                                # :146
                    f.outcome = "bail"
                else:
                    launches += 3                                           # k_fold_digits / _accumulate / _combine (:168-176)
                    if rnd in identity_rounds:                              # :184
                        f.outcome = "identity"
                    else:
                        launches += 1                                       # the new key's window table
                        f.new_c = fk_table_bits(f.m + (1 if indexed else 0), fk_small_c)
                        f.outcome = "materialised"
                        c, key_n, base = f.new_c, f.m, rnd
                sm.folds.append(f)
        sm.calls.append(("fold", launches))
        if s_n >= 2:
            round_call()
    kk = k - base                                              # ipa_api.inc:707
    sm.finish_tabs = half_tables(kk, key_n, no_ipa_tabs)
    sm.calls.append(("finish", sm.finish_tabs + plan(key_n, 1, table_c=c).launches))
    return sm


# ---- the case table -------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    name: str
    curve: int
    k: int
    rounds: int = DEFAULT_POLICY[0]
    min_log: int = DEFAULT_POLICY[1]
    table: Optional[int] = 0        # precompute(table) on the key (0: the key-size rule); None: no table
    indexed: bool = False           # h' = xi_0 * key[2^k] given by index, else as a point
    fk_small_c: int = 0             # ACCMSM_FK_C of the context
    no_ipa_tabs: bool = False       # ACCMSM_NO_IPA_TABS of the context
    seed: int = 0

    @property
    def table_c(self):
        return None if self.table is None else table_window_bits((1 << self.k) + 1, self.table)

    def model(self, **kw):
        args = dict(k=self.k, rounds=self.rounds, min_log=self.min_log, table_c=self.table_c, indexed=self.indexed,
                    fk_small_c=self.fk_small_c, no_ipa_tabs=self.no_ipa_tabs)
        args.update(kw)
        return model_session(**args)


PROD_CASES = [
    Case("Pallas 2^18, default policy, h' by index (bench)", 0, 18, indexed=True, seed=18),
    Case("Vesta 2^17, default policy, h' as a point", 1, 17, seed=17),
    Case("Pallas 2^20, default policy, h' by index", 0, 20, indexed=True, seed=20),
]

SWEEP_CASES = [
    Case("2^14, fold every round from 2^14: c = 15, cs = 1, MINB 4", 0, 14, 1, 14),
    Case("2^16, 7 rounds from 2^11: c = 17, widths [9, 8]", 1, 16, 7, 11, indexed=True),
    Case("2^13, 3 rounds from 2^2: four materialisations, slots reused", 0, 13, 3, 2),
    Case("2^12, 10 rounds over a c = 21 table: nlists 8200 > 8192, bail", 1, 12, 10, 0, table=21, indexed=True),
    Case("2^15, 2 rounds from 2^13 over a c = 4 table: WS 3 twice", 1, 15, 2, 13, table=4),
    Case("2^12, 3 rounds from 2^2 over a c = 4 table: G = 1", 0, 12, 3, 2, table=4, indexed=True),
    Case("2^13, 4 rounds from 2^6 over a c = 10 table", 1, 13, 4, 6, table=10, indexed=True),
    Case("2^12 without a table: the policy never materialises", 0, 12, 2, 2, table=None),
]
FK_C_CASE = Case("2^13, 3 rounds from 2^2, ACCMSM_FK_C=12", 0, 13, 3, 2, fk_small_c=12)
NO_TABS_CASE = Case("Pallas 2^18, ACCMSM_NO_IPA_TABS=1", 0, 18, indexed=True, no_ipa_tabs=True, seed=18)
IDENTITY_K, IDENTITY_P0 = 6, 5
REUSE_OPENINGS = [(0, 14), (0, 6), (0, 14)]         # (curve, k) in order on one context, each with set_ipa_fold(2, 2)
INTERLEAVED = [Case("interleaved Pallas 2^10", 0, 10, 2, 3, seed=101), Case("interleaved Vesta 2^9", 1, 9, 2, 3, indexed=True, seed=102)]
EVAL_SIZES = [1 << 20, (1 << 20) + 1, (1 << 21) + 3]
COMBINED_K = 21
FINAL_KEY_KS = (18, 20)


def _identity_model():
    return model_session(IDENTITY_K, 1, 0, table_window_bits((1 << IDENTITY_K) + 1), False, identity_rounds=(1,))


def _reuse_cases():
    return [Case(f"reuse {i}: 2^{k}", cv, k, 2, 2, seed=200 + i) for i, (cv, k) in enumerate(REUSE_OPENINGS)]


def _features(case, sm):
    f = set()
    n_mat = 0
    for s in sm.folds:
        if s.outcome == "bail":
            f.add("nlists bail")
            continue
        f.add(f"MINB {s.minb}")
        f.add(f"WS {s.WS}")
        if s.G == 1:
            f.add("G = 1")
        if s.cs == 1:
            f.add("cs = 1")
        if s.widths[-1] < s.cs:
            f.add("last group narrower than cs")
        if s.outcome == "identity":
            f.add("identity fallback")
        else:
            n_mat += 1
            if case is not None and case.fk_small_c and s.new_c == case.fk_small_c != table_window_bits(s.m + case.indexed):
                f.add("fk table from fk_small_c")
    if n_mat >= 2:
        f.add("second materialisation")
    if n_mat >= 3:
        f.add("third materialisation (slot reuse)")
    if not sm.folds:
        f.add("no materialisation")
    f.add("finish half tables" if sm.finish_tabs else "finish per-bit loop")
    f |= {"inner products, 1 pass" if p == 1 else "inner products, > 1 pass" for p in sm.ip_passes}
    return f


REQUIRED = {
    "MINB 3", "MINB 4", "WS 1", "WS 2", "WS 3", "WS 4", "G = 1", "cs = 1", "last group narrower than cs", "nlists bail",
    "identity fallback", "second materialisation", "third materialisation (slot reuse)", "fk table from fk_small_c",
    "no materialisation", "finish half tables", "finish per-bit loop", "inner products, 1 pass", "inner products, > 1 pass",
    "evaluation chunk 16", "evaluation chunk 64",
}


def test_case_table_reaches_every_branch():
    seen = set()
    for case in PROD_CASES + SWEEP_CASES + [FK_C_CASE, NO_TABS_CASE] + _reuse_cases() + INTERLEAVED:
        seen |= _features(case, case.model())
    seen |= _features(None, _identity_model())
    for n in EVAL_SIZES + [1 << COMBINED_K]:
        seen.add(f"evaluation chunk {poly_chunk(n)}")
    assert poly_chunk(1 << 20) == 16 and poly_chunk((1 << 20) + 1) == 64
    missing = REQUIRED - seen
    assert not missing, sorted(missing)
    # the knob cases leave their branch: per-bit finish where the default builds tables, fk_small_c where the rule differs
    assert NO_TABS_CASE.model().finish_tabs == 0 and NO_TABS_CASE.model(no_ipa_tabs=False).finish_tabs == 1
    assert [s.new_c for s in FK_C_CASE.model().folds] == [12, 12, 12, 12]
    assert [s.new_c for s in FK_C_CASE.model(fk_small_c=0).folds] == [10, 10, 10, 10]
    # inner products: one pass up to 2^15 products per half, two from 2^16 + 1 (k >= 17 makes more than one)
    assert inner_product_passes(1 << 15) == (128, 1) and inner_product_passes((1 << 15) + 1) == (128, 2)
    assert inner_product_passes(1 << 19) == (128, 16)
    # every fold call launches 1 (no attempt or bail), 4 (identity) or 5 (materialised)
    for case in PROD_CASES + SWEEP_CASES:
        assert {n for kind, n in case.model().calls if kind == "fold"} <= {1, 5}, case.name


def _shape_row(s):
    return (s.round, s.J, s.m, s.c, s.G, s.cs, s.widths, s.WS, s.minb)


def test_model_reproduces_the_materialisation_shapes():
    """The shapes of the production degrees and of the sweep, derived by hand from ipa_api.inc"""
    def rows(k, rounds, min_log, table, indexed=False, fk_small_c=0):
        c = table_window_bits((1 << k) + 1, table)
        return model_session(k, rounds, min_log, c, indexed, fk_small_c).folds

    r = rows(18, 5, 11, 0, True)
    assert [_shape_row(s) for s in r] == [(5, 5, 8192, 17, 3, 6, [6, 6, 5], 2, 3), (10, 5, 256, 15, 3, 5, [5, 5, 5], 4, 3)]
    assert [s.new_c for s in r] == [15, 10]
    r = rows(20, 5, 11, 0, True)
    assert [_shape_row(s) for s in r] == [(5, 5, 32768, 20, 4, 5, [5] * 4, 1, 4), (10, 5, 1024, 17, 3, 6, [6, 6, 5], 4, 3)]
    r = rows(17, 5, 11, 0)
    assert [_shape_row(s) for s in r] == [(5, 5, 4096, 17, 3, 6, [6, 6, 5], 4, 3), (10, 5, 128, 10, 2, 5, [5, 5], 4, 3)]
    r = rows(14, 1, 14, 0)
    assert [_shape_row(s) for s in r] == [(1, 1, 8192, 15, 15, 1, [1] * 15, 1, 4)]
    r = rows(16, 7, 11, 0)
    assert [_shape_row(s) for s in r] == [(7, 7, 512, 17, 2, 9, [9, 8], 4, 3)]
    r = rows(13, 3, 2, 0, fk_small_c=12)
    assert [(s.round, s.c, s.G, s.cs) for s in r] == [(3, 15, 5, 3), (6, 12, 4, 3), (9, 12, 4, 3), (12, 12, 4, 3)]
    assert all(s.outcome == "materialised" for s in r)
    r = rows(12, 10, 0, 21, True)
    assert [(s.round, s.G, s.cs, s.WS, s.nlists, s.outcome) for s in r] == [(10, 2, 11, 4, 8200, "bail")]
    bail = model_session(12, 10, 0, 21, True)
    assert [n for kind, n in bail.calls if kind == "fold"] == [1] * 12
    r = rows(15, 2, 13, 4)
    assert [(s.m, s.c, s.G, s.cs, s.WS) for s in r] == [(8192, 4, 2, 2, 3), (2048, 15, 8, 2, 3)]
    ident = _identity_model()
    assert [n for kind, n in ident.calls if kind == "fold"] == [4] + [1] * (IDENTITY_K - 1)


def fold_subdigits(s, c, G, cs, nwin):
    """signed sub-digits of k_fold_digits (ipa.cuh:194-205): [(w, g, digit)] and the carry left after the top window"""
    out, carry = [], 0
    for w in range(nwin):
        for g in range(G):
            width = min(cs, c - g * cs)
            half = 1 << (width - 1)
            raw = ((s >> (w * c + g * cs)) & ((1 << width) - 1)) + carry
            if raw > half:
                out.append((w, g, raw - (1 << width)))
                carry = 1
            else:
                out.append((w, g, raw))
                carry = 0
    return out, carry


def test_fold_subdigits_recompose_the_challenge_products():
    """sum_w sum_g digit 2^(c w + cs g) == C(u) with |digit| <= 2^(width - 1), and no carry after the top window, for every
    window width c = 4..21 of a table and every J = 1..10 of the fold policy"""
    for curve in (0, 1):
        q = pyref.scalar_modulus(curve)
        rng = pyref.SplitMix64(0xF01D + curve)
        xs = [rng.field(q) >> 126 | 1 for _ in range(5)]       # 128-bit challenges like the sponge's
        prods = [1]
        for u in range(1, 1 << len(xs)):                        # C(u) = prod of the challenges whose bit is set in u
            p = 1
            for r, x in enumerate(xs):
                if (u >> (len(xs) - 1 - r)) & 1:
                    p = p * x % q
            prods.append(p)
        # products near r: (-1) xi_1, (-1) xi_1 xi_2, and the largest elements
        near = [q - 1, q - 2, q - (1 << 64), q - xs[0], q - xs[0] * xs[1] % q, q >> 1, (1 << 253) + 1, (1 << 254) - 1]
        vals = prods + near
        assert all(0 < v < q for v in vals)
        for c in range(4, 22):
            nwin = -(-256 // c)
            for J in range(1, 11):
                f = fold_shape(J, J, 1 << 12, c)
                for v in vals:
                    digits, carry = fold_subdigits(v, c, f.G, f.cs, nwin)
                    assert carry == 0, (c, J, v)
                    assert all(abs(d) <= 1 << (f.widths[g] - 1) for _, g, d in digits), (c, J)
                    assert sum(d << (c * w + f.cs * g) for w, g, d in digits) == v, (c, J, v)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
_ORACLE = {}


def key_seed(case):
    return 0x1BA0 + 97 * case.curve + 7 * case.k + case.seed


def register_key(c, case):
    """2^k generators and the hiding generator h = key[2^k] (synthetic, deterministic in the seed)"""
    B = c.register_synthetic_bases(case.curve, key_seed(case), (1 << case.k) + 1)
    if case.table is not None:
        B.precompute(case.table)
    return B


def inputs(c, case, B):
    """(key points, coefficients, z, xi_0, h' = xi_0 h) of a case"""
    sf = cref.scalar_field(case.curve)
    n = 1 << case.k
    pts = c.download_bases(B)
    s = key_seed(case)
    coeffs = cref.gen_scalars(sf, s + 1, n, True)
    z = cref.gen_scalars(sf, s + 2, 1, True).reshape(4)
    xi0 = cref.gen_scalars(sf, s + 3, 1, True).reshape(4)
    hp, hp_inf = cref.point_mul(case.curve, pts[n], 0, cref.from_mont(sf, xi0.reshape(1, 4)).reshape(4))
    assert hp_inf == 0
    return pts, coeffs, z, xi0, hp


def oracle_proof(case, pts, coeffs, z, hp):
    """the oracle's proof, cached per key: it does not depend on how h' is passed, on the fold policy or on the context"""
    key = (case.curve, case.k, key_seed(case))
    if key not in _ORACLE:
        _ORACLE[key] = oracle_open(case.curve, pts[: 1 << case.k], coeffs, z, hp, sponge_stand_in(cref.scalar_field(case.curve)))
    return _ORACLE[key]


class Opening:
    """One session driven call by call; every call's launches are checked against the model in order.
    fold_round: one accmsm_ipa_open_fold_round per round like bench.py (the fold's and the round's launches together)."""

    def __init__(self, c, B, case, coeffs, z, xi0, hp, squeeze, sm, fold_round=False):
        self.c, self.case, self.squeeze, self.fold_round = c, case, squeeze, fold_round
        self.sf = cref.scalar_field(case.curve)
        self.expected = list(sm.calls)
        self.l_vec, self.r_vec, self.chs, self.lr, self.xi = [], [], [], None, None
        if case.indexed:
            self.sess = self._call("begin", lambda: c.ipa_open_begin(B, coeffs, case.k, z, None), lambda s: c.ipa_open_use_hiding_generator(s, 1 << case.k, xi0))
        else:
            self.sess = self._call("begin", lambda: c.ipa_open_begin(B, coeffs, case.k, z, hp))
        self.lr = self._call("round", lambda: c.ipa_open_round(self.sess)) if case.k else None

    def _call(self, kind, f, then=None):
        kinds = [kind] if kind != "fold_round" else ["fold", "round"]
        want = 0
        for kd in kinds:
            if kd == "round" and self.expected and self.expected[0][0] != "round":
                break                                          # the last fold_round runs no round
            ek, n = self.expected.pop(0)
            assert ek == kd, (self.case.name, ek, kd)
            want += n
        before = self.c.kernel_launches()
        out = f()
        if then is not None:
            then(out)
        got = self.c.kernel_launches() - before
        assert got == want, (self.case.name, kind, len(self.chs), got, want)
        return out

    def step(self):
        """fold with the challenge of the last (l, r) and run the next round; True while rounds remain"""
        l, r = self.lr
        self.xi = np.ascontiguousarray(self.squeeze(self.xi, l, r), dtype=np.uint64).reshape(4)
        self.l_vec.append(l); self.r_vec.append(r); self.chs.append(self.xi)
        if self.fold_round:
            self.lr = self._call("fold_round", lambda: self.c.ipa_open_fold_round(self.sess, self.xi))
        else:
            xinv = cref.fe_inv(self.sf, self.xi.reshape(1, 4)).reshape(4)
            self._call("fold", lambda: self.c.ipa_open_fold(self.sess, self.xi, xinv))
            self.lr = self._call("round", lambda: self.c.ipa_open_round(self.sess)) if self.expected[0][0] == "round" else None
        return self.lr is not None

    def finish(self):
        fk, cc = self._call("finish", lambda: self.c.ipa_open_finish(self.sess))
        assert not self.expected, (self.case.name, self.expected)
        return self.l_vec, self.r_vec, fk, cc, self.chs

    def run(self):
        if self.lr is not None:
            while self.step():
                pass
        return self.finish()


def assert_proof(name, got, exp):
    l_vec, r_vec, fk, c, chs = got
    el, er, efk, ec, echs = exp
    assert len(l_vec) == len(el) and len(chs) == len(echs), name
    for j, (a, b) in enumerate(zip(l_vec, el)):
        assert same_point(a, b), (name, "l", j)
    for j, (a, b) in enumerate(zip(r_vec, er)):
        assert same_point(a, b), (name, "r", j)
    for j, (a, b) in enumerate(zip(chs, echs)):
        assert np.array_equal(a, b), (name, "xi", j)
    assert np.array_equal(fk, efk), (name, "final key")
    assert np.array_equal(c, ec), (name, "c")


def open_case(c, case, B=None, fold_round=False, policy=None, **model_kw):
    """one opening of `case` on context c under the policy (rounds, min_log) (default: the case's), checked against the
    model and the oracle; returns the proof"""
    own = B is None
    B = register_key(c, case) if own else B
    rounds, min_log = policy if policy is not None else (case.rounds, case.min_log)
    try:
        pts, coeffs, z, xi0, hp = inputs(c, case, B)
        exp = oracle_proof(case, pts, coeffs, z, hp)
        c.set_ipa_fold(rounds, min_log)
        sm = case.model(rounds=rounds, min_log=min_log, **model_kw)
        got = Opening(c, B, case, coeffs, z, xi0, hp, sponge_stand_in(cref.scalar_field(case.curve)), sm, fold_round).run()
        assert_proof(case.name, got, exp)
        return got
    finally:
        c.set_ipa_fold()
        if own:
            B.release()


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(len(PROD_CASES)), ids=["pallas-18-index", "vesta-17-point", "pallas-20-index"])
def test_production_degrees(ctx, idx):
    """the degrees bench.py opens, with the default policy (two materialisations) and without materialisation, both bit for
    bit with one cached oracle proof; the decider accepts the final key"""
    case = PROD_CASES[idx]
    B = register_key(ctx, case)
    try:
        ck = ab.CommitterKey(B, 1 << case.k)
        for policy in (DEFAULT_POLICY, (0, 0)):
            got = open_case(ctx, case, B, fold_round=case.indexed, policy=policy)
            assert ab.InnerProductArgPC.check_final_key(ck, np.array(got[4]), got[2], 0), (case.name, policy)
        assert len(case.model().folds) == 2
    finally:
        B.release()


@pytest.mark.gpu
def test_production_degree_on_a_device_group():
    """a 2^18 opening on a virtual group of two contexts of one GPU gives the single-context proof (values only: the children
    run cyclic shards, which the single-context model does not describe)"""
    case = PROD_CASES[0]
    g = ab.Context(devices=[0, 0])
    try:
        B = register_key(g, case)
        pts, coeffs, z, xi0, hp = inputs(g, case, B)
        exp = oracle_proof(case, pts, coeffs, z, hp)
        ck = ab.CommitterKey(B, 1 << case.k)
        got = ab.InnerProductArgPC.open(ck, coeffs, z, None, sponge_stand_in(cref.scalar_field(case.curve)), log_d=case.k, xi0=xi0)
        assert_proof("group " + case.name, got, exp)
        assert ab.InnerProductArgPC.check_final_key(ck, np.array(got[4]), got[2], 0)
        B.release()
    finally:
        g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(len(SWEEP_CASES)), ids=[f"sweep{i}" for i in range(len(SWEEP_CASES))])
def test_fold_shape_sweep(ctx, idx):
    """cs = 1 and MINB 4, uneven sub-digit groups, repeated materialisations, the nlists bail, WS 3, G = 1, registered
    tables at c = 4, 10 and 21 and a key without a table"""
    open_case(ctx, SWEEP_CASES[idx])


def _canon_point(curve, xy, inf):
    if inf:
        return None
    x, y = cref.arr_to_ints(cref.from_mont(cref.base_field(curve), np.asarray(xy, dtype=np.uint64).reshape(2, 4)))
    return (x, y)


@pytest.mark.gpu
def test_identity_in_the_folded_key_falls_back(ctx):
    """A key with G[m + p0] = -xi_1^-1 G[p0] folds to the identity at p0 after round 1 (FK[p] = G[p] + xi_1 G[m + p]): the
    first fold call runs the fold kernels and abandons the result (4 launches), every later one launches 1, and the proof
    equals the unfolded run and the pure-Python restatement with the same challenges"""
    curve, k = 0, IDENTITY_K
    sf = cref.scalar_field(curve)
    q = pyref.scalar_modulus(curve)
    n, m = 1 << k, 1 << (k - 1)
    chs = cref.gen_scalars(sf, 0x1D0, k, True)
    xi1 = cref.arr_to_ints(cref.from_mont(sf, chs[:1]))[0]
    pts = cref.gen_points(curve, 0x1D1, n + 1)
    pts[m + IDENTITY_P0], inf = cref.point_mul(curve, pts[IDENTITY_P0], 0, cref.ints_to_arr([(-pow(xi1, -1, q)) % q]).reshape(4))
    assert inf == 0
    case = Case("identity fallback", curve, k, 1, 0)
    B = ctx.register_bases(curve, pts).precompute()
    try:
        coeffs = cref.gen_scalars(sf, 0x1D2, n, True)
        z = cref.gen_scalars(sf, 0x1D3, 1, True).reshape(4)
        hp = pts[n]
        proofs = []
        for policy, sm in (((1, 0), _identity_model()), ((0, 0), case.model(rounds=0))):
            ctx.set_ipa_fold(*policy)
            try:
                it = iter(list(chs))
                proofs.append(Opening(ctx, B, case, coeffs, z, None, hp, lambda prev, l, r: next(it), sm).run())
            finally:
                ctx.set_ipa_fold()
        assert_proof("identity fallback vs unfolded", proofs[0], proofs[1])
        key = [_canon_point(curve, p, 0) for p in pts[:n]]
        el, er, efk, ec = pyref.ipa_open(key, fe_ints(sf, coeffs), fe_ints(sf, z.reshape(1, 4))[0], _canon_point(curve, hp, 0),
                                         fe_ints(sf, chs), curve)
        l_vec, r_vec, fk, c, _ = proofs[0]
        assert [_canon_point(curve, *p) for p in l_vec] == el and [_canon_point(curve, *p) for p in r_vec] == er
        assert _canon_point(curve, fk, 0) == efk and fe_ints(sf, c.reshape(1, 4)) == [ec]
    finally:
        B.release()


def _fresh_context(monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    try:
        return ab.Context(0)
    finally:
        for k in env:
            monkeypatch.delenv(k)


@pytest.mark.gpu
def test_knob_fk_small_c(monkeypatch):
    """ACCMSM_FK_C=12: the materialised keys of <= 2^13 + 1 points get c = 12 tables, the proof stays the oracle's"""
    c2 = _fresh_context(monkeypatch, {"ACCMSM_FK_C": "12"})
    try:
        open_case(c2, FK_C_CASE)
    finally:
        c2.close()


@pytest.mark.gpu
def test_knob_no_ipa_tabs(ctx, monkeypatch):
    """ACCMSM_NO_IPA_TABS=1: the finish of a 2^18 opening and the decider's final key at 2^18 and 2^20 run the per-bit
    coefficient loop; the points equal the oracle's and the default context's"""
    c2 = _fresh_context(monkeypatch, {"ACCMSM_NO_IPA_TABS": "1"})
    try:
        open_case(c2, NO_TABS_CASE, fold_round=True)
        for k in FINAL_KEY_KS:
            sf = cref.scalar_field(0)
            ch = cref.gen_scalars(sf, 0xF1 + k, k, True)
            keys = [cc.register_synthetic_bases(0, 0xF10 + k, (1 << k) + 1).precompute() for cc in (ctx, c2)]
            try:
                c_tab = table_window_bits((1 << k) + 1)
                res = []
                for cc, B, tabs in ((ctx, keys[0], 1), (c2, keys[1], 0)):
                    before = cc.kernel_launches()
                    res.append(cc.ipa_final_key(B, ch))
                    assert cc.kernel_launches() - before == tabs + plan(1 << k, 1, table_c=c_tab).launches, (k, tabs)
                    assert half_tables(k, 1 << k, no_ipa_tabs=not tabs) == tabs
                assert same_point(res[0], res[1]), k
                pts = c2.download_bases(keys[1], 0, 1 << k)
                ok, exy, einf = cref.ipa_check_final_key(0, pts, ch, res[1][0], res[1][1])
                assert ok and einf == 0 and np.array_equal(exy, res[1][0]), k
                acc, _, _ = c2.ipa_check_final_key(keys[1], ch, res[1][0], 0)
                bad = res[1][0].copy(); bad[0] ^= np.uint64(1)
                rej, _, _ = c2.ipa_check_final_key(keys[1], ch, bad, 0)
                assert acc and not rej, k
            finally:
                for B in keys:
                    B.release()
    finally:
        c2.close()


@pytest.mark.gpu
def test_session_reuse_and_interleaving(monkeypatch):
    """On one context: 2^14 with set_ipa_fold(2, 2) materialises at rounds 2, 4, .., 12 (the two fk slots alternate), then
    2^6 and 2^14 again recycle the finished sessions with their stale slots; then the rounds of two sessions on different
    curves and keys interleave.  Every proof is the oracle's."""
    c2 = _fresh_context(monkeypatch, {})
    try:
        cases = _reuse_cases()
        assert len(cases[0].model().folds) == 6
        for case in cases:
            open_case(c2, case)
        keys = [register_key(c2, case) for case in INTERLEAVED]
        try:
            opens, exps = [], []
            c2.set_ipa_fold(INTERLEAVED[0].rounds, INTERLEAVED[0].min_log)      # one policy per context
            for case, B in zip(INTERLEAVED, keys):
                pts, coeffs, z, xi0, hp = inputs(c2, case, B)
                exps.append(oracle_proof(case, pts, coeffs, z, hp))
                opens.append(Opening(c2, B, case, coeffs, z, xi0, hp, sponge_stand_in(cref.scalar_field(case.curve)),
                                     case.model()))
            live = list(opens)
            while live:
                live = [o for o in live if o.step()]
            for case, o, exp in zip(INTERLEAVED, opens, exps):
                assert_proof(case.name, o.finish(), exp)
        finally:
            c2.set_ipa_fold()
            for B in keys:
                B.release()
    finally:
        c2.close()


@pytest.mark.gpu
def test_evaluation_above_2_20(ctx):
    """poly_evaluate on both sides of the switch to 64 coefficients per thread, and begin_combined at 2^21 (m = 2 and a
    random polynomial over a synthetic key of 2^21 points); finishing that session with its rounds left raises and
    releases it"""
    for i, n in enumerate(EVAL_SIZES):
        f = i % 2
        cf = cref.gen_scalars(f, 0xE0 + i, n, True)
        z = cref.gen_scalars(f, 0xE8 + i, 1, True).reshape(4)
        assert np.array_equal(ctx.poly_evaluate(f, cf, z), cref.poly_evaluate(f, cf, z)), n
    k, curve = COMBINED_K, 0
    sf = cref.scalar_field(curve)
    key = ctx.register_synthetic_bases(curve, 0xC21, 1 << k)
    try:
        chm = cref.gen_scalars(sf, 0xC22, 2 * k, True).reshape(2, k, 4)
        al = cref.gen_scalars(sf, 0xC23, 2, True)
        rp = cref.gen_scalars(sf, 0xC24, (1 << k) - 5, True)
        z = cref.gen_scalars(sf, 0xC25, 1, True).reshape(4)
        before = ctx.kernel_launches()
        sess, ev = ctx.ipa_open_begin_combined(key, chm, al, z, None, rp)
        assert ctx.kernel_launches() - before == 1 + 2 + 2          # k_powers, the two coefficient kernels, the evaluation
        assert np.array_equal(ev, cref.poly_evaluate(sf, cref.combine_check_polys(sf, chm, al, rp), z))
        with pytest.raises(ab.AccmsmError, match="rounds remain"):
            ctx.ipa_open_finish(sess)
        with pytest.raises(ab.AccmsmError):
            ctx.ipa_open_round(sess)
    finally:
        key.release()
