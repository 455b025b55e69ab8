"""Every branch of the MSM dispatch, each case known to run the branch it is named for.

msm_accumulate / msm_reduce (accumulation_b200/csrc/accmsm.cu) pick one of about a dozen device paths from the shape of a
pass: counting or radix sort, staged or direct writes in both radix passes, the skew gate that hands skewed inputs back to
the counting sort, warp-coop or balanced accumulation (and `into` accumulation across upload segments), three reduction
tiers with a coop, plain or split first level, coop or plain Horner in the finish.

The plan model below restates those host-side decisions in Python, citing the C++ line of each rule.  It predicts the
kernel launches of a call (the change of kernel_launches() across it), and every GPU case asserts that count, so a case
cannot drift off its branch unnoticed: a change that moves a threshold fails here, and the model is updated with it.
From canonical scalars the model also computes the device's signed digits (sort.cuh:142-147) and the pairs of every sort
partition, which tells the regime of the bucket pass (staged, direct, or gate closed).

test_case_table_reaches_every_branch runs without a GPU and checks that the case table reaches both sides of every
boundary and every bucket-pass regime.  The GPU tests compare every result bit for bit with the C oracle."""
import math
from dataclasses import dataclass
from typing import Optional

import numpy as np
import pytest

import accumulation_b200 as ab
from oracle import cref, pyref
from tests.util import same_point, scalar_distributions

# ---- constants of the pipeline (msm.cuh, sort.cuh, accmsm.cu) ------------------------------------------------------------
MAX_JOBS = 8                    # msm.cuh:38
SCAN_TILE = 4096                # msm.cuh:255
SCAN_ONE_CTA_TILES = 8          # msm.cuh:256
SORT_TILE = 1024                # sort.cuh:41
SORT_MAX_PARTS = 8192           # sort.cuh:44
SORT_MAX_LB = 12                # sort.cuh:45
SORT_STAGE_MAX = 24576          # sort.cuh:46
SORT_SMEM_OPT_IN = 220 * 1024   # accmsm.cu:399
SMEM_DEFAULT = 48 * 1024        # per-function dynamic shared memory without an opt-in
ACC_WARP_MAX_KEYS = 8192        # accmsm.cu:333
ACC_WARP_MAX_ENTRIES = 1 << 17  # accmsm.cu:334
RADIX_MIN_ENTRIES = 1 << 17     # accmsm.cu:431
RADIX_MIN_KEYS = 1024           # accmsm.cu:431
CHUNK_ELEMS = (4 << 20) // 32   # accmsm.cu:819, 826: 4 MiB upload chunks of 32-byte scalars


def _log2_floor(n):
    return n.bit_length() - 1


def pick_window_bits(n, window_bits=0):
    """window bits of a plain key (accmsm.cu:267-273)"""
    if 2 <= window_bits <= 16:
        return window_bits
    return min(16, max(4, _log2_floor(n) - 3))


def table_window_bits(key_n, window_bits=0):
    """window bits of precompute(window_bits) on a key of key_n points (accmsm.cu:291-293)"""
    if window_bits:
        return window_bits
    lg = _log2_floor(key_n)
    return 20 if lg >= 20 else 17 if lg >= 15 else 15 if lg >= 13 else 10


def scan_launches(nkeys):
    """launch_scan: one CTA up to 8 tiles of 4096 keys, three launches above (accmsm.cu:384-395)"""
    return 1 if (nkeys + SCAN_TILE - 1) // SCAN_TILE <= SCAN_ONE_CTA_TILES else 3


@dataclass
class Plan:
    n: int
    njobs: int
    c: int
    nwin: int
    nb: int
    sets_per_job: int
    hist_stride: int
    nkeys: int
    n_entries: int
    into: bool
    radix: bool
    lb: int = 0
    nparts: int = 0
    stage_pairs: int = 0
    bucket_cap: int = 0
    gate_thr: int = 0
    smem0: int = 0
    warp_coop: bool = False
    tier: int = 0
    first_level: str = ""
    sums_x_sets: int = 0
    finish: str = ""
    acc_launches: int = 0
    red_launches: int = 0

    @property
    def launches(self):
        return self.acc_launches + self.red_launches


def plan(n, njobs=1, table_c=None, window_bits=0, n_for_c=None, sort_lb=0, into=False, no_coop_finish=False):
    """One pass of msm_accumulate + msm_reduce.  table_c: window bits of the key's table (None: no table)."""
    # make_shape (accmsm.cu:349-373); the table is used unless a different window override is set (use_table, :327-331)
    if table_c is not None and window_bits in (0, table_c):
        c, sets = table_c, 1
    else:
        c, sets = pick_window_bits(n if n_for_c is None else n_for_c, window_bits), None
    nwin = -(-256 // c)
    nb = 1 << (c - 1)
    sets = nwin if sets is None else 1
    p = Plan(n=n, njobs=njobs, c=c, nwin=nwin, nb=nb, sets_per_job=sets, hist_stride=nb if sets > 1 else 0,
             nkeys=njobs * sets * nb, n_entries=n * nwin * njobs, into=into, radix=False)
    acc = 0
    # radix condition (accmsm.cu:431)
    p.radix = sort_lb >= 0 and p.n_entries >= RADIX_MIN_ENTRIES and p.nkeys >= RADIX_MIN_KEYS
    if p.radix:
        # lb escalation and nparts (:436-440)
        lb = sort_lb if sort_lb > 0 else 9
        lb = min(SORT_MAX_LB, max(9, lb))
        while -(-p.nkeys // (1 << lb)) > SORT_MAX_PARTS and lb < SORT_MAX_LB:
            lb += 1
        p.lb, p.nparts = lb, -(-p.nkeys // (1 << lb))
        assert p.nparts <= SORT_MAX_PARTS
        # write-pass staging, bucket-pass staging (:444-445) and the skew gate (:453)
        p.stage_pairs = SORT_TILE * nwin if SORT_TILE * nwin <= SORT_STAGE_MAX else 0
        p.bucket_cap = min(49152, max(4096, p.n_entries // p.nparts * 5 // 4 + 1024))
        p.gate_thr = min(0x7FFFFFFF, max(65536, 4 * p.n_entries // p.nparts))
        # dynamic shared memory of the count pass, the write pass and the bucket pass (:455-458)
        p.smem0 = 2 * p.nparts * 4
        assert p.smem0 + p.stage_pairs * 8 <= SORT_SMEM_OPT_IN and ((1 << lb) + p.bucket_cap) * 4 <= SORT_SMEM_OPT_IN
        acc += 2 + scan_launches(p.nparts) + 2         # count + tile scan, partition scan, write + bucket pass (:462-473)
    acc += 2 + scan_launches(p.nkeys)                  # counting sort: digits + scatter, scan over the keys (:479-490)
    # warp-coop accumulation of short passes (:495), else balanced accumulation + fix-up (:540-557; no batch-affine rounds)
    p.warp_coop = not into and p.nkeys <= ACC_WARP_MAX_KEYS and p.n_entries <= ACC_WARP_MAX_ENTRIES
    acc += 1 if p.warp_coop else 2
    p.acc_launches = acc
    # reduction tier (accmsm.cu:585-630)
    nsets = njobs * sets
    if nb > 1024:
        m = c - 1
        C0 = 1 << (m // 2)
        R0 = nb // C0
        p.sums_x_sets = (R0 + C0) * nsets
        split = p.sums_x_sets > 320 and R0 > C0                                 # :591
        p.first_level = "split" if split else "coop" if p.sums_x_sets <= 320 else "plain"   # :607-610
        p.tier, red = 2, 2
    elif nb > 32:
        p.tier, red = 1, 1
    else:
        p.tier, red = 0, 1
    red += 2 + 1                                       # leaf scan + combine, finish (:635-645)
    p.finish = "coop" if sets > 1 and not no_coop_finish else "plain"          # :641-644
    p.red_launches = red
    return p


def passes(n, rows, **kw):
    """msm_batch / msm_rows_host: groups of MAX_JOBS rows share one pass (accmsm.cu:935-950)"""
    return [plan(n, min(MAX_JOBS, rows - j0), **kw) for j0 in range(0, rows, MAX_JOBS)]


def host_segments(n, segments=0, seg_pcts=(), seg0_pct=25):
    """point segments [e0, e1) of a host-scalar MSM (msm_host_scalars, accmsm.cu:819-898); None: one plain pass"""
    if n * 32 < 4 * (4 << 20) or segments == 1:
        return None
    nchunks = -(-n // CHUNK_ELEMS)
    nseg = segments if segments > 1 else 2
    if seg_pcts:
        ends = [max(1, (nchunks * pc + 50) // 100) for pc in seg_pcts] + [nchunks]
    elif nseg == 2:
        ends = [max(1, (nchunks * seg0_pct + 50) // 100), nchunks]
    else:
        ends = [max(g, nchunks * g // nseg) for g in range(1, nseg + 1)]
    ends[-1] = nchunks
    out, c0 = [], 0
    for e in ends:
        c1 = min(e, nchunks)
        if c1 <= c0:
            continue
        out.append((c0 * CHUNK_ELEMS, min(n, c1 * CHUNK_ELEMS)))
        c0 = c1
    return out


def segmented_plans(n, table_c=None, **seg):
    """the `into` pass of every segment (window bits picked from the whole length) and the launches of the whole MSM"""
    segs = host_segments(n, **seg)
    plans = [plan(e1 - e0, 1, table_c=table_c, n_for_c=n, into=True) for e0, e1 in segs]
    return segs, plans, sum(p.acc_launches for p in plans) + plans[-1].red_launches


def signed_digits(canon, c, nwin):
    """(N, nwin) signed radix-2^c digits of canonical scalars, as the device forms them (sort.cuh:142-147, msm.cuh:227-237)"""
    s = np.ascontiguousarray(canon, dtype=np.uint64).reshape(-1, 4)
    limbs = [s[:, i] for i in range(4)]
    mask = np.uint64((1 << c) - 1)
    half = 1 << (c - 1)
    carry = np.zeros(s.shape[0], dtype=np.int64)
    out = np.empty((s.shape[0], nwin), dtype=np.int64)
    for w in range(nwin):
        li, off = divmod(w * c, 64)
        v = limbs[li] >> np.uint64(off) if li < 4 else np.zeros(s.shape[0], np.uint64)
        if off + c > 64 and li + 1 < 4:
            v = v | (limbs[li + 1] << np.uint64(64 - off))
        raw = (v & mask).astype(np.int64) + carry
        neg = raw > half
        out[:, w] = np.where(neg, raw - (1 << c), raw)
        carry = neg.astype(np.int64)
    return out


def partition_sizes(p, canon_rows):
    """pairs per sort partition of a radix pass: key = job key base + window * hist_stride + |digit| - 1 (sort.cuh:147-148)"""
    assert p.radix and len(canon_rows) == p.njobs
    sizes = np.zeros(p.nparts, dtype=np.int64)
    for j, canon in enumerate(canon_rows):
        mag = np.abs(signed_digits(canon, p.c, p.nwin))
        keys = j * p.sets_per_job * p.nb + np.arange(p.nwin, dtype=np.int64)[None, :] * p.hist_stride + mag - 1
        sizes += np.bincount((keys[mag != 0] >> p.lb), minlength=p.nparts)
    return sizes


def bucket_regime(p, sizes):
    """gate closed when any partition exceeds the threshold (the whole pass goes to the counting sort, sort.cuh:111, 202);
    else the largest partition is permuted in shared memory (staged) or scattered to HBM (direct, sort.cuh:207)"""
    big = int(sizes.max())
    return "gate closed" if big > p.gate_thr else "direct" if big > p.bucket_cap else "staged"


# ---- the case table -----------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    name: str
    curve: int
    n: int                          # scalars per row
    rows: int = 1                   # scalar vectors of the call: msm() for 1, msm_batch() above
    table_c: Optional[int] = None   # precompute(table_c) on the key; None: plain key
    window_bits: int = 0            # set_window_bits() for the call
    key_n: int = 1 << 14
    offset: int = 0
    mont: bool = True
    shape: tuple = ()               # how the scalars are shaped: (), ("dist", name), ("dists",), ("low", rows, share, windows, digit)
    seed: int = 0

    def passes(self, **kw):
        return passes(self.n, self.rows, table_c=self.table_c, window_bits=self.window_bits, **kw)

    def launches(self, **kw):
        return sum(p.launches for p in self.passes(**kw))


def set_low_windows(canon, c, share, windows, digit):
    """windows [0, windows) of the first share * N scalars become the digit `digit` (<= 2^(c-1), so no carry moves)"""
    k = int(round(share * canon.shape[0]))
    vals = cref.arr_to_ints(canon[:k]) if k else []
    mask = sum(((1 << c) - 1) << (c * w) for w in range(windows))
    put = sum(digit << (c * w) for w in range(windows))
    out = canon.copy()
    if k:
        out[:k] = cref.ints_to_arr([(v & ~mask) | put for v in vals])
    return out


def make_scalars(case):
    """-> (scalars of the call (rows, n, 4) in the case's form, canonical images (rows, n, 4))"""
    sf = cref.scalar_field(case.curve)
    seed = 0xD15 + 1000 * case.seed + 7 * case.n + case.rows
    kind = case.shape[0] if case.shape else None
    if kind in ("dist", "dists"):          # the distributions come in Montgomery form
        assert case.mont, case.name
        d = scalar_distributions(case.curve, case.n, seed)
        sc = np.stack([d[case.shape[1]]] if kind == "dist" else [d[k] for k in sorted(d)][: case.rows])
        return sc, cref.from_mont(sf, sc.reshape(-1, 4)).reshape(sc.shape)
    canon = cref.gen_scalars(sf, seed, case.n * case.rows, False).reshape(case.rows, case.n, 4)
    if kind == "low":
        _, which, share, windows, digit = case.shape
        c = case.passes()[0].c
        q = pyref.scalar_modulus(case.curve)
        for j in (range(case.rows) if which is None else which):
            canon[j] = set_low_windows(canon[j], c, share, windows, digit)
            assert max(cref.arr_to_ints(canon[j])) < q
    sc = cref.to_mont(sf, canon.reshape(-1, 4)).reshape(canon.shape) if case.mont else canon
    return np.ascontiguousarray(sc), canon


def _alternate(cases):
    """alternate the two curves and the two oracles (commit of Montgomery scalars, msm_ark of canonical ones)"""
    out = []
    for i, c in enumerate(cases):
        d = dict(c.__dict__)
        d["curve"] = i % 2
        if not c.shape:
            d["mont"] = (i // 2) % 2 == 0
        out.append(Case(**d))
    return out


# 7 or 8 jobs over 2^19 buckets each need more than 6144 partitions: the count pass of the radix sort asks for more than the
# 48 KB of shared memory a kernel gets without an opt-in.  6 jobs (c = 20) and 3 jobs (c = 21) are the last that fit.
BUG_CASES = _alternate(
    [Case(f"table c=20, {j} jobs", 0, 1 << 14, j, table_c=20) for j in (1, 6, 7, 8)]
    + [Case(f"table c=21, {j} jobs", 0, 1 << 14, j, table_c=21) for j in (3, 4, 5, 7, 8)]
    + [Case(f"plain c=16, {j} jobs", 0, 3000, j, window_bits=16, offset=999) for j in (6, 7, 8)]
    + [Case(f"table c=20, {k} rows: passes of 8 and a remainder", 0, 1 << 14, k, table_c=20) for k in (9, 17)])

SORT_CASES = _alternate([
    Case("2^17 - 16 pairs: counting sort", 0, 8191, table_c=16, offset=1),
    Case("2^17 pairs: radix sort", 0, 8192, table_c=16),
    Case("512 keys: counting sort of a long pass", 0, 1 << 14, table_c=10),
    Case("1024 keys: radix sort, direct write pass (26 windows)", 0, 1 << 14, 2, table_c=10),
    Case("1024 keys: radix sort, direct write pass (29 windows)", 0, 5000, 4, table_c=9, offset=77),
    Case("1024 keys: radix sort, staged write pass (24 windows)", 0, 1 << 14, table_c=11),
    Case("2^17 pairs over 8192 keys: radix sort feeds warp-coop accumulation", 0, 2048, 2, window_bits=8, offset=5),
    Case("2^17 + 64 pairs over 8192 keys: balanced accumulation", 0, 2049, 2, window_bits=8, offset=5),
])

REGIME_CASES = _alternate([
    Case("uniform: staged bucket pass", 0, 1 << 14, table_c=16),
    Case("a quarter of the low windows on one digit: direct bucket pass", 0, 1 << 14, table_c=16, shape=("low", None, 0.25, 1, 1000)),
    Case("five low windows on one digit: gate closed", 0, 1 << 14, table_c=16, shape=("low", None, 1.0, 5, 777)),
    Case("one skewed job among uniform ones closes the gate of the pass", 0, 1 << 14, 4, table_c=20, shape=("low", (2,), 1.0, 6, 4242)),
])

DIST_NAMES = ["a_a_a_0", "constant", "one", "one_hot", "q_minus_1", "trunc128", "uniform", "zero"]
DIST_CASES = _alternate(
    [Case(f"distribution {name}, 1 job over c = 20", 0, 1 << 14, table_c=20, shape=("dist", name)) for name in DIST_NAMES]
    + [Case(f"all distributions, 8 jobs over c = 20 (curve {cv})", cv, 1 << 14, 8, table_c=20, shape=("dists",)) for cv in (0, 1)])

ACC_CASES = _alternate([
    Case("8192 buckets: warp-coop accumulation", 0, 6000, table_c=14, offset=100),
    Case("16384 buckets: balanced accumulation", 0, 6000, 2, table_c=14, offset=100),
])

SWEEP_CASES = _alternate(
    [Case(f"sweep table c={c}, {j} jobs", 0, 700 + 13 * c, j, table_c=c, offset=17 * c, seed=c) for c in range(4, 22) for j in (1, 2, 3, 8)]
    + [Case(f"sweep plain c={c}, {j} jobs", 0, 700 + 13 * c, j, window_bits=c, offset=17 * c, seed=c) for c in range(4, 17) for j in (1, 2, 3, 8)])

TABLE_CASES = BUG_CASES + SORT_CASES + REGIME_CASES + DIST_CASES + ACC_CASES + SWEEP_CASES

# development knobs, each on a fresh context: (environment, model arguments, whether only plain keys are meaningful)
KNOBS = [
    ({"ACCMSM_SORT_LB": "-1"}, {"sort_lb": -1}, False),
    ({"ACCMSM_SORT_LB": "12"}, {"sort_lb": 12}, False),
    ({"ACCMSM_NO_AUX": "1"}, {}, False),
    ({"ACCMSM_NO_COOP_FINISH": "1"}, {"no_coop_finish": True}, True),
]
KNOB_CASE_NAMES = [
    "table c=20, 8 jobs", "table c=21, 5 jobs", "plain c=16, 7 jobs",
    "2^17 pairs over 8192 keys: radix sort feeds warp-coop accumulation", "1024 keys: radix sort, staged write pass (24 windows)",
    "a quarter of the low windows on one digit: direct bucket pass", "one skewed job among uniform ones closes the gate of the pass",
    "sweep plain c=13, 3 jobs", "sweep plain c=6, 8 jobs",
]
KNOB_CASES = [c for c in TABLE_CASES if c.name in KNOB_CASE_NAMES]

# host-scalar MSMs of 2^19 + 4097 points cut into `into` segments: (environment, model arguments, key window bits, chunk of
# constant scalars or None)
SEG_N = (1 << 19) + 4097
SEG_CASES = [
    ({"ACCMSM_SEG_PCTS": "20,40,60,80"}, {"seg_pcts": (20, 40, 60, 80)}, 0, 2),
    ({"ACCMSM_SEGMENTS": "3"}, {"segments": 3}, 0, None),
    ({"ACCMSM_SEGMENTS": "4"}, {"segments": 4}, None, 1),
]

FULL_N, FULL_ROWS = 1 << 20, 8
HPPC_N_IN, HPPC_LEN = 5, 2000
GROUP_KEY, GROUP_ROWS = 1 << 14, 8


def seg_scalars(curve, const_chunk):
    sc = cref.gen_scalars(cref.scalar_field(curve), 0x5E6 + curve, SEG_N, True)
    if const_chunk is not None:
        sc[const_chunk * CHUNK_ELEMS:(const_chunk + 1) * CHUNK_ELEMS] = sc[const_chunk * CHUNK_ELEMS]
    return sc


def _features(p):
    f = set()
    if p.radix:
        f.add("radix sort")
        f.add("lb 9" if p.lb == 9 else "lb > 9")
        f.add("count pass over 48 KB" if p.smem0 > SMEM_DEFAULT else "count pass within 48 KB")
        f.add("staged write pass" if p.stage_pairs else "direct write pass")
        if p.n_entries == RADIX_MIN_ENTRIES:
            f.add("radix sort at exactly 2^17 pairs")
        if p.warp_coop:
            f.add("radix sort feeds warp-coop")
    elif p.n_entries < RADIX_MIN_ENTRIES:
        f.add("counting sort: fewer than 2^17 pairs")
        if RADIX_MIN_ENTRIES - p.n_entries <= p.nwin * p.njobs and p.nkeys >= RADIX_MIN_KEYS:     # one scalar short
            f.add("counting sort: just below 2^17 pairs")
    elif p.nkeys < RADIX_MIN_KEYS:
        f.add("counting sort: long pass under 1024 keys")
    else:
        f.add("counting sort: radix switched off")
    f.add(f"key scan of {scan_launches(p.nkeys)} launches")
    if p.into:
        f.add("into accumulation after radix sort" if p.radix else "into accumulation after counting sort")
    elif p.warp_coop:
        f.add("warp-coop accumulation")
    else:
        f.add("balanced accumulation, > 8192 keys" if p.nkeys > ACC_WARP_MAX_KEYS else "balanced accumulation, > 2^17 pairs on <= 8192 keys")
    f.add(f"reduction tier {p.tier}")
    if p.tier == 2:
        f.add(f"first level {p.first_level}")
        f.add("(R0 + C0) nsets <= 320" if p.sums_x_sets <= 320 else "(R0 + C0) nsets > 320")
    f.add(f"{p.finish} finish")
    return f


REQUIRED = {
    "radix sort", "counting sort: fewer than 2^17 pairs", "counting sort: just below 2^17 pairs", "radix sort at exactly 2^17 pairs",
    "counting sort: long pass under 1024 keys", "counting sort: radix switched off",
    "lb 9", "lb > 9", "count pass within 48 KB", "count pass over 48 KB", "staged write pass", "direct write pass",
    "key scan of 1 launches", "key scan of 3 launches",
    "warp-coop accumulation", "radix sort feeds warp-coop", "balanced accumulation, > 8192 keys",
    "balanced accumulation, > 2^17 pairs on <= 8192 keys", "into accumulation after radix sort", "into accumulation after counting sort",
    "reduction tier 0", "reduction tier 1", "reduction tier 2", "first level coop", "first level plain", "first level split",
    "(R0 + C0) nsets <= 320", "(R0 + C0) nsets > 320", "coop finish", "plain finish",
    "bucket pass staged", "bucket pass direct", "bucket pass gate closed", "segment closes the gate alone", "segment of one chunk",
    "several passes in one call",
}


def test_case_table_reaches_every_branch():
    """The model on the case table: both sides of every boundary and every bucket-pass regime are reached, and the
    shapes that needed the count pass's shared-memory opt-in are the ones the analysis of the launch limit names."""
    seen = set()
    for case in TABLE_CASES:
        ps = case.passes()
        if len(ps) > 1:
            seen.add("several passes in one call")
        for p in ps:
            seen |= _features(p)
    for case in KNOB_CASES:
        for _, kw, _ in KNOBS:
            for p in case.passes(**kw):
                seen |= _features(p)
    for p in (plan(FULL_N, FULL_ROWS, table_c=table_window_bits(FULL_N)), plan(HPPC_LEN, 2 * HPPC_N_IN - 2, table_c=20),
              plan(GROUP_KEY // 2, GROUP_ROWS, table_c=20)):
        assert p.radix and p.nparts > 6144
        seen |= _features(p)

    # bucket-pass regimes from the digits of the scalars
    regimes = {}
    for case in REGIME_CASES + DIST_CASES + BUG_CASES[:4] + SORT_CASES:
        ps = case.passes()
        if len(ps) != 1 or not ps[0].radix:
            continue
        _, canon = make_scalars(case)
        regimes[case.name] = bucket_regime(ps[0], partition_sizes(ps[0], canon))
        seen.add("bucket pass " + regimes[case.name])
    assert regimes["uniform: staged bucket pass"] == "staged"
    assert regimes["a quarter of the low windows on one digit: direct bucket pass"] == "direct"
    assert regimes["five low windows on one digit: gate closed"] == "gate closed"
    assert regimes["one skewed job among uniform ones closes the gate of the pass"] == "gate closed"
    assert regimes["all distributions, 8 jobs over c = 20 (curve 0)"] == "direct"       # constant rows: one partition per window
    skewed = [c for c in REGIME_CASES if c.name.startswith("one skewed")][0]
    uniform = Case("the same pass without the skewed job", skewed.curve, skewed.n, skewed.rows, table_c=skewed.table_c)
    _, canon = make_scalars(uniform)
    assert bucket_regime(uniform.passes()[0], partition_sizes(uniform.passes()[0], canon)) == "staged"

    # segmented host-scalar MSMs
    for env, kw, table_bits, const_chunk in SEG_CASES:
        table_c = None if table_bits is None else table_window_bits(SEG_N, table_bits)
        segs, plans, _ = segmented_plans(SEG_N, table_c=table_c, **kw)
        assert 3 <= len(segs) <= 5, env
        for (e0, e1), p in zip(segs, plans):
            seen |= _features(p)
            if e1 - e0 == CHUNK_ELEMS:
                seen.add("segment of one chunk")
            if const_chunk is not None and p.radix and e0 <= const_chunk * CHUNK_ELEMS < e1:
                canon = cref.from_mont(cref.scalar_field(0), seg_scalars(0, const_chunk)[e0:e1])
                if bucket_regime(p, partition_sizes(p, [canon])) == "gate closed":
                    seen.add("segment closes the gate alone")
        if const_chunk is not None:
            whole = cref.from_mont(cref.scalar_field(0), seg_scalars(0, const_chunk))
            others = [bucket_regime(p, partition_sizes(p, [whole[e0:e1]])) for (e0, e1), p in zip(segs, plans)
                      if p.radix and not e0 <= const_chunk * CHUNK_ELEMS < e1]
            assert others and all(r != "gate closed" for r in others)
        assert segs[-1][1] - segs[-1][0] >= 4097
    seg5 = host_segments(SEG_N, seg_pcts=(20, 40, 60, 80))
    assert seg5[-1] == (4 * CHUNK_ELEMS, SEG_N) and not plan(4097, 1, table_c=17, into=True).radix

    missing = REQUIRED - seen
    assert not missing, sorted(missing)

    # the shapes whose count pass needs more than 48 KB: c = 20 and plain c = 16 with 7 or 8 jobs, c = 21 with 4, 7 or 8
    over = {c.name for c in BUG_CASES if any(p.radix and p.smem0 > SMEM_DEFAULT for p in c.passes())}
    assert over == {"table c=20, 7 jobs", "table c=20, 8 jobs", "table c=21, 4 jobs", "table c=21, 7 jobs", "table c=21, 8 jobs",
                    "plain c=16, 7 jobs", "plain c=16, 8 jobs", "table c=20, 9 rows: passes of 8 and a remainder",
                    "table c=20, 17 rows: passes of 8 and a remainder"}
    assert [plan(1 << 14, j, table_c=21).lb for j in (3, 4, 5, 7, 8)] == [9, 9, 10, 10, 10]


def test_model_digits_recompose_the_scalar():
    """sum_w d_w 2^(c w) == s for the model's signed digits, at every window width and at the edges of the field"""
    q = pyref.scalar_modulus(0)
    rng = pyref.SplitMix64(5)
    vals = [0, 1, q - 1, q - 2, 1 << 253, (1 << 254) - 1] + [rng.field(q) for _ in range(50)]
    canon = cref.ints_to_arr(vals)
    for c in range(2, 22):
        nwin = -(-256 // c)
        d = signed_digits(canon, c, nwin)
        assert (np.abs(d) <= 1 << (c - 1)).all()
        for i, v in enumerate(vals):
            assert sum(int(d[i, w]) << (c * w) for w in range(nwin)) == v, (c, i)


# ---- GPU ----------------------------------------------------------------------------------------------------------------
_POINTS = {}


def key_points(curve, n):
    if (curve, n) not in _POINTS:
        _POINTS[(curve, n)] = cref.gen_points(curve, 0xD150 + curve, n)
    return _POINTS[(curve, n)]


def oracle(curve, pts, row, mont):
    return cref.commit(curve, pts, row) if mont else cref.msm_ark(curve, pts, row)


def run_case(c, case, plan_kw=None, expected=None):
    """one call on context `c`: launches as the model predicts, every row bit-exact with the oracle (or `expected`)"""
    pts = key_points(case.curve, case.key_n)
    B = c.register_bases(case.curve, pts)
    try:
        if case.table_c is not None:
            B.precompute(case.table_c)
        if case.window_bits:
            c.set_window_bits(case.window_bits)
        sc, _ = make_scalars(case)
        before = c.kernel_launches()
        if case.rows == 1:
            got = [c.msm(B, sc[0], montgomery=case.mont, offset=case.offset)]
        else:
            xy, inf = c.msm_batch(B, sc, montgomery=case.mont, offset=case.offset)
            got = [(xy[j], int(inf[j])) for j in range(case.rows)]
        launched = c.kernel_launches() - before
    finally:
        c.set_window_bits(0)
        B.release()
    assert launched == case.launches(**(plan_kw or {})), (case.name, launched)
    seg = pts[case.offset:case.offset + case.n]
    exp = expected if expected is not None else [oracle(case.curve, seg, sc[j], case.mont) for j in range(case.rows)]
    for j in range(case.rows):
        assert same_point(got[j], exp[j]), (case.name, j)
    return exp


def _run_all(ctx, cases):
    for case in cases:
        run_case(ctx, case)


@pytest.mark.gpu
def test_count_pass_beyond_48kb_of_shared_memory(ctx):
    """7 and 8 jobs over 2^19 buckets (c = 20 tables, plain c = 16), 4, 7 and 8 over 2^20 (c = 21), msm_batch of 9 and 17
    rows: the count pass of the radix sort asks for up to 64 KB of dynamic shared memory; 1, 6, 3 and 5 jobs beside them"""
    _run_all(ctx, BUG_CASES)


@pytest.mark.gpu
def test_sort_boundaries(ctx):
    """radix against counting sort at 2^17 pairs and at 1024 keys, staged against direct write pass, radix sort into the
    warp-coop accumulation at exactly 2^17 pairs over 8192 keys"""
    _run_all(ctx, SORT_CASES)


@pytest.mark.gpu
def test_bucket_pass_regimes_and_gate(ctx):
    """staged, direct and gate-closed partitions; one skewed job among uniform ones closes the gate for the whole pass"""
    _run_all(ctx, REGIME_CASES)


@pytest.mark.gpu
def test_reference_distributions_through_radix_passes(ctx):
    """the reference's scalar distributions through radix-sized passes of 1 and 8 jobs over a c = 20 table"""
    _run_all(ctx, DIST_CASES)


@pytest.mark.gpu
def test_accumulation_and_reduction_sweep(ctx):
    """warp-coop against balanced accumulation at 8192 buckets; c = 4..21 with tables and 4..16 on plain keys x {1, 2, 3, 8}
    jobs: reduction tiers N0 <= 32, <= 1024 and > 1024, split / coop / plain first levels, coop and plain finish"""
    _run_all(ctx, ACC_CASES + SWEEP_CASES)


@pytest.mark.gpu
def test_full_size_batch_over_c20_table(ctx):
    """8 rows of 2^20 scalars over a 2^20 key with its default (c = 20) table: one pass over 8192 partitions"""
    key = ctx.register_synthetic_bases(0, 0xF011, FULL_N)
    try:
        key.precompute()
        pts = ctx.download_bases(key)
        sc = cref.gen_scalars(cref.FQ, 0xF012, FULL_N * FULL_ROWS, True).reshape(FULL_ROWS, FULL_N, 4)
        before = ctx.kernel_launches()
        xy, inf = ctx.msm_batch(key, sc)
        assert ctx.kernel_launches() - before == plan(FULL_N, FULL_ROWS, table_c=table_window_bits(FULL_N)).launches
        for j in range(FULL_ROWS):
            assert same_point((xy[j], int(inf[j])), cref.commit(0, pts, sc[j])), j
    finally:
        key.release()


@pytest.mark.gpu
def test_product_poly_comm_eight_commitments_in_one_pass(ctx):
    """hp_product_poly_comm with n_in = 5 commits 2 n_in - 2 = 8 t-vectors in one pass over a c = 20 table"""
    curve = 1
    sf = cref.scalar_field(curve)
    pts = key_points(curve, 1 << 14)
    B = ctx.register_bases(curve, pts).precompute(20)
    try:
        a = [cref.gen_scalars(sf, 0x990 + i, HPPC_LEN - 3 * i, True) for i in range(HPPC_N_IN)]
        b = [cref.gen_scalars(sf, 0x9A0 + i, HPPC_LEN, True) for i in range(HPPC_N_IN)]
        mu = cref.gen_scalars(sf, 0x9B0, HPPC_N_IN + 1, True)
        before = ctx.kernel_launches()
        (low, linf), (high, hinf), tv = ctx.hp_product_poly_comm(B, a, b, mu, HPPC_LEN, want_tvecs=True)
        assert ctx.kernel_launches() - before == 1 + plan(HPPC_LEN, 2 * HPPC_N_IN - 2, table_c=20).launches   # k_tvecs + one pass
        t = cref.tvecs(sf, a, b, mu, HPPC_LEN)
        assert np.array_equal(tv, t)
        for j in range(HPPC_N_IN - 1):
            assert same_point((low[j], int(linf[j])), cref.commit(curve, pts[:HPPC_LEN], t[j])), ("low", j)
            assert same_point((high[j], int(hinf[j])), cref.commit(curve, pts[:HPPC_LEN], t[HPPC_N_IN + j])), ("high", j)
    finally:
        B.release()


@pytest.mark.gpu
def test_group_batch_of_eight_rows_over_c20_tables():
    """msm_batch of 8 rows on a virtual group of two contexts of one GPU: each child runs one 8-job pass over its half of the
    key with its own c = 20 table, then child 0 combines"""
    g = ab.Context(devices=[0, 0], min_shard=16)
    try:
        curve = 0
        pts = key_points(curve, GROUP_KEY)
        B = g.register_bases(curve, pts).precompute(20)
        sc = cref.gen_scalars(cref.scalar_field(curve), 0x6A0, GROUP_KEY * GROUP_ROWS, True).reshape(GROUP_ROWS, GROUP_KEY, 4)
        before = g.kernel_launches()
        xy, inf = g.msm_batch(B, sc)
        assert g.kernel_launches() - before == 2 * plan(GROUP_KEY // 2, GROUP_ROWS, table_c=20).launches + 1   # + k_combine_batch
        for j in range(GROUP_ROWS):
            assert same_point((xy[j], int(inf[j])), cref.commit(curve, pts, sc[j])), j
        B.release()
    finally:
        g.close()


@pytest.mark.gpu
def test_development_knobs_give_the_same_points(ctx, monkeypatch):
    """counting sort only (ACCMSM_SORT_LB=-1), 4096-key partitions (=12), everything on one stream (ACCMSM_NO_AUX=1) and the
    plain Horner finish (ACCMSM_NO_COOP_FINISH=1, plain keys): same points as the default context and the oracle"""
    expected = {case.name: run_case(ctx, case) for case in KNOB_CASES}
    for env, kw, plain_only in KNOBS:
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        c2 = ab.Context(0)
        try:
            for case in KNOB_CASES:
                if plain_only and case.table_c is not None:
                    continue
                run_case(c2, case, plan_kw=kw, expected=expected[case.name])
        finally:
            c2.close()
            for k in env:
                monkeypatch.delenv(k)


@pytest.mark.gpu
def test_segmented_host_msm_into_accumulation(monkeypatch):
    """A host-scalar MSM of 2^19 + 4097 points cut into 3 to 5 segments that add into one bucket set: segments of one chunk,
    a last segment of 4097 scalars (counting sort inside the segmented path), one segment whose constant scalars alone
    close the gate, a plain key.  Same point as the unsegmented MSM of the device-resident scalars and as the oracle."""
    import torch
    for i, (env, kw, table_bits, const_chunk) in enumerate(SEG_CASES):
        curve = i % 2
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        c2 = ab.Context(0)
        try:
            key = c2.register_synthetic_bases(curve, 0x5E0 + i, SEG_N)
            table_c = None
            if table_bits is not None:
                key.precompute(table_bits)
                table_c = table_window_bits(SEG_N, table_bits)
            sc = seg_scalars(curve, const_chunk)
            before = c2.kernel_launches()
            got = c2.msm(key, sc)
            segs, _, launches = segmented_plans(SEG_N, table_c=table_c, **kw)
            assert c2.kernel_launches() - before == launches, env
            d_sc = torch.from_numpy(sc.view(np.int64)).cuda()
            before = c2.kernel_launches()
            dev = c2.msm_dev(key, d_sc.data_ptr(), SEG_N)
            assert c2.kernel_launches() - before == plan(SEG_N, 1, table_c=table_c).launches
            assert same_point(got, dev), env
            assert same_point(got, cref.commit(curve, c2.download_bases(key), sc)), env
            key.release()
        finally:
            c2.close()
            for k in env:
                monkeypatch.delenv(k)
