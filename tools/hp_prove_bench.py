"""ASForHadamardProducts::prove (src/hp_as/mod.rs:646-813; BASELINE config 2) on Pallas over a key of len generators + the hiding
generator with its window table, at len = 2^16 and 2^20, n = 2 and n = 6 pairs (6 is the largest n of the reference's
multiple_inputs_accumulation_test), with and without zero knowledge.  Each line times one whole prove, sponge stand-ins included:

  * session: accmsm_hp_prove_begin / _product_poly_comm / _finish (the pairs uploaded once; with zk one kernel and one 3-job
    pass for the hiding commitments; k_tvecs and the 2n - 2 commitments; two k_lincomb launches for a* and b*);
  * composed: the calls that existed before the session, each uploading the pairs it needs again: with zk two vec_hadamard, one
    vec_lincomb and three accmsm_commit for the hiding commitments; hp_product_poly_comm; two vec_scale and two vec_lincomb
    for a* and b*.

Every call returns its results to the host, so a host clock around a prove ends in a synchronise.  Session and composed runs
alternate within one process; medians are reported.  Nothing is printed unless both paths and the oracle give the same hiding
commitments, low and high commitments, a* and b*, and the device decide and the oracle's accept the accumulator.
Usage: python tools/hp_prove_bench.py [--logs 16,20] [--ns 2,6] [--reps 7]"""
import argparse, json, os, statistics, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import accumulation_b200 as ab
from oracle import cref
from tests.test_gpu_hp_prove import from_mont, make_inputs, mu_list, mu_stand_in, nu_stand_in, oracle_decide, oracle_prove, to_mont
from tests.util import same_point

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=7)
ap.add_argument("--logs", default="16,20")
ap.add_argument("--ns", default="2,6")
args = ap.parse_args()
SEED = 0x4850
CURVE = ab.PALLAS
F = ab.scalar_field(CURVE)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception:
        return "unknown"


def timed(fn):
    t0 = time.perf_counter()
    res = fn()
    return (time.perf_counter() - t0) * 1e3, res


def pts_of(xy, inf):
    return [(xy[j], int(inf[j])) for j in range(len(inf))]


def session_prove(c, B, L, a, b, hz):
    n = len(a)
    sess, hc = c.hp_prove_begin(B, a, b, L, *(None, None) if hz is None else hz[:2], hiding_index=L, hiding_rand=None if hz is None else hz[2])
    hcl = None if hc is None else pts_of(*hc)
    mu = mu_list(F, mu_stand_in(F, n)(hcl), hz is not None)
    (lo, li), (hi, hf) = c.hp_prove_product_poly_comm(sess, n, to_mont(F, mu))
    low, high = pts_of(lo, li), pts_of(hi, hf)
    nu = nu_stand_in(F)(low, high)
    a_s, b_s = c.hp_prove_finish(sess, nu, L)
    return hcl, low, high, a_s, b_s, mu, from_mont(F, nu)[0]


def composed_prove(c, B, L, a, b, hz):
    n = len(a)
    m = ab.mirror._MODULI[F]
    hcl = None
    if hz is not None:
        ha, hb, hr = hz
        one = to_mont(F, [1, 1])
        k0, k1 = min(L, b[0].shape[0]), min(L, a[-1].shape[0])
        cross = c.lincomb(F, [c.hadamard(F, ha[:k0], b[0][:k0]), c.hadamard(F, a[-1][:k1], hb[:k1])], one)
        hcl = [c.commit(B, v, hiding_index=L, randomizer_mont=hr[j]) for j, v in enumerate((ha, hb, cross))]
    mu = mu_list(F, mu_stand_in(F, n)(hcl), hz is not None)
    (lo, li), (hi, hf), _ = c.hp_product_poly_comm(B, a, b, to_mont(F, mu), L, *(None, None) if hz is None else hz[:2])
    low, high = pts_of(lo, li), pts_of(hi, hf)
    nu_m = nu_stand_in(F)(low, high)
    nu = from_mont(F, nu_m)[0]
    nus = [pow(nu, j, m) for j in range(n)]
    ha_s = None if hz is None else c.scale(F, hz[0], to_mont(F, [mu[n]]))
    hb_s = None if hz is None else c.scale(F, hz[1], to_mont(F, [mu[1]]))
    a_s = c.lincomb(F, a, to_mont(F, [mu[i] * nus[i] for i in range(n)]), ha_s)
    b_s = c.lincomb(F, b[::-1], to_mont(F, nus), hb_s)
    return hcl, low, high, a_s, b_s, mu, nu


def same_points(x, y):
    return (x is None) == (y is None) and (x is None or all(same_point(p, q) for p, q in zip(x, y)))


ctx = ab.Context(0)
gpu = card()
checks, records = {}, []
for lg in [int(x) for x in args.logs.split(",")]:
    L = 1 << lg
    B = ctx.register_synthetic_bases(CURVE, SEED, L + 1)
    B.precompute()
    ck = ab.CommitterKey(B, L)
    pts = ctx.download_bases(B, 0, L + 1).reshape(-1, 8)
    for n in [int(x) for x in args.ns.split(",")]:
        for zk in (True, False):
            tag = f"2^{lg}_n{n}_{'zk' if zk else 'plain'}"
            wits, insts, hz = make_inputs(CURVE, pts[:L], pts[L], n, [(L, L)] * n, SEED + lg + n, zk, L)
            a, b = [w[0] for w in wits], [w[1] for w in wits]
            s_out = session_prove(ctx, B, L, a, b, hz)
            c_out = composed_prove(ctx, B, L, a, b, hz)
            hc, low, high, a_s, b_s, mu, nu = s_out
            ohc, olow, ohigh, oa, ob, orand, onew = oracle_prove(CURVE, pts[:L], pts[L], L, wits, insts, mu, nu, hz)
            checks[f"hiding_{tag}"] = same_points(hc, c_out[0]) and same_points(hc, ohc)
            checks[f"low_high_{tag}"] = all(same_points(x, y) and same_points(x, z) for x, y, z in ((low, c_out[1], olow), (high, c_out[2], ohigh)))
            checks[f"ab_star_{tag}"] = all(np.array_equal(x, y) and np.array_equal(x, z) for x, y, z in ((a_s, c_out[3], oa), (b_s, c_out[4], ob)))
            checks[f"decide_{tag}"] = ab.ASForHadamardProducts.decide(ck, onew, (a_s, b_s, orand)) and oracle_decide(CURVE, pts[:L], pts[L], onew, oa, ob, orand)

            def sess():
                return session_prove(ctx, B, L, a, b, hz)

            def comp():
                return composed_prove(ctx, B, L, a, b, hz)

            for fn in (sess, comp, sess, comp):       # warm-up
                fn()
            ts, tc = [], []
            for _ in range(args.reps):               # alternate within the run
                ts.append(timed(sess)[0]); tc.append(timed(comp)[0])
            ms, mc = round(statistics.median(ts), 3), round(statistics.median(tc), 3)
            records.append(dict(metric=f"hp_prove_{tag}", session_ms=ms, composed_ms=mc, speedup=round(mc / ms, 2), len=L, n=n, zk=zk,
                                curve="pallas", table=True, reps=args.reps, gpu=gpu))
    B.release()

if not all(checks.values()):
    print(json.dumps({"error": "checks failed", "checks": checks}), file=sys.stderr)
    sys.exit(1)
for rec in records:
    print(json.dumps(rec), flush=True)
