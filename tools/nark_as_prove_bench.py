"""ASForR1CSNark::prove (src/r1cs_nark_as/mod.rs:713-926; SURVEY App. C.12) on Pallas: the scaling-nark circuit over a key of
n_rows generators + the hiding generator with its window table, 1 fresh input + 2 old accumulators (the shape of
examples/scaling-as.rs), with and without zero knowledge, at n_rows = 2^16 and 2^20.  Each line times the device part of one
prove, sponge stand-ins included (the host MSMs of the blinded commitments and of comm_M* are the same in both paths):

  * session: accmsm_nark_as_prove_begin / accmsm_hp_prove_product_poly_comm / accmsm_nark_as_prove_finish (one row-kernel launch
    writes the fresh mat-vecs into the hp pair buffers; with zk also M (r_x || r_w), the hiding rows and one 6-job pass; three
    k_lincomb launches for a*, b*, w*);
  * composed: the calls that existed before the session: csr_matvec per fresh input (A and B x_i || w'_i back to the host),
    with zk csr_matvec_commit for the randomness commitments, the hp session over the uploaded pairs, and vec_lincomb for w*.
    csr_matvec takes the matrices from the host and uploads A and B (row pointers, columns, coefficients) on every call, while
    the session reads the matrices registered once; part of the gap is that upload, not only the fused pass and the resident
    pair buffers.

Every call returns its results to the host, so a host clock around a prove ends in a synchronise.  Session and composed runs
alternate within one process; medians are reported.  Nothing is printed unless both paths and the oracle give the same begin
points, low and high commitments, a*, b* and w*, and the device decider accepts the new accumulator.
Usage: python tools/nark_as_prove_bench.py [--logs 16,20] [--reps 7]"""
import argparse, json, os, statistics, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import accumulation_b200 as ab
from oracle import cref
from tests.util import same_point
from tests.test_gpu_hp_prove import from_mont, mu_list, mu_stand_in, nu_stand_in, to_mont
from tests.test_gpu_nark import gamma_stand_in, scaling_system, zk_randomness
from tests.test_gpu_nark_as_prove import beta_stand_in, oracle_as_prove, prover_zk

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=7)
ap.add_argument("--logs", default="16,20")
args = ap.parse_args()
SEED = 0x4E41
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


def fresh_of(nark, x, w, zk, seed):
    """a fresh input from the device NARK prover -> the tuple shape of the test restatement (x, first, gamma, w', sigmas)"""
    g = gamma_stand_in(F)
    p = nark.prove(x, w, g, zk=zk_randomness(F, w.shape[0], seed) if zk else None)
    return x, p.first_msg, g(p.first_msg) if zk else None, np.asarray(p.blinded_witness), p.sigmas


def acc_tuple(inst, wit):
    a, b, hpr = wit.hp_witness
    return (np.asarray(inst.r1cs_input), np.asarray(wit.r1cs_blinded_witness), a, b, None if wit.randomness is None else np.array(wit.randomness),
            None if hpr is None else np.array(hpr), [inst.comm_a, inst.comm_b, inst.comm_c] + list(inst.hp_instance))


def session_prove(c, B, csr, M, fr, accs, z):
    n = 1 + len(accs)
    sess, pts = c.nark_as_prove_begin(B, csr, [fr[0]], [fr[3]], [a[1] for a in accs], [a[2] for a in accs], [a[3] for a in accs],
                                      zk=None if z is None else (z[0], z[1], z[3], z[4], np.concatenate([z[2], z[5]])), hiding_index=M)
    begin = None if pts is None else pts_of(*pts)
    mu = mu_list(F, mu_stand_in(F, n)(None if begin is None else begin[:3]), z is not None)
    (lo, li), (hi, hf) = c.hp_prove_product_poly_comm(sess, n, to_mont(F, mu))
    low, high = pts_of(lo, li), pts_of(hi, hf)
    nu_m = nu_stand_in(F)(low, high)
    beta = beta_of(begin, low, high, mu, nu_m, accs, fr, z)
    a_s, b_s, w_s = c.nark_as_prove_finish(sess, nu_m, to_mont(F, beta), M, fr[3].shape[0])
    return begin, low, high, a_s, b_s, w_s, (mu, from_mont(F, nu_m)[0], beta)


def beta_of(begin, low, high, mu, nu_m, accs, fr, z):
    """beta from the stand-in over the new hp instance (the mirror's combined_commitments, one small host-side batch)"""
    ck = CK
    n = 1 + len(accs)
    bl = ab.mirror._oneshot_equations(ck, [[(fr[1][i], 1), (fr[1][3 + i], from_mont(F, fr[2].reshape(1, 4))[0]), ((fr[1][i][0], 1), 0)]
                                           for i in range(3)] + [[(fr[1][2], 1), (fr[1][6], from_mont(F, fr[2].reshape(1, 4))[0]),
                                                                  (fr[1][7], from_mont(F, fr[2].reshape(1, 4))[0] ** 2)]]) \
        if z is not None else [fr[1][0], fr[1][1], fr[1][2], fr[1][2]]
    insts = [(bl[0], bl[1], bl[3])] + [tuple(a[6][3:]) for a in accs]
    hp_inst = ab.ASForHadamardProducts.combined_commitments(ck, insts, None if begin is None else begin[:3], low, high, mu, from_mont(F, nu_m)[0])
    return [1] + from_mont(F, beta_stand_in(F, n + (z is not None))(hp_inst, None if begin is None else begin[3:]))


def composed_prove(c, B, csr, mats, M, fr, accs, z):
    n = 1 + len(accs)
    x, _, _, wp, _ = fr
    t = c.csr_matvec(F, mats[:2], x, wp)                 # A (x || w'), B (x || w') back to the host
    comm_r = None
    if z is not None:
        _, xy, inf = c.csr_matvec_commit(B, csr, 3, M, z[0], z[1], hiding_index=M, blinders=z[2], want_vecs=False)
        comm_r = pts_of(xy, inf)
    a = [t[0]] + [v[2] for v in accs]
    b = [t[1]] + [v[3] for v in accs]
    sess, hc = c.hp_prove_begin(B, a, b, M, *(None, None) if z is None else (z[3], z[4]), hiding_index=M, hiding_rand=None if z is None else z[5])
    hcl = None if hc is None else pts_of(*hc)
    mu = mu_list(F, mu_stand_in(F, n)(hcl), z is not None)
    (lo, li), (hi, hf) = c.hp_prove_product_poly_comm(sess, n, to_mont(F, mu))
    low, high = pts_of(lo, li), pts_of(hi, hf)
    nu_m = nu_stand_in(F)(low, high)
    begin = None if z is None else hcl + comm_r
    beta = beta_of(begin, low, high, mu, nu_m, accs, fr, z)
    a_s, b_s = c.hp_prove_finish(sess, nu_m, M)
    ws = [wp] + [v[1] for v in accs]
    w_s = c.lincomb(F, ws, to_mont(F, beta[:n]), None if z is None else c.scale(F, z[1], to_mont(F, beta[n:])))
    return begin, low, high, a_s, b_s, w_s, (mu, from_mont(F, nu_m)[0], beta)


def same_points(x, y):
    return (x is None) == (y is None) and (x is None or all(same_point(p, q) for p, q in zip(x, y)))


ctx = ab.Context(0)
gpu = card()
checks, records = {}, []
for lg in [int(x) for x in args.logs.split(",")]:
    M = 1 << lg
    B = ctx.register_synthetic_bases(CURVE, SEED, M + 1)
    B.precompute()
    CK = ab.CommitterKey(B, M)
    pts = ctx.download_bases(B, 0, M + 1).reshape(-1, 8)
    mats, x, w = scaling_system(F, M, SEED + lg)
    nark = ab.R1CSNark(CK, mats, num_instance_variables=x.shape[0])
    for zk in (True, False):
        tag = f"2^{lg}_f1a2_{'zk' if zk else 'plain'}"
        # two valid old accumulators, each the mirror's prove over two device NARK proofs, then one fresh input
        accs = []
        for j in range(2):
            frs = [fresh_of(nark, x, w, zk, SEED + 10 * j + i) for i in range(2)]
            z0 = prover_zk(F, x.shape[0], w.shape[0], M, SEED + 50 + j) if zk else None
            inst, wit, _ = ab.ASForR1CSNark.prove(nark, [(f[0], ab.NarkProof(f[1], f[3], f[4])) for f in frs], [], gamma_stand_in(F),
                                                  mu_stand_in(F, 2), nu_stand_in(F), beta_stand_in(F, 2 + zk), zk=z0)
            accs.append(acc_tuple(inst, wit))
        fr = fresh_of(nark, x, w, zk, SEED + 90)
        z = prover_zk(F, x.shape[0], w.shape[0], M, SEED + 91) if zk else None
        s_out = session_prove(ctx, B, nark.csr, M, fr, accs, z)
        c_out = composed_prove(ctx, B, nark.csr, mats, M, fr, accs, z)
        ob, olow, ohigh, oacc, _ = oracle_as_prove(CURVE, mats, pts[:M], pts[M], [fr], accs, z, fixed=s_out[6])
        checks[f"begin_{tag}"] = same_points(s_out[0], c_out[0]) and same_points(s_out[0], ob)
        checks[f"low_high_{tag}"] = all(same_points(s_out[k], c_out[k]) and same_points(s_out[k], o) for k, o in ((1, olow), (2, ohigh)))
        checks[f"stars_{tag}"] = all(np.array_equal(s_out[k], c_out[k]) and np.array_equal(s_out[k], oacc[j]) for k, j in ((3, 2), (4, 3), (5, 1)))
        inst, wit, _ = ab.ASForR1CSNark.prove(nark, [(fr[0], ab.NarkProof(fr[1], fr[3], fr[4]))],
                                              [(ab.AccumulatorInstance(a[0], a[6][0], a[6][1], a[6][2], tuple(a[6][3:])),
                                                ab.AccumulatorWitness(a[1], (a[2], a[3], None if a[5] is None else list(a[5])),
                                                                      None if a[4] is None else list(a[4]))) for a in accs],
                                              gamma_stand_in(F), mu_stand_in(F, 3), nu_stand_in(F), beta_stand_in(F, 3 + zk), zk=z)
        checks[f"mirror_{tag}"] = np.array_equal(wit.r1cs_blinded_witness, oacc[1]) and all(
            same_point(p, q) for p, q in zip([inst.comm_a, inst.comm_b, inst.comm_c] + list(inst.hp_instance), oacc[6]))
        checks[f"decide_{tag}"] = ab.ASForR1CSNark.decide(nark, inst, wit)

        def sess():
            return session_prove(ctx, B, nark.csr, M, fr, accs, z)

        def comp():
            return composed_prove(ctx, B, nark.csr, mats, M, fr, accs, z)

        for fn in (sess, comp, sess, comp):       # warm-up
            fn()
        ts, tc = [], []
        for _ in range(args.reps):               # alternate within the run
            ts.append(timed(sess)[0]); tc.append(timed(comp)[0])
        ms, mc = round(statistics.median(ts), 3), round(statistics.median(tc), 3)
        records.append(dict(metric=f"nark_as_prove_{tag}", session_ms=ms, composed_ms=mc, speedup=round(mc / ms, 2), n_rows=M, n_fresh=1,
                            n_acc=2, zk=zk, curve="pallas", table=True, reps=args.reps, gpu=gpu))
    nark.release()
    B.release()

if not all(checks.values()):
    print(json.dumps({"error": "checks failed", "checks": checks}), file=sys.stderr)
    sys.exit(1)
for rec in records:
    print(json.dumps(rec), flush=True)
