"""R1CS NARK prove (zk) and verify on the scaling-nark circuit (examples/scaling-nark.rs; BASELINE config 3 is M = 2^16) at
M = 2^16 and 2^20 on Pallas, over a key of M generators + the hiding generator with its window table.  Lines:

  * zk prove first message: accmsm_nark_prove_zk (one vector launch + one 8-job pass) against the same 8 commitments
    composed from the calls that existed before it: csr_matvec_commit on (x, w) and on (0, r) with the six vectors
    downloaded, three vec_hadamard and one vec_lincomb for cross and rr, and two accmsm_commit;
  * verify: accmsm_nark_verify (one vector launch + one 4-job pass) against csr_matvec_commit on (x, w') with t_A, t_B
    downloaded, vec_hadamard and accmsm_commit, compared on the host;
  * the non-zk prove (csr_matvec_commit, 3 commitments) for reference;
  * the accumulation decider (ASForR1CSNark::decide) on the accumulator of the zk proof (x, w', sigma_A..C; hp part t_A, t_B
    with sigma_A, sigma_B, sigma_o): accmsm_nark_as_decide (one vector launch + one 6-job pass) against csr_matvec_commit with
    the sigmas plus hp_decide (a second vector launch and pass, after uploading t_A and t_B again), compared on the host.

Every call returns its results to the host, so a host clock around it ends in a synchronise.  Fused and composed runs
alternate within one run; medians are reported.  Nothing is printed unless both paths and the oracle give the same 8
commitments, both verify paths agree, the device verify accepts the device proof, and both decide paths and the oracle give
the same six decide commitments and accept.
Usage: python tools/nark_bench.py [--logs 16,20] [--reps 7]"""
import argparse, json, os, statistics, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import accumulation_b200 as ab
from oracle import cref
from tests.test_gpu_nark import gamma_stand_in, oracle_lhs, oracle_nark_prove, scaling_system, zk_randomness
from tests.test_gpu_nark_as import oracle_decide
from tests.util import same_point

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=7)
ap.add_argument("--logs", default="16,20")
args = ap.parse_args()
SEED = 0x4A4B
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


def composed_prove(c, B, csr, M, inp, wit, r, bl):
    one = cref.to_mont(F, cref.from_int(1).reshape(1, 4))
    z, cz, iz = c.csr_matvec_commit(B, csr, 3, M, inp, wit, hiding_index=M, blinders=bl[:3])
    rv, cr, ir = c.csr_matvec_commit(B, csr, 3, M, np.zeros_like(inp), r, hiding_index=M, blinders=bl[3:6])
    cross = c.lincomb(F, [c.hadamard(F, z[0], rv[1]), c.hadamard(F, z[1], rv[0])], np.concatenate([one, one]))
    rr = c.hadamard(F, rv[0], rv[1])
    c1 = c.commit(B, cross, hiding_index=M, randomizer_mont=bl[6])
    c2 = c.commit(B, rr, hiding_index=M, randomizer_mont=bl[7])
    return [(cz[i], int(iz[i])) for i in range(3)] + [(cr[i], int(ir[i])) for i in range(3)] + [c1, c2]


def composed_verify(c, B, csr, M, inp, wp, sig, lhs):
    t, ct, it = c.csr_matvec_commit(B, csr, 3, M, inp, wp, hiding_index=M, blinders=sig[:3])
    co = c.commit(B, c.hadamard(F, t[0], t[1]), hiding_index=M, randomizer_mont=sig[3])
    rhs = [(ct[i], int(it[i])) for i in range(3)] + [co]
    return all(same_point(a, b) for a, b in zip(lhs, rhs))


def composed_decide(c, B, csr, M, inp, wp, sig, a, b, hpr, exp):
    _, ct, it = c.csr_matvec_commit(B, csr, 3, M, inp, wp, hiding_index=M, blinders=sig, want_vecs=False)
    ok_hp, hxy, hinf = c.hp_decide(B, a, b, np.array([p[0] for p in exp[3:]]), [p[1] for p in exp[3:]], hiding_index=M, randomness=hpr)
    pts = [(ct[i], int(it[i])) for i in range(3)] + [(hxy[i], int(hinf[i])) for i in range(3)]
    return ok_hp and all(same_point(e, p) for e, p in zip(exp[:3], pts[:3])), pts


ctx = ab.Context(0)
gpu = card()
checks, records = {}, []
for lg in [int(x) for x in args.logs.split(",")]:
    M = 1 << lg
    B = ctx.register_synthetic_bases(CURVE, SEED, M + 1)
    B.precompute()
    ck = ab.CommitterKey(B, M)
    mats, inp, wit = scaling_system(F, M, SEED + lg)
    r, bl = zk_randomness(F, wit.shape[0], SEED + 100 + lg)
    nark = ab.R1CSNark(ck, mats)
    gam = gamma_stand_in(F)
    # parity: fused, composed and the oracle give the same 8 commitments; both verify paths accept the device proof
    _, fxy, finf = ctx.nark_prove_zk(B, nark.csr, M, inp, wit, r, bl, hiding_index=M, want_vecs=False)
    fused_first = [(fxy[i], int(finf[i])) for i in range(8)]
    comp_first = composed_prove(ctx, B, nark.csr, M, inp, wit, r, bl)
    pts = ctx.download_bases(B, 0, M + 1).reshape(-1, 8)
    _, ofirst, _, _, _ = oracle_nark_prove(CURVE, mats, pts[:M], pts[M], inp, wit, gam, (r, bl))
    checks[f"prove_fused_eq_composed_2^{lg}"] = all(same_point(a, b) for a, b in zip(fused_first, comp_first))
    checks[f"prove_fused_eq_oracle_2^{lg}"] = all(same_point(a, b) for a, b in zip(fused_first, ofirst))
    proof = nark.prove(inp, wit, gam, zk=(r, bl))
    gamma = gam(proof.first_msg)
    checks[f"verify_accepts_device_proof_2^{lg}"] = nark.verify(inp, proof, gamma)
    # the verifier's left-hand sides comm_M + gamma comm_rM, comm_C + gamma comm_1 + gamma^2 comm_2 (oracle point arithmetic),
    # shared by both timed verify paths
    lhs = oracle_lhs(CURVE, proof.first_msg, gamma)
    lhs_xy, lhs_inf = np.array([p[0] for p in lhs]), [p[1] for p in lhs]
    checks[f"verify_composed_accepts_2^{lg}"] = composed_verify(ctx, B, nark.csr, M, inp, proof.blinded_witness, proof.sigmas, lhs)

    # the accumulator of the zk proof; both decide paths and the oracle give the same six points and accept
    _, tv, _, _ = ctx.nark_verify(B, nark.csr, M, inp, proof.blinded_witness, lhs_xy, lhs_inf, hiding_index=M, sigmas=proof.sigmas,
                                  want_vecs=True)
    ta, tb = tv[0], tv[1]
    dsig, dhr = proof.sigmas[:3], np.stack([proof.sigmas[0], proof.sigmas[1], proof.sigmas[3]])
    dexp = [lhs[0], lhs[1], lhs[2], lhs[0], lhs[1], lhs[3]]
    dexp_xy, dexp_inf = np.array([p[0] for p in dexp]), [p[1] for p in dexp]
    okf, dxy, dinf = ctx.nark_as_decide(B, nark.csr, inp, proof.blinded_witness, ta, tb, dexp_xy, dexp_inf, hiding_index=M, sigmas=dsig,
                                        hp_randomness=dhr)
    okc, cpts = composed_decide(ctx, B, nark.csr, M, inp, proof.blinded_witness, dsig, ta, tb, dhr, dexp)
    oko, opts = oracle_decide(CURVE, mats, pts[:M], pts[M], inp, proof.blinded_witness, ta, tb, dexp, dsig, dhr)
    checks[f"decide_all_accept_2^{lg}"] = okf and okc and oko
    checks[f"decide_fused_eq_composed_eq_oracle_2^{lg}"] = all(same_point((dxy[j], dinf[j]), cpts[j]) and same_point(cpts[j], opts[j])
                                                               for j in range(6))

    def fused_d():
        return ctx.nark_as_decide(B, nark.csr, inp, proof.blinded_witness, ta, tb, dexp_xy, dexp_inf, hiding_index=M, sigmas=dsig,
                                  hp_randomness=dhr)[0]

    def comp_d():
        return composed_decide(ctx, B, nark.csr, M, inp, proof.blinded_witness, dsig, ta, tb, dhr, dexp)[0]

    def fused_p():
        return ctx.nark_prove_zk(B, nark.csr, M, inp, wit, r, bl, hiding_index=M, want_vecs=False)

    def comp_p():
        return composed_prove(ctx, B, nark.csr, M, inp, wit, r, bl)

    def fused_v():
        return ctx.nark_verify(B, nark.csr, M, inp, proof.blinded_witness, lhs_xy, lhs_inf, hiding_index=M, sigmas=proof.sigmas)[0]

    def comp_v():
        return composed_verify(ctx, B, nark.csr, M, inp, proof.blinded_witness, proof.sigmas, lhs)

    def nonzk_p():
        return ctx.csr_matvec_commit(B, nark.csr, 3, M, inp, wit, want_vecs=False)

    for fn in (fused_p, comp_p, fused_v, comp_v, nonzk_p, fused_d, comp_d):       # warm-up
        fn(); fn()
    t = {k: [] for k in ("fp", "cp", "fv", "cv", "np", "fd", "cd")}
    for _ in range(args.reps):                                    # alternate within the run
        t["fp"].append(timed(fused_p)[0]); t["cp"].append(timed(comp_p)[0])
        tv, okf = timed(fused_v); t["fv"].append(tv)
        tc, okc = timed(comp_v); t["cv"].append(tc)
        checks[f"verify_timed_accepts_2^{lg}"] = checks.get(f"verify_timed_accepts_2^{lg}", True) and okf and okc
        t["np"].append(timed(nonzk_p)[0])
        td, okd = timed(fused_d); t["fd"].append(td)
        tc, okcd = timed(comp_d); t["cd"].append(tc)
        checks[f"decide_timed_accepts_2^{lg}"] = checks.get(f"decide_timed_accepts_2^{lg}", True) and okd and okcd
    med = {k: round(statistics.median(v), 3) for k, v in t.items()}
    base = {"M": M, "curve": "pallas", "table": True, "reps": args.reps, "gpu": gpu}
    records += [
        dict(metric=f"nark_prove_zk_2^{lg}", fused_ms=med["fp"], composed_ms=med["cp"], speedup=round(med["cp"] / med["fp"], 2), **base),
        dict(metric=f"nark_verify_2^{lg}", fused_ms=med["fv"], composed_ms=med["cv"], speedup=round(med["cv"] / med["fv"], 2), **base),
        dict(metric=f"nark_prove_nonzk_2^{lg}", ms=med["np"], **base),
        dict(metric=f"nark_as_decide_2^{lg}", fused_ms=med["fd"], composed_ms=med["cd"], speedup=round(med["cd"] / med["fd"], 2), **base),
    ]
    nark.release(); B.release()

if not all(checks.values()):
    print(json.dumps({"error": "checks failed", "checks": checks}), file=sys.stderr)
    sys.exit(1)
for rec in records:
    print(json.dumps(rec), flush=True)
