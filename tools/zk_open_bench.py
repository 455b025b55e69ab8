"""Zero-knowledge AS-shaped prove (examples/scaling-as.rs runs MakeZK::Enabled) at degree 2^18 and 2^20: the sequence of
bench.py's ipa_as_prove line (3 batched succinct-check equations, the combined check polynomial built and evaluated on the
device) plus the hiding step of a zk opening -- accmsm_ipa_open_hide (upload, evaluate, shift, hiding_comm MSM), alpha
squeezed on the host, accmsm_ipa_open_hiding_challenge, C' = C + alpha hiding_comm - rand s (a 3-term one-shot MSM) and
xi_0 from C' -- then the rounds.  Reports the whole prove, the hiding step alone, and the non-zk prove of the same run.

Nothing is printed unless every check agrees: the 2^10 zk proof matches the oracle composition (poly_evaluate, commit,
combine_vectors, the round-by-round opening) bit for bit, the 2^18 / 2^20 proofs of a group (--devices) match the
single-device proof, and check_final_key accepts every proof.  The same-run CPU restatement of the host work the device
path replaces (the oracle's poly_evaluate + combine_vectors at 2^18) is timed too, with its thread count.
Usage: python tools/zk_open_bench.py [--devices 0,0] [--reps 5]   (a device listed twice makes a virtual group)"""
import argparse, hashlib, json, os, statistics, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import accumulation_b200 as ab
from accumulation_b200.mirror import _fe_to_int, _int_to_fe
from oracle import cref
from tests.test_gpu_ipa_open_zk import Case, assert_matches_oracle, run_zk, same_proof

ap = argparse.ArgumentParser()
ap.add_argument("--devices", default=None)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--logs", default="18,20")
args = ap.parse_args()
SEED = 0xACC5
F = 1          # curve 0 (Pallas): scalars in field 1


def rand_scalars(n, seed):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 1 << 64, size=(n, 4), dtype=np.uint64)
    a[:, 3] &= np.uint64((1 << 62) - 1)
    return a


def squeeze(prev, l, r):       # host transcript stand-in, 128-bit challenges (src/ipa_pc_as/mod.rs:42)
    h = hashlib.blake2s(b"" if prev is None else np.asarray(prev).tobytes())
    h.update(np.asarray(l[0]).tobytes()); h.update(np.asarray(r[0]).tobytes())
    return _int_to_fe(F, int.from_bytes(h.digest()[:16], "little") | 1)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception:
        return "unknown"


# ---- 1. the 2^10 zk proof against the oracle composition (single-device ctx and the group)
ref = ab.Context(0)
grp = ab.Context(devices=[int(d) for d in args.devices.split(",")], min_shard=0) if args.devices else None
case = Case(0, 10)
checks = {}
for name, c in (("single", ref), ("group", grp)):
    if c is None:
        continue
    B = c.register_bases(0, case.all); B.precompute()
    try:
        got = run_zk(c, B, case, True, True)
        assert_matches_oracle(case, got)
        checks[f"oracle_2^10_{name}"] = True
    finally:
        B.release()


# ---- 2. the AS-shaped prove, with and without the hiding step
def as_prove(c, B, k, zk, data):
    n, m_as = 1 << k, 3
    t0 = time.perf_counter()
    c.msm_oneshot_batch(ab.PALLAS, data["sc_pts"], data["sc_scal"], montgomery=False)
    sess, ev = c.ipa_open_begin_combined(B, data["chm"], data["al"], data["z"], None, data["rp"])
    t_hide = 0.0
    hc = rand = None
    if zk:
        th = time.perf_counter()
        hc = c.ipa_open_hide(sess, data["hiding"], n + 1, data["rho"])
        alpha = squeeze(None, (data["C"][0], 0), hc)                 # sponge over (C, z, v, hiding_comm)
        c.ipa_open_hiding_challenge(sess, alpha)
        rand = _int_to_fe(F, _fe_to_int(F, data["r"]) + _fe_to_int(F, alpha) * _fe_to_int(F, data["rho"]))
        c2 = ab.InnerProductArgPC.hiding_commitment(data["ck"], (data["C"][0], 0), hc, alpha, rand)
        xi0 = squeeze(None, c2, c2)                                  # xi_0 from C'
        t_hide = (time.perf_counter() - th) * 1e3
    else:
        xi0 = data["xi0"]
    c.ipa_open_use_hiding_generator(sess, n, xi0)
    xi, lr, l_vec, r_vec, chs = None, c.ipa_open_round(sess), [], [], []
    while lr is not None:
        xi = squeeze(xi, lr[0], lr[1])
        l_vec.append(lr[0]); r_vec.append(lr[1]); chs.append(xi)
        lr = c.ipa_open_fold_round(sess, xi)
    fk, cc = c.ipa_open_finish(sess)
    total = (time.perf_counter() - t0) * 1e3
    return total, t_hide, (l_vec, r_vec, fk, cc, chs), hc, rand


records = []
for k in [int(x) for x in args.logs.split(",")]:
    n = 1 << k
    B = ref.register_synthetic_bases(0, SEED, n + 2); B.precompute()      # generators || h || s
    ck = ab.CommitterKey(B, n, n + 1)
    data = dict(ck=ck, chm=rand_scalars(3 * k, SEED + 300).reshape(3, k, 4), al=rand_scalars(3, SEED + 301), rp=rand_scalars(2, SEED + 302),
                z=rand_scalars(1, SEED + 303).reshape(4), xi0=rand_scalars(1, SEED + 97).reshape(4), hiding=rand_scalars(n, SEED + 305),
                rho=rand_scalars(1, SEED + 306).reshape(4), r=rand_scalars(1, SEED + 307).reshape(4),
                sc_pts=np.stack([ref.download_bases(B, 0, 2 * k + 3)] * 3), sc_scal=np.stack([rand_scalars(2 * k + 3, SEED + 304)] * 3))
    data["al"][:, 2:] = 0
    data["C"] = (ref.download_bases(B, 7, 1).reshape(8), 0)                 # stand-in for the commitment being opened
    rec = {"metric": f"zk_as_prove_2^{k}", "gpu": card(), "reps": args.reps}
    for name, c in (("single", ref), ("group", grp)):
        if c is None:
            continue
        Bc = B if c is ref else c.register_synthetic_bases(0, SEED, n + 2)
        if c is not ref:
            Bc.precompute()
        dc = dict(data, ck=ab.CommitterKey(Bc, n, n + 1))
        for zk in (True, False):
            as_prove(c, Bc, k, zk, dc); as_prove(c, Bc, k, zk, dc)          # warm-up
        tz, th, tn, proofs = [], [], [], []
        for _ in range(args.reps):                                           # zk and non-zk alternate
            t, h, proof, hc, rand = as_prove(c, Bc, k, True, dc)
            tz.append(t); th.append(h); proofs.append((proof, hc, rand))
            tn.append(as_prove(c, Bc, k, False, dc)[0])
        proof, hc, rand = proofs[-1]
        checks[f"final_key_2^{k}_{name}"] = bool(c.ipa_check_final_key(Bc, np.array(proof[4]), proof[2], 0)[0])
        checks[f"repeatable_2^{k}_{name}"] = all(same_proof(p[0], proof) for p in proofs)
        if name == "single":
            single = (proof, hc)
        else:
            checks[f"group_matches_single_2^{k}"] = same_proof(proof, single[0]) and np.array_equal(hc[0], single[1][0])
            Bc.release()
        tag = "" if name == "single" else f"_group{args.devices.replace(',', '')}"
        rec.update({f"zk_prove_ms{tag}": round(statistics.median(tz), 3), f"hiding_step_ms{tag}": round(statistics.median(th), 3),
                    f"nonzk_prove_ms{tag}": round(statistics.median(tn), 3)})
    B.release()
    records.append(rec)

# ---- 3. CPU restatement of the host work the device hiding step replaces, 2^18: evaluate the hiding polynomial, combine
k = 18
hid = cref.gen_scalars(F, 5, 1 << k, True)
P = cref.gen_scalars(F, 6, 1 << k, True)
z = cref.gen_scalars(F, 7, 1, True).reshape(4)
al = np.stack([_int_to_fe(F, 1), cref.gen_scalars(F, 8, 1, True).reshape(4)])
ts = []
for _ in range(3):
    t0 = time.perf_counter()
    e = cref.poly_evaluate(F, hid, z)
    h2 = hid.copy(); h2[0] = cref.fe_sub(F, h2[0], e)
    cref.combine_vectors(F, [P, h2], al)
    ts.append((time.perf_counter() - t0) * 1e3)

if not all(checks.values()):
    print(json.dumps({"error": "checks failed", "checks": checks}), file=sys.stderr)
    sys.exit(1)
for rec in records:
    rec["checks"] = sorted(checks)
    print(json.dumps(rec), flush=True)
print(json.dumps({"metric": "cpu_restatement_eval_combine_2^18_ms", "ms": round(min(ts), 3), "oracle_threads": cref.num_threads(),
                  "cpu_cores": os.cpu_count(), "gpu": card()}), flush=True)
