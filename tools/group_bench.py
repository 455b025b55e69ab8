"""Device-group ctx (accmsm_init_multi) in ONE process, 1 / 2 / 4 / 8 GPUs: the reference-facing host-pointer calls with
keys sharded inside the library (no torch.distributed, no NCCL).  One JSON line per group size:
  weak   : one G * 2^20-point MSM from pinned host scalars (the bench.py e2e shape), Mpts/s
  strong : one 2^20-point MSM, the ipa-pc-as decide tail at degree 2^20 / 2^18 (config 4), hp-as decide with 2^16-element
           vectors (config 2), r1cs-nark A z / B z / C z + three commitments at 2^16 constraints (config 3), ms
  open   : IpaPC::open (h' by index, fold_round per round) at 2^20 and 2^18, sharded across the group at the default
           min_shard on >= 2 GPUs, and at 2^14, which stays on child 0: a workload on each side of the rule, ms
Every result is compared with the single-device ctx (which the GPU suite pins to the oracle) before it is printed.
Usage: python tools/group_bench.py [--gpus 1,2,4,8] [--devices 0,0]   (--devices: one group over exactly these devices;
a device listed twice makes a virtual group on one GPU, which runs every path but measures no multi-GPU speed)"""
import argparse, json, os, statistics, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import accumulation_b200 as ab
from tests.test_gpu_fused import scaling_nark_matrices
from tests.test_gpu_ipa_open import sponge_stand_in

ap = argparse.ArgumentParser()
ap.add_argument("--gpus", default="1,2,4,8")
ap.add_argument("--devices", default=None)
ap.add_argument("--reps", type=int, default=10)
args = ap.parse_args()
SEED = 0xACC5


def rand_scalars(n, seed):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 1 << 64, size=(n, 4), dtype=np.uint64)
    a[:, 3] &= np.uint64((1 << 62) - 1)
    return a


def timed(fn, reps):
    fn(); fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); r = fn(); ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts), r


def same(a, b):
    return int(a[1]) == int(b[1]) and np.array_equal(np.asarray(a[0]), np.asarray(b[0]))


ref = ab.Context(0)
N20 = 1 << 20
# single-device references (strong-scaling workloads)
key1 = ref.register_synthetic_bases(0, SEED, N20 + 1); key1.precompute()
sc20 = ab.pinned_array((N20, 4)); sc20[:] = rand_scalars(N20, SEED + 1)
ref_msm = ref.msm(key1, sc20, montgomery=False)
ch20 = rand_scalars(20, SEED + 77)
ref_fk20 = ref.ipa_final_key(key1, ch20)
ref_fk18 = ref.ipa_final_key(key1, ch20[:18])
OPEN_LOGS = (20, 18, 14)
open_coeffs = rand_scalars(N20, SEED + 31)
open_z, open_xi0 = rand_scalars(1, SEED + 32).reshape(4), rand_scalars(1, SEED + 33).reshape(4)
open_squeeze = sponge_stand_in(1)       # curve 0: scalars in field 1


def open_proof(c, B, lk):
    ck = ab.CommitterKey(B, N20)        # the hiding generator is base N20
    return ab.InnerProductArgPC.open(ck, open_coeffs[:1 << lk], open_z, None, open_squeeze, log_d=lk, xi0=open_xi0)


def same_proof(a, b):
    return (all(same(x, y) for x, y in zip(a[0] + a[1], b[0] + b[1])) and len(a[0]) == len(b[0])
            and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3]))


ref_open = {lk: open_proof(ref, key1, lk) for lk in OPEN_LOGS}
L = 1 << 16
keyL = ref.register_synthetic_bases(0, SEED + 9, L + 1); keyL.precompute()
a, b = rand_scalars(L, 11), rand_scalars(L, 12)
r3 = rand_scalars(3, 13)
_, hp_xy, hp_inf = ref.hp_decide(keyL, a, b, np.zeros((3, 8), np.uint64), np.zeros(3, np.uint8), hiding_index=L, randomness=r3)
mats, n_in, n_wit = scaling_nark_matrices(1, L, dense=True)
inp, wit, bl = rand_scalars(n_in, 21), rand_scalars(n_wit, 22), rand_scalars(3, 23)
csr1 = ref.register_csr(1, mats)
ref_vecs, ref_cxy, ref_cinf = ref.csr_matvec_commit(keyL, csr1, 3, L, inp, wit, hiding_index=L, blinders=bl)

groups = [[int(d) for d in args.devices.split(",")]] if args.devices else [list(range(int(G))) for G in args.gpus.split(",")]
for devs in groups:
    G = len(devs)
    g = ab.Context(devices=devs) if G > 1 else ab.Context(devs[0])
    rec = {"gpus": G, "devices": devs, "process": "one process, accmsm_init_multi" if G > 1 else "one process, accmsm_init"}
    # ---- weak: one G * 2^20-point MSM, host scalars (pinned), whole call timed
    n = N20 * G
    kw = g.register_synthetic_bases(0, SEED, n); kw.precompute()
    scw = ab.pinned_array((n, 4)); scw[:] = rand_scalars(n, SEED + 100)
    t, res = timed(lambda: g.msm(kw, scw, montgomery=False), args.reps)
    # verification: the same MSM as G single-device MSMs over the ranges, summed on the device by a (G + 0)-term one-shot MSM
    parts = []
    for r in range(G):
        kr = ref.register_synthetic_bases(0, SEED, N20, first_index=r * N20); kr.precompute()
        parts.append(ref.msm(kr, scw[r * N20:(r + 1) * N20], montgomery=False)); kr.release()
    one = np.zeros((G, 4), np.uint64); one[:, 0] = 1
    tot = ref.msm_oneshot(0, np.array([p[0] for p in parts]), one, montgomery=False, infinity=np.array([p[1] for p in parts], np.uint8))
    rec.update({"weak_msm_points": n, "weak_msm_ms": round(t, 4), "weak_msm_mpts": round(n / t / 1e3, 2), "weak_verified": same(res, tot)})
    kw.release(); ab.release_pinned(scw); del scw
    # ---- strong: the 2^20 workloads
    ks = g.register_synthetic_bases(0, SEED, N20 + 1); ks.precompute()
    t, res = timed(lambda: g.msm(ks, sc20, montgomery=False), args.reps)
    rec.update({"strong_msm_2^20_ms": round(t, 4), "strong_msm_verified": same(res, ref_msm)})
    t, res = timed(lambda: g.ipa_final_key(ks, ch20), args.reps)
    rec.update({"decide_tail_2^20_ms": round(t, 4), "decide_20_verified": same(res, ref_fk20)})
    t, res = timed(lambda: g.ipa_final_key(ks, ch20[:18]), args.reps)
    rec.update({"decide_tail_2^18_ms": round(t, 4), "decide_18_verified": same(res, ref_fk18)})
    bad = ch20.copy(); bad[7, 1] ^= np.uint64(8)
    rec["decide_rejects_corrupted"] = not g.ipa_check_final_key(ks, bad, ref_fk20[0], ref_fk20[1])[0]
    for lk in OPEN_LOGS:
        t, res = timed(lambda: open_proof(g, ks, lk), args.reps)
        rec.update({f"ipa_open_2^{lk}_ms": round(t, 4), f"ipa_open_{lk}_verified": same_proof(res, ref_open[lk])})
    ks.release()
    # ---- config 2 / 3 at 2^16 (below the default shard size: min_shard lowered so the group really splits them)
    g.set_min_shard(1 << 13) if G > 1 else None
    kl = g.register_synthetic_bases(0, SEED + 9, L + 1); kl.precompute()
    t, res = timed(lambda: g.hp_decide(kl, a, b, hp_xy, hp_inf, hiding_index=L, randomness=r3), args.reps)
    rec.update({"hp_decide_2^16_ms": round(t, 4), "hp_decide_accepts": bool(res[0])})
    csr = g.register_csr(1, mats)
    t, res = timed(lambda: g.csr_matvec_commit(kl, csr, 3, L, inp, wit, hiding_index=L, blinders=bl), args.reps)
    rec.update({"nark_matvec_commit_2^16_ms": round(t, 4),
                "nark_verified": all(np.array_equal(x, y) for x, y in zip(res[0], ref_vecs)) and np.array_equal(res[1], ref_cxy)})
    g.release_csr(csr); kl.release()
    rec["all_verified"] = all(v for k, v in rec.items() if k.endswith("verified") or k.endswith("accepts") or k.endswith("corrupted"))
    print(json.dumps(rec), flush=True)
    g.close()
