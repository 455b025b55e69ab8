#!/usr/bin/env python
"""bench.py -- BASELINE.json headline: Pallas variable-base MSM throughput (Mpts/s) at 2^20 points per GPU,
plus the ipa-pc-as decide tail (fused h(X) -> commitment-key MSM) in ms at degree 2^18 / 2^20.

One process per GPU (torchrun).  A "step" is ONE MSM over the whole (sharded) key: every rank runs the
Pippenger pipeline on its contiguous point range, one 128-byte XYZZ partial per rank is all-gathered over
NCCL, rank 0 adds them and normalises (SURVEY.md 8e).  Weak scaling: 2^20 points per GPU, so the job at N
GPUs is a single N * 2^20-point MSM (config 5 of BASELINE.json sweeps 2^12 .. 2^24).

  value : Mpts/s with scalars already resident in HBM (device-timed, CUDA events per step, L2 flushed
          between steps, max over ranks)
  e2e   : same metric through the host-buffer path: pinned host scalars -> H2D -> MSM -> affine point D2H
  --impl reference : the CPU restatement of ark-ec 0.2 VariableBaseMSM (oracle/, OpenMP over windows like
          ark's rayon path) on the box's host cores -- the reference itself is Rust and cannot be built here.
"""
from __future__ import annotations

import argparse
import shutil
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (it may be read-only)

import numpy as np  # noqa: E402

LOG_N_PER_GPU = 20
SEED = 0xACC5
MULS_PER_MADD = 10            # XYZZ madd-2008-s: 8M + 2S (one pair of the 8M shares a reduction)


def int_peaks():
    """Integer roofline denominators in the regime k_accumulate runs in: tools/ubench2.cu at 16 warps per SM (128
    registers), bursts of ~2.5 ms with the effective clock recorded per point (profiles/r02a_ubench2.jsonl).  STATIC: read
    from the committed profile, not measured in this run."""
    out = {"fe_mul_gmul_s": None, "fe_mul_eff_mhz": None, "madd_gmul_eq_s": None, "madd_eff_mhz": None, "source": "profiles/r02a_ubench2.jsonl"}
    try:
        with open(os.path.join(ROOT, "profiles", "r02a_ubench2.jsonl")) as f:
            for line in f:
                d = json.loads(line)
                if d.get("warps_per_sm") != 16:
                    continue
                if d.get("bench") == "fe_mul":
                    out["fe_mul_gmul_s"], out["fe_mul_eff_mhz"] = d["g_per_s"], d["eff_mhz"]
                if d.get("bench") == "madd":
                    out["madd_gmul_eq_s"], out["madd_eff_mhz"] = d["gmul_equiv_per_s"], d["eff_mhz"]
    except Exception:
        pass
    return out


def ncu_static(kernel):
    """pipe utilisation of the committed `ncu --set full` capture of the shipped build (STATIC, profiles/ncu_static.json)"""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_static.json")) as f:
            return json.load(f).get(kernel)
    except Exception:
        return None


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def rand_scalars(n, seed):
    """uniform 254-bit values (< both moduli; the moduli are 2^254 + ~2^125): valid canonical integers and valid
    Fp256 Montgomery images alike"""
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 1 << 64, size=(n, 4), dtype=np.uint64)
    a[:, 3] &= np.uint64((1 << 62) - 1)
    return a


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        pw = [float(r[3]) for r in self.rows if len(r) >= 9 and r[3].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def oracle_threads(world):
    """host threads each rank's oracle leg may use (torchrun exports OMP_NUM_THREADS=1; undo it for the checker)"""
    return max(1, (os.cpu_count() or 1) // max(world, 1))


def gather_cpu_points(cref, dist, torch, dev, world, part):
    """all-gather one CPU-computed affine point (xy, inf) per rank and add them with the oracle -> (xy, inf) on every rank"""
    row = np.concatenate([np.asarray(part[0], dtype=np.uint64).reshape(8), np.array([part[1]], dtype=np.uint64)])
    t = torch.from_numpy(row.view(np.int64).copy()).to(dev).reshape(1, 9)
    out = torch.empty((world, 9), dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(out, t)
    rows = out.cpu().numpy().view(np.uint64)
    acc = (rows[0, :8].copy(), int(rows[0, 8]))
    for r in range(1, world):
        acc = cref.point_add(0, acc[0], acc[1], rows[r, :8].copy(), int(rows[r, 8]))
    return acc


def same_pt(a, b):
    return a is not None and b is not None and int(a[1]) == int(b[1]) and np.array_equal(np.asarray(a[0], np.uint64), np.asarray(b[0], np.uint64))


def words_f64(limbs):
    """uint64 limbs (field elements, point coordinates in the library's Montgomery image) -> their 32-bit words, low word
    first, as float64: exact, since every word is below 2^53"""
    return np.ascontiguousarray(limbs, dtype=np.uint64).view(np.uint32).astype(np.float64)


def point_f64(p):
    """(xy, inf) as the library returns it -> the 16 words of x || y followed by the infinity flag"""
    return np.append(words_f64(p[0]).reshape(16), float(p[1]))


def proof_f64(name, l_vec, r_vec, final_key, c):
    """an IpaPC::open proof: l_vec and r_vec (one point per round), final_comm_key (affine x || y) and c"""
    return {f"{name}_l": np.stack([point_f64(p) for p in l_vec]), f"{name}_r": np.stack([point_f64(p) for p in r_vec]),
            f"{name}_final_key": words_f64(final_key), f"{name}_c": words_f64(c)}


def dump_outputs(outdir, outputs):
    """--dump-outputs: one DIR/<name>.npy per result of the timed path, for comparing two builds output for output"""
    os.makedirs(outdir, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(outdir, f"{name}.npy"), np.asarray(a, dtype=np.float64))


def run_reference(args, rank, world):
    """--impl reference: the ark-ec VariableBaseMSM restatement on host cores, same config / metric / unit."""
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the reference arm is meant to use all the host threads it can
    # (ark's rayon path does), so undo that before the OpenMP runtime of liboracle.so starts
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    from oracle import cref
    n_full = 1 << LOG_N_PER_GPU
    pts = cref.gen_points(0, SEED, n_full)
    sc = rand_scalars(n_full, SEED + 1)
    t0 = time.perf_counter()
    cref.msm_ark(0, pts, sc)                                   # warm-up, also sizes the sample
    t_full = time.perf_counter() - t0
    # each step is a bounded sample of the workload: the whole 2^20-point MSM when K of them fit in ~150 s of CPU
    # time, else the largest power-of-two prefix that does (the metric is size-normalised: Mpts/s)
    budget_s = 150.0
    n = n_full
    while n > (1 << 14) and args.steps * t_full * (n / n_full) > budget_s:
        n >>= 1
    pts, sc = pts[:n], sc[:n]
    for _ in range(max(args.warmup - 1, 0) if n < n_full else 0):
        cref.msm_ark(0, pts, sc)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = cref.msm_ark(0, pts, sc)
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"msm": point_f64(res)})
    mpts = n / dt / 1e6
    cores = ark_threads(n, cref.num_threads())
    print(json.dumps({
        "impl": "reference", "metric": "Pallas MSM Mpts/s @2^20", "value": round(mpts, 4), "unit": "Mpts/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt * 1e3, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32x8 (255-bit Montgomery)", "data": "synthetic",
        "config": {"workload": f"pallas_msm_2^{LOG_N_PER_GPU}_per_gpu", "points_per_gpu": n_full, "curve": "pallas",
                   "note": "CPU restatement of ark-ec 0.2.0 VariableBaseMSM (c = ln-rule, rayon-over-windows -> OpenMP over windows); "
                           "the Rust reference cannot be built in this image (no cargo)",
                   # SURVEY 8d: probe, do not assume -- with a toolchain on the box `cargo run --release --features parallel --example
                   # scaling-pc` of the reference would be the true arkworks number; none of the pool's boxes has one (no network either)
                   "cargo_on_this_box": shutil.which("cargo") is not None},
        "cpu_baseline": {"value": round(mpts, 4), "unit": "Mpts/s", "cores": cores, "kind": "port",
                         "sample": f"one {n}-point MSM per step (the per-GPU share of the workload is 2^{LOG_N_PER_GPU} points), canonical scalars"},
        "e2e": {"value": round(mpts, 4), "unit": "Mpts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log-n", type=int, default=LOG_N_PER_GPU, help="log2 points per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-open", action="store_true", help="skip the IpaPC::open timing")
    ap.add_argument("--no-precompute", action="store_true", help="skip the per-key window table (one-shot bases)")
    ap.add_argument("--window-bits", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path computed in its last step as DIR/<name>.npy "
                                                          "(float64: 32-bit words of the limbs; points end with their infinity flag)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import accumulation_b200 as ab
    from accumulation_b200.sharded import ShardedMSM, shard_range

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: accumulation_b200 has no CPU path")
    numa = pin_to_gpu_numa_node(local_rank) if world > 1 and not os.environ.get("ACCMSM_NO_AFFINITY") else None
    args.warmup = max(args.warmup, 3)
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    dev = torch.device(f"cuda:{local_rank}")
    ctx = ab.Context(local_rank)
    n_per = 1 << args.log_n
    n_total = n_per * world
    start, count = shard_range(n_total, rank, world)

    # ---- inputs: key shard generated on its own GPU; scalars seeded per rank, pinned on the host
    key = ctx.register_synthetic_bases(ab.PALLAS, SEED, count + 1, first_index=start)   # + 1: the hiding generator h
    if not args.no_precompute:       # commitment keys are registered once; the table is part of registration
        key.precompute(args.window_bits)
    elif args.window_bits:
        ctx.set_window_bits(args.window_bits)
    sh = ShardedMSM(ctx, ab.PALLAS, key, n_total, rank, world, device=str(dev))
    sc_np = rand_scalars(count, SEED + 1 + rank)
    h_sc = torch.empty((count, 4), dtype=torch.int64).pin_memory()
    h_sc.numpy().view(np.uint64)[:] = sc_np
    d_sc = h_sc.to(dev)
    d_stage = torch.empty_like(d_sc)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # > 126 MB L2
    stream = torch.cuda.current_stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_dev():
        return sh.msm_dev(d_sc, montgomery=False)

    h_np = h_sc.numpy().view(np.uint64)            # the same page-locked buffer as seen by the C-ABI

    def step_e2e():
        # N = 1: the reference-facing C-ABI call accmsm_msm with a HOST pointer (upload in 4 MiB chunks on a copy stream, the
        # digit kernel follows chunk by chunk, result read back); N > 1: pinned copy to the shard's GPU + partial + gather
        if world == 1:
            return ctx.msm(sh.bases, h_np, montgomery=False, n=count)
        if os.environ.get("ACCMSM_E2E_TORCH_COPY"):          # development switch: the first version's path (torch H2D copy + msm_partial_dev)
            d_stage.copy_(h_sc, non_blocking=True)
            return sh.msm_dev(d_stage, montgomery=False)
        return sh.msm_host(h_sc, montgomery=False)           # accmsm_msm_partial with the same host pointer + gather + combine

    # ---- warm-up (also sizes the workspace) and parity of the thing being timed
    res = None
    for _ in range(args.warmup):
        res = step_dev()
        step_e2e()
    barrier()

    # ---- timed region 1: device-resident scalars, per-step CUDA events, L2 flushed between steps
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.kernel_launches()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    stage_acc = {}
    barrier()
    for a, b in evs:
        flush.zero_()
        a.record(stream)
        res = step_dev()
        b.record(stream)
        if world == 1:
            for k, v in ctx.last_timings().items():
                stage_acc[k] = stage_acc.get(k, 0.0) + v
    barrier()
    launches = ctx.kernel_launches() - launches0
    t_dev_ms = sum(a.elapsed_time(b) for a, b in evs) / args.steps
    if world > 1:
        for k, v in ctx.last_timings().items():
            stage_acc[k] = v * args.steps

    # ---- timed region 2: end to end from pinned host scalars (H2D inside), affine result read back on rank 0
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res_e2e = step_e2e()
    barrier()
    t_e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    clocks = sampler.stop() if rank == 0 else None

    tt = torch.tensor([t_dev_ms, t_e2e_ms], dtype=torch.float64, device=dev)
    lt = torch.tensor([launches], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
    t_dev_ms, t_e2e_ms = float(tt[0]), float(tt[1])
    launches = int(lt[0])
    outputs = {"msm": point_f64(res), "msm_e2e": point_f64(res_e2e)} if rank == 0 else {}

    checks = {}
    # ---- parity of the timed multi-GPU step: every rank restates the MSM of its own shard on the CPU (oracle), the N affine
    #      partials are added on the CPU and compared with the combined GPU point (device-resident and end-to-end paths)
    if world > 1 and not args.no_verify:
        from oracle import cref
        cref.set_num_threads(oracle_threads(world))
        exp_weak = gather_cpu_points(cref, dist, torch, dev, world, cref.msm_ark(0, ctx.download_bases(key, 0, count), sc_np))
        if rank == 0:
            checks["weak_msm_equals_oracle"] = same_pt(res, exp_weak) and same_pt(res_e2e, exp_weak)

    # ---- ipa-pc-as decide tail (metric string: decide ms at degree 2^18, target 2^20), one GPU.  Each degree gets the
    #      key a trimmed CommitterKey of that degree would register: 2^k generators + the hiding generator
    decide = {}
    extras_cpu = {}
    ipa_keys = {}
    if rank == 0 and world == 1:
        for k in (18, 20):
            if (1 << k) > count:
                continue
            if (1 << k) + 1 == key.n:
                ipa_keys[k] = key
            else:
                ipa_keys[k] = ctx.register_synthetic_bases(ab.PALLAS, SEED + k, (1 << k) + 1)
                ipa_keys[k].precompute()
            ch = rand_scalars(k, SEED + 77)
            fk = ctx.ipa_final_key(ipa_keys[k], ch)
            ts = []
            for _ in range(5):
                flush.zero_(); torch.cuda.synchronize()
                t0 = time.perf_counter()
                ok, dxy, dinf = ctx.ipa_check_final_key(ipa_keys[k], ch, fk[0], fk[1])
                ts.append((time.perf_counter() - t0) * 1e3)
                assert ok
            decide[f"ipa_decide_tail_ms_2^{k}"] = round(statistics.median(ts), 4)
            outputs[f"ipa_decide_tail_2^{k}"] = np.append(point_f64((dxy, dinf)), float(ok))     # final key, then accept
            if k == 18 and not args.no_cpu_baseline:
                # CPU restatement of the same tail (compute_coeffs serial like upstream + VariableBaseMSM over windows), same key
                from oracle import cref
                kp = ctx.download_bases(ipa_keys[k], 0, 1 << k)
                t0 = time.perf_counter()
                okc, cxy, cinf = cref.ipa_check_final_key(0, kp, ch, fk[0], fk[1])
                dtc = (time.perf_counter() - t0) * 1e3
                assert okc, "decide tail: GPU final key differs from the oracle"
                extras_cpu["ipa_decide_tail_ms_2^18"] = {"value": round(dtc, 1), "unit": "ms", "cores": ark_threads(1 << k, cref.num_threads()), "kind": "port",
                                                         "sample": "whole tail at degree 2^18 (same key and challenges; the GPU key equals the oracle's)"}

    # ---- config 4: ipa-pc-as decide at degree 2^20 with the key sharded by point range over all ranks (strong scaling);
    #      every rank expands its own coefficient range of h(X); one all-gather of 128-byte partials
    if world > 1:
        kk = 20
        s_lo, s_cnt = shard_range(1 << kk, rank, world)
        dkey = ctx.register_synthetic_bases(ab.PALLAS, SEED, s_cnt, first_index=s_lo)
        dkey.precompute()
        dsh = ShardedMSM(ctx, ab.PALLAS, dkey, 1 << kk, rank, world, device=str(dev))
        ch = rand_scalars(kk, SEED + 77)
        for _ in range(3):
            dsh.ipa_final_key(ch, kk)
        ts = []
        for _ in range(10):
            flush.zero_()
            barrier()
            t0 = time.perf_counter()
            fk = dsh.ipa_final_key(ch, kk)
            barrier()
            ts.append((time.perf_counter() - t0) * 1e3)
        if not args.no_verify:
            # parity of the sharded decide tail: every rank restates its own slice on the CPU (h(X) coefficients of its
            # range x its key shard), the CPU partials are added, and rank 0 compares; a corrupted challenge must reject
            from oracle import cref
            cref.set_num_threads(oracle_threads(world))
            dpts = ctx.download_bases(dkey, 0, s_cnt)
            coeffs = cref.from_mont(cref.FQ, cref.compute_coeffs(cref.FQ, ch)[s_lo:s_lo + s_cnt])
            exp_fk = gather_cpu_points(cref, dist, torch, dev, world, cref.msm_ark(0, dpts, coeffs))
            ch_bad = ch.copy(); ch_bad[3, 0] ^= np.uint64(1)
            fk_bad = dsh.ipa_final_key(ch_bad, kk)
            if rank == 0:
                checks["sharded_decide_accepts_oracle_key"] = same_pt(fk, exp_fk)
                checks["sharded_decide_rejects_corrupted_challenge"] = not same_pt(fk_bad, exp_fk)
        tdec = torch.tensor([statistics.median(ts)], dtype=torch.float64, device=dev)
        dist.all_reduce(tdec, op=dist.ReduceOp.MAX)
        decide[f"ipa_decide_tail_sharded_ms_2^{kk}"] = round(float(tdec[0]), 4)
        if rank == 0:
            outputs[f"ipa_final_key_sharded_2^{kk}"] = point_f64(fk)
        # config 5 strong scaling: ONE 2^20-point MSM sharded over all ranks (scalars resident in HBM)
        d_sl = d_sc[:s_cnt]
        for _ in range(3):
            strong_res = dsh.msm_dev(d_sl, montgomery=False)
        if not args.no_verify:
            exp_strong = gather_cpu_points(cref, dist, torch, dev, world, cref.msm_ark(0, dpts, sc_np[:s_cnt]))
            if rank == 0:
                checks["sharded_strong_msm_equals_oracle"] = same_pt(strong_res, exp_strong)
        ts = []
        for _ in range(10):
            flush.zero_()
            barrier()
            t0 = time.perf_counter()
            strong_res = dsh.msm_dev(d_sl, montgomery=False)
            barrier()
            ts.append((time.perf_counter() - t0) * 1e3)
        tdec = torch.tensor([statistics.median(ts)], dtype=torch.float64, device=dev)
        dist.all_reduce(tdec, op=dist.ReduceOp.MAX)
        decide[f"msm_sharded_strong_ms_2^{kk}"] = round(float(tdec[0]), 4)
        if rank == 0:
            outputs[f"msm_sharded_strong_2^{kk}"] = point_f64(strong_res)
        dkey.release()
        # ipa-pc-as prove hot path sharded: IpaPC::open at degree 2^20 with key / coefficients / z-vector sharded
        # cyclically (ShardedIpaOpen): per round one all-gather of 2 x 128-byte shares, last log2(N) rounds replicated
        if not args.no_open and world & (world - 1) == 0:
            import hashlib
            from accumulation_b200.mirror import _int_to_fe
            from accumulation_b200.sharded import ShardedIpaOpen

            def squeeze_s(prev, l, r):
                h = hashlib.blake2s(b"" if prev is None else prev.tobytes())
                h.update(l[0].tobytes()); h.update(r[0].tobytes())
                return _int_to_fe(1, int.from_bytes(h.digest()[:16], "little") | 1)

            if not args.no_verify:
                # parity of the sharded opening at a small degree: over NCCL against the oracle's round-by-round folding
                checks["sharded_open_equals_oracle_2^10"] = sharded_open_check(ctx, ab, rank, world, str(dev), 10)
            n_loc = (1 << kk) // world
            tmp = ctx.register_synthetic_bases(ab.PALLAS, SEED + 5, n_loc, first_index=rank * n_loc)
            hgen = ctx.register_synthetic_bases(ab.PALLAS, SEED + 6, 1)            # the same hiding generator on every rank
            okey = ctx.register_bases(ab.PALLAS, np.concatenate([ctx.download_bases(tmp), ctx.download_bases(hgen)]))
            tmp.release(); hgen.release()
            okey.precompute()
            so = ShardedIpaOpen(ctx, ab.PALLAS, okey, kk, rank=rank, world=world, hiding_index=n_loc, device=str(dev))
            cf = rand_scalars(n_loc, SEED + 200 + rank)
            xi0 = rand_scalars(1, SEED + 97).reshape(4)
            z = rand_scalars(1, SEED + 98).reshape(4)
            ts = []
            for _ in range(3):
                barrier()
                t0 = time.perf_counter()
                proof = so.open(cf, z, squeeze_s, xi0_mont=xi0)
                barrier()
                ts.append((time.perf_counter() - t0) * 1e3)
            tdec = torch.tensor([min(ts[1:])], dtype=torch.float64, device=dev)
            dist.all_reduce(tdec, op=dist.ReduceOp.MAX)
            decide[f"ipa_open_sharded_ms_2^{kk}"] = round(float(tdec[0]), 3)
            if rank == 0:
                outputs.update(proof_f64(f"ipa_open_sharded_2^{kk}", *proof[:4]))
            okey.release()

    # ---- ipa-pc-as prove hot path: IpaPC::open on device (metric string: prove ms at degree 2^18), one GPU
    if rank == 0 and world == 1 and not args.no_open:
        import hashlib
        from accumulation_b200.mirror import CommitterKey, InnerProductArgPC, _int_to_fe

        def squeeze(prev, l, r):   # host transcript stand-in, 128-bit challenges (src/ipa_pc_as/mod.rs:42)
            h = hashlib.blake2s(b"" if prev is None else prev.tobytes())
            h.update(l[0].tobytes()); h.update(r[0].tobytes())
            return _int_to_fe(1, int.from_bytes(h.digest()[:16], "little") | 1)

        for k in (18, 20):
            if k not in ipa_keys:
                continue
            n = 1 << k
            ck = CommitterKey(ipa_keys[k], n)
            coeffs = rand_scalars(n, SEED + 99)
            xi0 = rand_scalars(1, SEED + 97).reshape(4)               # h' = xi_0 * h with h = base n of the key
            z = rand_scalars(1, SEED + 98).reshape(4)
            ts = []
            for _ in range(2):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                l_vec, r_vec, fk, c, chs = InnerProductArgPC.open(ck, coeffs, z, None, squeeze, log_d=k, xi0=xi0)
                ts.append((time.perf_counter() - t0) * 1e3)
            ok, _, _ = ctx.ipa_check_final_key(ipa_keys[k], np.array(chs), fk, 0)     # the proof's final key passes the decider
            assert ok
            decide[f"ipa_open_ms_2^{k}"] = round(min(ts), 3)
            outputs.update(proof_f64(f"ipa_open_2^{k}", l_vec, r_vec, fk, c))

        # ---- AS-shaped prove (examples/scaling-as.rs:91-103: 1 input + 2 copies of an accumulator, zk; src/ipa_pc_as/mod.rs:625-668):
        #      m = 3 succinct-check group equations (2k + 3 term one-shot MSMs), the combined check polynomial built, evaluated and
        #      opened on the device (combine + evaluate + open); the sponge stays on the host (Blake2s stand-in)
        for k in (18,):
            if k not in ipa_keys:
                continue
            n, m_as = 1 << k, 3
            chm = rand_scalars(m_as * k, SEED + 300).reshape(m_as, k, 4)
            al = rand_scalars(m_as, SEED + 301)
            al[:, 2:] = 0                                               # 128-bit linear-combination challenges (src/ipa_pc_as/mod.rs:292-299)
            rp = rand_scalars(2, SEED + 302)                            # the random linear polynomial of the zk variant
            zz = rand_scalars(1, SEED + 303).reshape(4)
            xi0 = rand_scalars(1, SEED + 97).reshape(4)
            sc_pts = ctx.download_bases(ipa_keys[k], 0, 2 * k + 3)      # stand-ins for C, l_i, r_i, h', final_comm_key of an input
            sc_scal = rand_scalars(2 * k + 3, SEED + 304)
            sc_pts_m, sc_scal_m = np.stack([sc_pts] * m_as), np.stack([sc_scal] * m_as)
            ts = []
            for _ in range(2):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                sc_res = ctx.msm_oneshot_batch(ab.PALLAS, sc_pts_m, sc_scal_m, montgomery=False)   # succinct_check of every input / accumulator, one batched call
                sess, ev = ctx.ipa_open_begin_combined(ipa_keys[k], chm, al, zz, None, rp)
                ctx.ipa_open_use_hiding_generator(sess, n, xi0)
                xi, lr, nround, l_vec, r_vec = None, ctx.ipa_open_round(sess), 0, [], []
                while lr is not None:
                    xi = squeeze(xi, lr[0], lr[1])
                    l_vec.append(lr[0]); r_vec.append(lr[1])
                    lr = ctx.ipa_open_fold_round(sess, xi)
                    nround += 1
                fk, c = ctx.ipa_open_finish(sess)
                ts.append((time.perf_counter() - t0) * 1e3)
            assert nround == k
            decide[f"ipa_as_prove_ms_2^{k}"] = round(min(ts), 3)
            outputs.update(proof_f64(f"ipa_as_prove_2^{k}", l_vec, r_vec, fk, c))
            outputs[f"ipa_as_prove_2^{k}_succinct_msms"] = np.stack([point_f64(p) for p in zip(*sc_res)])
            outputs[f"ipa_as_prove_2^{k}_evaluation"] = words_f64(ev)
            decide["ipa_as_prove_shape"] = f"m = {m_as} (1 input + 2 accumulator copies), zk, degree 2^{k}: {m_as} succinct-check equations + combine + evaluate + open"

        # ---- CPU restatement of the opening / the AS-shaped prove on a BOUNDED sample (degree 2^12: the CPU folds the key
        #      generator by generator like upstream, ~4 core-seconds per 2^12 opening), with the GPU's time on the same sample
        if not args.no_cpu_baseline:
            from oracle import cref
            from tests.test_gpu_ipa_open import oracle_open, sponge_stand_in
            ks = 12
            pts = cref.gen_points(0, SEED + 400, (1 << ks) + 1)
            key_s, hp = pts[: 1 << ks], pts[1 << ks]
            cks = CommitterKey.new(ctx, ab.PALLAS, key_s)
            cks.bases.precompute()
            cf = rand_scalars(1 << ks, SEED + 401)
            zs = rand_scalars(1, SEED + 402).reshape(4)
            sq = sponge_stand_in(1)
            InnerProductArgPC.open(cks, cf, zs, hp, sq, log_d=ks)
            t0 = time.perf_counter()
            g = InnerProductArgPC.open(cks, cf, zs, hp, sq, log_d=ks)
            t_gpu = (time.perf_counter() - t0) * 1e3
            t0 = time.perf_counter()
            e = oracle_open(0, key_s, cf, zs, hp, sq)
            t_cpu = (time.perf_counter() - t0) * 1e3
            assert np.array_equal(g[2], e[2]) and np.array_equal(g[3], e[3]) and all(same_pt(a, b) for a, b in zip(g[0] + g[1], e[0] + e[1])), \
                "IpaPC::open: GPU proof differs from the oracle"
            extras_cpu["ipa_open_ms_2^12"] = {"value": round(t_cpu, 1), "unit": "ms", "cores": cref.num_threads(), "kind": "port",
                                              "sample": f"one opening at degree 2^{ks} (bounded sample of the 2^18 workload; proof bit-exact with the GPU's)",
                                              "gpu_ms_same_sample": round(t_gpu, 3)}
            cks.bases.release()

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- CPU baseline beside it (rank 0, N = 1 only) and bit-exact check of the timed result against it
    cpu = None
    verified = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import cref   # checker + reported baseline only
        pts = ctx.download_bases(key, 0, count)
        t0 = time.perf_counter()
        exp = cref.msm_ark(0, pts, sc_np)
        dt = time.perf_counter() - t0
        cpu = {"value": round(count / dt / 1e6, 4), "unit": "Mpts/s", "ms": round(dt * 1e3, 1), "cores": ark_threads(count, cref.num_threads()), "kind": "port",
               "sample": f"one full 2^{args.log_n}-point MSM (same bases and scalars as the GPU step), {dt:.2f} s"}
        if not args.no_verify:
            verified = bool(res[1] == exp[1] and np.array_equal(res[0], exp[0]) and np.array_equal(res_e2e[0], exp[0]))
            if not verified:
                raise SystemExit("bench: GPU result differs from the oracle -- refusing to report a number")

    hbm_peak, peak_kind = peaks()
    value = n_total / (t_dev_ms * 1e-3) / 1e6
    e2e = n_total / (t_e2e_ms * 1e-3) / 1e6
    t_acc_ms = stage_acc.get("accumulate", 0.0) / args.steps
    c = args.window_bits or (table_window_bits(count) if not args.no_precompute else ctx_window_bits(count))
    nwin = (256 + c - 1) // c
    out = {
        "metric": "Pallas MSM Mpts/s @2^20", "value": round(value, 3), "unit": "Mpts/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(t_dev_ms, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32x8 (255-bit Montgomery)", "data": "synthetic",
        "config": {"workload": f"pallas_msm_2^{args.log_n}_per_gpu", "points_per_gpu": count, "points_total": n_total,
                   "curve": "pallas", "scalars": "uniform 254-bit canonical (BigInteger256)", "window_bits": c, "windows": nwin,
                   "key": "plain (per-window bucket sets)" if args.no_precompute else "precomputed window table 2^(cw)P (built once at registration, one bucket set)",
                   "sharding": f"point-range x{world}, all-gather of one 128 B partial per GPU" if world > 1 else "single GPU",
                   "host_affinity": numa,
                   "l2": "flushed (256 MiB memset) between timed steps", "timing": "CUDA events per step on the launching stream"},
        "e2e": {"value": round(e2e, 3), "unit": "Mpts/s", "ms_per_step": round(t_e2e_ms, 4), "h2d_bytes_per_step": count * 32 * world,
                "d2h_bytes_per_step": 128},    # one un-normalised XYZZ sum (4 x 32 B); the host thread converts it to affine
        "gpu_launches": launches,
        "clocks": clocks,
        "stages_ms": {k: round(v / args.steps, 4) for k, v in stage_acc.items() if v},
    }
    if t_acc_ms > 0:
        achieved = 96.0 * count / (t_acc_ms * 1e-3) / 1e9
        out["roofline"] = {"kernel": "k_accumulate", "bound": "hbm", "achieved": round(achieved, 2), "peak": hbm_peak,
                           "unit": "GB/s", "frac": round(achieved / hbm_peak, 5), "traffic": measured_traffic(args.log_n, c, not args.no_precompute),
                           "peak_kind": peak_kind,
                           "algorithmic_bytes": 96 * count, "kernel_ms": round(t_acc_ms, 4)}
        madds = count * nwin
        gmul = madds * MULS_PER_MADD / (t_acc_ms * 1e-3) / 1e9
        ip = int_peaks()
        ns = ncu_static("k_accumulate")
        out["roofline_int"] = {"kernel": "k_accumulate", "bound": "imad (255-bit Montgomery products)", "achieved": round(gmul, 2),
                               "peak": ip["fe_mul_gmul_s"], "unit": "Gmul/s", "frac": round(gmul / ip["fe_mul_gmul_s"], 4) if ip["fe_mul_gmul_s"] else None,
                               "peak_regime": "Fp::mul microbenchmark at the kernel's occupancy (16 warps/SM), ~2.5 ms bursts; the part lowers its clock under "
                                              "this load (effective MHz recorded)", "peak_eff_mhz": ip["fe_mul_eff_mhz"],
                               "madd_ceiling": ip["madd_gmul_eq_s"], "frac_of_madd_ceiling": round(gmul / ip["madd_gmul_eq_s"], 4) if ip["madd_gmul_eq_s"] else None,
                               "madd_ceiling_note": "the kernel's own loop body (XYZZ mixed adds) with operands in registers, no memory traffic",
                               "insertions": madds, "static_peaks_from": ip["source"],
                               "ncu_static": ns}
    t_sort_ms = sum(stage_acc.get(k, 0.0) for k in ("digits", "scan", "scatter")) / args.steps
    if t_sort_ms > 0 and world == 1:
        pairs = count * nwin
        # traffic the two-level sort has to move: scalars read by the count and the write pass, (key, entry) pairs written once
        # and read by the bucket pass, entries + bucket offsets written
        sort_bytes = 2 * 32 * count + 2 * 8 * pairs + 4 * pairs + 4 * (1 << (c - 1))
        out["roofline_sort"] = {"kernels": "k_sort_tiles<count> + k_sort_tile_scan + k_scan + k_sort_tiles<write> + k_sort_buckets", "bound": "hbm",
                                "achieved": round(sort_bytes / (t_sort_ms * 1e-3) / 1e9, 1), "peak": hbm_peak, "unit": "GB/s",
                                "frac": round(sort_bytes / (t_sort_ms * 1e-3) / 1e9 / hbm_peak, 4), "bytes": sort_bytes, "ms": round(t_sort_ms, 4),
                                "pairs": pairs}
    if cpu:
        out["cpu_baseline"] = cpu
    if world > 1 and not args.no_verify:
        verified = bool(checks) and all(checks.values())
        out["verified_checks"] = checks
        if not verified:
            raise SystemExit(f"bench: a multi-GPU result differs from the oracle -- refusing to report a number: {checks}")
    if verified is not None:
        out["verified_vs_oracle"] = verified
    out.update(decide)
    if extras_cpu:
        out["cpu_baselines_protocol"] = extras_cpu
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def sharded_open_check(ctx, ab, rank, world, device, k):
    """ShardedIpaOpen over NCCL at degree 2^k against the oracle's opening (both ways of passing h'); True on every rank
    only if l_vec, r_vec, final_comm_key and c all agree"""
    from accumulation_b200.sharded import ShardedIpaOpen, cyclic_shard
    from oracle import cref
    from tests.test_gpu_ipa_open import oracle_open, sponge_stand_in
    from tests.test_gpu_sharded_open import _case
    ok = True
    for indexed in (True, False):
        sf, key, h, xi0, hp, coeffs, z = _case(0, k, 500 + k)
        shard = cyclic_shard(key, rank, world)
        bases = ctx.register_bases(0, np.concatenate([shard, h.reshape(1, 8)]))
        bases.precompute()
        so = ShardedIpaOpen(ctx, 0, bases, k, rank=rank, world=world, hiding_index=shard.shape[0], device=device)
        squeeze = sponge_stand_in(sf)
        res = so.open(cyclic_shard(coeffs, rank, world), z, squeeze, h_prime_xy=None if indexed else hp, xi0_mont=xi0 if indexed else None)
        el, er, efk, ec, _ = oracle_open(0, key, coeffs, z, hp, squeeze)
        ok = ok and all(same_pt(x, y) for x, y in zip(res[0], el)) and all(same_pt(x, y) for x, y in zip(res[1], er))
        ok = ok and np.array_equal(res[2], efk) and np.array_equal(res[3], ec)
        bases.release()
    return bool(ok)


def pin_to_gpu_numa_node(gpu_index):
    """one process per GPU: run this rank (and first-touch its page-locked scalar buffer) on the CPUs that are local to its
    GPU's PCIe root, so eight concurrent uploads do not cross the socket interconnect.  Best effort; returns the cpu list."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        ncpu = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [64 * w + b for w, word in enumerate(mask) for b in range(64) if (word >> b) & 1 and 64 * w + b < ncpu]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"{cpus[0]}-{cpus[-1]} ({len(cpus)} cpus)"
    except Exception:
        pass
    return None


def ark_threads(n, omp_threads):
    """ark-ec 0.2 parallelises over windows only (SURVEY.md App. A.1): threads actually busy = min(threads, windows)"""
    lg = max(n - 1, 1).bit_length()
    c = 3 if n < 32 else lg * 69 // 100 + 2
    return min(omp_threads, (255 + c - 1) // c)


def measured_traffic(log_n, c, table):
    """dram bytes per k_accumulate launch from the committed ncu capture, when it matches this configuration"""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)["k_accumulate"]
        if t["log_n"] == log_n and t["window_bits"] == c and bool(t["table"]) == bool(table):
            return int(t["traffic_bytes"])
    except Exception:
        pass
    return None


def table_window_bits(n):
    """mirror of the automatic rule in accmsm_precompute_bases (reporting only)"""
    lg = max(n, 1).bit_length() - 1
    return 20 if lg >= 20 else 17 if lg >= 15 else 15 if lg >= 13 else 10


def ctx_window_bits(n):
    """mirror of pick_window_bits() in accumulation_b200/csrc/accmsm.cu (reporting only)"""
    lg = max(n, 1).bit_length() - 1
    return min(16, max(4, lg - 3))


if __name__ == "__main__":
    main()
