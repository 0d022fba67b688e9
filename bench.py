#!/usr/bin/env python3
"""Benchmark of the RTI-MPC hot path (BASELINE.json: "A1 centroidal MPC solves/sec").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--config NAME] [--dump-outputs DIR]

A "step" is one real-time-iteration solve (MPC::GetRealTimeUpdate: horizon maintenance -> linearise -> assemble ->
QP -> line search -> trajectory update) of every instance in the batch.  Workload at N=1: BASELINE config #2,
"A1 trot MPC batched over 4096 synthetic initial states" (apps/a1_configuration.yaml: 20 nodes x 0.05 s, 372
decision variables, 1012 constraint rows per instance).  With N>1 (torchrun, one rank per GPU) every rank runs its
own 4096 instances (weak scaling; instances are independent, there is no collective on the solve path; NCCL is
used for the barrier, the max-over-ranks time and the final gather of per-instance results).

Prints ONE JSON line.  --impl reference times the CPU oracle (the restated reference algorithm; the reference binary
itself cannot be built in this image, see DESIGN.md) on the host cores for the same metric.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "bilevel-gait-gen_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
import sharding  # noqa: E402
import workloads as wl  # noqa: E402

METRIC = "A1 SRB-MPC RTI solves/sec"
UNIT = "solves/s"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def ipm_algorithmic_bytes(N, nu, n_samples, n_eebox, n_eq):
    """Compulsory HBM traffic of one k_ipm instance: the structured QP it must read once + the solution it writes
    (DESIGN.md, "kernel 4"): H nu^2, g nu, position rows 2(N-3) nu, NodeLin records, samples, equality rows, offsets,
    header; u, lam, slack, nu_eq."""
    m = 6 * n_samples + 2 * n_eebox
    reads = 8 * (nu * nu + nu + 2 * (N - 3) * nu + 12 * (N + 1)) + 1696 * (N + 1) + 56 * n_samples + 48 * n_eq + 256
    writes = 8 * (nu + 2 * m + n_eq) + 64
    return reads + writes


def ipm_algorithmic_flops(N, nu, nf, n_samples, iters, refined_iters):
    """FP64 flops of one k_ipm instance (2 per multiply-add), DESIGN.md "kernel 4".  Per factorisation (iters + 1: the
    starting point has one): K assembly = rank-2(N-3) update of the nf x nf triangle, Cholesky nu^3/6.  Per iteration:
    3 solves (constant, affine, combined right-hand side: nu^2 each, forward + backward), 1 product with H (nu^2),
    4 products with the structured C and 4 with C' (dense position rows 2(N-3) nf + ~36 per force sample each).  An
    iteration that runs with refinement (the kernel counts them: bgg_sizes.refined_iters) adds, for the constant and the
    combined solve, one more solve, one product with H and one with C and C' each."""
    nkc = 2 * (N - 3)
    cprod = nkc * nf + 36 * n_samples
    fact = nkc * nf * (nf + 1) / 2 + nu ** 3 / 6
    per_it = 3 * nu * nu + nu * nu + 8 * cprod
    per_ref = 2 * (nu * nu + nu * nu + 2 * cprod)
    start = nu * nu + 2 * cprod
    return 2 * ((iters + 1) * fact + iters * per_it + refined_iters * per_ref + start)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(outputs, out_dir):
    """Write every per-instance array as out_dir/<name>.npy in float64.  Above DUMP_LIMIT_BYTES the same fixed, seeded sample of
    instances is kept from every array and its indices are written as sample_rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    arrs = {k: np.asarray(v, np.float64) for k, v in outputs.items()}
    B = len(next(iter(arrs.values())))
    row_bytes = sum(a[0].nbytes for a in arrs.values())
    if B * row_bytes > DUMP_LIMIT_BYTES:
        keep = (DUMP_LIMIT_BYTES - (1 << 16)) // (row_bytes + 8)   # 64 KB left for the .npy headers
        rows = np.sort(np.random.default_rng(0).choice(B, keep, replace=False))
        arrs = {k: a[rows] for k, a in arrs.items()}
        arrs["sample_rows"] = rows.astype(np.float64)
    for k, a in arrs.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def oracle_latency(cfg_name, solves):
    """Single-thread latency of the oracle's RTI solve on the nominal instance (ms): p50, p95."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import common
    cfg = wl.CONFIGS[cfg_name]
    init = np.asarray(cfg["srb_init"], float)
    o = common.make_oracle(cfg_name)
    o.initial_run(init, wl.EE_NOMINAL)
    ts = []
    for _ in range(solves):
        t = time.perf_counter()
        o.solve(init, 0.0, wl.EE_NOMINAL, real_time=True)
        ts.append(1e3 * (time.perf_counter() - t))
    return float(np.percentile(ts, 50)), float(np.percentile(ts, 95))


def oracle_throughput(cfg_name, sample, steps, warmup, threads):
    """CPU leg: the oracle's restatement of the live reference path (interior-point QP), `sample` instances of the same
    synthetic workload spread over `threads` host threads; every instance does `warmup` + `steps` RTI solves."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import common
    import pyoracle
    pyoracle.build()
    cfg = wl.CONFIGS[cfg_name]
    states, _, ee = wl.batched_trot_inputs(cfg, sample, seed=0)
    oracles = [common.make_oracle(cfg_name, states[b]) for b in range(sample)]

    def run(tid, nsteps):
        for b in range(tid, sample, threads):
            for _ in range(nsteps):
                oracles[b].solve(states[b], 0.0, ee[b], real_time=True)

    def parallel(nsteps):
        ts = [threading.Thread(target=run, args=(t, nsteps)) for t in range(threads)]
        t0 = time.perf_counter()
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        return time.perf_counter() - t0

    if warmup:
        parallel(warmup)
    el = parallel(steps)
    return sample * steps / el, el


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=4096, help="instances per GPU")
    ap.add_argument("--config", default="a1_configuration", choices=sorted(wl.CONFIGS))
    ap.add_argument("--cpu-sample", type=int, default=0)
    ap.add_argument("--ipm-refine", type=int, default=0, help="0 = library default, -1 = no refinement")
    ap.add_argument("--ipm-refine-after", type=int, default=0, help="refine once mu <= 10^-k of its first value (0 = library default, -1 = always)")
    ap.add_argument("--max-spline-vars", type=int, default=0)
    ap.add_argument("--latency-solves", type=int, default=200)
    ap.add_argument("--closed-loop", action="store_true",
                    help="BASELINE config #5: --scenarios closed-loop scenarios cut across the ranks (strong scaling); a step is one "
                         "closed-loop tick (plant step + RTI solve) of every scenario")
    ap.add_argument("--scenarios", type=int, default=65536)
    ap.add_argument("--no-extra-configs", action="store_true", help="skip the short legs of BASELINE configs #3 and #5 after the headline")
    ap.add_argument("--gait-opt", type=int, default=0, metavar="K",
                    help="BASELINE config #3: per step every instance does solve -> dH/dtheta -> contact-time LP -> line search over "
                         "K candidates (K + 1 RTI solves per instance and step); use with --config a1_gait_opt_config --batch 64")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0) to DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    cfg = wl.CONFIGS[args.config]
    cores = os.cpu_count() or 1
    workload = (f"{args.config}: A1 trot SRB-MPC, N={cfg['num_nodes']} nodes x {cfg['integrator_dt']} s, "
                f"{args.batch} synthetic initial states per GPU, t0=0")
    if args.gait_opt:
        workload = (f"{args.config}: gait optimisation, N={cfg['num_nodes']} nodes x {cfg['integrator_dt']} s, {args.batch} instances per GPU, "
                    f"per step solve + dH/dtheta + contact-time LP + line search over {args.gait_opt} candidates "
                    f"({1 + args.gait_opt} RTI solves per instance and step)")
    if args.closed_loop:
        workload = (f"{args.config}: disturbance-rejection sweep, N={cfg['num_nodes']} nodes x {cfg['integrator_dt']} s, "
                    f"{args.scenarios} closed-loop scenarios cut across {world} GPU(s), plant = node 1 of the solved trajectory")

    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes what the CUDA path computed: use it with --impl ours")
        if rank != 0:
            return
        sample = args.cpu_sample or 8 * cores
        v, el = oracle_throughput(args.config, sample, args.steps, args.warmup, cores)
        p50, p95 = oracle_latency(args.config, 30)
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": workload, "note": "CPU oracle (restated reference algorithm: same assembly, Clarabel's interior-point algorithm "
                           "with an envelope LDL'); the reference binary needs Eigen/pinocchio/Clarabel which are absent from this image"},
                "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                 "sample": f"{sample} instances x {args.steps} RTI solves on {cores} threads"},
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "latency": {"p50_ms": p50, "p95_ms": p95, "what": "one RTI solve of the nominal instance, one host thread"}}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    import bgg_b200 as bg

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_mpc(cfg_name, batch, states):
        c = wl.CONFIGS[cfg_name]
        m = bg.BatchedMPC(c["num_nodes"], c["integrator_dt"], wl.robot(), device=local_rank, ipm_refine=args.ipm_refine,
                          ipm_refine_after=args.ipm_refine_after, max_spline_vars=args.max_spline_vars, **wl.mpc_kwargs(c))
        m.AddQuadraticTrackingCost(wl.target_tangent(c), np.asarray(c["Q"], float))
        m.Reset(batch)
        m.SetStateTrajectoryWarmStart(states)
        return m

    def run_leg(cfg_name, mode, batch, steps, warmup, gait_k=0, scenarios=0, detail=False, capture=False):
        """One timed leg.  mode: 'solve' (config #2: `batch` instances per GPU, weak scaling), 'gait' (config #3: per step solve
        + dH/dtheta + contact-time LP + line search over gait_k candidates) or 'closed_loop' (config #5: `scenarios`
        closed-loop scenarios cut across the ranks, strong scaling).  Device time with CUDA events on the launching stream,
        barrier + synchronise on both sides, max over ranks; end-to-end time through the host-buffer API with the decision
        vectors copied back every step."""
        c = wl.CONFIGS[cfg_name]
        N = c["num_nodes"]
        if mode == "closed_loop":
            lo, hi = sharding.shard_range(scenarios, rank, world)
            B = hi - lo
            st, t0, ee = wl.disturbance_sweep_inputs(c, scenarios, seed=7)
            st, t0, ee = st[lo:hi].copy(), t0[lo:hi].copy(), ee[lo:hi].copy()
        else:
            B = batch
            st, t0, ee = wl.batched_trot_inputs(c, B, seed=1000 + rank)
        mpc = make_mpc(cfg_name, B, st)
        dt_plant = c["integrator_dt"]
        gait_stats = {"grad_ok": 0, "best_hist": np.zeros(max(gait_k, 1), np.int64)}
        last_gait = {}
        n_max = 12 * (N + 1) + (args.max_spline_vars or 160)
        # the buffer the decision vectors come back into: page-locked, as a controller that reads them every tick would hold it
        z_pinned = torch.zeros((B, n_max), dtype=torch.float64).pin_memory()
        z_host = z_pinned.numpy()

        def gait_tail():   # MPCController::GaitOpt + GaitOptimizer::LineSearch for every instance of the batch
            g = mpc.ComputeCostFcnDerivWrtContactTimes()
            lp = mpc.OptimizeContactTimes(t0)
            ls = mpc.LineSearch(st, t0, ee, lp["xk"], lp["step"], K=gait_k)
            gait_stats["grad_ok"] = int((g["status"] == 0).sum())
            gait_stats["best_hist"] += np.bincount(np.maximum(ls["best"], 0), minlength=gait_k)
            last_gait.update(grad_status=g["status"], n_contacts=g["n_contacts"], dHdtheta=g["raw"], lp_step=lp["step"], lp_xk=lp["xk"],
                             lp_new_times=lp["new_times"], lp_status=lp["status"], ls_best=ls["best"], ls_costs=ls["costs"],
                             ls_quality=ls["quality"])

        snapshot = []

        def step():
            if mode == "closed_loop":
                mpc.advance_plant(dt_plant)
            for b, inst in enumerate(snapshot):   # gait leg: every timed step starts from the same trajectories and contact times
                mpc.set_instance(b, inst)
            mpc.solve_resident()
            if mode == "gait":
                gait_tail()

        mpc.upload(st, t0, ee)
        mpc.solve_resident()
        for _ in range(warmup):
            step()
        if mode == "gait":
            # a gait-optimisation step moves the contact times, so consecutive steps are different problems (3x spread of the step
            # time over a dozen steps); the timed steps all repeat the one after the warm-up -- 19 KB per instance re-uploaded per step
            snapshot = [mpc.get_instance(b).copy() for b in range(B)]
        mpc.synchronize()
        barrier()
        l0 = mpc.launch_count()
        mpc.event_record(0)
        for _ in range(steps):
            step()
        mpc.event_record(1)
        ms_dev = mpc.event_elapsed_ms(0, 1)
        barrier()
        launches = mpc.launch_count() - l0
        res = mpc.download(z_out=z_host if capture else None)
        out = {"B": B, "N": N, "mpc": mpc, "res": res, "launches": launches, "sizes": mpc.sizes(0), "gait_stats": gait_stats}
        # with capture: the results of the last timed step's solve (in gait mode read back after its gradient, LP and line search, which
        # leave them in place) and its gait outputs, copied before the loops below reuse the buffers; z is [B][n_max], the columns past
        # an instance's own size stay zero
        if capture:
            out["outputs"] = {k: np.array(v) for k, v in {**res, **last_gait}.items()}

        kms = None
        if detail:   # per-kernel device time (CUDA events around each launch) over another `steps` steps, for the roofline entry
            mpc.set_profiling(True)
            kms = {"prepare": 0.0, "condense": 0.0, "ipm": 0.0, "finish": 0.0}
            for _ in range(steps):
                step()
                for k, v in mpc.last_kernel_ms().items():
                    kms[k] += v / steps
            mpc.set_profiling(False)
            refined = [mpc.sizes(b)["refined_iters"] for b in range(0, B, max(1, B // 64))]
            out["mean_refined_iters"] = float(np.mean(refined))
        out["kernel_ms"] = kms

        # end to end through the public call with HOST buffers: H2D of the step's inputs and D2H of its results (status, iteration
        # count, step length, cost AND the decision vector a controller consumes) inside the timed region
        if mode == "closed_loop":       # untimed: the first read-back allocates the pinned staging buffers of the decision vectors
            mpc.download(z_out=z_host)
        else:
            mpc.GetRealTimeUpdate(st, t0, ee, z_out=z_host)
        barrier()
        t_start = time.perf_counter()
        for _ in range(steps):
            if mode == "closed_loop":   # the plant lives on the device: no inputs travel, the per-scenario results do
                mpc.advance_plant(dt_plant)
                mpc.solve_resident()
                res2 = mpc.download(z_out=z_host)
            else:
                res2 = mpc.GetRealTimeUpdate(st, t0, ee, z_out=z_host)
                if mode == "gait":
                    gait_tail()
        mpc.synchronize()
        e2e_s = time.perf_counter() - t_start
        barrier()
        zs = z_host[res2["status"] == 0]
        assert np.all(np.isfinite(zs)) and (len(zs) == 0 or np.all(np.abs(zs).max(axis=1) > 0)), "the decision vectors did not come back"
        total = scenarios if mode == "closed_loop" else B * world
        status = res["status"].astype(np.int32)
        if world > 1:
            ms_dev, e2e_s = sharding.max_over_ranks([ms_dev, e2e_s], dist, "cuda")
            # the only data-path collective: gather of the per-instance results (status) at the end of the batch
            status = sharding.gather_to_root(status, total, dist, "cuda")
        spi = 1 + (gait_k if mode == "gait" else 0)
        out.update({"ms_dev": ms_dev, "e2e_s": e2e_s, "total": total, "solves_per_instance": spi,
                    "value": total * spi * steps / (ms_dev * 1e-3), "e2e_value": total * spi * steps / e2e_s,
                    "solved_fraction": (float(np.isin(status, (0, 1)).mean()) if rank == 0 else None),
                    "h2d": 0 if mode == "closed_loop" else B * (13 + 1 + 12) * 8,
                    "d2h": B * (2 * 4 + 2 * 8 + 8 * n_max) + (B * (4 * 12 * 8 + 16 + 4 + gait_k * 12) if mode == "gait" else 0)})
        return out

    main_mode = "closed_loop" if args.closed_loop else ("gait" if args.gait_opt else "solve")
    sampler = ClockSampler(local_rank)
    sampler.start()
    leg = run_leg(args.config, main_mode, args.batch, args.steps, args.warmup, gait_k=args.gait_opt, scenarios=args.scenarios, detail=True,
                  capture=bool(args.dump_outputs))
    clocks = sampler.stop()
    mpc, res, sz, kms, B, N = leg["mpc"], leg["res"], leg["sizes"], leg["kernel_ms"], leg["B"], leg["N"]

    # ---- single-instance latency (BASELINE metric's second half): one MPC, host buffers in, results out, per call
    lat = None
    if rank == 0:
        init = np.asarray(cfg["srb_init"], float)[None]
        one = make_mpc(args.config, 1, init)
        ee1 = wl.EE_NOMINAL[None].copy()
        one.CreateInitialRun(init, ee1)
        z1 = np.zeros((1, 12 * (N + 1) + 160))
        ts = []
        for _ in range(args.latency_solves):
            t = time.perf_counter()
            r1 = one.GetRealTimeUpdate(init, np.zeros(1), ee1, z_out=z1)
            ts.append(1e3 * (time.perf_counter() - t))
        lat = {"p50_ms": float(np.percentile(ts, 50)), "p95_ms": float(np.percentile(ts, 95)), "solves": len(ts),
               "status": int(r1["status"][0]), "ipm_iters": int(r1["iters"][0]),
               "what": "bgg_solve_batch with batch = 1 (host buffers in; status, cost and the decision vector out), wall clock per call"}
        one.close()
    mpc.close()

    # ---- the other GPU configurations of BASELINE.json under the same timing rules (short legs): #3 gait optimisation with 64
    #      candidates, #5 the 65 536-scenario closed-loop sweep cut across the ranks (strong scaling)
    extra = {}
    if main_mode == "solve" and not args.no_extra_configs:
        G3_STEPS, G3_WARM = 6, 3   # the contact times move every step: a few more steps than the solve legs, to average over them
        g3 = run_leg("a1_gait_opt_config", "gait", 64, G3_STEPS, G3_WARM, gait_k=64)
        g3["mpc"].close()
        extra["#3"] = {"workload": "a1_gait_opt_config: N=50, 64 instances per GPU, per step solve + dH/dtheta + contact-time LP + line search over 64 candidates (65 RTI solves per instance)",
                       "value": g3["value"], "unit": UNIT, "scaling": "weak", "steps": G3_STEPS, "warmup": G3_WARM, "ms_per_step": g3["ms_dev"] / G3_STEPS,
                       "gait_steps_per_s": g3["total"] * G3_STEPS / (g3["ms_dev"] * 1e-3), "e2e": g3["e2e_value"],
                       "instances_with_gradient": g3["gait_stats"]["grad_ok"], "solved_fraction_parents": g3["solved_fraction"]}
        C5_STEPS, C5_WARM = 25, 2   # SURVEY 8(d): T = 25 sequential closed-loop ticks -- long enough for the horizon to slide through
        #                              lift-offs and touch-downs (the QP grows from 120 to 148 spline variables and back)
        c5 = run_leg("a1_config_distr_rejection", "closed_loop", 0, C5_STEPS, C5_WARM, scenarios=args.scenarios)
        c5["mpc"].close()
        extra["#5"] = {"workload": f"a1_config_distr_rejection: N=50, {args.scenarios} closed-loop scenarios cut across {world} GPU(s), a step = plant step + RTI solve of every scenario",
                       "value": c5["value"], "unit": UNIT, "scaling": "strong", "steps": C5_STEPS, "warmup": C5_WARM, "ms_per_step": c5["ms_dev"] / C5_STEPS,
                       "e2e": c5["e2e_value"], "solved_fraction": c5["solved_fraction"],
                       "note": "the end-to-end loop continues the same closed loop (the next 25 ticks), where the disturbance has been "
                               "rejected and a solve takes 11-13 iterations instead of 14-17: its figure is not comparable tick for tick"}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")):
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    hbm_peak, peak_src = (peaks.get("hbm_gbs"), "measured") if peaks.get("hbm_gbs") else (6650.0, "fallback")
    alg_bytes = B * ipm_algorithmic_bytes(N, sz["nu"], sz["n_samples"], sz["n_eebox"], sz["n_eq"])
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ipm_dram_bytes_per_launch.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f)
    mean_iters = float(np.mean(res["iters"]))
    flops = B * ipm_algorithmic_flops(N, sz["nu"], sz["nf"], sz["n_samples"], mean_iters, leg["mean_refined_iters"])
    try:
        fp64_peak, fp64_src = bg.measure_fp64_peak(local_rank), "measured in this run: register-resident FP64 FMA chains (bgg_measure_fp64_peak)"
    except Exception as e:  # noqa: BLE001
        fp64_peak, fp64_src = 37.0, f"fallback, nominal ({e})"
    tf = flops / (kms["ipm"] * 1e-3) / 1e12
    line = {
        "metric": METRIC, "value": leg["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": leg["ms_dev"] / args.steps, "higher_is_better": True, "scaling": "strong" if args.closed_loop else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload, "decision_vars": sz["n"], "spline_vars": sz["nu"],
                   "ineq_rows": sz["m_ineq"], "eq_rows": 12 * (N + 1) + sz["n_eq"],
                   "qp_solver": "interior point (homogeneous self-dual embedding, Clarabel's algorithm), tolerances 1e-8",
                   "l2": "inputs larger than L2 (instance + workspace state is > 1 GB per 4096 instances)",
                   "solved_fraction": leg["solved_fraction"], "mean_ipm_iters": mean_iters, "mean_refined_iters": leg["mean_refined_iters"]},
        "clocks": clocks,
        "e2e": {"value": leg["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": leg["h2d"], "d2h_bytes_per_step": leg["d2h"],
                "timing": "wall clock around the host-buffer call (bgg_solve_batch: inputs up, status / iterations / step length / cost and "
                          "the decision vector of every instance back), synchronised both sides"},
        "gpu_launches": int(leg["launches"]),
        "gait_opt": ({"candidates": args.gait_opt, "instances_with_gradient": leg["gait_stats"]["grad_ok"],
                      "argmin_histogram": leg["gait_stats"]["best_hist"].tolist(),
                      "gait_steps_per_s": leg["total"] * args.steps / (leg["ms_dev"] * 1e-3)} if args.gait_opt else None),
        "kernel_ms": kms,
        "latency": lat,
        # the bound that binds: k_ipm keeps its QP in shared memory for the ~17 iterations of a solve, HBM sees only the
        # compulsory inputs and outputs (secondary entry below)
        "roofline": {"kernel": "k_ipm", "bound": "fp64", "achieved": tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac": tf / fp64_peak,
                     "traffic": (traffic or {}).get("dram_bytes_per_launch"),
                     "traffic_source": (traffic or {}).get("source", "none: no ncu capture of this build committed"),
                     "peak_source": fp64_src,
                     "flops_per_launch": flops, "kernel_share_of_step": kms["ipm"] / sum(kms.values()),
                     "hbm": {"achieved": alg_bytes / (kms["ipm"] * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": alg_bytes / (kms["ipm"] * 1e-3) / 1e9 / hbm_peak, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": alg_bytes}},
        "configs": extra or None,
    }
    if world == 1:
        sample = args.cpu_sample or 8 * cores
        v, el = oracle_throughput(args.config, sample, 20, 2, cores)
        p50, p95 = oracle_latency(args.config, 30)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                "what": "restated reference algorithm (same assembly, Clarabel's interior-point algorithm with an envelope LDL'); "
                                        "not the reference binary, which needs Eigen / pinocchio / Clarabel (absent here)",
                                "sample": f"{sample} instances of the same synthetic workload x 20 RTI solves (2 warm-up) on {cores} threads, {el:.1f} s",
                                "latency_p50_ms": p50, "latency_p95_ms": p95}
    if args.dump_outputs:
        dump_outputs(leg["outputs"], args.dump_outputs)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
