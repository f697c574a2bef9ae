#!/usr/bin/env python
"""Throughput harness of the NLP-evaluation hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            our arm (one process per GPU under torchrun)
  python bench.py --impl reference --gpus N ...            the reference arm: the CPU oracle ("port" of
                                                           the CasADi evaluation) on the host cores
  python bench.py ... --dump-outputs DIR                   also write the outputs of the last timed step
                                                           (see dump_outputs) as DIR/<name>.npy

A *step* is one evaluation of f, grad_f, g, jac_g and hess_l (what IPOPT requests at an iteration with
an exact Hessian) for every instance of the batch.  Workload at every N: BASELINE config 3,
``humanoid_kinodynamic single step on flat ground``, horizon 30, 1024 randomised instances PER GPU
(weak scaling: instances are sharded by rank, no data-path collective; the per-instance objective is
gathered with one all_gather per step).  Rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HORIZON = 30
INSTANCES_PER_GPU = 1024
METRIC = "knot_evals_per_s"
UNIT = "knot-evals/s (f+grad_f+g+jac_g+hess_l)"
WORKLOAD = "humanoid_kinodynamic single step flat ground (BASELINE config 3), horizon 30, 1024 instances per GPU"
PLANS_PER_GPU = 512  # BASELINE config 4: 4096 instances sharded over 8 GPUs
REFERENCE_BUDGET_S = 150.0  # wall-clock budget of the reference arm's timed + warm-up steps
DUMP_INSTANCES = 64  # instances whose full outputs --dump-outputs writes: 64 x 0.8 MB, under 64 MB in all


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=256, help="instances in the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float64): f of every instance of "
                         f"rank 0's shard, grad_f, g, jac and hess of {DUMP_INSTANCES} of them (dump_rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path; the reference arm keeps none")
    return args


def dump_rows(batch: int):
    """The instances whose grad_f, g, jac and hess --dump-outputs writes: a fixed, seeded, sorted sample of the batch."""
    import numpy as np

    rows = np.random.default_rng(0).choice(batch, min(DUMP_INSTANCES, batch), replace=False)
    return np.sort(rows)


def dump_outputs(out: dict, directory: str) -> None:
    """Write one evaluation's outputs (``KinoEvaluator.eval``'s dict of (B, ...) float64 device tensors) as
    directory/<name>.npy: ``f`` whole, the wider arrays only at the rows of ``dump_rows(B)``."""
    import numpy as np
    import torch

    os.makedirs(directory, exist_ok=True)
    f = out["f"]
    rows = torch.as_tensor(dump_rows(f.shape[0]), device=f.device)
    for name, t in out.items():
        a = t if name == "f" else t.index_select(0, rows)
        np.save(os.path.join(directory, f"{name}.npy"), a.cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1] or [r for (_, r) in self.rows[-3:]]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            c = [v.strip() for v in r.split(",")]
            try:
                sm.append(float(c[0]))
                mx.append(float(c[1]))
            except Exception:
                continue
            for nm, v in zip(names, c[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa_node(local_rank: int, world: int):
    """Pin this rank's threads to the CPUs of the NUMA node its GPU hangs off, so that the pinned host buffers of
    the end-to-end path are allocated (first touch) on that node and the copies of the ranks do not all cross one
    memory controller.  Node from sysfs (PCI device of the GPU); when the platform reports none (-1: a virtualised
    host) and several nodes exist, the ranks are spread evenly over them.  Returns a description for the JSON line."""
    try:
        nodes = sorted(int(d[4:]) for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit())
    except OSError:
        return {"nodes": 0, "bound": None}
    if len(nodes) < 2:
        return {"nodes": len(nodes), "bound": None}
    node = -1
    try:
        import torch

        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id  # type: ignore[attr-defined]
        node = int(open(f"/sys/bus/pci/devices/{str(bus).lower()}/numa_node").read())
    except Exception:  # noqa: BLE001
        node = -1
    how = "sysfs"
    if node < 0:
        node, how = nodes[(local_rank * len(nodes)) // max(world, 1) % len(nodes)], "spread"
    try:
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"nodes": len(nodes), "bound": node, "how": how, "cpus": len(cpus)}
    except Exception as exc:  # noqa: BLE001
        return {"nodes": len(nodes), "bound": None, "error": str(exc)}


def sharded_solves(model, ev, dev, rank, world):
    """Complete interior-point solves with the evaluator in the loop, one wave of instances per GPU: "keep standing"
    OCPs of the bench workload's size built from batched pose-finder solutions (hippopt_b200.workloads), stage-wise
    KKT on the GPU.  Returns (on every rank) the whole-job numbers: solves/s = converged instances of all ranks /
    slowest rank's wall time; results are gathered with one NCCL all_gather."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from hippopt_b200.evaluator import PoseEvaluator
    from hippopt_b200.ipsolver import BatchedInteriorPoint
    from hippopt_b200.workloads import pose_batch, standing_problem

    lay = ev.layout
    try:
        n_s = torch.cuda.get_device_properties(dev).multi_processor_count  # one wave of the LU kernels
        pev = PoseEvaluator(model)
        xq, pq, _, _ = pose_batch(pev.layout, model, n_s, seed=1 + 97 * rank, noise=0.02)
        lbq, ubq = pev.bounds(pq)
        po = BatchedInteriorPoint(pev, tol=1e-8, max_iter=300).solve(torch.tensor(xq, device=dev),
                                                                     torch.tensor(pq, device=dev), lbq, ubq)
        okp = po.success.cpu().numpy()
        pk, x0k = standing_problem(lay, model, po.values.cpu().numpy()[okp])
        lbs_, ubs_ = lay.bounds(pk)
        ip = BatchedInteriorPoint(ev, tol=1e-6, max_iter=150, kkt="stage", delta_c=1e-9, mu_init=1e-3)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        ts = time.perf_counter()
        # end to end: host arrays in (guess, parameters), solution and multipliers back on the host
        out = ip.solve(torch.tensor(x0k).pin_memory().to(dev, non_blocking=True), torch.tensor(pk).pin_memory().to(dev, non_blocking=True),
                       lbs_, ubs_)
        xs, lam = out.values.cpu(), out.constraint_multipliers.cpu()
        torch.cuda.synchronize(dev)
        secs = time.perf_counter() - ts
        mine = torch.tensor([float(okp.sum()), float(out.success.sum()), secs, float(out.iterations[out.success].median()) if
                             bool(out.success.any()) else -1.0, float(out.evaluations), float(ip.kkt_seconds),
                             float(xs.numel() * 8 + lam.numel() * 8), float(x0k.size * 8 + pk.size * 8)],
                            dtype=torch.float64, device=dev)
    except Exception as exc:  # noqa: BLE001 -- a solver failure must not cost the throughput line
        mine = torch.tensor([0.0, 0.0, 1e-9, -1.0, 0.0, 0.0, 0.0, 0.0], dtype=torch.float64, device=dev)
        err = f"{type(exc).__name__}: {exc}"
    else:
        err = None
    # ---- BASELINE config 4 AS POSED: periodic walking step plans, 4096 / 8 = 512 instances per GPU, built like
    # main_periodic_step.py:365-478 (keyframe poses by the pose finder, interpolated guess with the reference's planned
    # force of 100 N per point, mass-normalised as the planner does) and solved with the options the reference hands
    # to IPOPT (:111-134), hessian_approximation = limited-memory included
    plan = torch.zeros(6, dtype=torch.float64, device=dev)
    perr = None
    try:
        from hippopt_b200.evaluator import KinoEvaluator
        from hippopt_b200.initial_guess import periodic_step_guess
        from hippopt_b200.kino_layout import KinoSettings

        n_plans = PLANS_PER_GPU
        ev4 = KinoEvaluator(model, KinoSettings(horizon=HORIZON, final_state_constraint=True, periodicity_constraint=True))
        Ls = np.random.default_rng(5 + rank).uniform(0.1, 0.3, n_plans)
        torch.cuda.synchronize(dev)
        tg = time.perf_counter()
        gs = periodic_step_guess(model, pev, ev4, Ls, force_z=100.0, mass_normalised=True)
        torch.cuda.synchronize(dev)
        t_setup = time.perf_counter() - tg
        lb4, ub4 = ev4.layout.bounds(gs.parameters)
        ref_opts = {"tol": 1e-3, "dual_inf_tol": 1000.0, "compl_inf_tol": 1e-2, "constr_viol_tol": 1e-4,
                    "acceptable_tol": 10, "acceptable_iter": 2, "acceptable_compl_inf_tol": 1000.0,
                    "acceptable_obj_change_tol": 1e0, "nlp_scaling_method": "gradient-based", "max_iter": 400,
                    "hessian_approximation": "limited-memory"}
        ip4 = BatchedInteriorPoint(ev4, kkt="stage", delta_c=1e-9, mu_init=1e-1, ipopt_options=ref_opts)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        tp = time.perf_counter()
        r4 = ip4.solve(gs.x0, torch.tensor(gs.parameters, device=dev), lb4, ub4)
        x4 = r4.values.cpu()
        torch.cuda.synchronize(dev)
        t_plan = time.perf_counter() - tp
        g4 = ev4.eval(4, r4.values, torch.tensor(gs.parameters, device=dev))["g"].cpu().numpy()
        okk = r4.success.cpu().numpy()
        viol = float((np.maximum(lb4 - g4, 0) + np.maximum(g4 - ub4, 0))[okk].max()) if okk.any() else float("nan")
        plan = torch.tensor([float(n_plans), float(okk.sum()), t_plan, float(r4.iterations[r4.success].median()) if okk.any()
                             else -1.0, viol, t_setup], dtype=torch.float64, device=dev)
        del ev4, x4
    except Exception as exc:  # noqa: BLE001
        perr = f"{type(exc).__name__}: {exc}"
    from hippopt_b200.sharding import gather_rank_rows, whole_job_rate

    allr = gather_rank_rows(torch.cat([mine, plan]))
    a = allr.cpu().numpy()
    conv, slow, _ = whole_job_rate(allr, 1, 2)
    pconv, pslow, _ = whole_job_rate(allr, 9, 10)
    periodic = {"workload": f"BASELINE config 4 as posed: periodic walking step plans (step length U(0.1, 0.3) m, horizon {HORIZON}, "
                            f"final-state and periodicity rows), {PLANS_PER_GPU} per GPU, the reference's guess (100 N per point, "
                            f"mass-normalised) and IPOPT options (limited-memory Hessian, tol 1e-3, acceptable_tol 10)",
                "n_gpus": world, "instances": int(a[:, 8].sum()), "converged": int(pconv),
                "seconds_max_over_ranks": pslow, "solves_per_s": pconv / pslow if pslow > 0 else 0.0,
                "iterations_median_per_rank": [float(r[11]) for r in a],
                "constraint_violation_max": float(np.nanmax(a[:, 12])) if np.isfinite(a[:, 12]).any() else None,
                "setup_seconds_max_over_ranks": float(a[:, 13].max()), "error": perr}
    return {"periodic_step_plans": periodic, "workload": f"keep-standing OCPs at the bench size (horizon {HORIZON}, n_x {lay.n_x}, m {lay.m}), one wave of "
                        f"instances per GPU, stage-wise KKT on the batched LU kernels; host guess in, host solution out",
            "n_gpus": world, "instances": int(a[:, 0].sum()), "converged": int(conv), "seconds_max_over_ranks": slow,
            "solves_per_s": conv / slow if slow > 0 else 0.0, "per_rank_solves_per_s": [float(r[1] / r[2]) for r in a],
            "iterations_median_per_rank": [float(r[3]) for r in a], "batched_evaluations_per_rank": [int(r[4]) for r in a],
            "seconds_in_kkt_per_rank": [float(r[5]) for r in a], "h2d_bytes": float(a[:, 7].sum()),
            "d2h_bytes": float(a[:, 6].sum()), "error": err}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def run_reference(args):
    """The reference's own CPU evaluation of the path: CasADi is not installable here, so this is
    the oracle port (oracle/) on all host cores, on a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np

    from hippopt_b200.kino_layout import KinoLayout, KinoSettings
    from hippopt_b200.robot_model import synthetic_ergocub
    from hippopt_b200.workloads import kino_batch
    from oracle.cpu_baseline import OraclePool

    model = synthetic_ergocub()
    lay = KinoLayout(model, KinoSettings(horizon=HORIZON))
    pool = OraclePool(model, HORIZON)
    # --steps K --warmup W are honoured; each step is a BOUNDED SAMPLE of the workload, sized from a probe so that
    # the whole run stays within REFERENCE_BUDGET_S seconds (the contract: "ends within a few minutes")
    steps, warm = max(1, args.steps), max(0, args.warmup)
    xp, pp, lp, sp = kino_batch(lay, model, 16, seed=3)
    pool.step(xp, pp, lp, sp)
    dt_probe, _ = pool.step(xp, pp, lp, sp)
    rate = 16 / max(dt_probe, 1e-6)  # instances per second on this host
    n = int(max(min(8, args.cpu_sample), min(args.cpu_sample, REFERENCE_BUDGET_S * rate / (steps + warm))))
    x, p, lam, sigma = kino_batch(lay, model, n, seed=2)
    for _ in range(warm):
        pool.step(x, p, lam, sigma)
    t = 0.0
    for _ in range(steps):
        dt, ke = pool.step(x, p, lam, sigma)
        t += dt
    pool.close()
    value = steps * n * HORIZON / t
    sample = (f"{n} of the {INSTANCES_PER_GPU} instances x {HORIZON} knots per step ({steps} timed steps, {warm} warm-up); "
              f"{pool.description}")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": 1e3 * t / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "horizon": HORIZON, "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": pool.cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "CasADi/IPOPT are not installable offline; this is the repo's CPU oracle (an SX virtual machine "
                "restating CasADi's evaluation scheme, forward-mode sweeps for the derivatives), a stand-in CPU "
                "baseline, not CasADi",
    }
    print(json.dumps(line))


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    import numpy as np
    import torch
    import torch.distributed as dist

    import __graft_entry__ as entry
    from hippopt_b200.evaluator import ALL, HostPipeline, KinoEvaluator, probe_fp64_tflops
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.robot_model import synthetic_ergocub
    from hippopt_b200.sharding import gather_instances, shard_range
    from hippopt_b200.workloads import kino_batch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank, world)  # before any pinned allocation (first-touch placement)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep NCCL's version banner off stdout: ONE JSON line
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    if rank == 0:
        entry.build()
    if world > 1:
        dist.barrier()

    model = synthetic_ergocub()
    ev = KinoEvaluator(model, KinoSettings(horizon=HORIZON))
    lay = ev.layout
    total_instances = INSTANCES_PER_GPU * world
    lo, hi = shard_range(total_instances, rank, world)
    B = hi - lo
    # two rotating input sets; every step also streams ~1 GB of outputs, far beyond the 126 MB L2
    sets = []
    for s in range(2):
        x, p, lam, sigma = kino_batch(lay, model, B, seed=2 + 1000 * s + rank)
        sets.append(tuple(torch.tensor(a, device=dev) for a in (x, p, lam, sigma)))
    host = sets[0]

    def step(i):
        X, P, L, S = sets[i % 2]
        out = ev.eval(ALL, X, P, L, S)
        if world > 1:
            gather_instances(out["f"], total_instances)
        return out

    def fence():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for i in range(max(args.warmup, 3)):
        step(i)
    fence()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.15)
    fence()
    ev.profile(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for i in range(args.steps):
        last = step(i)
    e1.record()
    fence()
    t1 = time.perf_counter()
    ms_total = e0.elapsed_time(e1)
    launches_per_step = ev.last_launch_count()  # kernels one hb_eval of the timed region enqueued
    kernel_ms, n_evals = ev.profile_read()
    ev.profile(False)
    if args.dump_outputs and rank == 0:
        # now, while `last` still holds the timed step's values: ev.eval reuses its output buffers
        dump_outputs(last, args.dump_outputs)
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / args.steps
    value = total_instances * HORIZON / (ms_per_step * 1e-3)

    # ---- end-to-end through the host-buffer API (what a CPU-side IPOPT would call)
    pipe = HostPipeline(ev, B, ALL)
    xh, ph, lh, sh = (a.cpu().pin_memory() for a in host)
    pipe.set_parameters(ph)
    for _ in range(2):
        pipe.run(xh, lh, sh)
    fence()
    e2e_steps = max(3, min(args.steps, 10))
    te = time.perf_counter()
    for _ in range(e2e_steps):
        res = pipe.run(xh, lh, sh)
    fence()
    e2e_s = torch.tensor([(time.perf_counter() - te) / e2e_steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = total_instances * HORIZON / float(e2e_s.item())
    checksum = float(res["f"].sum())
    e2e_h2d, e2e_d2h = pipe.h2d_bytes, pipe.d2h_bytes
    del pipe
    # the same call with the mask IPOPT uses in the reference's own configuration of these planners
    # (hessian_approximation = limited-memory, main_single_step_flat_ground.py:112): f, grad_f, g, jac_g
    from hippopt_b200.evaluator import F, G, GRAD_F, JAC_G

    pipe1 = HostPipeline(ev, B, F | GRAD_F | G | JAC_G)
    pipe1.set_parameters(ph)
    for _ in range(2):
        pipe1.run(xh)
    fence()
    te = time.perf_counter()
    for _ in range(e2e_steps):
        pipe1.run(xh)
    fence()
    e2e1_s = torch.tensor([(time.perf_counter() - te) / e2e_steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e1_s, op=dist.ReduceOp.MAX)
    e2e_first_order = {"value": total_instances * HORIZON / float(e2e1_s.item()), "unit": "knot-evals/s (f+grad_f+g+jac_g)",
                       "h2d_bytes_per_step": pipe1.h2d_bytes, "d2h_bytes_per_step": pipe1.d2h_bytes,
                       "note": "mask of the reference's own IPOPT configuration (limited-memory Hessian: hess_l is never "
                               "requested)"}
    del pipe1

    # ---- row f1 at every world size (second half of BASELINE.json's metric: "solves/s at 1/2/4/8 B200"): every rank
    # solves its own wave of instances, results are gathered with NCCL
    solves_all = None
    if not args.no_cpu_baseline:
        solves_all = sharded_solves(model, ev, dev, rank, world)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (kinematics: FK + adjoint sweeps for Jacobian and Hessian)
    knot_evals_per_launch = B * HORIZON
    kin_ms = kernel_ms["kinematics"] / max(n_evals, 1)
    hbm_peak, hbm_src = measured_peaks()
    bytes_per_knot = lay.kernel_bytes_per_knot()["kinematics"]
    achieved_gbs = bytes_per_knot * knot_evals_per_launch / (kin_ms * 1e-3) / 1e9
    # fp64 roofline of the same kernel from EXECUTED flops: ncu's predicated-on thread-instruction counters of the
    # committed capture (profiles/ncu_counters.json, written by tools/ncu_counters.py from the ncu CSV of
    # `tools/time_kino.py`), not the oracle's tape count -- that one is kept as "reference_work"
    fp64_peak = probe_fp64_tflops()
    roofline_fp64 = None
    cpath = os.path.join(ROOT, "profiles", "ncu_counters.json")
    traffic = None
    if os.path.exists(cpath):
        prof = json.load(open(cpath))
        kin = prof["kernels"]["kino_kin_kernel<1>"]
        flops_launch = 2.0 * kin["dfma"] + kin["dadd"] + kin["dmul"]
        per_knot = flops_launch / prof["knot_evals_per_launch"]
        ach = per_knot * knot_evals_per_launch / (kin_ms * 1e-3) / 1e12
        sm_clock = (clocks or {}).get("sm_mhz") or 1965.0
        n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
        nominal = n_sm * 64 * 2 * sm_clock * 1e6 / 1e12
        counts_path = os.path.join(ROOT, "profiles", "algorithmic_counts.json")
        ref_work = json.load(open(counts_path))["kinematics_kernel_flops"] if os.path.exists(counts_path) else None
        # an fp64 warp instruction holds its scheduler's issue port for two cycles (64 lanes per SM and clock), every
        # other one for one: the share of issue cycles the kernel's instruction stream needs
        issue_cycles = kin["inst_executed"] + kin["inst_fp64"]
        issue_frac = issue_cycles / (kin["sm_cycles"] * n_sm * 4) if kin.get("sm_cycles") else None
        roofline_fp64 = {
            "bound": "fp64", "kernel": "kino_kin_kernel<true>", "achieved": ach, "peak": fp64_peak, "unit": "TFLOP/s",
            "frac": ach / fp64_peak,
            "peak_source": "measured in this run (hb_probe_fp64_tflops: 8 independent DFMA chains per thread, all SMs)",
            "peak_nominal": nominal, "peak_nominal_source": f"{n_sm} SMs x 64 DFMA/clk x 2 x {sm_clock:.0f} MHz",
            "executed_flops_per_knot_eval": per_knot,
            "flops_source": prof["source"],
            "pipe_fp64_active_pct_ncu": kin.get("fp64_pipe_active_pct"), "issue_active_pct_ncu": kin.get("issue_active_pct"),
            "issue_cycles_needed_frac_ncu": issue_frac,
            "reference_work_flops_per_knot_eval": ref_work,
            "note": "executed = 2 DFMA + DADD + DMUL predicated-on thread instructions (ncu) per knot-eval of the "
                    "committed capture x this run's launch rate; reference_work = operation count of the oracle's "
                    "(CasADi-style) tapes for the same rows, which the tree algorithm does not execute"}
        traffic = kin["dram_read"] + kin["dram_write"]

    # ---- the other BASELINE configs (device-resident, 10 timed steps each; parity cases, not the headline)
    other = None
    if world == 1 and not args.no_cpu_baseline:
        from hippopt_b200.evaluator import PoseEvaluator
        from hippopt_b200.workloads import pose_batch

        def quick(evx, data, knots, name):
            t = [torch.tensor(a, device=dev) for a in data]
            for _ in range(3):
                evx.eval(ALL, *t)
            torch.cuda.synchronize(dev)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(10):
                evx.eval(ALL, *t)
            a1.record()
            torch.cuda.synchronize(dev)
            ms = a0.elapsed_time(a1) / 10
            return {"workload": name, "ms_per_step": ms, "knot_evals_per_s": knots / (ms * 1e-3)}

        other = []
        pev = PoseEvaluator(model)
        other.append(quick(pev, pose_batch(pev.layout, model, 4096, seed=1), 4096,
                           "config 2: humanoid_pose_finder static pose, 4096 instances (1 knot each)"))
        ev4 = KinoEvaluator(model, KinoSettings(horizon=30, final_state_constraint=True, periodicity_constraint=True))
        other.append(quick(ev4, kino_batch(ev4.layout, model, 512, seed=3), 512 * 30,
                           "config 4: periodic walking step, 512-instance shard of 4096, horizon 30"))
        ev5 = KinoEvaluator(model, KinoSettings(horizon=50, terrain="smooth_steps", n_terrain_params=10,
                                                final_state_constraint=True))
        other.append(quick(ev5, kino_batch(ev5.layout, model, 512, seed=4), 512 * 50,
                           "config 5: walking on stairs (two smooth steps, randomised heights), 512-instance shard, horizon 50"))
        del pev, ev4, ev5

    # ---- row f2 (SURVEY 8(f)): the Newton (KKT) system of the same workload, stage-wise on the GPU
    kkt_line = None
    if world == 1 and not args.no_cpu_baseline:
        from hippopt_b200.kkt import StageKKT

        nk = min(B, 2 * torch.cuda.get_device_properties(dev).multi_processor_count)
        lbk, ubk = lay.bounds(host[1][:1].cpu().numpy())
        kkt, eqr, iner = StageKKT.for_evaluator(ev, lbk[0], ubk[0], device=dev)
        vals = ev.eval(ALL, *(a[:nk].contiguous() for a in sets[0]))
        gk = torch.Generator().manual_seed(0)
        sig = (torch.rand((nk, len(iner)), generator=gk, dtype=torch.float64) * 10.0).to(dev)
        dlt = torch.full((nk,), 1e-2, dtype=torch.float64, device=dev)
        rxk = torch.randn((nk, lay.n_x), generator=gk, dtype=torch.float64).to(dev)
        rEk = torch.randn((nk, len(eqr)), generator=gk, dtype=torch.float64).to(dev)
        for _ in range(2):
            torch.cuda.synchronize(dev)
            tk = time.perf_counter()
            kkt.solve(vals["hess"], vals["jac"], sig, dlt, 1e-9, rxk, rEk)
            torch.cuda.synchronize(dev)
            tk = time.perf_counter() - tk
        kkt_line = {"workload": f"Newton system of config 3 (n_x + m_E = {lay.n_x + len(eqr)}), {nk} instances: block-"
                                f"tridiagonal sweep over 30 stage blocks of {kkt.nb}^2, batched LU kernels (csrc/lu.cu)",
                    "ms_per_batched_solve": tk * 1e3, "kkt_solves_per_s": nk / tk}
        del kkt, vals

    # ---- row f1: complete solves with the evaluator in the loop (pose finder here; the "keep standing" OCPs of the
    # bench workload's size are in sharded_solves); informational, failures are reported, not hidden
    solves = None
    if world == 1 and not args.no_cpu_baseline:
        from hippopt_b200.evaluator import PoseEvaluator
        from hippopt_b200.ipsolver import BatchedInteriorPoint
        from hippopt_b200.workloads import pose_batch, standing_problem

        try:
            n_s = torch.cuda.get_device_properties(dev).multi_processor_count  # one wave of the LU kernels
            pev = PoseEvaluator(model)
            xq, pq, _, _ = pose_batch(pev.layout, model, n_s, seed=1, noise=0.02)
            lbq, ubq = pev.bounds(pq)
            torch.cuda.synchronize(dev)
            ts = time.perf_counter()
            po_out = BatchedInteriorPoint(pev, tol=1e-8, max_iter=300).solve(torch.tensor(xq, device=dev),
                                                                             torch.tensor(pq, device=dev), lbq, ubq)
            torch.cuda.synchronize(dev)
            t_pose = time.perf_counter() - ts
            okp = po_out.success.cpu().numpy()
            solves = {"pose_finder": {"instances": n_s, "converged": int(okp.sum()), "solves_per_s": int(okp.sum()) / t_pose,
                                      "iterations_median": int(po_out.iterations.median())},
                      "standing_ocp": "see solves_sharded (reported at every number of GPUs)"}
            # row f3: set-up of periodic-step plans (3 keyframe pose solves per instance + device interpolation of
            # the guess into the decision vector), hippopt_b200/initial_guess.py
            try:
                from hippopt_b200.evaluator import KinoEvaluator
                from hippopt_b200.initial_guess import periodic_step_guess
                from hippopt_b200.kino_layout import KinoSettings

                pev4 = KinoEvaluator(model, KinoSettings(horizon=HORIZON, final_state_constraint=True,
                                                         periodicity_constraint=True))
                Ls = np.random.default_rng(5).uniform(0.1, 0.3, n_s)
                periodic_step_guess(model, pev, pev4, Ls[:8])
                torch.cuda.synchronize(dev)
                ts = time.perf_counter()
                gs = periodic_step_guess(model, pev, pev4, Ls)
                torch.cuda.synchronize(dev)
                t_set = time.perf_counter() - ts
                solves["periodic_step_setup"] = {
                    "workload": f"{n_s} plans of config 4's structure: contact phases, {3 * n_s} keyframe pose solves, guess "
                                f"interpolated on the device into the decision vectors, parameters",
                    "instances": n_s, "keyframe_triples_converged": int(gs.ok.sum()), "setups_per_s": n_s / t_set}
            except Exception as exc:  # noqa: BLE001
                solves["periodic_step_setup"] = {"error": f"{type(exc).__name__}: {exc}"}
        except Exception as exc:  # noqa: BLE001 -- a solver failure must not cost the throughput line
            solves = {"error": f"{type(exc).__name__}: {exc}"}

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle.cpu_baseline import OraclePool

        n = args.cpu_sample
        x, p, lam, sigma = kino_batch(lay, model, n, seed=2)
        pool = OraclePool(model, HORIZON)
        pool.step(x[:8], p[:8], lam[:8], sigma[:8])
        dt, ke = pool.step(x, p, lam, sigma)
        pool.close()
        cpu_baseline = {"value": ke / dt, "unit": UNIT, "cores": pool.cores, "kind": "port",
                        "sample": f"{n} of the {B} instances x {HORIZON} knots, one pass ({dt:.1f} s), "
                                  f"{pool.description}"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "horizon": HORIZON, "instances_per_gpu": B, "n_x": lay.n_x, "m": lay.m,
                   "nnz_jac": lay.nnz_j, "nnz_hess": lay.nnz_h, "parallelism": f"instances sharded over {world} GPU(s)",
                   "l2": "two rotating input sets; each step streams ~1 GB of inputs+outputs (>> 126 MB L2)"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": e2e_h2d,
                "d2h_bytes_per_step": e2e_d2h, "steps": e2e_steps, "numa": numa,
                "path": "hb_eval_host (C ABI, host pointers): pinned host x/lam/sigma -> device, kernels, all five "
                        "outputs -> pinned host; 128-instance chunks over 3 internal streams",
                "checksum_f": checksum},
        "e2e_first_order": e2e_first_order,
        "gpu_launches": launches_per_step * args.steps,
        "kernel_ms_per_step": {k: v / max(n_evals, 1) for k, v in kernel_ms.items()},
        "roofline": {"bound": "hbm", "kernel": "kino_kin_kernel<true>", "achieved": achieved_gbs, "peak": hbm_peak,
                     "unit": "GB/s", "frac": achieved_gbs / hbm_peak, "traffic": traffic, "peak_source": hbm_src,
                     "bytes_per_knot_eval": bytes_per_knot,
                     "note": "the kernel is fp64-FMA bound, not HBM bound: see roofline_fp64"},
        "roofline_fp64": roofline_fp64,
        "cpu_baseline": cpu_baseline,
        "other_configs": other,
        "kkt": kkt_line,
        "solves": solves,
        "solves_sharded": solves_all,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
