#!/usr/bin/env python
"""bench.py -- dual-simplex iterations/sec (and wall-to-optimal) of the B200 engine on BASELINE.json's workloads.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c2|c3|small]
                  [--dump-outputs DIR]

Workloads
  N = 1 (default c2): BASELINE.json configs[1] -- synthetic random LP m=10k n=100k 1% nnz, fp64, dual
      steepest edge, no presolve / scaling / perturbation.  A *step* is one factorization cycle of the
      hot path: `cycle` = 550 dual simplex iterations (twice the reference's default interval) plus the
      refactorization + recompute that ends the cycle.  The timed window starts from a mid-solve basis (tests/golden/c2_status_it12000.npz:
      the basis the CPU oracle reaches after 12 000 iterations) so that the nucleus of the basis has a
      representative size.  The line also carries C2's objective after the window and `wall_to_optimal_s`
      of the same generator at 3 000 x 30 000 (C2 itself needs > 10^6 iterations, see DESIGN.md section 11).
  N > 1 (default c3): BASELINE.json configs[2] -- m=50k n=500k 1% nnz (2.5e8 nonzeros), the size
      north_star assigns to several GPUs.  One process per GPU; the matrix is column-sharded for the
      pricing pass and the factors (rows of the nucleus inverse, rows of the eta panel) are row-sharded;
      every rank holds the same m-vectors after ONE in-place NCCL all-gather per solve / pricing pass.
      A step is half a factorization cycle (541 iterations; one refactorization per two steps).  `python bench.py --gpus 1 --workload c3` measures the
      same workload on one GPU (profiles/ holds that line; quoted in `strong_scaling_reference`).
  Inputs are larger than L2 (CSC copy of A >= 120 MB + factors), no L2 flush is needed.

W warm-up steps run untimed, then exactly K steps are timed with CUDA events on the engine's stream
(max over ranks).

--dump-outputs DIR writes what the timed call hands its caller after the last timed step -- primal and
dual column / row solutions, the status array and the objective -- as DIR/<name>.npy (rank 0).  The
inputs are generated from fixed seeds and start from a committed basis, so two builds run with the
same arguments can be compared output for output.

--impl reference times the reference's CPU implementation of the path.  coin-or/Clp cannot be built
here (its CoinUtils dependency is absent), so the arm runs the CPU restatement in oracle/
("kind": "port") on all host cores on the same workload, window and configuration; each step is a
bounded sample (25 iterations) of the factorization cycle, refactorizing at the reference's own
default frequency.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (m, n, density, seed, generator)
    "c2": (10000, 100000, 0.01, 20260923, "random_sparse_lp"),
    "c3": (50000, 500000, 0.01, 20260924, "random_sparse_lp_large"),
    "small": (1000, 10000, 0.01, 20260923, "random_sparse_lp"),
}
REF_ITERS_PER_STEP = 25


def clp_default_frequency(m):
    # ClpSimplex::defaultFactorizationFrequency (src/ClpSimplex.cpp:11401-11431)
    return min(10000, 75 + m // 50 if m < 10000 else 75 + 200 + (m - 10000) // 150)


def default_cycle(m):
    # Engine::setupDevice (clp_b200/csrc/engine.cu): twice Clp's default, capped at 2048
    return max(8, min(2048, 2 * clp_default_frequency(m)))


def step_iterations(name, cycle):
    return cycle // 2 if name == "c3" else cycle


def build_workload(name, local_rank=0):
    """Returns (lp, start status or None, description of the start).  The c3 matrix (4 GB of host
    arrays) is generated once per node by local rank 0 and shared through /dev/shm."""
    from clp_b200 import generators as G

    m, n, dens, seed, gen = WORKLOADS[name]
    if name == "c3":
        shm = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
        path = os.path.join(shm, f"clpb_{name}_{m}x{n}_{seed}.npz")
        if not os.path.exists(path):
            if local_rank == 0:
                lp = getattr(G, gen)(m, n, dens, seed, name=f"rand-{m}x{n}")
                tmp = path + f".tmp{os.getpid()}.npz"
                np.savez(tmp, name=lp.name, m=lp.m, n=lp.n, col_start=lp.col_start, row_index=lp.row_index,
                         element=lp.element, col_lower=lp.col_lower, col_upper=lp.col_upper,
                         objective=lp.objective, row_lower=lp.row_lower, row_upper=lp.row_upper,
                         known_objective=lp.known_objective, expect_status=0)
                os.replace(tmp, path)
            else:
                t0 = time.time()
                while not os.path.exists(path):
                    time.sleep(1.0)
                    if time.time() - t0 > 1200:
                        raise SystemExit("bench.py: timed out waiting for the shared c3 matrix")
        lp = G.LP.load(path)
    else:
        lp = getattr(G, gen)(m, n, dens, seed, name=f"rand-{m}x{n}")
    status, start = None, "all-slack basis"
    fx = os.path.join(ROOT, "tests", "golden", f"{name}_status.npz")
    if name == "c2":
        fx = os.path.join(ROOT, "tests", "golden", "c2_status_it12000.npz")
    if os.path.exists(fx):
        z = np.load(fx)
        status = z["status"].astype(np.uint8)
        who = "CPU oracle" if name == "c2" else "GPU engine"
        start = f"basis of the {who} after {int(z['iterations'])} iterations (tests/golden/{os.path.basename(fx)})"
    return lp, status, start


def workload_config(name, lp, start, cycle, world):
    """The `config` object -- identical for the b200 arm and the reference arm of the same run."""
    si = step_iterations(name, cycle)
    step = (f"{cycle} iterations + 1 refactorization" if si == cycle
            else f"{si} iterations (1 refactorization per {cycle} iterations)")
    return {"workload": lp.name, "m": lp.m, "n": lp.n, "nnz": lp.nnz, "start": start, "step": step,
            "pricing": "dual steepest edge", "presolve": "off", "scaling": "off", "perturbation": "off",
            "l2": "inputs larger than L2 (CSC copy >= 120 MB + factors), no flush",
            "parallelism": "single GPU" if world == 1 else
            f"{world} GPUs: column-sharded pricing, row-sharded factors, one all-gather per solve / pricing pass"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.lines, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (copy, of measured)"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def oracle_sample(lp, status, cores, warm_iters, total_iters=None, seconds=None):
    """The oracle port on the host cores over a bounded sample of the window; returns
    (iterations/s, iterations, seconds, refactorizations, split)."""
    from oracle.oracle import OracleSimplex

    o = OracleSimplex(lp)
    if status is not None:
        o.set_status(status)
    o.set_option("threads", cores)
    o.set_option("factorizationFrequency", clp_default_frequency(lp.m))  # the reference's own cadence
    o.set_option("warmupIterations", warm_iters)
    if total_iters is not None:
        o.set_option("maximumIterations", total_iters)
    if seconds is not None:
        o.set_option("maximumSeconds", seconds)
    o.dual()
    sec, its = o.timed_window()
    return (its / sec if sec > 0 else 0.0), its, sec, o.refactorizations


def highs_line(lp, seconds, status=None):
    """External sanity line (BASELINE.md section 2): HiGHS serial dual simplex on the same LP for a bounded
    time -- different code, same algorithm class -- from its own slack start, or (status given) from the
    window's start basis.  None when the module is absent."""
    try:
        from scipy.optimize._highspy import _core as hp
    except Exception:
        return None
    try:
        h = hp._Highs()
        for k, v in (("output_flag", False), ("solver", "simplex"), ("simplex_strategy", 1), ("presolve", "off"),
                     ("threads", 1), ("time_limit", float(seconds))):
            h.setOptionValue(k, v)
        inf = hp.kHighsInf

        def cl(v):
            v = np.array(v, dtype=float)
            v[v >= 1e29] = inf
            v[v <= -1e29] = -inf
            return v
        L = hp.HighsLp()
        L.num_col_, L.num_row_ = lp.n, lp.m
        L.col_cost_ = np.asarray(lp.objective, float)
        L.col_lower_, L.col_upper_ = cl(lp.col_lower), cl(lp.col_upper)
        L.row_lower_, L.row_upper_ = cl(lp.row_lower), cl(lp.row_upper)
        L.a_matrix_.format_ = hp.MatrixFormat.kColwise
        L.a_matrix_.start_ = np.asarray(lp.col_start, np.int32)
        L.a_matrix_.index_ = np.asarray(lp.row_index, np.int32)
        L.a_matrix_.value_ = np.asarray(lp.element, float)
        h.passModel(L)
        where = "its own all-slack start"
        if status is not None:
            S = hp.HighsBasisStatus  # ClpSimplex::Status -> HighsBasisStatus
            mp = {0: S.kZero, 1: S.kBasic, 2: S.kUpper, 3: S.kLower, 4: S.kNonbasic, 5: S.kLower}
            st = np.asarray(status)
            basis = hp.HighsBasis()
            basis.col_status = [mp[int(x)] for x in st[:lp.n]]
            basis.row_status = [mp[int(x)] for x in st[lp.n:]]
            basis.valid = True
            h.setBasis(basis)
            where = "the window's start basis (its first factorization is inside the time)"
        t = time.perf_counter()
        h.run()
        dt = time.perf_counter() - t
        info = h.getInfo()
        its = int(info.simplex_iteration_count)
        return {"value": its / dt if dt > 0 else 0.0, "unit": "iterations/s", "cores": 1,
                "kind": "highs-ds" if status is None else "highs-ds-window",
                "sample": f"HiGHS {getattr(hp, 'HIGHS_VERSION_MAJOR', '')} serial dual simplex, presolve off, from {where}: "
                          f"{its} iterations in {dt:.1f} s (time limit {seconds:.0f} s), "
                          f"model status {str(h.getModelStatus()).split('.')[-1]}"}
    except Exception as ex:  # the sanity line must never break the bench
        return {"value": None, "kind": "highs-ds", "sample": f"failed: {ex!r}"}


def highs_line_bounded(lp, seconds, status, wall_limit):
    """highs_line in a forked child with a hard wall-clock limit: HiGHS does not look at its time limit while
    it factorizes a start basis (C2's window basis: > 100 s on 8 cores), and the bench must stay bounded."""
    import multiprocessing as mp

    try:
        ctx = mp.get_context("fork")
        parent, child = ctx.Pipe(duplex=False)

        def work(conn):
            conn.send(highs_line(lp, seconds, status))
            conn.close()
        p = ctx.Process(target=work, args=(child,), daemon=True)
        t0 = time.perf_counter()
        p.start()
        child.close()
        if parent.poll(wall_limit):
            res = parent.recv()
            p.join(5)
            return res
        p.kill()  # exactly the child started above
        p.join(5)
        return {"value": 0.0, "unit": "iterations/s", "cores": 1, "kind": "highs-ds-window",
                "sample": f"HiGHS serial dual simplex from the window's start basis: no iteration within the hard limit of "
                          f"{time.perf_counter() - t0:.0f} s (still in its first factorization)"}
    except Exception as ex:
        return {"value": None, "kind": "highs-ds-window", "sample": f"failed: {ex!r}"}


def clp_probe():
    """Run-time probe for a real Clp on the measurement box (BASELINE.md section 2 line 1)."""
    exe = shutil.which("clp")
    lib = None
    try:
        import ctypes.util

        lib = ctypes.util.find_library("Clp")
    except Exception:
        pass
    return {"clp_binary": exe, "libClp": lib,
            "note": "coin-or/Clp not present on this box" if not (exe or lib) else "present (not timed: no MPS hand-off wired)"}


def run_reference(args, name, lp, status, start, cycle):
    """CPU arm: the oracle port on all host cores; rank 0 only."""
    cores = os.cpu_count() or 1
    note = ""
    if name == "c3":
        status = None  # the port cannot factorize the window's basis (13k structurals) in bounded time
        note = "; sampled from the all-slack basis (the CPU port needs minutes to factorize the configured start basis)"
    value, its, sec, nref = oracle_sample(lp, status, cores, args.warmup * REF_ITERS_PER_STEP,
                                          total_iters=(args.warmup + args.steps) * REF_ITERS_PER_STEP)
    sample = (f"{its} iterations ({args.steps} steps x {REF_ITERS_PER_STEP}) of the same window, after "
              f"{args.warmup * REF_ITERS_PER_STEP} warm-up iterations, refactorizing at the reference's default "
              f"frequency ({clp_default_frequency(lp.m)}; {nref} refactorizations in the run); oracle/ port of Clp's dual "
              f"path, {cores} threads in price, LU solves serial{note}")
    return {
        "metric": "dual_simplex_iterations_per_sec", "value": value, "unit": "iterations/s",
        "impl": "reference", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * sec / max(1, args.steps), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(name, lp, start, cycle, args.gpus),
        "sample": f"each step is a bounded sample of {REF_ITERS_PER_STEP} iterations of the configured step",
        "cpu_baseline": {"value": value, "unit": "iterations/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def dump_outputs(path, s):
    """The arrays a caller of the timed dual() receives, in float64 (status codes in float32): 2.2 MB at
    c2 and 11 MB at c3, so every entry is written."""
    os.makedirs(path, exist_ok=True)
    outputs = {"primalColumnSolution": s.primalColumnSolution(), "primalRowSolution": s.primalRowSolution(),
               "dualColumnSolution": s.dualColumnSolution(), "dualRowSolution": s.dualRowSolution(),
               "statusArray": s.statusArray().astype(np.float32),
               "objectiveValue": np.array([s.objectiveValue()], dtype=np.float64)}
    for name, a in outputs.items():
        np.save(os.path.join(path, name + ".npy"), a)


def _claim_stdout():
    """Rank 0 must print exactly ONE JSON line: park the real stdout and point fd 1 at stderr, so that
    library banners (NCCL prints its version to stdout) cannot precede or follow the line."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, "w")


def main():
    out = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--no-optimal", action="store_true", help="skip the solve-to-optimality leg (N=1, c2)")
    ap.add_argument("--save-status", default=None, help="write the status array after the run (fixture generation)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the outputs of the timed call after its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b200 path; the reference arm only samples the window")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else max(args.warmup, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    name = args.workload or ("c2" if max(world, args.gpus) == 1 else "c3")

    m = WORKLOADS[name][0]
    cycle = default_cycle(m)
    step_its = step_iterations(name, cycle)

    if args.impl == "reference":
        if rank != 0:
            return 0
        lp, status, start = build_workload(name, 0)
        print(json.dumps(run_reference(args, name, lp, status, start, cycle)), file=out, flush=True)
        return 0

    os.environ.setdefault("NCCL_DEBUG", "WARN")  # NCCL's version banner would go to stdout
    import torch

    import clp_b200

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (clp_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lp, status, start = build_workload(name, local_rank)

    def new_model(**params):
        s = clp_b200.ClpSimplex()
        model_lp = params.pop("_lp", None)
        s.loadLP(model_lp if model_lp is not None else lp)
        if model_lp is None and status is not None and not params.pop("_from_slack", False):
            s.copyinStatus(status)
        params.pop("_from_slack", None)
        single = params.pop("_single", False)
        for k, v in params.items():
            s.setParameter(k, v)
        if world > 1 and not single:
            from clp_b200.sharding import broadcast_unique_id

            uid = clp_b200.ClpSimplex.ncclUniqueId() if rank == 0 else np.zeros(128, dtype=np.uint8)
            uid = broadcast_unique_id(uid, src=0)
            s.initSharding(rank, world, uid)
        return s

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    W, K = args.warmup, args.steps
    nm = lp.n + lp.m
    # ---------------- device-timed run: inputs resident in HBM before the window opens.  The same
    # call is also the end-to-end measurement at N > 1 (host buffers in, solution read back).
    barrier()
    t_e2e = time.perf_counter()
    s = new_model(batch=args.batch, warmupIterations=W * step_its, maximumIterations=(W + K) * step_its,
                  factorizationFrequency=cycle)
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    st = s.dual()
    barrier()
    clocks = sampler.stop()
    s.primalColumnSolution(); s.dualRowSolution(); s.statusArray(); s.objectiveValue()
    wall_e2e = time.perf_counter() - t_e2e
    ms, its = s.timedWindow()
    if dist is not None:
        t = torch.tensor([ms, wall_e2e], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, wall_e2e = float(t[0].item()), float(t[1].item())
    value = its / (ms / 1000.0) if ms > 0 else 0.0
    steps_done = its / step_its
    launches = s.kernelLaunches()
    nucleus = s.nucleusSize()
    if args.save_status and rank == 0:
        np.savez_compressed(args.save_status, status=s.statusArray(), iterations=s.numberIterations())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, s)

    result = {
        "metric": "dual_simplex_iterations_per_sec", "value": value, "unit": "iterations/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / max(1e-9, steps_done),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": workload_config(name, lp, start, cycle, world),
        "timed_iterations": its, "status_after_window": st, "nucleus_size": nucleus,
        "refactorizations": s.numberRefactorizations(),
        "clocks": clocks, "gpu_launches": int(launches),
    }
    h2d = (4 * (lp.n + 1) + 12 * lp.nnz) + (4 * (lp.m + 1) + 12 * lp.nnz) + 8 * 7 * nm + nm + 12 * lp.m
    d2h = 8 * 2 * nm + 8 * lp.m + nm + 4 * lp.m
    if world > 1:
        total_steps = max(1.0, s.numberIterations() / step_its)
        result["e2e"] = {"value": s.numberIterations() / wall_e2e, "unit": "iterations/s",
                         "h2d_bytes_per_step": int(h2d / total_steps), "d2h_bytes_per_step": int(d2h / total_steps),
                         "includes": "per rank: Clpb_loadProblem (pageable host arrays -> HBM), NCCL communicator set-up, "
                                     "basis hand-over, Clpb_dual for W+K steps, solution read-back; max over ranks",
                         "wall_s": wall_e2e, "iterations": s.numberIterations()}
        ref = os.path.join(ROOT, "profiles", f"r2_bench_{name}_n1.json")
        if os.path.exists(ref):
            try:
                r1 = json.load(open(ref))
                result["strong_scaling_reference"] = {"n1_value": r1["value"], "n1_ms_per_step": r1["ms_per_step"],
                                                      "source": f"profiles/r2_bench_{name}_n1.json (python bench.py --gpus 1 --workload {name})",
                                                      "speedup_vs_n1": value / r1["value"] if r1["value"] else None}
            except Exception:
                pass

    if world > 1:
        # ---------------- parity of the sharded path inside the scaling run itself: a small LP of the same
        # family solved (a) by all ranks with every shard forced on (pricing columns, GEMV rows, eta panel
        # rows, inverse columns) and (b) by rank 0 alone on one GPU; all ranks must take the same pivots and
        # both must end at the planted optimum
        try:
            from clp_b200 import generators as G

            plp = G.random_sparse_lp(1500, 20000, 0.01, 31, name="rand-1500x20000")
            a = new_model(_lp=plp, shardMinNnzPerRank=0, shardPanel=1)
            ast = a.dual()
            mine = {"rank": rank, "status": ast, "objective": a.objectiveValue(), "iterations": a.numberIterations()}
            everyone = [None] * world
            dist.all_gather_object(everyone, mine)
            if rank == 0:
                b1 = new_model(_lp=plp, _single=True)
                bst = b1.dual()
                tol = 1e-8 * (1.0 + abs(plp.known_objective))
                result["sharded_parity"] = {
                    "workload": plp.name, "ranks": everyone,
                    "ranks_identical": all(e["objective"] == everyone[0]["objective"] and e["iterations"] == everyone[0]["iterations"]
                                           and e["status"] == everyone[0]["status"] for e in everyone),
                    "single_gpu": {"status": bst, "objective": b1.objectiveValue(), "iterations": b1.numberIterations()},
                    "planted_objective": plp.known_objective,
                    "ok": bool(ast == 0 and bst == 0 and abs(everyone[0]["objective"] - plp.known_objective) <= tol
                               and abs(b1.objectiveValue() - plp.known_objective) <= tol)}
                del b1
            del a
        except Exception as ex:  # the parity leg must never cost the bench line
            if rank == 0:
                result["sharded_parity"] = {"ok": False, "error": repr(ex)}

    if rank == 0 and world == 1:
        # ---------------- per-kernel timing (CUDA events around single kernels, no graph replay)
        # one full factorization cycle, so that the eta-panel costs (which grow with the number of
        # updates since the last refactorization) are averaged the way the timed window sees them
        p = new_model(batch=16, timing=1, maximumIterations=cycle, factorizationFrequency=cycle)
        p.dual()
        ph = p.phaseTimes()
        ns = max(1.0, ph["samples"])
        k = p.nucleusSize()
        peak, peak_src = measured_peak_gbs()
        nb = max(1, int((np.asarray(status) == 1)[: lp.n].sum())) if status is not None else 0
        kern = {
            # algorithmic bytes per launch (DESIGN.md "Roofline accounting")
            "price": (12.0 * lp.nnz + 4.0 * (lp.n + 1) + 1.0 * lp.n + 8.0 * lp.m + 8.0 * lp.n, ph["priceKernel"] / ns),
            # mean over the timed launches: the nucleus size changes when the accuracy gate forces a
            # refactorization inside the cycle
            "ftran_gemv": (ph["ftranGemvBytes"] / ns, ph["ftranGemv"] / ns),
            "btran_gemv": (ph["btranGemvBytes"] / ns, ph["btranGemv"] / ns),
        }
        dom = max(kern, key=lambda q: kern[q][1])
        b, t_ms = kern[dom]
        ach = b / (t_ms * 1e-3) / 1e9 if t_ms > 0 else 0.0
        # DRAM bytes per launch of that kernel from the committed ncu --set full capture (same
        # workload, same nucleus size); null when the nucleus differs from the captured one
        traffic, traffic_src, capture = None, None, None
        for tp in ("r2_ncu_traffic.json", "r1_ncu_traffic.json"):
            tp = os.path.join(ROOT, "profiles", tp)
            if not os.path.exists(tp):
                continue
            rec = json.load(open(tp)).get(dom)
            if rec:
                kc = int(rec.get("nucleus_size", 0))
                cap = {"price": kern["price"][0], "ftran_gemv": 8.0 * kc * ((kc + 7) // 8 * 8) + 48.0 * kc,
                       "btran_gemv": 8.0 * kc * ((kc + 7) // 8 * 8) + 16.0 * kc}[dom]
                # reported as roofline.traffic only when this run's launches have the size of the
                # captured one; otherwise the capture is quoted separately (traffic_capture)
                if abs(b - cap) <= 0.005 * cap:
                    traffic, traffic_src = rec["traffic"], rec["source"]
                capture = {"nucleus_size": kc, "algorithmic_bytes": cap, "traffic": rec["traffic"],
                           "traffic_over_algorithmic": rec["traffic"] / cap, "source": rec["source"]}
                break
        result["roofline"] = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                              "frac": ach / peak, "frac_of_nominal_8TBps": ach / 8000.0, "traffic": traffic,
                              "traffic_source": traffic_src,
                              "traffic_capture": capture,
                              "peak_source": peak_src,
                              "bytes_per_launch": b, "ms_per_launch": t_ms, "nucleus_size": k,
                              "all": {q: {"bytes": v[0], "ms": v[1], "GBps": (v[0] / (v[1] * 1e-3) / 1e9 if v[1] > 0 else 0.0),
                                          "frac": (v[0] / (v[1] * 1e-3) / 1e9 / peak if v[1] > 0 else 0.0)}
                                      for q, v in kern.items()},
                              "phase_us_per_iteration": {q: 1000.0 * ph[q] / ns for q in
                                                         ("chuzr", "btran", "price", "chuzc", "dualUpdate", "ftran", "update")},
                              "refactor_ms_total": ph["refactor"], "basic_structurals_at_start": nb}
        del p
        # ---------------- end to end through the C ABI with host buffers
        # the problem is uploaded once per solve, so the copies are amortised over the K steps of the call
        t0 = time.perf_counter()
        e = new_model(batch=args.batch, maximumIterations=K * step_its, factorizationFrequency=cycle)
        e.dual()
        e.primalColumnSolution(); e.dualRowSolution(); e.statusArray(); e.objectiveValue()
        wall = time.perf_counter() - t0
        result["e2e"] = {"value": e.numberIterations() / wall, "unit": "iterations/s",
                         "h2d_bytes_per_step": int(h2d / max(1, K)), "d2h_bytes_per_step": int(d2h / max(1, K)),
                         "includes": "Clpb_loadProblem (pageable host arrays -> HBM), basis hand-over, "
                                     "Clpb_dual for K steps, solution read-back", "wall_s": wall,
                         "iterations": e.numberIterations()}
        del e
        # ---------------- wall-to-optimal (the other half of BASELINE.json's metric).  C2 itself approaches
        # its planted optimum only asymptotically (-25 534 after 8.4e5 iterations / 400 s against -25 267.64,
        # profiles/r2_fullsize.json; HiGHS serial: 1e4 iterations in 3000 s), far beyond a bench run: the
        # line carries C2's objective after the timed window, and the wall-to-optimal of the SAME generator
        # at 3 000 x 30 000 solved from the all-slack basis through the public API (host buffers in,
        # solution out), checked against the planted optimum c^T x* the generator certifies
        result["objective_after_window"] = {"objective": s.objectiveValue(), "planted_objective": lp.known_objective,
                                            "iterations_from_start_basis": s.numberIterations()}
        try:
            if name in ("c2", "small") and not args.no_optimal:
                from clp_b200 import generators as G
                from oracle.oracle import kkt_violations  # checker only, outside every timed region

                olp = G.random_sparse_lp(3000, 30000, 0.01, 20260923, name="rand-3000x30000")
                t0 = time.perf_counter()
                f = clp_b200.ClpSimplex()
                f.loadLP(olp)
                f.setParameter("batch", args.batch)
                f.setParameter("maximumSeconds", 300)
                fst = f.dual()
                xs = f.primalColumnSolution()
                wall = time.perf_counter() - t0
                rel = abs(f.objectiveValue() - olp.known_objective) / (1.0 + abs(olp.known_objective))
                result["wall_to_optimal_s"] = wall
                result["optimal"] = {"workload": olp.name, "m": olp.m, "n": olp.n, "nnz": olp.nnz,
                                     "status": fst, "objective": f.objectiveValue(), "planted_objective": olp.known_objective,
                                     "rel_diff": rel, "iterations": f.numberIterations(),
                                     "refactorizations": f.numberRefactorizations(), "seconds_in_loop": f.secondsInLoop(),
                                     "iterations_per_sec": f.numberIterations() / max(1e-9, f.secondsInLoop()),
                                     "kkt_violations": int(kkt_violations(olp, xs, f.primalRowSolution(), f.dualColumnSolution())) if fst == 0 else None,
                                     "n_basic": int((f.statusArray() == 1).sum()),
                                     "parity_ok": bool(fst == 0 and rel <= 1e-8),
                                     "includes": "Clpb_loadProblem, Clpb_dual from the all-slack basis to status 0, solution read-back"}
                del f
        except Exception as ex:  # never lose the line to an auxiliary leg
            result["optimal"] = {"parity_ok": False, "error": repr(ex)}
        # ---------------- CPU baselines on the host cores, bounded samples
        try:
            cores = os.cpu_count() or 1
            # at c3 the CPU port needs ~10 minutes for the FIRST factorization of the window's basis (13k
            # structurals, dense tail): its bounded sample starts from the all-slack basis instead
            cpu_status = status if name != "c3" else None
            v, cits, sec, nref = oracle_sample(lp, cpu_status, cores, 5, seconds=args.cpu_seconds)
            where = "of the same window" if cpu_status is not None or status is None else "from the all-slack basis (the window's basis takes the port minutes to factorize)"
            result["cpu_baseline"] = {"value": v, "unit": "iterations/s", "cores": cores, "kind": "port",
                                      "sample": f"first {cits} iterations ({sec:.1f} s) {where} on the host; "
                                                "oracle/ restatement of Clp's dual path (coin-or/Clp itself cannot be "
                                                "built: CoinUtils absent)",
                                      "others": [x for x in (highs_line(lp, args.cpu_seconds),
                                                             highs_line_bounded(lp, args.cpu_seconds, status, 90.0)
                                                             if (status is not None and name == "c2") else None) if x],
                                      "clp_probe": clp_probe()}
        except Exception as ex:
            result["cpu_baseline"] = {"value": None, "unit": "iterations/s", "cores": os.cpu_count() or 1, "kind": "port", "sample": f"failed: {ex!r}"}
    if rank == 0:
        print(json.dumps(result), file=out, flush=True)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
