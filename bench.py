#!/usr/bin/env python
"""bench.py — throughput of the ARMOUR reach-set / constraint-evaluation hot path on B200.

Workload (BASELINE.json configs[1], SURVEY.md 8d "config 2"): per GPU 1,024 random Kinova Gen3 worlds x 10
obstacles (seed 20261017 + rank), 128 time intervals; a STEP is one batch of Ipopt-style queries: for each
of `--iters` (16) k-iterates, one eval_g + one eval_jac_g for every problem of the batch (metric M2,
"planning iters/s": one unit = one eval_g + eval_jac_g pair on built reach sets).  The reach-set build
(metric M1) is timed separately and reported in the "m1" object, next to the single-problem latency
BASELINE.json targets (< 1 ms for one Kinova planning iteration's build + eval).

  value   : M2 units/s, reach sets, k and outputs resident in HBM (device pointers, CUDA events)
  e2e     : M2 units/s through the C-ABI host-buffer call (armour_batch_eval: pinned k -> device,
            kernel, g and dense Jacobian -> pinned host), copies inside the timed region
  roofline: k_constraints, the only kernel of the timed region; algorithmic bytes per launch = B_eval of
            SURVEY.md 8d from the stored monomial counts of THIS batch
  cpu_baseline / --impl reference: the REFERENCE ITSELF when oracle/_ref/libarmour_ref_cuda.so travelled to the box
            (the reference's own PZsparse / Trajectory / Dynamics / CollisionChecking / NLPclass sources compiled by
            nvcc with its flags against stand-in Eigen / Boost / Ipopt headers: OpenMP host slices on all cores + its
            7 collision-kernel launches and blocking copies per call, exactly what armtd_NLP::eval_g / eval_jac_g do;
            kind "reference"), else the CPU oracle (C++ restatement, kind "port").  One world at a time, like the
            reference; a bounded sample of worlds of the same generator.
  Extra objects of the line (the driver reads them, the headline stays M2): "m1" (builds), "config1_host_abi" (one
  planning iteration through host pointers, eval_g and eval_jac_g called separately like Ipopt does), "solver_e2e"
  (armour_batch_solve, host in/out, beside the CPU planner), "config3" / "config4" (BASELINE configs 3 and 4),
  "sweep" (BASELINE config 5: 65,536-world sweep split over the ranks, strong scaling, per-world verdicts gathered
  over NCCL), "controller" (SURVEY 8f-4: the robust controller's interval Newton-Euler pass and robust input over 2^20
  sampled states, beside the reference's own MEX sources on one host thread), "armtd" (SURVEY 8f-3: the ARMTD comparison
  planner on one saved world, beside the reference's own KPA sources).

Multi-GPU: problems are independent -> every rank owns its own 1,024 worlds, no collective on the data
path ("weak" scaling); NCCL only reduces the timing (max over ranks) and gathers the verdict counts.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

os.environ.setdefault("OMP_NUM_THREADS", "1")  # oracle legs parallelise over problems, one thread each

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

NF, T = 7, 128
METRIC = "planning iters/s (eval_g + eval_jac_g pairs on built reach sets; Kinova 7-DOF, 128 steps, 10 obstacles)"
UNIT = "evals/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nprob", type=int, default=1024, help="worlds per GPU")
    ap.add_argument("--nobs", type=int, default=10)
    ap.add_argument("--iters", type=int, default=16, help="k-iterates per step")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline eval loop")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-m1", action="store_true")
    ap.add_argument("--sweep-worlds", type=int, default=65536, help="BASELINE config 5: total worlds of the sweep (0: skip)")
    ap.add_argument("--sweep-seconds", type=float, default=45.0, help="wall-clock box of the sweep per rank")
    ap.add_argument("--no-configs", action="store_true", help="skip the config 1 / 3 / 4 objects")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write g and the dense Jacobian of the last k-iterate of the last step as "
                         "DIR/g.npy and DIR/jac.npy (float64; rank 0's worlds, a fixed sample of them beyond 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 timed path")
    return args


DUMP_BYTES = 64 * 10 ** 6


def dump_sample(nprob, m):
    """Worlds whose g [m] and dense Jacobian [m, 7] --dump-outputs writes: all of them when they fit in DUMP_BYTES (less
    room for the .npy headers), else a sorted sample drawn with a fixed seed, so that runs with the same arguments write
    the same worlds."""
    n = min(nprob, (DUMP_BYTES - 1024) // (8 * m * (1 + NF)))
    if n < 1:
        raise SystemExit(f"bench.py: g and the Jacobian of one world ({m} constraints) exceed {DUMP_BYTES} bytes")
    if n == nprob:
        return np.arange(nprob)
    return np.sort(np.random.default_rng(0).choice(nprob, n, replace=False))


def dump_outputs(out_dir, d_g, d_j):
    """What the timed step hands its caller (g [nprob, m] and the dense Jacobian [nprob, m, 7] of its last k-iterate,
    on the device) for the worlds of dump_sample, as float64 .npy files."""
    import torch

    sel = torch.as_tensor(dump_sample(*d_g.shape), device=d_g.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "g.npy"), d_g[sel].cpu().numpy())
    np.save(os.path.join(out_dir, "jac.npy"), d_j[sel].cpu().numpy())


_WORLDS = None


def load_worlds():
    """armour_b200/worlds.py (pure numpy input generators) loaded by path: importing the armour_b200 PACKAGE would map
    libarmour_b200.so, which the reference arm must never do."""
    global _WORLDS
    if _WORLDS is None:
        import importlib.util
        spec = importlib.util.spec_from_file_location("armour_worlds", os.path.join(ROOT, "armour_b200", "worlds.py"))
        _WORLDS = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(_WORLDS)
    return _WORLDS


# ---------------------------------------------------------------------------------------------------
def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms while the timed regions run."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._pump, daemon=True)
            self.thr.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark(self):
        return time.time()

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self, windows):
        """`windows`: (t0, t1) wall-clock pairs of the timed regions, the device-timed one first.  The device
        region of the default run lasts ~50 ms, so when it holds fewer than 3 samples the other timed regions
        of the same run (host-buffer path, M1), equally under load, are added; `window` says which were used."""
        out = self._summary(windows[:1])
        out["window"] = "device-timed region"
        if out["samples"] < 3 and len(windows) > 1:
            out = self._summary(windows)
            out["window"] = "all timed regions of the run (device, host-buffer, M1)"
        return out

    def _summary(self, windows):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            if not any(t0 <= ts <= t1 + 0.05 for t0, t1 in windows):
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# CPU oracle legs (the checker timed as the CPU baseline; never on the product path)
def oracle_run(nthreads, nobs, iters, steps, warmup, seed, seconds=None):
    """`nthreads` problems, one host thread each (ctypes releases the GIL; the oracle is thread-safe).
    Returns build seconds (all problems, in parallel) and the per-step seconds of `iters` eval pairs per
    problem.  With `seconds` set, runs steps until the budget is spent (at least one)."""
    from concurrent.futures import ThreadPoolExecutor

    worlds = load_worlds()
    from oracle.pyoracle import OracleProblem, lib
    lib()
    q0, qd0, qdd0, _, obs = worlds.random_problems(nthreads, nobs, seed=seed)
    ks = worlds.halton_k(iters * max(1, nthreads)).reshape(iters, -1, NF)
    probs = [OracleProblem(max_obstacles=max(40, nobs)) for _ in range(nthreads)]
    pool = ThreadPoolExecutor(nthreads)
    t0 = time.perf_counter()
    list(pool.map(lambda i: probs[i].build(q0[i], qd0[i], qdd0[i], obs[i], nthreads=1), range(nthreads)))
    build_s = time.perf_counter() - t0

    def one(i):
        for it in range(iters):
            probs[i].eval_g(ks[it, i])
            probs[i].eval_jac_g(ks[it, i])

    times = []
    n = 0
    tstart = time.perf_counter()
    while True:
        t0 = time.perf_counter()
        list(pool.map(one, range(nthreads)))
        dt = time.perf_counter() - t0
        n += 1
        if n > warmup:
            times.append(dt)
        if seconds is None:
            if len(times) >= steps:
                break
        elif len(times) >= 1 and time.perf_counter() - tstart > seconds:
            break
    pool.shutdown()
    return build_s, times


def workload_config(nprob, nobs, iters, world):
    """The `config` object of the line: identical in both arms (the reference arm times a bounded SAMPLE of this workload,
    described in its cpu_baseline.sample)."""
    return {"workload": f"Kinova Gen3 batched {nprob} random worlds x {nobs} obstacles per GPU, one eval_g + eval_jac_g per "
                        f"world per k-iterate, {iters} k-iterates per step",
            "time_intervals": T, "obstacles": nobs, "constraints_per_world": NF * T + 7 * T * nobs + 4 * NF,
            "k_iterates_per_step": iters, "worlds_per_gpu": nprob, "parallelism": f"worlds sharded x{world}",
            "l2": "outputs (g + dense Jacobian) and reach-set tables per launch exceed the 126 MB L2"}


def reference_available():
    """The reference's own planner path (oracle/_ref/libarmour_ref_cuda.so) needs the prebuilt library and a GPU."""
    try:
        from oracle import pyrefcuda
        return pyrefcuda.available()
    except Exception:
        return False


def reference_run(nworlds, nobs, iters, steps, warmup, seed, seconds=None):
    """The REFERENCE ITSELF: `nworlds` worlds, one after the other like kinova_planner_realtime (one process, one world):
    build (OpenMP over the 128 intervals on all cores, then its hyper-plane kernels), then per step `iters` x (eval_g,
    eval_jac_g) per world through armtd_NLP.  Returns (build seconds per world, per-step seconds)."""
    cores = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(cores)  # before libgomp of the reference library starts (it is loaded lazily)
    worlds = load_worlds()
    from oracle import pyrefcuda
    q0, qd0, qdd0, q_des, obs = worlds.random_problems(nworlds, nobs, seed=seed)
    ks = worlds.halton_k(iters * max(1, nworlds)).reshape(iters, -1, NF)
    probs, build_s = [], []
    devnull = os.open(os.devnull, os.O_WRONLY)
    for i in range(nworlds):
        t0 = time.perf_counter()
        probs.append(pyrefcuda.ReferencePlanner(q0[i], qd0[i], qdd0[i], q_des[i], obs[i], nthreads=cores))
        build_s.append(time.perf_counter() - t0)
    os.close(devnull)
    times, n = [], 0
    tstart = time.perf_counter()
    while True:
        t0 = time.perf_counter()
        for i in range(nworlds):
            for it in range(iters):
                probs[i].eval_g(ks[it, i])
                probs[i].eval_jac_g(ks[it, i])
        dt = time.perf_counter() - t0
        n += 1
        if n > warmup:
            times.append(dt)
        if seconds is None:
            if len(times) >= steps:
                break
        elif len(times) >= 1 and time.perf_counter() - tstart > seconds:
            break
    return build_s, times


def cpu_leg(nobs, iters, steps, warmup, seconds=None):
    """The CPU side of the comparison on this box: the reference itself when it travelled, else the port.  Returns the
    cpu_baseline object (value in M2 units/s) and, for the line, ms per step."""
    cores = os.cpu_count() or 1
    if reference_available():
        nworlds = 4
        build_s, times = reference_run(nworlds, nobs, iters, steps, warmup, 20261017, seconds)
        value = nworlds * iters * len(times) / sum(times)
        obj = {"value": value, "unit": UNIT, "cores": cores, "kind": "reference",
               "sample": f"{nworlds} worlds of the same generator (seed 20261017), one after the other like the reference "
                         f"planner, x {iters} k-iterates x {len(times)} steps ({sum(times):.1f} s); the reference's own "
                         f"sources (KPR PZsparse / Trajectory / Dynamics / CollisionChecking / NLPclass .cu, nvcc -O2 "
                         f"-Xcompiler -fopenmp) against stand-in Eigen / Boost.Interval / Ipopt headers: OpenMP slices on "
                         f"{cores} threads + its own collision kernels on the GPU",
               "build_s_per_world": float(np.median(build_s)), "builds_per_s": 1.0 / float(np.median(build_s)),
               "sample_worlds": nworlds}
    else:
        build_s, times = oracle_run(cores, nobs, iters, steps, warmup, seed=20261017, seconds=seconds)
        value = cores * iters * len(times) / sum(times)
        obj = {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{cores} worlds of the same generator (seed 20261017), one per host thread, x {iters} "
                         f"k-iterates x {len(times)} steps ({sum(times):.1f} s); oracle = C++ restatement of the reference "
                         f"(oracle/_ref/libarmour_ref_cuda.so absent or no GPU)",
               "build_s_per_world_1thread": build_s, "builds_per_s_all_cores": cores / build_s, "sample_worlds": cores}
    return obj, 1e3 * sum(times) / len(times)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    obj, ms_per_step = cpu_leg(args.nobs, args.iters, args.steps, args.warmup)
    value = obj["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.nprob, args.nobs, args.iters, args.gpus),
        "sample_note": "per-world throughput of the same generator; the GPU arm runs 1,024 worlds per GPU, the CPU arm a "
                       "bounded sample of them, one world at a time like the reference planner (cpu_baseline.sample)",
        "cpu_baseline": obj,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------------
def config1_host_abi(device):
    """BASELINE config 1 through the reference-facing calls: armour_reachsets_build + 20 x (armour_eval_g,
    armour_eval_jac_g) with HOST pointers on saved world 016_006, wall clock (Python ctypes call overhead included,
    ~10 us per call).  Beside it the same problem on the CPU: the reference itself when it travelled (OpenMP over the
    intervals on all cores, its own threading: KPR/armour_main.cu:99,117, KPR/NLPclass.cu:304,376), and the port."""
    from armour_b200 import ReachSetEngine
    worlds = load_worlds()
    q0, qd0, qdd0, q_des, obs = worlds.config1_problem(os.path.join(ROOT, "tests", "golden", "worlds", "scene_016_006.csv"))
    ks = np.vstack([np.zeros(NF), worlds.halton_k(19)])
    eng = ReachSetEngine(max_problems=1, max_obstacles=obs.shape[0], device=device)
    rc = eng.lib.armour_ctx_reserve(eng._h, 1, obs.shape[0])
    assert rc == 0
    build, pair, total = [], [], []
    for rep in range(15):
        t0 = time.perf_counter()
        eng.build(q0, qd0, qdd0, obs)
        t1 = time.perf_counter()
        for k in ks:
            eng.eval_g(k)
            eng.eval_jac_g(k)
        t2 = time.perf_counter()
        if rep >= 3:
            build.append(1e3 * (t1 - t0))
            pair.append(1e3 * (t2 - t1) / len(ks))
            total.append(1e3 * (t1 - t0) + 1e3 * (t2 - t1) / len(ks))
    fused = []
    for rep in range(6):  # the same pair as ONE call (armour_eval_g_jac: one launch, one synchronisation)
        t1 = time.perf_counter()
        for k in ks:
            eng.eval(k)
        if rep >= 1:
            fused.append(1e3 * (time.perf_counter() - t1) / len(ks))
    eng.close()
    out = {"world": "scene_016_006.csv", "obstacles": int(obs.shape[0]), "iterates": len(ks),
           "eval_g_jac_fused_ms": float(np.median(fused)),
           "one_iteration_fused_ms": float(np.median(build) + np.median(fused)),
           "build_ms": float(np.median(build)), "eval_g_plus_eval_jac_g_ms": float(np.median(pair)),
           "one_iteration_ms": float(np.median(total)), "target_ms": 1.0,
           "replan_ms_build_plus_20_iterates": float(np.median(build) + len(ks) * np.median(pair)),
           "timing": "wall clock around the host-pointer C-ABI calls (H2D of inputs / k, kernels, D2H of g / dense J, "
                     "synchronisation inside each call)"}
    cores = os.cpu_count() or 1
    from oracle.pyoracle import OracleProblem
    orc, ob, op = OracleProblem(), [], []
    for rep in range(3):
        t0 = time.perf_counter()
        orc.build(q0, qd0, qdd0, obs, nthreads=cores)
        t1 = time.perf_counter()
        for k in ks[:5]:
            orc.eval_g(k)
            orc.eval_jac_g(k)
        ob.append(1e3 * (t1 - t0))
        op.append(1e3 * (time.perf_counter() - t1) / 5)
    out["cpu_port"] = {"build_ms": float(min(ob)), "eval_g_plus_eval_jac_g_ms": float(min(op)), "threads": cores,
                       "one_iteration_ms": float(min(ob) + min(op))}
    if reference_available():
        from oracle import pyrefcuda
        os.environ["OMP_NUM_THREADS"] = str(cores)
        rb, rp = [], []
        for rep in range(3):
            t0 = time.perf_counter()
            ref = pyrefcuda.ReferencePlanner(q0, qd0, qdd0, q_des, obs, nthreads=cores)
            t1 = time.perf_counter()
            for k in ks[:5]:
                ref.eval_g(k)
                ref.eval_jac_g(k)
            rb.append(1e3 * (t1 - t0))
            rp.append(1e3 * (time.perf_counter() - t1) / 5)
            del ref
        out["cpu_reference"] = {"build_ms": float(min(rb)), "eval_g_plus_eval_jac_g_ms": float(min(rp)), "threads": cores,
                                "one_iteration_ms": float(min(rb) + min(rp)),
                                "note": "build includes the Obstacles constructor's cudaMalloc calls, as one process per "
                                        "replan does in the reference"}
        out["speedup_vs_reference_one_iteration"] = out["cpu_reference"]["one_iteration_ms"] / out["one_iteration_ms"]
    return out


def config_m1(device, stream, dev, nworlds, nobs, seed, label, **engine_kw):
    """M1 (build + one eval_g + eval_jac_g) of a small batch of another BASELINE configuration on the device, and the
    share of the evaluation spent on the torque rows (the same launch with the obstacles taken away)."""
    import torch

    from armour_b200 import ReachSetEngine
    worlds = load_worlds()
    q0, qd0, qdd0, _, obs = worlds.random_problems(nworlds, nobs, seed=seed)
    eng = ReachSetEngine(max_problems=nworlds, max_obstacles=nobs, device=device, **engine_kw)
    eng.set_stream(stream.cuda_stream)
    t = [torch.tensor(x, dtype=torch.float64, device=dev) for x in (q0, qd0, qdd0, obs)]
    m = eng.lib.armour_num_constraints(eng._h, nobs)
    d_k = torch.tensor(worlds.halton_k(nworlds), dtype=torch.float64, device=dev)
    d_g = torch.empty((nworlds, m), dtype=torch.float64, device=dev)
    d_j = torch.empty((nworlds, m, NF), dtype=torch.float64, device=dev)
    tb, te = [], []
    for rep in range(3):
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record(stream)
        eng.build_device(nworlds, nobs, *(x.data_ptr() for x in t))
        e1.record(stream)
        eng.eval_device(nworlds, d_k.data_ptr(), d_g.data_ptr(), d_j.data_ptr())
        e2.record(stream)
        torch.cuda.synchronize()
        tb.append(e0.elapsed_time(e1))
        te.append(e1.elapsed_time(e2))
    failures = int((eng.build_status() != 0).sum())
    ln, un = eng.monomial_counts()
    # torque-row share: the same reach sets evaluated without obstacles (torque + Bezier rows only)
    eng.build_device(nworlds, 0, t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), 0)
    m0 = eng.lib.armour_num_constraints(eng._h, 0)
    tt = []
    for rep in range(3):
        e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(2))
        e1.record(stream)
        eng.eval_device(nworlds, d_k.data_ptr(), d_g.data_ptr(), d_j.data_ptr())
        e2.record(stream)
        torch.cuda.synchronize()
        tt.append(e1.elapsed_time(e2))
    eng.close()
    b, e, t0 = min(tb), min(te), min(tt)
    return {"label": label, "worlds": nworlds, "obstacles": nobs, "constraints_per_world": int(m),
            "capacity_failures": failures, "build_ms_per_world": b / nworlds, "eval_ms_per_batch": e,
            "m1_problems_per_s": nworlds / ((b + e) * 1e-3), "m2_evals_per_s": nworlds / (e * 1e-3),
            "torque_rows_share_of_eval": t0 / e, "torque_only_eval_ms": t0, "rows_without_obstacles": int(m0),
            "link_monomials_max": int(ln.max()), "torque_monomials_max": int(un.max())}


def armtd_leg(device, cpu):
    """SURVEY 8f-3: the ARMTD comparison planner (KPA) on one saved world through the host-pointer ABI: build (imported joint
    reachable set -> link reach sets -> half-space candidates) and one eval_g + eval_jac_g pair, wall clock; the reference's own
    KPA sources (oracle/_ref/libarmour_ref_armtd.so, its CUDA collision kernels included) or the oracle beside it."""
    from armour_b200 import ArmtdPlanner
    worlds = load_worlds()
    q0, qd0, q_des, jrs, k_range, obs = worlds.armtd_problem(os.path.join(ROOT, "tests", "golden", "worlds", "scene_016_006.csv"), 1)
    k = np.array([0.5, 0.6, 0.7, 0.0, -0.5, -0.6, -0.7])
    p = ArmtdPlanner(device=device)
    p.build(q0, qd0, jrs, k_range, obs)
    p.eval(k)

    def best(fn, reps=7):
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return 1e3 * min(ts)

    out = {"world": "scene_016_006.csv", "obstacles": int(obs.shape[0]), "constraints": int(p.m),
           "build_ms": best(lambda: p.build(q0, qd0, jrs, k_range, obs)), "eval_g_plus_eval_jac_g_ms": best(lambda: p.eval(k)),
           "timing": "wall clock around the host-pointer C-ABI calls (copies and synchronisation inside)"}
    out["one_iteration_ms"] = out["build_ms"] + out["eval_g_plus_eval_jac_g_ms"]
    if cpu:
        from oracle import pyrefarmtd
        if pyrefarmtd.available():
            mk, kind = (lambda: pyrefarmtd.ReferenceArmtd(q0, qd0, q_des, jrs, k_range, obs)), "reference"
        else:
            from oracle.pyoracle import OracleArmtd
            mk, kind = (lambda: OracleArmtd().build(q0, qd0, jrs, k_range, obs)), "port"
        ref = mk()
        out["cpu_baseline"] = {"kind": kind, "cores": os.cpu_count() or 1, "build_ms": best(mk, 3),
                               "eval_g_plus_eval_jac_g_ms": best(lambda: (ref.eval_g(k), ref.eval_jac_g(k)), 5)}
        out["cpu_baseline"]["one_iteration_ms"] = out["cpu_baseline"]["build_ms"] + out["cpu_baseline"]["eval_g_plus_eval_jac_g_ms"]
        out["speedup_one_iteration"] = out["cpu_baseline"]["one_iteration_ms"] / out["one_iteration_ms"]
    p.close()
    return out


def controller_leg(device, stream, dev, cpu, n=1 << 20):
    """SURVEY 8f-4: RobustController::update (MEX/robust_controller.cpp:67-181) for n sampled states in one launch:
    device-resident states/s (CUDA events), the same through the host-pointer ABI call, and the reference's own sources
    (oracle/_ref/libarmour_ref_controller.so; the oracle's restatement if that library is absent) on one host thread."""
    import torch

    from armour_b200 import RobustController
    model = os.path.join(ROOT, "tests", "golden", "robot_models", "kinova_without_gripper.txt")
    ctl = RobustController(model, 0.03, device)
    ctl.set_stream(stream.cuda_stream)
    rng = np.random.default_rng(20261018)
    q = rng.uniform(-np.pi, np.pi, (n, 7))
    qd = rng.uniform(-1.5, 1.5, (n, 7))
    q_des, qd_des, qdd_des = q + rng.uniform(-0.05, 0.05, (n, 7)), qd + rng.uniform(-0.1, 0.1, (n, 7)), rng.uniform(-2, 2, (n, 7))
    Kr, gains = np.full(7, 10.0), (1.0, 1e-2, 1e-10)
    host = (q, qd, q_des, qd_des, qdd_des)
    t = [torch.tensor(a, dtype=torch.float64, device=dev) for a in host]
    u = torch.empty((n, 7), dtype=torch.float64, device=dev)
    lo, hi = torch.empty_like(u), torch.empty_like(u)
    st = torch.empty(n, dtype=torch.int32, device=dev)

    def timed(fn, reps=5):
        for _ in range(3):
            fn()
        torch.cuda.synchronize(dev)
        ms = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            torch.cuda.synchronize(dev)
            ms.append(e0.elapsed_time(e1))
        return float(np.median(ms))

    ms_upd = timed(lambda: ctl.update_device(n, Kr, *gains, *(x.data_ptr() for x in t), d_u=u.data_ptr(), d_status=st.data_ptr()))
    ms_int = timed(lambda: ctl.rnea_device(n, *(x.data_ptr() for x in t[:4]), d_tau_lo=lo.data_ptr(), d_tau_hi=hi.data_ptr()))
    out = {"metric": "controller updates/s (RobustController::update, ARMOUR method: nominal + interval Newton-Euler pass, "
                     "interval M(q) r, robust input) over sampled states, device-resident", "states": n,
           "value": n / (ms_upd * 1e-3), "unit": "states/s", "ms_per_launch": ms_upd,
           "interval_pass_only": {"value": n / (ms_int * 1e-3), "unit": "states/s", "ms_per_launch": ms_int},
           "status_nonzero": int(st.sum().item()), "kernel_launches": ctl.kernel_launches,
           "timing": "CUDA events on the launching stream, median of 5 launches after 3 warm-up launches; inputs of "
                     f"{5 * n * 56 / 1e6:.0f} MB, larger than L2 together with the outputs"}
    m = 1 << 16
    sub = [a[:m] for a in host]
    ctl.update(Kr, *gains, *sub)
    t0 = time.perf_counter()
    ctl.update(Kr, *gains, *sub)
    dt = time.perf_counter() - t0
    out["e2e"] = {"value": m / dt, "unit": "states/s", "states": m, "h2d_bytes": int(7 * m * 56), "d2h_bytes": int(3 * m * 56 + 4 * m),
                  "note": "armour_controller_update with host pointers: sin / cos on the host like the reference, copies, "
                          "launch, copies back, synchronised"}
    if cpu:
        from oracle import pycontroller
        kind = "reference" if pycontroller.reference_available() else "port"
        ref = (pycontroller.ReferenceController if kind == "reference" else pycontroller.OracleController)()
        k = 1500
        t0 = time.perf_counter()
        for i in range(k):
            ref.update(Kr, *gains, *(a[i] for a in host))
        dtc = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": k / dtc, "unit": "states/s", "cores": 1, "kind": kind,
                               "sample": f"{k} states, one update() per state like the MEX entry (MEX/kinova_controller.cpp), "
                                         "one host thread"}
        out["ratio_vs_cpu_one_thread"] = out["value"] / out["cpu_baseline"]["value"]
    ctl.close()
    return out


def run_sweep(args, eng, stream, dev, rank, world, dist):
    """BASELINE config 5: `--sweep-worlds` random worlds (config-2 generator), split over the ranks with
    sharding.shard_bounds (STRONG scaling: the total is fixed), each rank walking its shard in batches through the
    bench's context: build (M1) + 4 eval_g + eval_jac_g pairs per world (M2) + device verdict of the last iterate.
    Device-timed (CUDA events, max over ranks); the next batch's inputs are generated on the host while the GPU works.
    Per-world verdicts come back in global world order through sharding.gather_results (NCCL all-gather)."""
    import zlib

    import torch

    from armour_b200 import sharding
    worlds = load_worlds()
    nobs, iters, total = args.nobs, 4, args.sweep_worlds
    batch = min(args.nprob, 2048)
    lo, hi = sharding.shard_bounds(total, world, rank)
    m = eng.lib.armour_num_constraints(eng._h, nobs)
    d_g = torch.empty((batch, m), dtype=torch.float64, device=dev)
    d_j = torch.empty((batch, m, NF), dtype=torch.float64, device=dev)
    ks = torch.tensor(worlds.halton_k(iters * batch).reshape(iters, batch, NF), dtype=torch.float64, device=dev)
    verdict = torch.full((hi - lo,), -2, dtype=torch.int32, device=dev)  # -2: not run (time box), else feasible 0 / 1
    first = torch.full((hi - lo,), -2, dtype=torch.int32, device=dev)
    d_ok = torch.empty(batch, dtype=torch.int32, device=dev)
    d_first = torch.empty(batch, dtype=torch.int32, device=dev)
    t_build = t_eval = 0.0
    done = failed = 0
    wall0 = time.perf_counter()

    def gen(b0):
        n = min(batch, hi - b0)
        q0, qd0, qdd0, _, obs = worlds.random_problems(n, nobs, seed=1000003 + b0)
        return n, [torch.tensor(x, dtype=torch.float64).pin_memory() for x in (q0, qd0, qdd0, obs)]

    nxt = gen(lo) if hi > lo else None
    b0 = lo
    while nxt is not None:
        n, host = nxt
        t = [x.to(dev, non_blocking=True) for x in host]
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record(stream)
        eng.build_device(n, nobs, *(x.data_ptr() for x in t))
        e1.record(stream)
        for it in range(iters):
            eng.eval_device(n, ks[it].data_ptr(), d_g.data_ptr(), d_j.data_ptr())
        eng.verdict_device(n, d_g.data_ptr(), d_ok.data_ptr(), d_first.data_ptr())
        e2.record(stream)
        verdict[b0 - lo:b0 - lo + n].copy_(d_ok[:n], non_blocking=True)
        first[b0 - lo:b0 - lo + n].copy_(d_first[:n], non_blocking=True)
        b0 += n
        # host work for the next batch overlaps the device work of this one
        nxt = gen(b0) if (b0 < hi and time.perf_counter() - wall0 < args.sweep_seconds) else None
        torch.cuda.synchronize()
        t_build += e0.elapsed_time(e1)
        t_eval += e1.elapsed_time(e2)
        failed += int((eng.build_status()[:n] != 0).sum())
        done += n
    wall = time.perf_counter() - wall0
    tb, te = sharding.reduce_max(t_build, dev), sharding.reduce_max(t_eval, dev)
    counts = torch.tensor([done, failed], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(counts)
    res = sharding.gather_results({"feasible": verdict, "first_violation": first}, total)
    if rank != 0:
        return None
    v = res["feasible"].cpu().numpy()
    f = res["first_violation"].cpu().numpy()
    n_done = int(counts[0].item())
    return {"config": "BASELINE config 5: replanning sweep, strong scaling", "worlds": total, "worlds_done": n_done,
            "complete": n_done == total, "n_gpus": world, "batch_per_context": batch, "obstacles": nobs,
            "k_iterates_per_world": iters, "build_s": tb * 1e-3, "eval_s": te * 1e-3, "wall_s_rank0": wall,
            "m1_problems_per_s": n_done / ((tb + te / iters) * 1e-3), "m2_evals_per_s": n_done * iters / (te * 1e-3),
            "feasible_last_iterate": int((v == 1).sum()), "capacity_failures": int(counts[1].item()),
            "verdicts_gathered": int((v >= 0).sum()), "verdict_crc32": int(zlib.crc32(v.tobytes()) ^ zlib.crc32(f.tobytes())),
            "gather": "sharding.gather_results: all_gather of the per-world (feasible, first violated row) over NCCL",
            "timing": "CUDA events on the launching stream per batch, summed per rank, max over ranks"}


# ---------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch

    from armour_b200 import ReachSetEngine, worlds
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # NCCL prints its version banner on stdout when the communicator is created (NCCL_DEBUG=VERSION/WARN boxes):
        # stdout must carry exactly one JSON line, so the banner goes to stderr
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            warm = torch.zeros(1, device=torch.device("cuda", local))
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    dev = torch.device("cuda", local)
    nprob, nobs, iters = args.nprob, args.nobs, args.iters

    # ---- inputs (synthetic, config-2 generator), reach sets built once per problem -------------------
    q0, qd0, qdd0, q_des, obs = worlds.random_problems(nprob, nobs, seed=20261017 + rank)
    eng = ReachSetEngine(max_problems=nprob, max_obstacles=nobs, device=local)
    # the library launches on THIS stream and the CUDA events below are recorded on it (a NULL handle would
    # make the context fall back to its own stream, which torch events do not see)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    eng.set_stream(stream.cuda_stream)
    tq0, tqd0, tqdd0, tobs = (torch.tensor(a, dtype=torch.float64, device=dev) for a in (q0, qd0, qdd0, obs))
    launches0 = eng.kernel_launches
    eng.build_device(nprob, nobs, tq0.data_ptr(), tqd0.data_ptr(), tqdd0.data_ptr(), tobs.data_ptr())
    torch.cuda.synchronize()
    build_launches = eng.kernel_launches - launches0
    status = eng.build_status()
    if status.any():
        raise SystemExit(f"reach-set build overflowed a monomial table for {int((status != 0).sum())} problems")
    m = eng.m
    ks_host = worlds.halton_k(iters * nprob).reshape(iters, nprob, NF)
    d_k = torch.tensor(ks_host, dtype=torch.float64, device=dev)
    d_g = torch.empty((nprob, m), dtype=torch.float64, device=dev)
    d_j = torch.empty((nprob, m, NF), dtype=torch.float64, device=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def step_device():
        for it in range(iters):
            eng.eval_device(nprob, d_k[it].data_ptr(), d_g.data_ptr(), d_j.data_ptr())

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        timed.launches = eng.kernel_launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        timed.launches = eng.kernel_launches - timed.launches
        barrier()
        t1 = time.time()
        ms = e0.elapsed_time(e1)
        timed.per_rank = [ms]
        if dist is not None:  # max over ranks is the time of the job; the per-rank list tells variance from contention
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            parts = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(parts, t)
            timed.per_rank = [float(x.item()) for x in parts]
            ms = max(timed.per_rank)
        return ms, t0, t1

    # One step = 16 k-iterates x (k_constraints + k_constraints_slow), captured ONCE in a CUDA graph and replayed: the
    # device-timed region then does not depend on how fast each rank's host thread can enqueue 32 launches per step
    # (with 8 ranks + NCCL threads + clock samplers sharing the host, slow enqueueing showed up as 10-30 % slower ranks).
    step_timed, launches_per_step, graph_used = step_device, None, False
    try:
        step_device()  # warm: modules loaded, nothing allocated inside the capture
        torch.cuda.synchronize()
        l0 = eng.kernel_launches
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            step_device()
        launches_per_step = eng.kernel_launches - l0
        torch.cuda.set_stream(stream)
        graph.replay()
        torch.cuda.synchronize()
        step_timed, graph_used = graph.replay, True
    except Exception as exc:  # capture not possible on this stack: plain launches
        sys.stderr.write(f"bench.py: CUDA graph capture of the step failed ({exc!r}); timing plain launches\n")
        torch.cuda.synchronize()
        torch.cuda.set_stream(stream)

    clocks = ClockSampler(local).start()
    time.sleep(0.3)
    la = eng.kernel_launches
    ms_dev, c0, c1 = timed(step_timed, args.steps, args.warmup)
    launches_timed = timed.launches if not graph_used else launches_per_step * args.steps
    per_rank_dev = list(timed.per_rank)
    clock_windows = [(c0, c1)]
    value = world * nprob * iters * args.steps / (ms_dev * 1e-3)
    if args.dump_outputs and rank == 0:  # before anything below overwrites d_g / d_j
        dump_outputs(args.dump_outputs, d_g, d_j)

    # verdicts of the last iterate (on the device), gathered as counts: the only cross-rank traffic
    d_ok = torch.empty(nprob, dtype=torch.int32, device=dev)
    d_first = torch.empty(nprob, dtype=torch.int32, device=dev)
    eng.verdict_device(nprob, d_g.data_ptr(), d_ok.data_ptr(), d_first.data_ptr())
    feas = d_ok.sum().to(torch.float64).reshape(1)
    if dist is not None:
        dist.all_reduce(feas)
    feasible_total = int(feas.item())

    # ---- roofline of k_constraints (the only kernel of the timed region) ----------------------------
    ln, un = eng.monomial_counts()
    NJ = eng.NJ
    reads = (int(ln.sum()) * (24 + 8) + int(un.sum()) * (8 + 8) + nprob * (T * NJ * 24 + T * NF * 8 + T * NJ * 144 +
                                                                         nobs * 96 + 56))
    writes = nprob * 8 * m * (1 + NF)
    alg_bytes = reads + writes
    n_launch = args.steps * iters
    kernel_ms = ms_dev / n_launch
    peak, peak_src = peaks()
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    roofline = {"kernel": "k_constraints", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": kernel_ms,
                "launch_ms_per_rank": [x / n_launch for x in per_rank_dev], "bytes_per_unit": alg_bytes / nprob,
                "note": "launch = k_constraints + k_constraints_slow (the latter returns at once here: ~1 % of the time)"}
    prof = os.path.join(ROOT, "profiles", "k_constraints_traffic.json")
    if os.path.exists(prof):  # dram bytes per launch from the committed ncu --set full capture of this command
        with open(prof) as f:
            pj = json.load(f)
        if pj.get("nprob") == nprob and pj.get("nobs") == nobs:
            roofline["traffic"] = pj.get("dram_bytes_per_launch")

    # ---- e2e: the host-buffer C-ABI call, copies inside the timed region --------------------------------
    e2e = None
    if not args.no_e2e:
        h_k = torch.empty((iters, nprob, NF), dtype=torch.float64, pin_memory=True)
        h_k.copy_(torch.from_numpy(ks_host))
        h_g = torch.empty((nprob, m), dtype=torch.float64, pin_memory=True)
        h_j = torch.empty((nprob, m, NF), dtype=torch.float64, pin_memory=True)
        k_np, g_np, j_np = h_k.numpy(), h_g.numpy(), h_j.numpy()

        def step_host():
            for it in range(iters):
                eng.eval_into(k_np[it], g_np, j_np)

        ms_e2e, h0, h1 = timed(step_host, args.steps, args.warmup)
        clock_windows.append((h0, h1))
        e2e = {"value": world * nprob * iters * args.steps / (ms_e2e * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": iters * nprob * NF * 8, "d2h_bytes_per_step": iters * nprob * m * (1 + NF) * 8,
               "ms_per_step": ms_e2e / args.steps, "ms_per_step_per_rank": [x / args.steps for x in timed.per_rank],
               "note": "dense m x 7 Jacobian of every world crosses PCIe every iterate (the reference's TNLP contract): "
                       "PCIe-bound; see solver_e2e for the path that keeps g and J on the device"}
        # the structured variant of the same call: g + the non-zeros of the Jacobian (39 % fewer Jacobian bytes)
        try:
            nnz = eng.jacobian_nnz
            h_v = torch.empty((nprob, nnz), dtype=torch.float64, pin_memory=True)
            v_np = h_v.numpy()

            def step_host_structured():
                for it in range(iters):
                    eng.eval_structured_into(k_np[it], g_np, v_np)

            ms_s, h0, h1 = timed(step_host_structured, args.steps, args.warmup)
            e2e["structured"] = {"value": world * nprob * iters * args.steps / (ms_s * 1e-3), "unit": UNIT,
                                 "d2h_bytes_per_step": iters * nprob * (m + nnz) * 8, "nnz_per_world": int(nnz),
                                 "dense_values_per_world": int(m * NF), "ms_per_step": ms_s / args.steps,
                                 "note": "armour_batch_eval_structured: same g, the Jacobian as its fixed non-zero pattern "
                                         "(armour_jacobian_structure) — offered beside the dense call, which keeps the "
                                         "reference's contract"}
            del h_v
        except Exception as exc:
            e2e["structured"] = {"error": repr(exc)}
        # the host path must deliver what the device path computed
        eng.eval_device(nprob, d_k[iters - 1].data_ptr(), d_g.data_ptr(), d_j.data_ptr())
        torch.cuda.synchronize()
        if not (torch.equal(d_g.cpu(), h_g) and torch.equal(d_j.cpu(), h_j)):
            raise SystemExit("bench.py: host-buffer and device-pointer evaluations disagree")
        del h_g, h_j

    # ---- M1: reach-set build + one evaluation --------------------------------------------------------
    m1 = None
    if not args.no_m1:
        def step_m1():
            eng.build_device(nprob, nobs, tq0.data_ptr(), tqd0.data_ptr(), tqdd0.data_ptr(), tobs.data_ptr())
            eng.eval_device(nprob, d_k[0].data_ptr(), d_g.data_ptr(), d_j.data_ptr())

        ms_m1, h0, h1 = timed(step_m1, 2, 1)
        clock_windows.append((h0, h1))

        def step_build():
            eng.build_device(nprob, nobs, tq0.data_ptr(), tqd0.data_ptr(), tqdd0.data_ptr(), tobs.data_ptr())

        ms_b, _, _ = timed(step_build, 2, 0)
        m1 = {"metric": "reach-set build + eval_g + eval_jac_g per problem (M1)", "value": world * nprob * 2 / (ms_m1 * 1e-3),
              "unit": "problems/s", "ms_per_batch": ms_m1 / 2, "build_ms_per_batch": ms_b / 2,
              "build_us_per_problem": 1e3 * ms_b / 2 / nprob}
        if rank == 0:
            # latency of ONE planning iteration (BASELINE config 1; target < 1 ms): saved world 016_006
            csv = os.path.join(ROOT, "tests", "golden", "worlds", "scene_016_006.csv")
            a0, a1, a2, _, aobs = worlds.config1_problem(csv)
            e1 = ReachSetEngine(max_problems=1, max_obstacles=aobs.shape[0], device=local)
            e1.set_stream(stream.cuda_stream)
            t0_, t1_, t2_, to_ = (torch.tensor(a, dtype=torch.float64, device=dev) for a in (a0, a1, a2, aobs))
            k1 = torch.zeros(NF, dtype=torch.float64, device=dev)
            g1 = torch.empty(e1.lib.armour_num_constraints(e1._h, aobs.shape[0]), dtype=torch.float64, device=dev)
            j1 = torch.empty((g1.numel(), NF), dtype=torch.float64, device=dev)
            lat_b, lat_e = [], []
            for rep in range(25):
                ea, eb, ec = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                ea.record(stream)
                e1.build_device(1, aobs.shape[0], t0_.data_ptr(), t1_.data_ptr(), t2_.data_ptr(), to_.data_ptr())
                eb.record(stream)
                e1.eval_device(1, k1.data_ptr(), g1.data_ptr(), j1.data_ptr())
                ec.record(stream)
                torch.cuda.synchronize()
                if rep >= 5:
                    lat_b.append(ea.elapsed_time(eb))
                    lat_e.append(eb.elapsed_time(ec))
            m1["single_problem_latency_ms"] = {"build": float(np.median(lat_b)), "eval": float(np.median(lat_e)),
                                               "total": float(np.median(lat_b) + np.median(lat_e)),
                                               "world": "scene_016_006.csv", "target_ms": 1.0}
            e1.close()
        fp64 = eng.measure_fp64_peak()
        # F_build: FP64 flops of the coefficient products of one build (counted by the oracle on a sample problem,
        # SURVEY.md 8d: ~83-89 MFLOP per problem at the default threshold)
        m1["fp64_peak_tflops_measured"] = fp64

    # ---- BASELINE config 1 where the reference measures it: ONE planning problem through HOST pointers, eval_g and
    # eval_jac_g called separately like Ipopt does (KPR/NLPclass.cu:272-396), wall clock around the C-ABI calls
    config1 = None
    if rank == 0 and not args.no_configs:
        try:
            config1 = config1_host_abi(local)
        except Exception as exc:
            config1 = {"error": repr(exc)}

    # ---- batched planning end to end: q_des in (host), k_opt / verdict out (host); g and J never leave the device
    solver_e2e = None
    if not args.no_m1:
        try:
            eng.solve(q_des)  # warm-up: workspace allocation
            reps = []
            for _ in range(3):
                barrier()
                t0s = time.perf_counter()
                ksol, oksol, firstsol, itsol = eng.solve(q_des)  # every rank plans its own worlds
                reps.append(time.perf_counter() - t0s)
            dts_rank = float(np.median(reps))
            dts, per_rank_s = dts_rank, [dts_rank]
            if dist is not None:
                tt = torch.tensor([dts_rank], dtype=torch.float64, device=dev)
                parts = [torch.empty_like(tt) for _ in range(world)]
                dist.all_gather(parts, tt)
                per_rank_s = [float(x.item()) for x in parts]
                dts = max(per_rank_s)
            solver_e2e = {"metric": "plans/s (armour_batch_solve: whole NLP loop per world on the device; host q_des in, "
                                    "k_opt + verdict + iterations out), all ranks, max over ranks",
                          "value": world * nprob / dts, "unit": "plans/s", "n_gpus": world,
                          "seconds": dts, "seconds_per_rank": per_rank_s, "worlds": world * nprob,
                          "feasible_rank0": int(oksol.sum()),
                          "iterations_mean": float(itsol.mean()), "iterations_max": int(itsol.max()),
                          "h2d_bytes_per_gpu": nprob * NF * 8, "d2h_bytes_per_gpu": nprob * (NF * 8 + 12),
                          "constraint_evals_per_s": float((2 * itsol + 2).sum() / dts)}
            if rank == 0 and world == 1 and not args.no_cpu_baseline:
                # CPU arm: the same solver algorithm (armour_b200/host/local_solver.cpp) over the CPU oracle, one world per
                # host thread, on the first worlds of the same batch; no wall-clock limit on either side
                from concurrent.futures import ThreadPoolExecutor

                from oracle.pyoracle import OracleProblem
                cores = os.cpu_count() or 1
                nw = min(2 * cores, nprob)
                probs = [OracleProblem(max_obstacles=max(40, nobs)) for _ in range(nw)]
                pool = ThreadPoolExecutor(cores)
                list(pool.map(lambda i: probs[i].build(q0[i], qd0[i], qdd0[i], obs[i], nthreads=1), range(nw)))
                t0c = time.perf_counter()
                res = list(pool.map(lambda i: probs[i].solve(q_des[i]), range(nw)))
                dtc = time.perf_counter() - t0c
                pool.shutdown()
                agree = sum(int(res[i][1] == bool(oksol[i])) for i in range(nw))
                solver_e2e["cpu"] = {"value": nw / dtc, "unit": "plans/s", "cores": cores, "worlds": nw, "seconds": dtc,
                                     "kind": "host local solver over the CPU oracle (reach sets already built)",
                                     "verdicts_agreeing_with_device": agree,
                                     "max_abs_k_opt_diff_feasible": float(max(
                                         [np.max(np.abs(res[i][0] - ksol[i])) for i in range(nw) if res[i][1] and oksol[i]] or [0.0]))}
                solver_e2e["ratio_vs_cpu"] = solver_e2e["value"] / solver_e2e["cpu"]["value"]
        except Exception as exc:  # an extra, never allowed to take the bench line down
            solver_e2e = {"error": repr(exc)}

    # ---- BASELINE configs 3 and 4 (rank 0; small batches, M1 = build + one evaluation, torque-row share of the eval)
    config3 = config4 = None
    if rank == 0 and not args.no_configs:
        try:
            config3 = config_m1(local, stream, dev, nworlds=128, nobs=40, seed=3, robot_model=1, mass_uncertainty=0.10,
                                inertia_uncertainty=0.10, cap_link=64, cap_torque=128,
                                label="config 3: gripper link (8 links), 40 obstacles, 10 % mass / inertia uncertainty")
            config4 = [config_m1(local, stream, dev, nworlds=16, nobs=100, seed=4, simplify_threshold=thr, cap_link=128,
                                 cap_torque=256, cap_work=cw, label=f"config 4: 100 obstacles, SIMPLIFY_THRESHOLD {thr:g}")
                       for thr, cw in ((5e-5, 4096), (5e-6, 16384))]
        except Exception as exc:
            config3 = config3 or {"error": repr(exc)}
            config4 = config4 or {"error": repr(exc)}

    # ---- SURVEY 8f-4: robust controller (interval Newton-Euler pass + robust input) over sampled states, rank 0
    controller = None
    if rank == 0 and not args.no_configs:
        try:
            controller = controller_leg(local, stream, dev, cpu=(world == 1 and not args.no_cpu_baseline))
        except Exception as exc:
            controller = {"error": repr(exc)}

    # ---- SURVEY 8f-3: ARMTD comparison planner, one problem through the host-pointer ABI, rank 0
    armtd = None
    if rank == 0 and not args.no_configs:
        try:
            armtd = armtd_leg(local, cpu=(world == 1 and not args.no_cpu_baseline))
        except Exception as exc:
            armtd = {"error": repr(exc)}

    # ---- BASELINE config 5: the 65,536-world sweep, split over the ranks (strong scaling), per-world verdicts gathered
    sweep = None
    if args.sweep_worlds > 0:
        try:
            sweep = run_sweep(args, eng, stream, dev, rank, world, dist)
        except Exception as exc:
            sweep = {"error": repr(exc)}

    clocks.stop()
    clk = clocks.summary(clock_windows)

    # ---- CPU baseline on this box's host cores, bounded sample: the reference itself when it travelled, else the port
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        cpu, _ = cpu_leg(nobs, iters, 1, 0, seconds=args.cpu_seconds)
        if cpu["kind"] == "reference":  # the port beside it, for the record (one world per host thread)
            pb, pt = oracle_run(cores, nobs, iters, 1, 0, seed=20261017, seconds=min(6.0, args.cpu_seconds))
            cpu["port"] = {"value": cores * iters * len(pt) / sum(pt), "unit": UNIT, "cores": cores,
                           "build_s_per_world_1thread": pb, "builds_per_s_all_cores": cores / pb}
        if m1 is not None:
            # FP64 roofline of the build kernel: flops counted by the oracle on one problem of this batch
            from oracle.pyoracle import OracleProblem
            ref = OracleProblem(max_obstacles=max(40, nobs)).build(q0[0], qd0[0], qdd0[0], obs[0], nthreads=cores)
            fl = ref.stats()["flops"]
            ach = fl * nprob / (m1["build_ms_per_batch"] * 1e-3) / 1e12
            m1["roofline_build"] = {"kernel": "k_reachsets", "bound": "fp64", "flops_per_problem": fl,
                                    "achieved": ach, "peak": m1["fp64_peak_tflops_measured"], "unit": "TFLOP/s",
                                    "frac": ach / m1["fp64_peak_tflops_measured"],
                                    "note": "2x counted flops (nominal + interval RNEA) in the oracle; the kernel runs "
                                            "RNEA once with two radius lanes"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(nprob, nobs, iters, world),
            "step_submission": "CUDA graph replay (one graph = one step)" if graph_used else "plain launches",
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "m1": m1, "config1_host_abi": config1,
            "solver_e2e": solver_e2e, "config3": config3, "config4": config4, "sweep": sweep,
            "controller": controller, "armtd": armtd, "gpu_launches": int(launches_timed), "clocks": clk,
            "feasible_worlds_last_iterate": feasible_total, "build_launches": int(build_launches),
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    args = parse_args()
    sys.dont_write_bytecode = True  # the tree may be read-only: no __pycache__ beside the modules imported from here on
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
