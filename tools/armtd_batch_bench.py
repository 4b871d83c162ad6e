"""Measurement of the batched ARMTD comparison planner (ArmtdBatch / armour_armtd_batch_*) on one GPU.

Workload: 1 024 worlds x 10 obstacles from worlds.armtd_random_problems.  Reports, as one JSON document:
  - the batched build per problem: the device-pointer build (inputs resident) timed with CUDA events on the context's stream,
    the window ending in a synchronise; and the host-pointer build (copies included), wall clock;
  - device-resident evaluation pairs (eval_g + eval_jac_g) per second, CUDA events;
  - armour_armtd_batch_solve plans per second (host pointers, wall clock), iteration counts, number feasible;
  - in the same run, the single-problem context (ArmtdPlanner) on a sample of 32 of the same worlds: build ms and one
    eval_g + eval_jac_g pair through host pointers, as bench.py's armtd leg measures them;
  - how many sampled worlds' batched verdict and k_opt agree with OracleArmtd.solve (the host solver over the CPU oracle).
Every shape is warmed up before it is timed.  The card's name and power limit are read (read-only) in the same run.

usage: python tools/armtd_batch_bench.py [--nprob 1024] [--nobs 10] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
import numpy as np  # noqa: E402
import torch  # noqa: E402

from armour_b200 import ArmtdBatch, ArmtdPlanner, worlds  # noqa: E402


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        out["nvidia_smi"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        out["nvidia_smi"] = repr(exc)
    return out


def events_ms(fn, reps):
    """median of `reps` CUDA-event windows around fn() on the current stream, each ending in a synchronise"""
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts))


def wall_ms(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nprob", type=int, default=1024)
    ap.add_argument("--nobs", type=int, default=10)
    ap.add_argument("--sample", type=int, default=32)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("armtd_batch_bench: no CUDA device (there is no CPU path)")
    n, nobs = a.nprob, a.nobs
    t0 = time.perf_counter()
    q0, qd0, q_des, kr, jrs, obs = worlds.armtd_random_problems(n, nobs)
    gen_s = time.perf_counter() - t0
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)  # a stream of its own (a NULL handle would leave the context on its private stream)
    torch.cuda.set_stream(stream)
    b = ArmtdBatch(max_problems=n, max_obstacles=nobs)
    b._check(b.lib.armour_ctx_set_stream(b._h, C_void(stream.cuda_stream)))  # the events below are recorded on this stream
    d_in = [torch.as_tensor(np.ascontiguousarray(x), device=dev) for x in (q0, qd0, jrs, kr, obs)]
    ptrs = [x.data_ptr() for x in d_in]
    k = worlds.halton_k(n)
    d_k = torch.as_tensor(k, device=dev)
    m = b.NJ * 100 * nobs + 28
    d_g = torch.empty((n, m), dtype=torch.float64, device=dev)
    d_J = torch.empty((n, m, 7), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()

    def build_device():
        b.build_device(n, nobs, *ptrs, None)

    def eval_device():
        b.eval_device(n, d_k.data_ptr(), d_g.data_ptr(), d_J.data_ptr())

    # warm-up of every shape
    b.build(q0, qd0, jrs, kr, obs)
    build_device()
    eval_device()
    b.solve(q_des)
    torch.cuda.synchronize()
    status = b.build_status()
    build_dev_ms = events_ms(build_device, 7)
    build_host_ms = wall_ms(lambda: b.build(q0, qd0, jrs, kr, obs), 5)
    reps = 20
    eval_ms = events_ms(lambda: [eval_device() for _ in range(reps)], 5) / reps
    t0 = time.perf_counter()
    k_opt, ok, first, iters = b.solve(q_des)
    solve_s = time.perf_counter() - t0

    # the single-problem context on a sample of the same worlds (host pointers, as bench.py's armtd leg)
    rng = np.random.default_rng(0)
    sample = np.sort(rng.choice(n, size=min(a.sample, n), replace=False))
    p = ArmtdPlanner(max_obstacles=nobs)
    p.build(q0[sample[0]], qd0[sample[0]], jrs[sample[0]], kr[sample[0]], obs[sample[0]])
    p.eval(k[sample[0]])
    single_build, single_eval = [], []
    for s in sample:
        single_build.append(wall_ms(lambda: p.build(q0[s], qd0[s], jrs[s], kr[s], obs[s]), 3))
        single_eval.append(wall_ms(lambda: p.eval(k[s]), 3))
    p.close()

    # agreement with the host solver over the CPU oracle on the sample
    from oracle.pyoracle import OracleArmtd
    agree, disagree = 0, []
    for s in sample:
        o = OracleArmtd().build(q0[s], qd0[s], jrs[s], kr[s], obs[s])
        k_ref, ok_ref, first_ref, _ = o.solve(q_des[s])
        same = (bool(ok[s]), int(first[s])) == (ok_ref, first_ref) and (not ok_ref or np.max(np.abs(k_opt[s] - k_ref)) <= 1e-8)
        agree += int(same)
        if not same:
            disagree.append(int(s))

    single_build_ms = float(np.median(single_build))
    out = {
        "tool": "tools/armtd_batch_bench.py",
        "card": card(),
        "workload": {"worlds": n, "obstacles": nobs, "generator": "worlds.armtd_random_problems(seed=20261017)",
                     "constraints_per_world": m, "generator_seconds": gen_s},
        "build_failures": int(np.sum(status != 0)),
        "batched_build": {
            "device_pointers_ms": build_dev_ms, "device_pointers_ms_per_problem": build_dev_ms / n,
            "host_pointers_ms": build_host_ms, "host_pointers_ms_per_problem": build_host_ms / n,
            "timing": "device pointers: CUDA events on the context's stream around the build, median of 7, window ends in a "
                      "synchronise; host pointers (H2D of the offline tables and the status readback included): wall clock, "
                      "median of 5"},
        "device_eval": {"ms_per_batch": eval_ms, "pairs_per_s": n / (eval_ms * 1e-3),
                        "timing": f"CUDA events around {reps} back-to-back eval_g + eval_jac_g batches, median of 5"},
        "batched_solve": {"ms": solve_s * 1e3, "plans_per_s": n / solve_s, "feasible": int(ok.sum()),
                          "iterations_mean": float(iters.mean()), "iterations_max": int(iters.max()),
                          "iterations_histogram": np.bincount(iters, minlength=61).tolist(),
                          "timing": "wall clock around armour_armtd_batch_solve (host pointers, copies included), after a warm-up solve"},
        "single_problem_context": {"sample": int(len(sample)), "build_ms_median": single_build_ms,
                                   "eval_pair_ms_median": float(np.median(single_eval)),
                                   "timing": "wall clock around the host-pointer C-ABI calls, median of 3 per world, median over the sample"},
        "build_speedup_per_problem": {
            "device_pointers": single_build_ms / (build_dev_ms / n), "host_pointers": single_build_ms / (build_host_ms / n)},
        "oracle_agreement": {"sample": int(len(sample)), "agree": agree, "disagree": disagree,
                             "criterion": "same verdict and first row as OracleArmtd.solve (tol 1e-7), k_opt within 1e-8 where feasible"},
    }
    b.close()
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


def C_void(x):
    import ctypes
    return ctypes.c_void_p(x)


if __name__ == "__main__":
    main()
