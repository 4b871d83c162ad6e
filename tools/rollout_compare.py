"""ARMOUR against its ARMTD comparison planner in closed loop, on the same worlds and under the same audit, on one GPU: the
question the reference's system test (kinova_run_100_worlds.m -> simulator_armtd.run) asks of the two planners.

Workload: N worlds x 10 obstacles from worlds.random_episodes; worlds whose start already intersects an obstacle (exact
clearance, ReachSetEngine.clearance) are dropped and counted.  Both planners run the kept worlds with the same replan budget,
audit samples, collision_tol and max_iter (each with its own solver tolerance: 1e-4 for ARMOUR, KPA's 1e-7 for ARMTD),
alternated over the reps.  Reports, as one JSON document, per planner: outcome counts, infeasible replans, build failures, the
median replans to arrival, the smallest audited clearance and world-replans per second (wall clock around ReachSetEngine.rollout /
ArmtdBatch.rollout, host pointers, copies included, the call ends in a synchronise).  Also: CUDA-event times of the stand-in
table kernel (armour_armtd_offline_jrs_device) and of the ARMTD build (armour_armtd_batch_build_device) at N worlds, and the
card's name and power limit, read in the same run.

usage: python tools/rollout_compare.py [--worlds 1024] [--obstacles 10] [--replans 40] [--reps 2] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True
import numpy as np  # noqa: E402
import torch  # noqa: E402

from armour_b200 import ArmtdBatch, ReachSetEngine, _lib, worlds  # noqa: E402
from rollout_bench import card  # noqa: E402


def summary(res, seconds):
    li = res["log_int"]
    planned = li[..., 0] >= 0
    arrived = res["outcome"] == _lib.ROLLOUT_ARRIVED
    total = int(res["replans"].sum())
    med = float(np.median(seconds))
    return {
        "outcomes": {"budget": int(np.sum(res["outcome"] == _lib.ROLLOUT_BUDGET)), "arrived": int(np.sum(arrived)),
                     "collision": int(np.sum(res["outcome"] == _lib.ROLLOUT_COLLISION)),
                     "limit": int(np.sum(res["outcome"] == _lib.ROLLOUT_LIMIT))},
        "infeasible_replans": int(res["infeasible"].sum()),
        "build_failures": int(np.sum(li[..., 3][planned] != 0)),
        "median_replans_to_arrival": float(np.median(res["replans"][arrived])) if np.any(arrived) else None,
        "min_clearance_m": float(np.min(res["min_clearance"])),
        "world_replans": total,
        "seconds": seconds,
        "seconds_median": med,
        "world_replans_per_s": total / med,
    }


def event_ms(fn, reps, stream):
    """mean CUDA-event time of fn() over reps launches on `stream`, after one warm-up launch"""
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(reps):
        fn()
    b.record(stream)
    b.synchronize()
    return a.elapsed_time(b) / reps


def table_and_build(b, n, nobs, seed):
    """CUDA-event times (ms) of the stand-in table kernel and of the ARMTD device build for n worlds on b's context, both on
    one torch stream; moving start states of worlds.random_problems, so k_range > pi / 24 on some joints."""
    q0, qd0, _, _, obs = worlds.random_problems(n, nobs, seed)
    kr = worlds.armtd_k_range(qd0)
    dev = torch.device("cuda", 0)
    dq0, dqd0, dkr, dobs = (torch.as_tensor(np.ascontiguousarray(x), device=dev) for x in (q0, qd0, kr, obs))
    djrs = torch.empty((n, 6, 7, 100), dtype=torch.float64, device=dev)
    stream = torch.cuda.Stream(dev)  # not the legacy default stream: a NULL handle would leave the context on its own stream
    b.lib.armour_ctx_set_stream(b._h, C.c_void_p(stream.cuda_stream))
    torch.cuda.synchronize(dev)
    table = event_ms(lambda: b.offline_jrs_device(n, dqd0.data_ptr(), dkr.data_ptr(), djrs.data_ptr()), 20, stream)
    build = event_ms(lambda: b.build_device(n, nobs, dq0.data_ptr(), dqd0.data_ptr(), djrs.data_ptr(), dkr.data_ptr(),
                                            dobs.data_ptr()), 5, stream)
    b.synchronize()
    ok = bool(np.array_equal(djrs.cpu().numpy()[:8], b.offline_jrs(qd0[:8], kr[:8])))
    return {"worlds": n, "table_ms": table, "table_us_per_world": 1e3 * table / n, "build_ms": build,
            "build_us_per_world": 1e3 * build / n, "table_over_build": table / build,
            "sincos_per_call": n * 7 * 100 * (9 * 33 + 1),
            "timing": "CUDA events around 20 table launches / 5 builds on one stream, after a warm-up launch; the build "
                      "is armour_armtd_batch_build_device with the device's sincos (its own k_armtd_jrs, k_reachsets_fk, "
                      "k_hyperplanes)", "device_table_equals_host_call": ok}


def armtd_contact_link(eng, res, w, obs_w, S):
    """link of the smallest clearance over the audit samples of world w's last executed ARMTD segment (the plan of the last
    feasible replan, over [0, 0.5] if that is the last replan, else its braking half), recomputed from the logs"""
    r = res["replans"][w] - 1
    rp = max(x for x in range(r + 1) if res["log_int"][x, w, 0])
    st = res["log_state"][rp, w]
    q0, qd0 = st[:7], st[7:14]
    k_a = worlds.armtd_k_range(qd0) * res["log_k"][rp, w]
    t0, t1 = (0.0, 0.5) if rp == r else (0.5, 1.0)
    q = []
    for t in t0 + (t1 - t0) * np.arange(S) / (S - 1):
        if t <= 0.5:
            q.append(q0 + qd0 * t + k_a * t * t / 2)
        else:
            qp, vp, tau = q0 + qd0 * 0.5 + k_a * 0.125, qd0 + k_a * 0.5, t - 0.5
            q.append(qp + vp * tau - vp * tau * tau)
    clr, which = eng.clearance(np.stack(q), obs_w)
    return int(which[np.argmin(clr)] // obs_w.shape[0])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worlds", type=int, default=1024)
    ap.add_argument("--obstacles", type=int, default=10)
    ap.add_argument("--replans", type=int, default=40)
    ap.add_argument("--audit-samples", type=int, default=16)
    ap.add_argument("--max-iter", type=int, default=60)
    ap.add_argument("--collision-tol", type=float, default=1e-4)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--seed", type=int, default=20261017)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("rollout_compare: no CUDA device (there is no CPU path)")
    n, nobs, R, S = a.worlds, a.obstacles, a.replans, a.audit_samples
    start, goal, obs = worlds.random_episodes(n, nobs, a.seed)
    eng = ReachSetEngine(max_problems=n, max_obstacles=nobs)
    c0, _ = eng.clearance(start, obs, np.arange(n))
    keep = np.flatnonzero(c0 > 0)
    start, goal, obs = start[keep], goal[keep], obs[keep]
    b = ArmtdBatch(max_problems=n, max_obstacles=nobs)
    common = dict(audit_samples=S, max_iter=a.max_iter, collision_tol=a.collision_tol)
    runs = {"armour": lambda r: eng.rollout(start, goal, obs, max_replans=r, **common),
            "armtd": lambda r: b.rollout(start, goal, obs, max_replans=r, **common)}
    for run in runs.values():  # warm-up: loads the modules, allocates the grow-only scratch
        run(1)
    seconds = {k: [] for k in runs}
    res = {}
    for _ in range(a.reps):
        for name, run in runs.items():
            t0 = time.perf_counter()
            res[name] = run(R)
            seconds[name].append(time.perf_counter() - t0)
    out = {
        "tool": "tools/rollout_compare.py",
        "card": card(),
        "workload": {"worlds_drawn": n, "worlds": int(keep.size), "starts_in_collision_dropped": int(n - keep.size),
                     "obstacles": nobs, "max_replans": R, "audit_samples": S, "max_iter": a.max_iter,
                     "collision_tol": a.collision_tol, "solver_tol": {"armour": 1e-4, "armtd": 1e-7},
                     "generator": f"worlds.random_episodes(seed={a.seed}), starts with clearance > 0"},
        "timing": "wall clock around each planner's rollout call (host pointers, copies included, ends in a synchronise), "
                  "the two planners alternated over the reps",
        "armour": summary(res["armour"], seconds["armour"]),
        "armtd": summary(res["armtd"], seconds["armtd"]),
        "armtd_table_and_build": table_and_build(b, n, nobs, a.seed),
    }
    hit = np.flatnonzero(res["armtd"]["outcome"] == _lib.ROLLOUT_COLLISION)
    if hit.size:  # the link that touched, over the audit samples of the last segment
        out["armtd"]["collision_links"] = [armtd_contact_link(eng, res["armtd"], w, obs[w], S) for w in hit]
    eng.close()
    b.close()
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
