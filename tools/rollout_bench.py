"""Measurement of closed-loop replanning episodes on the device (ReachSetEngine.rollout / armour_batch_rollout) on one GPU.

Workload: N worlds x 10 obstacles from worlds.random_episodes, a stated replan budget.  Reports, as one JSON document:
  - the wall time of armour_batch_rollout (host pointers, copies included; the call ends in a synchronise), Sum of replans
    over the worlds and world-replans per second, outcome counts, infeasible replans, build failures, the smallest clearance;
  - in the same run and alternated with it, a host-driven loop of the same steps: per replan the host-pointer build + solve
    of the running worlds (ReachSetEngine.build / solve), the waypoint and the advance in numpy (the device's arithmetic, operation
    for operation), the audit through ReachSetEngine.clearance.  Both loops must log the same k_opt and verdict rows; the tool
    fails otherwise.
The card's name and power limit are read (read-only) in the same run.

usage: python tools/rollout_bench.py [--worlds 1024] [--obstacles 10] [--replans 10] [--reps 2] [--out FILE]
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

from armour_b200 import ArmourError, ReachSetEngine, _lib, worlds  # noqa: E402

NF = 7
CONT = worlds.CONTINUOUS


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        out["nvidia_smi"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        out["nvidia_smi"] = repr(exc)
    return out


# ---- the device's arithmetic in numpy, operation for operation (bezier.cuh, rollout.cuh) ----------------------------------
def pw2(x): return x * x
def pw3(x): return x * x * x
def pw4(x): y = x * x; return y * y
def pw5(x): y = x * x; return y * y * x


def bez(q0, a, b, k, t):
    """(q, q', q'') of the Bezier at normalised time t (a = qd0 * D, b = qdd0 * D * D), as bez_q / bez_qd / bez_qdd"""
    B = [-pw5(t - 1), 5 * t * pw4(t - 1), -10 * pw2(t) * pw3(t - 1), 10 * pw3(t) * pw2(t - 1), -5 * pw4(t) * (t - 1), pw5(t)]
    dB = [pw4(t - 1.0) * -5.0, t * pw3(t - 1.0) * 2.0E+1 + pw4(t - 1.0) * 5.0,
          t * pw3(t - 1.0) * -2.0E+1 - (t * t) * pw2(t - 1.0) * 3.0E+1,
          pw3(t) * (t * 2.0 - 2.0) * 1.0E+1 + (t * t) * pw2(t - 1.0) * 3.0E+1, pw3(t) * (t - 1.0) * -2.0E+1 - pw4(t) * 5.0,
          pw4(t) * 5.0]
    u = 1.0 - t
    ddB = [20.0 * pw3(u), -40.0 * pw3(u) + 60.0 * t * pw2(u), 20.0 * pw3(u) - 120.0 * t * pw2(u) + 60.0 * pw2(t) * u,
           60.0 * t * pw2(u) - 120.0 * pw2(t) * u + 20.0 * pw3(t), 60.0 * pw2(t) * u - 40.0 * pw3(t), 20.0 * pw3(t)]
    beta1 = q0 + a / 5
    beta2 = q0 + (2 * a) / 5 + b / 20
    beta3 = q0 + k
    return tuple(C[0] * q0 + C[1] * beta1 + C[2] * beta2 + C[3] * beta3 + C[4] * beta3 + C[5] * beta3 for C in (B, dB, ddB))


def eval_plan(P, s, D=1.0):
    q, qd, qdd = bez(P[:, 0:7], P[:, 7:14] * D, P[:, 14:21] * D * D, P[:, 21:28], s)
    return q, qd / D, qdd / (D * D)


def goal_diff(q, goal):
    d = goal - q
    m = np.fmod(d + np.pi, 2 * np.pi)
    m = np.where((m != 0) & (m < 0), m + 2 * np.pi, m)
    return np.where(CONT[None, :], m - np.pi, d)


def seqnorm(d):
    s = np.zeros(d.shape[0])
    for j in range(NF):
        s = s + d[:, j] * d[:, j]
    return np.sqrt(s)


def host_loop(eng, start, goal, obs, R, S, lookahead=0.1, goal_radius=0.05, collision_tol=1e-4):
    """The episode loop driven from the host through the host-pointer build + solve; returns log_k, log_int, outcome, replans"""
    n = start.shape[0]
    k_range = np.full(NF, np.pi / 48)
    state = np.concatenate([start, np.zeros((n, 14))], axis=1)
    plan = np.concatenate([start, np.zeros((n, 21))], axis=1)
    outcome = np.full(n, -1, np.int32)
    replans = np.zeros(n, np.int32)
    log_k = np.full((R, n, NF), np.nan)
    log_int = np.full((R, n, 4), -1, np.int32)
    run = np.arange(n)
    lb = np.array([-1000.0, -2.41, -1000.0, -2.66, -1000.0, -2.23, -1000.0])  # raw position limits of the robot model
    ub, sp = -lb, worlds.SPEED_LIMITS
    for r in range(R):
        if run.size == 0:
            break
        st = state[run]
        d = goal_diff(st[:, :7], goal[run])
        nrm = seqnorm(d)
        at = nrm <= lookahead
        q_des = np.where(at[:, None], st[:, :7] + d, st[:, :7] + lookahead * d / np.where(at, 1.0, nrm)[:, None])
        try:
            eng.build(st[:, :7], st[:, 7:14], st[:, 14:21], obs[run])
        except ArmourError as e:
            if e.code != _lib.ERR_CAPACITY:
                raise
        bs = eng.build_status()
        k, ok, first, iters = eng.solve(q_des)
        log_k[r, run] = k
        log_int[r, run] = np.stack([ok.astype(np.int32), first, iters, bs], axis=1)
        P = plan[run]
        newP = np.concatenate([st, k_range * k], axis=1)
        P = np.where(ok[:, None], newP, P)
        samp = np.empty((run.size, S, NF))
        lim = np.zeros(run.size, bool)
        for m in range(S):
            q = np.empty((run.size, NF))
            qd = np.empty((run.size, NF))
            for grp in (True, False):
                sel = ok == grp
                s = (0.0 + (0.5 - 0.0) * float(m) / float(S - 1)) if grp else (0.5 + (1.0 - 0.5) * float(m) / float(S - 1))
                qa, qda, _ = eval_plan(P[sel], s)
                q[sel], qd[sel] = qa, qda
            samp[:, m] = q
            lim |= np.any(~CONT[None, :] & ((q < lb) | (q > ub)), axis=1) | np.any(np.abs(qd) > sp, axis=1)
        qa, qda, qdda = eval_plan(P, 0.5)
        q1, _, _ = eval_plan(P, 1.0)
        z = np.zeros_like(q1)
        nxt = np.where(ok[:, None], np.concatenate([qa, qda, qdda], axis=1), np.concatenate([q1, z, z], axis=1))
        P = np.where(ok[:, None], P, np.concatenate([q1, z, z, z], axis=1))
        state[run], plan[run] = nxt, P
        replans[run] = r + 1
        clr, _ = eng.clearance(samp.reshape(-1, NF), obs, np.repeat(run, S))
        cl = clr.reshape(run.size, S).min(axis=1)
        arrived = seqnorm(goal_diff(nxt[:, :7], goal[run])) <= goal_radius
        oc = np.where(cl < -collision_tol, 2, np.where(lim, 3, np.where(arrived, 1, np.where(r + 1 >= R, 0, -1))))
        outcome[run] = oc
        run = run[oc < 0]
    return log_k, log_int, outcome, replans


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worlds", type=int, default=1024)
    ap.add_argument("--obstacles", type=int, default=10)
    ap.add_argument("--replans", type=int, default=10)
    ap.add_argument("--audit-samples", type=int, default=16)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--seed", type=int, default=20261017)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("rollout_bench: no CUDA device (there is no CPU path)")
    n, nobs, R, S = a.worlds, a.obstacles, a.replans, a.audit_samples
    start, goal, obs = worlds.random_episodes(n, nobs, a.seed)
    eng = ReachSetEngine(max_problems=n, max_obstacles=nobs)
    # warm-up of both loops on a small batch and a short budget (loads the modules, allocates the grow-only scratch)
    eng.rollout(start, goal, obs, max_replans=1, audit_samples=S)
    host_loop(eng, start[:64], goal[:64], obs[:64], 1, S)
    dev_s, host_s, res = [], [], None
    for _ in range(a.reps):
        t0 = time.perf_counter()
        res = eng.rollout(start, goal, obs, max_replans=R, audit_samples=S)
        dev_s.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        hk, hi, ho, hr = host_loop(eng, start, goal, obs, R, S)
        host_s.append(time.perf_counter() - t0)
    same_k = bool(np.array_equal(hk, res["log_k"], equal_nan=True))
    same_i = bool(np.array_equal(hi, res["log_int"]))
    same_o = bool(np.array_equal(ho, res["outcome"]) and np.array_equal(hr, res["replans"]))
    total = int(res["replans"].sum())
    li = res["log_int"]
    planned = li[..., 0] >= 0
    dev, host = float(np.median(dev_s)), float(np.median(host_s))
    out = {
        "tool": "tools/rollout_bench.py",
        "card": card(),
        "workload": {"worlds": n, "obstacles": nobs, "max_replans": R, "audit_samples": S,
                     "generator": f"worlds.random_episodes(seed={a.seed})", "solver": "armour_solver_options_default"},
        "device_loop": {"seconds": dev_s, "seconds_median": dev, "world_replans": total, "world_replans_per_s": total / dev,
                        "timing": "wall clock around ReachSetEngine.rollout (armour_batch_rollout, host pointers, copies "
                                  "included, ends in a synchronise), alternated with the host-driven loop"},
        "host_driven_loop": {"seconds": host_s, "seconds_median": host, "world_replans_per_s": total / host,
                             "timing": "wall clock around the same episodes driven from Python: host-pointer build + solve per "
                                       "replan, numpy waypoint and advance, audit through ReachSetEngine.clearance"},
        "speedup_device_over_host_loop": host / dev,
        "outcomes": {"budget": int(np.sum(res["outcome"] == 0)), "arrived": int(np.sum(res["outcome"] == 1)),
                     "collision": int(np.sum(res["outcome"] == 2)), "limit": int(np.sum(res["outcome"] == 3))},
        "infeasible_replans": int(res["infeasible"].sum()),
        "build_failures": int(np.sum(li[..., 3][planned] != 0)),
        "min_clearance_m": float(np.min(res["min_clearance"])),
        "starts_in_collision": int(np.sum(eng.clearance(start, obs, np.arange(n))[0] < 0)),
        "host_loop_agrees": {"log_k": same_k, "log_int": same_i, "outcome_and_replans": same_o},
    }
    eng.close()
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    if not (same_k and same_i):
        sys.exit("rollout_bench: the device loop and the host-driven loop logged different plans")


if __name__ == "__main__":
    main()
