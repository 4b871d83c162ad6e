"""numpy reference of the episodes of the ARMTD comparison planner (armour_armtd_batch_rollout), written from the semantics in
include/armour_b200.h and sharing no code with the library: the constant-acceleration trajectory, k_range of a planning state
and the replay of an episode's executed segments from its logs alone."""
import numpy as np

NF = 7
T_MOVE = 0.5


def k_range(qd0):
    """max(pi / 24, |qd0| / 3) per joint"""
    return np.maximum(np.pi / 24, np.abs(np.asarray(qd0, dtype=np.float64)) / 3)


def const_acc(q0, qd0, k_a, t):
    """(q, qd) at time t in [0, 1] of the trajectory that accelerates at k_a up to t = 0.5 and then brakes at a constant rate
    to rest at t = 1: q0 + qd0 t + k_a t^2 / 2, then q_peak + qd_peak tau - qd_peak tau^2 with tau = t - 0.5."""
    q0, qd0, k_a = (np.asarray(a, dtype=np.float64) for a in (q0, qd0, k_a))
    if t <= T_MOVE:
        return q0 + qd0 * t + k_a * t * t / 2, qd0 + k_a * t
    q_peak = q0 + qd0 * T_MOVE + k_a * T_MOVE * T_MOVE / 2
    qd_peak = qd0 + k_a * T_MOVE
    tau = t - T_MOVE
    return q_peak + qd_peak * tau - qd_peak * tau * tau, qd_peak - 2 * qd_peak * tau


def replay(res, start):
    """The executed plan of every (replan, world) from the logs alone: seg[r, w] = ((q0, qd0, k_a), t0, t1), and the state
    after the segment nxt[r, w] = (q, qd, 0) [21]."""
    R, n = res["log_k"].shape[:2]
    cur = [(np.asarray(start[w], dtype=np.float64).copy(), np.zeros(NF), np.zeros(NF)) for w in range(n)]  # rest at the start
    seg, nxt = {}, {}
    for r in range(R):
        for w in range(n):
            if r >= res["replans"][w]:
                continue
            st = res["log_state"][r, w]
            if res["log_int"][r, w, 0]:
                cur[w] = (st[:NF], st[NF:2 * NF], k_range(st[NF:2 * NF]) * res["log_k"][r, w])
                seg[r, w] = (cur[w], 0.0, T_MOVE)
                q, qd = const_acc(*cur[w], T_MOVE)
            else:
                seg[r, w] = (cur[w], T_MOVE, 1.0)
                q, qd = const_acc(*cur[w], 1.0)[0], np.zeros(NF)
                cur[w] = (q, np.zeros(NF), np.zeros(NF))
            nxt[r, w] = np.concatenate([q, qd, np.zeros(NF)])
    return seg, nxt
