"""Planning-problem inputs: saved worlds, the armour.in text format and the synthetic generators of
the benchmark configurations (SURVEY.md §8d).

File formats follow the reference: world CSVs (kinova_src/saved_worlds/random/*.csv: row 1 start,
row 2 goal, row 3 NaN, rows 4+ `cx,cy,cz,sx,sy,sz,NaN`; obstacle zonotope = [c, diag(s/2)],
simulator/worlds/obstacles/box_obstacle_zonotope.m:21-26) and `armour.in` (4 lines of 7 `%.10f`,
the obstacle count, one line of 12 `%.10f` per obstacle: kinova_simulator_interfaces/uarmtd_planner.m:158-185,
parsed by kinova_planner_realtime/armour_main.cu:53-76).
"""
from __future__ import annotations

import numpy as np

NF = 7
STATE_LB = np.array([-np.pi, -2.41, -np.pi, -2.66, -np.pi, -2.23, -np.pi])  # continuous joints sampled in [-pi, pi]
STATE_UB = -STATE_LB
SPEED_LIMITS = np.array([1.3963, 1.3963, 1.3963, 1.3963, 1.2218, 1.2218, 1.2218])
CONTINUOUS = np.array([True, False, True, False, True, False, True])


def quantize(x):
    """Round-trip through the `%.10f` text MATLAB writes, so every consumer sees the same doubles."""
    a = np.asarray(x, dtype=np.float64)
    return np.array([float("%.10f" % v) for v in a.ravel()]).reshape(a.shape)


def boxes_to_zonotopes(boxes):
    """[n, 6] (centre, side lengths) -> [n, 12] (centre, 3 generators = diag(side/2), column-major Z)."""
    boxes = np.asarray(boxes, dtype=np.float64).reshape(-1, 6)
    out = np.zeros((boxes.shape[0], 12))
    out[:, 0:3] = boxes[:, 0:3]
    for a in range(3):
        out[:, 3 + 4 * a] = boxes[:, 3 + a] / 2
    return out


def load_world_csv(path):
    rows = np.genfromtxt(path, delimiter=",")
    start, goal = rows[0, :NF].copy(), rows[1, :NF].copy()
    return start, goal, boxes_to_zonotopes(rows[3:, :6])


def angdiff(a, b):
    """MATLAB angdiff(a, b): b - a wrapped to [-pi, pi]."""
    d = np.asarray(b) - np.asarray(a)
    return (d + np.pi) % (2 * np.pi) - np.pi


def straight_line_waypoint(q_cur, q_goal, lookahead=0.1):
    """robot_arm_straight_line_HLP.get_waypoint (simulator/planners/high_level_planners/...:45-57)."""
    d = np.asarray(q_goal, dtype=np.float64) - np.asarray(q_cur, dtype=np.float64)
    d[CONTINUOUS] = angdiff(np.asarray(q_cur)[CONTINUOUS], np.asarray(q_goal)[CONTINUOUS])
    return np.asarray(q_cur) + lookahead * d / np.linalg.norm(d)


def write_armour_in(path, q0, qd0, qdd0, q_des, obstacles):
    obstacles = np.asarray(obstacles, dtype=np.float64).reshape(-1, 12)
    with open(path, "w") as f:
        for v in (q0, qd0, qdd0, q_des):
            f.write("".join("%.10f " % x for x in v) + "\n")
        f.write("%d\n" % obstacles.shape[0])
        for o in obstacles:
            f.write("".join("%.10f " % x for x in o) + "\n")


def read_armour_in(path):
    tok = open(path).read().split()
    vals = [float(x) for x in tok[:4 * NF]]
    q0, qd0, qdd0, q_des = (np.array(vals[i * NF:(i + 1) * NF]) for i in range(4))
    nobs = int(tok[4 * NF])
    obs = np.array([float(x) for x in tok[4 * NF + 1:4 * NF + 1 + nobs * 12]]).reshape(nobs, 12)
    return q0, qd0, qdd0, q_des, obs


def config1_problem(csv_path):
    """BASELINE config 1: one saved world, qd0 = qdd0 = 0, straight-line waypoint, %.10f-quantised."""
    start, goal, obs = load_world_csv(csv_path)
    q_des = straight_line_waypoint(start, goal, 0.1)
    z = np.zeros(NF)
    return quantize(start), z, z.copy(), quantize(q_des), quantize(obs)


def random_problems(nprob, nobs, seed=20261017, moving=True):
    """BASELINE config 2 generator: random start / goal / motion state and `nobs` random boxes per problem."""
    q0, goal, qd0, qdd0, obs = _random_draws(nprob, nobs, seed, moving)
    q_des = np.stack([straight_line_waypoint(q0[p], goal[p]) for p in range(nprob)])
    return quantize(q0), quantize(qd0), quantize(qdd0), quantize(q_des), quantize(obs)


def random_episodes(nworlds, nobs, seed=20261017):
    """Closed-loop episodes from the draws of random_problems(nworlds, nobs, seed, moving=False): start, goal [n, 7] and
    obstacles [n, nobs, 12], %.10f-quantised like random_problems' outputs (start and obstacles equal its q0 and obstacles)."""
    q0, goal, _, _, obs = _random_draws(nworlds, nobs, seed, False)
    return quantize(q0), quantize(goal), quantize(obs)


PAD_CENTRE = np.array([10.0, 10.0, 10.0])  # m: far beyond the arm's reach (about 1.3 m from the base)
PAD_HALF_SIZE = 0.005


def pad_obstacles(obstacles, n):
    """Pad every world's obstacle list ([n_i, 12] each) to n obstacles with small boxes (1 cm) far outside the workspace, so
    that worlds with different counts form one batch.  Returns [len(obstacles), n, 12]; the padding boxes lie along x from
    PAD_CENTRE, one per slot."""
    out = np.empty((len(obstacles), n, 12))
    for w, o in enumerate(obstacles):
        o = np.asarray(o, dtype=np.float64).reshape(-1, 12)
        if o.shape[0] > n:
            raise ValueError(f"world {w} has {o.shape[0]} obstacles, more than {n}")
        out[w, :o.shape[0]] = o
        for s in range(o.shape[0], n):
            out[w, s] = 0.0
            out[w, s, 0:3] = PAD_CENTRE + np.array([0.1 * s, 0.0, 0.0])
            out[w, s, 3] = out[w, s, 7] = out[w, s, 11] = PAD_HALF_SIZE
    return out


def _random_draws(nprob, nobs, seed, moving):
    rng = np.random.default_rng(seed)
    q0 = rng.uniform(STATE_LB, STATE_UB, (nprob, NF))
    goal = rng.uniform(STATE_LB, STATE_UB, (nprob, NF))
    qd0 = rng.uniform(-0.5, 0.5, (nprob, NF)) * SPEED_LIMITS if moving else np.zeros((nprob, NF))
    qdd0 = rng.uniform(-1, 1, (nprob, NF)) if moving else np.zeros((nprob, NF))
    boxes = np.empty((nprob, nobs, 6))
    for p in range(nprob):
        n = 0
        while n < nobs:
            c = rng.uniform([-0.8, -0.8, 0.0], [0.8, 0.8, 1.2])
            s = rng.uniform(0.01, 0.5, 3)
            if np.all(np.abs(c - np.array([0, 0, 0.05])) <= s / 2 + 0.1):  # would swallow the robot base
                continue
            boxes[p, n] = np.concatenate([c, s])
            n += 1
    obs = boxes_to_zonotopes(boxes.reshape(-1, 6)).reshape(nprob, nobs, 12)
    return q0, goal, qd0, qdd0, obs


def halton_k(n, dim=NF, skip=1):
    """Deterministic k schedule in [-1, 1]^7 (Halton points) for exercising eval_g / eval_jac_g."""
    primes = [2, 3, 5, 7, 11, 13, 17][:dim]
    out = np.empty((n, dim))
    for j, b in enumerate(primes):
        for i in range(n):
            f, r, x = 1.0, 0.0, i + skip
            while x > 0:
                f /= b
                r += f * (x % b)
                x //= b
            out[i, j] = 2 * r - 1
    return out


# ---- inputs of the ARMTD comparison planner (SURVEY 8f-3) ------------------------------------------------------------------
ARMTD_T = 100  # KPA/Parameters.h:17


def armtd_k_range(qd0):
    """k_range of the constant-acceleration parameterisation, as ARMTD's offline tables define it: max(pi/24, |qd0| / 3)"""
    return np.maximum(np.pi / 24, np.abs(np.asarray(qd0, dtype=np.float64)) / 3)


def armtd_offline_jrs(qd0, k_range, T=ARMTD_T):
    """Synthetic stand-in for the reference's offline joint-reachable-set tables (generated with MATLAB / CORA by
    KPA/offline_jrs/create_orig_offline_jrs.m and sliced by load_offline_jrs.m: not in the reference tree).  For joint i and
    interval j it returns zonotope enclosures  cos(q_des - q0) in c + g*k +- r  (same for sin), k in [-1, 1], of the trajectory
    q_des(t) - q0 = qd0 t + k_a t^2 / 2 (t <= 0.5), braking to a stop at t = 1 afterwards, k_a = k_range * k: centre and slope from
    the interval's mid-time, r from the largest residual over a sample grid times 1.1.  Returns [6, 7, T] in the input file's
    order c_cos, g_cos, r_cos, c_sin, g_sin, r_sin (KPA/armtd_main.cu:70-88)."""
    qd0 = np.asarray(qd0, dtype=np.float64)
    k_range = np.asarray(k_range, dtype=np.float64)
    out = np.zeros((6, NF, T))
    ts = np.linspace(0.0, 1.0, 9)
    ks = np.linspace(-1.0, 1.0, 33)

    def coeffs(t):  # q_des - q0 = A(t) + B(t) * k_a
        if t <= 0.5:
            return qd0 * t, np.full(NF, 0.5 * t * t)
        tau = t - 0.5  # peak state, then constant deceleration -qd_peak / 0.5
        return qd0 * 0.5 + qd0 * tau - qd0 * tau * tau, 0.125 + 0.5 * tau - 0.5 * tau * tau

    for j in range(T):
        t0, t1 = j / T, (j + 1) / T
        A, B = coeffs(0.5 * (t0 + t1))
        c_cos, c_sin = np.cos(A), np.sin(A)
        g_cos, g_sin = -np.sin(A) * B * k_range, np.cos(A) * B * k_range
        r_cos, r_sin = np.zeros(NF), np.zeros(NF)
        for s in ts:
            At, Bt = coeffs(t0 + s * (t1 - t0))
            for k in ks:
                d = At + Bt * k_range * k
                r_cos = np.maximum(r_cos, np.abs(np.cos(d) - (c_cos + g_cos * k)))
                r_sin = np.maximum(r_sin, np.abs(np.sin(d) - (c_sin + g_sin * k)))
        out[:, :, j] = np.stack([c_cos, g_cos, 1.1 * r_cos + 1e-6, c_sin, g_sin, 1.1 * r_sin + 1e-6])
    return out


def armtd_offline_jrs_batch(qd0, k_range, T=ARMTD_T):
    """armtd_offline_jrs for n problems at once: qd0, k_range [n, 7] -> [n, 6, 7, T], the same arithmetic vectorised over the
    problems and the intervals."""
    qd0 = np.asarray(qd0, dtype=np.float64)[:, :, None]          # [n, 7, 1]
    k_range = np.asarray(k_range, dtype=np.float64)[:, :, None]
    j = np.arange(T, dtype=np.float64)
    t0, t1 = j / T, (j + 1) / T                                   # [T]

    def coeffs(t):  # as armtd_offline_jrs: q_des - q0 = A(t) + B(t) * k_a, t [T] -> A [n, 7, T], B [1, 1, T]
        tau = t - 0.5
        A = np.where(t <= 0.5, qd0 * t, qd0 * 0.5 + qd0 * tau - qd0 * tau * tau)
        B = np.where(t <= 0.5, 0.5 * t * t, 0.125 + 0.5 * tau - 0.5 * tau * tau)[None, None, :]
        return A, B

    A, B = coeffs(0.5 * (t0 + t1))
    c_cos, c_sin = np.cos(A), np.sin(A)
    g_cos, g_sin = -np.sin(A) * B * k_range, np.cos(A) * B * k_range
    r_cos, r_sin = np.zeros_like(A), np.zeros_like(A)
    for s in np.linspace(0.0, 1.0, 9):
        At, Bt = coeffs(t0 + s * (t1 - t0))
        for k in np.linspace(-1.0, 1.0, 33):
            d = At + Bt * k_range * k
            r_cos = np.maximum(r_cos, np.abs(np.cos(d) - (c_cos + g_cos * k)))
            r_sin = np.maximum(r_sin, np.abs(np.sin(d) - (c_sin + g_sin * k)))
    return np.stack([c_cos, g_cos, 1.1 * r_cos + 1e-6, c_sin, g_sin, 1.1 * r_sin + 1e-6], axis=1)


def armtd_random_problems(nprob, nobs, seed=20261017):
    """A sweep of comparison-planner problems: the start states, waypoints and `nobs` random boxes of random_problems(nprob,
    nobs, seed) with the synthetic offline JRS of each start velocity.  Returns q0, qd0, q_des, k_range [n, 7], jrs [n, 6, 7, 100]
    and obstacles [n, nobs, 12]."""
    q0, qd0, _, q_des, obs = random_problems(nprob, nobs, seed)
    k_range = armtd_k_range(qd0)
    return q0, qd0, q_des, k_range, armtd_offline_jrs_batch(qd0, k_range), obs


def armtd_problem(path, seed=0):
    """A planning problem of the comparison planner from a saved world: start from the CSV, a random initial velocity,
    straight-line waypoint, the synthetic offline JRS.  Returns q0, qd0, q_des, jrs[6, 7, T], k_range, obstacles."""
    q0, _, _, q_des, obs = config1_problem(path)
    rng = np.random.default_rng(seed)
    qd0 = np.round(rng.uniform(-0.4, 0.4, NF), 10)
    k_range = armtd_k_range(qd0)
    return q0, qd0, q_des, armtd_offline_jrs(qd0, k_range), k_range, obs


def write_armtd_in(path, q0, qd0, q_des, jrs, k_range, obstacles):
    """buffer/armtd.in as KPA/armtd_main.cu:54-103 parses it: q0, qd0, q_des, then per joint the six offline-JRS arrays
    (100 values each) followed by its k_range, the obstacle count and 12 numbers per obstacle."""
    obstacles = np.asarray(obstacles, dtype=np.float64).reshape(-1, 12)
    with open(path, "w") as f:
        for v in (q0, qd0, q_des):
            f.write(" ".join(repr(float(x)) for x in v) + "\n")
        for i in range(NF):
            for a in range(6):
                f.write(" ".join(repr(float(x)) for x in jrs[a, i]) + "\n")
            f.write(repr(float(k_range[i])) + "\n")
        f.write(f"{obstacles.shape[0]}\n")
        for o in obstacles:
            f.write(" ".join(repr(float(x)) for x in o) + "\n")
