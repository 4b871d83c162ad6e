"""numpy reference of the closed-loop episodes (armour_batch_rollout) and of the exact clearance (armour_batch_clearance),
written from the semantics in include/armour_b200.h and the robot model of armour_b200/csrc/robot_constants.h, sharing no code
with the library: the Bezier state update, the straight-line waypoint with its clamp at the goal, the forward kinematics of the
link boxes and the separating-axis test of two parallelepipeds."""
import numpy as np

NF = 7
CONTINUOUS = np.array([True, False, True, False, True, False, True])
T_MOVE = 0.5  # t_plan of the robot model (duration 1)
K_RANGE = np.full(NF, np.pi / 48)
STATE_LB = np.array([-1000.0, -2.41, -1000.0, -2.66, -1000.0, -2.23, -1000.0])
SPEED = np.array([1.3963, 1.3963, 1.3963, 1.3963, 1.2218, 1.2218, 1.2218])

_TRANS = np.array([0, 0, 0.15643, 0, 0.005375, -0.12838, 0, -0.21038, -0.006375, 0, 0.006375, -0.21038, 0, -0.20843,
                   -0.006375, 0, 0.00017505, -0.10593, 0, -0.10593, -0.00017505, 0, 0, 0]).reshape(8, 3)
_LC = np.array([0.000000, -0.001297, -0.088375, 0.000000, -0.089400, -0.007877, 0.000000, -0.001502, -0.129375, 0.000000,
                -0.087450, -0.013648, 0.000001, -0.009023, -0.071752, 0.000000, -0.041661, -0.009251, 0.000000, -0.018585,
                -0.033462, 0.0, -0.00, -0.0]).reshape(8, 3)
_LG = np.array([0.046358, 0.047354, 0.086000, 0.046000, 0.135400, 0.047501, 0.046000, 0.047501, 0.127000, 0.046000, 0.133450,
                0.042293, 0.034999, 0.044023, 0.069252, 0.035000, 0.076739, 0.044076, 0.045500, 0.056085, 0.030963, 0.07, 0.09,
                0.07]).reshape(8, 3)


def _rpy(roll, pitch, yaw):
    cr, sr, cp, sp, cy, sy = np.cos(roll), np.sin(roll), np.cos(pitch), np.sin(pitch), np.cos(yaw), np.sin(yaw)
    return np.array([[cp * cy, -cp * sy, sp],
                     [cr * sy + cy * sp * sr, cr * cy - sp * sr * sy, -cp * sr],
                     [sr * sy - cr * cy * sp, cy * sr + cr * sp * sy, cp * cr]])


def robot(model=0):
    """(trans [NJ, 3], rrpy [NJ, 3, 3], link centre [NJ, 3], link half-extents [NJ, 3]) of robot model 0 (7 links) or 1
    (with the fixed gripper link)."""
    nj = 8 if model == 1 else 7
    trans = _TRANS[:nj].copy()
    if model == 1:
        trans[7, 2] = -0.061525 - 0.10155
    rrpy = np.stack([_rpy(np.pi if i == 0 else (np.pi / 2 if i % 2 == 1 else -np.pi / 2), 0.0, 0.0) for i in range(nj)])
    return trans, rrpy, _LC[:nj], _LG[:nj]


def link_boxes(q, model=0):
    """Exact link boxes of configuration q: centres [NJ, 3], generator columns [NJ, 3 generators, 3]."""
    trans, rrpy, lc, lg = robot(model)
    R, T = np.eye(3), np.zeros(3)
    cs, gs = [], []
    for i in range(trans.shape[0]):
        T = T + R @ trans[i]
        J = rrpy[i]
        if i < NF:
            c, s = np.cos(q[i]), np.sin(q[i])
            J = J @ np.array([[c, -s, 0], [s, c, 0], [0, 0, 1.0]])
        R = R @ J
        cs.append(T + R @ lc[i])
        gs.append((R * lg[i][None, :]).T)
    return np.array(cs), np.array(gs)


def sat_clearance(ca, A, cb, B):
    """Signed clearance of two parallelepipeds (centre, generators as rows): the largest gap over the 15 separating axes."""
    d = np.asarray(cb) - np.asarray(ca)
    axes = [np.cross(A[a], A[b]) for a, b in ((0, 1), (1, 2), (0, 2))]
    axes += [np.cross(B[a], B[b]) for a, b in ((0, 1), (1, 2), (0, 2))]
    axes += [np.cross(A[a], B[b]) for a in range(3) for b in range(3)]
    best = -np.inf
    for n in axes:
        nn = np.sqrt(n @ n)
        if nn < 1e-12:
            continue
        gap = (abs(d @ n) - np.sum(np.abs(A @ n)) - np.sum(np.abs(B @ n))) / nn
        best = max(best, gap)
    return best


def zono(z):
    z = np.asarray(z, dtype=np.float64)
    return z[:3], z[3:12].reshape(3, 3)


def clearance(q, obstacles, model=0):
    """(smallest clearance, l * nobs + o of the first pair attaining it) of configuration q; (inf, -1) without obstacles."""
    obstacles = np.asarray(obstacles).reshape(-1, 12)
    cs, gs = link_boxes(q, model)
    best, which = np.inf, -1
    for l in range(cs.shape[0]):
        for o in range(obstacles.shape[0]):
            cb, B = zono(obstacles[o])
            v = sat_clearance(cs[l], gs[l], cb, B)
            if v < best:
                best, which = v, l * obstacles.shape[0] + o
    return best, which


def angdiff(a, b):
    d = np.asarray(b) - np.asarray(a)
    return (d + np.pi) % (2 * np.pi) - np.pi


def goal_diff(q, goal):
    d = np.asarray(goal, dtype=np.float64) - np.asarray(q, dtype=np.float64)
    d[CONTINUOUS] = angdiff(np.asarray(q)[CONTINUOUS], np.asarray(goal)[CONTINUOUS])
    return d


def waypoint(q, goal, lookahead=0.1):
    """The straight-line waypoint, or the goal itself (q + d) within lookahead of it."""
    d = goal_diff(q, goal)
    n = np.linalg.norm(d)
    return q + d if n <= lookahead else q + lookahead * d / n


def bezier(q0, qd0, qdd0, k, s):
    """(q, qd, qdd) at normalised time s of the degree-5 Bezier with q(0) = q0, q'(0) = qd0, q''(0) = qdd0, q(1) = q0 + k,
    q'(1) = q''(1) = 0 (duration 1): the control points and Bernstein derivatives written out independently."""
    b = np.stack([q0, q0 + qd0 / 5, q0 + 2 * qd0 / 5 + qdd0 / 20, q0 + k, q0 + k, q0 + k])  # [6, 7]
    from math import comb
    B = np.array([comb(5, i) * s ** i * (1 - s) ** (5 - i) for i in range(6)])
    d1 = 5 * (b[1:] - b[:-1])
    B4 = np.array([comb(4, i) * s ** i * (1 - s) ** (4 - i) for i in range(5)])
    d2 = 4 * (d1[1:] - d1[:-1])
    B3 = np.array([comb(3, i) * s ** i * (1 - s) ** (3 - i) for i in range(4)])
    return B @ b, B4 @ d1, B3 @ d2
