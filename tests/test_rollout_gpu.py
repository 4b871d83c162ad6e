"""Closed-loop replanning episodes on the device (armour_batch_rollout) and the exact clearance kernel (armour_batch_clearance).

Every replan of an episode must be the existing planner, bit for bit: the sub-batch of worlds still running at replan r,
rebuilt in ascending world order from the logged planning states, plans the logged k_opt and verdict through the host-pointer
build + solve.  The state update and the waypoint are checked against the numpy reference of tests/rollout_ref.py, the audit
against its forward kinematics and separating-axis test, the plans against the CPU oracle."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import WORLDS
from rollout_ref import K_RANGE, T_MOVE, bezier, clearance, goal_diff, link_boxes, waypoint

pytestmark = pytest.mark.gpu

KEYS = ("outcome", "replans", "infeasible", "final_state", "min_clearance", "log_state", "log_q_des", "log_k", "log_int",
        "log_clearance")


def _random_obstacles(rng, n, general):
    out = np.zeros((n, 12))
    out[:, 0:3] = rng.uniform([-0.6, -0.6, 0.0], [0.6, 0.6, 1.1], (n, 3))
    for o in range(n):
        G = np.diag(rng.uniform(0.02, 0.2, 3))
        if general:  # a general parallelepiped: sheared and rotated generators
            G = rng.uniform(-0.15, 0.15, (3, 3)) + G
        out[o, 3:12] = G.T.ravel()  # generator columns, column-major as the zonotopes of the ABI
    return out


@pytest.mark.parametrize("model", [0, 1])
def test_clearance_matches_the_numpy_reference(built, model):
    from armour_b200 import ReachSetEngine
    rng = np.random.default_rng(11 + model)
    nsets, nobs, n = 4, 6, 48
    obs = np.stack([_random_obstacles(rng, nobs, general=s % 2 == 1) for s in range(nsets)])
    q = rng.uniform(-np.pi, np.pi, (n, 7))
    world = rng.integers(0, nsets, n)
    eng = ReachSetEngine(max_problems=1, max_obstacles=nobs, robot_model=model)
    clr, which = eng.clearance(q, obs, world)
    for i in range(n):
        ref, ref_which = clearance(q[i], obs[world[i]], model)
        assert abs(clr[i] - ref) <= 1e-12, (i, clr[i], ref)
        assert which[i] == ref_which, (i, which[i], ref_which)
    assert np.any(clr < 0) and np.any(clr > 0), "expected both intersecting and separated configurations"
    # world=None is obstacle set 0
    c0, w0 = eng.clearance(q[:5], obs[0])
    c1, w1 = eng.clearance(q[:5], obs, np.zeros(5, np.int32))
    assert np.array_equal(c0, c1) and np.array_equal(w0, w1)


def test_clearance_of_constructed_cases(built):
    from armour_b200 import ReachSetEngine
    eng = ReachSetEngine(max_problems=1, max_obstacles=4)
    q = np.zeros(7)  # the arm stretched upwards: every link box axis-aligned
    cs, gs = link_boxes(q)
    top = np.abs(gs[:, :, 2]).sum(axis=1) + cs[:, 2]
    lt = int(np.argmax(top))
    for gap in (0.2, 0.01, 0.0, -0.01):
        box = np.zeros(12)  # a wide slab whose underside is `gap` above the highest point of the arm
        box[0:3] = [cs[lt, 0], cs[lt, 1], top[lt] + gap + 0.05]
        box[3], box[7], box[11] = 0.4, 0.4, 0.05
        far = np.zeros(12)
        far[0:3] = [5.0, 0.0, 0.0]
        far[3] = far[7] = far[11] = 0.1
        clr, which = eng.clearance(q, np.stack([far, box]))
        assert abs(clr[0] - gap) <= 1e-12, (gap, clr[0])
        assert which[0] == lt * 2 + 1
    clr, which = eng.clearance(np.zeros((3, 7)), np.zeros((0, 12)))
    assert np.all(np.isinf(clr)) and np.all(clr > 0) and np.all(which == -1)


def _numpy_replay(res, start):
    """The executed plan of every (replan, world) from the logs alone: (plan (q0, qd0, qdd0, k in rad), s0, s1), and the
    state after the segment."""
    R, n = res["log_k"].shape[:2]
    cur = [(start[w].copy(), np.zeros(7), np.zeros(7), np.zeros(7)) for w in range(n)]  # the rest plan at the start
    seg, nxt = {}, {}
    for r in range(R):
        for w in range(n):
            if r >= res["replans"][w]:
                continue
            st = res["log_state"][r, w]
            if res["log_int"][r, w, 0]:
                cur[w] = (st[:7], st[7:14], st[14:21], K_RANGE * res["log_k"][r, w])
                seg[r, w] = (cur[w], 0.0, T_MOVE)
                q, qd, qdd = bezier(*cur[w], T_MOVE)
            else:
                seg[r, w] = (cur[w], T_MOVE, 1.0)
                q, qd, qdd = bezier(*cur[w], 1.0)[0], np.zeros(7), np.zeros(7)
                cur[w] = (q, np.zeros(7), np.zeros(7), np.zeros(7))
            nxt[r, w] = np.concatenate([q, qd, qdd])
    return seg, nxt


@pytest.fixture(scope="module")
def episodes16(built):
    from armour_b200 import ReachSetEngine, worlds
    start, goal, obs = worlds.random_episodes(16, 20, seed=5)
    eng = ReachSetEngine(max_problems=16, max_obstacles=20)
    res = eng.rollout(start, goal, obs, max_replans=12)
    return eng, start, goal, obs, res


def test_each_replan_is_the_existing_planner(episodes16):
    from armour_b200 import ArmourError
    eng, start, goal, obs, res = episodes16
    R = 12
    li = res["log_int"]
    planned = np.arange(R)[:, None] < res["replans"][None, :]
    assert np.all(res["replans"] >= 1) and np.all(res["replans"] <= R)
    assert np.any(li[..., 0][planned] == 1) and np.any(li[..., 0][planned] == 0), "seed 5: feasible and infeasible replans"
    assert np.all(np.isnan(res["log_k"][~planned])) and np.all(li[~planned] == -1)
    assert np.array_equal(res["infeasible"], ((li[..., 0] == 0) & planned).sum(axis=0))
    seg, nxt = _numpy_replay(res, start)
    for r in range(R):
        idx = np.flatnonzero(res["replans"] > r)
        if idx.size == 0:
            break
        st = res["log_state"][r, idx]
        try:
            eng.build(st[:, :7], st[:, 7:14], st[:, 14:21], obs[idx])
        except ArmourError as e:  # a table overflowed: the rollout logged it and the solve below is fail-safe
            assert e.code == -4
        assert np.array_equal(eng.build_status(), li[r, idx, 3])
        k, ok, first, iters = eng.solve(res["log_q_des"][r, idx])
        assert np.array_equal(k, res["log_k"][r, idx]), r
        assert np.array_equal(ok.astype(np.int32), li[r, idx, 0]) and np.array_equal(first, li[r, idx, 1])
        assert np.array_equal(iters, li[r, idx, 2])
        for j, w in enumerate(idx):
            assert np.max(np.abs(res["log_q_des"][r, w] - waypoint(st[j, :7], goal[w]))) <= 1e-13
            after = res["log_state"][r + 1, w] if r + 1 < res["replans"][w] else res["final_state"][w]
            assert np.max(np.abs(after - nxt[r, w])) <= 1e-12, (r, w)
            if not li[r, w, 0]:
                assert not np.any(after[7:])
    assert np.array_equal(res["log_state"][0], np.concatenate([start, np.zeros((16, 14))], axis=1))


def test_rollout_is_deterministic_and_worlds_are_independent(episodes16):
    eng, start, goal, obs, res = episodes16
    again = eng.rollout(start, goal, obs, max_replans=12)
    for key in KEYS:
        assert np.array_equal(res[key], again[key], equal_nan=True), key
    perm = np.random.default_rng(2).permutation(16)
    p = eng.rollout(start[perm], goal[perm], obs[perm], max_replans=12)
    for key in KEYS:
        a = res[key]
        if a.ndim >= 2 and key.startswith("log_"):
            assert np.array_equal(p[key], a[:, perm], equal_nan=True), key
        else:
            assert np.array_equal(p[key], a[perm], equal_nan=True), key


def test_logged_plans_agree_with_the_oracle(episodes16):
    from oracle.pyoracle import OracleProblem
    eng, start, goal, obs, res = episodes16
    pairs = [(r, w) for w in range(16) for r in range(res["replans"][w]) if res["log_int"][r, w, 3] == 0]
    rng = np.random.default_rng(4)
    pick = [pairs[i] for i in rng.choice(len(pairs), 4, replace=False)]
    fe = [p for p in pairs if res["log_int"][p[0], p[1], 0]]
    if not any(res["log_int"][r, w, 0] for r, w in pick):
        pick[-1] = fe[0]
    for r, w in pick:
        st = res["log_state"][r, w]
        orc = OracleProblem().build(st[:7], st[7:14], st[14:21], obs[w])
        k, ok, first, _ = orc.solve(res["log_q_des"][r, w])
        assert ok == bool(res["log_int"][r, w, 0]), (r, w)
        assert np.max(np.abs(k - res["log_k"][r, w])) <= 1e-8, (r, w, k, res["log_k"][r, w])
        if ok:  # the oracle's own verdict accepts the logged plan
            good, row = orc.verdict(orc.eval_g(res["log_k"][r, w]))
            assert good, (r, w, row)


def test_certified_motion_is_collision_free(built):
    """64 worlds whose start is collision-free (a world that starts inside an obstacle collides whatever is planned), 10
    obstacles, 30 replans, 32 audit samples: no executed segment hits an obstacle or exceeds a limit."""
    from armour_b200 import ReachSetEngine, _lib, worlds
    start, goal, obs = worlds.random_episodes(160, 10, seed=20261020)
    eng = ReachSetEngine(max_problems=64, max_obstacles=10)
    c0, _ = eng.clearance(start, obs, np.arange(160))
    keep = np.flatnonzero(c0 > 0)[:64]
    assert keep.size == 64
    start, goal, obs = start[keep], goal[keep], obs[keep]
    res = eng.rollout(start, goal, obs, max_replans=30, audit_samples=32)
    assert not np.any(res["outcome"] == _lib.ROLLOUT_COLLISION), np.flatnonzero(res["outcome"] == _lib.ROLLOUT_COLLISION)
    assert not np.any(res["outcome"] == _lib.ROLLOUT_LIMIT)
    lc = res["log_clearance"]
    assert np.all(lc[~np.isnan(lc)] >= -1e-4)
    assert np.array_equal(res["min_clearance"], np.nanmin(lc, axis=0))
    seg, _ = _numpy_replay(res, start)
    keys = sorted(seg)
    rng = np.random.default_rng(9)
    chosen = [keys[i] for i in rng.choice(len(keys), 5, replace=False)]
    chosen += [k for k in keys if not res["log_int"][k[0], k[1], 0]][:1]  # a braking segment too
    for r, w in chosen:
        plan, s0, s1 = seg[r, w]
        ref = min(clearance(bezier(*plan, s)[0], obs[w])[0] for s in s0 + (s1 - s0) * np.arange(32) / 31)
        assert abs(ref - lc[r, w]) <= 1e-12, (r, w, ref, lc[r, w])


def test_episodes_end_as_specified(built):
    from armour_b200 import ReachSetEngine, _lib, worlds
    eng = ReachSetEngine(max_problems=2, max_obstacles=10)
    start = np.array([0.3, 0.4, -0.2, 1.2, 0.1, 0.6, -0.4])
    v = np.array([1.0, -0.5, 0.8, 0.6, -1.0, 0.4, 0.9])
    goal = start + 0.3 * v / np.linalg.norm(v)
    pad = worlds.pad_obstacles([np.zeros((0, 12))], 10)
    res = eng.rollout(start[None], goal[None], pad, max_replans=40)
    assert res["outcome"][0] == _lib.ROLLOUT_ARRIVED
    n = res["replans"][0]
    assert res["infeasible"][0] == 0 and np.all(res["log_int"][:n, 0, 0] == 1)
    assert np.linalg.norm(goal_diff(res["final_state"][0, :7], goal)) <= 0.05
    assert res["min_clearance"][0] > 5.0

    # a saved world padded from 6 to 10 obstacles plans what the world itself plans
    s, g, o = worlds.load_world_csv(os.path.join(WORLDS, "scene_013_001.csv"))
    assert o.shape[0] == 6
    a = eng.rollout(s[None], g[None], o[None], max_replans=6)
    b = eng.rollout(s[None], g[None], worlds.pad_obstacles([o], 10), max_replans=6)
    assert np.array_equal(a["replans"], b["replans"])
    n = a["replans"][0]
    assert np.max(np.abs(a["log_k"][:n] - b["log_k"][:n])) <= 1e-9
    assert np.array_equal(a["log_int"][:n, :, 0], b["log_int"][:n, :, 0])


def test_argument_errors(built):
    from armour_b200 import ArmourError, ArmtdBatch, ReachSetEngine, _lib
    eng = ReachSetEngine(max_problems=2, max_obstacles=3)
    s = np.zeros((2, 7))
    o = np.zeros((2, 3, 12))
    with pytest.raises(ArmourError) as e:
        eng.rollout(np.zeros((3, 7)), np.zeros((3, 7)), np.zeros((3, 3, 12)))
    assert e.value.code == _lib.ERR_STATE
    with pytest.raises(ArmourError) as e:
        eng.rollout(s, s, np.zeros((2, 4, 12)))
    assert e.value.code == _lib.ERR_OBSTACLES
    for kw in (dict(max_replans=0), dict(audit_samples=1), dict(lookahead=0.0), dict(goal_radius=-1.0), dict(max_iter=0)):
        with pytest.raises(ArmourError) as e:
            eng.rollout(s, s, o, **kw)
        assert e.value.code == _lib.ERR_ARG, kw
    lib = eng.lib
    opt = _lib.RolloutOptions()
    lib.armour_rollout_options_default(C.byref(opt))
    assert (opt.max_replans, opt.audit_samples, opt.lookahead, opt.goal_radius) == (100, 16, 0.1, 0.05)
    out = _lib.RolloutOut()
    dp = s.ctypes.data_as(_lib.dp)
    assert lib.armour_batch_rollout(eng._h, 2, None, dp, o.ctypes.data_as(_lib.dp), 3, C.byref(opt), C.byref(out)) == _lib.ERR_ARG
    assert lib.armour_batch_rollout(eng._h, 2, dp, dp, None, 3, C.byref(opt), C.byref(out)) == _lib.ERR_ARG
    assert lib.armour_batch_rollout(eng._h, 2, dp, dp, None, 0, None, C.byref(out)) == _lib.ERR_ARG
    opt.struct_size = 8
    assert lib.armour_batch_rollout(eng._h, 2, dp, dp, None, 0, C.byref(opt), C.byref(out)) == _lib.ERR_ARG
    with pytest.raises(ArmourError) as e:
        eng.clearance(np.zeros(7), np.zeros((4, 12)))
    assert e.value.code == _lib.ERR_OBSTACLES
    c = np.zeros(1)
    assert lib.armour_batch_clearance(eng._h, 1, None, None, None, 0, c.ctypes.data_as(_lib.dp), None) == _lib.ERR_ARG
    assert lib.armour_batch_clearance(eng._h, 0, dp, None, None, 0, c.ctypes.data_as(_lib.dp), None) == _lib.ERR_ARG
    # the episodes run the main planner: a context of the ARMTD comparison planner is refused
    armtd = ArmtdBatch(max_problems=2, max_obstacles=3)
    lib.armour_rollout_options_default(C.byref(opt))
    assert lib.armour_batch_rollout(armtd._h, 2, dp, dp, o.ctypes.data_as(_lib.dp), 3, C.byref(opt), C.byref(out)) == _lib.ERR_STATE
    assert lib.armour_batch_rollout_device(armtd._h, 2, None, None, None, 3, C.byref(opt), C.byref(out)) == _lib.ERR_STATE
