"""Closed-loop episodes of the ARMTD comparison planner on the device (armour_armtd_batch_rollout, ArmtdBatch.rollout) and the
stand-in offline table they build from (armour_armtd_offline_jrs).

Every replan of an episode must be the existing ARMTD planner, bit for bit: the sub-batch of worlds still running at replan r,
rebuilt in ascending world order from the logged planning states through the table call + the device-pointer build + the
batched solve, plans the logged k_opt and verdict.  The state update and the waypoint are checked against the numpy reference
of tests/armtd_rollout_ref.py, the audit against the forward kinematics and separating-axis test of tests/rollout_ref.py, the
plans against the CPU oracle."""
import ctypes as C
import os

import numpy as np
import pytest

from armtd_rollout_ref import const_acc, k_range, replay
from conftest import WORLDS
from rollout_ref import clearance, goal_diff, waypoint

pytestmark = pytest.mark.gpu

KEYS = ("outcome", "replans", "infeasible", "final_state", "min_clearance", "log_state", "log_q_des", "log_k", "log_int",
        "log_clearance")
R16 = 12


def _device(*arrays):
    import torch
    return [torch.as_tensor(np.ascontiguousarray(a), device=torch.device("cuda", 0)) for a in arrays]


def test_device_table_matches_the_numpy_generator(built):
    from armour_b200 import ArmtdBatch, worlds
    rng = np.random.default_rng(3)
    qd0 = np.concatenate([np.zeros((2, 7)), rng.uniform(-0.5, 0.5, (20, 7)) * worlds.SPEED_LIMITS,
                          np.stack([worlds.SPEED_LIMITS * 0.999, -worlds.SPEED_LIMITS, worlds.SPEED_LIMITS])])
    kr = worlds.armtd_k_range(qd0)
    ref = worlds.armtd_offline_jrs_batch(qd0, kr)
    b = ArmtdBatch(max_problems=4, max_obstacles=10)
    jrs = b.offline_jrs(qd0, kr)  # more rows than max_problems: the table call does not use the batch
    assert jrs.shape == ref.shape
    assert np.max(np.abs(jrs - ref)) <= 1e-14
    assert np.all(jrs[:, [2, 5]] >= ref[:, [2, 5]] - 1e-15)
    # the device-pointer call writes the same table
    dq, dk, dj = _device(qd0, kr, np.zeros_like(ref))
    import torch
    torch.cuda.synchronize()
    b.offline_jrs_device(qd0.shape[0], dq.data_ptr(), dk.data_ptr(), dj.data_ptr())
    b.synchronize()
    assert np.array_equal(dj.cpu().numpy(), jrs)
    b.close()


@pytest.fixture(scope="module")
def episodes16(built):
    from armour_b200 import ArmtdBatch, worlds
    start, goal, obs = worlds.random_episodes(16, 20, seed=5)
    b = ArmtdBatch(max_problems=16, max_obstacles=20)
    res = b.rollout(start, goal, obs, max_replans=R16)
    yield b, start, goal, obs, res
    b.close()


def test_each_replan_is_the_existing_planner(episodes16):
    import torch
    b, start, goal, obs, res = episodes16
    li = res["log_int"]
    planned = np.arange(R16)[:, None] < res["replans"][None, :]
    assert np.all(res["replans"] >= 1) and np.all(res["replans"] <= R16)
    assert np.any(li[..., 0][planned] == 1) and np.any(li[..., 0][planned] == 0), "seed 5: feasible and infeasible replans"
    assert np.all(np.isnan(res["log_k"][~planned])) and np.all(li[~planned] == -1)
    assert np.array_equal(res["infeasible"], ((li[..., 0] == 0) & planned).sum(axis=0))
    for r in range(R16):
        idx = np.flatnonzero(res["replans"] > r)
        if idx.size == 0:
            break
        st = res["log_state"][r, idx]
        q0, qd0 = st[:, :7], st[:, 7:14]
        kr = worlds_k_range(qd0)
        dq0, dqd0, dkr, dobs, djrs = _device(q0, qd0, kr, obs[idx], np.zeros((idx.size, 6, 7, 100)))
        torch.cuda.synchronize()
        b.offline_jrs_device(idx.size, dqd0.data_ptr(), dkr.data_ptr(), djrs.data_ptr())
        b.build_device(idx.size, obs.shape[1], dq0.data_ptr(), dqd0.data_ptr(), djrs.data_ptr(), dkr.data_ptr(), dobs.data_ptr())
        b.synchronize()
        assert np.array_equal(b.build_status(), li[r, idx, 3]), r
        k, ok, first, iters = b.solve(res["log_q_des"][r, idx])
        assert np.array_equal(k, res["log_k"][r, idx]), r
        assert np.array_equal(ok.astype(np.int32), li[r, idx, 0]) and np.array_equal(first, li[r, idx, 1]), r
        assert np.array_equal(iters, li[r, idx, 2]), r
    assert np.array_equal(res["log_state"][0], np.concatenate([start, np.zeros((16, 14))], axis=1))


def worlds_k_range(qd0):
    from armour_b200 import worlds
    kr = worlds.armtd_k_range(qd0)
    assert np.array_equal(kr, k_range(qd0))
    return kr


def test_state_update_and_waypoint(episodes16):
    b, start, goal, obs, res = episodes16
    seg, nxt = replay(res, start)
    planned = np.arange(R16)[:, None] < res["replans"][None, :]
    assert not np.any(res["log_state"][..., 14:][planned]) and not np.any(res["final_state"][:, 14:]), "no acceleration input"
    braked = 0
    for (r, w), after_ref in nxt.items():
        st = res["log_state"][r, w]
        assert np.max(np.abs(res["log_q_des"][r, w] - waypoint(st[:7], goal[w]))) <= 1e-13, (r, w)
        after = res["log_state"][r + 1, w] if r + 1 < res["replans"][w] else res["final_state"][w]
        assert np.max(np.abs(after - after_ref)) <= 1e-12, (r, w)
        if not res["log_int"][r, w, 0]:
            assert not np.any(after[7:]), (r, w)  # braked to rest
            braked += 1
    assert braked > 0


def test_rollout_is_deterministic_and_worlds_are_independent(episodes16):
    b, start, goal, obs, res = episodes16
    again = b.rollout(start, goal, obs, max_replans=R16)
    for key in KEYS:
        assert np.array_equal(res[key], again[key], equal_nan=True), key
    perm = np.random.default_rng(2).permutation(16)
    p = b.rollout(start[perm], goal[perm], obs[perm], max_replans=R16)
    for key in KEYS:
        a = res[key]
        if a.ndim >= 2 and key.startswith("log_"):
            assert np.array_equal(p[key], a[:, perm], equal_nan=True), key
        else:
            assert np.array_equal(p[key], a[perm], equal_nan=True), key


def test_logged_plans_agree_with_the_oracle(episodes16):
    from oracle.pyoracle import OracleArmtd
    b, start, goal, obs, res = episodes16
    li = res["log_int"]
    pairs = [(r, w) for w in range(16) for r in range(res["replans"][w]) if li[r, w, 3] == 0]
    rng = np.random.default_rng(4)
    pick = [pairs[i] for i in rng.choice(len(pairs), 4, replace=False)]
    fe = [p for p in pairs if li[p[0], p[1], 0]]
    if not any(li[r, w, 0] for r, w in pick):
        pick[-1] = fe[0]
    for r, w in pick:
        st = res["log_state"][r, w]
        kr = k_range(st[7:14])
        jrs = b.offline_jrs(st[None, 7:14], kr[None])[0]
        o = OracleArmtd().build(st[:7], st[7:14], jrs, kr, obs[w])
        k, ok, first, _ = o.solve(res["log_q_des"][r, w])
        assert ok == bool(li[r, w, 0]) and first == li[r, w, 1], (r, w)
        if ok:
            # the episode's build takes cos q0 / sin q0 from the device's sincos, the oracle from the host's libm: inputs a few
            # ulp apart move the solver's stopping point within its tolerance (KPA's 1e-7; 2.3e-8 observed on one plan of four)
            assert np.max(np.abs(k - res["log_k"][r, w])) <= 1e-7, (r, w, k, res["log_k"][r, w])
            good, row = o.verdict(o.eval_g(res["log_k"][r, w]))  # the oracle's own verdict accepts the logged plan
            assert good, (r, w, row)


def test_certified_motion_is_collision_free(built):
    """64 worlds whose start is collision-free, 10 obstacles, 30 replans, 32 audit samples: no executed segment exceeds a
    limit, and none hits an obstacle except through the reference's NUM_FACTORS - 1 quirk: KPA's verdict does not check the
    last link's collision rows, so a plan it accepts may move the last link into an obstacle.  Every such contact must be the
    last link's, on a plan the verdict accepted, whose last-link collision rows are violated."""
    from armour_b200 import ArmtdBatch, ReachSetEngine, _lib, worlds
    start, goal, obs = worlds.random_episodes(160, 10, seed=20261020)
    b = ArmtdBatch(max_problems=64, max_obstacles=10)
    eng = ReachSetEngine(max_problems=1, max_obstacles=10)  # the clearance of robot model 0, the ARMTD planner's model
    c0, _ = eng.clearance(start, obs, np.arange(160))
    keep = np.flatnonzero(c0 > 0)[:64]
    assert keep.size == 64
    start, goal, obs = start[keep], goal[keep], obs[keep]
    res = b.rollout(start, goal, obs, max_replans=30, audit_samples=32)
    assert not np.any(res["outcome"] == _lib.ROLLOUT_LIMIT)
    lc = res["log_clearance"]
    assert np.array_equal(res["min_clearance"], np.nanmin(lc, axis=0))
    seg, _ = replay(res, start)
    hit = np.flatnonzero(res["outcome"] == _lib.ROLLOUT_COLLISION)
    for w in hit:  # the quirk, shown: the last link, a plan KPA's verdict accepted, its last-link rows violated
        r = res["replans"][w] - 1
        plan, t0, t1 = seg[r, w]
        samples = np.stack([const_acc(*plan, t)[0] for t in t0 + (t1 - t0) * np.arange(32) / 31])
        clr, which = eng.clearance(samples, obs[w])
        assert abs(np.min(clr) - lc[r, w]) <= 1e-12 and lc[r, w] < -1e-4
        link = which[np.argmin(clr)] // 10
        assert link == 6, (w, link)
        rp = max(x for x in range(r + 1) if res["log_int"][x, w, 0])  # the replan that made the executed plan
        st = res["log_state"][rp, w]
        kr = k_range(st[7:14])
        one = ArmtdBatch(max_problems=1, max_obstacles=10).build(st[None, :7], st[None, 7:14], b.offline_jrs(st[None, 7:14], kr[None]),
                                                                kr[None], obs[w][None])
        g, _ = one.eval(res["log_k"][rp, w][None], want_jac=False)
        ok, _ = one.finalize_solution(g)
        rows = g[0, :7 * 100 * 10].reshape(7, 100, 10)
        assert ok[0] and np.max(rows[6]) > 0, (w, rp, np.max(rows[:6]), np.max(rows[6]))
        one.close()
    others = np.setdiff1d(np.arange(64), hit)
    lo = lc[:, others]
    assert np.all(lo[~np.isnan(lo)] >= -1e-4)
    keys = sorted(seg)
    rng = np.random.default_rng(9)
    chosen = [keys[i] for i in rng.choice(len(keys), 5, replace=False)]
    chosen += [k for k in keys if not res["log_int"][k[0], k[1], 0]][:1]  # a braking segment too
    for r, w in chosen:
        plan, t0, t1 = seg[r, w]
        ref = min(clearance(const_acc(*plan, t)[0], obs[w])[0] for t in t0 + (t1 - t0) * np.arange(32) / 31)
        assert abs(ref - lc[r, w]) <= 1e-12, (r, w, ref, lc[r, w])
    b.close()
    eng.close()


def test_episodes_end_as_specified(built):
    from armour_b200 import ArmtdBatch, ReachSetEngine, _lib, worlds
    b = ArmtdBatch(max_problems=4, max_obstacles=10)
    start = np.array([0.3, 0.4, -0.2, 1.2, 0.1, 0.6, -0.4])
    v = np.array([1.0, -0.5, 0.8, 0.6, -1.0, 0.4, 0.9])
    goal = start + 0.3 * v / np.linalg.norm(v)
    pad = worlds.pad_obstacles([np.zeros((0, 12))], 10)
    res = b.rollout(start[None], goal[None], pad, max_replans=100)
    assert res["outcome"][0] == _lib.ROLLOUT_ARRIVED
    n = res["replans"][0]
    assert res["infeasible"][0] == 0 and np.all(res["log_int"][:n, 0, 0] == 1)
    assert np.linalg.norm(goal_diff(res["final_state"][0, :7], goal)) <= 0.05
    assert res["min_clearance"][0] > 5.0

    # a saved world padded from 6 to 10 obstacles plans what the world itself plans
    s, g, o = worlds.load_world_csv(os.path.join(WORLDS, "scene_013_001.csv"))
    assert o.shape[0] == 6
    a = b.rollout(s[None], g[None], o[None], max_replans=6)
    p = b.rollout(s[None], g[None], worlds.pad_obstacles([o], 10), max_replans=6)
    assert np.array_equal(a["replans"], p["replans"])
    n = a["replans"][0]
    assert np.max(np.abs(a["log_k"][:n] - p["log_k"][:n])) <= 1e-9
    assert np.array_equal(a["log_int"][:n, :, 0], p["log_int"][:n, :, 0])

    # both planners take the same episode arrays and return the same dict
    start4, goal4, obs4 = worlds.random_episodes(4, 10, seed=11)
    eng = ReachSetEngine(max_problems=4, max_obstacles=10)
    ra = eng.rollout(start4, goal4, obs4, max_replans=5)
    rt = b.rollout(start4, goal4, obs4, max_replans=5)
    assert set(ra) == set(rt) == set(KEYS)
    for key in KEYS:
        assert ra[key].shape == rt[key].shape and ra[key].dtype == rt[key].dtype, key
    assert np.array_equal(ra["log_state"][0], rt["log_state"][0])
    eng.close()
    b.close()


def test_argument_errors(built):
    from armour_b200 import ArmourError, ArmtdBatch, ReachSetEngine, _lib
    b = ArmtdBatch(max_problems=2, max_obstacles=3)
    s = np.zeros((2, 7))
    o = np.zeros((2, 3, 12))
    with pytest.raises(ArmourError) as e:
        b.rollout(np.zeros((3, 7)), np.zeros((3, 7)), np.zeros((3, 3, 12)))
    assert e.value.code == _lib.ERR_STATE
    with pytest.raises(ArmourError) as e:
        b.rollout(s, s, np.zeros((2, 4, 12)))
    assert e.value.code == _lib.ERR_OBSTACLES
    for kw in (dict(max_replans=0), dict(audit_samples=1), dict(lookahead=0.0), dict(goal_radius=-1.0), dict(max_iter=0),
               dict(tol=0.0)):
        with pytest.raises(ArmourError) as e:
            b.rollout(s, s, o, **kw)
        assert e.value.code == _lib.ERR_ARG, kw
    lib = b.lib
    opt = _lib.RolloutOptions()
    lib.armour_rollout_options_default(C.byref(opt))
    out = _lib.RolloutOut()
    dp = s.ctypes.data_as(_lib.dp)
    op = o.ctypes.data_as(_lib.dp)
    assert lib.armour_armtd_batch_rollout(b._h, 2, None, dp, op, 3, C.byref(opt), C.byref(out)) == _lib.ERR_ARG
    assert lib.armour_armtd_batch_rollout(b._h, 2, dp, dp, None, 3, C.byref(opt), C.byref(out)) == _lib.ERR_ARG
    assert lib.armour_armtd_batch_rollout(b._h, 2, dp, dp, None, 0, None, C.byref(out)) == _lib.ERR_ARG
    assert lib.armour_armtd_batch_rollout(b._h, 0, dp, dp, None, 0, C.byref(opt), C.byref(out)) == _lib.ERR_ARG
    assert lib.armour_armtd_batch_rollout_device(b._h, 2, None, None, None, 0, C.byref(opt), C.byref(out)) == _lib.ERR_ARG
    opt.struct_size = 8
    assert lib.armour_armtd_batch_rollout(b._h, 2, dp, dp, None, 0, C.byref(opt), C.byref(out)) == _lib.ERR_ARG
    # the episode calls of each planner refuse the other planner's context
    lib.armour_rollout_options_default(C.byref(opt))
    assert lib.armour_batch_rollout(b._h, 2, dp, dp, op, 3, C.byref(opt), C.byref(out)) == _lib.ERR_STATE
    eng = ReachSetEngine(max_problems=2, max_obstacles=3)
    assert lib.armour_armtd_batch_rollout(eng._h, 2, dp, dp, op, 3, C.byref(opt), C.byref(out)) == _lib.ERR_STATE
    assert lib.armour_armtd_batch_rollout_device(eng._h, 2, None, None, None, 3, C.byref(opt), C.byref(out)) == _lib.ERR_STATE
    # the table calls: ARMTD contexts only, n >= 1, non-null arrays
    z = np.zeros((2, 7))
    jrs = np.zeros((2, 6, 7, 100))
    zp, jp = z.ctypes.data_as(_lib.dp), jrs.ctypes.data_as(_lib.dp)
    assert lib.armour_armtd_offline_jrs(eng._h, 2, zp, zp, jp) == _lib.ERR_STATE
    assert lib.armour_armtd_offline_jrs_device(eng._h, 2, None, None, None) == _lib.ERR_STATE
    assert lib.armour_armtd_offline_jrs(b._h, 0, zp, zp, jp) == _lib.ERR_ARG
    assert lib.armour_armtd_offline_jrs(b._h, 2, zp, None, jp) == _lib.ERR_ARG
    assert lib.armour_armtd_offline_jrs_device(b._h, 2, None, None, None) == _lib.ERR_ARG
    with pytest.raises(ValueError):
        b.offline_jrs(np.zeros((2, 7)), np.zeros((3, 7)))
    eng.close()
    b.close()
