"""Inputs of the closed-loop episodes (worlds.random_episodes, worlds.pad_obstacles) and the numpy separating-axis reference
the GPU tests of armour_batch_clearance / armour_batch_rollout compare with (no GPU needed)."""
import numpy as np
import pytest

from rollout_ref import link_boxes, sat_clearance, clearance, bezier, waypoint


def test_random_episodes_are_the_draws_of_random_problems(built):
    from armour_b200 import worlds
    start, goal, obs = worlds.random_episodes(9, 4, seed=7)
    assert start.shape == (9, 7) and goal.shape == (9, 7) and obs.shape == (9, 4, 12)
    q0, qd0, qdd0, q_des, obs_p = worlds.random_problems(9, 4, seed=7, moving=False)
    assert np.array_equal(start, q0) and np.array_equal(obs, obs_p)
    assert not np.any(qd0) and not np.any(qdd0)
    # the goal is the one random_problems aimed its waypoint at
    for p in range(9):
        assert np.allclose(worlds.straight_line_waypoint(start[p], goal[p]), q_des[p], atol=1e-9)
    assert np.all(goal >= worlds.STATE_LB) and np.all(goal <= worlds.STATE_UB)
    s2, g2, o2 = worlds.random_episodes(9, 4, seed=7)
    assert np.array_equal(s2, start) and np.array_equal(g2, goal) and np.array_equal(o2, obs)
    s3, g3, _ = worlds.random_episodes(9, 4, seed=8)
    assert not np.array_equal(s3, start) and not np.array_equal(g3, goal)


def test_pad_obstacles_pads_beyond_the_arms_reach(built):
    from armour_b200 import worlds
    a = np.arange(3 * 12, dtype=float).reshape(3, 12)
    b = np.arange(5 * 12, dtype=float).reshape(5, 12) + 100
    out = worlds.pad_obstacles([a, b, np.zeros((0, 12))], 6)
    assert out.shape == (3, 6, 12)
    assert np.array_equal(out[0, :3], a) and np.array_equal(out[1, :5], b)
    pads = np.concatenate([out[0, 3:], out[1, 5:], out[2]])
    assert pads.shape == (3 + 1 + 6, 12)
    for z in pads:  # small boxes: diagonal generators of 1 cm
        assert np.allclose(z[3:12].reshape(3, 3), np.eye(3) * worlds.PAD_HALF_SIZE)
    with pytest.raises(ValueError):
        worlds.pad_obstacles([b], 4)
    # no configuration of either robot model comes near a padding box: every link box lies within 2 m of the base
    rng = np.random.default_rng(3)
    for model in (0, 1):
        for q in rng.uniform(-np.pi, np.pi, (20, 7)):
            c, _ = clearance(q, pads, model)
            assert c > 10.0
            cs, gs = link_boxes(q, model)
            assert np.max(np.linalg.norm(cs, axis=1) + np.abs(gs).sum(axis=(1, 2))) < 2.0


def _box(c, h, R=np.eye(3)):
    return np.asarray(c, dtype=float), (R * np.asarray(h, dtype=float)[None, :]).T


def test_sat_reference_on_analytic_cases():
    ca, A = _box([0, 0, 0], [0.1, 0.2, 0.3])
    cb, B = _box([0.5, 0, 0], [0.1, 0.1, 0.1])
    assert sat_clearance(ca, A, cb, B) == pytest.approx(0.3, abs=1e-15)          # a known gap
    assert sat_clearance(cb, B, ca, A) == pytest.approx(0.3, abs=1e-15)
    cb, B = _box([0.2, 0, 0], [0.1, 0.1, 0.1])
    assert sat_clearance(ca, A, cb, B) == pytest.approx(0.0, abs=1e-15)          # touching
    cb, B = _box([0.0, 0.05, 0], [0.05, 0.05, 0.05])
    assert sat_clearance(ca, A, cb, B) == pytest.approx(-0.15, abs=1e-15)        # nested: -penetration along x
    cb, B = _box([0.3, -0.4, 1.0], [0.1, 0.1, 0.1])
    assert sat_clearance(ca, A, cb, B) == pytest.approx(0.6, abs=1e-15)          # separated along z most
    c45, s45 = np.cos(np.pi / 4), np.sin(np.pi / 4)
    Rz = np.array([[c45, -s45, 0], [s45, c45, 0], [0, 0, 1]])
    ca, A = _box([0, 0, 0], [0.1, 0.1, 0.1])
    for d in (0.5, 0.25, 0.2):  # rotated by 45 degrees: the vertex of B meets the face of A at x = d - 0.1 sqrt 2
        cb, B = _box([d, 0, 0], [0.1, 0.1, 0.1], Rz)
        assert sat_clearance(ca, A, cb, B) == pytest.approx(d - 0.1 - 0.1 * np.sqrt(2), abs=1e-15)
    # B rotated 45 degrees about x, an edge towards A's top face
    Rx = np.array([[1, 0, 0], [0, c45, -s45], [0, s45, c45]])
    cb, B = _box([0.0, 0.0, 0.5], [0.1, 0.1, 0.1], Rx)
    assert sat_clearance(ca, A, cb, B) == pytest.approx(0.5 - 0.1 - 0.1 * np.sqrt(2), abs=1e-15)
    # degenerate generators (a flat box) skip the vanishing axes
    cb, B = _box([0.0, 0.0, 0.35], [0.1, 0.1, 0.0])
    assert sat_clearance(ca, A, cb, B) == pytest.approx(0.25, abs=1e-15)


def test_bezier_and_waypoint_reference():
    q0, qd0, qdd0, k = np.full(7, 0.3), np.full(7, -0.2), np.full(7, 0.7), np.full(7, 0.05)
    q, qd, qdd = bezier(q0, qd0, qdd0, k, 0.0)
    assert np.allclose(q, q0, atol=1e-15) and np.allclose(qd, qd0, atol=1e-15) and np.allclose(qdd, qdd0, atol=1e-14)
    q, qd, qdd = bezier(q0, qd0, qdd0, k, 1.0)
    assert np.allclose(q, q0 + k, atol=1e-15) and np.allclose(qd, 0, atol=1e-15) and np.allclose(qdd, 0, atol=1e-14)
    h = 1e-5  # the derivatives are those of q
    qa, qda, _ = bezier(q0, qd0, qdd0, k, 0.4 - h)
    qb, qdb, _ = bezier(q0, qd0, qdd0, k, 0.4 + h)
    _, qd, qdd = bezier(q0, qd0, qdd0, k, 0.4)
    assert np.allclose((qb - qa) / (2 * h), qd, atol=1e-9) and np.allclose((qdb - qda) / (2 * h), qdd, atol=1e-8)
    goal = np.array([3.0, 0.5, -3.0, 0.0, 0.0, 0.0, 0.0])
    q = np.array([-3.0, 0.45, 3.0, 0.0, 0.0, 0.0, 0.0])
    # continuous joints go the short way round; within lookahead the waypoint is the goal (unwrapped next to q)
    w = waypoint(q, goal)
    d = np.array([6.0 - 2 * np.pi, 0.05, 2 * np.pi - 6.0, 0, 0, 0, 0])
    assert np.linalg.norm(d) > 0.1
    assert np.allclose(w, q + 0.1 * d / np.linalg.norm(d), atol=1e-14)
    near = q + np.array([0.01, 0.02, -0.03, 0, 0, 0, 0.04])
    assert np.allclose(waypoint(q, near), near, atol=1e-15)
