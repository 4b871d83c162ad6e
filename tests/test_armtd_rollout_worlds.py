"""The trajectory the episodes of the ARMTD comparison planner execute (tests/armtd_rollout_ref.py) and the soundness of the
synthetic offline table (worlds.armtd_offline_jrs_batch) their builds rely on, no GPU needed."""
import numpy as np
import pytest

from armtd_rollout_ref import const_acc, k_range


def test_constant_acceleration_trajectory():
    rng = np.random.default_rng(1)
    q0, qd0 = rng.uniform(-2, 2, 7), rng.uniform(-1.2, 1.2, 7)
    k_a = k_range(qd0) * rng.uniform(-1, 1, 7)
    q, qd = const_acc(q0, qd0, k_a, 0.0)
    assert np.array_equal(q, q0) and np.array_equal(qd, qd0)
    # continuous at t = 0.5, position and velocity
    h = 1e-9
    qa, qda = const_acc(q0, qd0, k_a, 0.5)
    qb, qdb = const_acc(q0, qd0, k_a, 0.5 + h)
    assert np.max(np.abs(qb - qa)) <= 1e-8 and np.max(np.abs(qdb - qda)) <= 1e-8
    # at rest at t = 1, at the q_stop of the KPA joint-limit rows (csrc/armtd.cuh armtd_joint_extremum), written out here
    t_move, t_to_stop = 0.5, 0.5
    q_peak = q0 + qd0 * t_move + k_a * t_move * t_move * 0.5
    q_dot_peak = qd0 + k_a * t_move
    q_ddot_to_stop = -q_dot_peak / t_to_stop
    q_stop = q_peak + q_dot_peak * t_to_stop + 0.5 * q_ddot_to_stop * t_to_stop * t_to_stop
    q1, qd1 = const_acc(q0, qd0, k_a, 1.0)
    assert np.array_equal(q1, q_stop) and not np.any(qd1)
    assert np.array_equal(qa, q_peak) and np.array_equal(qda, q_dot_peak)
    # the velocity is the derivative of the position in both phases
    for t in (0.2, 0.8):
        qm, _ = const_acc(q0, qd0, k_a, t - 1e-6)
        qp, _ = const_acc(q0, qd0, k_a, t + 1e-6)
        _, v = const_acc(q0, qd0, k_a, t)
        assert np.allclose((qp - qm) / 2e-6, v, atol=1e-8)


@pytest.mark.parametrize("case", ["rest", "random", "near_speed_limits"])
def test_stand_in_table_encloses_the_trajectory(built, case):
    """cos / sin of q(t) - q0 lie inside c + g k +- r on a grid much denser than the table's own 9 x 33 per interval
    (65 times x 257 values of k)."""
    from armour_b200 import worlds
    rng = np.random.default_rng(2)
    qd0 = {"rest": np.zeros((1, 7)),
           "random": rng.uniform(-0.5, 0.5, (3, 7)) * worlds.SPEED_LIMITS,
           "near_speed_limits": np.stack([worlds.SPEED_LIMITS * 0.999, -worlds.SPEED_LIMITS, worlds.SPEED_LIMITS])}[case]
    kr = worlds.armtd_k_range(qd0)
    jrs = worlds.armtd_offline_jrs_batch(qd0, kr)
    k = np.linspace(-1, 1, 257)
    worst = -np.inf
    for j in range(100):
        t = j / 100 + np.linspace(0, 1, 65) / 100
        for p in range(qd0.shape[0]):
            for i in range(7):
                d = np.stack([const_acc(0.0, qd0[p, i], kr[p, i] * k, tt)[0] for tt in t])  # [65, 257]
                c, g, r, cs, gs, rs = jrs[p, :, i, j]
                worst = max(worst, np.max(np.abs(np.cos(d) - (c + g * k)) - r), np.max(np.abs(np.sin(d) - (cs + gs * k)) - rs))
    assert worst <= 0.0, worst
