"""worlds.armtd_random_problems: the vectorised sweep generator of the ARMTD comparison planner (no GPU needed)."""
import numpy as np


def test_armtd_random_problems_is_deterministic_and_matches_the_per_problem_tables():
    from armour_b200 import worlds
    a = worlds.armtd_random_problems(6, 3, seed=11)
    b = worlds.armtd_random_problems(6, 3, seed=11)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    q0, qd0, q_des, k_range, jrs, obs = a
    assert q0.shape == qd0.shape == q_des.shape == k_range.shape == (6, 7)
    assert jrs.shape == (6, 6, 7, 100) and obs.shape == (6, 3, 12)
    r0, rd0, _, rq_des, robs = worlds.random_problems(6, 3, seed=11)
    assert np.array_equal(q0, r0) and np.array_equal(qd0, rd0) and np.array_equal(q_des, rq_des) and np.array_equal(obs, robs)
    assert np.array_equal(k_range, worlds.armtd_k_range(qd0))
    for p in range(6):
        assert np.max(np.abs(jrs[p] - worlds.armtd_offline_jrs(qd0[p], k_range[p]))) <= 1e-15
    assert not np.array_equal(worlds.armtd_random_problems(6, 3, seed=12)[4], jrs)
