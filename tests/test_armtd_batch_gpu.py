"""Batched ARMTD comparison planner (armour_armtd_batch_*, ArmtdBatch): many worlds per context, against the frozen KPA outputs,
the single-problem path, the oracle and the armtd_main CLI.  Batches of 2 problems (208 units) run the latency configuration of
k_reachsets, batches of 3 or more (>= 312 units, beyond two waves of 148 CTAs) the throughput configuration."""
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
WORLDS = os.path.join(HERE, "golden", "worlds")
GOLD = os.path.join(HERE, "golden", "armtd", "reference.npz")
TEN_OBSTACLE_WORLDS = ["scene_013_006", "scene_016_006", "scene_016_007", "scene_016_010", "scene_022_001", "scene_022_009",
                       "scene_025_010", "scene_031_004", "scene_031_010", "scene_037_001", "scene_037_004", "scene_037_005",
                       "scene_040_010"]


def _stack(problems):
    """list of armtd_problem tuples -> q0, qd0, q_des, jrs, k_range, obstacles stacked over the problems"""
    return [np.stack([p[i] for p in problems]) for i in range(6)]


@pytest.fixture(scope="module")
def sweep():
    """the 13 ten-obstacle saved worlds x 2 seeds of armtd_problem"""
    from armour_b200 import worlds
    return _stack([worlds.armtd_problem(os.path.join(WORLDS, w + ".csv"), seed=s) for w in TEN_OBSTACLE_WORLDS for s in (0, 1)])


@pytest.fixture(scope="module")
def batch(built, sweep):
    from armour_b200 import ArmtdBatch
    q0, qd0, q_des, jrs, kr, obs = sweep
    b = ArmtdBatch(max_problems=32).build(q0, qd0, jrs, kr, obs)
    yield b
    b.close()


def test_frozen_reference_batched(built):
    from armour_b200 import ArmtdBatch
    gold = np.load(GOLD)
    b = ArmtdBatch(max_problems=12)
    for cases, reps in (([0, 2, 3], 4), ([1], 2)):  # 12 problems (throughput path), then a batch of 2 in the same context
        order = [c for c in cases for _ in range(reps)]
        get = lambda key: np.stack([gold[f"c{c}_{key}"] for c in order])  # noqa: E731
        b.build(get("q0"), get("qd0"), get("jrs"), get("k_range"), get("obs"))
        assert b.m == gold[f"c{cases[0]}_g"].shape[1]
        assert np.all(b.build_status() == 0)
        lg, ref = b.link_independent_generators(), get("link_gens")
        assert np.max(np.abs(lg - ref) / (1e-300 + np.abs(ref) + 1e-12)) <= 1e-9 and np.all(lg[..., 9:] >= ref[..., 9:] - 1e-15)
        for i in range(5):
            k = get("k")[:, i]
            g, J = b.eval(k)
            g_ref, J_ref = get("g")[:, i], get("J")[:, i]
            assert np.max(np.abs(g - g_ref)) <= 1e-11 and np.max(np.abs(J - J_ref)) <= 1e-11, f"k {i}"
            assert np.array_equal(g[:, -28:], g_ref[:, -28:]) and np.array_equal(J[:, -28:], J_ref[:, -28:])
            ok, _ = b.finalize_solution(g)
            assert np.array_equal(ok, get("feasible")[:, i].astype(bool))
            f, df = b.cost(get("q_des"), k)
            assert np.array_equal(f, get("f")[:, i]) and np.array_equal(df, get("df")[:, i])
            for p in range(len(order)):  # repeats of a case are bit-identical to each other
                q = order.index(order[p])
                assert np.array_equal(g[p], g[q]) and np.array_equal(J[p], J[q])
    b.close()


def test_batch_against_single_problems_and_the_oracle(batch, sweep):
    from armour_b200 import ArmtdPlanner, worlds
    from oracle.pyoracle import OracleArmtd
    q0, qd0, q_des, jrs, kr, obs = sweep
    n = q0.shape[0]
    ks = worlds.halton_k(3 * n).reshape(3, n, 7)
    res = [batch.eval(k) for k in ks]
    lg = batch.link_independent_generators()
    single = ArmtdPlanner(max_obstacles=10)
    for p in range(n):
        single.build(q0[p], qd0[p], jrs[p], kr[p], obs[p])
        # throughput (batch) and latency (single) configurations of k_reachsets: same generators, radii to rounding
        ls = single.link_independent_generators()
        assert np.array_equal(lg[p][..., :9], ls[..., :9])
        assert np.max(np.abs(lg[p][..., 9:] - ls[..., 9:]) / (np.abs(ls[..., 9:]) + 1e-300)) <= 1e-13
        for r, k in zip(res, ks):
            g, J = single.eval(k[p])
            assert np.max(np.abs(r[0][p] - g)) <= 1e-12 and np.max(np.abs(r[1][p] - J)) <= 1e-12, p
            # (the single-problem verdict runs the same k_armtd_verdict: this checks the batch indexing, not the predicate;
            # the oracle's verdict below and test_verdict_kernel_row_classes check the predicate itself)
            assert single.finalize_solution(r[0][p]) == tuple(x[p] for x in batch.finalize_solution(r[0]))
    single.close()
    for p in (0, 7, 14, 25):
        o = OracleArmtd().build(q0[p], qd0[p], jrs[p], kr[p], obs[p])
        for r, k in zip(res, ks):
            assert np.max(np.abs(r[0][p] - o.eval_g(k[p]))) <= 1e-11 and np.max(np.abs(r[1][p] - o.eval_jac_g(k[p]))) <= 1e-11
            assert o.verdict(r[0][p]) == tuple(x[p] for x in batch.finalize_solution(r[0]))


def test_device_pointer_calls(batch, sweep):
    import torch
    from armour_b200 import ArmtdBatch
    q0, qd0, q_des, jrs, kr, obs = sweep
    n, m = q0.shape[0], batch.m
    dev = torch.device("cuda", 0)
    k = np.random.default_rng(4).uniform(-1, 1, (n, 7))
    g_h, J_h = batch.eval(k)
    dk = torch.as_tensor(k, device=dev)
    dg = torch.empty((n, m), dtype=torch.float64, device=dev)
    dJ = torch.empty((n, m, 7), dtype=torch.float64, device=dev)
    verdict = torch.empty((2, n), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    batch.eval_device(n, dk.data_ptr(), dg.data_ptr(), dJ.data_ptr())
    batch.verdict_device(n, dg.data_ptr(), verdict[0].data_ptr(), verdict[1].data_ptr())
    batch.synchronize()
    assert np.array_equal(dg.cpu().numpy(), g_h) and np.array_equal(dJ.cpu().numpy(), J_h)
    ok, first = batch.finalize_solution(g_h)
    assert np.array_equal(verdict[0].cpu().numpy().astype(bool), ok) and np.array_equal(verdict[1].cpu().numpy(), first)
    # a device-pointer build with the device's sincos: within a few ulp of the host-pointer build
    b2 = ArmtdBatch(max_problems=32)
    t = [torch.as_tensor(np.ascontiguousarray(a), device=dev) for a in (q0, qd0, jrs, kr, obs)]
    torch.cuda.synchronize()
    b2.build_device(n, obs.shape[1], *(x.data_ptr() for x in t), None)
    b2.synchronize()
    assert np.all(b2.build_status() == 0)
    g2, J2 = b2.eval(k)
    assert np.max(np.abs(g2 - g_h)) <= 1e-12 and np.max(np.abs(J2 - J_h)) <= 1e-12
    f2, df2 = b2.cost(q_des, k)  # host copies of the inputs fetched after a device build
    f1, df1 = batch.cost(q_des, k)
    assert np.array_equal(f1, f2) and np.array_equal(df1, df2)
    b2.close()


def test_verdict_kernel_row_classes(batch, sweep):
    from armour_b200 import ArmtdPlanner
    from oracle.pyoracle import OracleArmtd
    q0, qd0, q_des, jrs, kr, obs = sweep
    g, _ = batch.eval(np.zeros((q0.shape[0], 7)), want_jac=False)
    o = OracleArmtd().build(q0[0], qd0[0], jrs[0], kr[0], obs[0])
    single = ArmtdPlanner(max_obstacles=10).build(q0[0], qd0[0], jrs[0], kr[0], obs[0])
    g0 = g[0].copy()
    g0[:6 * 100 * 10] = np.minimum(g0[:6 * 100 * 10], -1.0)  # a clean start: every checked collision row satisfied
    g0[6 * 100 * 10:-28] = -1.0
    gl, gu = single.get_bounds_info()
    g0[-28:] = 0.5 * (gl[-28:] + gu[-28:])
    m = batch.m
    cases = [(), (3,), (6 * 100 * 10 + 5,), (m - 28 + 2,), (m - 21 + 1,), (m - 14 + 4,), (m - 7 + 6,), (3 * 100 * 10 + 7, 50)]
    gs = []
    for rows in cases:
        gv = g0.copy()
        for r in rows:
            gv[r] = 1e3
        gs.append(gv)
    ok, first = batch.finalize_solution(np.stack(gs))
    for i, rows in enumerate(cases):
        assert (ok[i], first[i]) == o.verdict(gs[i]) == single.finalize_solution(gs[i]), rows
    assert ok[0] and ok[2]  # the last link's collision rows are not checked (the reference's NUM_FACTORS - 1 loop)
    assert first[1] == 3 and first[7] == 50 and not any(ok[3:7])
    single.close()


def test_cost_per_problem(batch, sweep):
    """The batched cost picks each problem's own inputs: the single-problem call on that problem alone (the same armtd_cost
    code, so bit-identical) and the CPU oracle's cost (an independent restatement)."""
    from armour_b200 import ArmtdPlanner
    from oracle.pyoracle import OracleArmtd
    q0, qd0, q_des, jrs, kr, obs = sweep
    k = np.random.default_rng(5).uniform(-1, 1, (q0.shape[0], 7))
    f, df = batch.cost(q_des, k)
    single = ArmtdPlanner(max_obstacles=10)
    for p in range(q0.shape[0]):
        single.build(q0[p], qd0[p], jrs[p], kr[p], obs[p])
        assert single.eval_f(q_des[p], k[p]) == f[p] and np.array_equal(single.eval_grad_f(q_des[p], k[p]), df[p])
    single.close()
    for p in (0, 9, 18):
        o = OracleArmtd().build(q0[p], qd0[p], jrs[p], kr[p], obs[p])
        assert abs(o.cost(q_des[p], k[p]) - f[p]) <= 1e-14 * abs(f[p]) + 1e-300
        assert np.max(np.abs(o.cost_grad(q_des[p], k[p]) - df[p])) <= 1e-14 * np.max(np.abs(df[p]))


def test_batched_solve_against_the_host_solver_over_the_oracle(batch, sweep):
    from oracle.pyoracle import OracleArmtd
    q0, qd0, q_des, jrs, kr, obs = sweep
    n = q0.shape[0]
    k_opt, ok, first, iters = batch.solve(q_des)
    assert np.all(iters >= 1)
    for p in range(n):
        o = OracleArmtd().build(q0[p], qd0[p], jrs[p], kr[p], obs[p])
        k_ref, ok_ref, first_ref, _ = o.solve(q_des[p])
        assert (ok[p], first[p]) == (ok_ref, first_ref), p
        if ok[p]:
            assert np.max(np.abs(k_opt[p] - k_ref)) <= 1e-8, p
            assert o.verdict(o.eval_g(k_opt[p]))[0]
    # a permuted batch gives bit-identical per-problem results
    perm = np.random.default_rng(6).permutation(n)
    from armour_b200 import ArmtdBatch
    b2 = ArmtdBatch(max_problems=32).build(q0[perm], qd0[perm], jrs[perm], kr[perm], obs[perm])
    k2, ok2, first2, it2 = b2.solve(q_des[perm])
    assert np.array_equal(k2, k_opt[perm]) and np.array_equal(ok2, ok[perm]) and np.array_equal(first2, first[perm])
    assert np.array_equal(it2, iters[perm])
    b2.close()


def test_batched_solve_against_the_armtd_main_cli(built, tmp_path):
    from armour_b200 import ArmtdBatch, worlds
    exe = os.path.join(os.path.dirname(HERE), "armour_b200", "armtd_main")
    probs = [worlds.armtd_problem(os.path.join(WORLDS, w + ".csv"), seed=1) for w in ("scene_016_006", "scene_031_004", "scene_037_005")]
    q0, qd0, q_des, jrs, kr, obs = _stack(probs)
    k_opt, ok, _, _ = ArmtdBatch(max_problems=3).build(q0, qd0, jrs, kr, obs).solve(q_des)
    ran = 0
    for p in range(3):
        d = tmp_path / str(p)
        d.mkdir()
        worlds.write_armtd_in(str(d / "armtd.in"), q0[p], qd0[p], q_des[p], jrs[p], kr[p], obs[p])
        res = subprocess.run([exe, str(d)], capture_output=True, text=True, timeout=120)
        assert res.returncode == 0, res.stdout + res.stderr
        if "wall time exceeded" in res.stdout:
            continue  # the cold process ran into the reference's 0.4 s optimiser budget
        ran += 1
        lines = (d / "armtd.out").read_text().split()
        if not ok[p]:
            assert lines[0] == "-1"
            continue
        assert len(lines) == 8
        assert np.max(np.abs(np.array([float(x) for x in lines[:7]]) - k_opt[p])) <= 1e-8
    if ran == 0:
        pytest.skip("every CLI run ran into the reference's 0.4 s optimiser budget")


def test_capacity_failures_are_per_problem_and_fail_safe(built, sweep):
    """A link-table capacity too small for some problems of the batch and not for others.  At the default simplify_threshold
    (5e-4) a link table of this planner holds at most 7 monomials; at 1e-4 the largest table of a world holds 11 to 18 (the
    CPU oracle's tables of this sweep), so the capacity is chosen from the monomial counts of a clean build."""
    from armour_b200 import ArmourError, ArmtdBatch
    from armour_b200._lib import ERR_CAPACITY
    q0, qd0, q_des, jrs, kr, obs = sweep
    n = q0.shape[0]
    clean = ArmtdBatch(max_problems=32, simplify_threshold=1e-4).build(q0, qd0, jrs, kr, obs)
    assert np.all(clean.build_status() == 0)
    most = clean.monomial_counts().reshape(n, -1).max(axis=1)
    caps = [c for c in range(8, clean_cap(clean) + 1, 8) if np.any(most <= c) and np.any(most > c)]
    assert caps, f"no capacity separates the problems: {sorted(most)}"
    cap = caps[len(caps) // 2]
    b = ArmtdBatch(max_problems=32, simplify_threshold=1e-4, cap_link_monomials=cap)
    with pytest.raises(ArmourError) as ei:
        b.build(q0, qd0, jrs, kr, obs)
    assert ei.value.code == ERR_CAPACITY
    failed = b.build_status() != 0
    assert np.array_equal(failed, most > cap)
    k = np.full((n, 7), 0.2)
    g, J = b.eval(k)
    g_clean, J_clean = clean.eval(k)
    ok, _ = b.finalize_solution(g)
    assert not np.any(ok[failed]) and np.all(g[failed, :6 * 100 * 10] == 1e300)
    assert np.all(J[failed, :7 * 100 * 10] == 0)
    assert np.array_equal(g[~failed], g_clean[~failed]) and np.array_equal(J[~failed], J_clean[~failed])
    _, ok_s, _, _ = b.solve(q_des)
    assert not np.any(ok_s[failed])
    b.close()
    clean.close()


def clean_cap(b):
    """cap_link_monomials of the context (the default configuration's)"""
    import ctypes as C
    from armour_b200 import _lib
    cfg = _lib.Config()
    b.lib.armour_config_default(C.byref(cfg))
    return cfg.cap_link_monomials


def test_argument_errors(built, sweep):
    from armour_b200 import ArmourError, ArmtdBatch, ArmtdPlanner, ReachSetEngine
    from armour_b200._lib import ERR_OBSTACLES, ERR_STATE
    q0, qd0, q_des, jrs, kr, obs = sweep
    b = ArmtdBatch(max_problems=4, max_obstacles=10)
    with pytest.raises(ArmourError) as ei:
        b.eval(np.zeros((1, 7)))  # before a build
    assert ei.value.code == ERR_STATE
    with pytest.raises(ArmourError) as ei:
        b.build(q0[:5], qd0[:5], jrs[:5], kr[:5], obs[:5])  # more than max_problems
    assert ei.value.code == ERR_STATE
    with pytest.raises(ArmourError) as ei:
        b.build(q0[:2], qd0[:2], jrs[:2], kr[:2], np.zeros((2, 11, 12)))  # more than max_obstacles
    assert ei.value.code == ERR_OBSTACLES
    with pytest.raises(ValueError):
        b.build(q0[:2], qd0[:2], jrs[:2, :, :, :99], kr[:2], obs[:2])
    b.build(q0[:2], qd0[:2], jrs[:2], kr[:2], obs[:2])
    with pytest.raises(ArmourError) as ei:
        b.eval(np.zeros((3, 7)))  # more problems than built
    assert ei.value.code == ERR_STATE
    b.close()
    eng = ReachSetEngine(max_problems=2, max_obstacles=10)  # the main planner's context
    h, lib = eng._h, eng.lib
    z = np.zeros(2 * 7)
    from armour_b200._lib import ip
    from armour_b200.armtd import _dp
    assert lib.armour_armtd_batch_build(h, 1, _dp(z), _dp(z), _dp(np.zeros(4200)), _dp(z), None, 0) == ERR_STATE
    assert lib.armour_armtd_batch_eval(h, 1, _dp(z), _dp(np.zeros(100)), None) == ERR_STATE
    ok = np.zeros(2, np.int32)
    assert lib.armour_armtd_batch_solve(h, 1, _dp(z), None, _dp(z), ok.ctypes.data_as(ip), None, None) == ERR_STATE
    eng.close()
    single = ArmtdPlanner(max_obstacles=10)  # a single-problem ARMTD context takes batches of one only
    rc = single.lib.armour_armtd_batch_build(single._h, 2, _dp(q0[:2].copy()), _dp(qd0[:2].copy()), _dp(jrs[:2].copy()),
                                             _dp(kr[:2].copy()), _dp(obs[:2].copy()), 10)
    assert rc == ERR_STATE
    single.close()
