"""Evaluation images: at the end of every build the tables and candidate lists of each chunk are packed into one
contiguous image, the only input of k_constraints.  These tests decode the images on the host and check them against
the padded tables (armour_export_reachsets) and the candidate counts, then check the evaluation against the CPU oracle
(or, for a batch with capacity failures, against the same batch built with room to spare: bit-identical)."""
import os

import numpy as np
import pytest

from conftest import WORLDS
from halfspace_ref import chunk_candidates, chunk_rows, half_spaces, row_generators

pytestmark = pytest.mark.gpu
NF = 7
K_TEST = np.array([0.5, 0.6, 0.7, 0.0, -0.5, -0.6, -0.7])


def _check_images(eng, failed=(), obs=None, g0=None):
    """Decode every chunk image and compare it with the padded tables and the candidate counts.  With the batch's
    obstacles [nprob, O, 12], every row's records must be, bit for bit and in order, a subsequence of the row's 72
    half-spaces computed from the generators; with g0 (the g of problem 0 at a k inside the lists' box, evaluated just
    before), the row maximum over the records at the sliced link centres must equal both g0 and the maximum over all 72."""
    img, lay = eng.eval_images()
    T, NJ, O = eng.T, eng.NJ, max(eng.nobs, 0)
    C_ = eng.lib.armour_chunk_intervals()
    cnt_all = eng.candidate_counts() if O > 0 else None
    rows = NJ * C_ * O
    for p in range(eng.nprob):
        if p in failed:
            continue
        ex = eng.export_reachsets(p)
        for tb in range(T // C_):
            b = img[p, tb]
            d = b.view(np.float64)
            u16 = b.view(np.uint16)
            lt = b[:C_ * NJ * 8].view(np.int32).reshape(C_ * NJ, 2)
            ut = b[lay["torque_tables"]:lay["torque_tables"] + C_ * NF * 16].view(np.int32).reshape(C_ * NF, 4)
            lc = b[lay["link_c"]:lay["link_c"] + C_ * NJ * 24].view(np.float64).reshape(C_ * NJ, 3)
            lr = b[lay["link_r"]:lay["link_r"] + C_ * NJ * 24].view(np.float64).reshape(C_ * NJ, 3)
            uc = b[lay["u_c"]:lay["u_c"] + C_ * NF * 8].view(np.float64)
            ur = b[lay["u_r"]:lay["u_r"] + C_ * NF * 8].view(np.float64)
            for tt in range(C_):
                t = tb * C_ + tt
                for l in range(NJ):
                    i, src = tt * NJ + l, t * NJ + l
                    off, n = lt[i]
                    assert n == ex["nl"][src]
                    recs = d[off:off + 4 * n].reshape(n, 4)
                    assert np.array_equal(recs[:, :3], ex["gl"][src, :n])
                    keys = u16[(off * 4):(off + 4 * n) * 4].reshape(n, 16)[:, 12]
                    assert np.array_equal(keys.astype(np.uint64), ex["hl"][src, :n] & 0xFFFF)
                    assert np.array_equal(lc[i], ex["cl"][src])
                    assert np.array_equal(lr[i], ex["link_gens"][t, l][[9, 13, 17]])
                for j in range(NF):
                    i, src = tt * NF + j, t * NF + j
                    coff, koff, n, _ = ut[i]
                    assert n == ex["nu"][src]
                    assert np.array_equal(d[coff:coff + n], ex["gu"][src, :n])
                    assert np.array_equal(u16[koff:koff + n].astype(np.uint64), ex["hu"][src, :n] & 0xFFFF)
                    assert uc[i] == ex["cu"][src] and ur[i] == ex["ru"][src]
            if rows == 0:
                continue
            cnt, grp, recs, first = chunk_candidates(b, lay, rows)
            assert np.array_equal(cnt, cnt_all[p, tb].reshape(-1))
            stored = np.where(cnt == 255, 0, cnt).astype(np.int64)
            assert np.array_equal(grp, first[0:rows:32])
            if obs is not None:
                _check_records(eng, ex, obs[p], tb, C_, cnt, recs, g0 if p == 0 else None)
            # the link tables follow the records directly
            assert lt[0, 0] == lay["records"] // 8 + 4 * stored.sum()


def _check_records(eng, ex, ob, tb, C_, cnt, recs, g0):
    NJ, O, T = eng.NJ, ob.shape[0], eng.T
    t, l, o = chunk_rows(NJ, C_, O, tb)
    x = np.arange(NJ * C_ * O)
    hs, nz = half_spaces(*row_generators(ob, ex["link_gens"], t, l, o))
    if g0 is not None:
        centres = eng.link_sliced_center()[t, l]  # [rows, 3] of problem 0
    first = 0
    for r in range(len(x)):
        n = int(cnt[r])
        if n == 255:
            continue
        mine = recs[first:first + n]
        first += n
        pos = -1
        for rec in mine:  # a subsequence of the scan order, bit for bit
            hit = np.nonzero(np.all(hs[r] == rec, axis=1) & nz[r])[0]
            hit = hit[hit > pos]
            assert hit.size, f"row {r}: a stored record is not one of its half-spaces after position {pos}"
            pos = hit[0]
        if g0 is not None:
            c0, c1, c2 = centres[r]
            best = -100000000.0
            for rec in mine:
                v = (rec[0] * c0 + rec[1] * c1 + rec[2] * c2) - rec[3]
                if v > best:
                    best = v
            full = -100000000.0
            for q in np.nonzero(nz[r])[0]:
                v = (hs[r, q, 0] * c0 + hs[r, q, 1] * c1 + hs[r, q, 2] * c2) - hs[r, q, 3]
                if v > full:
                    full = v
            row = NF * T + (l[r] * T + t[r]) * O + o[r]
            assert -best == g0[row] and best == full


def _oracle_check(eng, ref, ks, tol=1e-9):
    for k in ks:
        g, jac = eng.eval(k)
        assert np.max(np.abs(g[0] - ref.eval_g(k))) <= tol
        assert np.max(np.abs(jac[0] - ref.eval_jac_g(k))) <= tol


def test_gripper_model_image(built):
    from armour_b200 import ReachSetEngine, worlds
    from oracle.pyoracle import OracleProblem
    q0, qd0, qdd0, q_des, obs = worlds.random_problems(1, 5, seed=11)
    eng = ReachSetEngine(max_problems=1, max_obstacles=5, robot_model=1, cap_link=64, cap_torque=128)
    eng.build(q0[0], qd0[0], qdd0[0], obs[0])
    assert eng.NJ == 8
    _check_images(eng, obs=obs, g0=eng.eval(K_TEST)[0][0])
    ref = OracleProblem(model_id=1).build(q0[0], qd0[0], qdd0[0], obs[0])
    _oracle_check(eng, ref, [np.zeros(7), K_TEST, 1.5 * np.ones(7)])


def test_no_obstacles_image(built):
    from armour_b200 import ReachSetEngine, worlds
    from oracle.pyoracle import OracleProblem
    q0, qd0, qdd0, q_des, obs = worlds.random_problems(1, 1, seed=3)
    eng = ReachSetEngine(max_problems=1, max_obstacles=4)
    eng.build(q0[0], qd0[0], qdd0[0], np.zeros((0, 12)))
    _check_images(eng)
    ref = OracleProblem().build(q0[0], qd0[0], qdd0[0], np.zeros((0, 12)))
    _oracle_check(eng, ref, [np.zeros(7), K_TEST])


def test_import_path_image(built):
    from armour_b200 import ReachSetEngine, worlds
    from oracle.pyoracle import OracleProblem
    q0, qd0, qdd0, q_des, obs = worlds.config1_problem(os.path.join(WORLDS, "scene_016_006.csv"))
    ref = OracleProblem().build(q0, qd0, qdd0, obs)
    eng = ReachSetEngine(max_problems=1, max_obstacles=obs.shape[0])
    eng.import_reachsets(0, 1, ref.tables(), q0, qd0, qdd0, obs)
    _check_images(eng, obs=obs[None], g0=eng.eval(K_TEST)[0][0])
    _oracle_check(eng, ref, [np.zeros(7), K_TEST, -np.ones(7), 2.0 * np.ones(7)], tol=1e-12)


def test_capacity_failure_batch_image(built):
    """A batch in which some problems overflow their tables: those evaluate to fail-safe rows, the others are
    bit-identical to the same batch built with room to spare (their images are packed normally)."""
    from armour_b200 import ArmourError, ReachSetEngine, worlds
    n = 16
    q0, qd0, qdd0, q_des, obs = worlds.random_problems(n, 6, seed=8)
    # a link or torque capacity (multiple of 8) between the smallest and the largest table maximum of the batch's problems
    probe = ReachSetEngine(max_problems=n, max_obstacles=6)
    probe.build(q0, qd0, qdd0, obs)
    ln, un = probe.monomial_counts()
    ml, mu = ln.reshape(n, -1).max(axis=1), un.reshape(n, -1).max(axis=1)
    split = [(c, 64) for c in range(8, 33, 8) if ml.min() <= c < ml.max()]
    split += [(32, c) for c in range(8, 65, 8) if mu.min() <= c < mu.max()]
    assert split, f"the batch's tables are too alike to split it by capacity: {ml} {mu}"
    cl, cu = split[0]
    must_fail = {p for p in range(n) if ml[p] > cl or mu[p] > cu}
    eng = ReachSetEngine(max_problems=n, max_obstacles=6, cap_link=cl, cap_torque=cu)
    with pytest.raises(ArmourError) as ei:
        eng.build(q0, qd0, qdd0, obs)
    assert ei.value.code == -4
    eng.nprob, eng.nobs = n, 6  # (the Python mirror only records a successful build)
    failed = {p for p, s in enumerate(eng.build_status()) if s != 0}
    assert must_fail <= failed and len(failed) < n
    g, jac = eng.eval(np.vstack([K_TEST] * n))
    _check_images(eng, failed, obs=obs, g0=g[0] if 0 not in failed else None)
    g1, j1 = probe.eval(np.vstack([K_TEST] * n))
    for p in range(n):
        if p in failed:
            assert np.all(g[p][:7 * 128 + 7 * 128 * 6] >= 1e299)
        else:
            assert np.array_equal(g1[p], g[p]) and np.array_equal(j1[p], jac[p])


def test_out_of_domain_rows_forty_obstacles(built):
    """Every row at a k outside the box the lists were built for goes to k_constraints_slow; inside the box the rows come
    from the image.  40 obstacles: 2 240 rows per chunk, three tiles of the pack kernel.  Checked against the oracle."""
    from armour_b200 import ReachSetEngine, worlds
    from oracle.pyoracle import OracleProblem
    q0, qd0, qdd0, q_des, obs = worlds.random_problems(1, 40, seed=21)
    eng = ReachSetEngine(max_problems=1, max_obstacles=40)
    eng.build(q0[0], qd0[0], qdd0[0], obs[0])
    _check_images(eng, obs=obs, g0=eng.eval(K_TEST)[0][0])
    ref = OracleProblem().build(q0[0], qd0[0], qdd0[0], obs[0])
    _oracle_check(eng, ref, [K_TEST, 1.2 * np.ones(7)])


def test_solver_subbatch_reads_the_right_images(built):
    """The batched solver evaluates its still-running worlds through a problem list: each world's result equals the
    same world solved alone."""
    from armour_b200 import ReachSetEngine, worlds
    n = 6
    q0, qd0, qdd0, q_des, obs = worlds.random_problems(n, 10, seed=31)
    eng = ReachSetEngine(max_problems=n, max_obstacles=10)
    eng.build(q0, qd0, qdd0, obs)
    _check_images(eng, obs=obs)
    k, ok, first, iters = eng.solve(q_des)
    assert len(set(iters.tolist())) > 1, "worlds finish at different iterations: later evaluations run on a sub-batch"
    for p in (int(np.argmax(iters)), int(np.argmin(iters))):
        one = ReachSetEngine(max_problems=1, max_obstacles=10)
        one.build(q0[p], qd0[p], qdd0[p], obs[p])
        k1, ok1, first1, it1 = one.solve(q_des[p:p + 1])
        assert np.array_equal(k1[0], k[p]) and ok1[0] == ok[p] and it1[0] == iters[p]


def test_later_context_with_fewer_obstacles(built):
    """Contexts are independent: creating one for fewer obstacles does not limit the builds of one created earlier for
    more, and a context may be created for many obstacles."""
    from armour_b200 import ReachSetEngine, worlds
    from oracle.pyoracle import OracleProblem
    q0, qd0, qdd0, q_des, obs = worlds.random_problems(2, 20, seed=13)
    big = ReachSetEngine(max_problems=2, max_obstacles=40)
    small = ReachSetEngine(max_problems=1, max_obstacles=4)
    small.build(q0[0], qd0[0], qdd0[0], obs[0][:4])
    big.build(q0, qd0, qdd0, obs)
    g = big.eval(np.vstack([K_TEST] * 2))[0]
    _check_images(big, obs=obs, g0=g[0])
    ref = OracleProblem().build(q0[1], qd0[1], qdd0[1], obs[1])
    assert np.max(np.abs(g[1] - ref.eval_g(K_TEST))) <= 1e-9
    ReachSetEngine(max_problems=1, max_obstacles=2000)


def test_overflow_rows_image(built):
    """A world with rows of more than HP_CAP candidates (world 427 of the 40-obstacle generator at seed 6: 99 such rows):
    those rows store no records, the pack skips them, k_constraints_slow evaluates them.  Checked against the oracle."""
    from armour_b200 import ReachSetEngine, worlds
    from oracle.pyoracle import OracleProblem
    q0, qd0, qdd0, q_des, obs = worlds.random_problems(1024, 40, seed=6)
    w = [427, 19]
    eng = ReachSetEngine(max_problems=2, max_obstacles=40)
    eng.build(q0[w], qd0[w], qdd0[w], obs[w])
    assert (eng.candidate_counts()[0] == 255).sum() > 0, "the world has overflow rows"
    g = eng.eval(np.vstack([K_TEST] * 2))[0]
    _check_images(eng, obs=obs[w], g0=g[0])
    ref = OracleProblem().build(q0[427], qd0[427], qdd0[427], obs[427])
    assert np.max(np.abs(g[0] - ref.eval_g(K_TEST))) <= 1e-9
