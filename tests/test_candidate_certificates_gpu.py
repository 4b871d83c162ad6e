"""Exactness of the collision candidate lists (DESIGN §3 K3a).  k_hyperplanes stores, per (link, interval, obstacle) row,
only the half-spaces that can attain the row maximum for some |k_j| <= K_DOMAIN.  For worlds chosen for the edges of its
filters, every row of every built problem is decoded from its evaluation image and each half-space left out must carry an
exact certificate (tests/halfspace_ref.py), for the device build and for the import of the oracle's tables.  Then the
evaluation is compared with the oracle's full scan where the stored lists are most likely to be wrong: at the points of
the box where the two best stored half-spaces of a row tie, just beside them, and on the edge of K_DOMAIN."""
import os

import numpy as np
import pytest
from scipy.optimize import minimize

from conftest import WORLDS
from halfspace_ref import (K_DOMAIN, MAX_LINK_DEGREE, NF, Certificates, certify, chunk_candidates, chunk_rows,
                           full_scan, kept_planes, monomials, row_inputs)

pytestmark = pytest.mark.gpu
EDGE = (1.0 + 5e-7, K_DOMAIN, float(np.nextafter(K_DOMAIN, 2.0)))  # list path, list path, generators path


def _certify_images(eng, obs, tag):
    """Certify every row of every successfully built problem of eng (obstacles obs [nprob, O, 12]).  Returns the merged
    Certificates, the mean kept / certified-dropped ratio per problem and the kept masks of problem 0 in g-row order."""
    img, lay = eng.eval_images()
    T, NJ, O = eng.T, eng.NJ, obs.shape[1]
    C_ = eng.lib.armour_chunk_intervals()
    status = eng.build_status()
    total, ratios = Certificates(), []
    kept0 = np.zeros((NJ * T * O, 72), bool)
    for p in range(eng.nprob):
        if status[p] != 0:
            continue
        ex = eng.export_reachsets(p)
        ex["hl"] &= np.uint64(0xFFFF)
        per = Certificates()
        for tb in range(T // C_):
            t, l, o = chunk_rows(NJ, C_, O, tb)
            A, b, nz, c, gm, deg, _ = row_inputs(ex, obs[p], t, l, o)
            assert deg.max(initial=0) <= MAX_LINK_DEGREE, f"{tag}: a link monomial of degree {deg.max()}"
            cnt, _, recs, first = chunk_candidates(img[p, tb], lay, len(t))
            kept, skip = kept_planes(A, b, nz, cnt, recs, first)
            assert np.all(cnt[skip] == 255), f"{tag}: problem {p} chunk {tb}: records that are not the row's half-spaces"
            live = np.setdiff1d(np.arange(len(t)), skip)
            res = certify(A[live], b[live], nz[live], c[live], gm[live], deg[live], kept[live], K_DOMAIN)
            for r, i, gap in res.failures:
                x = live[r]
                pytest.fail(f"{tag}: problem {p}, row (link {l[x]}, interval {t[x]}, obstacle {o[x]}): half-space {i} "
                            f"dropped without a certificate (best gap {gap:.3e}); {len(res.failures)} such")
            per.merge(res)
            if p == 0:
                kept0[(l * T + t) * O + o] = kept
        ratios.append(per.n_kept / max(per.n_dropped, 1))
        total.merge(per)
    print(f"\n{tag}: {total}; kept / dropped {np.mean(ratios):.4f}")
    return total, float(np.mean(ratios)), kept0


def _tie_points(tables, ob, T, NJ, kept, nrows, rng):
    """Points of the box where the two best stored half-spaces (at k = 0) of a row tie, and the same points moved by
    +-1e-9 along the gradient of their difference; nrows rows with at least two stored half-spaces, spread over the
    world."""
    O = ob.shape[0]
    multi = np.nonzero(kept.sum(axis=1) >= 2)[0]
    if multi.size == 0:
        return []
    rows = multi[np.linspace(0, multi.size - 1, min(nrows, multi.size)).astype(int)]
    o, t, l = rows % O, (rows // O) % T, rows // (O * T)
    A, b, nz, c, gm, deg, keys = row_inputs(tables, ob, t, l, o)
    ks = []
    for r in range(len(rows)):
        K = np.nonzero(kept[rows[r]])[0]
        v0 = A[r, K] @ c[r] - b[r, K]
        ia, ib = K[np.argsort(-v0, kind="stable")[:2]]
        D, db = A[r, ia] - A[r, ib], b[r, ia] - b[r, ib]
        Dg = gm[r] @ D                                                   # [M]

        def f(k):
            mu, dmu = monomials(keys[r], k)
            diff = D @ c[r] + mu[0] @ Dg - db
            return diff * diff, 2 * diff * (Dg @ dmu[0])

        best = min((minimize(f, x0, jac=True, method="L-BFGS-B", bounds=[(-1, 1)] * NF)
                    for x0 in rng.uniform(-1, 1, (3, NF))), key=lambda s: s.fun)
        k = best.x
        grad = Dg @ monomials(keys[r], k)[1][0]
        ks.append(k)
        if np.linalg.norm(grad) > 0:
            u = grad / np.linalg.norm(grad)
            ks += [k + 1e-9 * u, k - 1e-9 * u]
    return ks


def _edge_points():
    ks = []
    for v in EDGE:
        for j in range(NF):
            k = np.zeros(NF)
            k[j] = v if j % 2 == 0 else -v
            ks.append(k)
        ks += [np.full(NF, v), np.full(NF, -v)]
    return ks


def _adversarial(tag, q0, qd0, qdd0, ob, eng_kw=None, ref_kw=None, tables_kw=None, nrows=8, seed=0):
    """Import the oracle's tables of one world into P problem slots, certify its lists, and evaluate P points at once:
    tie points of stored half-spaces and K_DOMAIN edge points, each against the oracle's full scan."""
    from armour_b200 import ReachSetEngine
    from oracle.pyoracle import OracleProblem
    eng_kw, ref_kw, tables_kw = eng_kw or {}, ref_kw or {}, tables_kw or {}
    ref = OracleProblem(max_obstacles=max(ob.shape[0], 1), **ref_kw).build(q0, qd0, qdd0, ob)
    tables = ref.tables(**tables_kw)
    T, NJ, O = ref.T, ref.NJ, ob.shape[0]
    one = ReachSetEngine(max_problems=1, max_obstacles=O, **eng_kw)
    one.import_reachsets(0, 1, tables, q0, qd0, qdd0, ob)
    res, ratio, kept = _certify_images(one, ob[None], tag + " (import)")
    one.close()
    ks = np.array(_tie_points(tables, ob, T, NJ, kept, nrows, np.random.default_rng(seed)) + _edge_points())
    P = len(ks)
    eng = ReachSetEngine(max_problems=P, max_obstacles=O, **eng_kw)
    for p in range(P):
        eng.import_reachsets(p, P, tables, q0, qd0, qdd0, ob)
    g, jac = eng.eval(ks)
    coll = NF * T
    for p, k in enumerate(ks):
        g_ref, j_ref = ref.eval_g(k), ref.eval_jac_g(k)
        err = np.abs(g[p] - g_ref)
        assert err.max() <= 1e-12, f"{tag}: k = {k.tolist()}: g row {int(np.argmax(err))} off by {err.max():.3e}"
        bad = np.nonzero(np.abs(jac[p] - j_ref).max(axis=1) > 1e-12)[0]
        if bad.size == 0:
            continue
        # only a row whose two best half-spaces tie (within 1e-12) may carry the other one's gradient
        assert np.all((bad >= coll) & (bad < coll + NJ * T * O)), f"{tag}: k = {k.tolist()}: Jacobian rows {bad[:8]}"
        eng.eval(k[None])                                         # problem 0 holds the same world: its sliced centres
        centres = eng.link_sliced_center()
        x = bad - coll
        o, t, l = x % O, (x // O) % T, x // (O * T)
        A, b, nz, _, _, _, _ = row_inputs(tables, ob, t, l, o)
        pc = centres[t, l]
        v = np.where(nz, (A[..., 0] * pc[:, None, 0] + A[..., 1] * pc[:, None, 1] + A[..., 2] * pc[:, None, 2]) - b, -np.inf)
        top = np.sort(v, axis=1)[:, -2:]
        assert np.all(top[:, 1] - top[:, 0] < 1e-12), (
            f"{tag}: k = {k.tolist()}: Jacobian rows {bad[top[:, 1] - top[:, 0] >= 1e-12][:8]} carry another plane's gradient "
            f"(full scan winners {full_scan(A, b, nz, pc)[1][:8]})")
    eng.close()
    return res, ratio


def _build_and_certify(tag, q0, qd0, qdd0, obs, **eng_kw):
    from armour_b200 import ReachSetEngine
    q0, qd0, qdd0 = (np.asarray(a, dtype=np.float64).reshape(-1, NF) for a in (q0, qd0, qdd0))
    obs = np.asarray(obs, dtype=np.float64).reshape(q0.shape[0], -1, 12)
    eng = ReachSetEngine(max_problems=q0.shape[0], max_obstacles=obs.shape[1], **eng_kw)
    eng.build(q0, qd0, qdd0, obs)
    out = _certify_images(eng, obs, tag + " (build)")
    return eng, out


@pytest.mark.parametrize("scene", ["scene_016_006", "scene_040_010"])
def test_saved_worlds(built, scene):
    from armour_b200 import worlds
    q0, qd0, qdd0, _, obs = worlds.config1_problem(os.path.join(WORLDS, scene + ".csv"))
    eng, _ = _build_and_certify(scene, q0, qd0, qdd0, obs)
    eng.close()
    _adversarial(scene, q0, qd0, qdd0, obs)


def test_throughput_batch_with_a_repeated_world(built):
    """Four problems (the batched build's throughput configuration), world 0 at slots 0 and 2: every slot certifies, and
    the repeated world stores the same lists at both slots."""
    from armour_b200 import worlds
    q0, qd0, qdd0, _, obs = worlds.random_problems(3, 10, seed=41)
    w = [0, 1, 0, 2]
    eng, _ = _build_and_certify("batch", q0[w], qd0[w], qdd0[w], obs[w])
    cnt = eng.candidate_counts()
    assert np.array_equal(cnt[0], cnt[2])
    img, _ = eng.eval_images()
    assert np.array_equal(img[0], img[2])
    eng.close()
    _adversarial("batch world 0", q0[0], qd0[0], qdd0[0], obs[0])


def _axis_boxes():
    from armour_b200 import worlds
    return worlds.boxes_to_zonotopes(np.array([[0.35, 0.0, 0.6, 0.2, 0.2, 0.2], [0.0, -0.4, 0.9, 0.1, 0.3, 0.2],
                                               [-0.3, 0.25, 0.3, 0.2, 0.1, 0.4], [0.0, 0.0, 1.5, 0.3, 0.3, 0.1],
                                               [0.5, 0.5, 0.2, 0.1, 0.1, 0.1]]))


def test_arm_at_rest_among_axis_aligned_boxes(built):
    """qd0 = qdd0 = 0 at q0 = 0 and at a pose with the links along the base axes, among axis-aligned boxes: exact ties,
    duplicate normals and degenerate generator pairs.  Certificate (c) and degenerate pairs must actually occur."""
    q0 = np.array([np.zeros(NF), [0.0, np.pi / 2, 0.0, -np.pi / 2, 0.0, 0.0, 0.0]])
    z = np.zeros((2, NF))
    obs = np.stack([_axis_boxes()] * 2)
    eng, (res, _, _) = _build_and_certify("rest", q0, z, z, obs)
    eng.close()
    assert res.n_c > 0 and res.n_degenerate > 0, res
    res, _ = _adversarial("rest q0 = 0", q0[0], z[0], z[0], obs[0])
    assert res.n_c > 0 and res.n_degenerate > 0, res


def test_boxes_on_the_swept_links(built):
    """Boxes centred on the links' sliced centres at k = 0: row values near 0 and below."""
    from armour_b200 import worlds
    from oracle.pyoracle import OracleProblem
    q0, qd0, qdd0, _, obs = worlds.random_problems(1, 3, seed=17)
    ref = OracleProblem().build(q0[0], qd0[0], qdd0[0], obs[0])
    ref.eval_g(np.zeros(NF))
    cen = ref.link_sliced_center()
    boxes = [np.r_[cen[t, l], 0.06, 0.05, 0.08] for t, l in ((10, 2), (64, 4), (120, 6))]
    ob = worlds.boxes_to_zonotopes(np.array(boxes))
    eng, _ = _build_and_certify("swept", q0[0], qd0[0], qdd0[0], ob)
    g = eng.eval(np.zeros(NF))[0][0]
    assert np.sum(g[NF * eng.T:NF * eng.T + eng.NJ * eng.T * 3] > 0) > 0, "some rows are in collision"
    eng.close()
    _adversarial("swept", q0[0], qd0[0], qdd0[0], ob)


def test_padded_obstacle_list(built):
    """worlds.pad_obstacles: 1 cm boxes 10 m away, |d| large next to small deltas."""
    from armour_b200 import worlds
    q0, qd0, qdd0, _, obs = worlds.random_problems(1, 3, seed=23)
    ob = worlds.pad_obstacles([obs[0]], 10)[0]
    eng, _ = _build_and_certify("padded", q0[0], qd0[0], qdd0[0], ob)
    eng.close()
    _adversarial("padded", q0[0], qd0[0], qdd0[0], ob)


@pytest.mark.parametrize("nobs", [1, 3, 5])
def test_obstacle_counts_off_the_row_groups(built, nobs):
    """Rows per chunk 56, 168, 280: not multiples of 32."""
    from armour_b200 import worlds
    q0, qd0, qdd0, _, obs = worlds.random_problems(2, nobs, seed=50 + nobs)
    eng, _ = _build_and_certify(f"O={nobs}", q0, qd0, qdd0, obs)
    eng.close()
    _adversarial(f"O={nobs}", q0[0], qd0[0], qdd0[0], obs[0], nrows=6)


def test_gripper_model_with_uncertainty(built):
    from armour_b200 import worlds
    q0, qd0, qdd0, _, obs = worlds.random_problems(1, 5, seed=11)
    unc = dict(mass_uncertainty=0.10, inertia_uncertainty=0.10)
    eng_kw = dict(robot_model=1, cap_link=64, cap_torque=128, **unc)
    eng, _ = _build_and_certify("gripper", q0[0], qd0[0], qdd0[0], obs[0], **eng_kw)
    assert eng.NJ == 8
    eng.close()
    _adversarial("gripper", q0[0], qd0[0], qdd0[0], obs[0], eng_kw=eng_kw, ref_kw=dict(model_id=1, **unc))


def test_long_link_tables(built):
    """simplify_threshold 5e-5 (config 4): link tables longer than the 24 monomials k_hyperplanes stages in shared
    memory, so that its variation sums continue from global memory."""
    from armour_b200 import worlds
    q0, qd0, qdd0, _, obs = worlds.random_problems(1, 10, seed=4)
    eng_kw = dict(simplify_threshold=5e-5, cap_link=128, cap_torque=256, cap_work=4096)
    eng, _ = _build_and_certify("5e-5", q0[0], qd0[0], qdd0[0], obs[0], **eng_kw)
    assert eng.monomial_counts()[0].max() > 24
    eng.close()
    _adversarial("5e-5", q0[0], qd0[0], qdd0[0], obs[0], eng_kw=eng_kw, ref_kw=dict(simplify_threshold=5e-5),
                 tables_kw=dict(cap_link=128, cap_u=256))
