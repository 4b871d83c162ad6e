"""Collision rows of k_constraints, bit for bit.  Every listed collision row of problem 0 is recomputed on the host from the
decoded evaluation image: the same expression (n . c) - b at the sliced link centres, a sequential strict '>' scan from
-1e8 (KPR/CollisionChecking.cu:264-276), and g = -max; a row that no record wins has a zero Jacobian row.  Any reordering
of the row phase (DESIGN §3 K3) must keep this.  The worlds are chosen so that the 32 rows of one warp pass hold more than
32 records, the counts and row-group bases are read from global memory (40 obstacles), and exact ties occur (the arm at
rest among axis-aligned boxes, the tie points of the certificate tests)."""
import numpy as np
import pytest

from halfspace_ref import NF, chunk_candidates, chunk_rows, kept_planes, row_inputs
from test_candidate_certificates_gpu import _axis_boxes, _tie_points

pytestmark = pytest.mark.gpu
K_TEST = np.array([0.5, 0.6, 0.7, 0.0, -0.5, -0.6, -0.7])


def _decode(eng, ob):
    """The listed collision rows of problem 0: g-row index, interval, link and records (padded to the longest list, with
    their count), the kept masks [NJ*T*O, 72] in g-row order (for the tie points), and the largest number of records the
    32 rows of one pass hold."""
    img, lay = eng.eval_images()
    T, NJ, O = eng.T, eng.NJ, ob.shape[0]
    C_ = eng.lib.armour_chunk_intervals()
    ex = eng.export_reachsets(0)
    ex["hl"] &= np.uint64(0xFFFF)
    kept0 = np.zeros((NJ * T * O, 72), bool)
    out, pass_max = [], 0
    for tb in range(T // C_):
        t, l, o = chunk_rows(NJ, C_, O, tb)
        cnt, _, recs, first = chunk_candidates(img[0, tb], lay, len(t))
        stored = np.where(cnt == 255, 0, cnt).astype(np.int64)
        pass_max = max(pass_max, int(np.add.reduceat(stored, np.arange(0, len(t), 32)).max()))
        A, b, nz, _, _, _, _ = row_inputs(ex, ob, t, l, o)
        kept, _ = kept_planes(A, b, nz, cnt, recs, first)
        g_row = (l * T + t) * O + o
        kept0[g_row] = kept
        live = np.nonzero(cnt != 255)[0]
        pad = np.zeros((len(live), 32, 4))
        for s in range(int(stored.max(initial=0))):
            on = stored[live] > s
            pad[on, s] = recs[first[live[on]] + s]
        out.append((g_row[live], t[live], l[live], pad, stored[live]))
    rows = tuple(np.concatenate(a) for a in zip(*out))
    return rows, kept0, ex, pass_max


def _check_at(eng, rows, k):
    """Evaluate problem 0 at k and compare every listed collision row with the sequential scan, bit for bit."""
    g, jac = eng.eval(k[None])
    centres = eng.link_sliced_center()  # [T, NJ, 3]: the centres the kernel's rows use
    g_row, t, l, recs, n = rows
    c = centres[t, l]
    best = np.full(len(n), -100000000.0)
    win = np.full(len(n), -1)
    for s in range(int(n.max(initial=0))):
        r = recs[:, s]
        v = (r[:, 0] * c[:, 0] + r[:, 1] * c[:, 1] + r[:, 2] * c[:, 2]) - r[:, 3]
        with np.errstate(invalid="ignore"):
            up = (n > s) & (v > best)
        best = np.where(up, v, best)
        win = np.where(up, s, win)
    coll = NF * eng.T
    got = g[0, coll + g_row]
    bad = np.nonzero(got.view(np.int64) != (-best).view(np.int64))[0]
    assert bad.size == 0, (f"k = {k.tolist()}: {bad.size} rows differ from the sequential scan, e.g. row {g_row[bad[0]]} "
                           f"({n[bad[0]]} records): g {got[bad[0]]!r}, scan {-best[bad[0]]!r}")
    assert not np.any(jac[0, coll + g_row[win < 0]]), f"k = {k.tolist()}: a row without a winner has a Jacobian"


def _run(tag, eng, ob, ks, min_pass=33):
    rows, kept0, ex, pass_max = _decode(eng, ob)
    print(f"\n{tag}: {len(rows[0])} listed rows, up to {pass_max} records in one pass of 32 rows")
    assert pass_max >= min_pass, f"{tag}: no pass crosses a step of 32 records"
    ks = list(ks) + _tie_points(ex, ob, eng.T, eng.NJ, kept0, 8, np.random.default_rng(3))
    for k in ks:
        _check_at(eng, rows, np.asarray(k, dtype=np.float64))


def _engine(q0, qd0, qdd0, ob, **kw):
    from armour_b200 import ReachSetEngine
    eng = ReachSetEngine(max_problems=1, max_obstacles=ob.shape[0], **kw)
    eng.build(q0, qd0, qdd0, ob)
    assert eng.build_status()[0] == 0
    return eng


def test_long_link_tables(built):
    """simplify_threshold 5e-5 (config 4): longer tables, more candidates per row."""
    from armour_b200 import worlds
    q0, qd0, qdd0, _, obs = worlds.random_problems(1, 10, seed=4)
    eng = _engine(q0[0], qd0[0], qdd0[0], obs[0], simplify_threshold=5e-5, cap_link=128, cap_torque=256, cap_work=4096)
    _run("5e-5", eng, obs[0], [np.zeros(NF), K_TEST])
    eng.close()


def test_many_boxes_on_the_swept_links(built):
    """Ten boxes centred on the links' sliced centres at k = 0: the passes of those links hold many records."""
    from armour_b200 import worlds
    q0, qd0, qdd0, _, obs = worlds.random_problems(1, 10, seed=17)
    eng = _engine(q0[0], qd0[0], qdd0[0], obs[0])
    eng.eval(np.zeros((1, NF)))
    cen = eng.link_sliced_center()
    eng.close()
    tl = [(8, 3), (20, 4), (36, 5), (50, 6), (64, 4), (77, 5), (90, 6), (101, 3), (115, 5), (126, 6)]
    ob = worlds.boxes_to_zonotopes(np.array([np.r_[cen[t, l], 0.05, 0.06, 0.07] for t, l in tl]))
    eng = _engine(q0[0], qd0[0], qdd0[0], ob)
    _run("swept", eng, ob, [np.zeros(NF), K_TEST, np.full(NF, 0.9)])
    eng.close()


def test_forty_obstacles(built):
    """2 240 rows per chunk: the counts and row-group bases are read from global memory."""
    from armour_b200 import worlds
    q0, qd0, qdd0, _, obs = worlds.random_problems(1, 40, seed=29)
    eng = _engine(q0[0], qd0[0], qdd0[0], obs[0])
    assert eng.NJ * eng.lib.armour_chunk_intervals() * 40 > 2048
    _run("O=40", eng, obs[0], [np.zeros(NF), K_TEST])
    eng.close()


def test_arm_at_rest_among_axis_aligned_boxes(built):
    """qd0 = qdd0 = 0, links along the base axes, axis-aligned boxes: exact ties between stored half-spaces."""
    z = np.zeros(NF)
    ob = _axis_boxes()
    for q0 in (np.zeros(NF), np.array([0.0, np.pi / 2, 0.0, -np.pi / 2, 0.0, 0.0, 0.0])):
        eng = _engine(q0, z, z, ob)
        _run("rest", eng, ob, [np.zeros(NF), K_TEST], min_pass=1)
        eng.close()
