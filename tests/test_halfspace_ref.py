"""The host certificate checker of the collision candidate lists (tests/halfspace_ref.py) on the oracle's tables and on
constructed rows: it accepts sound prunings and flags every half-space dropped although it can win somewhere in the box."""
import os
import time

import numpy as np
import pytest

from conftest import WORLDS
from halfspace_ref import (K_DOMAIN, NPLANES, certify, certify_row, full_scan, monomial_degrees, monomials, row_inputs)

K_TEST = np.array([0.5, 0.6, 0.7, 0.0, -0.5, -0.6, -0.7])


@pytest.fixture(scope="module")
def world():
    """Every collision row of a saved ten-obstacle world, from the oracle's k-only tables (g order (l * T + t) * O + o)."""
    from armour_b200 import worlds
    from oracle.pyoracle import OracleProblem
    q0, qd0, qdd0, q_des, obs = worlds.config1_problem(os.path.join(WORLDS, "scene_016_006.csv"))
    ref = OracleProblem().build(q0, qd0, qdd0, obs)
    T, NJ, O = ref.T, ref.NJ, obs.shape[0]
    x = np.arange(NJ * T * O)
    o, t, l = x % O, (x // O) % T, x // (O * T)
    return ref, row_inputs(ref.tables(), obs, t, l, o)


def _kernel_pruning(A, b, nz, c, gm, rho_scale=1.0 + 3e-5):
    """Binary64 model of k_hyperplanes' filters (interval bound, pairwise test against the holder of the best lower
    bound, same normal): the kept mask [rows, 72]."""
    R = A.shape[0]
    vc = (A[..., 0] * c[:, None, 0] + A[..., 1] * c[:, None, 1] + A[..., 2] * c[:, None, 2]) - b
    slop = 1e-10 + 1e-12 * (np.abs(vc[:, 0::2] + b[:, 0::2]) + np.abs(b[:, 0::2]) + np.abs(b[:, 1::2]))
    rho = np.repeat(np.abs(np.einsum("rpe,rme->rpm", A[:, 0::2], gm)).sum(axis=2) * rho_scale + slop, 2, axis=1)
    up = np.where(nz, vc + rho, -1e300)
    lo = np.where(nz[:, 0::2], np.maximum(vc[:, 0::2], vc[:, 1::2]) - rho[:, 0::2], -1e300)
    bi = np.argmax(lo, axis=1)
    lo_max = np.maximum(lo[np.arange(R), bi], -100000000.0)
    jb = 2 * bi + (vc[np.arange(R), 2 * bi + 1] > vc[np.arange(R), 2 * bi])
    rr = np.arange(R)[:, None]
    D = A[rr, jb[:, None]] - A
    rd = np.abs(np.einsum("rpe,rme->rpm", D, gm)).sum(axis=2)
    vj, bj = vc[rr, jb[:, None]], b[rr, jb[:, None]]
    margin = rd * rho_scale + (1e-10 + 1e-12 * (np.abs(vc) + np.abs(vj) + np.abs(b) + np.abs(bj)))
    drop = ((vj - vc) > margin) & (np.arange(NPLANES)[None] != jb[:, None])
    listed = nz & (up >= lo_max[:, None]) & ~drop
    same = np.all(A[:, :, None] == A[:, None, :], axis=3) & (b[:, :, None] <= b[:, None, :]) & listed[:, :, None]
    same &= np.arange(NPLANES)[:, None] < np.arange(NPLANES)[None, :]
    return listed & ~same.any(axis=1)


def test_full_candidate_set_certifies(world):
    """Nothing dropped: nothing to certify, and every degenerate pair is left alone."""
    _, (A, b, nz, c, gm, deg, _) = world
    res = certify(A, b, nz, c, gm, deg, nz.copy(), K_DOMAIN)
    assert not res.failures and res.n_dropped == 0 and res.n_kept == int(nz.sum())
    assert deg.max() <= 21


def test_kernel_filters_certify_on_a_whole_world(world):
    """The filters of k_hyperplanes, restated in binary64 on the host, keep about two half-spaces per row; every other
    one carries a certificate, and the whole world (8 960 rows) certifies in seconds."""
    _, (A, b, nz, c, gm, deg, _) = world
    kept = _kernel_pruning(A, b, nz, c, gm)
    t0 = time.perf_counter()
    res = certify(A, b, nz, c, gm, deg, kept, K_DOMAIN)
    dt = time.perf_counter() - t0
    assert not res.failures, res
    assert res.n_a > 0 and res.n_b > 0 and res.n_kept < 4 * A.shape[0], res
    assert dt < 15.0, dt


def test_halved_variation_bound_is_flagged(world):
    """The same filters with the variation bounds halved drop half-spaces that can still win: the checker names them."""
    _, (A, b, nz, c, gm, deg, _) = world
    res = certify(A, b, nz, c, gm, deg, _kernel_pruning(A, b, nz, c, gm, rho_scale=0.5), K_DOMAIN)
    assert res.failures and min(g for _, _, g in res.failures) < -1e-9, res


def test_a_dropped_winner_is_flagged(world):
    """Remove by hand the half-space that wins a row at some k of the box: the checker names that row and plane."""
    ref, (A, b, nz, c, gm, deg, keys) = world
    rows = np.arange(0, A.shape[0], 97)
    for k in (K_TEST, -np.ones(7)):
        p = np.stack([c[r] + monomials(keys[r], k)[0][0] @ gm[r] for r in rows])
        val, win = full_scan(A[rows], b[rows], nz[rows], p)
        v = np.where(nz[rows], (A[rows] @ p[:, :, None])[..., 0] - b[rows], -np.inf)
        second = np.sort(v, axis=1)[:, -2]
        r_i = int(np.argmax(val - second))          # the clearest winner among the sampled rows
        r, i = int(rows[r_i]), int(win[r_i])
        g = ref.eval_g(k)
        assert g[7 * ref.T + r] == pytest.approx(-val[r_i], abs=1e-12)
        kept = nz[r].copy()
        kept[i] = False
        res = certify_row(A[r], b[r], nz[r], c[r], gm[r], deg[r], np.nonzero(kept)[0], K_DOMAIN)
        assert [(f[0], f[1]) for f in res.failures] == [(0, i)] and res.failures[0][2] <= 0


def _constructed_row(b2):
    """Two pairs: plane 0 = (e_x, 0), plane 2 = ((0.6, 0.8, 0), b2); planes 1, 3 far below; every other pair degenerate.
    p(k) = (mu(k), 0, 0) with mu = k_0^3 ... k_6^3 (total degree 21).  v_2 - v_0 = -0.4 mu - b2: plane 2 wins where
    mu < -b2 / 0.4."""
    A = np.zeros((NPLANES, 3))
    b = np.zeros(NPLANES)
    nz = np.zeros(NPLANES, bool)
    A[0], A[1], A[2], A[3] = (1, 0, 0), (-1, 0, 0), (0.6, 0.8, 0), (-0.6, -0.8, 0)
    b[1], b[2], b[3] = 10.0, b2, 10.0
    nz[:4] = True
    keys = np.array([0x3FFF], np.uint64)
    return A, b, nz, np.zeros(3), np.array([[1.0, 0.0, 0.0]]), monomial_degrees(keys), keys


def test_degree_bound_matters():
    """Plane 2 is dominated for |k_j| <= 1 but wins at k = -K_DOMAIN (all seven): the checker must accept it at kdom = 1
    and flag it at K_DOMAIN, which needs the exact K_DOMAIN^21 of its degree-21 monomial."""
    A, b, nz, c, gm, deg, keys = _constructed_row(0.4 * (1 + 1e-5))
    assert deg.tolist() == [21]
    assert not certify_row(A, b, nz, c, gm, deg, [0], 1.0).failures
    res = certify_row(A, b, nz, c, gm, deg, [0], K_DOMAIN)
    assert [(f[0], f[1]) for f in res.failures] == [(0, 2)]
    p = c + monomials(keys, -K_DOMAIN * np.ones(7))[0][0] @ gm
    assert full_scan(A, b, nz, p)[1] == 2
    p = c + monomials(keys, -np.ones(7))[0][0] @ gm
    assert full_scan(A, b, nz, p)[1] == 0


def test_duplicate_normal_row():
    """A later plane with the same normal, bit for bit, and an offset >= the earlier one's is dropped by certificate (c)
    alone (its pairwise gap is exactly 0); dropping the EARLIER of two equal planes instead changes the first attaining
    index and is flagged."""
    A, b, nz, c, gm, deg, _ = _constructed_row(0.5)
    A[4], b[4], A[5], b[5] = A[0], b[0], A[1], b[1] + 1.0
    nz[4:6] = True
    res = certify_row(A, b, nz, c, gm, deg, [0], K_DOMAIN)
    assert not res.failures and res.n_c == 1, res
    res = certify_row(A, b, nz, c, gm, deg, [4], K_DOMAIN)
    assert [(f[0], f[1]) for f in res.failures] == [(0, 0)] and res.failures[0][2] == 0.0


def test_monomial_degrees():
    assert monomial_degrees(np.array([0, 1, 2, 3, 0x3FFF, 0b01_00_11_10], np.uint64)).tolist() == [0, 1, 2, 3, 21, 6]
    with pytest.raises(ValueError):
        monomial_degrees(np.array([1 << 14], np.uint64))
