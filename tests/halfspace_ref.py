"""Host reference for the collision half-space candidate lists (k_hyperplanes, DESIGN §3 K3a).

Each collision row of a (link, interval, obstacle) is the maximum over 72 signed half-spaces (A_i, b_i) of
v_i(k) = A_i . p(k) - b_i, where p(k) = c + sum_m g_m mu_m(k) is the sliced link centre and mu_m(k) a monomial of total
degree deg_m in k.  The build stores only a short list of those half-spaces per row.  certify() proves, in exact rational
arithmetic on the binary64 inputs, that every half-space left out can never be the first attaining maximum of the full
scan for any |k_j| <= kdom; full_scan() is that scan.  Needs no GPU: the GPU tests feed it decoded evaluation images,
the CPU tests feed it the oracle's tables."""
from fractions import Fraction

import numpy as np

NF = 7
NPLANES = 72
PAIRS = [(a, b) for a in range(8) for b in range(a + 1, 9)]  # generator pairs in the reference's scan order
EPS = 2.0 ** -53                                              # unit round-off of binary64
K_DOMAIN = 1.0 + 1e-6        # layout.h: the candidate lists are exact for |k_j| <= K_DOMAIN
MAX_LINK_DEGREE = 21         # layout.h: HP_RHO_SCALE >= K_DOMAIN^21


def half_spaces(G, oc):
    """All 72 signed half-spaces (s*C, b) of rows with generators G [rows, 9, 3] and obstacle centres oc [rows, 3], in scan
    order pos_0, neg_0, pos_1, ..., computed with the expressions of k_hyperplanes (no contraction): [rows, 72, 4] and the
    mask of non-degenerate normals [rows, 72]."""
    rows = G.shape[0]
    out = np.zeros((rows, NPLANES, 4))
    nzs = np.zeros((rows, NPLANES), bool)
    for i, (a, b) in enumerate(PAIRS):
        ga, gb = G[:, a], G[:, b]
        cx = ga[:, 1] * gb[:, 2] - ga[:, 2] * gb[:, 1]
        cy = ga[:, 2] * gb[:, 0] - ga[:, 0] * gb[:, 2]
        cz = ga[:, 0] * gb[:, 1] - ga[:, 1] * gb[:, 0]
        nrm = np.sqrt(cx * cx + cy * cy + cz * cz)
        safe = np.where(nrm > 0, nrm, 1.0)
        C0, C1, C2 = (np.where(nrm > 0, c / safe, 0.0) for c in (cx, cy, cz))
        d = C0 * oc[:, 0] + C1 * oc[:, 1] + C2 * oc[:, 2]
        delta = np.zeros(rows)
        for g in range(9):
            delta = delta + np.abs(C0 * G[:, g, 0] + C1 * G[:, g, 1] + C2 * G[:, g, 2])
        nz = np.sqrt(C0 * C0 + C1 * C1 + C2 * C2) > 0
        out[:, 2 * i] = np.stack([C0, C1, C2, d + delta], axis=1)
        out[:, 2 * i + 1] = np.stack([-C0, -C1, -C2, -d + delta], axis=1)
        nzs[:, 2 * i] = nzs[:, 2 * i + 1] = nz
    return out, nzs


def chunk_rows(NJ, C_, O, tb):
    """(t, l, o) of the rows of chunk tb in its x order x = (l * C_ + tt) * O + o."""
    x = np.arange(NJ * C_ * O)
    o, tt, l = x % O, (x // O) % C_, x // (O * C_)
    return tb * C_ + tt, l, o


def row_generators(ob, link_gens, t, l, o):
    """Generators [rows, 9, 3] (3 of the obstacle, then the 3 x 6 link matrix) and obstacle centres [rows, 3] of the rows
    (t, l, o); ob [O, 12], link_gens [T, NJ, 18] column-major."""
    G = np.concatenate([ob[o, 3:12].reshape(-1, 3, 3), link_gens[t, l].reshape(-1, 6, 3)], axis=1)
    return G, ob[o, 0:3]


def row_inputs(tables, ob, t, l, o):
    """Inputs of certify() for the rows (t, l, o) of one problem: the 72 half-spaces A [rows, 72, 3], b, nz [rows, 72],
    the sliced-centre polynomial c [rows, 3], gm [rows, M, 3] (zero padded), deg [rows, M], and its keys [rows, M].
    tables: the k-only link tables (nl, cl, gl, hl, link_gens [T, NJ, 18]) of export_reachsets / OracleProblem.tables."""
    NJ = tables["link_gens"].shape[1]
    G, oc = row_generators(ob, tables["link_gens"], t, l, o)
    hs, nz = half_spaces(G, oc)
    src = t * NJ + l
    n = tables["nl"][src]
    M = int(n.max(initial=0))
    live = np.arange(M)[None] < n[:, None]
    gm = np.where(live[..., None], tables["gl"][src, :M], 0.0)
    keys = np.where(live, tables["hl"][src, :M], 0).astype(np.uint64)
    return hs[..., :3], hs[..., 3], nz, tables["cl"][src], gm, monomial_degrees(keys), keys


def chunk_candidates(b, lay, rows):
    """Candidate lists of one chunk's evaluation image b (uint8): (counts uint8 [rows], row-group bases uint32, records
    [stored, 4] in CSR order, first record of each row [rows]).  A count of 255 (HP_OVERFLOW) stores no record."""
    d = b.view(np.float64)
    cnt = b[lay["counts"]:lay["counts"] + rows]
    stored = np.where(cnt == 255, 0, cnt).astype(np.int64)
    grp = b[lay["groups"]:lay["groups"] + 4 * ((rows + 31) // 32)].view(np.uint32)
    recs = d[lay["records"] // 8:lay["records"] // 8 + 4 * stored.sum()].reshape(-1, 4)
    first = np.concatenate([[0], np.cumsum(stored)])[:rows]
    return cnt, grp, recs, first


def kept_planes(A, b, nz, cnt, recs, first):
    """Match every row's stored records, bit for bit and in order, to a subsequence of its 72 half-spaces (the earliest
    match after the previous one).  Returns the kept mask [rows, 72] and the rows whose records do not match (or whose
    count is 255: those rows have no list)."""
    rows = A.shape[0]
    hs = np.concatenate([A, b[..., None]], axis=-1)
    kept = np.zeros((rows, NPLANES), bool)
    n = np.where(cnt == 255, 0, cnt).astype(np.int64)
    pos = np.full(rows, -1)
    bad = np.zeros(rows, bool)
    for s in range(int(n.max(initial=0))):
        r = np.nonzero(n > s)[0]
        rec = recs[first[r] + s]
        hit = np.all(hs[r] == rec[:, None, :], axis=2) & nz[r] & (np.arange(NPLANES)[None] > pos[r, None])
        ok = hit.any(axis=1)
        bad[r[~ok]] = True
        q = np.argmax(hit, axis=1)
        pos[r[ok]] = q[ok]
        kept[r[ok], q[ok]] = True
    return kept, np.nonzero(bad | (cnt == 255))[0]


def monomial_degrees(keys):
    """Total k-degree of each exported link monomial.  The degree hash gives each k_j two bits (oracle/pz.h, var_bits and
    hash_to_degree); a k-only monomial uses the low 2 * 7 bits, and a key with higher bits set is not one."""
    keys = np.asarray(keys).astype(np.uint64)
    if np.any(keys >> np.uint64(2 * NF)):
        raise ValueError("a monomial key with degrees outside k_0..k_6")
    return sum(((keys >> np.uint64(2 * j)) & np.uint64(3)).astype(np.int64) for j in range(NF))


def monomials(keys, k):
    """mu_m(k) [n, M] and d mu_m / d k [n, M, 7] of the monomials keys [M] at the points k [n, 7]."""
    keys = np.asarray(keys).astype(np.uint64)
    e = np.stack([((keys >> np.uint64(2 * j)) & np.uint64(3)).astype(np.int64) for j in range(NF)], axis=1)  # [M, 7]
    k = np.atleast_2d(k)
    pw = k[:, None, :] ** e[None]                                             # [n, M, 7]
    mu = np.prod(pw, axis=2)
    dmu = np.empty(mu.shape + (NF,))
    for j in range(NF):
        dj = np.where(e[None, :, j] > 0, e[None, :, j] * k[:, None, j] ** np.maximum(e[None, :, j] - 1, 0), 0.0)
        dmu[:, :, j] = dj * np.prod(np.delete(pw, j, axis=2), axis=2)
    return mu, dmu


def full_scan(A, b, nz, p):
    """Row value and first attaining index of the full scan under strict '>' from -1e8 (checkCollisionKernel), with the
    kernel's expression (A0 p0 + A1 p1 + A2 p2) - b.  A [..., 72, 3], b, nz [..., 72], p [..., 3]; index -1 when no
    half-space exceeds the start value."""
    v = (A[..., 0] * p[..., None, 0] + A[..., 1] * p[..., None, 1] + A[..., 2] * p[..., None, 2]) - b
    v = np.where(nz, v, -np.inf)
    i = np.argmax(v, axis=-1)
    best = np.take_along_axis(v, i[..., None], axis=-1)[..., 0]
    above = best > -100000000.0
    return np.where(above, best, -100000000.0), np.where(above, i, -1)


class Certificates:
    """Outcome of certify(): failures [(row, plane, best gap)], counts of certificates by kind, kept / droppable / degenerate
    planes, and the smallest gap among planes certified by (a) or (b) only."""

    def __init__(self):
        self.failures = []
        self.n_a = self.n_b = self.n_c = 0
        self.n_kept = self.n_dropped = self.n_degenerate = 0
        self.min_gap = np.inf

    def merge(self, o, row0=0):
        self.failures += [(r + row0, i, g) for r, i, g in o.failures]
        for f in ("n_a", "n_b", "n_c", "n_kept", "n_dropped", "n_degenerate"):
            setattr(self, f, getattr(self, f) + getattr(o, f))
        self.min_gap = min(self.min_gap, o.min_gap)

    def __repr__(self):
        return (f"Certificates(kept={self.n_kept}, dropped={self.n_dropped} [a={self.n_a} b={self.n_b} c={self.n_c}], "
                f"degenerate={self.n_degenerate}, min_gap={self.min_gap:.3e}, failures={self.failures[:5]})")


def _exact_terms(A, b, c, gm, wq):
    """Exact A . c - b and the exact |A . g_m| kdom^deg_m summed, for one half-space (rational)."""
    Af = [Fraction(float(x)) for x in A]
    vc = sum(Af[e] * Fraction(float(c[e])) for e in range(3)) - Fraction(float(b))
    rho = sum(abs(sum(Af[e] * Fraction(float(gm[m, e])) for e in range(3))) * wq[m] for m in range(gm.shape[0]))
    return vc, rho


def _exact_gap_a(A, b, nz, c, gm, wq, i):
    lo = [None] * NPLANES
    for q in range(0, NPLANES, 2):
        if nz[q]:
            vp, rho = _exact_terms(A[q], b[q], c, gm, wq)
            vn, _ = _exact_terms(A[q + 1], b[q + 1], c, gm, wq)
            lo[q] = max(vp, vn) - rho
    L = max(x for x in lo if x is not None)
    vi, rhoi = _exact_terms(A[i], b[i], c, gm, wq)
    return L - (vi + rhoi)


def _exact_gap_b(A, b, c, gm, wq, i, j):
    vi, _ = _exact_terms(A[i], b[i], c, gm, wq)
    vj, _ = _exact_terms(A[j], b[j], c, gm, wq)
    D = [Fraction(float(A[j, e])) - Fraction(float(A[i, e])) for e in range(3)]
    rd = sum(abs(sum(D[e] * Fraction(float(gm[m, e])) for e in range(3))) * wq[m] for m in range(gm.shape[0]))
    return (vj - vi) - rd


def certify(A, b, nz, c, gm, deg, kept, kdom, block=512):
    """Certify every non-degenerate half-space that is not kept, for rows A [R, 72, 3], b, nz, kept [R, 72], centres
    c [R, 3], monomial coefficients gm [R, M, 3] and total degrees deg [R, M] (padding: zero coefficients), |k_j| <= kdom.

    A dropped half-space i is certified by
      (a) U_i < L, U_i = A_i.c - b_i + sum_m |A_i.g_m| kdom^deg_m and L = max over the pairs of
          max(v_pos(c), v_neg(c)) - sum_m |C.g_m| kdom^deg_m (the row's guaranteed lower bound), or
      (b) (A_j.c - b_j) - (A_i.c - b_i) - sum_m |(A_j - A_i).g_m| kdom^deg_m > 0 for some half-space j, or
      (c) an earlier half-space with the same normal, bit for bit, and an offset <= b_i.
    Each must hold in exact arithmetic on the binary64 inputs.  (a) and (b) are evaluated in binary64 with the bound
    (3 M + 64) u S on the rounding error of the gap, S the same sums taken over absolute values of every term (u = 2^-53;
    it covers the M + 8 rounded additions of each sum and the rounding of kdom^deg); gaps inside that bound are decided
    with fractions.Fraction.  Candidates j of (b): the three pairs with the best lower bounds (larger centre value of the
    two signs) and every kept half-space; a certificate against any j suffices for exactness, and the kernel's own pairwise
    test is against the first of them."""
    out = Certificates()
    for r0 in range(0, A.shape[0], block):
        sl = slice(r0, r0 + block)
        part = _certify_block(A[sl], b[sl], nz[sl], c[sl], gm[sl], deg[sl], kept[sl], kdom)
        out.merge(part, r0)
    return out


def certify_row(A, b, nz, c, gm, deg, kept, kdom):
    """certify() for one row: A [72, 3], b, nz [72], c [3], gm [M, 3], deg [M], kept the indices of the stored planes."""
    mask = np.zeros(NPLANES, bool)
    mask[np.asarray(kept, dtype=np.int64)] = True
    return certify(A[None], b[None], nz[None], np.asarray(c)[None], np.asarray(gm).reshape(1, -1, 3),
                   np.asarray(deg).reshape(1, -1), mask[None], kdom)


def _certify_block(A, b, nz, c, gm, deg, kept, kdom):
    R, M = A.shape[0], gm.shape[1]
    res = Certificates()
    w = float(kdom) ** deg.astype(np.float64)                                # [R, M]
    tol = (3 * M + 64) * EPS
    vc = (A[..., 0] * c[:, None, 0] + A[..., 1] * c[:, None, 1] + A[..., 2] * c[:, None, 2]) - b
    Sc = np.abs(A[..., 0] * c[:, None, 0]) + np.abs(A[..., 1] * c[:, None, 1]) + np.abs(A[..., 2] * c[:, None, 2]) + np.abs(b)
    Ag = np.einsum("rpe,rme->rpm", A, gm)                                    # [R, 72, M]
    rho = np.einsum("rpm,rm->rp", np.abs(Ag), w)
    Srho = np.einsum("rpe,rme,rm->rp", np.abs(A), np.abs(gm), w)
    S = Sc + Srho                                                            # bounds every term of v_c and rho
    U = vc + rho
    lo = np.maximum(vc[:, 0::2], vc[:, 1::2]) - rho[:, 0::2]                 # [R, 36]
    lo = np.where(nz[:, 0::2], lo, -np.inf)
    L = lo.max(axis=1)
    SL = np.where(nz[:, 0::2], np.maximum(S[:, 0::2], S[:, 1::2]), 0.0).max(axis=1)
    drop = nz & ~kept
    res.n_kept = int((nz & kept).sum())
    res.n_dropped = int(drop.sum())
    res.n_degenerate = int((~nz).sum())
    if not drop.any():
        return res
    # (c): bit-identical normal earlier in the scan order, offset <= b_i
    same = np.all(A[:, :, None, :] == A[:, None, :, :], axis=3)              # [R, q, i]
    same &= nz[:, :, None] & (b[:, :, None] <= b[:, None, :])
    same &= np.arange(NPLANES)[:, None] < np.arange(NPLANES)[None, :]
    cert_c = drop & same.any(axis=1)
    # (a)
    gap_a = L[:, None] - U
    err_a = tol * (S + SL[:, None])
    cert_a = drop & (gap_a > err_a)
    open_a = drop & (np.abs(gap_a) <= err_a)
    # (b): candidates j per row
    best3 = np.argsort(-lo, axis=1, kind="stable")[:, :3]
    sgn = (np.take_along_axis(vc[:, 1::2], best3, 1) > np.take_along_axis(vc[:, 0::2], best3, 1)).astype(np.int64)
    cand = [(2 * best3[:, s] + sgn[:, s], np.take_along_axis(lo, best3[:, s:s + 1], 1)[:, 0] > -np.inf) for s in range(3)]
    nk = kept.sum(axis=1)
    order = np.argsort(~kept, axis=1, kind="stable")                         # kept planes first, in scan order
    cand += [(order[:, s], nk > s) for s in range(int(nk.max(initial=0)))]
    gap_b = np.full((R, NPLANES), -np.inf)
    cert_b = np.zeros((R, NPLANES), bool)
    open_b = {}                                                              # (r, i) -> undecided j
    need = drop & ~cert_a & ~cert_c
    for j, valid in cand:
        rr, ii = np.nonzero(need & valid[:, None])
        if rr.size == 0:
            continue
        jj = j[rr]
        D = A[rr, jj] - A[rr, ii]                                            # [P, 3]
        rd = np.einsum("pm,pm->p", np.abs(np.einsum("pe,pme->pm", D, gm[rr])), w[rr])
        g = (vc[rr, jj] - vc[rr, ii]) - rd
        err = tol * (S[rr, ii] + S[rr, jj])
        gap_b[rr, ii] = np.maximum(gap_b[rr, ii], g)
        cert_b[rr[g > err], ii[g > err]] = True
        for p_ in np.nonzero(np.abs(g) <= err)[0]:
            open_b.setdefault((rr[p_], ii[p_]), []).append(int(jj[p_]))
    # exact decisions where the binary64 gap is inside its error bound
    certified = cert_a | cert_b | cert_c
    wq = None
    for r, i in zip(*np.nonzero(drop & ~certified)):
        if wq is None or wq[0] != r:
            wq = (r, [Fraction(float(kdom)) ** int(d) for d in deg[r]])
        ok = False
        if open_a[r, i] and _exact_gap_a(A[r], b[r], nz[r], c[r], gm[r], wq[1], i) > 0:
            ok, kind = True, "a"
        for j_ in ([] if ok else open_b.get((r, i), [])):
            if _exact_gap_b(A[r], b[r], c[r], gm[r], wq[1], i, j_) > 0:
                ok, kind = True, "b"
                break
        if ok:
            (cert_a if kind == "a" else cert_b)[r, i] = True
        else:
            res.failures.append((int(r), int(i), float(max(gap_a[r, i], gap_b[r, i]))))
    cert_b &= ~cert_a
    res.n_a, res.n_b = int(cert_a.sum()), int(cert_b.sum())
    res.n_c = int((cert_c & ~cert_a & ~cert_b).sum())
    ab = (cert_a | cert_b) & ~cert_c
    if ab.any():
        res.min_gap = float(np.maximum(gap_a, gap_b)[ab].min())
    return res
