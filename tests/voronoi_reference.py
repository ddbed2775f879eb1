"""CPU reference of the Voronoi tessellation of ljmd_voronoi (csrc/voronoi.cu, rules in include/ljmd.h):
scipy.spatial.Voronoi (Qhull) on the fp32 sites promoted to double, with their periodic images in a margin strip.

The edge rule is the kernel's: a ridge of site i counts when its length l > TAU R_i, R_i the largest distance
from i to a vertex of its region.  A cell is known exactly once 2 R_i < margin (every site that can cut it is in
the strip: the security radius) and complete when also 2 R_i < box / 2.  Coincident sites are merged before
Qhull: every particle of a coincident group gets the cell of the group, and neighbours see only the group's
smallest index, as the kernel does.

    tessellate(R, box, ms=(4, 6))                     every particle (the margin grows to box / 2 if needed)
    tessellate(R, box, ms, window=(lo, hi), margin=M)  only the particles in [lo, hi]^2 whose 2 R_i < M

Returns a dict: nvor (N,) int64 (-1 incomplete or non-finite, -2 not determined: outside the window or 2 R_i
>= margin), area (N,), adj (N, ADJ) int64 in angle order padded with -1, psi {m: (N, 2)}, and tau_ratio: the
smallest max(l / (TAU R), TAU R / l) over the ridges of the determined particles, so tau_ratio >= 2 means no
ridge length lies within a factor 2 of the threshold.
"""
import numpy as np
from scipy.spatial import Voronoi

TAU = 2.0 ** -30
ADJ = 64


def min_image(xj, xi, box):
    """The kernel's exact minimum-image difference of fp32 coordinates, in double."""
    d = np.asarray(xj, np.float64) - np.asarray(xi, np.float64)
    half = 0.5 * box
    return np.where(d > half, d - box, np.where(d < -half, d + box, d))


def weighted_psi(dx, dy, ell, m):
    """sum_k (l_k / L) (d_k / |d_k|)^m over the columns in order (rows padded with l = 0 contribute 0), with the
    kernel's operations: u = d / |d|, m - 1 sequential complex products, the weights l / L."""
    with np.errstate(invalid="ignore", divide="ignore"):
        r = np.sqrt(dx * dx + dy * dy)
        ux, uy = dx / r, dy / r
        wx, wy = ux.copy(), uy.copy()
        for _ in range(1, m):
            wx, wy = wx * ux - wy * uy, wx * uy + wy * ux
        L = np.zeros(ell.shape[0])
        for k in range(ell.shape[1]):
            L = L + ell[:, k]
        sx, sy = np.zeros(ell.shape[0]), np.zeros(ell.shape[0])
        for k in range(ell.shape[1]):
            c = ell[:, k] / L
            on = ell[:, k] > 0
            sx = np.where(on, sx + c * wx[:, k], sx)
            sy = np.where(on, sy + c * wy[:, k], sy)
    return np.stack([sx, sy], axis=1)


def _cells(X, box, lo, hi, M):
    """Qhull on the sites X (distinct, double) and their periodic images within [lo - M, hi + M]^2.  Returns the
    region radius R of every point, the ridges (p, q, l) in both directions (q as an index into X), and slot:
    the point of each site's own copy (-1 when it is outside the strip)."""
    pts, orig = [], []
    slot = np.full(X.shape[0], -1)
    off = 0
    for sx in (-1, 0, 1):
        for sy in (-1, 0, 1):
            P = X + np.array([sx * box, sy * box])
            keep = np.flatnonzero(((P >= lo - M) & (P <= hi + M)).all(axis=1))
            if sx == 0 and sy == 0:
                slot[keep] = off + np.arange(keep.size)
            pts.append(P[keep])
            orig.append(keep)
            off += keep.size
    pts = np.concatenate(pts)
    orig = np.concatenate(orig)
    vor = Voronoi(pts)
    V = vor.vertices
    rp = vor.ridge_points
    rv = np.asarray(vor.ridge_vertices, dtype=np.int64)
    inf = (rv < 0).any(axis=1)
    ell = np.where(inf, np.inf, np.linalg.norm(V[np.maximum(rv[:, 0], 0)] - V[np.maximum(rv[:, 1], 0)], axis=1))
    R = np.zeros(pts.shape[0])
    for side in (0, 1):
        for v in (0, 1):
            dv = np.where(inf, np.inf, np.linalg.norm(V[np.maximum(rv[:, v], 0)] - pts[rp[:, side]], axis=1))
            np.maximum.at(R, rp[:, side], dv)
    p = np.concatenate([rp[:, 0], rp[:, 1]])
    q = orig[np.concatenate([rp[:, 1], rp[:, 0]])]
    return R, p, q, np.concatenate([ell, ell]), slot


def tessellate(R, box, ms=(), window=None, margin=None):
    R = np.asarray(R, np.float32)
    N = R.shape[0]
    box = float(np.float32(box))
    X64 = R.astype(np.float64)
    active = np.isfinite(X64).all(axis=1)
    act = np.flatnonzero(active)
    # coincident sites: one Qhull site per distinct fp32 position, represented by its smallest index
    uniq, inv = np.unique(R[act], axis=0, return_inverse=True)
    inv = inv.reshape(-1)
    rep_of_u = np.full(uniq.shape[0], np.iinfo(np.int64).max)
    np.minimum.at(rep_of_u, inv, act)
    X = uniq.astype(np.float64)
    a = box / np.sqrt(max(act.size, 1))
    if window is None:
        lo, hi = 0.0, box
        in_t = np.ones(uniq.shape[0], bool)
        M = min(0.5 * box, 10.0 * a) if margin is None else margin
    else:
        lo, hi = window
        in_t = ((X >= lo) & (X <= hi)).all(axis=1)
        M = margin
    targets = np.flatnonzero(in_t)
    while True:
        Rc, p, q, l, slot = _cells(X, box, lo, hi, M)
        Rt = Rc[slot[targets]]
        known = 2 * Rt < M
        if window is None and M < 0.5 * box and not known.all():
            M = 0.5 * box
            continue
        if window is None and M >= 0.5 * box:
            known[:] = True
        break
    complete = known & (2 * Rt < 0.5 * box)
    # per target u (index into uniq): its ridges
    t_of_slot = np.full(Rc.shape[0], -1)
    t_of_slot[slot[targets]] = targets
    u = t_of_slot[p]
    Ru = np.zeros(uniq.shape[0])
    Ru[targets] = Rt
    ok_u = np.zeros(uniq.shape[0], bool)
    ok_u[targets[complete]] = True
    known_u = np.zeros(uniq.shape[0], bool)
    known_u[targets[known]] = True
    sel = (u >= 0)
    sel[sel] = known_u[u[sel]]
    u, q, l = u[sel], q[sel], l[sel]
    xi = X[u]
    dx = min_image(X[q][:, 0], xi[:, 0], box)
    dy = min_image(X[q][:, 1], xi[:, 1], box)
    # area: the shoelace of the region as the sum of its ridge triangles from the site (l |d| / 4 each)
    area_u = np.zeros(uniq.shape[0])
    np.add.at(area_u, u, l * np.sqrt(dx * dx + dy * dy) / 4.0)
    ratio = l / (TAU * Ru[u])
    tau_ratio = float(np.min(np.maximum(ratio, 1.0 / ratio))) if ratio.size else np.inf
    cnt = ratio > 1.0
    u, q, l, dx, dy = u[cnt], q[cnt], l[cnt], dx[cnt], dy[cnt]
    qn = rep_of_u[q]
    ang = np.arctan2(dy, dx)
    order = np.lexsort((ang, u))
    u, qn, l, dx, dy = u[order], qn[order], l[order], dx[order], dy[order]
    nU = uniq.shape[0]
    n_u = np.bincount(u, minlength=nU)
    start = np.concatenate([[0], np.cumsum(n_u)[:-1]])
    col = np.arange(u.size) - start[u]
    K = max(int(n_u.max()) if n_u.size else 0, 1)
    Q = np.full((nU, max(K, ADJ)), -1, np.int64)
    Q[u, col] = qn
    Lm = np.zeros((nU, K))
    DX = np.ones((nU, K))
    DY = np.zeros((nU, K))
    Lm[u, col], DX[u, col], DY[u, col] = l, dx, dy

    out_n = np.full(N, -2, np.int64)
    out_n[~active] = -1
    out_a = np.full(N, np.nan)
    out_adj = np.full((N, ADJ), -1, np.int64)
    psis = {m: np.full((N, 2), np.nan) for m in ms}
    pu = {m: weighted_psi(DX, DY, Lm, m) for m in ms}
    for_u = inv                                   # active particle k -> its unique site
    kn = known_u[for_u]
    ok = ok_u[for_u]
    idx = act[kn]
    out_n[idx] = np.where(ok[kn], n_u[for_u[kn]], -1)
    okidx = act[ok]
    out_a[okidx] = area_u[for_u[ok]]
    out_adj[okidx] = Q[for_u[ok], :ADJ]
    for m in ms:
        psis[m][okidx] = pu[m][for_u[ok]]
    return {"nvor": out_n, "area": out_a, "adj": out_adj, "psi": psis, "tau_ratio": tau_ratio}
