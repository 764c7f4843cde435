"""Float64 reference of the raster geometry, independent of the raster contract.  TEST INFRASTRUCTURE ONLY.

`oracle/wr_oracle.c`, `oracle/raster_numpy.py` and `csrc/raster.cu` restate DESIGN.md section 3 line by line, so a
mistake in section 3 itself would be made by all three alike.  This module answers the other question -- "is the
contract right?" -- from the geometry alone.  It imports and copies no arithmetic from those files: no fixed point, no
snapping, no guard-band clipper, no fill rule.  In float64 it

* clips a face with a vertex at w <= 0 against z = -w and z = w (its own clipper; after both, w >= |z| >= 0, so the
  projection is defined, and the far clip removes only points that the depth test rejects anyway),
* projects the polygon to pixel space, where pixel (c, r) has its centre at (c, r), i.e. NDC ((2c+1)/W - 1, (2r+1)/H - 1),
* measures the signed distance in pixels from each sample to each polygon edge, and z/w on the polygon's plane,
* takes perspective-correct barycentrics of the parent triangle from the inverse of its homogeneous 3 x 3 vertex
  matrix [x; y; w] (b ~ T^-1 (x_ndc, y_ndc, 1), normalised to sum 1).

What an implementation of the contract may do differently is bounded, not restated:

Snap margin.  A snapped vertex lies within e_i of the float64 one: at most 1/32 px per axis from round-to-nearest in
1/16-px units, plus the float32 error of the projection `(x * 8W) * (1/w)` (C_PROJ ulps of |x/w|), of a clip transform
computed in float32 (C_CLIP ulps of the sum of |m_ij v_j|, render() only) and, for vertices made by clipping, of the
float32 interpolation `(b - a) t + a` with `t = d_i / (d_i - d_j)` (C_LERP ulps of |a| + |b|, t's own error
carried along the edge).  Moving the endpoints A, B of an edge of length L by at most e_A, e_B moves the sign of the
edge function at a sample p with signed distance d only if
    |d| (1 - (e_A + e_B) / L) <= |1 - s| e_A + |s| e_B + e_A e_B / L,
s being p's position along the edge (exact, not first order; expand cross(B'-A', p-A') with p - A = s (B-A) + d n).
That right-hand side, divided by (1 - (e_A + e_B) / L), is the inside margin delta of the edge at p (infinite when
L <= e_A + e_B).  A sample farther than e_max = max_i e_i outside any edge is outside the snapped polygon (every
snapped vertex stays within e_max of the edge's half-plane).  With no float32 error, delta = sqrt(2)/32 px = 0.044 px
at mid-edge.

Depth margin eps_d.  The contract's depth is the plane through the snapped vertices with the vertices' own z/w; at a
covered sample it differs from the float64 plane by at most |grad z/w| * e_max (the sample's barycentrics in the
snapped triangle are >= 0 and sum to 1), plus the float32 rounding of the vertex z/w and of the plane evaluation,
C_ZD ulps of sum |z/w_i| (clip vertices: their interpolation error over w).

Classification of (sample, triangle): *inside* if every edge distance exceeds its delta and -1 + eps_d < z/w <
1 - eps_d; *outside* if some edge distance is below -e_max or z/w is outside [-1, 1] by more than eps_d; *ambiguous*
otherwise.  A sample is *decided* if no triangle is inside or ambiguous (it must be background), or if the triangle
with the smallest z/w - eps_d is inside and its z/w + eps_d is below z/w - eps_d of every other inside or ambiguous
triangle (it must win).  Depth ties (the lowest-id rule) and samples on an edge (the top-left rule) are undecided by
construction: the bit-exact parity tests cover them.

Values at decided samples.  Each float result r of an implementation that evaluates the section 3.4-3.6 / section 4
expressions in float32 is held to |r - r64| <= c * 2^-24 * (sum of |terms|), the terms' absolute values computed in
float64 from the same expression; c is one constant per quantity (the C_* below), calibrated once against the C
oracle and never set per case.  Clamps are 1-Lipschitz and applied to the float64 value as section 3.4 says.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import numpy as np

EPS = 2.0 ** -24
SNAP = 1.0 / 32.0          # half of the 1/16-px snap step, per axis

# ulp multipliers of the error model (see the module docstring and DESIGN.md section 6)
C_PROJ = 4.0               # (x * 8W) * (1/w): three roundings of |x/w|
C_CLIP = 4.0               # ((m0 x + m1 y) + m2 z) + m3 in float32
C_LERP = 4.0               # clip-vertex interpolation and its t
C_ZD = 8.0                 # vertex z/w and the snapped depth plane
C_BARY = 8.0               # u, v of section 3.4
C_ZW = 8.0                 # z/w of section 3.4
C_INTERP = 4.0             # section 3.5 on top of the error of u, v
C_TEX = 8.0                # section 3.6 bilinear weights and sum
C_DEPTH = 4.0              # view depth -(((r0 px + r1 py) + r2 pz) + r3)
C_NORMAL = 8.0             # n / max(sqrt((x^2 + y^2) + z^2), 1e-12)
NEAREST_MARGIN = 1e-6      # nearest filter: a sample this close to a texel boundary (texel units) is undecided

_BIG = np.inf


def pixel_sample(H: int, W: int, max_pixels: int = 1 << 18, row_step: Optional[int] = None, seed: int = 0):
    """(rows, cols) of the samples to check: the whole image when it has at most max_pixels pixels, else every
    row_step-th row plus a seeded random set of about as many pixels."""
    if H * W <= max_pixels:
        r, c = np.divmod(np.arange(H * W, dtype=np.int64), W)
        return r, c
    if row_step is None:
        row_step = max(1, (2 * H * W) // max_pixels)
    rows = np.arange(row_step // 2, H, row_step, dtype=np.int64)
    lin = (rows[:, None] * W + np.arange(W, dtype=np.int64)[None]).reshape(-1)
    rng = np.random.default_rng(seed)
    extra = rng.integers(0, H * W, max(0, max_pixels - lin.size), dtype=np.int64)
    lin = np.unique(np.concatenate([lin, extra]))
    return np.divmod(lin, W)


# ---------------------------------------------------------------------------------------------------------------
# clip positions in float64 with the bound of a float32 transform
# ---------------------------------------------------------------------------------------------------------------

def clip_positions(v_pos, mvp):
    """v_pos [V,3], mvp [B,4,4] -> (clip [B,V,4] float64 of the float32 inputs, abs [B,V,4] = sum_j |m_ij v_j| + |m_i3|)."""
    v = np.asarray(v_pos, np.float64)
    m = np.asarray(mvp, np.float64).reshape(-1, 4, 4)
    vh = np.concatenate([v, np.ones((v.shape[0], 1))], 1)
    clip = np.einsum("bij,vj->bvi", m, vh)
    mag = np.einsum("bij,vj->bvi", np.abs(m), np.abs(vh))
    return clip, mag


# ---------------------------------------------------------------------------------------------------------------
# one view: primitives (clipped polygons) with their margins
# ---------------------------------------------------------------------------------------------------------------

@dataclass
class _Prims:
    parent: np.ndarray      # [P] face id
    n: np.ndarray           # [P] vertex count (3..NV)
    X: np.ndarray           # [P,NV] pixel x (padded by repeating vertex 0)
    Y: np.ndarray
    E: np.ndarray           # [P,NV] vertex error (px)
    ZW: np.ndarray          # [P,NV] z/w
    EZ: np.ndarray          # [P,NV] z/w error
    gx: np.ndarray          # [P] d(z/w)/dx (px)
    gy: np.ndarray
    degenerate: np.ndarray  # [P] bool: area too small for a plane / an edge frame
    unstable: np.ndarray    # [P] bool: a clip vertex whose float32 position is undetermined (see _build_prims)
    edges: tuple            # (AX, AY, DX, DY, L, EA, EB) [P,NV] of edge k = vertex k -> k+1


# Planes of the clipper, as clip-space normals: near z + w >= 0, far w - z >= 0, then |x|, |y| <= GUARD_K w.  The
# last four only cut geometry far outside the viewport (any K >= 1 keeps every pixel's coverage); they keep the
# vertices of a face that passes by the eye at a finite, well-conditioned screen position.
GUARD_K = 64.0
_PLANES = np.array([[0, 0, 1, 1], [0, 0, -1, 1], [1, 0, 0, GUARD_K], [-1, 0, 0, GUARD_K],
                    [0, 1, 0, GUARD_K], [0, -1, 0, GUARD_K]], np.float64)
NV = 9                      # a triangle cut by six planes has at most nine vertices


def _clip_face(P, M):
    """Sutherland-Hodgman of one triangle (rows of P [3,4], transform magnitudes M [3,4]) against _PLANES.
    Returns (poly [m,4], magnitudes [m,4], err [m,4] of the float32 interpolation each vertex carries)."""
    poly = [(P[i], M[i], np.zeros(4)) for i in range(P.shape[0])]
    for nrm in _PLANES:
        out = []
        n = len(poly)
        for i in range(n):
            a, ma, ea = poly[i]
            b, mb, eb = poly[(i + 1) % n]
            da, db = nrm @ a, nrm @ b
            if da >= 0:
                out.append(poly[i])
            if (da >= 0) != (db >= 0):
                t = da / (da - db)
                q = a + t * (b - a)
                # interpolation error of each component, plus t's error carried along the edge
                dt = (np.abs(nrm) @ (np.abs(a) + ma + ea + np.abs(b) + mb + eb)) / abs(da - db)
                e = C_LERP * EPS * (np.abs(a) + np.abs(b) + ma + mb + dt * np.abs(b - a)) + (1 - t) * ea + t * eb
                out.append((q, (1 - t) * ma + t * mb, e))
        poly = out
        if len(poly) < 3:
            return None
    return (np.array([p[0] for p in poly]), np.array([p[1] for p in poly]), np.array([p[2] for p in poly]))


def _project(P, M, Eabs, H, W):
    """Pixel coordinates, vertex errors (px), z/w and z/w errors of clip vertices P [...,4] (w > 0)."""
    w = P[..., 3]
    nx, ny, zw = P[..., 0] / w, P[..., 1] / w, P[..., 2] / w
    # error of the NDC coordinate: projection rounding + transform / interpolation error of x and w
    ex = C_PROJ * EPS * np.abs(nx) + (C_CLIP * EPS * M[..., 0] + Eabs[..., 0]
                                      + np.abs(nx) * (C_CLIP * EPS * M[..., 3] + Eabs[..., 3])) / w
    ey = C_PROJ * EPS * np.abs(ny) + (C_CLIP * EPS * M[..., 1] + Eabs[..., 1]
                                      + np.abs(ny) * (C_CLIP * EPS * M[..., 3] + Eabs[..., 3])) / w
    ez = C_ZD * EPS * np.abs(zw) + (C_CLIP * EPS * M[..., 2] + Eabs[..., 2]
                                    + np.abs(zw) * (C_CLIP * EPS * M[..., 3] + Eabs[..., 3])) / w
    X = (nx + 1.0) * (0.5 * W) - 0.5
    Y = (ny + 1.0) * (0.5 * H) - 0.5
    E = np.hypot(ex * (0.5 * W) + SNAP, ey * (0.5 * H) + SNAP)
    return X, Y, E, zw, ez


def _build_prims(P, M, tri, H, W):
    """P [V,4] float64 clip positions, M [V,4] their float32-transform magnitudes (zeros: exact inputs)."""
    V = P.shape[0]
    tri = np.asarray(tri, np.int64).reshape(-1, 3)
    F = tri.shape[0]
    ok = np.all((tri >= 0) & (tri < V), 1)
    t = np.where(ok[:, None], tri, 0)
    Pf = P[t]                                    # [F,3,4]
    Mf = M[t]
    ok &= np.all(np.isfinite(Pf), (1, 2))
    needs_clip = ok & np.any(Pf[..., 3] <= 0, 1)
    direct = ok & ~needs_clip
    ids = np.nonzero(direct)[0]
    X, Y, E, ZW, EZ = _project(Pf[ids], Mf[ids], np.zeros_like(Pf[ids]), H, W)
    parts = [(ids, np.full(ids.size, 3), X, Y, E, ZW, EZ)]
    clipped = []
    for f in np.nonzero(needs_clip)[0]:
        r = _clip_face(Pf[f], Mf[f])
        if r is None:
            continue
        poly, mag, err = r
        if np.any(poly[:, 3] <= 0):
            continue
        clipped.append((f, *_project(poly, mag, err, H, W)))
    if clipped:
        pad = lambda a: np.concatenate([a, np.repeat(a[:1], NV - a.size)])
        parts.append((np.array([c[0] for c in clipped]), np.array([len(c[1]) for c in clipped]),
                      *[np.stack([pad(c[k]) for c in clipped]) for k in range(1, 6)]))
    pad5 = lambda a: np.concatenate([a, np.repeat(a[:, :1], NV - a.shape[1], 1)], 1) if a.shape[1] < NV else a
    parent = np.concatenate([p[0] for p in parts]).astype(np.int64)
    n = np.concatenate([p[1] for p in parts]).astype(np.int64)
    X, Y, E, ZW, EZ = (np.concatenate([pad5(p[k]) for p in parts]) for k in range(2, 7))
    # z/w plane in pixel space from vertices 0, 1, 2 (the polygon is planar; z/w is affine on its projection)
    ax, ay, az = X[:, 1] - X[:, 0], Y[:, 1] - Y[:, 0], ZW[:, 1] - ZW[:, 0]
    bx, by, bz = X[:, 2] - X[:, 0], Y[:, 2] - Y[:, 0], ZW[:, 2] - ZW[:, 0]
    det = ax * by - ay * bx
    area = np.zeros(parent.size)
    for k in range(NV):
        k1 = np.where(k + 1 < n, k + 1, 0)
        live = k < n
        area += np.where(live, X[:, k] * np.take_along_axis(Y, k1[:, None], 1)[:, 0]
                         - np.take_along_axis(X, k1[:, None], 1)[:, 0] * Y[:, k], 0.0)
    extent = np.maximum(np.ptp(X[:, :3], 1), np.ptp(Y[:, :3], 1))
    degenerate = ~(np.abs(det) > 1e-9 * np.maximum(extent, 1.0) ** 2) | ~np.isfinite(det)
    with np.errstate(divide="ignore", invalid="ignore"):
        gx = np.where(degenerate, 0.0, (az * by - ay * bz) / det)
        gy = np.where(degenerate, 0.0, (ax * bz - az * bx) / det)
    # orientation: make every polygon counter-clockwise in (X, Y)
    flip = area < 0
    for A in (X, Y, E, ZW, EZ):
        for i in np.nonzero(flip)[0]:
            A[i, :n[i]] = A[i, :n[i]][::-1].copy()
            A[i, n[i]:] = A[i, 0]
    # A clip vertex near the apex w = z = 0 of the clip volume (a face passing by the eye between its near and far
    # planes) has a float32 position that is not even determined in sign: its error exceeds the viewport.  Such a
    # face is ambiguous over its float64 footprint grown by UNSTABLE_GROW in barycentric units, outside elsewhere.
    unstable = np.max(E, 1) > 0.5 * (W + H)
    k1 = (np.arange(NV)[None] + 1) % n[:, None]
    k1 = np.where(np.arange(NV)[None] < n[:, None], k1, 0)
    BX, BY, EB = (np.take_along_axis(A, k1, 1) for A in (X, Y, E))
    DX, DY = BX - X, BY - Y
    L = np.hypot(DX, DY)
    L = np.where(np.arange(NV)[None] < n[:, None], L, np.nan)
    return _Prims(parent, n, X, Y, E, ZW, EZ, gx, gy, degenerate, unstable, (X, Y, DX, DY, L, E, EB))


def _pairs(pr: _Prims, rows, cols, H, W, cross_threshold=None):
    """Candidate (prim, sample) pairs by screen bounding box: small prims enumerate their box, large ones are
    crossed with the sample list."""
    S = rows.size
    smap = np.full(H * W, -1, np.int64)
    smap[rows * W + cols] = np.arange(S)
    m = np.max(pr.E, 1) + 1.0
    live = np.arange(NV)[None] < pr.n[:, None]
    Xl = np.where(live, pr.X, np.nan)
    Yl = np.where(live, pr.Y, np.nan)
    with np.errstate(invalid="ignore"):
        c0 = np.clip(np.ceil(np.nanmin(Xl, 1) - m), 0, W)
        c1 = np.clip(np.floor(np.nanmax(Xl, 1) + m), -1, W - 1)
        r0 = np.clip(np.ceil(np.nanmin(Yl, 1) - m), 0, H)
        r1 = np.clip(np.floor(np.nanmax(Yl, 1) + m), -1, H - 1)
    c0, c1, r0, r1 = (a.astype(np.int64) for a in (c0, c1, r0, r1))
    nw, nh = np.maximum(c1 - c0 + 1, 0), np.maximum(r1 - r0 + 1, 0)
    area = nw * nh
    if cross_threshold is None:
        cross_threshold = max(64, S // 2)
    small = (area > 0) & (area <= cross_threshold)
    big = np.nonzero(area > cross_threshold)[0]
    si = np.nonzero(small)[0]
    cnt = area[si]
    pi = np.repeat(si, cnt)
    off = np.arange(pi.size) - np.repeat(np.cumsum(cnt) - cnt, cnt)
    pr_r = r0[pi] + off // nw[pi]
    pr_c = c0[pi] + off % nw[pi]
    sj = smap[pr_r * W + pr_c]
    keep = sj >= 0
    out_p, out_s = [pi[keep]], [sj[keep]]
    for b in big:
        sel = np.nonzero((rows >= r0[b]) & (rows <= r1[b]) & (cols >= c0[b]) & (cols <= c1[b]))[0]
        out_p.append(np.full(sel.size, b, np.int64))
        out_s.append(sel)
    return np.concatenate(out_p), np.concatenate(out_s)


UNSTABLE_GROW = 0.05
CHUNK = 1 << 19


def _classify(pr: _Prims, p, rows, cols, P, tri, H, W):
    """Per pair: (status 0 outside / 1 ambiguous / 2 inside, z/w, eps_d)."""
    cx, cy = cols.astype(np.float64), rows.astype(np.float64)
    n = pr.n[p]
    emax = np.max(pr.E[p], 1)
    inside = np.ones(p.size, bool)
    outside = np.zeros(p.size, bool)
    AX, AY, DX, DY, LL, EA, EB = pr.edges
    for k in range(NV):
        live = n > k
        if not np.any(live):
            break
        q = p[live]
        ax, ay, dx, dy, L, ea, eb = AX[q, k], AY[q, k], DX[q, k], DY[q, k], LL[q, k], EA[q, k], EB[q, k]
        rx, ry = cx[live] - ax, cy[live] - ay
        with np.errstate(divide="ignore", invalid="ignore"):
            # inward normal of a counter-clockwise polygon is (-dy, dx) / L
            d = (dx * ry - dy * rx) / L
            s = (dx * rx + dy * ry) / (L * L)
            qq = 1.0 - (ea + eb) / L
            delta = np.where(qq > 0, (np.abs(1 - s) * ea + np.abs(s) * eb + ea * eb / L) / qq, _BIG)
        inside[live] &= d > delta
        outside[live] |= d < -emax[live]
    X, Y = pr.X[p], pr.Y[p]
    zw = pr.ZW[p, 0] + pr.gx[p] * (cx - X[:, 0]) + pr.gy[p] * (cy - Y[:, 0])
    epsd = np.hypot(pr.gx[p], pr.gy[p]) * emax + np.max(pr.EZ[p], 1) + C_ZD * EPS * np.sum(np.abs(pr.ZW[p][:, :3]), 1)
    deg = pr.degenerate[p]
    d_in = (zw > -1 + epsd) & (zw < 1 - epsd)
    d_out = (zw < -1 - epsd) | (zw > 1 + epsd)
    inside &= d_in & ~deg & ~pr.unstable[p]
    outside |= d_out & ~deg
    if np.any(deg):   # no plane, no edge frame: outside only when clear of the box grown by e_max
        live = np.arange(NV)[None] < n[:, None]
        Xl, Yl = np.where(live, X, np.nan), np.where(live, Y, np.nan)
        far = ((cx < np.nanmin(Xl, 1) - emax) | (cx > np.nanmax(Xl, 1) + emax)
               | (cy < np.nanmin(Yl, 1) - emax) | (cy > np.nanmax(Yl, 1) + emax))
        outside = np.where(deg, far, outside)
        zw = np.where(deg, -_BIG, zw)
        epsd = np.where(deg, 0.0, epsd)
    un = pr.unstable[p]
    if np.any(un):    # footprint of the parent triangle from its homogeneous barycentrics (exact inputs)
        i = np.nonzero(un)[0]
        t = np.asarray(tri, np.int64).reshape(-1, 3)[pr.parent[p[i]]]
        Pv = P[t]
        fx, fy = (2 * cx[i] + 1) / W - 1.0, (2 * cy[i] + 1) / H - 1.0
        T = np.stack([Pv[..., 0], Pv[..., 1], Pv[..., 3]], 1)
        k = np.linalg.solve(T, np.stack([fx, fy, np.ones_like(fx)], -1)[..., None])[..., 0]
        b = k / np.sum(k, 1, keepdims=True)
        lam = np.sum(b * Pv[..., 3], 1)
        zwh = np.sum(b * Pv[..., 2], 1) / lam
        near = np.all(b > -UNSTABLE_GROW, 1) & (lam > 0) & (np.abs(zwh) < 1 + UNSTABLE_GROW)
        outside[i] = ~near
        zw[i], epsd[i] = -_BIG, 0.0
    status = np.where(outside, 0, np.where(inside, 2, 1))
    return status, zw, epsd


@dataclass
class ViewRaster:
    """Decided samples of one view.  rows, cols: the sample; decided: bool; winner: face id, -1 = background,
    meaningful where decided."""
    rows: np.ndarray
    cols: np.ndarray
    decided: np.ndarray
    winner: np.ndarray


def raster_view(P, tri, H, W, rows, cols, M=None) -> ViewRaster:
    """Coverage and visibility of one view.  P [V,4] float64 clip positions; M [V,4] magnitudes of a float32 clip
    transform that produced the implementation's clip positions (None: the implementation received P as float32)."""
    P = np.asarray(P, np.float64)
    M = np.zeros_like(P) if M is None else np.asarray(M, np.float64)
    pr = _build_prims(P, M, tri, H, W)
    S = rows.size
    p_all, s_all = _pairs(pr, rows, cols, H, W)
    # per sample: the smallest z/w - eps_d over the inside / ambiguous triangles, that triangle, and the runner-up
    lo1 = np.full(S, _BIG)
    lo2 = np.full(S, _BIG)
    hi1 = np.full(S, _BIG)
    arg1 = np.full(S, -1, np.int64)
    in1 = np.zeros(S, bool)
    for c0 in range(0, p_all.size, CHUNK):
        p, s = p_all[c0:c0 + CHUNK], s_all[c0:c0 + CHUNK]
        status, zw, epsd = _classify(pr, p, rows[s], cols[s], P, tri, H, W)
        cand = status > 0
        p, s, status, lo, hi = p[cand], s[cand], status[cand], (zw - epsd)[cand], (zw + epsd)[cand]
        # merge this chunk's candidates into the running first / second minimum of every sample
        m = np.full(S, _BIG)
        np.minimum.at(m, s, lo)
        is_min = lo == m[s]
        first = np.zeros(s.size, bool)
        sel = np.nonzero(is_min)[0]
        _, u = np.unique(s[sel], return_index=True)
        first[sel[u]] = True                      # one minimum per sample; a tie leaves the other as runner-up
        m2 = np.full(S, _BIG)
        np.minimum.at(m2, s[~first], lo[~first])
        f = np.nonzero(first)[0]
        sf = s[f]
        better = lo[f] < lo1[sf]
        lo2[sf] = np.where(better, np.minimum(lo1[sf], m2[sf]), np.minimum(lo2[sf], lo[f]))
        keep = sf[better]
        lo1[keep], hi1[keep], arg1[keep], in1[keep] = lo[f][better], hi[f][better], p[f][better], status[f][better] == 2
        rest = np.setdiff1d(np.arange(S), sf, assume_unique=True)
        lo2[rest] = np.minimum(lo2[rest], m2[rest])
    empty = arg1 < 0
    win_ok = ~empty & in1 & (hi1 < lo2)
    decided = empty | win_ok
    winner = np.where(win_ok, pr.parent[np.maximum(arg1, 0)], -1) if pr.parent.size else np.full(S, -1, np.int64)
    return ViewRaster(rows, cols, decided, winner)


# ---------------------------------------------------------------------------------------------------------------
# values at decided samples, with their bounds
# ---------------------------------------------------------------------------------------------------------------

def barycentrics(P, M, tri, face, rows, cols, H, W):
    """Perspective-correct barycentrics of `face` at pixel centres and the error bounds of section 3.4.
    Returns dict(b [n,3], zw, bu, bv, bzw)."""
    t = np.asarray(tri, np.int64).reshape(-1, 3)[face]
    Pv = np.asarray(P, np.float64)[t]                  # [n,3,4]
    Mv = np.asarray(M, np.float64)[t]
    fx = (2 * cols + 1) / W - 1.0
    fy = (2 * rows + 1) / H - 1.0
    T = np.stack([Pv[..., 0], Pv[..., 1], Pv[..., 3]], 1)   # [n, (x,y,w), vertex]
    k = np.linalg.solve(T, np.stack([fx, fy, np.ones_like(fx)], -1)[..., None])[..., 0]
    b = k / np.sum(k, 1, keepdims=True)
    zw = np.sum(b * Pv[..., 2], 1) / np.sum(b * Pv[..., 3], 1)
    # absolute terms of section 3.4: p_i = x_i - f w_i, a0 = p1x p2y - p1y p2x, ...
    Ax = np.abs(Pv[..., 0]) + np.abs(fx[:, None] * Pv[..., 3]) + C_CLIP * (Mv[..., 0] + np.abs(fx[:, None]) * Mv[..., 3])
    Ay = np.abs(Pv[..., 1]) + np.abs(fy[:, None] * Pv[..., 3]) + C_CLIP * (Mv[..., 1] + np.abs(fy[:, None]) * Mv[..., 3])
    px = Pv[..., 0] - fx[:, None] * Pv[..., 3]
    py = Pv[..., 1] - fy[:, None] * Pv[..., 3]
    qx, qy = np.abs(px), np.abs(py)
    # a_i = p_jx p_ky - p_jy p_kx of rounded differences: each factor errs by ~eps * A, the products by eps * |p p|
    Tn = np.stack([Ax[:, j] * qy[:, k] + qx[:, j] * Ay[:, k] + Ay[:, j] * qx[:, k] + qy[:, j] * Ax[:, k]
                   + qx[:, j] * qy[:, k] + qy[:, j] * qx[:, k] for j, k in ((1, 2), (2, 0), (0, 1))], 1)
    a = np.stack([px[:, 1] * py[:, 2] - py[:, 1] * px[:, 2], px[:, 2] * py[:, 0] - py[:, 2] * px[:, 0],
                  px[:, 0] * py[:, 1] - py[:, 0] * px[:, 1]], 1)
    ssum = np.abs(np.sum(a, 1))
    S = np.sum(Tn, 1)
    bu = C_BARY * EPS * (Tn[:, 0] + np.abs(b[:, 0]) * S) / ssum
    bv = C_BARY * EPS * (Tn[:, 1] + np.abs(b[:, 1]) * S) / ssum
    Za = np.abs(Pv[..., 2]) + C_CLIP * Mv[..., 2]
    Wa = np.abs(Pv[..., 3]) + C_CLIP * Mv[..., 3]
    den = np.abs(np.sum(Pv[..., 3] * a, 1))
    bzw = C_ZW * EPS * (np.sum(Za * (np.abs(a) + Tn), 1) + np.abs(zw) * np.sum(Wa * (np.abs(a) + Tn), 1)) / den
    return dict(b=b, zw=zw, bu=bu, bv=bv, bzw=bzw)


def interpolate(attr, tri, face, bc):
    """Section 3.5 in float64 from the float64 barycentrics, and its bound given the bounds of u and v.
    attr [V,A]; returns (value [n,A], bound [n,A])."""
    t = np.asarray(tri, np.int64).reshape(-1, 3)[face]
    a = np.asarray(attr, np.float64)[t]            # [n,3,A]
    b = bc["b"]
    val = np.einsum("ni,nia->na", b, a)
    bu, bv = bc["bu"][:, None], bc["bv"][:, None]
    aa = np.abs(a)
    bound = (aa[:, 0] * bu + aa[:, 1] * bv + aa[:, 2] * (bu + bv)
             + C_INTERP * EPS * (np.einsum("ni,nia->na", np.abs(b), aa) + aa[:, 2] * (1 + np.abs(b[:, :1]) + np.abs(b[:, 1:2]))))
    return val, bound


def texture(tex, uv, filter_mode: str, boundary_mode: str, uv_bound=None):
    """Section 3.6 in float64.  tex [TH,TW,C], uv [n,2] (the implementation's own input, float32 values).
    Returns (value [n,C], bound [n,C], decided [n])."""
    tex = np.asarray(tex, np.float64)
    TH, TW, C = tex.shape
    u = np.asarray(uv, np.float64)[:, 0]
    v = np.asarray(uv, np.float64)[:, 1]
    n = u.size
    decided = np.isfinite(u) & np.isfinite(v)
    uu, vv = np.where(decided, u, 0.0), np.where(decided, v, 0.0)
    # float32 error of the texel coordinate: the wrap subtraction, the scale and the bilinear half-texel shift
    ex = C_TEX * EPS * (np.abs(uu) + 1.0) * TW + (0 if uv_bound is None else uv_bound[:, 0] * TW)
    ey = C_TEX * EPS * (np.abs(vv) + 1.0) * TH + (0 if uv_bound is None else uv_bound[:, 1] * TH)
    if boundary_mode == "wrap":
        uu, vv = uu - np.floor(uu), vv - np.floor(vv)
    x, y = uu * TW, vv * TH
    if boundary_mode == "clamp":
        x, y = np.clip(x, 0, TW), np.clip(y, 0, TH)

    def fetch(ix, iy):
        if boundary_mode == "wrap":
            ix, iy = np.mod(ix, TW), np.mod(iy, TH)
            inb = np.ones(ix.shape, bool)
        elif boundary_mode == "clamp":
            ix, iy = np.clip(ix, 0, TW - 1), np.clip(iy, 0, TH - 1)
            inb = np.ones(ix.shape, bool)
        else:
            inb = (ix >= 0) & (ix < TW) & (iy >= 0) & (iy < TH)
            ix, iy = np.clip(ix, 0, TW - 1), np.clip(iy, 0, TH - 1)
        return np.where(inb[:, None], tex[iy, ix], 0.0)

    if filter_mode == "nearest":
        fxl, fyl = np.floor(x), np.floor(y)
        # a sample on a texel boundary (or, with wrap, on the texture's own edge) can go either way -- except on the
        # outer edges of a clamped texture, where both sides fetch the same texel
        for t, e, size in ((x, ex, TW), (y, ey, TH)):
            k = np.round(t)
            near = np.abs(t - k) <= np.maximum(NEAREST_MARGIN, e)
            if boundary_mode == "clamp":
                near &= (k > 0) & (k < size)
            decided &= ~near
        val = fetch(fxl.astype(np.int64), fyl.astype(np.int64))
        return val, np.zeros((n, C)), decided
    xs, ys = x - 0.5, y - 0.5
    x0, y0 = np.floor(xs), np.floor(ys)
    wx1, wy1 = xs - x0, ys - y0
    ix, iy = x0.astype(np.int64), y0.astype(np.int64)
    taps = [(fetch(ix, iy), (1 - wx1) * (1 - wy1)), (fetch(ix + 1, iy), wx1 * (1 - wy1)),
            (fetch(ix, iy + 1), (1 - wx1) * wy1), (fetch(ix + 1, iy + 1), wx1 * wy1)]
    val = sum(t * w[:, None] for t, w in taps)
    # bilinear filtering is continuous in (x, y) in all three modes: a coordinate error moves the value by at most
    # the largest tap difference per texel; the float32 weights and sum add a rounding term
    lip = 2 * np.max(np.abs(tex)) if tex.size else 0.0
    absum = sum(np.abs(t) * w[:, None] for t, w in taps)
    bound = lip * (ex + ey)[:, None] + C_TEX * EPS * (absum + np.max(np.abs(tex)))
    return val, bound, decided


def view_depth(pos, w2c_row2, pos_bound):
    """-(((r0 px + r1 py) + r2 pz) + r3) in float64 and its bound."""
    r = np.asarray(w2c_row2, np.float64)
    d = -(pos @ r[:3] + r[3])
    bound = pos_bound @ np.abs(r[:3]) + C_DEPTH * EPS * (np.abs(pos) @ np.abs(r[:3]) + abs(r[3]))
    return d, bound


def normalize(n, n_bound):
    """n / |n| in float64 and its bound (2 |dn| / |n| per component, plus rounding)."""
    ln = np.linalg.norm(n, axis=1, keepdims=True)
    val = n / np.maximum(ln, 1e-12)
    bound = 2.0 * np.linalg.norm(n_bound, axis=1, keepdims=True) / np.maximum(ln, 1e-30) + C_NORMAL * EPS
    return val, np.broadcast_to(bound, n.shape)


# ---------------------------------------------------------------------------------------------------------------
# checks an implementation's output against the reference
# ---------------------------------------------------------------------------------------------------------------

class Report:
    """Decided fraction and the largest error / bound per quantity over everything checked."""

    def __init__(self):
        self.samples = 0
        self.decided = 0
        self.covered = 0
        self.ratio = {}

    def add_ratio(self, name, err, bound, extra=0.0):
        err = np.asarray(err, np.float64)
        bound = np.asarray(bound, np.float64) + extra
        bad = ~(err <= bound)
        if np.any(bad):
            i = np.argmax(np.where(bad, err - bound, -np.inf).reshape(-1))
            raise AssertionError(f"{name}: {int(bad.sum())} decided values outside their bound; worst "
                                 f"err {err.reshape(-1)[i]:.3g} > bound {bound.reshape(-1)[i]:.3g}")
        if err.size:
            r = float(np.max(err / np.maximum(bound, 1e-300)))
            self.ratio[name] = max(self.ratio.get(name, 0.0), r)

    @property
    def fraction(self):
        return self.decided / max(self.samples, 1)

    def __str__(self):
        rs = " ".join(f"{k} {v:.3f}" for k, v in sorted(self.ratio.items()))
        return f"decided {self.fraction:.4f} of {self.samples} ({self.covered} covered); max err/bound: {rs}"


def check_rasterize(P, tri, H, W, rast, tri_id=None, rows=None, cols=None, report=None, M=None):
    """Hold one implementation's dr.rasterize output to the reference at the sampled pixels.
    P [B,V,4] clip positions (float32 values as the implementation got them, or float64 exact ones with M);
    rast [B,H,W,4] numpy; tri_id [B,H,W] or None (the id is then rast[...,3] - 1)."""
    P = np.asarray(P, np.float64)
    if P.ndim == 2:
        P = P[None]
    B = rast.shape[0]
    if P.shape[0] == 1 and B > 1:
        P = np.broadcast_to(P, (B,) + P.shape[1:])
    Ms = np.zeros_like(P) if M is None else np.broadcast_to(np.asarray(M, np.float64), P.shape)
    if rows is None:
        rows, cols = pixel_sample(H, W)
    report = report or Report()
    views = []
    for b in range(B):
        vr = raster_view(P[b], tri, H, W, rows, cols, Ms[b])
        got = rast[b, rows, cols]
        gid = (got[:, 3].astype(np.int64) - 1) if tri_id is None else tri_id[b, rows, cols].astype(np.int64)
        d = vr.decided
        bad = d & (gid != vr.winner)
        if np.any(bad):
            i = np.nonzero(bad)[0][:5]
            raise AssertionError(f"view {b}: {int(bad.sum())} decided pixels have the wrong triangle; (row, col, "
                                 f"expected, got): {list(zip(rows[i].tolist(), cols[i].tolist(), vr.winner[i].tolist(), gid[i].tolist()))}")
        if tri_id is not None:   # the id channel of rast must carry the same triangle, + 1
            bad = d & (vr.winner >= 0) & (got[:, 3].astype(np.float64) != vr.winner + 1)
            if np.any(bad):
                raise AssertionError(f"view {b}: {int(bad.sum())} decided pixels with rast[..., 3] != id + 1")
        bg = d & (vr.winner < 0)
        if np.any(got[bg] != 0):
            raise AssertionError(f"view {b}: background pixels with non-zero rast")
        cov = np.nonzero(d & (vr.winner >= 0))[0]
        if cov.size:
            bc = barycentrics(P[b], Ms[b], tri, vr.winner[cov], rows[cov], cols[cov], H, W)
            g = got[cov].astype(np.float64)
            report.add_ratio("u", np.abs(g[:, 0] - np.clip(bc["b"][:, 0], 0, 1)), bc["bu"])
            report.add_ratio("v", np.abs(g[:, 1] - np.clip(bc["b"][:, 1], 0, 1)), bc["bv"])
            report.add_ratio("z/w", np.abs(g[:, 2] - np.clip(bc["zw"], -1, 1)), bc["bzw"])
        report.samples += rows.size
        report.decided += int(d.sum())
        report.covered += int(cov.size)
        views.append(vr)
    return report, views


_ULP_REL = {"float32": 0.0, "float16": 2.0 ** -10, "bfloat16": 2.0 ** -7}


def check_render(v_pos, tri, mvp, w2c, v_nrm, H, W, out, rows=None, cols=None, report=None, dtype="float32",
                 tri_nrm=None, v_tang=None, v_tex=None, tri_tex=None, tex=None, filter_mode="linear",
                 normal_background=0.0, tangent_background=0.0, attr_background=0.5):
    """Hold render()'s mask, pos, normal and raw view depth (no normaliser) to the reference at the sampled pixels.
    The implementation computes the clip positions itself in float32 (section 3.0): the reference takes them in
    float64 and widens every margin and bound by that transform's error.  out: dict of numpy maps (float maps may be
    float16 / bfloat16 values, `dtype` names them: one ulp of that type is allowed on top of the float32 bound).
    Optional maps: "tangent" (v_tang over tri_nrm, normalised like the normals) and "attr" (tex [TH,TW,C] sampled at
    the UV interpolated over tri_tex, wrap mode).  Backgrounds (section 4): pos 0, normal / tangent / attr their background
    values, raw view depth the per-view minimum over all pixels, the background's own depth -w2c[2][3] included."""
    clip, mag = clip_positions(v_pos, mvp)
    w2c = np.asarray(w2c, np.float64).reshape(-1, 4, 4)
    B = clip.shape[0]
    if rows is None:
        rows, cols = pixel_sample(H, W)
    report = report or Report()
    rel = _ULP_REL[dtype]
    tn = tri if tri_nrm is None else tri_nrm
    for b in range(B):
        vr = raster_view(clip[b], tri, H, W, rows, cols, mag[b])
        d = vr.decided
        mask = np.asarray(out["mask"][b, rows, cols]).astype(bool)
        bad = d & (mask != (vr.winner >= 0))
        if np.any(bad):
            i = np.nonzero(bad)[0][:5]
            raise AssertionError(f"view {b}: {int(bad.sum())} decided pixels with the wrong mask at "
                                 f"{list(zip(rows[i].tolist(), cols[i].tolist()))}")
        bg = np.nonzero(d & (vr.winner < 0))[0]
        for k, want in (("pos", 0.0), ("normal", normal_background), ("tangent", tangent_background),
                        ("attr", attr_background)):
            if k in out and np.any(np.asarray(out[k][b, rows[bg], cols[bg]], np.float64) != np.float32(want)):
                raise AssertionError(f"view {b}: background {k} is not {want}")
        if "depth" in out and bg.size:
            full = np.asarray(out["depth"][b], np.float64)
            covered = np.asarray(out["mask"][b]).astype(bool)
            fill = float(-np.float32(w2c[b, 2, 3]))
            if covered.any():
                fill = min(fill, float(full[covered].min()))
            g = full[rows[bg], cols[bg]]
            if np.any(np.abs(g - fill) > rel * abs(fill)):
                raise AssertionError(f"view {b}: background depth is not the per-view minimum {fill}")
        cov = np.nonzero(d & (vr.winner >= 0))[0]
        report.samples += rows.size
        report.decided += int(d.sum())
        report.covered += int(cov.size)
        if not cov.size:
            continue
        face = vr.winner[cov]
        bc = barycentrics(clip[b], mag[b], tri, face, rows[cov], cols[cov], H, W)
        pos, pb = interpolate(v_pos, tri, face, bc)
        if "pos" in out:
            g = np.asarray(out["pos"][b, rows[cov], cols[cov]], np.float64)
            report.add_ratio("pos", np.abs(g - pos), pb + rel * np.abs(pos), 1e-30)
        if "depth" in out:
            dv, db = view_depth(pos, w2c[b, 2], pb)
            g = np.asarray(out["depth"][b, rows[cov], cols[cov]], np.float64)
            report.add_ratio("depth", np.abs(g - dv), db + rel * np.abs(dv), 1e-30)
        if "normal" in out:
            n, nb = interpolate(v_nrm, tn, face, bc)
            nv, nvb = normalize(n, nb)
            g = np.asarray(out["normal"][b, rows[cov], cols[cov]], np.float64)
            report.add_ratio("normal", np.abs(g - nv), nvb + rel * np.abs(nv), 1e-30)
        if "tangent" in out:
            t, tb = interpolate(v_tang, tn, face, bc)
            tv, tvb = normalize(t, tb)
            ok = np.all(np.isfinite(tv), 1)         # a vertex without a tangent frame (NaN) is not compared
            g = np.asarray(out["tangent"][b, rows[cov], cols[cov]], np.float64)[ok]
            report.add_ratio("tangent", np.abs(g - tv[ok]), tvb[ok] + rel * np.abs(tv[ok]), 1e-30)
        if "attr" in out:
            uv, uvb = interpolate(v_tex, tri_tex, face, bc)
            val, vb, ok = texture(tex, uv, filter_mode, "wrap", uv_bound=uvb)
            g = np.asarray(out["attr"][b, rows[cov], cols[cov]], np.float64)[ok]
            report.add_ratio("attr", np.abs(g - val[ok]), vb[ok] + rel * np.abs(val[ok]), 1e-30)
    return report
