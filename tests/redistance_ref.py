"""NumPy restatement of the closest-point redistancing contract (``lsm_redistance``, include/lsm_b200.h).

The three phases — band scan, jump flooding, write — vectorised, with the same operation order as ``csrc/lsm_redistance.cu``, so
that the device result equals this one bit for bit.  The primitives come from ``interface_ref.extract``: a primitive's cell is the
componentwise minimum of the lower nodes (``key // (2^N - 1)``) of its vertices, and ``extract`` lists primitives in cell order,
then simplex order, which is the order the band scan visits them in.
"""
from __future__ import annotations

import itertools

import numpy as np

import interface_ref as IR


# ---- geometry, in the contract's operation order --------------------------------------------------
def dot(u, v):
    r = u[..., 0] * v[..., 0]
    for d in range(1, u.shape[-1]):
        r = r + u[..., d] * v[..., d]
    return r


def dist(x, p):
    """sqrt(((x1 - p1)^2 + (x2 - p2)^2) + (x3 - p3)^2) over the last axis."""
    r = (x[..., 0] - p[..., 0]) * (x[..., 0] - p[..., 0])
    for d in range(1, x.shape[-1]):
        r = r + (x[..., d] - p[..., d]) * (x[..., d] - p[..., d])
    return np.sqrt(r)


def closest_segment(x, a, b):
    """a + t (b - a), t = clamp(dot(x - a, b - a) / dot(b - a, b - a), 0, 1); a where a == b."""
    ab, ax = b - a, x - a
    with np.errstate(all="ignore"):
        t = dot(ax, ab) / dot(ab, ab)
        t = np.where(t < 0.0, 0.0, np.where(t > 1.0, 1.0, t))
        q = a + t[..., None] * ab
    return np.where(np.all(a == b, axis=-1)[..., None], a, q)


def closest_triangle(p, a, b, c):
    """Ericson's ClosestPtPointTriangle (Real-Time Collision Detection 5.1.5) in its operation order; where the divisor of the
    region reached is 0, the closest of the projections on ab, ac, bc (a later one only if strictly closer)."""
    with np.errstate(all="ignore"):
        ab, ac, ap, bp, cp = b - a, c - a, p - a, p - b, p - c
        d1, d2, d3, d4, d5, d6 = dot(ab, ap), dot(ac, ap), dot(ab, bp), dot(ac, bp), dot(ab, cp), dot(ac, cp)
        vc, vb, va = d1 * d4 - d3 * d2, d5 * d2 - d1 * d6, d3 * d6 - d5 * d4
        q = np.full(p.shape, np.nan)
        done = np.zeros(p.shape[:-1], bool)
        degen = np.zeros(p.shape[:-1], bool)

        def put(mask, val):
            m = mask & ~done & ~degen
            q[m] = np.broadcast_to(val, q.shape)[m]
            done[m] = True

        def divide(mask, num, den, val):
            reach = mask & ~done & ~degen
            put(reach & (den != 0.0), val(num / den))
            degen[reach & (den == 0.0)] = True

        put((d1 <= 0.0) & (d2 <= 0.0), a)
        put((d3 >= 0.0) & (d4 <= d3), b)
        divide((vc <= 0.0) & (d1 >= 0.0) & (d3 <= 0.0), d1, d1 - d3, lambda v: a + v[..., None] * ab)
        put((d6 >= 0.0) & (d5 <= d6), c)
        divide((vb <= 0.0) & (d2 >= 0.0) & (d6 <= 0.0), d2, d2 - d6, lambda w: a + w[..., None] * ac)
        divide((va <= 0.0) & ((d4 - d3) >= 0.0) & ((d5 - d6) >= 0.0), d4 - d3, (d4 - d3) + (d5 - d6),
               lambda w: b + w[..., None] * (c - b))
        den = (va + vb) + vc
        denom = 1.0 / den
        v, w = vb * denom, vc * denom
        put(den != 0.0, (a + ab * v[..., None]) + ac * w[..., None])
    rest = ~done
    if np.any(rest):
        pr, ar, br, cr = p[rest], a[rest], b[rest], c[rest]
        best_q = closest_segment(pr, ar, br)
        best = dist(pr, best_q)
        for u, v in ((ar, cr), (br, cr)):
            s = closest_segment(pr, u, v)
            ds = dist(pr, s)
            take = ds < best
            best = np.where(take, ds, best)
            best_q = np.where(take[..., None], s, best_q)
        q[rest] = best_q
    return q


def closest_point(x, V):
    """Closest point of primitive(s) V (..., N vertices, N coordinates) to x (..., N)."""
    N = x.shape[-1]
    if N == 1:
        return V[..., 0, :].copy()
    if N == 2:
        return closest_segment(x, V[..., 0, :], V[..., 1, :])
    return closest_triangle(x, V[..., 0, :], V[..., 1, :], V[..., 2, :])


# ---- the mesh as primitives with their cells -------------------------------------------------------
def primitives(phi, lc, h):
    """(V (np, N, N) vertex coordinates of each primitive, cell (np, N) lower corner of its cell), in the extraction's order."""
    phi = np.asarray(phi)
    N, n = phi.ndim, phi.shape
    X, F, K = IR.extract(phi, lc, h)
    if not len(F):
        return np.empty((0, N, N)), np.empty((0, N), np.int64)
    ncode = (1 << N) - 1
    low = np.stack(np.unravel_index(K[F.astype(np.int64)] // ncode, n, order="F"), axis=-1)   # (np, N vertices, N)
    return X[F.astype(np.int64)], low.min(axis=1).astype(np.int64)


def node_coords(n, lc, h):
    """x (n..., N): x_d = lc_d + i_d h_d."""
    idx = np.indices(n)
    return np.stack([float(lc[d]) + idx[d].astype(np.float64) * float(h[d]) for d in range(len(n))], axis=-1)


# ---- the three phases ------------------------------------------------------------------------------
def band_phase(phi, lc, h, band):
    """Closest points of the band scan: (P (n..., N) float64, NaN where no point; is_band (n...) bool)."""
    phi = np.asarray(phi)
    N, n = phi.ndim, phi.shape
    V, cell = primitives(phi, lc, h)
    nodes = int(np.prod(n))
    best = np.full(nodes, np.inf)
    best_j = np.full(nodes, np.iinfo(np.int64).max)
    P = np.full((nodes, N), np.nan)
    is_band = np.zeros(nodes, bool)
    jall = np.arange(len(V))
    for r in itertools.product(range(-band + 1, band + 1), repeat=N):
        node = cell + np.array(r)
        ok = np.all((node >= 0) & (node < np.array(n)), axis=1)
        j, nd = jall[ok], node[ok]
        if not len(j):
            continue
        lin = np.ravel_multi_index(tuple(nd.T), n, order="F")
        is_band[lin] = True
        x = np.stack([float(lc[d]) + nd[:, d].astype(np.float64) * float(h[d]) for d in range(N)], axis=-1)
        q = closest_point(x, V[j])
        d = dist(x, q)
        fin = d < np.inf                      # NaN never wins
        j, lin, q, d = j[fin], lin[fin], q[fin], d[fin]
        # the first (in primitive order) of the smallest distances per node, then against what the node already holds
        o = np.lexsort((j, d, lin))
        first = o[np.r_[True, lin[o][1:] != lin[o][:-1]]] if len(o) else o
        l_, d_, j_ = lin[first], d[first], j[first]
        better = (d_ < best[l_]) | ((d_ == best[l_]) & (j_ < best_j[l_]))
        l_, d_, j_, q_ = l_[better], d_[better], j_[better], q[first][better]
        best[l_], best_j[l_], P[l_] = d_, j_, q_
    shape = tuple(n) + (N,)
    return P.reshape(shape, order="F"), is_band.reshape(n, order="F")


def flood_steps(n):
    L = 0
    while (1 << L) < max(n):
        L += 1
    return [1 << e for e in range(L - 1, -1, -1)] + [1]


def _shifted(P, s):
    """P[i + s] (NaN outside the box)."""
    n = P.shape[:-1]
    out = np.full(P.shape, np.nan)
    dst, src = [], []
    for d, sd in enumerate(s):
        if abs(sd) >= n[d]:
            return out
        dst.append(slice(max(0, -sd), n[d] - max(0, sd)))
        src.append(slice(max(0, sd), n[d] + min(0, sd)))
    out[tuple(dst)] = P[tuple(src)]
    return out


def propagate(P, lc, h):
    """Jump flooding over closest points (k = 2^(L-1) .. 1, then 1 again)."""
    n = P.shape[:-1]
    N = len(n)
    x = node_coords(n, lc, h)
    offsets = [tuple(reversed(o)) for o in itertools.product((-1, 0, 1), repeat=N)]      # column-major: o_1 fastest
    offsets = [o for o in offsets if any(o)]
    for k in flood_steps(n):
        best = np.full(n, np.inf)
        out = np.full(P.shape, np.nan)
        for o in [(0,) * N] + offsets:
            q = P if not any(o) else _shifted(P, [k * v for v in o])
            with np.errstate(invalid="ignore"):
                d = dist(x, q)
                take = d < best
            best = np.where(take, d, best)
            out[take] = q[take]
        P = out
    return P


def write(phi, P, lc, h):
    phi = np.asarray(phi)
    s = phi.astype(np.float64)
    x = node_coords(phi.shape, lc, h)
    with np.errstate(invalid="ignore"):
        d = dist(x, P)
    neg = (-d).astype(phi.dtype)
    pos = d.astype(phi.dtype)
    pos[pos == 0] = np.finfo(phi.dtype).smallest_subnormal
    out = phi.copy()
    keep = np.isnan(s) | np.isnan(P[..., 0])
    val = np.where(s <= 0, neg, pos)
    out[~keep] = val[~keep]
    return out


def redistance(phi, lc, h, band=3):
    """(the redistanced field in phi's dtype, number of band nodes)."""
    P, is_band = band_phase(phi, lc, h, band)
    return write(phi, propagate(P, lc, h), lc, h), int(is_band.sum())


def brute_force(phi, lc, h, chunk=1 << 18):
    """The distance of every node to the whole mesh: min over all primitives of dist(x, closest point) (inf without a mesh)."""
    phi = np.asarray(phi)
    n, N = phi.shape, phi.ndim
    V, _ = primitives(phi, lc, h)
    x = node_coords(n, lc, h).reshape(-1, N)
    best = np.full(len(x), np.inf)
    if len(V):
        step = max(1, chunk // len(V))
        for b in range(0, len(x), step):
            xb = x[b:b + step]
            q = closest_point(np.broadcast_to(xb[:, None, :], (len(xb), len(V), N)), np.broadcast_to(V, (len(xb),) + V.shape))
            with np.errstate(invalid="ignore"):
                best[b:b + step] = np.fmin.reduce(dist(xb[:, None, :], q), axis=1)
    return best.reshape(n)
