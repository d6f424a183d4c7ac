"""NumPy restatement of the closest-point extension contract (``lsm_extend_closest_point``, include/lsm_b200.h).

The geometry is ``redistance_ref``'s: the same primitives, band scan, closest points and jump flooding.  This file adds the value
of F, with the same operation order as ``csrc/lsm_redistance.cu`` so that the device result equals this one bit for bit: at the
mesh vertices (``Fa + t (Fb - Fa)`` on the vertex's lattice edge), at the closest point of a primitive (following the branch the
closest-point routine takes), carried through the jump flooding with its point, and written where the point is.
"""
from __future__ import annotations

import itertools

import numpy as np

import interface_ref as IR
import redistance_ref as R


# ---- value at the closest point of a primitive ---------------------------------------------------
def closest_segment(x, a, b, fa, fb):
    """(``redistance_ref.closest_segment(x, a, b)``, F there): fa + t (fb - fa) with the clamped t of the projection; fa where
    a == b."""
    ab, ax = b - a, x - a
    with np.errstate(all="ignore"):
        t = R.dot(ax, ab) / R.dot(ab, ab)
        t = np.where(t < 0.0, 0.0, np.where(t > 1.0, 1.0, t))
        q = a + t[..., None] * ab
        f = fa + t * (fb - fa)
    same = np.all(a == b, axis=-1)
    return np.where(same[..., None], a, q), np.where(same, fa, f)


def closest_triangle(p, a, b, c, f0, f1, f2):
    """(``redistance_ref.closest_triangle(p, a, b, c)``, F there): F0 / F1 / F2 in the vertex regions, F0 + v (F1 - F0),
    F0 + w (F2 - F0), F1 + w (F2 - F1) on the edges ab, ac, bc, (F0 + (F1 - F0) v) + (F2 - F0) w inside, with Ericson's own v, w;
    the degenerate fallback takes the value of the segment it picks."""
    with np.errstate(all="ignore"):
        ab, ac, ap, bp, cp = b - a, c - a, p - a, p - b, p - c
        d1, d2, d3, d4, d5, d6 = R.dot(ab, ap), R.dot(ac, ap), R.dot(ab, bp), R.dot(ac, bp), R.dot(ab, cp), R.dot(ac, cp)
        vc, vb, va = d1 * d4 - d3 * d2, d5 * d2 - d1 * d6, d3 * d6 - d5 * d4
        q = np.full(p.shape, np.nan)
        f = np.full(p.shape[:-1], np.nan)
        done = np.zeros(p.shape[:-1], bool)
        degen = np.zeros(p.shape[:-1], bool)

        def put(mask, val, fval):
            m = mask & ~done & ~degen
            q[m] = np.broadcast_to(val, q.shape)[m]
            f[m] = np.broadcast_to(fval, f.shape)[m]
            done[m] = True

        def divide(mask, num, den, val, fval):
            reach = mask & ~done & ~degen
            r = num / den
            put(reach & (den != 0.0), val(r), fval(r))
            degen[reach & (den == 0.0)] = True

        put((d1 <= 0.0) & (d2 <= 0.0), a, f0)
        put((d3 >= 0.0) & (d4 <= d3), b, f1)
        divide((vc <= 0.0) & (d1 >= 0.0) & (d3 <= 0.0), d1, d1 - d3, lambda v: a + v[..., None] * ab,
               lambda v: f0 + v * (f1 - f0))
        put((d6 >= 0.0) & (d5 <= d6), c, f2)
        divide((vb <= 0.0) & (d2 >= 0.0) & (d6 <= 0.0), d2, d2 - d6, lambda w: a + w[..., None] * ac,
               lambda w: f0 + w * (f2 - f0))
        divide((va <= 0.0) & ((d4 - d3) >= 0.0) & ((d5 - d6) >= 0.0), d4 - d3, (d4 - d3) + (d5 - d6),
               lambda w: b + w[..., None] * (c - b), lambda w: f1 + w * (f2 - f1))
        den = (va + vb) + vc
        denom = 1.0 / den
        v, w = vb * denom, vc * denom
        put(den != 0.0, (a + ab * v[..., None]) + ac * w[..., None], (f0 + (f1 - f0) * v) + (f2 - f0) * w)
    rest = ~done
    if np.any(rest):
        pr, ar, br, cr = p[rest], a[rest], b[rest], c[rest]
        g0, g1, g2 = (np.broadcast_to(z, p.shape[:-1])[rest] for z in (f0, f1, f2))
        best_q, best_f = closest_segment(pr, ar, br, g0, g1)
        best = R.dist(pr, best_q)
        for u, v, fu, fv in ((ar, cr, g0, g2), (br, cr, g1, g2)):
            s, fs = closest_segment(pr, u, v, fu, fv)
            ds = R.dist(pr, s)
            take = ds < best
            best = np.where(take, ds, best)
            best_q = np.where(take[..., None], s, best_q)
            best_f = np.where(take, fs, best_f)
        q[rest] = best_q
        f[rest] = best_f
    return q, f


def closest_point(x, V, FV):
    """(closest point, F there) of primitive(s) V (..., N vertices, N coordinates) with vertex values FV (..., N) to x (..., N)."""
    N = x.shape[-1]
    if N == 1:
        return V[..., 0, :].copy(), FV[..., 0].copy()
    if N == 2:
        return closest_segment(x, V[..., 0, :], V[..., 1, :], FV[..., 0], FV[..., 1])
    return closest_triangle(x, V[..., 0, :], V[..., 1, :], V[..., 2, :], FV[..., 0], FV[..., 1], FV[..., 2])


# ---- the mesh with the values of F at its vertices --------------------------------------------------
def primitives(phi, F, lc, h):
    """(V, cell) as ``redistance_ref.primitives``, and FV (np, N): F at each primitive's vertices.  A vertex with key
    a * (2^N - 1) + e - 1 lies on the lattice edge (a, a + bits(e)) at t = s_a / (s_a - s_b); its value is Fa + t (Fb - Fa)."""
    phi = np.asarray(phi)
    N, n = phi.ndim, phi.shape
    X, Fc, K = IR.extract(phi, lc, h)
    if not len(Fc):
        return np.empty((0, N, N)), np.empty((0, N), np.int64), np.empty((0, N))
    ncode = (1 << N) - 1
    a, e = K // ncode, K % ncode + 1
    ia = np.stack(np.unravel_index(a, n, order="F"), axis=-1)
    ib = ia + np.stack([(e >> d) & 1 for d in range(N)], axis=-1)
    b = np.ravel_multi_index(tuple(ib.T), n, order="F")
    s = phi.astype(np.float64).reshape(-1, order="F") - 0.0
    f = np.asarray(F).astype(np.float64).reshape(-1, order="F")
    with np.errstate(all="ignore"):
        t = s[a] / (s[a] - s[b])
        fv = f[a] + t * (f[b] - f[a])
    Fi = Fc.astype(np.int64)
    low = ia[Fi]                                                  # (np, N vertices, N): the lower node of each vertex's edge
    return X[Fi], low.min(axis=1).astype(np.int64), fv[Fi]


# ---- the three phases ------------------------------------------------------------------------------
def band_phase(phi, F, lc, h, band):
    """The band scan of ``redistance_ref.band_phase`` with values: (P (n..., N), value at P (n...), NaN where no point; is_band)."""
    phi = np.asarray(phi)
    N, n = phi.ndim, phi.shape
    V, cell, FV = primitives(phi, F, lc, h)
    nodes = int(np.prod(n))
    best = np.full(nodes, np.inf)
    best_j = np.full(nodes, np.iinfo(np.int64).max)
    P = np.full((nodes, N), np.nan)
    val = np.full(nodes, np.nan)
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
        q, fq = closest_point(x, V[j], FV[j])
        d = R.dist(x, q)
        fin = d < np.inf
        j, lin, q, fq, d = j[fin], lin[fin], q[fin], fq[fin], d[fin]
        o = np.lexsort((j, d, lin))
        first = o[np.r_[True, lin[o][1:] != lin[o][:-1]]] if len(o) else o
        l_, d_, j_ = lin[first], d[first], j[first]
        better = (d_ < best[l_]) | ((d_ == best[l_]) & (j_ < best_j[l_]))
        l_, d_, j_ = l_[better], d_[better], j_[better]
        best[l_], best_j[l_], P[l_], val[l_] = d_, j_, q[first][better], fq[first][better]
    return P.reshape(tuple(n) + (N,), order="F"), val.reshape(n, order="F"), is_band.reshape(n, order="F")


def propagate(P, val, lc, h):
    """``redistance_ref.propagate`` with the value travelling with its point: (P, val) after the jump-flooding passes."""
    n = P.shape[:-1]
    N = len(n)
    x = R.node_coords(n, lc, h)
    Q = np.concatenate([P, val[..., None]], axis=-1)
    offsets = [tuple(reversed(o)) for o in itertools.product((-1, 0, 1), repeat=N)]      # column-major: o_1 fastest
    offsets = [o for o in offsets if any(o)]
    for k in R.flood_steps(n):
        best = np.full(n, np.inf)
        out = np.full(Q.shape, np.nan)
        for o in [(0,) * N] + offsets:
            q = Q if not any(o) else R._shifted(Q, [k * v for v in o])
            with np.errstate(invalid="ignore"):
                d = R.dist(x, q[..., :N])
                take = d < best
            best = np.where(take, d, best)
            out[take] = q[take]
        Q = out
    return Q[..., :N], Q[..., N]


def write(F, phi, P, val):
    """F = val, rounded to F's dtype, on the nodes with a point and a non-NaN phi; every other node keeps its F."""
    F = np.asarray(F)
    keep = np.isnan(np.asarray(phi).astype(np.float64)) | np.isnan(P[..., 0])
    out = F.copy()
    with np.errstate(all="ignore"):
        out[~keep] = val[~keep].astype(F.dtype)
    return out


def extend(F, phi, lc, h, band=3, redistance=False):
    """(F extended in its dtype, phi (its signed distance when ``redistance``, else unchanged), number of band nodes)."""
    P, val, is_band = band_phase(phi, F, lc, h, band)
    P, val = propagate(P, val, lc, h)
    phi_out = R.write(phi, P, lc, h) if redistance else np.array(phi, copy=True)
    return write(F, phi, P, val), phi_out, int(is_band.sum())
