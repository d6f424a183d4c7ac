"""NumPy restatement of the cubic interpolant (``lsm_interpolate_cubic``) and of the cubic closest-point redistancing
(``lsm_redistance_cubic``), include/lsm_b200.h.

Vectorised, with the operation order of ``csrc/lsm_cubic.cuh`` and the refinement pass of ``csrc/lsm_redistance.cu`` (both
compiled with -fmad=false), so that the device results equal these bit for bit.  The seeds are ``redistance_ref``'s linear
closest points after jump flooding, and the write pass is ``redistance_ref.write``.
"""
from __future__ import annotations

import numpy as np

import redistance_ref as R

NEWTON_ITERS = 20


def weights(xi):
    """(M, 3, 4): the Lagrange weights L, L' and L'' on the nodes 0..3 at xi (M,)."""
    a, b, c = xi - 1.0, xi - 2.0, xi - 3.0
    L = [((a * b) * c) / (-6.0), ((xi * b) * c) / 2.0, ((xi * a) * c) / (-2.0), ((xi * a) * b) / 6.0]
    D = [((a * b + a * c) + b * c) / (-6.0), ((xi * b + xi * c) + b * c) / 2.0, ((xi * a + xi * c) + a * c) / (-2.0),
         ((xi * a + xi * b) + a * b) / 6.0]
    S = [((a + b) + c) / (-3.0), (xi + b) + c, -((xi + a) + c), ((xi + a) + b) / 3.0]
    return np.stack([np.stack(L, -1), np.stack(D, -1), np.stack(S, -1)], -2)


def _contract(F, W, orders):
    """Contract the stencil F (M, 4, ..., 4; axis 1 first) with the weights of derivative order orders[d] on axis d."""
    r = F
    for d, o in enumerate(orders):
        w = W[d][:, o, :].reshape((len(F), 4) + (1,) * (r.ndim - 2))
        t = w * r
        r = ((t[:, 0] + t[:, 1]) + t[:, 2]) + t[:, 3]
    return r


def evaluate(phi, lc, h, Y):
    """(P (M,), g (M, N), H (M, N, N)) of the interpolant of phi at the points Y (M, N); NaN outside the box."""
    phi = np.asarray(phi)
    N, n = phi.ndim, phi.shape
    Y = np.asarray(Y, dtype=np.float64).reshape(-1, N)
    M = len(Y)
    P, g, H = np.full(M, np.nan), np.full((M, N), np.nan), np.full((M, N, N), np.nan)
    with np.errstate(invalid="ignore"):
        u = np.stack([(Y[:, d] - float(lc[d])) / float(h[d]) for d in range(N)], -1)
        inside = np.all((u >= 0.0) & (u <= np.array([n[d] - 1 for d in range(N)], np.float64)), axis=1)
    if not inside.any():
        return P, g, H
    u = u[inside]
    Mi = len(u)
    W, starts = [], []
    for d in range(N):
        c = np.minimum(np.floor(u[:, d]).astype(np.int64), n[d] - 2)
        s = np.minimum(np.maximum(c - 1, 0), n[d] - 4)
        W.append(weights(u[:, d] - s.astype(np.float64)))
        starts.append(s)
    k = np.arange(4)
    idx = []
    for d in range(N):
        shp = [Mi] + [1] * N
        shp[1 + d] = 4
        idx.append((starts[d][:, None] + k[None, :]).reshape(shp))
    F = phi.astype(np.float64)[tuple(idx)]                    # (Mi, 4, ..., 4): axis d of the stencil = axis d of phi
    zero = [0] * N
    Pi = _contract(F, W, zero)
    gi = np.empty((Mi, N))
    Hi = np.empty((Mi, N, N))
    for d in range(N):
        o = list(zero)
        o[d] = 1
        gi[:, d] = _contract(F, W, o) / float(h[d])
        o[d] = 2
        Hi[:, d, d] = (_contract(F, W, o) / float(h[d])) / float(h[d])
        for e in range(d + 1, N):
            o = list(zero)
            o[d] = o[e] = 1
            Hi[:, d, e] = Hi[:, e, d] = (_contract(F, W, o) / float(h[d])) / float(h[e])
    P[inside], g[inside], H[inside] = Pi, gi, Hi
    return P, g, H


def _finite(v):
    return np.abs(v) < np.inf


def _solve(M, r):
    """Gaussian elimination with partial pivoting (strictly larger |entry| replaces the pivot), as the device does it, on a batch:
    (z, ok); ok is False where a pivot is 0."""
    M, r = M.copy(), r.copy()
    K = M.shape[1]
    ok = np.ones(len(M), bool)
    rows = np.arange(len(M))
    with np.errstate(all="ignore"):
        for k in range(K):
            p = np.full(len(M), k)
            big = np.abs(M[:, k, k])
            for i in range(k + 1, K):
                take = np.abs(M[:, i, k]) > big
                big = np.where(take, np.abs(M[:, i, k]), big)
                p = np.where(take, i, p)
            ok &= ~(big == 0.0)
            rk, rp = M[rows, k].copy(), M[rows, p].copy()
            M[rows, k], M[rows, p] = rp, rk
            bk, bp = r[rows, k].copy(), r[rows, p].copy()
            r[rows, k], r[rows, p] = bp, bk
            for i in range(k + 1, K):
                f = M[:, i, k] / M[:, k, k]
                for j in range(k + 1, K):
                    M[:, i, j] = M[:, i, j] - f * M[:, k, j]
                r[:, i] = r[:, i] - f * r[:, k]
        z = np.empty_like(r)
        for i in range(K - 1, -1, -1):
            s = r[:, i]
            for j in range(i + 1, K):
                s = s - M[:, i, j] * z[:, j]
            z[:, i] = s / M[:, i, i]
    return z, ok


def refine(phi, lc, h, x, y0):
    """Newton on the KKT conditions of min |y - x| subject to P(y) = 0 from the seeds y0 (M, N), for the nodes x (M, N):
    (y (M, N) the refined point or y0 where it falls back, fell (M,) bool, iterations (M,) int)."""
    phi = np.asarray(phi)
    N = phi.ndim
    x, y0 = np.asarray(x, np.float64).reshape(-1, N), np.asarray(y0, np.float64).reshape(-1, N)
    M = len(x)
    y = y0.copy()
    iters = np.zeros(M, np.int64)
    done = np.zeros(M, bool)
    hmin, hmax = min(abs(float(v)) for v in h[:N]), max(abs(float(v)) for v in h[:N])
    tol, reach = 1e-10 * hmin, 2.0 * hmax
    with np.errstate(all="ignore"):
        _, g, _ = evaluate(phi, lc, h, y0)
        gg = R.dot(g, g)
        lam = R.dot(x - y0, g) / gg
    fell = ~_finite(gg) | (gg == 0.0) | ~_finite(lam)
    nmax = np.array([phi.shape[d] - 1 for d in range(N)], np.float64)
    for _ in range(NEWTON_ITERS):
        ia = np.nonzero(~fell & ~done)[0]
        if not len(ia):
            break
        iters[ia] += 1
        ya, xa, la = y[ia], x[ia], lam[ia]
        P, g, H = evaluate(phi, lc, h, ya)
        fin = _finite(P) & np.all(_finite(g), axis=1) & np.all(_finite(H), axis=(1, 2))
        with np.errstate(all="ignore"):
            K = np.zeros((len(ia), N + 1, N + 1))
            K[:, :N, :N] = la[:, None, None] * H
            for d in range(N):
                K[:, d, d] = 1.0 + la * H[:, d, d]
            K[:, :N, N] = g
            K[:, N, :N] = g
            r = np.empty((len(ia), N + 1))
            r[:, :N] = -((ya - xa) + la[:, None] * g)
            r[:, N] = -P
            z, ok = _solve(K, r)
            ok &= fin & np.all(_finite(z), axis=1)
            yn = ya + z[:, :N]
            ln = la + z[:, N]
            u = np.stack([(yn[:, d] - float(lc[d])) / float(h[d]) for d in range(N)], -1)
            ok &= _finite(ln) & np.all(_finite(yn) & (u >= 0.0) & (u <= nmax), axis=1)
            ok &= ~(R.dist(yn, y0[ia]) > reach)
            conv = ok & (R.dist(z[:, :N], np.zeros((len(ia), N))) <= tol)
        fell[ia[~ok]] = True
        y[ia[ok]], lam[ia[ok]] = yn[ok], ln[ok]
        done[ia[conv]] = True
    fell |= ~done
    y[fell] = y0[fell]
    return y, fell, iters


def redistance_cubic(phi, lc, h, band=3):
    """(the redistanced field in phi's dtype, band nodes, nodes that fell back)."""
    phi = np.asarray(phi)
    P, is_band = R.band_phase(phi, lc, h, band)
    P = R.propagate(P, lc, h)
    x = R.node_coords(phi.shape, lc, h)
    s = phi.astype(np.float64)
    todo = ~np.isnan(P[..., 0]) & ~np.isnan(s)
    y, fell, _ = refine(phi, lc, h, x[todo], P[todo])
    Q = P.copy()
    Q[todo] = y
    return R.write(phi, Q, lc, h), int(is_band.sum()), int(fell.sum())
