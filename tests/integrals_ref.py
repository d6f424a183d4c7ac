"""NumPy restatement of the level-set integrals contract (``lsm_level_set_integrals``, include/lsm_b200.h).

Vectorised over cells, one simplex and one inside mask at a time, with the operation order of ``csrc/lsm_integrals.cu`` for every
contribution; the simplices, their primitives and the vertex coordinates are ``interface_ref``'s.  Only the order of the final sums
differs from the device (NumPy's pairwise sums against the device's per-plane sums), so the two agree to rounding, not bit for bit.
"""
from __future__ import annotations

import math

import numpy as np

import interface_ref as IR


def _corner(a, k, N):
    """The values at corner k of every cell (cells indexed like the nodes, one fewer along each axis)."""
    return a[tuple(slice((k >> d) & 1, a.shape[d] - 1 + ((k >> d) & 1)) for d in range(N))]


def _measure(V, N):
    if N == 1:
        return np.ones(V[0].shape[0])
    if N == 2:
        dx, dy = V[1][:, 0] - V[0][:, 0], V[1][:, 1] - V[0][:, 1]
        return np.sqrt(dx * dx + dy * dy)
    u, w = V[1] - V[0], V[2] - V[0]
    cx = u[:, 1] * w[:, 2] - u[:, 2] * w[:, 1]
    cy = u[:, 2] * w[:, 0] - u[:, 0] * w[:, 2]
    cz = u[:, 0] * w[:, 1] - u[:, 1] * w[:, 0]
    return np.sqrt((cx * cx + cy * cy) + cz * cz) / 2.0


def _mean(Fv, N):
    if N == 1:
        return Fv[0]
    if N == 2:
        return (Fv[0] + Fv[1]) / 2.0
    return ((Fv[0] + Fv[1]) + Fv[2]) / 3.0


def cell_integrals(phi, lc, h, level=0.0, F=None):
    """Per-cell contributions (vol, area, fvol, farea), each an array over the cells (fvol / farea None without F)."""
    phi = np.asarray(phi)
    N = phi.ndim
    lc = [float(v) for v in lc]
    h = [float(v) for v in h]
    hsign = -1 if sum(1 for v in h if v < 0) & 1 else 1
    s = phi.astype(np.float64) - float(level)
    f = None if F is None else np.asarray(F).astype(np.float64)
    V = abs(h[0])
    for d in range(1, N):
        V = V * abs(h[d])
    Vs = V / math.factorial(N)
    S = [_corner(s, k, N) for k in range(1 << N)]
    Fk = None if f is None else [_corner(f, k, N) for k in range(1 << N)]
    shape = S[0].shape
    cells = np.indices(shape)
    valid = np.all([~np.isnan(v) for v in S], axis=0)
    allin = valid & np.all([v <= 0 for v in S], axis=0)
    allout = valid & np.all([v > 0 for v in S], axis=0)
    vol, area = np.zeros(shape), np.zeros(shape)
    fvol, farea = (np.zeros(shape), np.zeros(shape)) if f is not None else (None, None)
    vol[allin] = V
    if f is not None:
        if N == 1:
            mean = (Fk[0] + Fk[1]) / 2.0
        elif N == 2:
            mean = (Fk[0] + Fk[3]) / 3.0 + (Fk[1] + Fk[2]) / 6.0
        else:
            mean = (Fk[0] + Fk[7]) / 4.0 + (((((Fk[1] + Fk[2]) + Fk[3]) + Fk[4]) + Fk[5]) + Fk[6]) / 12.0
        fvol[allin] = V * mean[allin]
    walk = ~allin & ~allout
    for p in range(len(IR.permutations(N))):
        w = IR.chain(N, p)
        ok = walk & np.all([~np.isnan(S[wk]) for wk in w], axis=0)
        mask = np.zeros(shape, np.int64)
        for x, wk in enumerate(w):
            mask |= (S[wk] <= 0).astype(np.int64) << x
        for m in range(1, 1 << (N + 1)):
            sel = ok & (mask == m)
            if not sel.any():
                continue
            sw = [S[wk][sel] for wk in w]
            fw = None if f is None else [Fk[wk][sel] for wk in w]

            def Fc(x, y):
                a, b = min(x, y), max(x, y)
                t = sw[a] / (sw[a] - sw[b])
                return fw[a] + t * (fw[b] - fw[a])

            k = bin(m).count("1")
            if k == N + 1:
                vol[sel] += Vs
                if f is not None:
                    tot = fw[0]
                    for x in range(1, N + 1):
                        tot = tot + fw[x]
                    fvol[sel] += Vs * (tot / float(N + 1))
                continue
            if k == 1 or k == N:
                bits = m if k == 1 else (~m & ((1 << (N + 1)) - 1))
                q = (bits & -bits).bit_length() - 1
                o = [x for x in range(N + 1) if x != q]
                u = [sw[q] / (sw[q] - sw[x]) for x in o]
                corner = u[0]
                for j in range(1, N):
                    corner = corner * u[j]
                if k == 1:
                    vol[sel] += Vs * corner
                    if f is not None:
                        tot = fw[q]
                        for x in o:
                            tot = tot + Fc(q, x)
                        fvol[sel] += (Vs * corner) * (tot / float(N + 1))
                elif N == 2:
                    va, vb = Vs * (1.0 - u[1]), Vs * (u[1] * (1.0 - u[0]))
                    vol[sel] += va
                    vol[sel] += vb
                    if f is not None:
                        Fr, Fs, fr = Fc(q, o[0]), Fc(q, o[1]), fw[o[0]]
                        fvol[sel] += va * (((fr + fw[o[1]]) + Fs) / 3.0)
                        fvol[sel] += vb * (((fr + Fs) + Fr) / 3.0)
                else:
                    vol[sel] += Vs * (1.0 - corner)
                    if f is not None:
                        whole = Vs * ((((fw[0] + fw[1]) + fw[2]) + fw[3]) / 4.0)
                        cut = (Vs * corner) * ((((fw[q] + Fc(q, o[0])) + Fc(q, o[1])) + Fc(q, o[2])) / 4.0)
                        fvol[sel] += whole - cut
            else:
                a, b = [x for x in range(4) if (m >> x) & 1]
                c, d = [x for x in range(4) if not (m >> x) & 1]
                tac, tad = sw[a] / (sw[a] - sw[c]), sw[a] / (sw[a] - sw[d])
                tbc, tbd = sw[b] / (sw[b] - sw[c]), sw[b] / (sw[b] - sw[d])
                v1, v2, v3 = Vs * ((tac * tad) * (1.0 - tbd)), Vs * ((tac * (1.0 - tbc)) * tbd), Vs * (tbc * tbd)
                vol[sel] += v1
                vol[sel] += v2
                vol[sel] += v3
                if f is not None:
                    Fac, Fad, Fbc, Fbd = Fc(a, c), Fc(a, d), Fc(b, c), Fc(b, d)
                    fvol[sel] += v1 * ((((fw[a] + Fac) + Fad) + Fbd) / 4.0)
                    fvol[sel] += v2 * ((((fw[a] + Fac) + Fbc) + Fbd) / 4.0)
                    fvol[sel] += v3 * ((((fw[a] + fw[b]) + Fbc) + Fbd) / 4.0)
            # the primitives, with interface_ref's vertex coordinates
            cs = [cells[d][sel] for d in range(N)]
            for prim in IR.simplex_primitives(N, p, m, hsign):
                Vx, Fv = [], []
                for (x, y) in prim:
                    a, b = w[x], w[y]
                    t = sw[x] / (sw[x] - sw[y])
                    X = np.empty((len(t), N))
                    for d in range(N):
                        g = (cs[d] + ((a >> d) & 1)).astype(np.float64)
                        X[:, d] = lc[d] + (g + t) * h[d] if ((a ^ b) >> d) & 1 else lc[d] + g * h[d]
                    Vx.append(X)
                    if f is not None:
                        Fv.append(fw[x] + t * (fw[y] - fw[x]))
                meas = _measure(Vx, N)
                area[sel] += meas
                if f is not None:
                    farea[sel] += meas * _mean(Fv, N)
    return vol, area, fvol, farea


def integrals(phi, lc, h, level=0.0, F=None):
    """(|{s <= 0}|, |{s = 0}|, integral of F over the region, over the interface); the last two NaN without F."""
    vol, area, fvol, farea = cell_integrals(phi, lc, h, level, F)
    if fvol is None:
        return float(vol.sum()), float(area.sum()), math.nan, math.nan
    return float(vol.sum()), float(area.sum()), float(fvol.sum()), float(farea.sum())


def scales(phi, lc, h, level=0.0, F=None):
    """The sums of the absolute per-cell contributions: the scale against which a relative tolerance of the signed sums is fair."""
    parts = cell_integrals(phi, lc, h, level, F)
    return tuple(math.nan if a is None else float(np.abs(a).sum()) for a in parts)


def mesh_integrals(phi, lc, h, level=0.0, F=None):
    """The interface measure and the integral of F over it, recomputed from interface_ref.extract's mesh: F at a vertex from the
    lattice edge its key names, Fa + t (Fb - Fa)."""
    phi = np.asarray(phi)
    N = phi.ndim
    X, P, K = IR.extract(phi, lc, h, level)
    if len(P) == 0:
        return 0.0, 0.0
    meas = _measure([X[P[:, j]] for j in range(N)], N)
    if F is None:
        return float(meas.sum()), math.nan
    ncode = (1 << N) - 1
    lin, e = K // ncode, K % ncode + 1
    a = np.stack(np.unravel_index(lin, phi.shape, order="F"))
    b = a + np.stack([(e >> d) & 1 for d in range(N)])
    s = phi.astype(np.float64) - float(level)
    f = np.asarray(F).astype(np.float64)
    sa, sb = s[tuple(a)], s[tuple(b)]
    fa, fb = f[tuple(a)], f[tuple(b)]
    t = sa / (sa - sb)
    fv = fa + t * (fb - fa)
    return float(meas.sum()), float((meas * _mean([fv[P[:, j]] for j in range(N)], N)).sum())
