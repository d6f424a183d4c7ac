"""NumPy restatement of the zero-level-set extraction contract (``lsm_interface_extract``, include/lsm_b200.h).

Marching simplices on the Freudenthal–Kuhn triangulation of the node lattice, vectorised over cells, with the same operation
order as ``csrc/lsm_interface.cu``, so that the device mesh equals this one bit for bit.  ``simplex_primitives`` is the per-simplex
rule (which cut edges form which primitive, in which order); ``extract`` applies it to a whole field.
"""
from __future__ import annotations

import itertools

import numpy as np


def permutations(N):
    """The N! permutations of the axes in lexicographic order (one simplex each)."""
    return list(itertools.permutations(range(N)))


def perm_sign(seq):
    inv = sum(1 for x in range(len(seq)) for y in range(x + 1, len(seq)) if seq[x] > seq[y])
    return -1 if inv & 1 else 1


def chain(N, p):
    """Corner indices w_0 .. w_N of simplex p (corner k = c + sum_d bit_d(k) e_d)."""
    w = [0]
    for ax in permutations(N)[p]:
        w.append(w[-1] | (1 << ax))
    return w


def simplex_primitives(N, p, inside, hsign=1):
    """Primitives of simplex p of a cell whose chain vertices w_k are inside where bit k of ``inside`` is set (all vertices
    valid).  Each primitive is a tuple of N edges (x, y), x < y chain positions; the edge's vertex is the crossing on it."""
    full = (1 << (N + 1)) - 1
    k = bin(inside).count("1")
    if k == 0 or k == N + 1:
        return []
    if N == 1:
        return [((0, 1),)]
    sgn = perm_sign(permutations(N)[p]) * hsign
    edge = lambda x, y: (min(x, y), max(x, y))
    if N == 2 or k != 2:
        lone_outside = k == N
        bits = (~inside & full) if lone_outside else inside
        q = (bits & -bits).bit_length() - 1
        others = [x for x in range(N + 1) if x != q]
        sigma = -sgn if q & 1 else sgn
        flip = (sigma < 0) != lone_outside
        e = [edge(q, o) for o in others]
        if N == 2:
            return [(e[1], e[0]) if flip else (e[0], e[1])]
        return [(e[0], e[2], e[1]) if flip else (e[0], e[1], e[2])]
    ins = [x for x in range(4) if (inside >> x) & 1]
    outs = [x for x in range(4) if not (inside >> x) & 1]
    sigma = perm_sign(ins + outs) * sgn
    ac, ad, bd, bc = edge(ins[0], outs[0]), edge(ins[0], outs[1]), edge(ins[1], outs[1]), edge(ins[1], outs[0])
    return [(ac, ad, bd), (ac, bd, bc)] if sigma > 0 else [(ac, bd, ad), (ac, bc, bd)]


def _bits(k, N):
    return np.array([(k >> d) & 1 for d in range(N)], dtype=np.int64)


def extract(phi, lc, h, level=0.0, first_last=0, nglob_last=None):
    """The mesh of {phi = level}: (vertices (nv, N) float64, faces (np, N) int32, keys (nv,) int64).

    ``phi`` is indexed [i1, i2, i3] (dim 1 first, like the column-major device array).  ``first_last`` / ``nglob_last`` describe a
    box that is a slab of a larger grid along the last axis (its global offset and the global node count there); the default is
    the whole grid."""
    phi = np.asarray(phi)
    N = phi.ndim
    n = phi.shape
    nglob = tuple(n[:-1]) + ((nglob_last if nglob_last is not None else n[-1]),)
    lc = [float(v) for v in lc]
    h = [float(v) for v in h]
    hsign = -1 if sum(1 for v in h if v < 0) & 1 else 1
    s = phi.astype(np.float64) - float(level)
    inside = s <= 0
    outside = s > 0
    ncode = (1 << N) - 1

    def glin(idx):
        g = list(idx)
        g[-1] = g[-1] + first_last
        return np.ravel_multi_index(tuple(g), nglob, order="F").astype(np.int64)

    keys, X = [], []
    for e in range(1, ncode + 1):
        ev = _bits(e, N)
        sa_sl = tuple(slice(0, n[d] - ev[d]) for d in range(N))
        sb_sl = tuple(slice(ev[d], n[d]) for d in range(N))
        cut = (inside[sa_sl] & outside[sb_sl]) | (outside[sa_sl] & inside[sb_sl])
        idx = np.nonzero(cut)
        sa, sb = s[sa_sl][idx], s[sb_sl][idx]
        t = sa / (sa - sb)
        x = np.empty((len(t), N))
        for d in range(N):
            ad = (idx[d] + (first_last if d == N - 1 else 0)).astype(np.float64)
            x[:, d] = lc[d] + (ad + t) * h[d] if ev[d] else lc[d] + ad * h[d]
        keys.append(glin(idx) * ncode + (e - 1))
        X.append(x)
    keys = np.concatenate(keys)
    X = np.concatenate(X, axis=0)
    order = np.argsort(keys, kind="stable")
    keys, X = keys[order], X[order]

    if any(v < 2 for v in n):
        return X, np.empty((0, N), np.int32), keys
    cells = np.indices(tuple(v - 1 for v in n)).reshape(N, -1)       # column-major order below via the lexsort on glin
    cell_lin = glin(tuple(cells))
    rows = []      # (cell_lin, simplex, sub, vertex indices)
    for p in range(len(permutations(N))):
        w = chain(N, p)
        sv = [s[tuple(slice(b, b + v - 1) for b, v in zip(_bits(wk, N), n))].reshape(-1, order="C") for wk in w]
        valid = np.all([~np.isnan(v) for v in sv], axis=0)
        mask = np.zeros(valid.shape, np.int64)
        for k, v in enumerate(sv):
            mask |= (v <= 0).astype(np.int64) << k
        for m in range(1, (1 << (N + 1)) - 1):
            sel = np.nonzero(valid & (mask == m))[0]
            if not len(sel):
                continue
            for j, prim in enumerate(simplex_primitives(N, p, m, hsign)):
                cols = []
                for (x, y) in prim:
                    a = cells[:, sel] + _bits(w[x], N)[:, None]
                    key = glin(tuple(a)) * ncode + ((w[x] ^ w[y]) - 1)
                    pos = np.searchsorted(keys, key)
                    assert np.all(keys[pos] == key)
                    cols.append(pos)
                rows.append((cell_lin[sel], np.full(len(sel), p), np.full(len(sel), j), np.stack(cols, axis=1)))
    if not rows:
        return X, np.empty((0, N), np.int32), keys
    cl = np.concatenate([r[0] for r in rows])
    sp = np.concatenate([r[1] for r in rows])
    sj = np.concatenate([r[2] for r in rows])
    F = np.concatenate([r[3] for r in rows], axis=0)
    order = np.lexsort((sj, sp, cl))
    return X, F[order].astype(np.int32), keys


# ---- mesh checks ----------------------------------------------------------------------------------
def edge_counts(F):
    """(undirected edge -> uses, directed edge -> uses) of a triangle mesh."""
    F = F.astype(np.int64)
    a = np.concatenate([F[:, 0], F[:, 1], F[:, 2]])
    b = np.concatenate([F[:, 1], F[:, 2], F[:, 0]])
    nv = int(F.max()) + 1 if F.size else 1
    _, cu = np.unique(np.minimum(a, b) * nv + np.maximum(a, b), return_counts=True)
    _, cd = np.unique(a * nv + b, return_counts=True)
    return cu, cd


def euler_characteristic(X, F):
    cu, _ = edge_counts(F)
    return len(np.unique(F)) - len(cu) + len(F)


def area(X, F):
    a, b, c = X[F[:, 0]], X[F[:, 1]], X[F[:, 2]]
    return 0.5 * np.linalg.norm(np.cross(b - a, c - a), axis=1).sum()


def enclosed_volume(X, F):
    """Divergence theorem: positive when the normals point out of the enclosed (inside) region."""
    a, b, c = X[F[:, 0]], X[F[:, 1]], X[F[:, 2]]
    return np.einsum("ij,ij->i", a, np.cross(b, c)).sum() / 6.0


def signed_area_2d(X, F):
    """Shoelace over the segments: positive when the inside lies on the left of every segment."""
    a, b = X[F[:, 0]], X[F[:, 1]]
    return 0.5 * (a[:, 0] * b[:, 1] - b[:, 0] * a[:, 1]).sum()
