"""SciPy restatement of the semi-implicit (inflow-implicit / outflow-explicit) advection step of include/lsm_b200.h
(LSM_SEMI_IMPLICIT): the linear system of one step is assembled with scipy.sparse and solved directly with spsolve, so the
engine's Jacobi sweeps are checked against the exact solution of the same system.

One step of phi_t + u.grad phi = 0 with u given at the nodes (at mid-step), for each node I and dimension d:
    c_d = dt u_d / h_d,  a_d = |c_d| / 2,  s_d = +1 if c_d > 0 else -1
    (1 + sum_d a_d) x_I - sum_d a_d x_{I - s_d e_d}  =  phi_I - sum_d a_d (phi_{I + s_d e_d} - phi_I)
Off-grid indices go through the boundary condition's index map on both sides: "periodic" (node n duplicates node 1),
"neumann" (ExtrapolationBC{0}) and "symmetry".  Arrays are N-d with the engine's column-major node order."""
import math

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

PERIODIC, NEUMANN, SYMMETRY = "periodic", "neumann", "symmetry"


def bc_map(j, n, lo, hi):
    """The in-grid node standing for indices j (one step off the grid at most) along an axis of n nodes."""
    j = np.asarray(j)
    out = j.copy()
    for mask, kind, left in ((j < 0, lo, True), (j >= n, hi, False)):
        jm = j[mask]
        if kind == PERIODIC:
            out[mask] = (n - 1) + jm if left else 1 + jm - n
        elif kind == SYMMETRY:
            out[mask] = -jm if left else 2 * (n - 1) - jm
        elif kind == NEUMANN:
            out[mask] = 0 if left else n - 1
        else:
            raise ValueError(kind)
    return out


def step(phi, u, h, dt, bcs):
    """phi^{n+1} from phi^n (N-d array), the velocity u (N arrays at the nodes), mesh sizes h, step dt and bcs[d] = (lo, hi)."""
    phi = np.asarray(phi, dtype=np.float64)
    shape, N, M = phi.shape, phi.ndim, phi.size
    lin = np.arange(M).reshape(shape, order="F")
    I = np.indices(shape)
    f = phi.ravel(order="F")
    diag = np.ones(M)
    S = np.zeros(M)
    rows, cols, vals = [], [], []
    for d in range(N):
        c = ((dt * np.asarray(u[d], dtype=np.float64)) / h[d]).ravel(order="F")
        a = np.abs(c) / 2
        s = np.where(c > 0, 1, -1)
        Id = I[d].ravel(order="F")

        def neighbour(offset):
            J = [I[e].ravel(order="F") for e in range(N)]
            J[d] = bc_map(Id + offset, shape[d], *bcs[d])
            return lin[tuple(J)]

        S = S + a * (f[neighbour(s)] - f)
        diag = diag + a
        rows.append(np.arange(M)); cols.append(neighbour(-s)); vals.append(-a)
    A = sp.coo_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(M, M)).tocsr()
    A = (A + sp.diags(diag)).tocsc()          # a ghost that maps onto the node itself lands on the diagonal
    x = spla.spsolve(A, f - S)
    return x.reshape(shape, order="F")


def cfl_dt(u, h):
    """The advection CFL step 1 / max_I sum_d |u_d| / h_d (levelsetterms.jl:90-96)."""
    m = np.abs(u[0]) / h[0]
    for d in range(1, len(u)):
        m = m + np.abs(u[d]) / h[d]
    return 1.0 / float(np.max(m))


def integrate(phi, velocity, h, bcs, tf, cfl=2.0, t0=0.0, dt_max=math.inf):
    """The loop of _integrate! with dt = min(dt_max, cfl * cfl_dt(u(tc)), tf - tc); velocity(t) -> N arrays.  (phi, steps)."""
    tc, steps = t0, 0
    while tc <= tf - np.spacing(abs(tc)):
        dt = min(dt_max, cfl * cfl_dt(velocity(tc), h), tf - tc)
        phi = step(phi, velocity(tc + 0.5 * dt), h, dt, bcs)
        tc += dt
        steps += 1
    return phi, steps


def sweeps(courant, f64=True):
    """Jacobi sweeps of a step at Courant number `courant`: ceil(log tol / log q), q = (C/2) / (1 + C/2), at least 1."""
    q = (courant / 2) / (1 + courant / 2)
    tol = 1e-15 if f64 else 1e-8
    return 1 if q == 0 else max(1, math.ceil(math.log(tol) / math.log(q)))
