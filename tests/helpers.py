"""Shared builders for the parity tests: the same synthetic, seed-free configuration is materialised
once for the CPU oracle (``oracle.Field`` / ``oracle.Term``) and once for the engine
(``lsm_b200.MeshField`` / terms).  Configurations follow SURVEY.md §8(d) / BASELINE.json ``configs``.
"""
from __future__ import annotations

import numpy as np

import oracle as O


def coords(lc, hc, n):
    out = []
    N = len(n)
    for d in range(N):
        h = (hc[d] - lc[d]) / (n[d] - 1)
        x = lc[d] + np.arange(n[d], dtype=np.float64) * h
        shape = [1] * N
        shape[d] = n[d]
        out.append(x.reshape(shape))
    return out


def bcast(a, n):
    return np.asfortranarray(np.broadcast_to(a, n).copy())


class Case:
    """A named configuration: grid, phi0, list of term specs, BC spec, integrator, dtype."""

    def __init__(self, name, lc, hc, n, phi0, terms, bc, dtype=np.float64):
        self.name, self.lc, self.hc, self.n = name, tuple(lc), tuple(hc), tuple(n)
        self.phi0 = np.asfortranarray(phi0.astype(dtype))
        self.terms, self.bc, self.dtype = terms, bc, dtype

    def coef_field(self, t):
        """A term's stored coefficient, in its own ``field_dtype`` when it sets one (a Float64 field with a Float32 state)."""
        return np.asfortranarray(t["field"].astype(t.get("field_dtype", self.dtype)))

    # ---- oracle side ----
    def oracle_bc(self):
        def one(b):
            k = b[0]
            return {"periodic": O.PERIODIC, "neumann": O.NEUMANN, "symmetry": O.SYMMETRY}.get(k) or O.EXTRAP(b[1])
        if isinstance(self.bc, tuple) and isinstance(self.bc[0], str):
            return one(self.bc)
        return [one(b) if isinstance(b[0], str) else (one(b[0]), one(b[1])) for b in self.bc]

    def oracle_field(self):
        return O.Field(self.phi0.copy(order="F"), self.lc, self.hc, bc=self.oracle_bc())

    def oracle_terms(self, s0=None):
        out = []
        for t in self.terms:
            k = t["kind"]
            if k == "advection":
                sch = O.UPWIND if t.get("scheme") == "upwind" else O.WENO5
                ts = O.TS_COS if "cos_period" in t else O.TS_NONE
                tp = t.get("cos_period", 1.0)
                if "separable" in t:
                    sc, tabs = t["separable"]
                    out.append(O.advection_separable(sc, tabs, scheme=sch, tscale=ts, tparam=tp))
                elif "field" in t:
                    out.append(O.advection(self.coef_field(t), scheme=sch, tscale=ts, tparam=tp))
                else:
                    out.append(O.advection(t["const"], scheme=sch, tscale=ts, tparam=tp))
            elif k == "normal":
                out.append(O.normal_motion(self.coef_field(t) if "field" in t else t["const"]))
            elif k == "curvature":
                out.append(O.curvature(self.coef_field(t) if "field" in t else t["const"]))
            elif k == "eikonal":
                if t.get("frozen", True):
                    out.append(O.eikonal(O.eikonal_s0(self.oracle_field()) if s0 is None else s0))
                else:
                    out.append(O.eikonal())
        return out

    # ---- engine side (lsm_b200 host mirror) ----
    def engine_bc(self, m):
        def one(b):
            k = b[0]
            if k == "periodic":
                return m.PeriodicBC()
            if k == "neumann":
                return m.NeumannBC()
            if k == "symmetry":
                return m.SymmetryBC()
            return m.ExtrapolationBC(b[1])
        if isinstance(self.bc, tuple) and isinstance(self.bc[0], str):
            return one(self.bc)
        return tuple(one(b) if isinstance(b[0], str) else (one(b[0]), one(b[1])) for b in self.bc)

    def engine_grid(self, m):
        return m.CartesianGrid(self.lc, self.hc, self.n)

    def engine_field(self, m, ctx=None):
        return m.MeshField(self.phi0.copy(order="F"), self.engine_grid(m), bc=self.engine_bc(m), ctx=ctx)

    def engine_terms(self, m, phi, ctx=None):
        out = []
        g = phi.mesh
        for t in self.terms:
            k = t["kind"]
            if k == "advection":
                sch = m.Upwind() if t.get("scheme") == "upwind" else m.WENO5()
                if "separable" in t:
                    sc, tabs = t["separable"]
                    base = m.SeparableVelocity(g, sc, tabs, ctx=ctx)
                elif "field" in t:
                    base = m.MeshField(self.coef_field(t), g, ctx=ctx)
                else:
                    base = tuple(t["const"])
                if "cos_period" in t:
                    base = m.TimeScaled(base, ("cos", t["cos_period"]))
                out.append(m.AdvectionTerm(base, sch))
            elif k == "normal":
                v = m.MeshField(self.coef_field(t), g, ctx=ctx) if "field" in t else t["const"]
                out.append(m.NormalMotionTerm(v))
            elif k == "curvature":
                b = m.MeshField(self.coef_field(t), g, ctx=ctx) if "field" in t else t["const"]
                out.append(m.CurvatureTerm(b))
            elif k == "eikonal":
                out.append(m.EikonalReinitializationTerm(phi) if t.get("frozen", True) else m.EikonalReinitializationTerm())
        return tuple(out)


# ---- BASELINE.json configs, scaled (SURVEY.md §8d) ----------------------------------------------
def c1_circle_rotation(n=128, dtype=np.float64, bc=("periodic",)):
    """C1: 2-D circle SDF under rigid rotation, WENO5, periodic."""
    lc, hc, nn = (-1, -1), (1, 1), (n, n)
    x, y = coords(lc, hc, nn)
    phi = np.hypot(x - 0.3, y) - 0.4
    u = np.stack([bcast(-y, nn), bcast(x, nn)], axis=0)
    return Case("C1", lc, hc, nn, phi, [dict(kind="advection", field=u)], bc, dtype)


def c2_zalesak_curvature(n=256, dtype=np.float64):
    """C2: Zalesak disk rotation + curvature (b = -0.01), Neumann (docs/src/example-zalesak.md:21-40)."""
    lc, hc, nn = (-1.5, -1.5), (1.5, 1.5), (n, n)
    x, y = coords(lc, hc, nn)
    cx, cy, r, w, hgt = -0.75, 0.0, 0.5, 0.2, 1.0
    disk = np.hypot(x - cx, y - cy) - r
    rec = np.maximum(np.abs(x - cx) - w / 2, np.abs(y - (cy - r)) - hgt / 2)
    phi = np.maximum(disk, -rec)
    u = np.stack([bcast(-y, nn), bcast(x, nn)], axis=0)
    return Case("C2", lc, hc, nn, bcast(phi, nn), [dict(kind="advection", field=u), dict(kind="curvature", const=-0.01)],
                ("neumann",), dtype)


def enright_tables(lc, hc, n):
    x, y, z = [c.ravel() for c in coords(lc, hc, n)]
    s2 = lambda a: np.sin(np.pi * a) ** 2
    s = lambda a: np.sin(2 * np.pi * a)
    tabs = [[s2(x), s(y), s(z)], [s(x), s2(y), s(z)], [s(x), s(y), s2(z)]]
    return (2.0, -1.0, -1.0), tabs


def c3_enright(n=64, dtype=np.float64, separable=False, period=3.0):
    """C3: 3-D sphere in the Enright/LeVeque deformation field x cos(pi t / T), WENO5, Neumann."""
    lc, hc, nn = (0, 0, 0), (1, 1, 1), (n, n, n)
    x, y, z = coords(lc, hc, nn)
    phi = np.sqrt((x - 0.35) ** 2 + (y - 0.35) ** 2 + (z - 0.35) ** 2) - 0.15
    sc, tabs = enright_tables(lc, hc, nn)
    if separable:
        term = dict(kind="advection", separable=(sc, tabs), cos_period=period)
    else:
        X, Y, Z = np.meshgrid(*[np.arange(k) for k in nn], indexing="ij", sparse=True)
        u = np.stack([((sc[d] * tabs[d][0][X]) * tabs[d][1][Y]) * tabs[d][2][Z] for d in range(3)], axis=0)
        term = dict(kind="advection", field=u, cos_period=period)
    return Case("C3", lc, hc, nn, phi, [term], ("neumann",), dtype)


def c4_eikonal(n=64, dtype=np.float64, frozen=True):
    """C4: Eikonal reinitialisation of a perturbed sphere SDF, Neumann."""
    lc, hc, nn = (-1, -1, -1), (1, 1, 1), (n, n, n)
    x, y, z = coords(lc, hc, nn)
    r = np.sqrt(x * x + y * y + z * z)
    phi = (r - 0.5) * (1 + 0.4 * np.sin(3 * np.pi * x) * np.sin(3 * np.pi * y) * np.sin(3 * np.pi * z))
    return Case("C4", lc, hc, nn, phi, [dict(kind="eikonal", frozen=frozen)], ("neumann",), dtype)


def c5_normal_advection(n=64, dtype=np.float64):
    """C5: NormalMotionTerm(v field = 0.2) + AdvectionTerm(u = (-y, x, 0) field), Neumann."""
    lc, hc, nn = (-1, -1, -1), (1, 1, 1), (n, n, n)
    x, y, z = coords(lc, hc, nn)
    phi = np.sqrt((x - 0.3) ** 2 + y * y + z * z) - 0.4
    v = np.full(nn, 0.2)
    u = np.stack([bcast(-y, nn), bcast(x, nn), np.zeros(nn)], axis=0)
    return Case("C5", lc, hc, nn, phi, [dict(kind="normal", field=v), dict(kind="advection", field=u)], ("neumann",), dtype)


# ---- the term / BC matrix of the stage-kernel parity tests ----------------------------------------------------------
def small_problem(n):
    """Grid corners, phi0 and the stored velocity u, speed v and curvature coefficient b of the term / BC matrix on an n grid
    (1-, 2- or 3-D; anisotropic mesh sizes, sign changes of every coefficient)."""
    N = len(n)
    lc, hc = [-1.0] * N, [1.0 + 0.1 * d for d in range(N)]
    X = coords(lc, hc, n)
    r = np.sqrt(sum((x - 0.1) ** 2 for x in X))
    phi = bcast((r - 0.5) * (1 + 0.3 * np.sin(3 * X[0])), n)
    u = np.stack([bcast(np.sin(2 * X[d] + d) + 0.2, n) for d in range(N)], axis=0)
    v = bcast(0.3 + 0.5 * np.cos(2 * X[0]), n)
    b = bcast(-0.02 - 0.01 * np.sin(X[-1]), n)
    return lc, hc, phi, u, v, b


def small_termsets(u, v, b, N):
    """Every term kind and coefficient kind alone, and the two- and three-term lists the stage kernels dispatch on."""
    return {
        "adv_weno": [dict(kind="advection", field=u)],
        "adv_upwind": [dict(kind="advection", field=u, scheme="upwind")],
        "adv_const_cos": [dict(kind="advection", const=tuple([0.7, -0.4, 0.5][:N]), cos_period=0.05)],
        "normal": [dict(kind="normal", field=v)],
        "normal_const": [dict(kind="normal", const=-0.8)],
        "curv": [dict(kind="curvature", field=b)],
        "curv_const": [dict(kind="curvature", const=-0.05)],
        "eik_frozen": [dict(kind="eikonal", frozen=True)],
        "eik_live": [dict(kind="eikonal", frozen=False)],
        "three": [dict(kind="normal", field=v), dict(kind="advection", field=u), dict(kind="curvature", const=-0.01)],
        # two-term lists: the BASELINE orders run the static-signature kernels (C5: normal+adv fields, C2: adv field + const
        # curvature); the reversed orders / other coefficient kinds must take the runtime-dispatch kernels of the same masks
        "normal_adv": [dict(kind="normal", field=v), dict(kind="advection", field=u)],
        "adv_normal": [dict(kind="advection", field=u), dict(kind="normal", field=v)],
        "normalc_adv": [dict(kind="normal", const=0.6), dict(kind="advection", field=u)],
        "adv_curvc": [dict(kind="advection", field=u), dict(kind="curvature", const=-0.03)],
        "curvc_adv": [dict(kind="curvature", const=-0.03), dict(kind="advection", field=u)],
        "adv_curvf": [dict(kind="advection", field=u), dict(kind="curvature", field=b)],
    }


SMALL_BCS = (("periodic",), ("neumann",), ("extrap", 2), ("symmetry",), ("extrap", 1))
SMALL_SPLIT = (("neumann",), ("extrap", 1))


def small_bc(i, N, bcs=SMALL_BCS, split=SMALL_SPLIT):
    """BC of the i-th term set: bcs[(i + d) % len(bcs)] along axis d; every third set (2-D and 3-D) has `split`'s two
    different sides along y."""
    bc = tuple(bcs[(i + d) % len(bcs)] for d in range(N))
    if N > 1 and i % 3 == 0:
        bc = (bc[0], split) + bc[2:]
    return bc


def small_cases(n, bcs=SMALL_BCS, split=SMALL_SPLIT):
    """[(f"{N}d-{term set}", Case)] of the term / BC matrix on an n grid."""
    N = len(n)
    lc, hc, phi, u, v, b = small_problem(n)
    return [(f"{N}d-{tn}", Case(tn, lc, hc, n, phi, ts, small_bc(i, N, bcs, split)))
            for i, (tn, ts) in enumerate(small_termsets(u, v, b, N).items())]


# ---- integration through the oracle and the engine -----------------------------------------------------------------
INTEG = {"FE": 0, "RK2": 1, "RK3": 2}


def run_oracle(O, case, integ="RK3", steps=100, tf=None, cfl=0.5):
    """Integrate `case` with the oracle; return (phi, t, nsteps, tf).  Without `tf`, tf is chosen from the initial CFL step so
    that exactly `steps` steps are taken when dt is constant."""
    fo = case.oracle_field()
    to = case.oracle_terms()
    if tf is None:
        dt0 = cfl * O.compute_cfl(fo, to, 0.0)
        tf = dt0 * steps * (1 - 1e-12)
    t_o, n_o = O.integrate(fo, INTEG[integ], to, tf, cfl=cfl)
    return fo.vals, t_o, n_o, tf


def run_engine(m, case, integ, tf, cfl=0.5):
    """Integrate `case` to `tf` with the engine (the context's current kernel options); return the equation."""
    phi = case.engine_field(m)
    terms = case.engine_terms(m, phi)
    eq = m.LevelSetEquation(terms=terms, ic=phi, integrator=getattr(m, {"FE": "ForwardEuler"}.get(integ, integ))(cfl))
    m.integrate(eq, tf)
    return eq


def run_pair(m, O, case, integ="RK3", steps=100, tf=None, cfl=0.5):
    """Integrate `case` with the oracle and the engine; return (phi_oracle, phi_engine, t, nsteps)."""
    a, t_o, n_o, tf = run_oracle(O, case, integ, steps, tf, cfl)
    eq = run_engine(m, case, integ, tf, cfl)
    assert eq.t == t_o
    assert eq.steps_taken == n_o
    return a, eq.state.peek(), t_o, n_o


def check_parity(a, b, tol):
    assert not np.isnan(b).any()
    d = np.abs(a.astype(np.float64) - b.astype(np.float64)).max()
    assert d <= tol, f"max-abs difference {d:.3e} > {tol:.1e}"
    assert np.array_equal(np.sign(a), np.sign(b)), "zero-level-set node classification differs"
    assert np.array_equal(cut_cells(a), cut_cells(b)), "cut-cell classification differs"
    return d


def cut_cells(phi):
    """Per-cell cut flag over all 2^N corners: vmin <= 0 <= vmax (meshfield.jl:566-575)."""
    N = phi.ndim
    vmin = vmax = None
    for corner in np.ndindex(*([2] * N)):
        sl = tuple(slice(c, phi.shape[d] - 1 + c) for d, c in enumerate(corner))
        v = phi[sl]
        vmin = v if vmin is None else np.minimum(vmin, v)
        vmax = v if vmax is None else np.maximum(vmax, v)
    return (vmin <= 0) & (vmax >= 0)
