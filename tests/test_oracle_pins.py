"""Pins the CPU oracle against every exact-value / known-answer check the reference's own
test-suite and doctests hold for the dense-grid integration path (SURVEY.md §8c).

Each test names the reference test it re-expresses (paths relative to the root of the LevelSetMethods.jl repository).
"""
import json
import math
import os

import numpy as np
import pytest


GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
KNOWN = json.load(open(os.path.join(GOLDEN, "reference_known_answers.json")))      # numbers the reference itself states, with citations


def mk(O, f, lc, hc, n, bc=None, dtype=np.float64):
    fld = O.Field(np.zeros(n, dtype=dtype, order="F"), lc, hc, bc=bc)
    X = fld.nodes()
    fld.vals[...] = np.broadcast_to(f(*X), fld.vals.shape).astype(dtype)
    return fld


# ---- src/levelsetops.jl:14-25 and :126-137 (jldoctest scalars) : the only stored numbers ----
def test_doctest_volume_perimeter_bitexact(O):
    k = KNOWN["doctest_circle_200x200"]
    f = mk(O, lambda x, y: np.sqrt(x * x + y * y) - k["radius"], k["lc"], k["hc"], tuple(k["n"]))
    assert f.volume() == k["volume"] == 0.7854362890190668
    assert f.perimeter() == k["perimeter"] == 3.1426415491430384


# ---- test/test-meshes.jl:6-14 ----
def test_grid_nodes_exact(O):
    f = mk(O, lambda x, y: x + y, (-1, 0), (1, 3), (100, 50))
    assert f.getnode((1, 1)) == [-1.0, 0.0]
    assert f.getnode((100, 50)) == [1.0, 3.0]
    assert f.meshsize() == [2 / 99, 3 / 49]


# ---- test/test-meshfield.jl:44-55 ----
def test_periodic_getindex_exact(O):
    rng = np.random.default_rng(0)
    vals = rng.random((10, 5))
    mf = O.Field(vals, (0, 0), (1, 1), bc=[O.PERIODIC, O.PERIODIC])
    assert mf[1, 1] == vals[0, 0]
    assert mf[1, 0] == vals[0, 3]          # mf[1,0] == vals[1,4] (1-based)
    assert mf[11, 5] == mf[2, 5]
    # period is n-1 cells: ghost(1-k) = node(n-k), ghost(n+k) = node(1+k)
    for k in (1, 2, 3):
        assert mf[1 - k, 2] == vals[10 - k - 1, 1]
        assert mf[10 + k, 2] == vals[k, 1]


# ---- test/test-meshfield.jl:57-98 ----
def test_extrapolation_getindex(O):
    a, b, n = -0.3, 1.7, 10
    h = (b - a) / (n - 1)
    for P in range(0, 6):
        for k in range(0, P + 1):
            f = mk(O, lambda x: x ** k, (a,), (b,), (n,), bc=[O.EXTRAP(P)])
            for j in range(1, P + 2):
                assert f[1 - j] == pytest.approx((a - j * h) ** k, abs=1e-10)
                assert f[n + j] == pytest.approx((b + j * h) ** k, abs=1e-10)
    a1, a2, b1, b2, n1, n2 = -0.3, 0.5, 1.7, 2.1, 8, 6
    h1, h2 = (b1 - a1) / (n1 - 1), (b2 - a2) / (n2 - 1)
    for P in (1, 2, 3):
        for j in range(P + 1):
            for k in range(P + 1):
                g = lambda x, y: x ** j * y ** k
                f = mk(O, g, (a1, a2), (b1, b2), (n1, n2), bc=[O.EXTRAP(P), O.EXTRAP(P)])
                y3 = f.getnode((1, 3))[1]
                assert f[0, 3] == pytest.approx(g(a1 - h1, y3), abs=1e-10)
                assert f[n1 + 1, 3] == pytest.approx(g(b1 + h1, y3), abs=1e-10)
                assert f[0, 0] == pytest.approx(g(a1 - h1, a2 - h2), abs=1e-10)
                assert f[n1 + 1, n2 + 1] == pytest.approx(g(b1 + h1, b2 + h2), abs=1e-10)


def test_extrapolation_weight_table():
    """SURVEY.md §8a table for w_j(k,P) (boundaryconditions.jl:90-97) via ghost reads of unit vectors."""
    import oracle as O
    wt = KNOWN["lagrange_extrapolation_weights"]
    table = {(P, k): wt[f"P{P}"][f"k{k}"] for P in range(4) for k in (1, 2, 3)}
    assert table[(2, 3)] == [10, -15, 6] and table[(3, 2)] == [10, -20, 15, -4]
    n = 8
    for (P, k), w in table.items():
        for j, wj in enumerate(w):
            e = np.zeros(n); e[j] = 1.0
            assert O.Field(e, (0,), (1,), bc=[O.EXTRAP(P)])[1 - k] == pytest.approx(wj, abs=1e-12)
            e = np.zeros(n); e[n - 1 - j] = 1.0
            assert O.Field(e, (0,), (1,), bc=[O.EXTRAP(P)])[n + k] == pytest.approx(wj, abs=1e-12)


# ---- test/test-meshfield.jl:100-125 ----
def test_symmetry_getindex(O):
    f = mk(O, lambda x: x, (0.0,), (4.0,), (5,), bc=[O.SYMMETRY])
    fn = mk(O, lambda x: x, (0.0,), (4.0,), (5,), bc=[O.NEUMANN])
    assert f[0] == 1.0 and f[-1] == 2.0 and f[6] == 3.0 and f[7] == 2.0
    assert fn[0] == 0.0 and f[0] != fn[0]
    g = mk(O, lambda x: x * x, (0.0,), (4.0,), (5,), bc=[O.SYMMETRY])
    assert g[0] == pytest.approx(1.0) and g[-1] == pytest.approx(4.0)
    f2 = mk(O, lambda x, y: x + 10 * y, (0.0, 0.0), (4.0, 4.0), (5, 5), bc=[O.SYMMETRY, O.SYMMETRY])
    assert f2[0, 0] == f2[2, 2]


# ---- test/test-boundaryconditions.jl ----
def test_normalize_bc(O):
    P, N, E2 = O.PERIODIC, O.NEUMANN, O.EXTRAP(2)
    assert O._norm_bc(P, 2) == [(P, P), (P, P)]
    assert O._norm_bc([P, N], 2) == [(P, P), (N, N)]
    r = O._norm_bc([P, (E2, N)], 2)
    assert r[0] == (P, P) and r[1] == (E2, N)
    with pytest.raises(ValueError):
        O._norm_bc([(P, E2), (E2, N)], 2)


# ---- test/test-derivatives.jl:15-42 ----
def test_derivative_stencils(O):
    f = mk(O, lambda x, y: x ** 3 + x * y ** 2, (-2.0, -2.0), (2.0, 2.0), (400, 200))
    h = f.meshsize()
    I = (9, 7)
    x, y = f.getnode(I)
    exact = (3 * x * x + y * y, 2 * x * y)
    for dim in (1, 2):
        hd = h[dim - 1]
        assert abs(f.deriv("D+", I, dim) - exact[dim - 1]) < 10 * hd
        assert abs(f.deriv("D-", I, dim) - exact[dim - 1]) < 10 * hd
        assert abs(f.deriv("D0", I, dim) - exact[dim - 1]) < 5 * hd ** 2
        assert abs(f.deriv("weno5-", I, dim) - exact[dim - 1]) < 5 * hd ** 2
        assert abs(f.deriv("weno5+", I, dim) - exact[dim - 1]) < 5 * hd ** 2
    diag = (6 * x, 2 * x)
    for dim in (1, 2):
        hd = h[dim - 1]
        assert abs(f.deriv("D2_0", I, dim) - diag[dim - 1]) < 5 * hd
        assert abs(f.deriv("D2++", I, dim) - diag[dim - 1]) < 10 * hd
        assert abs(f.deriv("D2--", I, dim) - diag[dim - 1]) < 10 * hd
    for d1, d2 in ((1, 2), (2, 1)):
        assert abs(f.deriv("D2", I, d1, d2) - 2 * y) < 5 * h[0] * h[1]


def test_weno5_known_answers(O):
    L = O.lib()
    # linear data: every candidate equals the common slope; smooth weights are the ideal ones
    assert L.orc_weno5(2.0, 2.0, 2.0, 2.0, 2.0) == pytest.approx(2.0, rel=1e-15)
    # flat data must give finite (zero) result thanks to the 1e-99 floor (test-levelsetterms.jl:53-77)
    assert L.orc_weno5(0.0, 0.0, 0.0, 0.0, 0.0) == 0.0
    # linear-in-i data v_i = i: all three third-order candidates equal 3.5, so any convex combination is 3.5
    assert L.orc_weno5(1.0, 2.0, 3.0, 4.0, 5.0) == pytest.approx(3.5, rel=1e-15)
    # a shock on the right: weight collapses onto the left candidate d1 = 1/3 v1 - 7/6 v2 + 11/6 v3
    v = (1.0, 1.0, 1.0, 1.0, 1000.0)
    assert L.orc_weno5(*v) == pytest.approx(1.0, rel=1e-6)
    # minmod limiter (levelsetterms.jl:184-187)
    assert L.orc_limiter(1.0, 2.0) == 1.0 and L.orc_limiter(-3.0, -2.0) == -2.0
    assert L.orc_limiter(1.0, -2.0) == 0.0 and L.orc_limiter(0.0, 5.0) == 0.0


# ---- test/test-levelsetterms.jl:7-31 ----
def test_cfl_closed_forms(O):
    f = mk(O, lambda x: x, (-1.0,), (1.0,), (100,))
    dx = f.meshsize(1)
    assert O.compute_cfl(f, [O.advection((2.0,))]) == pytest.approx(dx / 2.0, rel=1e-15)
    assert O.compute_cfl(f, [O.normal_motion(3.0)]) == pytest.approx(dx / 3.0, rel=1e-15)
    g = mk(O, lambda x, y: np.sqrt(x * x + y * y) - 0.5, (-1.0, -1.0), (1.0, 1.0), (50, 50))
    dxm = min(g.meshsize())
    assert O.compute_cfl(g, [O.curvature(0.5)]) == pytest.approx(dxm ** 2 / (2 * 0.5), rel=1e-15)
    # min over terms; stored velocity field; NaN / zero velocity semantics (SURVEY A.6)
    u = np.zeros((2, 50, 50), order="F"); u[0] = 1.0; u[1] = -3.0
    hx, hy = g.meshsize()
    assert O.compute_cfl(g, [O.advection(u), O.curvature(1e-9)]) == 1 / (1.0 / hx + 3.0 / hy)
    assert O.compute_cfl(g, [O.advection(np.zeros_like(u))]) == math.inf
    u[0, 3, 4] = np.nan
    with pytest.raises(O.CFLError):
        O.compute_cfl(g, [O.advection(u)])
    u[0, 3, 4] = np.inf
    with pytest.raises(O.CFLError):
        O.compute_cfl(g, [O.advection(u)])


# ---- test/test-levelsetterms.jl:33-51 ----
def test_eikonal_1d_reinit(O):
    f = mk(O, lambda x: 2 * (x - 0.3), (-1.0,), (1.0,), (101,), bc=[O.EXTRAP(1)])
    s0 = O.eikonal_s0(f)
    O.integrate(f, O.RK2, [O.eikonal(s0)], 2.0)
    x = f.nodes()[0]
    err = np.where(np.abs(f.vals) > 0.5, 0.0, np.abs(f.vals - (x - 0.3))).max()
    assert err < 0.05


# ---- test/test-levelsetterms.jl:53-77 ----
def test_nan_robustness(O):
    f = mk(O, lambda x, y: np.sqrt(x * x + y * y) - 0.7, (-2.0, -2.0), (2.0, 2.0), (31, 31), bc=O.NEUMANN)
    O.integrate(f, O.RK2, [O.curvature(-0.1)], 0.1)
    assert not np.isnan(f.vals).any()
    g = mk(O, lambda x: 0.0 * x, (-1.0,), (1.0,), (31,), bc=O.NEUMANN)
    O.integrate(g, O.RK2, [O.eikonal()], 0.1)
    assert not np.isnan(g.vals).any()
    # flat field under WENO5 advection stays finite too (epsilon floor)
    hflat = mk(O, lambda x: 0.0 * x + 1.0, (-1.0,), (1.0,), (31,), bc=O.PERIODIC)
    O.integrate(hflat, O.RK3, [O.advection((1.0,))], 0.1)
    assert np.all(hflat.vals == 1.0)


# ---- test/test-timestepping.jl:8-46 ----
def _adv_err_1d(O, integ, N, u=1.0, tf=0.5, cfl=0.5, scheme=None):
    f = mk(O, lambda x: np.sin(np.pi * x), (-1.0,), (1.0,), (N,), bc=O.PERIODIC)
    sch = O.WENO5 if scheme is None else scheme
    O.integrate(f, integ, [O.advection((u,), scheme=sch)], tf, cfl=cfl)
    x = f.nodes()[0]
    return np.abs(f.vals - np.sin(np.pi * (x - u * tf))).max()


def test_timestepping_accuracy(O):
    assert _adv_err_1d(O, O.FE, 200) < 0.05
    assert _adv_err_1d(O, O.RK2, 200) < 1.0e-3
    assert _adv_err_1d(O, O.RK3, 200) < 1.0e-5


def test_timestepping_orders(O):
    Ns = [50, 100, 200, 400]
    for integ, p in ((O.FE, 1), (O.RK2, 2), (O.RK3, 3)):
        e = [_adv_err_1d(O, integ, N) for N in Ns]
        for i in range(len(Ns) - 1):
            assert math.log(e[i] / e[i + 1]) / math.log(Ns[i + 1] / Ns[i]) >= p - 0.5


# ---- test/test-levelsetequation.jl:26-65 ----
def test_weno5_exact_rational_vectors(O):
    """`_weno5` against the reference formula evaluated in exact rational arithmetic (tests/golden/make_weno5_vectors.py;
    dyadic inputs, exact values of the Float64 literals): independent of any rounding order, so it pins coefficients, signs
    and the structure of the weights to a few ulp."""
    import json
    L = O.lib()
    g = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_known_answers.json")))["weno5_exact"]
    assert len(g["cases"]) >= 7
    for c in g["cases"]:
        got = L.orc_weno5(*c["v"])
        assert got == pytest.approx(c["expected"], rel=g["rel_tol"], abs=0.0), (c, got)


def test_weno5_and_upwind_spatial_order(O):
    Ns = [20, 40, 80]
    e = [_adv_err_1d(O, O.RK3, N, cfl=1e-2) for N in Ns]
    assert all(math.log(e[i] / e[i + 1]) / math.log(2) >= 4.5 for i in range(2))
    Ns = [50, 100, 200]
    e = [_adv_err_1d(O, O.RK3, N, cfl=1e-2, scheme=O.UPWIND) for N in Ns]
    assert all(math.log(e[i] / e[i + 1]) / math.log(2) >= 0.8 for i in range(2))


# ---- test/test-levelsetequation.jl:67-119 ----
def test_normal_motion_and_curvature_order(O):
    def run(N, term, exact):
        f = mk(O, lambda x, y: np.sqrt(x * x + y * y) - r0, (-2.0, -2.0), (2.0, 2.0), (N, N), bc=O.EXTRAP(2))
        O.integrate(f, O.RK3, [term], 0.2)
        x, y = f.nodes()
        r = np.sqrt(x * x + y * y)
        return np.where((r >= 0.5) & (r <= 1.5), np.abs(f.vals - exact(r)), 0.0).max()

    r0, v, tf = 0.5, 0.5, 0.2
    e = [run(N, O.normal_motion(v), lambda r: r - r0 - v * tf) for N in (30, 60, 120)]
    assert all(math.log(e[i] / e[i + 1]) / math.log(2) >= 1.5 for i in range(2))
    r0, b = 0.7, -0.1
    e = [run(N, O.curvature(b), lambda r: np.sqrt(r * r - 2 * b * tf) - r0) for N in (30, 60, 120)]
    assert all(math.log(e[i] / e[i + 1]) / math.log(2) >= 1.5 for i in range(2))


# ---- src/levelsetequation.jl:194-203 / timestepping.jl:101-122 : loop semantics ----
def test_integrate_loop_semantics(O):
    f = mk(O, lambda x: np.sin(np.pi * x), (-1.0,), (1.0,), (101,), bc=O.PERIODIC)
    h = f.meshsize(1)
    t, steps = O.integrate(f, O.RK3, [O.advection((1.0,))], 0.5)
    assert t == 0.5 and steps == math.ceil(0.5 / (0.5 * h) - 1e-9)
    with pytest.raises(ValueError):
        O.integrate(f, O.RK3, [O.advection((1.0,))], -1.0)
    # tf == t0 : zero steps, state untouched
    before = f.vals.copy()
    t, steps = O.integrate(f, O.RK3, [O.advection((1.0,))], 0.5, t0=0.5)
    assert steps == 0 and np.array_equal(before, f.vals)
    # dt_max caps the step
    t, steps = O.integrate(f, O.FE, [O.advection((1.0,))], 0.01, dt_max=0.001)
    assert steps in (10, 11)


def test_stage_api_equals_advance(O):
    """orc_stage x nstages == orc_advance, for all three integrators, two terms."""
    rng = np.random.default_rng(1)
    for integ in (O.FE, O.RK2, O.RK3):
        f = mk(O, lambda x, y: np.sqrt(x * x + y * y) - 0.5, (-1, -1), (1, 1), (24, 20), bc=O.NEUMANN)
        g = O.Field(f.vals.copy(order="F"), (-1, -1), (1, 1), bc=O.NEUMANN)
        u = np.asfortranarray(rng.standard_normal((2, 24, 20)))
        terms = [O.advection(u), O.curvature(-0.01)]
        O.advance(f, integ, terms, 0.0, 1e-3)
        b1, b2 = g.vals.copy(order="F"), g.vals.copy(order="F")
        for s in range(1, O.nstages(integ) + 1):
            O.stage(g, integ, s, b1, b2, terms, 0.0, 1e-3)
        assert np.array_equal(f.vals, g.vals)


# ---- test/test-velocityextension.jl:19-44 "Extend Along Normals" and :46-87 "Circle periodic extension" ----
def test_extend_along_normals_reference_tests(O):
    f = mk(O, lambda x, y: x + 0 * y, (-1.0, -1.0), (1.0, 1.0), (81, 61))
    X = f.nodes()
    d = min(f.meshsize(1), f.meshsize(2))
    frozen = np.asfortranarray(np.abs(f.vals) <= d)
    Fref = np.broadcast_to(np.sin(np.pi * X[1]), f.vals.shape)
    F = np.asfortranarray(np.where(frozen, Fref, 0.0))
    seed = F.copy()
    out = O.extend_along_normals(F, f, nb_iters=150, frozen=frozen, cfl=0.45)
    assert np.abs(out - Fref).max() < 0.08
    assert np.array_equal(out[frozen], seed[frozen])

    R = 0.55
    f = mk(O, lambda x, y: np.sqrt(x * x + y * y) - R, (-1.0, -1.0), (1.0, 1.0), (121, 121), bc=O.PERIODIC)
    X = f.nodes()
    d = f.meshsize(1)
    r = np.sqrt(X[0] ** 2 + X[1] ** 2)
    frozen = np.asfortranarray(np.abs(f.vals) <= 1.1 * d)
    v = np.asfortranarray(np.where(frozen, np.broadcast_to(X[1], r.shape) / np.maximum(r, np.finfo(float).eps), 0.0))
    seed = v.copy()
    out = O.extend_along_normals(v, f, nb_iters=100, frozen=frozen, cfl=0.45)
    assert np.array_equal(out[frozen], seed[frozen])
    vf = O.Field(out, (-1.0, -1.0), (1.0, 1.0), bc=O.PERIODIC)
    tot, cnt = 0.0, 0
    for i in range(1, 121):            # active_nodeindices of a periodic field: node n duplicates node 1
        for j in range(1, 121):
            if abs(f.vals[i - 1, j - 1]) <= 5.0 * d and not frozen[i - 1, j - 1]:
                gx, gy = f.deriv("D0", (i, j), 1), f.deriv("D0", (i, j), 2)
                nn = math.hypot(gx, gy)
                if nn == 0 or math.isnan(nn):
                    continue
                tot += abs(gx / nn * vf.deriv("D0", (i, j), 1) + gy / nn * vf.deriv("D0", (i, j), 2))
                cnt += 1
    assert cnt > 100 and tot / cnt < 0.12
    # default mask = |phi| <= interface_band * dx; nb_iters = 0 leaves F untouched
    F0 = np.asfortranarray(np.random.default_rng(0).standard_normal(f.vals.shape))
    assert np.array_equal(O.extend_along_normals(F0.copy(order="F"), f, nb_iters=0), F0)
    out = O.extend_along_normals(F0.copy(order="F"), f, nb_iters=3)
    band = np.abs(f.vals) <= 1.5 * d
    assert np.array_equal(out[band], F0[band]) and not np.array_equal(out[~band], F0[~band])


# ---- src/levelsetops.jl:253-325 : set operations, Julia min/max semantics ----
def test_csg_semantics(O):
    a = np.array([1.0, -2.0, 0.0, -0.0, np.nan, 3.0, 0.5])
    b = np.array([0.5, -1.0, -0.0, 0.0, 1.0, np.nan, 0.5])
    u, i, d, c = O.csg("union", a, b), O.csg("intersect", a, b), O.csg("setdiff", a, b), O.csg("complement", a)
    assert np.array_equal(u[[0, 1, 6]], [0.5, -2.0, 0.5]) and np.isnan(u[4]) and np.isnan(u[5])
    assert np.signbit(u[2]) and np.signbit(u[3])                 # min(0.0, -0.0) == -0.0 either way round
    assert np.array_equal(i[[0, 1, 6]], [1.0, -1.0, 0.5]) and not np.signbit(i[2]) and not np.signbit(i[3])
    assert np.array_equal(d[[0, 1, 6]], [1.0, 1.0, 0.5]) and np.isnan(d[4]) and np.isnan(d[5])
    assert np.array_equal(c[[0, 1, 6]], [-1.0, 2.0, -0.5]) and np.signbit(c[2]) and not np.signbit(c[3])
    # test/test-levelsetops.jl style identity: a \ b == a ∩ complement(b)
    assert np.array_equal(O.csg("setdiff", a[:4], b[:4]), O.csg("intersect", a[:4], O.csg("complement", b[:4])))


# ---- tests/golden/oracle_vectors.npz : the oracle pinned against its own committed outputs ----
def test_oracle_golden_vectors(O):
    """Regression pin: the oracle must keep reproducing the committed vectors of the five BASELINE configurations (small
    instances, f64 and f32; generated by tests/golden/make_oracle_vectors.py).  Same compiler flags -> equality; the
    tolerance only allows for a different libm (sin/cos in the input fields)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_oracle_vectors", os.path.join(GOLDEN, "make_oracle_vectors.py"))
    gen = importlib.util.module_from_spec(spec); spec.loader.exec_module(gen)
    gold = np.load(os.path.join(GOLDEN, "oracle_vectors.npz"))
    O.set_threads(4)
    for name in gen.CASES:
        for dtype, tag in ((np.float64, "f64"), (np.float32, "f32")):
            v, tf, n = gen.run(name, dtype)
            g = gold[f"{name}_{tag}"]
            assert g.dtype == v.dtype and g.shape == v.shape
            assert gold[f"{name}_{tag}_tf_steps"][1] == n
            assert np.abs(v.astype(np.float64) - g.astype(np.float64)).max() <= (1e-13 if dtype == np.float64 else 1e-6), (name, tag)
    # the periodic wrap pairs of the reference (boundaryconditions.jl:107-119)
    k = KNOWN["periodic_wrap"]
    f = O.Field(np.arange(1.0, k["n"] + 1), (0,), (1,), bc=O.PERIODIC)
    for i, j in k["pairs"]:
        assert f[i] == float(j)
