"""GPU parity tests proper: every call goes through the C ABI (liblsm_b200.so) and is compared with
the CPU oracle on the same seed-free inputs.  Tolerances are the ones BASELINE.json states:
max-abs phi difference <= 1e-10 (Float64) / <= 1e-4 (Float32) after 100 RK3 steps, identical sign and
cut-cell classification.  The strict generic kernel is additionally required to match the oracle to
rounding level (<= 1e-13 relative) on every term / BC / dimension / dtype combination.
"""
import math
import os

import numpy as np
import pytest

import helpers as H

pytestmark = pytest.mark.gpu

OPT_KERNEL = 0


@pytest.fixture(scope="module")
def m():
    import lsm_b200
    return lsm_b200


@pytest.fixture()
def strict(m):
    ctx = m.default_context()
    ctx.set_option(OPT_KERNEL, 1)
    yield ctx
    ctx.set_option(OPT_KERNEL, 0)


# ------------------------------------------------------------------------------------------------
# ghost cells on the device (test/test-meshfield.jl:44-125) against the oracle
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_device_getindex_matches_oracle(m, O, dtype):
    rng = np.random.default_rng(0)
    bcs = [("periodic",), ("neumann",), ("extrap", 1), ("extrap", 2), ("extrap", 3), ("symmetry",)]
    for n in [(12,), (10, 7), (8, 6, 7)]:
        N = len(n)
        vals = rng.standard_normal(n).astype(dtype)
        for i, b in enumerate(bcs):
            bc = tuple(bcs[(i + d) % len(bcs)] if d else b for d in range(N))      # mix kinds across dims
            case = H.Case("g", [0.0] * N, [1.0] * N, n, vals, [], bc, dtype)
            fo = case.oracle_field()
            phi = case.engine_field(m)
            for _ in range(40):
                I = tuple(int(rng.integers(-2, n[d] + 4)) for d in range(N))      # 1-based, up to 3 outside
                assert phi[I] == fo[I], (n, bc, I)


def test_device_getindex_reference_cases(m):
    g = m.CartesianGrid((0, 0), (1, 1), (10, 5))
    vals = np.random.default_rng(1).random((10, 5))
    mf = m.MeshField(vals, g, bc=(m.PeriodicBC(), m.PeriodicBC()))
    assert mf[1, 1] == vals[0, 0] and mf[1, 0] == vals[0, 3] and mf[11, 5] == mf[2, 5]
    g1 = m.CartesianGrid((0.0,), (4.0,), (5,))
    s = m.MeshField(lambda x: x[0], g1, bc=m.SymmetryBC())
    assert (s[0], s[-1], s[6], s[7]) == (1.0, 2.0, 3.0, 2.0)
    nb = m.MeshField(lambda x: x[0], g1)
    with pytest.raises(m.BCError):
        nb[0]                                     # meshfield.jl:222-232: no BC to resolve a ghost
    a, b, n = -0.3, 1.7, 10
    h = (b - a) / (n - 1)
    for P in range(0, 6):
        for k in range(0, P + 1):
            f = m.MeshField(lambda x: x[0] ** k, m.CartesianGrid((a,), (b,), (n,)), bc=m.ExtrapolationBC(P))
            for j in range(1, P + 2):
                assert f[1 - j] == pytest.approx((a - j * h) ** k, abs=1e-10)
                assert f[n + j] == pytest.approx((b + j * h) ** k, abs=1e-10)


# ------------------------------------------------------------------------------------------------
# CFL (test/test-levelsetterms.jl:7-31) : bit-exact against the oracle
# ------------------------------------------------------------------------------------------------
def test_cfl_bitexact_and_errors(m, O):
    for case in (H.c1_circle_rotation(64), H.c3_enright(24), H.c5_normal_advection(24), H.c2_zalesak_curvature(64),
                 H.c3_enright(24, separable=True), H.c1_circle_rotation(48, np.float32)):
        fo, to = case.oracle_field(), case.oracle_terms()
        phi = case.engine_field(m)
        terms = case.engine_terms(m, phi)
        for t in (0.0, 0.37, 1.4):
            assert m.compute_cfl(terms, phi, t) == O.compute_cfl(fo, to, t), case.name
    g = m.CartesianGrid((-1.0,), (1.0,), (100,))
    phi = m.MeshField(lambda x: x[0], g, bc=m.NeumannBC())
    dx = g.meshsize(1)
    assert m.compute_cfl((m.AdvectionTerm(lambda x, t: (2.0,)),), phi, 0.0) == pytest.approx(dx / 2.0, rel=1e-15)
    assert m.compute_cfl((m.NormalMotionTerm(lambda x, t: 3.0),), phi, 0.0) == pytest.approx(dx / 3.0, rel=1e-15)
    assert m.compute_cfl((m.AdvectionTerm((0.0,)),), phi, 0.0) == math.inf
    u = np.ones((1, 100)); u[0, 17] = np.nan
    with pytest.raises(m.CFLError):
        m.compute_cfl((m.AdvectionTerm(m.MeshField(u, g)),), phi, 0.0)
    u[0, 17] = np.inf
    with pytest.raises(m.CFLError):
        m.compute_cfl((m.AdvectionTerm(m.MeshField(u, g)),), phi, 0.0)


# ------------------------------------------------------------------------------------------------
# strict kernel: every term x BC x dim x dtype x integrator, a few steps, rounding-level agreement
# ------------------------------------------------------------------------------------------------
def _small_cases():
    return [c for n in ((40,), (26, 22), (14, 12, 13)) for c in H.small_cases(n)]


@pytest.mark.parametrize("name,case", _small_cases(), ids=[c[0] for c in _small_cases()])
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_strict_kernel_all_terms(m, O, strict, name, case, dtype):
    case = H.Case(case.name, case.lc, case.hc, case.n, case.phi0, case.terms, case.bc, dtype)
    for integ in ("FE", "RK2", "RK3"):
        a, b, _, n = H.run_pair(m, O, case, integ=integ, steps=4)
        assert n == 4 or "cos" in name
        tol = 1e-13 if dtype == np.float64 else 2e-6
        d = np.abs(a.astype(np.float64) - b.astype(np.float64)).max()
        assert d <= tol * max(1.0, np.abs(a).max()), (name, integ, d)


@pytest.mark.parametrize("name,case", [c for c in _small_cases() if not c[0].startswith("1d")],
                         ids=[c[0] for c in _small_cases() if not c[0].startswith("1d")])
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_tiled_kernel_all_terms(m, O, name, case, dtype):
    """The same matrix through the default kernel selection, i.e. the tiled kernels (2-D and 3-D): every term, every BC
    kind (index-remap and polynomial-extrapolation instantiations), all three integrators.  The grids are small: 26 x 22 is
    one tile in x and two in y, 14 x 12 x 13 one tile and one z chunk, so every tile is partial and resolves its ghosts;
    none takes the plain-copy or TMA fill.  Grids of many tiles are in test_tiled_multitile.py.  Tolerance = the BASELINE
    bar (1e-10 / 1e-4), far above what 8 steps accumulate."""
    case = H.Case(case.name, case.lc, case.hc, case.n, case.phi0, case.terms, case.bc, dtype)
    for integ in ("FE", "RK2", "RK3"):
        a, b, _, n = H.run_pair(m, O, case, integ=integ, steps=8)
        tol = 1e-10 if dtype == np.float64 else 1e-4
        d = np.abs(a.astype(np.float64) - b.astype(np.float64)).max()
        assert not np.isnan(b).any() and d <= tol * max(1.0, np.abs(a).max()), (name, integ, d)


# ------------------------------------------------------------------------------------------------
# BASELINE.json configs, 100 RK3 steps, default kernel selection (tiled where available)
# ------------------------------------------------------------------------------------------------
CONFIGS = [
    ("C1-128", lambda dt: H.c1_circle_rotation(128, dt)),
    ("C2-192", lambda dt: H.c2_zalesak_curvature(192, dt)),
    ("C3-48", lambda dt: H.c3_enright(48, dt)),
    ("C3sep-48", lambda dt: H.c3_enright(48, dt, separable=True)),
    ("C4-48", lambda dt: H.c4_eikonal(48, dt)),
    ("C5-48", lambda dt: H.c5_normal_advection(48, dt)),
]


@pytest.mark.parametrize("name,mk", CONFIGS, ids=[c[0] for c in CONFIGS])
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_config_parity_100_steps(m, O, name, mk, dtype):
    case = mk(dtype)
    steps = 50 if name.startswith("C4") else 100
    a, b, t, n = H.run_pair(m, O, case, integ="RK3", steps=steps)
    assert n >= 0.9 * steps
    d = H.check_parity(a, b, 1e-10 if dtype == np.float64 else 1e-4)
    print(f"{name} {np.dtype(dtype).name}: {n} steps, max-abs diff {d:.3e}")


# SURVEY.md §8(d) sizes: 128^3 (3-D) / 512^2 (2-D), 100 RK3 steps (C4: 50).  At these sizes interior tiles take the TMA ring
# path of every kernel family, z marching spans several chunks per block column and the 3-blocks/SM instantiations are resident,
# so the production kernels are compared with the oracle DIRECTLY (not through the strict kernel).  The observed max-abs
# difference is printed for each case (-s / -rP shows it; profiles/parity_rNN.txt keeps a copy).
CONFIGS_BIG = [
    ("C2-512", lambda dt: H.c2_zalesak_curvature(512, dt)),
    ("C3-128", lambda dt: H.c3_enright(128, dt)),
    ("C3sep-128", lambda dt: H.c3_enright(128, dt, separable=True)),
    ("C4-128", lambda dt: H.c4_eikonal(128, dt)),
    ("C5-128", lambda dt: H.c5_normal_advection(128, dt)),
]


@pytest.mark.parametrize("name,mk", CONFIGS_BIG, ids=[c[0] for c in CONFIGS_BIG])
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_config_parity_survey_sizes(m, O, name, mk, dtype):
    case = mk(dtype)
    steps = 50 if name.startswith("C4") else 100
    O.set_threads(O.max_threads())
    a, b, t, n = H.run_pair(m, O, case, integ="RK3", steps=steps)
    assert n >= 0.9 * steps
    d = H.check_parity(a, b, 1e-10 if dtype == np.float64 else 1e-4)
    print(f"PARITY {name} {np.dtype(dtype).name}: {n} steps, max-abs diff {d:.3e} (bar {'1e-10' if dtype == np.float64 else '1e-4'})")


def _pair_case(n, bc, dtype, separable):
    lc, hc = (0, 0, 0), (1, 1, 1)
    x, y, z = H.coords(lc, hc, n)
    phi = np.sqrt((x - 0.35) ** 2 + (y - 0.4) ** 2 + (z - 0.45) ** 2) - 0.15 + 0.02 * np.sin(9 * x) * np.cos(7 * y) * np.sin(5 * z)
    sc, tabs = H.enright_tables(lc, hc, n)
    tabs = [[t + 0.05 * (a + 1) for a, t in enumerate(row)] for row in tabs]       # sign changes in every direction, no exact zeros
    if separable:
        term = dict(kind="advection", separable=(sc, tabs), cos_period=3.0)
    else:
        X, Y, Z = np.meshgrid(*[np.arange(k) for k in n], indexing="ij", sparse=True)
        u = np.stack([((sc[d] * tabs[d][0][X]) * tabs[d][1][Y]) * tabs[d][2][Z] for d in range(3)], axis=0)
        term = dict(kind="advection", field=u, cos_period=3.0)
    return H.Case("P", lc, hc, n, phi, [term], bc, dtype)


PAIR_SHAPES = [(128, 64, 40), (72, 52, 37), (64, 8, 8), (200, 30, 70), (136, 9, 130)]
PAIR_BCS = [("neumann",), ("periodic",), ("symmetry",),
            ((("neumann",), ("symmetry",)), ("periodic",), (("symmetry",), ("neumann",)))]


@pytest.mark.parametrize("n", PAIR_SHAPES, ids=["x".join(map(str, s)) for s in PAIR_SHAPES])
def test_pair_kernel_bitwise_vs_tiled(m, n):
    """The x-pair kernel (csrc/lsm_pair3d.cu: TMA for every tile, lazy ghost fix-up, direction branches, shared differences)
    performs the same operations as the general tiled kernel when it is run with the exact epsilon maximum (LSM_OPT_KERNEL = 4;
    anisotropic mesh sizes, so the per-dimension scaling is not folded), so kernels 4 and 3 must give BIT-IDENTICAL states:
    partial tiles on every side, every index-map BC (also mixed per side), FE / RK2 / RK3, stored and separable velocity,
    sign changes of the velocity inside warps and pairs, both dtypes.  The default mode (20-bit epsilon maximum) must stay at
    rounding level of it."""
    ctx = m.default_context()
    k = 0
    for bc in PAIR_BCS:
        for dtype in (np.float64, np.float32):
            if dtype == np.float32 and n[0] % 4:
                continue
            k += 1
            case = _pair_case(n, bc, dtype, separable=(k % 3 == 0))
            integ = (m.RK3, m.RK2, m.ForwardEuler)[k % 3]
            outs = []
            for kernel in (4, 3, 0):
                ctx.set_option(OPT_KERNEL, kernel)
                ctx.reset_counters()
                phi = case.engine_field(m)
                eq = m.LevelSetEquation(terms=case.engine_terms(m, phi), ic=phi, integrator=integ())
                dt = 0.5 * m.compute_cfl(eq.terms, eq.state, 0.0)
                m.integrate(eq, 3 * dt * (1 - 1e-12))
                outs.append((eq.t, eq.steps_taken, eq.state.peek().copy(), ctx.counters()["pair_launches"]))
            ctx.set_option(OPT_KERNEL, 0)
            assert outs[0][3] > 0 and outs[1][3] == 0 and outs[2][3] > 0, "kernel selection"
            assert outs[0][:2] == outs[1][:2] == outs[2][:2]
            assert np.array_equal(outs[0][2], outs[1][2]), (n, bc, np.dtype(dtype).name, float(np.abs(outs[0][2] - outs[1][2]).max()))
            tol = 1e-12 if dtype == np.float64 else 0.0
            assert np.abs(outs[2][2].astype(np.float64) - outs[1][2].astype(np.float64)).max() <= tol


@pytest.mark.parametrize("n", [(128, 64, 40), (72, 52, 37), (48, 48, 48)], ids=["128x64x40", "72x52x37", "48cube"])
def test_pair_kernel_two_terms_vs_tiled(m, n):
    """BASELINE config 5's term list (NormalMotionTerm(stored speed), AdvectionTerm(stored velocity)) through the x-pair kernel,
    which shares the first / second differences between the ENO2 Godunov norm and WENO5 (the general tiled kernel forms
    phi+ - 2 phi0 + phi- directly): same result up to rounding.  Speed with sign changes, every index-map BC, the three
    integrators, anisotropic and isotropic meshes."""
    ctx = m.default_context()
    lc, hc = (0, 0, 0), (1, 1, 1)
    x, y, z = H.coords(lc, hc, n)
    phi = np.sqrt((x - 0.45) ** 2 + (y - 0.5) ** 2 + (z - 0.55) ** 2) - 0.25 + 0.03 * np.sin(7 * x) * np.cos(5 * y) * np.sin(6 * z)
    v = H.bcast(0.2 * np.sin(4 * x + 1) * np.cos(3 * y) + 0.1 * z - 0.05, n)
    sc, tabs = H.enright_tables(lc, hc, n)
    tabs = [[t + 0.05 * (a + 1) for a, t in enumerate(row)] for row in tabs]
    X, Y, Z = np.meshgrid(*[np.arange(k) for k in n], indexing="ij", sparse=True)
    u = np.stack([((sc[d] * tabs[d][0][X]) * tabs[d][1][Y]) * tabs[d][2][Z] for d in range(3)], axis=0)
    for k, bc in enumerate(PAIR_BCS):
        case = H.Case("P5", lc, hc, n, phi, [dict(kind="normal", field=v), dict(kind="advection", field=u)], bc, np.float64)
        integ = (m.RK3, m.RK2, m.ForwardEuler)[k % 3]
        outs = []
        for kernel in (4, 0, 3):
            ctx.set_option(OPT_KERNEL, kernel)
            ctx.reset_counters()
            f = case.engine_field(m)
            eq = m.LevelSetEquation(terms=case.engine_terms(m, f), ic=f, integrator=integ())
            dt = 0.5 * m.compute_cfl(eq.terms, eq.state, 0.0)
            m.integrate(eq, 4 * dt * (1 - 1e-12))
            outs.append((eq.t, eq.steps_taken, eq.state.peek().copy(), ctx.counters()["pair_launches"]))
        ctx.set_option(OPT_KERNEL, 0)
        assert outs[0][3] > 0 and outs[1][3] > 0 and outs[2][3] == 0, "kernel selection"
        assert outs[0][:2] == outs[1][:2] == outs[2][:2]
        for o in outs[:2]:
            d = np.abs(o[2] - outs[2][2]).max()
            assert d <= 1e-12, (n, bc, integ.__name__, d)


@pytest.mark.parametrize("n", [(256, 96), (520, 70), (40, 33), (1032, 24)], ids=["256x96", "520x70", "40x33", "1032x24"])
def test_pair2d_kernel_vs_tiled(m, n):
    """The 2-D x-pair kernel (csrc/lsm_pair2d.cu: strips marching along y on a TMA row ring, lazy x-ghost fix-up two rows ahead
    for the curvature corners) against the general tiled 2-D kernel (LSM_OPT_KERNEL = 3): advection alone (C1's term list) and
    advection + constant-b curvature (C2's), every index-map BC, FE / RK2 / RK3, both dtypes, partial strips, sign changes of
    the velocity.  Same operations, so the states must agree to rounding level (bit-identical in practice)."""
    ctx = m.default_context()
    lc, hc = (-1.0, -1.0), (1.0, 1.0)
    x, y = H.coords(lc, hc, n)
    phi = np.hypot(x - 0.1, y + 0.05) - 0.45 + 0.03 * np.sin(9 * x) * np.cos(7 * y)
    phi = np.maximum(phi, -(np.maximum(np.abs(x - 0.1) - 0.08, np.abs(y + 0.4) - 0.3)))        # a notch: kinks for the curvature term
    u = np.stack([H.bcast(-y + 0.2 * np.sin(5 * x), n), H.bcast(x + 0.1 * np.cos(4 * y), n)], axis=0)
    bcs = [("neumann",), ("periodic",), ("symmetry",), ((("neumann",), ("symmetry",)), ("periodic",))]
    k = 0
    for bc in bcs:
        for dtype in (np.float64, np.float32):
            if dtype == np.float32 and n[0] % 4:
                continue
            for curv in (False, True):
                k += 1
                terms = [dict(kind="advection", field=u)] + ([dict(kind="curvature", const=-0.01)] if curv else [])
                case = H.Case("P2", lc, hc, n, phi, terms, bc, dtype)
                integ = (m.RK3, m.RK2, m.ForwardEuler)[k % 3]
                outs = []
                for kernel in (2, 3):                      # 2: x-pair kernel forced (also below its size threshold), 3: tiled only
                    ctx.set_option(OPT_KERNEL, kernel)
                    ctx.reset_counters()
                    f = case.engine_field(m)
                    eq = m.LevelSetEquation(terms=case.engine_terms(m, f), ic=f, integrator=integ())
                    dt = 0.5 * m.compute_cfl(eq.terms, eq.state, 0.0)
                    m.integrate(eq, 4 * dt * (1 - 1e-12))
                    outs.append((eq.t, eq.steps_taken, eq.state.peek().copy(), ctx.counters()["pair_launches"]))
                ctx.set_option(OPT_KERNEL, 0)
                assert outs[0][3] > 0 and outs[1][3] == 0, "kernel selection"
                assert outs[0][:2] == outs[1][:2]
                d = np.abs(outs[0][2].astype(np.float64) - outs[1][2].astype(np.float64)).max()
                assert d <= (1e-13 if dtype == np.float64 else 1e-6), (n, bc, np.dtype(dtype).name, curv, integ.__name__, d)


@pytest.mark.parametrize("n", [(128, 128), (40, 48), (130, 49), (33, 70), (170, 170), (8, 300)], ids=["128x128", "40x48", "130x49", "33x70", "170x170", "8x300"])
def test_resident_kernel_bitwise_vs_tiled(m, n):
    """Small 2-D grids run the WHOLE time loop in one cluster kernel (csrc/lsm_resident2d.cu: state, stage buffers and velocity in
    the distributed shared memory of 16 CTAs, every result pushed into the ghost columns / the neighbouring CTAs' halo rows that
    mirror it, the dt sequence replayed on the host).  Same arithmetic as the tiled 2-D kernel (LSM_OPT_KERNEL = 3), so time,
    step count and state must be BIT-IDENTICAL: every index-map BC, FE / RK2 / RK3, both dtypes, strips of exactly 3 rows
    (40x48), uneven strips (130x49: 4 rows and 3 rows), 2 and 4 nodes per thread, a final step shorter than the others (two
    dt runs), sign changes of the velocity."""
    ctx = m.default_context()
    lc, hc = (-1.0, -1.0), (1.0, 1.0)
    x, y = H.coords(lc, hc, n)
    phi = np.hypot(x - 0.1, y + 0.05) - 0.45 + 0.03 * np.sin(9 * x) * np.cos(7 * y)
    u = np.stack([H.bcast(-y + 0.2 * np.sin(5 * x), n), H.bcast(x + 0.1 * np.cos(4 * y), n)], axis=0)
    bcs = [("periodic",), ("neumann",), ("symmetry",), ((("neumann",), ("symmetry",)), ("periodic",)),
           (("periodic",), (("symmetry",), ("neumann",)))]
    k = 0
    for bc in bcs:
        for dtype in (np.float64, np.float32):
            k += 1
            case = H.Case("R2", lc, hc, n, phi, [dict(kind="advection", field=u)], bc, dtype)
            integ = (m.RK3, m.RK2, m.ForwardEuler)[k % 3]
            outs = []
            for kernel in (0, 3):                      # 0: automatic selection (resident kernel), 3: tiled per-stage kernels
                ctx.set_option(OPT_KERNEL, kernel)
                ctx.reset_counters()
                f = case.engine_field(m)
                eq = m.LevelSetEquation(terms=case.engine_terms(m, f), ic=f, integrator=integ())
                dt = 0.5 * m.compute_cfl(eq.terms, eq.state, 0.0)
                m.integrate(eq, 6.4 * dt)
                n1 = eq.steps_taken
                m.integrate(eq, 9.0 * dt)                # a second call starts from the state the first one left on the device
                c = ctx.counters()
                outs.append((eq.t, (n1, eq.steps_taken), eq.state.peek().copy(), c["resident_steps"], c["stage_launches"]))
            ctx.set_option(OPT_KERNEL, 0)
            assert outs[0][3] == sum(outs[0][1]) >= 9 and outs[0][4] == 0 and outs[1][3] == 0, ("kernel selection", outs[0][3:], outs[1][3:])
            assert outs[0][:2] == outs[1][:2], (outs[0][:2], outs[1][:2])
            assert np.array_equal(outs[0][2], outs[1][2]), (n, bc, np.dtype(dtype).name, integ.__name__,
                                                            np.abs(outs[0][2].astype(np.float64) - outs[1][2].astype(np.float64)).max())


def test_resident_kernel_c1_long_run(m):
    """BASELINE configs[0] (128^2 circle rotation, periodic, Float64 RK3) for 300 steps through the resident cluster kernel against
    the per-stage tiled kernels (bit-identical) — and the options that must switch it off do."""
    ctx = m.default_context()
    case = H.c1_circle_rotation(128)
    outs = []
    for kernel, resident in ((0, 1), (3, 1), (0, 0)):
        ctx.set_option(OPT_KERNEL, kernel)
        ctx.set_option(m._lib.OPT_RESIDENT, resident)
        ctx.reset_counters()
        f = case.engine_field(m)
        eq = m.LevelSetEquation(terms=case.engine_terms(m, f), ic=f, integrator=m.RK3())
        dt = 0.5 * m.compute_cfl(eq.terms, eq.state, 0.0)
        m.integrate(eq, 300 * dt * (1 - 1e-12))
        outs.append((eq.t, eq.steps_taken, eq.state.peek().copy(), ctx.counters()["resident_steps"]))
    ctx.set_option(OPT_KERNEL, 0)
    ctx.set_option(m._lib.OPT_RESIDENT, 1)
    assert outs[0][3] == 300 and outs[1][3] == 0 and outs[2][3] == 0
    for o in outs[1:]:
        assert o[:2] == outs[0][:2] and np.array_equal(o[2], outs[0][2])


@pytest.mark.parametrize("n", [(128, 64, 40), (72, 52, 37), (64, 8, 8)], ids=["128x64x40", "72x52x37", "64x8x8"])
def test_pair_kernel_eikonal_bitwise_vs_tiled(m, n):
    """BASELINE config 4's term (EikonalReinitializationTerm with a frozen stored S0) through the x-pair kernel: the same
    operations as the general tiled kernel (direct second differences), so the states must be BIT-IDENTICAL — partial tiles,
    every index-map BC, FE / RK2 / RK3."""
    ctx = m.default_context()
    lc, hc = (-1, -1, -1), (1, 1, 1)
    x, y, z = H.coords(lc, hc, n)
    r = np.sqrt(x * x + y * y + z * z)
    phi = (r - 0.5) * (1 + 0.4 * np.sin(3 * np.pi * x) * np.sin(3 * np.pi * y) * np.sin(3 * np.pi * z))
    for k, bc in enumerate(PAIR_BCS):
        case = H.Case("P4", lc, hc, n, phi, [dict(kind="eikonal", frozen=True)], bc, np.float64)
        integ = (m.RK3, m.RK2, m.ForwardEuler)[k % 3]
        outs = []
        for kernel in (0, 3):
            ctx.set_option(OPT_KERNEL, kernel)
            ctx.reset_counters()
            f = case.engine_field(m)
            eq = m.LevelSetEquation(terms=case.engine_terms(m, f), ic=f, integrator=integ())
            dt = 0.5 * m.compute_cfl(eq.terms, eq.state, 0.0)
            m.integrate(eq, 5 * dt * (1 - 1e-12))
            outs.append((eq.t, eq.steps_taken, eq.state.peek().copy(), ctx.counters()["pair_launches"]))
        ctx.set_option(OPT_KERNEL, 0)
        assert outs[0][3] > 0 and outs[1][3] == 0, "kernel selection"
        assert outs[0][:2] == outs[1][:2]
        assert np.array_equal(outs[0][2], outs[1][2]), (n, bc, integ.__name__, float(np.abs(outs[0][2] - outs[1][2]).max()))


def _notched_sphere_case(n, dtype=np.float64):
    """3-D Zalesak-type body (sphere with a slot: kinks along the slot edges) in the Enright velocity: the sharp-feature
    counterpart of C3 for the x-pair kernel."""
    case = H.c3_enright(n, dtype)
    x, y, z = H.coords(case.lc, case.hc, case.n)
    sphere = np.sqrt((x - 0.5) ** 2 + (y - 0.6) ** 2 + (z - 0.5) ** 2) - 0.25
    slot = np.maximum(np.abs(x - 0.5) - 0.05, np.abs(y - 0.5) - 0.25) + 0 * z
    case.phi0 = np.asfortranarray(np.maximum(sphere, -slot).astype(dtype))
    return case


def test_pair_kernel_kinked_body_parity(m, O):
    """Default kernels on non-smooth data, 96^3 cube (isotropic mesh: folded scaling + 20-bit epsilon maximum), 100 RK3 steps
    against the oracle: the BASELINE bar with the observed value printed."""
    O.set_threads(O.max_threads())
    a, b, t, n = H.run_pair(m, O, _notched_sphere_case(96), integ="RK3", steps=100)
    d = H.check_parity(a, b, 1e-10)
    print(f"PARITY notched-sphere-96 float64: {n} steps, max-abs diff {d:.3e} (bar 1e-10)")
    assert d <= 2e-11


def test_cfl_candidates_are_exact(m, O):
    """Time-scaled static coefficients: from the third CFL request on, the maximum is evaluated on the HOST over the candidate
    nodes (lsm_api.cu, CflMemo) — no reduction pass, no D2H, no sync per step.  It must be bit-identical to the full reduction
    (LSM_OPT_CFL_CANDIDATES = 0) for every scale: stored and separable velocity, both dtypes, a scalar speed, a field of ties
    (constant velocity stored as a field: the candidate list overflows and the full pass answers), and whole integrations
    must take the same steps and produce the same bits."""
    OPT_CAND = 6
    ctx = m.default_context()
    cases = [H.c3_enright(40), H.c3_enright(40, separable=True), H.c3_enright(32, np.float32), H.c1_circle_rotation(96)]
    cases[3].terms[0]["cos_period"] = 2.0
    flat = H.c3_enright(24)
    flat.terms[0]["field"] = np.broadcast_to(np.array([0.3, -0.2, 0.1]).reshape(3, 1, 1, 1), (3, 24, 24, 24)).copy()
    cases.append(flat)
    ts = [0.0, 0.11, 0.37, 0.9, 1.4, 1.5 - 1e-9, 2.2, 2.9]
    for case in cases:
        fo, to = case.oracle_field(), case.oracle_terms()
        phi = case.engine_field(m)
        terms = case.engine_terms(m, phi)
        ctx.reset_counters()
        got = [m.compute_cfl(terms, phi, t) for t in ts]
        passes = ctx.counters()["cfl_passes"]
        assert got == [O.compute_cfl(fo, to, t) for t in ts], case.name
        if case is not flat:
            assert passes <= 2, (case.name, passes)                    # first request + the unscaled maximum of the build
    # normal motion with a time-scaled stored speed (host g(t)): |fl(v g)| is monotone in |v|
    g = m.CartesianGrid((-1, -1), (1, 1), (80, 64))
    X, Y = g.coords()
    v = np.asfortranarray(0.3 + 0.2 * np.sin(3 * X) * np.cos(2 * Y))
    phi = m.MeshField(np.asfortranarray(np.hypot(X, Y) - 0.5), g, bc=m.NeumannBC())
    term = m.NormalMotionTerm(m.TimeScaled(m.MeshField(v, g), lambda t: math.cos(t) - 0.2))
    ref = []
    for opt in (0, 1):
        ctx.set_option(OPT_CAND, opt)
        ref.append([m.compute_cfl((term,), phi, t) for t in ts])
    assert ref[0] == ref[1]
    # whole integrations: identical step counts, times and states with and without candidates
    for case in (H.c3_enright(40), H.c3_enright(40, separable=True)):
        outs = []
        for cand in (1, 0):
            ctx.set_option(OPT_CAND, cand)
            phi = case.engine_field(m)
            eq = m.LevelSetEquation(terms=case.engine_terms(m, phi), ic=phi, integrator=m.RK3())
            ctx.reset_counters()
            m.integrate(eq, 0.25)
            outs.append((eq.t, eq.steps_taken, eq.state.peek().copy(), ctx.counters()))
        ctx.set_option(OPT_CAND, 1)
        assert outs[0][1] > 12
        for o in outs[1:]:
            assert o[:2] == outs[0][:2] and np.array_equal(o[2], outs[0][2])
        assert outs[0][3]["d2h_bytes"] < outs[1][3]["d2h_bytes"]       # no 8-byte readback per step any more


def test_device_generated_fields_match_numpy(m):
    """lsm_field_fill_shape / lsm_field_fill_separable (MeshField(f, grid) for analytic f, meshfield.jl:208-211, evaluated on the
    device) against the NumPy construction tests/helpers.py uses for the BASELINE configurations: bit for bit, both dtypes,
    2-D and 3-D; the Zalesak disk of docs/src/example-zalesak.md:21-40 is assembled with the device set operations."""
    for dtype in (np.float64, np.float32):
        c3 = H.c3_enright(40, dtype)
        g3 = c3.engine_grid(m)
        sph = m.MeshField.from_shape(g3, "sphere", (0.35, 0.35, 0.35, 0.15), bc=m.NeumannBC(), dtype=dtype)
        assert np.array_equal(sph.peek(), c3.phi0)
        sc, tabs = H.enright_tables(c3.lc, c3.hc, c3.n)
        vel = m.MeshField.from_separable(m.SeparableVelocity(g3, sc, tabs), dtype=dtype)
        assert np.array_equal(vel.peek(), c3.terms[0]["field"].astype(dtype))
        c5 = H.c5_normal_advection(24, dtype)
        g5 = c5.engine_grid(m)
        x, y, z = [c.ravel() for c in H.coords(c5.lc, c5.hc, c5.n)]
        one = [np.ones_like(x), np.ones_like(y), np.ones_like(z)]
        rot = m.SeparableVelocity(g5, (-1.0, 1.0, 0.0), [[one[0], y, one[2]], [x, one[1], one[2]], one])
        assert np.array_equal(m.MeshField.from_separable(rot, dtype=dtype).peek(), c5.terms[1]["field"].astype(dtype))
        assert np.array_equal(m.MeshField.from_shape(g5, "sphere", (0.3, 0.0, 0.0, 0.4), dtype=dtype).peek(), c5.phi0)
        assert np.array_equal(m.MeshField.from_shape(g5, "const", (0.2,), dtype=dtype).peek(), c5.terms[0]["field"].astype(dtype))
        cv = m.MeshField.from_shape(g5, "const", (0.5, -1.5, 2.0), dtype=dtype).peek()
        assert cv.shape == (3, 24, 24, 24) and np.all(cv[0] == dtype(0.5)) and np.all(cv[1] == dtype(-1.5)) and np.all(cv[2] == dtype(2.0))
        # 2-D: Zalesak = setdiff(disk, rec) with the reference's rectangle formula
        c2 = H.c2_zalesak_curvature(96, dtype)
        g2 = c2.engine_grid(m)
        X, Y = H.coords(c2.lc, c2.hc, c2.n)
        disk = m.MeshField.from_shape(g2, "sphere", (-0.75, 0.0, 0.5), bc=m.NeumannBC(), dtype=dtype)
        assert np.array_equal(disk.peek(), (np.sqrt((X + 0.75) ** 2 + (Y - 0.0) ** 2) - 0.5).astype(dtype))
        rec = m.MeshField.from_shape(g2, "box", (-0.75, -0.5, 0.2, 1.0), dtype=dtype)
        rec_np = np.maximum(np.abs(X + 0.75) - 0.2 / 2, np.abs(Y + 0.5) - 1.0 / 2)
        assert np.array_equal(rec.peek(), rec_np.astype(dtype))
        zal = m.setdiff(disk, rec)
        assert np.array_equal(zal.peek(), np.maximum(disk.peek(), -rec.peek()))
        pl = m.MeshField.from_shape(g2, "plane", (0.6, -0.8, 0.1), dtype=dtype)
        assert np.array_equal(pl.peek(), ((0.6 * X + -0.8 * Y) - 0.1).astype(dtype))
    with pytest.raises(m.LSMError):
        m.MeshField.from_shape(g2, "sphere", (0.0, 0.0), dtype=np.float64)          # wrong parameter count
    # a device-generated state integrates like an uploaded one (no host array is ever created for it)
    case = H.c3_enright(40)
    g = case.engine_grid(m)
    outs = []
    for dev in (False, True):
        phi = m.MeshField.from_shape(g, "sphere", (0.35, 0.35, 0.35, 0.15), bc=m.NeumannBC()) if dev else case.engine_field(m)
        sc, tabs = H.enright_tables(case.lc, case.hc, case.n)
        vel = m.MeshField.from_separable(m.SeparableVelocity(g, sc, tabs)) if dev else m.MeshField(case.terms[0]["field"], g)
        eq = m.LevelSetEquation(terms=(m.AdvectionTerm(m.TimeScaled(vel, ("cos", 3.0)), m.WENO5()),), ic=phi, integrator=m.RK3())
        if dev:
            assert vel._vals is None
        m.integrate(eq, 0.05)
        outs.append((eq.t, eq.steps_taken, eq.state.peek().copy()))
    assert outs[0][:2] == outs[1][:2] and np.array_equal(outs[0][2], outs[1][2])


def test_against_committed_vectors(m):
    """The engine against tests/golden/oracle_vectors.npz (committed oracle outputs for small instances of C1..C5, f64 and
    f32): catches a change that moves the oracle and the engine together."""
    import importlib.util
    gdir = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    spec = importlib.util.spec_from_file_location("make_oracle_vectors", os.path.join(gdir, "make_oracle_vectors.py"))
    gen = importlib.util.module_from_spec(spec); spec.loader.exec_module(gen)
    gold = np.load(os.path.join(gdir, "oracle_vectors.npz"))
    for name, (mk, integ, steps) in gen.CASES.items():
        for dtype, tag in ((np.float64, "f64"), (np.float32, "f32")):
            case = mk(dtype)
            tf, n = gold[f"{name}_{tag}_tf_steps"]
            phi = case.engine_field(m)
            eq = m.LevelSetEquation(terms=case.engine_terms(m, phi), ic=phi, integrator={"RK2": m.RK2, "RK3": m.RK3}[integ]())
            m.integrate(eq, float(tf))
            assert eq.steps_taken == int(n), (name, tag)
            H.check_parity(gold[f"{name}_{tag}"], eq.state.peek(), 1e-10 if dtype == np.float64 else 1e-4)


def test_c4_rk2_reference_default(m, O):
    a, b, _, n = H.run_pair(m, O, H.c4_eikonal(40), integ="RK2", steps=50)
    H.check_parity(a, b, 1e-10)


def test_strict_and_default_kernels_agree(m, O, strict):
    """Same run through the strict generic kernel: must also be inside the tolerance (and is in fact at rounding level)."""
    a, b, _, _ = H.run_pair(m, O, H.c3_enright(40), steps=60)
    d = H.check_parity(a, b, 1e-10)
    assert d <= 1e-13


# ------------------------------------------------------------------------------------------------
# BASELINE.json's FULL sizes, through size-independent properties (the oracle would need minutes per step there)
# ------------------------------------------------------------------------------------------------
def test_full_size_linear_field_is_advected_exactly(m):
    """512^3 Float64: WENO5 differentiates a linear field exactly (all smoothness indicators vanish) and
    LinearExtrapolationBC continues it exactly, so phi(x, t) = phi0(x) - t * (u . grad phi0) up to rounding."""
    n = 512
    g = m.CartesianGrid((0, 0, 0), (1, 1, 1), (n, n, n))
    a, u, c = (0.3, -0.2, 0.5), (0.7, -0.4, 0.5), 0.1
    phi = m.MeshField(lambda x: a[0] * x[0] + a[1] * x[1] + a[2] * x[2] + c, g)
    eq = m.LevelSetEquation(terms=(m.AdvectionTerm(u),), ic=phi, bc=m.LinearExtrapolationBC(), integrator=m.RK3())
    h = g.meshsize(1)
    tf = 12 * 0.5 / (sum(abs(v) for v in u) / h) * (1 - 1e-12)
    m.integrate(eq, tf)
    assert eq.steps_taken == 12
    x, y, z = g.coords()
    exact = a[0] * x + a[1] * y + a[2] * z + c - tf * sum(ai * ui for ai, ui in zip(a, u))
    assert np.abs(eq.state.peek() - exact).max() <= 1e-12


def test_full_size_flat_field_is_a_fixed_point(m):
    """512^3 Float32 under the Enright velocity: every difference of a constant field is zero, the epsilon floor keeps
    the WENO weights finite, so the field must stay bit-identical (test-levelsetterms.jl:53-77 at scale)."""
    case = H.c3_enright(512, np.float32)
    case.phi0[...] = 1.0
    phi = case.engine_field(m)
    eq = m.LevelSetEquation(terms=case.engine_terms(m, phi), ic=phi, integrator=m.RK3())
    m.integrate(eq, 3 * 0.5 * m.compute_cfl(eq.terms, eq.state, 0.0))
    out = eq.state.peek()
    assert eq.steps_taken >= 3 and np.all(out == np.float32(1.0))


def test_full_size_strict_and_tiled_kernels_agree(m):
    """256^3 Float64 C3 and C5: the reference-ordered strict kernel and the restructured tiled kernels (TMA fill, fused
    CFL, one reciprocal ...) must agree far inside the 1e-10 bar, with identical step sizes."""
    ctx = m.default_context()
    for case in (H.c3_enright(256), H.c5_normal_advection(192)):
        outs = []
        for kernel in (1, 0):
            ctx.set_option(OPT_KERNEL, kernel)
            phi = case.engine_field(m)
            eq = m.LevelSetEquation(terms=case.engine_terms(m, phi), ic=phi, integrator=m.RK3())
            m.integrate(eq, 3 * 0.5 * m.compute_cfl(eq.terms, eq.state, 0.0) * (1 - 1e-12))
            outs.append((eq.t, eq.steps_taken, eq.state.peek().copy()))
        ctx.set_option(OPT_KERNEL, 0)
        assert outs[0][:2] == outs[1][:2]
        d = np.abs(outs[0][2] - outs[1][2]).max()
        assert d <= 1e-13, d
        assert np.array_equal(np.sign(outs[0][2]), np.sign(outs[1][2]))


# ------------------------------------------------------------------------------------------------
# the reference's own integration tests, run through the engine (test-timestepping.jl, test-levelsetequation.jl)
# ------------------------------------------------------------------------------------------------
def _adv_err_1d(m, integ, N, u=1.0, tf=0.5, scheme=None):
    g = m.CartesianGrid((-1.0,), (1.0,), (N,))
    phi = m.MeshField(lambda x: np.sin(np.pi * x[0]), g)
    term = m.AdvectionTerm(lambda x, t: (u,), scheme or m.WENO5())
    eq = m.LevelSetEquation(terms=(term,), ic=phi, bc=m.PeriodicBC(), integrator=integ)
    m.integrate(eq, tf)
    x = g.coords()[0]
    return np.abs(eq.state.peek() - np.sin(np.pi * (x - u * tf))).max()


def test_reference_timestepping_tests(m):
    assert _adv_err_1d(m, m.ForwardEuler(), 200) < 0.05
    assert _adv_err_1d(m, m.RK2(), 200) < 1.0e-3
    assert _adv_err_1d(m, m.RK3(), 200) < 1.0e-5
    Ns = [50, 100, 200, 400]
    for mk, p in ((m.ForwardEuler, 1), (m.RK2, 2), (m.RK3, 3)):
        e = [_adv_err_1d(m, mk(), N) for N in Ns]
        for i in range(len(Ns) - 1):
            assert math.log(e[i] / e[i + 1]) / math.log(Ns[i + 1] / Ns[i]) >= p - 0.5


def test_reference_spatial_orders(m):
    e = [_adv_err_1d(m, m.RK3(1e-2), N) for N in (20, 40, 80)]
    assert all(math.log(e[i] / e[i + 1]) / math.log(2) >= 4.5 for i in range(2))
    e = [_adv_err_1d(m, m.RK3(1e-2), N, scheme=m.Upwind()) for N in (50, 100, 200)]
    assert all(math.log(e[i] / e[i + 1]) / math.log(2) >= 0.8 for i in range(2))


def test_reference_normal_and_curvature_orders(m):
    def run(N, term, exact, r0):
        g = m.CartesianGrid((-2.0, -2.0), (2.0, 2.0), (N, N))
        phi = m.MeshField(lambda x: np.sqrt(x[0] ** 2 + x[1] ** 2) - r0, g)
        eq = m.LevelSetEquation(terms=(term,), ic=phi, bc=m.ExtrapolationBC(2), integrator=m.RK3())
        m.integrate(eq, 0.2)
        x, y = g.coords()
        r = np.sqrt(x * x + y * y)
        return np.where((r >= 0.5) & (r <= 1.5), np.abs(eq.state.peek() - exact(r)), 0.0).max()

    e = [run(N, m.NormalMotionTerm(lambda x, t: 0.5), lambda r: r - 0.5 - 0.5 * 0.2, 0.5) for N in (30, 60, 120)]
    assert all(math.log(e[i] / e[i + 1]) / math.log(2) >= 1.5 for i in range(2))
    e = [run(N, m.CurvatureTerm(lambda x, t: -0.1), lambda r: np.sqrt(r * r + 0.2 * 0.2) - 0.7, 0.7) for N in (30, 60, 120)]
    assert all(math.log(e[i] / e[i + 1]) / math.log(2) >= 1.5 for i in range(2))


def test_reference_eikonal_and_nan_robustness(m):
    g = m.CartesianGrid((-1.0,), (1.0,), (101,))
    phi = m.MeshField(lambda x: 2 * (x[0] - 0.3), g)
    eq = m.LevelSetEquation(terms=(m.EikonalReinitializationTerm(phi),), ic=phi, bc=m.LinearExtrapolationBC())
    m.integrate(eq, 2.0)
    out, x = eq.state.peek(), g.coords()[0]
    assert np.where(np.abs(out) > 0.5, 0.0, np.abs(out - (x - 0.3))).max() < 0.05
    g2 = m.CartesianGrid((-2.0, -2.0), (2.0, 2.0), (31, 31))
    phi2 = m.MeshField(lambda x: np.sqrt(x[0] ** 2 + x[1] ** 2) - 0.7, g2)
    eq2 = m.LevelSetEquation(terms=(m.CurvatureTerm(lambda x, t: -0.1),), ic=phi2, bc=m.NeumannBC(), integrator=m.RK2())
    m.integrate(eq2, 0.1)
    assert not np.isnan(eq2.state.peek()).any()
    g3 = m.CartesianGrid((-1.0,), (1.0,), (31,))
    eq3 = m.LevelSetEquation(terms=(m.EikonalReinitializationTerm(),), ic=m.MeshField(lambda x: 0.0 * x[0], g3),
                             bc=m.NeumannBC(), integrator=m.RK2())
    m.integrate(eq3, 0.1)
    assert not np.isnan(eq3.state.peek()).any()


# ------------------------------------------------------------------------------------------------
# API semantics: hooks, update_func, incremental integrate!, ic untouched
# ------------------------------------------------------------------------------------------------
def test_hooks_update_func_and_incremental(m, O):
    case = H.c1_circle_rotation(48)
    phi = case.engine_field(m)
    terms = case.engine_terms(m, phi)
    before = phi.peek().copy()
    eq = m.LevelSetEquation(terms=terms, ic=phi, integrator=m.RK3())
    calls = {"pre": 0, "post": 0, "upd": 0}
    # two-leg integration with hooks == one-leg device loop (hooks here only count)
    m.integrate(eq, 0.05, prehook=lambda e: calls.__setitem__("pre", calls["pre"] + 1),
                posthook=lambda e: calls.__setitem__("post", calls["post"] + 1))
    m.integrate(eq, 0.1)
    assert calls["pre"] == calls["post"] > 0 and eq.t == 0.1
    assert np.array_equal(phi.peek(), before)                     # ic never mutated (levelsetequation.jl:66)
    fo = case.oracle_field()
    O.integrate(fo, O.RK3, case.oracle_terms(), 0.05)
    O.integrate(fo, O.RK3, case.oracle_terms(), 0.1, t0=0.05)
    assert np.abs(fo.vals - eq.state.peek()).max() <= 1e-12
    # update_func hook semantics (test-velocityextension.jl:4-17): called as f(coeff, phi, t) before the CFL and every stage
    g = m.CartesianGrid((-1.0, -1.0), (1.0, 1.0), (21, 21))
    p = m.MeshField(lambda x: np.sqrt(x[0] ** 2 + x[1] ** 2) - 0.5, g, bc=m.PeriodicBC())
    v = m.MeshField(np.zeros((21, 21)), g)
    seen = []

    def upd(speed, phi_stage, t):
        speed.vals[...] = 2 * t + 0.1
        seen.append(t)

    term = m.NormalMotionTerm(v, upd)
    m.update_term(term, p, 0.3)
    assert np.all(v.peek() == 0.7)
    eq = m.LevelSetEquation(terms=(term,), ic=p, integrator=m.RK3())
    m.integrate(eq, 1e-3, 5e-4)
    assert eq.steps_taken == 2 and len(seen) == 1 + 2 * (1 + 3)     # CFL refresh + 3 stages per step
    assert np.isfinite(eq.state.peek()).all()


def test_device_volume_and_perimeter(m, O):
    """SURVEY §8f row 1: volume / perimeter reduced on the device (levelsetops.jl:27-33,139-149) against the oracle, which
    reproduces the reference's doctest scalars bit for bit; the parallel sum only changes the summation order."""
    g = m.CartesianGrid((-1, -1), (1, 1), (200, 200))
    phi = m.MeshField(lambda x: np.sqrt(x[0] ** 2 + x[1] ** 2) - 0.5, g)           # no BCs: perimeter supplies LinearExtrapolationBC
    assert m.volume(phi) == pytest.approx(0.7854362890190668, rel=1e-13)           # levelsetops.jl:14-25
    assert m.perimeter(phi) == pytest.approx(3.1426415491430384, rel=1e-13)        # levelsetops.jl:126-137
    for case in (H.c3_enright(40), H.c2_zalesak_curvature(96), H.c4_eikonal(24, np.float32)):
        fo = case.oracle_field()
        f = case.engine_field(m)
        assert m.volume(f) == pytest.approx(fo.volume(), rel=1e-12)
        assert m.perimeter(f) == pytest.approx(fo.perimeter(), rel=1e-12)
    # as a posthook payload: the state is never downloaded
    case = H.c1_circle_rotation(64)
    f = case.engine_field(m)
    eq = m.LevelSetEquation(terms=case.engine_terms(m, f), ic=f, integrator=m.RK3())
    vols = []
    ctx = m.default_context()
    eq.state.device(); ctx.reset_counters()
    m.integrate(eq, 0.05, posthook=lambda e: vols.append(m.volume(e)))
    assert len(vols) == eq.steps_taken and ctx.counters()["d2h_bytes"] < 64 * (len(vols) + 2)
    assert abs(vols[-1] - vols[0]) < 2e-3 * vols[0]                                # rigid rotation preserves the area


def test_eikonal_reinitialize_prehook(m, O):
    """Eikonal reinitialisation as an in-place device prehook: restores |grad phi| = 1 near the interface of a distorted
    level set without moving the zero set much, and equals the same pseudo-time steps taken by the oracle."""
    g = m.CartesianGrid((-1, -1), (1, 1), (96, 96))
    f0 = lambda x: (np.sqrt(x[0] ** 2 + x[1] ** 2) - 0.5) * (1.5 + 0.8 * np.sin(4 * x[0]))
    phi = m.MeshField(f0, g, bc=m.NeumannBC())
    before = phi.peek().copy()
    m.eikonal_reinitialize(phi, iterations=30)
    out = phi.peek()
    fo = O.Field(before.copy(order="F"), (-1, -1), (1, 1), bc=O.NEUMANN)
    s0 = O.eikonal_s0(fo)
    dt = 0.5 * min(fo.meshsize())
    O.integrate(fo, O.RK2, [O.eikonal(s0)], dt * 30 * (1 - 1e-12))
    assert np.abs(out - fo.vals).max() <= 1e-10
    h = g.meshsize(1)
    gx, gy = np.gradient(out, h, h)
    band = np.abs(out) < 3 * h
    assert np.abs(np.hypot(gx, gy)[band] - 1).max() < 0.12 and np.abs(np.hypot(*np.gradient(before, h, h))[band] - 1).max() > 0.4
    assert (np.sign(out) != np.sign(before)).mean() < 5e-3        # the PDE reinitialisation moves the interface slightly (levelsetterms.jl:203-206)
    # as a prehook inside integrate! (docs/src/index.md:106-114 idiom)
    case = H.c1_circle_rotation(64)
    f = case.engine_field(m)
    eq = m.LevelSetEquation(terms=case.engine_terms(m, f), ic=f, integrator=m.RK3())
    m.integrate(eq, 0.03, prehook=lambda e: m.eikonal_reinitialize(m.current_state(e), iterations=2))
    assert np.isfinite(eq.state.peek()).all()


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_extend_along_normals(m, O, strict, dtype):
    """SURVEY §8f row 2: extend_along_normals! on the device against the oracle's restatement of velocityextension.jl:20-116,
    2-D (the grid of test-velocityextension.jl) and 3-D, default band mask and an explicit Bool mask, strict and tiled kernels."""
    ctx = m.default_context()
    for n, lc, hc in (((81, 61), (-1, -1), (1, 1)), ((30, 28, 26), (-1, -1, -1), (1, 1, 1))):
        X = H.coords(lc, hc, n)
        r = np.sqrt(sum(x * x for x in X))
        phi0 = H.bcast((r - 0.5) * (1 + 0.2 * X[0]), n).astype(dtype)
        F0 = H.bcast(np.sin(3 * X[0]) + X[1] ** 2, n).astype(dtype)
        mask = np.asfortranarray(np.abs(phi0) < 0.08)
        for frozen in (None, mask):
            for bc in (None, "neumann"):
                fo = O.Field(phi0.copy(order="F"), lc, hc, bc=None if bc is None else O.NEUMANN)
                Fo = O.extend_along_normals(F0.copy(order="F"), fo, nb_iters=12, frozen=frozen)
                for kernel in (1, 0):
                    ctx.set_option(OPT_KERNEL, kernel)
                    g = m.CartesianGrid(lc, hc, n)
                    phi = m.MeshField(phi0.copy(order="F"), g, bc=None if bc is None else m.NeumannBC())
                    F = m.MeshField(F0.copy(order="F"), g)
                    m.extend_along_normals(F, phi, nb_iters=12, frozen=frozen)
                    d = np.abs(F.peek().astype(np.float64) - Fo.astype(np.float64)).max()
                    tol = (1e-13 if kernel == 1 else 1e-11) if dtype == np.float64 else 2e-5
                    assert d <= tol, (n, frozen is not None, bc, kernel, d)
                    if frozen is not None:
                        assert np.array_equal(F.peek()[mask], F0[mask])          # Dirichlet constraint on frozen nodes
    with pytest.raises(ValueError):
        m.extend_along_normals(F, phi, nb_iters=-1)
    # F undefined (NaN) away from the interface: frozen nodes keep their values exactly (velocityextension.jl:53-56 copies them),
    # even where a neighbour is NaN — 0 * NaN must not leak into them
    n, lc, hc = (64, 56), (-1, -1), (1, 1)
    X = H.coords(lc, hc, n)
    phi0 = H.bcast(np.sqrt(X[0] ** 2 + X[1] ** 2) - 0.5, n).astype(dtype)
    mask = np.asfortranarray(np.abs(phi0) < 0.06)
    near = np.asfortranarray(np.abs(phi0) < 0.075)
    F0 = np.where(near, H.bcast(np.sin(3 * X[0]) + X[1] ** 2, n), np.nan).astype(dtype)
    for kernel in (1, 0):
        ctx.set_option(OPT_KERNEL, kernel)
        g = m.CartesianGrid(lc, hc, n)
        F = m.MeshField(F0.copy(order="F"), g)
        m.extend_along_normals(F, m.MeshField(phi0.copy(order="F"), g, bc=m.NeumannBC()), nb_iters=3, frozen=mask)
        assert np.array_equal(F.peek()[mask], F0[mask]) and not np.isnan(F.peek()[mask]).any()
    ctx.set_option(OPT_KERNEL, 0)


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_csg_on_device(m, O, dtype):
    """SURVEY §8f row 3: union!/intersect!/setdiff!/complement! on device fields, bit-identical to the oracle (Julia min/max
    semantics incl. NaN and signed zeros), and composing with the integrator without a host round trip."""
    n = (33, 29, 17)
    g = m.CartesianGrid((-1, -1, -1), (1, 1, 1), n)
    X = H.coords((-1, -1, -1), (1, 1, 1), n)
    a0 = H.bcast(np.sqrt((X[0] - 0.2) ** 2 + X[1] ** 2 + X[2] ** 2) - 0.5, n).astype(dtype)
    b0 = H.bcast(np.maximum(np.abs(X[0] + 0.1), np.maximum(np.abs(X[1]), np.abs(X[2]))) - 0.4, n).astype(dtype)
    a0[0, 0, 0], b0[1, 0, 0] = np.nan, np.nan
    a0[2, 0, 0], b0[2, 0, 0], a0[3, 0, 0], b0[3, 0, 0] = 0.0, -0.0, -0.0, 0.0
    bits = np.uint64 if dtype == np.float64 else np.uint32

    def same(x, y):          # bit-level comparison (signed zeros matter); NaNs must coincide, payloads may differ
        nx, ny = np.isnan(x), np.isnan(y)
        return np.array_equal(nx, ny) and np.array_equal(np.where(nx, 0, x).astype(dtype).view(bits), np.where(ny, 0, y).astype(dtype).view(bits))

    for name, fn_ip, fn in (("union", m.union_, m.union), ("intersect", m.intersect_, m.intersect), ("setdiff", m.setdiff_, m.setdiff)):
        a, b = m.MeshField(a0.copy(order="F"), g), m.MeshField(b0.copy(order="F"), g)
        ref = O.csg(name, a0, b0)
        out = fn(a, b)
        assert out is not a and np.array_equal(a.peek(), a0, equal_nan=True)
        assert same(out.peek(), ref), name
        assert fn_ip(a, b) is a and same(a.peek(), ref), name
    a = m.MeshField(a0.copy(order="F"), g)
    assert same(m.complement_(a).peek(), O.csg("complement", a0))
    with pytest.raises(ValueError):
        m.union_(a, m.MeshField(np.zeros((4, 4, 4), dtype=dtype), m.CartesianGrid((-1, -1, -1), (1, 1, 1), (4, 4, 4))))
    # device-resident composition: build a shape with set operations, then integrate it without touching the host copy
    a0[0, 0, 0], b0[1, 0, 0] = 1.0, 1.0
    phi = m.setdiff_(m.MeshField(a0.copy(order="F"), g, bc=m.NeumannBC()), m.MeshField(b0.copy(order="F"), g))
    eq = m.LevelSetEquation(terms=(m.AdvectionTerm((1.0, 0.0, 0.0)),), ic=phi, bc=m.NeumannBC(), integrator=m.RK3())
    m.integrate(eq, 0.05)
    fo = O.Field(O.csg("setdiff", a0, b0), (-1, -1, -1), (1, 1, 1), bc=O.NEUMANN)
    O.integrate(fo, O.RK3, [O.advection((1.0, 0.0, 0.0))], 0.05)
    assert np.abs(eq.state.peek().astype(np.float64) - fo.vals.astype(np.float64)).max() <= (1e-10 if dtype == np.float64 else 1e-4)


def test_graph_replay_is_invisible(m, O):
    """Small grids: lsm_integrate replays a captured CUDA graph of one step's stage launches (LSM_OPT_GRAPH).  States, times,
    step counts and launch counters must be identical with the option on and off, for RK3 and RK2, 2-D and 3-D, including a
    final shorter step (different dt -> direct launches) and a second integrate! call on the same equation."""
    ctx = m.default_context()
    OPT_GRAPH = m._lib.OPT_GRAPH
    ctx.set_option(m._lib.OPT_RESIDENT, 0)            # the resident cluster kernel would take the first case whole
    try:
        for mk, integ in ((lambda: H.c1_circle_rotation(64), m.RK3), (lambda: H.c2_zalesak_curvature(96), m.RK2),
                          (lambda: H.c5_normal_advection(24), m.RK3)):
            res = []
            for on in (1, 0):
                ctx.set_option(OPT_GRAPH, on)
                case = mk()
                phi = case.engine_field(m)
                eq = m.LevelSetEquation(terms=case.engine_terms(m, phi), ic=phi, integrator=integ())
                dt0 = 0.5 * m.compute_cfl(eq.terms, eq.state, 0.0)
                ctx.reset_counters()
                m.integrate(eq, dt0 * 17.3)               # 17 full steps + one shorter
                n1 = eq.steps_taken
                m.integrate(eq, dt0 * 25.0)
                c = ctx.counters()
                res.append((eq.state.peek().copy(), eq.t, n1, eq.steps_taken, c["kernel_launches"], c["stage_launches"]))
            ctx.set_option(OPT_GRAPH, 1)
            assert np.array_equal(res[0][0], res[1][0]) and res[0][1:] == res[1][1:], res[0][1:]
            fo = mk().oracle_field()
            O.integrate(fo, {m.RK3: O.RK3, m.RK2: O.RK2}[integ], mk().oracle_terms(), res[0][1])
            # two integrate calls vs one oracle call to the same final time: the step sequences differ, so compare loosely
            assert np.abs(res[0][0] - fo.vals).max() < 1e-3
    finally:
        ctx.set_option(OPT_GRAPH, 1)
        ctx.set_option(m._lib.OPT_RESIDENT, 1)


@pytest.mark.parametrize("integ", ["RK3", "RK2", "FE"])
def test_counters_and_launch_accounting(m, integ):
    """Launch accounting of the two ways the per-step CFL maximum of a time-scaled velocity is obtained, for all three
    integrators (both exact, so the states are bit-identical): (a) default — host evaluation over the candidate nodes: one
    reduction for the first step, the unscaled reduction + one extraction kernel when the set is built, nothing afterwards;
    (b) candidates off, which is also what a field with more ties at the maximum than the candidate list holds gets — one
    reduction pass per step.  Option 4 (the retired next-step reduction in the last stage) is refused."""
    ctx = m.default_context()
    with pytest.raises(m.LSMError) as ei:
        ctx.set_option(4, 0)
    assert ei.value.code == m._lib.ERR_ARG
    case = H.c3_enright(32)
    mk, nst = {"RK3": (m.RK3, 3), "RK2": (m.RK2, 2), "FE": (m.ForwardEuler, 1)}[integ]
    results = []
    for cand in (1, 0):
        ctx.set_option(m._lib.OPT_CFL_CANDIDATES, cand)
        phi = case.engine_field(m)
        eq = m.LevelSetEquation(terms=case.engine_terms(m, phi), ic=phi, integrator=mk())
        eq.state.device()
        eq.terms[0].velocity.base.device()            # upload the coefficient (AoS->SoA kernels) before counting
        ctx.reset_counters()
        m.integrate(eq, 0.02)
        c = ctx.counters()
        assert eq.steps_taken >= 3
        assert c["stage_launches"] == nst * eq.steps_taken
        if cand:
            assert c["cfl_passes"] == 2 and c["kernel_launches"] == c["stage_launches"] + 3
        else:
            assert c["cfl_passes"] == eq.steps_taken
            assert c["kernel_launches"] == c["stage_launches"] + c["cfl_passes"]
        results.append((eq.t, eq.steps_taken, eq.state.peek().copy()))
    ctx.set_option(m._lib.OPT_CFL_CANDIDATES, 1)
    assert results[0][:2] == results[1][:2] and np.array_equal(results[0][2], results[1][2])
