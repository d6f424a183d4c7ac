"""The semi-implicit (inflow-implicit / outflow-explicit) advection integrator, LSM_SEMI_IMPLICIT: the SciPy restatement's
behaviour on the CPU, and the engine against that restatement on the GPU, through the C ABI."""
import math

import numpy as np
import pytest

import semi_implicit_ref as R


# ---- the restatement (CPU) -------------------------------------------------------------------------------------------------
def _sine_error(n, cfl):
    x = np.linspace(-1.0, 1.0, n)
    h = 2.0 / (n - 1)
    phi, _ = R.integrate(np.sin(np.pi * x), lambda t: [np.ones(n)], [h], [(R.PERIODIC, R.PERIODIC)], 0.5, cfl=cfl)
    return float(np.max(np.abs(phi - np.sin(np.pi * (x - 0.5)))))


@pytest.mark.parametrize("cfl", [0.5, 2.0, 4.0])
def test_restatement_is_second_order_in_1d(cfl):
    ns = [51, 101, 201, 401]
    err = [_sine_error(n, cfl) for n in ns]
    orders = [math.log(err[i] / err[i + 1]) / math.log((ns[i + 1] - 1) / (ns[i] - 1)) for i in range(3)]
    assert min(orders) >= 1.9, (err, orders)


@pytest.mark.parametrize("cfl", [0.5, 2.0, 4.0])
def test_restatement_keeps_a_kinked_profile_in_range(cfl):
    n = 201
    x = np.linspace(-1.0, 1.0, n)
    phi0 = np.abs(x) - 0.5
    phi, _ = R.integrate(phi0, lambda t: [np.ones(n)], [2.0 / (n - 1)], [(R.PERIODIC, R.PERIODIC)], 0.5, cfl=cfl)
    assert phi.min() >= phi0.min() - 1e-14 and phi.max() <= phi0.max() + 1e-14
    inside = phi[:-1] <= 0                                           # nodes 1 .. n-1: one period, counted cyclically
    assert np.count_nonzero(inside != np.roll(inside, 1)) == 2


@pytest.mark.parametrize("cfl", [0.5, 2.0, 4.0])
def test_restatement_is_neutrally_stable_for_a_constant_velocity(cfl):
    n, k = 65, 3
    P = n - 1
    j = np.arange(n)
    phi = np.cos(2 * np.pi * k * j / P)
    h = 2.0 / P
    a0 = abs(np.fft.fft(phi[:P])[k])
    for _ in range(10):
        phi = R.step(phi, [np.full(n, 0.7)], [h], cfl * h / 0.7, [(R.PERIODIC, R.PERIODIC)])
    assert abs(abs(np.fft.fft(phi[:P])[k]) - a0) / a0 <= 1e-12


def test_host_sweep_count():
    import lsm_b200 as m
    for c in [0.0, 1e-3, 0.5, 1.0, 2.0, 4.0, 17.5]:
        for f64 in (True, False):
            assert m.semi_implicit_sweeps(c, np.float64 if f64 else np.float32) == R.sweeps(c, f64), (c, f64)
    assert m.semi_implicit_sweeps(2.0) == 50              # q = 0.5: 2^-50 < 1e-15
    for bad in (-1.0, math.inf, math.nan):
        with pytest.raises(m.LSMError) as ei:
            m.semi_implicit_sweeps(bad)
        assert ei.value.code == m._lib.ERR_ARG


def test_integrator_codes():
    import lsm_b200 as m
    assert m._lib.SEMI_IMPLICIT == 3 and m.SemiImplicit().cfl == 2.0 and m.SemiImplicit.nstages == 1
    assert m._lib.lib().lsm_nstages(m._lib.SEMI_IMPLICIT) == 1


# ---- the engine (GPU) --------------------------------------------------------------------------------------------------------
BCS = {"periodic": R.PERIODIC, "neumann": R.NEUMANN, "symmetry": R.SYMMETRY}


def _engine_bc(m, kind):
    return {"periodic": m.PeriodicBC(), "neumann": m.NeumannBC(), "symmetry": m.SymmetryBC()}[kind]


def _grid(ndim, n):
    lc, hc = (-1.0, -0.9, -1.1)[:ndim], (1.0, 1.1, 0.8)[:ndim]
    return lc, hc, n[:ndim]


def _base_velocity(X, ndim):
    """A velocity with sign changes in every component (N arrays at the nodes)."""
    x = X[0]
    if ndim == 1:
        return [np.sin(np.pi * x) + 0.3 + 0 * x]
    y = X[1]
    if ndim == 2:
        return [-(y - 0.2) + 0 * x, (x + 0.1) + 0 * y]
    z = X[2]
    return [-(y - 0.2) + 0 * x * z, (x + 0.1) + 0 * y * z, 0.5 * np.sin(np.pi * x) + 0 * y * z]


_EXPRS = {1: ("(sin(pi * x1) + 0.3) * cos(pi * t)",),
          2: ("-(x2 - 0.2) * cos(pi * t)", "(x1 + 0.1) * cos(pi * t)"),
          3: ("-(x2 - 0.2) * cos(pi * t)", "(x1 + 0.1) * cos(pi * t)", "0.5 * sin(pi * x1) * cos(pi * t)")}


def _setup(m, ndim, n, kind, bcs, dtype):
    """(engine equation, numpy phi0, velocity(t) -> N arrays in float64, grid spacing h)."""
    lc, hc, n = _grid(ndim, n)
    grid = m.CartesianGrid(lc, hc, n)
    X = [np.asarray(c, dtype=np.float64) for c in grid.coords()]
    h = grid.meshsize()
    r2 = sum((X[d] - 0.1 * (d + 1)) ** 2 for d in range(ndim))
    phi0 = np.broadcast_to(np.sqrt(r2) - 0.5, n).astype(dtype)
    base = [np.broadcast_to(b, n).astype(np.float64) for b in _base_velocity(X, ndim)]
    T = 0.8
    if kind == "const":
        cv = (0.7, -0.4, 0.3)[:ndim]
        vel, velocity = tuple(cv), (lambda t: [np.full(n, c) for c in cv])
    elif kind == "field":
        stored = np.stack(base).astype(dtype)
        vel, velocity = m.MeshField(stored, grid), (lambda t: [stored[d].astype(np.float64) for d in range(ndim)])
    elif kind == "timescaled":
        stored = np.stack(base).astype(dtype)
        vel = m.TimeScaled(m.MeshField(stored, grid), ("cos", T))
        velocity = lambda t: [stored[d].astype(np.float64) * math.cos(math.pi * t / T) for d in range(ndim)]
    elif kind == "separable":
        # u_d = s_d X_d[i1] Y_d[i2] Z_d[i3]: the rotation-like field (-(y - 0.2), x + 0.1, ...) as rank-1 products
        xs = [np.asarray(grid.coords()[a], dtype=np.float64).ravel() for a in range(ndim)]
        tabs = [[np.ones(n[a]) for a in range(ndim)] for _ in range(ndim)]
        scales = [1.0] * ndim
        tabs[0][0] = np.sin(np.pi * xs[0]) + 0.3
        if ndim > 1:
            tabs[0][0] = np.ones(n[0]); tabs[0][1] = -(xs[1] - 0.2)
            tabs[1][0] = xs[0] + 0.1
        if ndim > 2:
            tabs[2][0] = 0.5 * np.sin(np.pi * xs[0]); tabs[2][2] = np.cos(xs[2])
        vel = m.SeparableVelocity(grid, scales, tabs)

        def velocity(t):
            out = []
            for d in range(ndim):
                v = scales[d] * tabs[d][0].reshape([-1] + [1] * (ndim - 1))
                for a in range(1, ndim):
                    shp = [1] * ndim; shp[a] = -1
                    v = v * tabs[d][a].reshape(shp)
                out.append(np.broadcast_to(v, n).astype(np.float64))
            return out
    else:   # expression
        vel = m.DeviceExpr(_EXPRS[ndim])
        # the engine materialises the expressions in the state's dtype
        velocity = lambda t: [np.broadcast_to(eval_expr(e, X, t), n).astype(dtype).astype(np.float64) for e in _EXPRS[ndim]]
    phi = m.MeshField(phi0.copy(), grid, bc=[_engine_bc(m, b) for b in bcs], dtype=dtype)
    eq = m.LevelSetEquation(terms=m.AdvectionTerm(vel, m.Upwind()), ic=phi, integrator=m.SemiImplicit())
    return eq, phi0, velocity, h


def eval_expr(e, X, t):
    env = {"sin": np.sin, "cos": np.cos, "pi": np.pi, "t": t}
    env.update({f"x{d + 1}": X[d] for d in range(len(X))})
    return eval(e, env)


def _advance(m, eq, tc, dt):
    """One lsm_advance step of the state through the C ABI."""
    phi = eq.state
    low = m.api._Lowered(eq.terms, phi, tc)
    m._lib.check(m._lib.lib().lsm_advance(phi._context().handle, m._lib.SEMI_IMPLICIT, phi.device(), low.arr, len(eq.terms),
                                           float(tc), float(dt)))
    phi._mark_device_advanced()


def _run_both(m, eq, phi0, velocity, h, bcs, cfl, steps=20):
    ndim = len(h)
    dt = cfl * R.cfl_dt(velocity(0.0), h)
    ref, tc = phi0.astype(np.float64), 0.0
    rbcs = [(BCS[b], BCS[b]) for b in bcs]
    for _ in range(steps):
        _advance(m, eq, tc, dt)
        ref = R.step(ref, velocity(tc + 0.5 * dt), h, dt, rbcs)
        tc += dt
    return np.asarray(eq.state.peek(), dtype=np.float64), ref


CASES = []
for ndim, n in ((1, (57,)), (2, (24, 19)), (3, (12, 10, 9))):
    for kind in ("const", "field", "separable", "timescaled", "expr"):
        for cfl in (0.5, 2.0, 4.0):
            CASES.append((ndim, n, kind, cfl))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("ndim,n,kind,cfl", CASES)
def test_engine_matches_restatement(ndim, n, kind, cfl, dtype):
    import lsm_b200 as m
    bcs = [("periodic", "neumann", "symmetry")[(d + int(cfl)) % 3] for d in range(ndim)]
    eq, phi0, velocity, h = _setup(m, ndim, n, kind, bcs, dtype)
    out, ref = _run_both(m, eq, phi0, velocity, h, bcs, cfl)
    tol = 1e-12 if dtype == np.float64 else 1e-5
    assert np.max(np.abs(out - ref)) <= tol * max(1.0, np.max(np.abs(ref)))


# larger grids (many thread blocks per sweep launch) and every BC on every axis
BIG = [(1, (5000,)), (2, (100, 90)), (3, (30, 20, 17))]


@pytest.mark.gpu
@pytest.mark.parametrize("bc", ["periodic", "neumann", "symmetry", "mixed"])
@pytest.mark.parametrize("ndim,n", BIG)
def test_engine_matches_restatement_on_many_tiles(ndim, n, bc):
    import lsm_b200 as m
    bcs = [("periodic", "neumann", "symmetry")[d % 3] if bc == "mixed" else bc for d in range(ndim)]
    if bc == "mixed" and ndim == 1:
        bcs = ["neumann"]
    eq, phi0, velocity, h = _setup(m, ndim, n, "field", bcs, np.float64)
    out, ref = _run_both(m, eq, phi0, velocity, h, bcs, 2.0, steps=6)
    assert np.max(np.abs(out - ref)) <= 1e-12


@pytest.mark.gpu
def test_mixed_bc_box():
    """Neumann on the left and symmetry on the right of one axis, periodic on the other."""
    import lsm_b200 as m
    grid = m.CartesianGrid((-1.0, -1.0), (1.0, 1.0), (70, 61))
    X = [np.asarray(c, dtype=np.float64) for c in grid.coords()]
    phi0 = np.broadcast_to(np.sqrt((X[0] - 0.3) ** 2 + X[1] ** 2) - 0.4, grid.n).astype(np.float64)
    u = np.stack([np.broadcast_to(b, grid.n) for b in _base_velocity(X, 2)]).astype(np.float64)
    bc = [(m.NeumannBC(), m.SymmetryBC()), m.PeriodicBC()]
    phi = m.MeshField(phi0.copy(), grid, bc=bc)
    eq = m.LevelSetEquation(terms=m.AdvectionTerm(m.MeshField(u, grid)), ic=phi, integrator=m.SemiImplicit())
    h = grid.meshsize()
    dt = 2.0 * R.cfl_dt([u[0], u[1]], h)
    ref = phi0
    for s in range(10):
        _advance(m, eq, s * dt, dt)
        ref = R.step(ref, [u[0], u[1]], h, dt, [(R.NEUMANN, R.SYMMETRY), (R.PERIODIC, R.PERIODIC)])
    assert np.max(np.abs(np.asarray(eq.state.peek()) - ref)) <= 1e-12


@pytest.mark.gpu
def test_sweep_count_in_counters():
    import lsm_b200 as m
    ctx = m.default_context()
    eq, phi0, velocity, h = _setup(m, 2, (40, 30), "field", ["periodic", "periodic"], np.float64)
    ctx.reset_counters()
    m.integrate(eq, 0.3)
    c = ctx.counters()
    dt_cfl = R.cfl_dt(velocity(0.0), h)
    assert eq.steps_taken >= 2
    # every full step is at Courant number 2 (the last one may be shorter)
    assert c["jacobi_sweeps"] >= (eq.steps_taken - 1) * R.sweeps(2.0 * (1 + 1e-12)) - 1
    assert c["jacobi_sweeps"] <= eq.steps_taken * R.sweeps(2.0 * (1 + 1e-12))
    assert abs(eq.t - 0.3) == 0 and dt_cfl > 0


@pytest.mark.gpu
def test_integrate_lands_on_tf_like_the_restatement_loop():
    import lsm_b200 as m
    bcs = ["periodic", "symmetry"]
    eq, phi0, velocity, h = _setup(m, 2, (33, 29), "timescaled", bcs, np.float64)
    tf = 0.37
    m.integrate(eq, tf)
    ref, steps = R.integrate(phi0, velocity, h, [(BCS[b], BCS[b]) for b in bcs], tf, cfl=2.0)
    assert eq.steps_taken == steps and eq.t == tf
    assert np.max(np.abs(np.asarray(eq.state.peek()) - ref)) <= 1e-12
    # with a posthook every step goes through the stage entry point: the same steps, bit for bit
    eq2, *_ = _setup(m, 2, (33, 29), "timescaled", bcs, np.float64)
    seen = []
    m.integrate(eq2, tf, posthook=lambda ls: seen.append(ls.t))
    assert len(seen) == steps
    assert np.array_equal(np.asarray(eq2.state.peek()), np.asarray(eq.state.peek()))


# a smooth profile whose zero level set is the same circle: 0.5 - exp(-(r / s)^2) with exp(-(0.3 / s)^2) = 1/2
_SMOOTH_S = 0.3 / math.sqrt(math.log(2.0))


def _rotation(m, n, integ, smooth=False):
    """Rigid rotation about the origin over one revolution of a level set whose zero level set is the circle of radius 0.3 around
    (0.4, 0): its signed distance, or with `smooth` the profile above.  Returns the max error in the band |r - 0.3| <= 0.15."""
    grid = m.CartesianGrid((-1.0, -1.0), (1.0, 1.0), (n, n))
    X = [np.asarray(c, dtype=np.float64) for c in grid.coords()]
    r = np.broadcast_to(np.sqrt((X[0] - 0.4) ** 2 + X[1] ** 2), grid.n)
    phi0 = (0.5 - np.exp(-(r / _SMOOTH_S) ** 2) if smooth else r - 0.3).astype(np.float64)
    u = np.stack([np.broadcast_to(-2 * np.pi * X[1], grid.n), np.broadcast_to(2 * np.pi * X[0], grid.n)]).astype(np.float64)
    phi = m.MeshField(phi0.copy(), grid, bc=[m.NeumannBC(), m.NeumannBC()])
    eq = m.LevelSetEquation(terms=m.AdvectionTerm(m.MeshField(u, grid), m.WENO5()), ic=phi, integrator=integ)
    m.integrate(eq, 1.0)
    out = np.asarray(eq.state.peek())
    band = np.abs(r - 0.3) <= 0.15
    return float(np.max(np.abs(out - phi0)[band])), eq.steps_taken, out, grid.meshsize()[0]


@pytest.mark.gpu
def test_rigid_rotation_order_interface_and_step_count():
    import lsm_b200 as m
    # Second order on a smooth profile.  The signed distance of the circle is not a fair test of the order: its kink at the centre
    # and its non-zero slope at the clamped Neumann boundary leave errors that this neutrally stable scheme (|G| = 1) never damps,
    # so on it the SciPy restatement shows only 0.8-1.5 at these resolutions.
    e = [_rotation(m, n, m.SemiImplicit(2.0), smooth=True)[0] for n in (64, 128, 256)]
    orders = [math.log2(e[0] / e[1]), math.log2(e[1] / e[2])]
    assert min(orders) >= 1.8, (e, orders)
    res = {n: _rotation(m, n, m.SemiImplicit(2.0)) for n in (64, 128, 256)}
    for n in (64, 128, 256):
        err, steps, out, h = res[n]
        # the zero level set stays within 2h of the exact circle: on every cut grid edge the crossing is within 2h of radius 0.3
        grid = m.CartesianGrid((-1.0, -1.0), (1.0, 1.0), (n, n))
        X = [np.asarray(c, dtype=np.float64) for c in grid.coords()]
        xs, ys = np.broadcast_to(X[0], (n, n)), np.broadcast_to(X[1], (n, n))
        a, b = out[:-1, :], out[1:, :]
        cut = (a <= 0) != (b <= 0)
        t = a[cut] / (a[cut] - b[cut])
        px, py = xs[:-1, :][cut] + t * h, ys[:-1, :][cut]
        assert cut.any() and np.max(np.abs(np.hypot(px - 0.4, py) - 0.3)) <= 2 * h
    steps_rk3 = _rotation(m, 64, m.RK3(0.5))[1]
    assert abs(res[64][1] * 4 - steps_rk3) <= 4, (res[64][1], steps_rk3)


@pytest.mark.gpu
def test_refusals():
    import lsm_b200 as m
    L = m._lib
    grid = m.CartesianGrid((-1.0, -1.0), (1.0, 1.0), (20, 20))
    X = grid.coords()
    phi0 = np.broadcast_to(np.sqrt(X[0] ** 2 + X[1] ** 2) - 0.5, grid.n).astype(np.float64)

    def run(terms, bc):
        phi = m.MeshField(phi0.copy(), grid, bc=bc)
        eq = m.LevelSetEquation(terms=terms, ic=phi, integrator=m.SemiImplicit())
        with pytest.raises(m.LSMError) as ei:
            m.integrate(eq, 0.1)
        with pytest.raises(m.LSMError) as es:
            _advance(m, eq, 0.0, 0.01)
        assert es.value.code == ei.value.code
        return ei.value

    e = run((m.AdvectionTerm((1.0, 0.5)), m.CurvatureTerm(0.1)), m.PeriodicBC())
    assert e.code == L.ERR_ARG and "exactly one AdvectionTerm" in str(e)
    e = run(m.NormalMotionTerm(1.0), m.PeriodicBC())
    assert e.code == L.ERR_ARG and "exactly one AdvectionTerm" in str(e)
    e = run(m.AdvectionTerm((1.0, 0.5)), [m.PeriodicBC(), m.LinearExtrapolationBC()])
    assert e.code == L.ERR_UNSUPPORTED and "ExtrapolationBC{1}" in str(e)
    e = run(m.AdvectionTerm((1.0, 0.5)), [m.ExtrapolationBC(2), m.NeumannBC()])
    assert e.code == L.ERR_UNSUPPORTED and "ExtrapolationBC{2}" in str(e)
    # lsm_stage: one stage only
    phi = m.MeshField(phi0.copy(), grid, bc=m.PeriodicBC())
    low = m.api._Lowered((m.AdvectionTerm((1.0, 0.5)),), phi, 0.0)
    rc = L.lib().lsm_stage(phi._context().handle, L.SEMI_IMPLICIT, 2, phi.device(), low.arr, 1, 0.0, 0.01, None)
    assert rc == L.ERR_ARG


@pytest.mark.gpu
def test_slab_decomposition_is_refused():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs for a slab-decomposed context")
    import lsm_b200 as m
    mc = m.MultiContext([0, 1])
    grid = m.CartesianGrid((-1.0, -1.0), (1.0, 1.0), (16, 16))
    eqs = []
    for c in mc.ranks:
        X = grid.coords(*c.slab(16))
        phi = m.MeshField(np.sqrt(X[0] ** 2 + X[1] ** 2) - 0.5 + 0 * X[0], grid, bc=m.PeriodicBC(), ctx=c)
        eqs.append(m.LevelSetEquation(terms=m.AdvectionTerm((1.0, 0.5)), ic=phi, integrator=m.SemiImplicit()))
    with pytest.raises(m.LSMError) as ei:
        m.integrate_multi(mc, eqs, 0.1)
    assert ei.value.code == m._lib.ERR_UNSUPPORTED and "slab decomposition is not supported" in str(ei.value)
