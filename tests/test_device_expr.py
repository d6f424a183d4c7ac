"""Function-valued coefficients f(x, t) (levelsetterms.jl:42-43) written as CUDA C++ expressions (DeviceExpr, lsm_expr_check,
lsm_field_set_expr, lsm_field_fill_expr).  The first tests need no GPU: validation and NVRTC compilation run on the host.  The
`gpu` tests check the generated kernel against NumPy, the device path against today's host path (a Python callable evaluated with
NumPy and uploaded at every CFL and stage time) bit for bit, the static case against stored fields, the oracle, launch accounting,
graph replay, the hooked host loop and the multi-GPU fan-out."""
import ctypes as C

import numpy as np
import pytest

import helpers as H


@pytest.fixture(scope="module")
def m():
    import lsm_b200
    return lsm_b200


def _check(m, ndim, ncomp, exprs):
    arr = (C.c_char_p * (len(exprs) + 1))(*[e.encode() for e in exprs], None)
    return m._lib.lib().lsm_expr_check(ndim, ncomp, arr), m._lib.last_error()


VALID = [
    (1, ("sqrt(fabs(x1)) - 0.5",)),
    (1, ("-x1*(1.0 + t)",)),
    (2, ("fmin(x1, x2)*fmax(x1, 0.25) - pi/4",)),
    (2, ("-x2*(1.0+t)", "x1*(1.0+t)")),
    (3, ("sqrt(x1*x1 + x2*x2 + x3*x3) - 0.5",)),
    (3, ("2.0*sin(pi*x1)*sin(pi*x1)*sin(2.0*pi*x2)*sin(2.0*pi*x3)*cos(pi*t/3.0)",
         "-sin(2.0*pi*x1)*sin(pi*x2)*sin(pi*x2)*sin(2.0*pi*x3)*cos(pi*t/3.0)",
         "-sin(2.0*pi*x1)*sin(2.0*pi*x2)*sin(pi*x3)*sin(pi*x3)*cos(pi*t/3.0)")),
]


@pytest.mark.parametrize("ndim,exprs", VALID, ids=[f"{d}d_{len(e)}comp_{i}" for i, (d, e) in enumerate(VALID)])
def test_valid_expressions_compile_without_a_gpu(m, ndim, exprs):
    rc, msg = _check(m, ndim, len(exprs), exprs)
    assert rc == m._lib.OK, msg
    e = m.DeviceExpr(exprs if len(exprs) > 1 else exprs[0])
    assert e.ncomp == len(exprs) and e.exprs == tuple(exprs)


REJECTED = [
    ("", "empty expression"),
    ("   ", "empty expression"),
    ("x1; x2", "';' is not allowed"),
    ("{x1}", "'{' is not allowed"),
    ("x1 }", "'}' is not allowed"),
    ("#x1", "'#' is not allowed"),
    ('x1 + "a"', "'\"' is not allowed"),
    ("x1 + 'a'", "''' is not allowed"),
    ("x1 \\ 2.0", "'\\' is not allowed"),
    ("x1 + `a`", "'`' is not allowed"),
    ("lsm_a.t", "'lsm_a' is reserved"),
    ("__sinf(x1)", "'__sinf' is reserved"),
    ("1/3*x1", "integer division 1/3"),
    ("x1 * (2 / -3)", "integer division 2/3"),
]


@pytest.mark.parametrize("expr,why", REJECTED, ids=[f"r{i}" for i in range(len(REJECTED))])
def test_rejected_forms_name_the_reason(m, expr, why):
    rc, msg = _check(m, 2, 1, (expr,))
    assert rc == m._lib.ERR_ARG and why in msg, msg
    with pytest.raises(m.LSMError) as ei:
        m.DeviceExpr(expr)
    assert ei.value.code == m._lib.ERR_ARG and why in str(ei.value)


def test_floating_divisions_and_count_checks(m):
    for ok in ("1.0/3*x1", "1/3.0*x1", "x1/3", "1e3/2*x1", "0x10/2.0"):
        rc, msg = _check(m, 1, 1, (ok,))
        assert rc == m._lib.OK, (ok, msg)
    rc, msg = _check(m, 2, 2, ("x1",))
    assert rc == m._lib.ERR_ARG and "fewer than ncomp" in msg
    rc, msg = _check(m, 2, 1, ("x1", "x2"))
    assert rc == m._lib.ERR_ARG and "more than ncomp" in msg
    rc, msg = _check(m, 2, 3, ("x1", "x2", "x1"))
    assert rc == m._lib.ERR_ARG and "ncomp must be 1 or ndim" in msg
    rc, msg = _check(m, 4, 1, ("x1",))
    assert rc == m._lib.ERR_ARG and "ndim must be" in msg


def test_compile_error_returns_the_nvrtc_log(m):
    rc, msg = _check(m, 1, 1, ("x1 + ",))
    assert rc == m._lib.ERR_ARG and "x1 + " in msg and "error" in msg, msg
    rc, msg = _check(m, 2, 1, ("x3",))                       # no x3 in 2-D
    assert rc == m._lib.ERR_ARG and "x3" in msg and "undefined" in msg, msg
    with pytest.raises(m.LSMError) as ei:
        m.DeviceExpr("cos(x1) +* 2.0")
    assert ei.value.code == m._lib.ERR_ARG and "cos(x1) +* 2.0" in str(ei.value)


def test_time_scaled_expression_is_refused(m):
    with pytest.raises(ValueError):
        m.TimeScaled(m.DeviceExpr(("-x2", "x1")), ("cos", 3.0))
    with pytest.raises(TypeError):
        m.DeviceExpr(("x1", 2.0))


# =================================================================================================================================
# GPU
# =================================================================================================================================
NS = dict(sqrt=np.sqrt, fabs=np.abs, fmin=np.fmin, fmax=np.fmax, sin=np.sin, cos=np.cos, exp=np.exp, pi=np.pi)
GRIDS = {1: ((-1.0,), (1.5,), (37,)), 2: ((-1.0, -0.5), (1.0, 2.0), (33, 29)), 3: ((-1.0, 0.0, -0.3), (1.0, 1.0, 0.7), (17, 13, 11))}
EXACT = {1: ("sqrt(fabs(x1)) - 0.5*x1/3.0", ("fmax(x1, -0.25)*x1 - pi",)),
         2: ("sqrt(x1*x1 + x2*x2) - 0.5*fabs(x1 - x2)/3.0 + fmin(x1, x2)*fmax(x1, 0.25)", ("-x2*x1 + pi", "x1/(1.5 + x2*x2)")),
         3: ("sqrt((x1 - 0.35)*(x1 - 0.35) + (x2 - 0.35)*(x2 - 0.35) + x3*x3) - 0.15",
             ("-x2 + 0.5*x3", "x1*x3 - fmin(x2, 0.5)", "fabs(x1 - x2)/(2.0 + x3)"))}
TRANSC = {1: "sin(pi*x1)*exp(-x1*x1)", 2: "cos(2.0*pi*x1)*sin(pi*x2) + exp(x1 - x2)", 3: "sin(pi*x1)*cos(pi*x2)*exp(-x3)"}


def _numpy(grid, exprs, dtype):
    X = grid.coords()
    ns = dict(NS, **{f"x{d + 1}": X[d] for d in range(grid.ndim)}, t=0.0)
    vals = [np.broadcast_to(eval(e, {"__builtins__": {}}, ns), grid.n) for e in exprs]
    v = np.stack(vals, axis=0) if len(exprs) > 1 else vals[0]
    return v.astype(dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("ndim", [1, 2, 3])
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_from_expr_matches_numpy(m, ndim, dtype):
    """MeshField.from_expr in 1-3 D, scalar and vector: bit-identical to NumPy evaluating the same formula on grid.coords() with
    + - * / sqrt fabs fmin fmax; within 1e-14 relative with sin, cos and exp."""
    grid = m.CartesianGrid(*GRIDS[ndim])
    bits = np.uint64 if dtype == np.float64 else np.uint32
    scalar, vector = EXACT[ndim]
    for exprs in ((scalar,), vector):
        f = m.MeshField.from_expr(grid, exprs if len(exprs) > 1 else exprs[0], dtype=dtype)
        got, want = f.peek(), _numpy(grid, exprs, dtype)
        assert got.shape == want.shape and got.dtype == want.dtype
        assert np.array_equal(got.view(bits), want.view(bits)), (exprs, np.abs(got - want).max())
    if dtype == np.float64:
        got = m.MeshField.from_expr(grid, TRANSC[ndim]).peek()
        want = _numpy(grid, (TRANSC[ndim],), np.float64)
        assert np.abs(got - want).max() <= 1e-14 * np.abs(want).max()


def _flow(ndim):
    """(device expressions, the equivalent Python callable) of time-dependent coefficients, + - * / only."""
    if ndim == 2:
        return ("-x2*(1.0+t)", "x1*(1.0+t)"), lambda x, t: (-x[1] * (1.0 + t), x[0] * (1.0 + t))
    return (("-x2*(1.0+0.5*t)", "x1*(1.0+0.5*t)", "0.25*(1.0-t)+0.1*x3"),
            lambda x, t: (-x[1] * (1.0 + 0.5 * t), x[0] * (1.0 + 0.5 * t), 0.25 * (1.0 - t) + 0.1 * x[2]))


SPEED = ("0.2 + 0.1*t*x1", lambda x, t: 0.2 + 0.1 * t * x[0])
BCURV = ("-0.01*(1.0 + t) - 0.001*x1*x1", lambda x, t: -0.01 * (1.0 + t) - 0.001 * x[0] * x[0])


def _terms(m, kind, device):
    pick = (lambda pair: m.DeviceExpr(pair[0])) if device else (lambda pair: pair[1])
    if kind == "adv2d_weno":
        return (m.AdvectionTerm(pick(_flow(2)), m.WENO5()),)
    if kind == "adv3d_upwind":
        return (m.AdvectionTerm(pick(_flow(3)), m.Upwind()),)
    if kind == "normal":
        return (m.NormalMotionTerm(pick(SPEED)),)
    if kind == "curvature":
        return (m.CurvatureTerm(pick(BCURV)),)
    return (m.AdvectionTerm(pick(_flow(2)), m.WENO5()), m.CurvatureTerm(pick(BCURV)))


def _phi0(m, ndim, dtype, ctx=None):
    if ndim == 2:
        grid = m.CartesianGrid((-1.0, -1.0), (1.0, 1.0), (48, 40))
        f = lambda x: np.sqrt((x[0] - 0.3) ** 2 + x[1] ** 2) - 0.4
    else:
        grid = m.CartesianGrid((-1.0, -1.0, -1.0), (1.0, 1.0, 1.0), (24, 20, 18))
        f = lambda x: np.sqrt((x[0] - 0.3) ** 2 + x[1] ** 2 + x[2] ** 2) - 0.4
    return m.MeshField(f, grid, bc=m.NeumannBC(), dtype=dtype, ctx=ctx)


def _run(m, kind, integ, dtype, device, tf_steps=7.3, **kw):
    ndim = 3 if kind == "adv3d_upwind" else 2
    phi = _phi0(m, ndim, dtype)
    eq = m.LevelSetEquation(terms=_terms(m, kind, device), ic=phi, integrator=integ())
    dt0 = integ().cfl * m.compute_cfl(eq.terms, eq.state, 0.0)
    m.integrate(eq, dt0 * tf_steps, **kw)
    return eq


INTEGS = ["ForwardEuler", "RK2", "RK3"]
KINDS = ["adv2d_weno", "adv3d_upwind", "normal", "curvature", "adv_curv"]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("integ", INTEGS)
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_time_dependent_expression_equals_host_callable(m, kind, integ, dtype):
    """integrate with a time-dependent DeviceExpr == integrate with the equivalent Python callable (host path) bit for bit: same
    state, time and step count.  The final time is 7.3 initial CFL steps, so the run ends in a shorter final step."""
    I = getattr(m, integ)
    dev = _run(m, kind, I, dtype, True)
    host = _run(m, kind, I, dtype, False)
    assert dev.t == host.t and dev.steps_taken == host.steps_taken >= 5
    assert np.array_equal(dev.state.peek(), host.state.peek()), np.abs(dev.state.peek() - host.state.peek()).max()


@pytest.mark.gpu
def test_static_expression_runs_like_a_stored_field(m):
    """An expression without `t` is materialised once and then IS a stored field: C1 with DeviceExpr(("-x2", "x1")) equals
    helpers.c1_circle_rotation bit for bit and takes the resident cluster kernel; a 3-D 64^3 case takes the x-pair kernel."""
    ctx = m.default_context()
    case = H.c1_circle_rotation(128)
    outs = []
    for device in (True, False):
        f = case.engine_field(m)
        terms = (m.AdvectionTerm(m.DeviceExpr(("-x2", "x1")), m.WENO5()),) if device else case.engine_terms(m, f)
        eq = m.LevelSetEquation(terms=terms, ic=f, integrator=m.RK3())
        dt = 0.5 * m.compute_cfl(eq.terms, eq.state, 0.0)
        ctx.reset_counters()
        m.integrate(eq, 60 * dt * (1 - 1e-12))
        outs.append((eq.t, eq.steps_taken, eq.state.peek().copy(), ctx.counters()["resident_steps"]))
    assert outs[0][3] > 0 and outs[0][:2] == outs[1][:2] and np.array_equal(outs[0][2], outs[1][2])
    n = (64, 64, 64)
    lc, hc = (-1, -1, -1), (1, 1, 1)
    x, y, z = H.coords(lc, hc, n)
    phi = np.sqrt((x - 0.3) ** 2 + y * y + z * z) - 0.4
    u = np.stack([H.bcast(-y, n), H.bcast(x, n), np.full(n, 0.5)], axis=0)
    case = H.Case("S3", lc, hc, n, phi, [dict(kind="advection", field=u)], ("neumann",))
    outs = []
    for device in (True, False):
        f = case.engine_field(m)
        terms = (m.AdvectionTerm(m.DeviceExpr(("-x2", "x1", "0.5")), m.WENO5()),) if device else case.engine_terms(m, f)
        eq = m.LevelSetEquation(terms=terms, ic=f, integrator=m.RK3())
        dt = 0.5 * m.compute_cfl(eq.terms, eq.state, 0.0)
        ctx.reset_counters()
        m.integrate(eq, 12 * dt * (1 - 1e-12))
        c = ctx.counters()
        outs.append((eq.t, eq.steps_taken, eq.state.peek().copy(), c["pair_launches"], c["cfl_passes"]))
    assert outs[0][3] > 0 and outs[0][4] <= 1 and outs[0][:2] == outs[1][:2] and np.array_equal(outs[0][2], outs[1][2])


def _enright_expr(m):
    return m.DeviceExpr(VALID[-1][1])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_c3_enright_expression_oracle_parity(m, O, dtype):
    """C3 at 64^3 with the Enright velocity written as a time-dependent expression, 100 RK3 steps: within 1e-10 (f64) / 1e-4 (f32)
    of the oracle's stored-field x cos(pi t / 3) run, identical sign and cut-cell classification."""
    case = H.c3_enright(64, dtype)
    fo, to = case.oracle_field(), case.oracle_terms()
    dt0 = 0.5 * O.compute_cfl(fo, to, 0.0)
    tf = dt0 * 100 * (1 - 1e-12)
    O.integrate(fo, O.RK3, to, tf, dt_max=dt0)
    phi = case.engine_field(m)
    eq = m.LevelSetEquation(terms=(m.AdvectionTerm(_enright_expr(m), m.WENO5()),), ic=phi, integrator=m.RK3())
    m.integrate(eq, tf, dt0)
    assert eq.t == tf and abs(eq.steps_taken - 100) <= 1
    out = eq.state.peek()
    assert not np.isnan(out).any()
    d = np.abs(fo.vals.astype(np.float64) - out.astype(np.float64)).max()
    assert d <= (1e-10 if dtype == np.float64 else 1e-4), d
    assert np.array_equal(np.sign(fo.vals), np.sign(out))
    assert np.array_equal(H.cut_cells(fo.vals), H.cut_cells(out))


@pytest.mark.gpu
@pytest.mark.parametrize("integ,fills", [("ForwardEuler", lambda n: n), ("RK2", lambda n: n + 1), ("RK3", lambda n: 3 * n)])
def test_launch_accounting(m, integ, fills):
    """A time-dependent expression needs no CFL pass: the fill that materialises it at the CFL time reduces the maximum, and a stage
    at the next step's CFL time (RK2's tc + dt) serves that request too."""
    ctx = m.default_context()
    I = getattr(m, integ)
    phi = _phi0(m, 2, np.float64)
    eq = m.LevelSetEquation(terms=_terms(m, "adv2d_weno", True), ic=phi, integrator=I())
    eq.state.device()
    ctx.reset_counters()
    m.integrate(eq, 0.05)
    c = ctx.counters()
    n = eq.steps_taken
    assert n >= 3 and c["cfl_passes"] == 0 and c["resident_steps"] == 0
    assert c["stage_launches"] == I.nstages * n
    assert c["kernel_launches"] == c["stage_launches"] + fills(n), (c, n)


@pytest.mark.gpu
def test_graph_option_and_hooked_loop_are_invisible(m):
    """OPT_GRAPH on and off give identical states (a captured fill would freeze t), and a prehook run (host loop through
    lsm_compute_cfl / lsm_stage) equals the one-call run."""
    ctx = m.default_context()
    res = []
    for on, hook in ((1, False), (0, False), (1, True)):
        ctx.set_option(m._lib.OPT_GRAPH, on)
        try:
            eq = _run(m, "adv_curv", m.RK3, np.float64, True, tf_steps=20.5, **({"prehook": lambda e: None} if hook else {}))
        finally:
            ctx.set_option(m._lib.OPT_GRAPH, 1)
        res.append((eq.t, eq.steps_taken, eq.state.peek().copy()))
    for r in res[1:]:
        assert r[:2] == res[0][:2] and np.array_equal(r[2], res[0][2])


@pytest.mark.gpu
def test_errors(m):
    """NaN in the expression raises CFLError like the host callable; TimeScaled(DeviceExpr), a wrong component count, a time
    factor on LSM_COEF_EXPR and a field of another context are refused."""
    with pytest.raises(m.CFLError):
        _run_nan = _phi0(m, 2, np.float64)
        m.integrate(m.LevelSetEquation(terms=(m.AdvectionTerm(m.DeviceExpr(("sqrt(-1.0 - t)", "x1"))),), ic=_run_nan), 0.1)
    with pytest.raises(m.CFLError):
        with np.errstate(invalid="ignore"):
            m.integrate(m.LevelSetEquation(terms=(m.AdvectionTerm(lambda x, t: (np.sqrt(-1.0 - t + 0 * x[0]), x[0])),),
                                           ic=_phi0(m, 2, np.float64)), 0.1)
    with pytest.raises(ValueError):
        m.TimeScaled(m.DeviceExpr(("-x2", "x1")), ("cos", 3.0))
    phi = _phi0(m, 2, np.float64)
    with pytest.raises(ValueError):
        m.compute_cfl((m.AdvectionTerm(m.DeviceExpr("x1")),), phi, 0.0)
    # C level: a time factor, a field without expressions, a field of another context
    lib, L = m._lib.lib(), m._lib
    ctx = m.default_context()
    grid = phi.mesh
    f = m.MeshField.from_expr(grid, ("-x2", "x1"))
    plain = m.MeshField(np.zeros((2,) + grid.n), grid)
    other = m.Context(0)
    try:
        g = m.MeshField.from_expr(grid, ("-x2", "x1"), ctx=other)
        for field, ts, why in ((f, L.TS_COS, "no time factor"), (plain, L.TS_NONE, "attached expressions"), (g, L.TS_NONE, "another context")):
            t = (L.lsm_term * 1)()
            t[0].kind, t[0].scheme, t[0].coef_kind, t[0].tscale_kind, t[0].tparam, t[0].field = L.TERM_ADVECTION, L.WENO5, L.COEF_EXPR, ts, 3.0, field.device()
            dt = C.c_double()
            rc = lib.lsm_compute_cfl(ctx.handle, phi.device(), t, 1, 0.0, None, C.byref(dt))
            assert rc == L.ERR_ARG and why in L.last_error(), (why, rc, L.last_error())
        assert lib.lsm_field_fill_expr(plain.device(), 0.0) == L.ERR_ARG
        del g
    finally:
        other.close()


@pytest.mark.gpu
def test_multi_gpu_expression_matches_single_gpu(m):
    """integrate_multi with a time-dependent expression on 2 ranks == the 1-GPU run bit for bit (each rank materialises its slab,
    the CFL maximum goes through the all-reduce)."""
    n = C.c_int32(0)
    m._lib.lib().lsm_device_count(C.byref(n))
    if n.value < 2:
        pytest.skip("needs 2 GPUs")
    mc = m.MultiContext([0, 1])
    solo = m.Context(0)
    try:
        expr = m.DeviceExpr(_flow(3)[0])

        def build(ctx):
            phi = _phi0(m, 3, np.float64, ctx=ctx)
            return m.LevelSetEquation(terms=(m.AdvectionTerm(expr, m.WENO5()),), ic=phi, integrator=m.RK3())
        ref = build(solo)
        tf = 8.5 * 0.5 * m.compute_cfl(ref.terms, ref.state, 0.0)
        m.integrate(ref, tf)
        eqs = [build(c) for c in mc.ranks]
        m.integrate_multi(mc, eqs, tf)
        got = m.MultiContext.gather([e.state for e in eqs])
        assert eqs[0].t == ref.t and eqs[0].steps_taken == ref.steps_taken
        assert np.array_equal(got, ref.state.peek())
    finally:
        mc.close()
        solo.close()
