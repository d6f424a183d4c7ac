"""Time-scaled coefficients through the sign change of their factor, on every stage-kernel family, against the CPU oracle.

C3 (Enright), the single vortex and every ``TimeScaled(base, ("cos", T))`` term multiply a velocity, speed or curvature coefficient
by g(t) = cos(pi t / T).  Past t = T/2 the factor is negative and the flow runs backwards.  The sign of u g chooses the upwind WENO5
stencil, and each kernel family forms it its own way: the sign bits of u and g in lsm_tiled.cu, lsm_pair3d.cu and lsm_pair2d.cu,
v * g in the strict kernel; on an isotropic mesh the 3-D x-pair kernel folds g / h into the stage coefficient, and with a normal
term it scales the speed by that term's own factor.  Near T/2, |g| is tiny and the CFL step is huge.

1. Reversal windows: dt0 = half the CFL step at t = 0 (where g = 1), T = 6 dt0, 8 steps with dt_max = dt0 from t0 = 0 or from
   T/2 - 1.5 dt0.  |g| <= 1 keeps every step at dt0, a stage time lands on T/2 and g reaches -1 (test_windows_cross_the_reversal
   checks this with the oracle alone), so the window never takes the huge steps.
2. The single step that a tiny |g| selects without dt_max, the CFL candidates on and off, and one coefficient field shared by two
   terms with different factors (one CFL memo per field).
3. The host-callable factor against the device one, factors of exactly +0.0 and -0.0, and a NaN factor.
4. Whole periods of the Enright deformation (3-D) and of the single vortex (2-D): the shape comes back, the engine stays at the
   BASELINE bar of the oracle.

Every difference is measured relative to max(1, max|phi|) of the reference state; every engine run asserts from the counters which
kernel family ran its stages, so no case passes on a fallback to another kernel.
"""
import ctypes as C
import functools
import math

import numpy as np
import pytest

import helpers as H
import integrals_ref as IR
import test_tiled_multitile as TM

OPT_KERNEL, OPT_CAND = 0, 6
STEPS = 8
# (integrator, t0): t0 = 0 puts the stage time 3 dt0 on T/2 for every integrator; t0 = T/2 - 1.5 dt0 reaches T/2 through the
# half-step stage of RK3
WINDOWS = (("FE", 0), ("RK2", 0), ("RK3", 0), ("RK3", 1))
NSTAGES = {"FE": 1, "RK2": 2, "RK3": 3}
DTYPES = {"f64": np.float64, "f32": np.float32}
BAR_STRICT = {"f64": 1e-13, "f32": 2e-6}
BAR_TILED = {"f64": 1e-10, "f32": 1e-4}


@pytest.fixture(scope="module")
def m():
    import lsm_b200
    return lsm_b200


@pytest.fixture(scope="module")
def fast_oracle(O):
    O.set_threads(O.max_threads())
    return O


# ---- windows ---------------------------------------------------------------------------------------------------------
def timed(case, T):
    """`case` with the factor cos(pi t / T) on every term."""
    terms = [dict(t, cos_period=T) for t in case.terms]
    return H.Case(case.name, case.lc, case.hc, case.n, case.phi0, terms, case.bc, case.dtype)


def dt_half(O, case):
    """Half the CFL step at t = 0, where every factor is cos(0) = 1."""
    return 0.5 * O.compute_cfl(case.oracle_field(), case.oracle_terms(), 0.0)


def window(O, case, offset):
    """(timed case, t0, tf, dt0) of the reversal window of `case`."""
    dt0 = dt_half(O, case)
    T = 6 * dt0
    t0 = T / 2 - 1.5 * dt0 if offset else 0.0
    return timed(case, T), t0, t0 + STEPS * dt0 * (1 - 1e-12), dt0


def stage_factors(O, case, integ, t0, tf, dt_max):
    """orc_integrate's loop replayed with the oracle's CFL: (step sizes, the factor of every term at every stage time)."""
    fo, to = case.oracle_field(), case.oracle_terms()
    tc, dts, gs = t0, [], []
    while tc <= tf - np.spacing(abs(tc)):
        dt = min(dt_max, 0.5 * O.compute_cfl(fo, to, tc), tf - tc)
        for ts in {"FE": (tc,), "RK2": (tc, tc + dt), "RK3": (tc, tc + dt, tc + 0.5 * dt)}[integ]:
            gs += [O.lib().orc_tscale(C.byref(t.c()), ts) for t in to]
        dts.append(dt)
        tc += dt
    return dts, gs


# ---- runs ------------------------------------------------------------------------------------------------------------
def run_oracle(O, case, integ, t0, tf, dt_max=math.inf):
    fo = case.oracle_field()
    t, n = O.integrate(fo, H.INTEG[integ], case.oracle_terms(), tf, t0=t0, dt_max=dt_max)
    return t, n, fo.vals


def run(m, case, integ, t0, tf, dt_max=math.inf, kernel=0, terms=None):
    """Integrate `case` from t0 to tf through LSM_OPT_KERNEL = kernel; `terms(m, phi)` replaces the case's engine terms.
    Returns (t, steps, state, counters)."""
    ctx = m.default_context()
    ctx.set_option(OPT_KERNEL, kernel)
    try:
        ctx.reset_counters()
        phi = case.engine_field(m)
        eq = m.LevelSetEquation(terms=(terms or case.engine_terms)(m, phi), ic=phi, t=t0,
                                integrator=getattr(m, {"FE": "ForwardEuler"}.get(integ, integ))())
        m.integrate(eq, tf, dt_max)
        return eq.t, eq.steps_taken, eq.state.peek().copy(), ctx.counters()
    finally:
        ctx.set_option(OPT_KERNEL, 0)


def ran(out, integ, pair, what):
    """Every stage of the run `out` went to the x-pair kernel (pair) or none did."""
    _, n, _, c = out
    assert c["stage_launches"] == NSTAGES[integ] * n and c["resident_steps"] == 0, (what, "stage launches", c)
    assert c["pair_launches"] == (c["stage_launches"] if pair else 0), (what, "x-pair launches", c["pair_launches"], c["stage_launches"])


def rel(a, b):
    """(max |a - b| / max(1, max|a|), location of the worst node); a NaN counts as the worst.  Grids of 2-D and 3-D name the
    tile seams of the worst node (test_tiled_multitile.where), 1-D ones its index."""
    d = np.abs(a.astype(np.float64) - b.astype(np.float64))
    worst = np.unravel_index(np.argmax(np.where(np.isnan(d), np.inf, d)), d.shape)
    loc = TM.where(worst, a.shape) if a.ndim > 1 else f"worst node {int(worst[0])} of {a.shape[0]}"
    return float(np.max(d)) / max(1.0, float(np.abs(a).max())), loc


def label(integ, off):
    return f"{integ}{'@T/2-1.5dt0' if off else ''}"


# ---- term lists ------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=4)
def small_sets(n):
    """Grid, phi0 and the term lists of the strict and tiled windows on an n grid (no factor yet): every coefficient kind of
    every term kind and the multi-term lists of the stage kernels, each coefficient changing sign in space."""
    lc, hc, phi, u, v, b = H.small_problem(n)
    N = len(n)
    ts = H.small_termsets(u, v, b, N)
    X = [x.ravel() for x in H.coords(lc, hc, n)]
    tabs = [[np.sin(2 * X[a] + d) + 0.2 if a == d else np.cos(X[a] - 0.5 * d) for a in range(N)] for d in range(N)]
    sep, c = ((1.0, -0.7, 0.5)[:N], tabs), tuple([0.7, -0.4, 0.5][:N])
    sets = {k: ts[k] for k in ("adv_weno", "adv_upwind")}
    sets["adv_sep"] = [dict(kind="advection", separable=sep)]
    sets["adv_sep_upwind"] = [dict(kind="advection", separable=sep, scheme="upwind")]
    sets["adv_const"] = [dict(kind="advection", const=c)]
    sets["adv_const_upwind"] = [dict(kind="advection", const=c, scheme="upwind")]
    sets.update({k: ts[k] for k in ("normal", "normal_const", "curv", "curv_const", "three", "normal_adv")})
    return lc, hc, phi, sets


SMALL_SETS = list(small_sets((8, 8))[3])


def small_case(n, termset, dt, bcs=H.SMALL_BCS, split=H.SMALL_SPLIT):
    lc, hc, phi, sets = small_sets(n)
    return H.Case(termset, lc, hc, n, phi, sets[termset], H.small_bc(SMALL_SETS.index(termset), len(n), bcs, split), DTYPES[dt])


@functools.lru_cache(maxsize=2)
def pair3d_sets(n):
    """The Enright-type deformation of test_pair_kernel_bitwise_vs_tiled (shifted tables: sign changes in every direction, no
    exact zeros) as a stored and as a separable velocity, and C5's list (stored speed with sign changes, stored velocity)."""
    lc, hc = (0, 0, 0), (1, 1, 1)
    x, y, z = H.coords(lc, hc, n)
    phi = np.sqrt((x - 0.45) ** 2 + (y - 0.5) ** 2 + (z - 0.55) ** 2) - 0.25 + 0.03 * np.sin(7 * x) * np.cos(5 * y) * np.sin(6 * z)
    sc, tabs = H.enright_tables(lc, hc, n)
    tabs = [[t + 0.05 * (a + 1) for a, t in enumerate(row)] for row in tabs]
    X, Y, Z = np.meshgrid(*[np.arange(k) for k in n], indexing="ij", sparse=True)
    u = np.stack([((sc[d] * tabs[d][0][X]) * tabs[d][1][Y]) * tabs[d][2][Z] for d in range(3)], axis=0)
    v = H.bcast(0.2 * np.sin(4 * x + 1) * np.cos(3 * y) + 0.1 * z - 0.05, n)
    return lc, hc, H.bcast(phi, n), {"adv": [dict(kind="advection", field=u)],
                                     "adv_sep": [dict(kind="advection", separable=(sc, tabs))],
                                     "normal_adv": [dict(kind="normal", field=v), dict(kind="advection", field=u)]}


def pair3d_case(n, termset, dt, bc=("neumann",)):
    lc, hc, phi, sets = pair3d_sets(n)
    return H.Case(termset, lc, hc, n, phi, sets[termset], bc, DTYPES[dt])


@functools.lru_cache(maxsize=2)
def pair2d_problem(n):
    """test_pair2d_kernel_vs_tiled's notched circle (kinks for the curvature term) and rotation-like velocity."""
    lc, hc = (-1.0, -1.0), (1.0, 1.0)
    x, y = H.coords(lc, hc, n)
    phi = np.hypot(x - 0.1, y + 0.05) - 0.45 + 0.03 * np.sin(9 * x) * np.cos(7 * y)
    phi = np.maximum(phi, -(np.maximum(np.abs(x - 0.1) - 0.08, np.abs(y + 0.4) - 0.3)))
    u = np.stack([H.bcast(-y + 0.2 * np.sin(5 * x), n), H.bcast(x + 0.1 * np.cos(4 * y), n)], axis=0)
    return lc, hc, H.bcast(phi, n), u


def pair2d_case(n, curv, dt, bc=("neumann",)):
    lc, hc, phi, u = pair2d_problem(n)
    terms = [dict(kind="advection", field=u)] + ([dict(kind="curvature", const=-0.01)] if curv else [])
    return H.Case("adv_curv" if curv else "adv", lc, hc, n, phi, terms, bc, DTYPES[dt])


# ---- section 1: the matrices -----------------------------------------------------------------------------------------
STRICT_GRIDS = ((40,), (26, 22), (14, 12, 13))
STRICT = [(n, ts, dt) for n in STRICT_GRIDS for ts in SMALL_SETS for dt in DTYPES]

TILED = [(s, dt, bs, ts) for s in TM.SHAPES for dt in DTYPES for bs in TM.BCSETS for ts in SMALL_SETS]

PAIR_SHAPES = [(128, 64, 40), (72, 52, 37), (64, 8, 8), (200, 30, 70), (136, 9, 130)]
PAIR_BCS = [("neumann",), ("periodic",), ("symmetry",),
            ((("neumann",), ("symmetry",)), ("periodic",), (("symmetry",), ("neumann",)))]
PAIR = [(n, b, dt, ts) for n in PAIR_SHAPES for b in range(len(PAIR_BCS)) for dt in DTYPES for ts in ("adv", "adv_sep", "normal_adv")
        if not (dt == "f32" and (n[0] % 4 or ts == "normal_adv"))]

ISO_N = (48, 48, 48)
ISO = [(dt, ts, b) for dt in DTYPES for ts in ("adv", "adv_sep", "normal_adv") for b in (0, 1) if not (dt == "f32" and ts == "normal_adv")]

PAIR2D_SHAPES = [(256, 96), (520, 70), (40, 33), (1032, 24)]
PAIR2D_BCS = [("neumann",), ("periodic",), ("symmetry",), ((("neumann",), ("symmetry",)), ("periodic",))]
PAIR2D = [(n, b, dt, curv) for n in PAIR2D_SHAPES for b in range(len(PAIR2D_BCS)) for dt in DTYPES for curv in (False, True)
          if not (dt == "f32" and n[0] % 4)]


def _rot(k):
    return WINDOWS[k % len(WINDOWS)]


def section1_windows():
    """(name, untimed case, windows) of every reversal window the GPU tests of section 1 run."""
    for n, ts, dt in STRICT:
        yield f"strict-{len(n)}d-{ts}-{dt}", small_case(n, ts, dt), WINDOWS
    for k, (s, dt, bs, ts) in enumerate(TILED):
        yield f"tiled-{s}-{dt}-{bs}-{ts}", tiled_case(s, dt, bs, ts), (_rot(k),)
    for k, (n, b, dt, ts) in enumerate(PAIR):
        yield f"pair3d-{n}-{b}-{dt}-{ts}", pair3d_case(n, ts, dt, PAIR_BCS[b]), (_rot(k),)
    for dt, ts, b in ISO:
        yield f"iso-{dt}-{ts}-{b}", pair3d_case(ISO_N, ts, dt, PAIR_BCS[b]), WINDOWS
    for k, (n, b, dt, curv) in enumerate(PAIR2D):
        yield f"pair2d-{n}-{b}-{dt}-{curv}", pair2d_case(n, curv, dt, PAIR2D_BCS[b]), (_rot(k),)


def tiled_case(shape, dt, bcset, termset):
    n = TM.SHAPES[shape]
    lc, hc, phi, sets = small_sets(n)
    bcs, split = TM.BCSETS[bcset]
    return H.Case(termset, lc, hc, n, phi, sets[termset], H.small_bc(SMALL_SETS.index(termset), len(n), bcs, split), DTYPES[dt])


def test_windows_cross_the_reversal(O):
    """Without a GPU: in every window of section 1 all steps but the (shortened) last are exactly dt0, the factors of the stage
    times take both signs, and one stage time lands on T/2 (|g| < 1e-3)."""
    count = 0
    for name, case, wins in section1_windows():
        for integ, off in wins:
            tcase, t0, tf, dt0 = window(O, case, off)
            dts, gs = stage_factors(O, tcase, integ, t0, tf, dt0)
            assert len(dts) == STEPS and all(d == dt0 for d in dts[:-1]) and dt0 * (1 - 1e-9) < dts[-1] <= dt0, (name, integ, off, dts)
            assert max(gs) > 0.5 and min(gs) < -0.5, (name, integ, off, gs)
            assert min(abs(g) for g in gs) < 1e-3, (name, integ, off, gs)
            count += 1
    assert count == len(STRICT) * len(WINDOWS) + len(TILED) + len(PAIR) + len(ISO) * len(WINDOWS) + len(PAIR2D)


@pytest.mark.gpu
@pytest.mark.parametrize("n,termset,dt", STRICT, ids=[f"{len(n)}d-{ts}-{dt}" for n, ts, dt in STRICT])
def test_strict_kernel_reversal(m, O, n, termset, dt):
    """The strict kernel (1), the reference's operation order, against the oracle at rounding level through every window."""
    case = small_case(n, termset, dt)
    lines = []
    for integ, off in WINDOWS:
        tcase, t0, tf, dt0 = window(O, case, off)
        t_o, n_o, a = run_oracle(O, tcase, integ, t0, tf, dt0)
        out = run(m, tcase, integ, t0, tf, dt0, kernel=1)
        assert out[:2] == (t_o, n_o) and n_o == STEPS, (integ, off, out[:2], t_o, n_o)
        ran(out, integ, False, "strict")
        d, loc = rel(a, out[2])
        assert d <= BAR_STRICT[dt], f"{termset} {label(integ, off)}: {d:.3e} > {BAR_STRICT[dt]:.0e} ({loc})"
        lines.append(f"{label(integ, off)} {d:.2e}")
    print(f"TSCALE strict {len(n)}d-{termset}-{dt}: " + ", ".join(lines))


@pytest.mark.gpu
@pytest.mark.parametrize("shape,dt,bcset,termset", TILED, ids=["-".join(c) for c in TILED])
def test_tiled_kernel_reversal(m, fast_oracle, shape, dt, bcset, termset):
    """The tiled kernel alone (3) on grids of many tiles (test_tiled_multitile.SHAPES) against the oracle: the BASELINE bar."""
    O = fast_oracle
    integ, off = _rot(TILED.index((shape, dt, bcset, termset)))
    tcase, t0, tf, dt0 = window(O, tiled_case(shape, dt, bcset, termset), off)
    t_o, n_o, a = run_oracle(O, tcase, integ, t0, tf, dt0)
    out = run(m, tcase, integ, t0, tf, dt0, kernel=3)
    assert out[:2] == (t_o, n_o) and n_o == STEPS
    ran(out, integ, False, "tiled")
    d, loc = rel(a, out[2])
    assert d <= BAR_TILED[dt], f"{label(integ, off)}: {d:.3e} > {BAR_TILED[dt]:.0e} ({loc})"
    print(f"TSCALE tiled {shape}-{dt}-{bcset}-{termset} {label(integ, off)}: {d:.3e} (bar {BAR_TILED[dt]:.0e})")


@pytest.mark.gpu
@pytest.mark.parametrize("n,b,dt,termset", PAIR, ids=[f"{'x'.join(map(str, n))}-bc{b}-{dt}-{ts}" for n, b, dt, ts in PAIR])
def test_pair3d_kernel_reversal(m, fast_oracle, n, b, dt, termset):
    """The 3-D x-pair kernel with the exact epsilon maximum (4) performs the tiled kernel's operations (anisotropic meshes: no
    folded scaling), so one-term lists must give BIT-IDENTICAL states through the sign change of g.  C5's list, with the speed
    and the velocity both time-scaled, shares differences between its two terms and stays within 1e-12, as in
    test_pair_kernel_two_terms_vs_tiled.  The default mode (0) is within 1e-12 (Float64) and bit-identical (Float32) of the
    tiled kernel (3), which is held to the BASELINE bar of the oracle."""
    O = fast_oracle
    integ, off = _rot(PAIR.index((n, b, dt, termset)))
    tcase, t0, tf, dt0 = window(O, pair3d_case(n, termset, dt, PAIR_BCS[b]), off)
    t_o, n_o, a = run_oracle(O, tcase, integ, t0, tf, dt0)
    outs = {k: run(m, tcase, integ, t0, tf, dt0, kernel=k) for k in (4, 3, 0)}
    for k, o in outs.items():
        assert o[:2] == (t_o, n_o) and n_o == STEPS, (k, o[:2], t_o, n_o)
        ran(o, integ, k != 3, f"kernel {k}")
    d3, loc = rel(a, outs[3][2])
    assert d3 <= BAR_TILED[dt], f"tiled vs oracle {d3:.3e} ({loc})"
    d4, loc4 = rel(outs[3][2], outs[4][2])
    d0, loc0 = rel(outs[3][2], outs[0][2])
    if termset == "normal_adv":
        assert d4 <= 1e-12, f"exact-epsilon x-pair vs tiled {d4:.3e} ({loc4})"
    else:
        assert np.array_equal(outs[4][2], outs[3][2]), f"exact-epsilon x-pair vs tiled {d4:.3e} ({loc4})"
    if dt == "f64":
        assert d0 <= 1e-12, f"default vs tiled {d0:.3e} ({loc0})"
    else:
        assert np.array_equal(outs[0][2], outs[3][2]), f"default vs tiled {d0:.3e} ({loc0})"
    print(f"TSCALE pair3d {n}-bc{b}-{dt}-{termset} {label(integ, off)}: tiled vs oracle {d3:.3e}, exact-eps vs tiled {d4:.3e}, "
          f"default vs tiled {d0:.3e}")


@pytest.mark.gpu
@pytest.mark.parametrize("dt,termset,b", ISO, ids=[f"{dt}-{ts}-bc{b}" for dt, ts, b in ISO])
def test_pair3d_iso_reversal(m, fast_oracle, dt, termset, b):
    """The default 3-D x-pair kernel on a cube, where it folds c g / h into the stage coefficient (and, with C5's list, scales
    the speed by the normal term's own factor), against the oracle through every window: the BASELINE bar."""
    O = fast_oracle
    case = pair3d_case(ISO_N, termset, dt, PAIR_BCS[b])
    lines = []
    for integ, off in WINDOWS:
        tcase, t0, tf, dt0 = window(O, case, off)
        t_o, n_o, a = run_oracle(O, tcase, integ, t0, tf, dt0)
        out = run(m, tcase, integ, t0, tf, dt0, kernel=0)
        assert out[:2] == (t_o, n_o) and n_o == STEPS
        ran(out, integ, True, "iso x-pair")
        d, loc = rel(a, out[2])
        assert d <= BAR_TILED[dt], f"{label(integ, off)}: {d:.3e} > {BAR_TILED[dt]:.0e} ({loc})"
        lines.append(f"{label(integ, off)} {d:.2e}")
    print(f"TSCALE iso48 {dt}-{termset}-bc{b}: " + ", ".join(lines))


@pytest.mark.gpu
@pytest.mark.parametrize("n,b,dt,curv", PAIR2D, ids=[f"{'x'.join(map(str, n))}-bc{b}-{dt}-{'adv_curv' if c else 'adv'}" for n, b, dt, c in PAIR2D])
def test_pair2d_kernel_reversal(m, fast_oracle, n, b, dt, curv):
    """The 2-D x-pair kernel (2: forced, also below its size threshold) against the tiled kernel (3) through the sign change of
    the velocity's factor and of the constant curvature's: within 1e-13 (Float64) / 1e-6 (Float32), as
    test_pair2d_kernel_vs_tiled claims; the tiled kernel against the oracle at the BASELINE bar."""
    O = fast_oracle
    integ, off = _rot(PAIR2D.index((n, b, dt, curv)))
    tcase, t0, tf, dt0 = window(O, pair2d_case(n, curv, dt, PAIR2D_BCS[b]), off)
    t_o, n_o, a = run_oracle(O, tcase, integ, t0, tf, dt0)
    outs = {k: run(m, tcase, integ, t0, tf, dt0, kernel=k) for k in (2, 3)}
    for k, o in outs.items():
        assert o[:2] == (t_o, n_o) and n_o == STEPS
        ran(o, integ, k == 2, f"kernel {k}")
    d3, loc = rel(a, outs[3][2])
    assert d3 <= BAR_TILED[dt], f"tiled vs oracle {d3:.3e} ({loc})"
    d2, loc2 = rel(outs[3][2], outs[2][2])
    assert d2 <= (1e-13 if dt == "f64" else 1e-6), f"x-pair vs tiled {d2:.3e} ({loc2})"
    print(f"TSCALE pair2d {n}-bc{b}-{dt}-{'adv_curv' if curv else 'adv'} {label(integ, off)}: tiled vs oracle {d3:.3e}, "
          f"x-pair vs tiled {d2:.3e}")


# ---- section 2: the step a tiny |g| selects; the CFL memo across the sign change -------------------------------------
BIG_STEP = {
    "3d-pair-c5-f64": (lambda: pair3d_case((64, 48, 40), "normal_adv", "f64"), True),
    "3d-pair-adv-f32": (lambda: pair3d_case((64, 48, 40), "adv", "f32", PAIR_BCS[3]), True),
    "3d-iso-sep-f64": (lambda: pair3d_case(ISO_N, "adv_sep", "f64", ("periodic",)), True),
    "2d-tiled-adv_curv-f64": (lambda: pair2d_case((256, 96), True, "f64"), False),
    "2d-pair-adv-f64": (lambda: pair2d_case((512, 512), False, "f64", ("periodic",)), True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(BIG_STEP))
def test_tiny_factor_takes_one_clipped_step(m, fast_oracle, name):
    """No dt_max, first step at T/2 - 1e-3 dt0: |g| ~ 5e-4 makes the CFL step ~2000 dt0, so the loop clips it to tf - t0 = 4 dt0
    and takes ONE step.  The default kernels must take the same step (time and count) and land within the BASELINE bar."""
    O = fast_oracle
    mk, pair = BIG_STEP[name]
    case = mk()
    dt0 = dt_half(O, case)
    tcase = timed(case, 6 * dt0)
    t0 = 3 * dt0 - 1e-3 * dt0
    tf = t0 + 4 * dt0
    assert 0.5 * O.compute_cfl(tcase.oracle_field(), tcase.oracle_terms(), t0) > 1000 * dt0
    t_o, n_o, a = run_oracle(O, tcase, "RK3", t0, tf)
    assert n_o == 1
    out = run(m, tcase, "RK3", t0, tf)
    assert out[:2] == (t_o, n_o), (out[:2], t_o, n_o)
    ran(out, "RK3", pair, name)
    dt = "f64" if tcase.dtype == np.float64 else "f32"
    d, loc = rel(a, out[2])
    assert d <= BAR_TILED[dt], f"{d:.3e} ({loc})"
    print(f"TSCALE one clipped step {name}: {d:.3e} (bar {BAR_TILED[dt]:.0e})")


CAND = {
    "stored": lambda: H.c3_enright(40),
    "separable": lambda: H.c3_enright(40, separable=True),
    "normal-field": lambda: small_case((40, 36, 32), "normal", "f64"),
    "c5-f64": lambda: pair3d_case((64, 48, 40), "normal_adv", "f64"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CAND))
def test_cfl_candidates_through_the_reversal(m, fast_oracle, name):
    """Whole integrations through the reversal, with dt_max = dt0 and without, take the same steps and produce the same bits
    with the CFL candidates (LSM_OPT_CFL_CANDIDATES) on and off, and the steps of the oracle.  The CFL equals the oracle's bit
    for bit at a dense set of times around T/2, T/2 itself included, either way."""
    O = fast_oracle
    case = CAND[name]()
    dt0 = dt_half(O, case)
    T = 6 * dt0
    tcase = timed(case, T)
    fo, to = tcase.oracle_field(), tcase.oracle_terms()
    ts = [0.0, dt0, T / 2, T / 2 * (1 - 2 ** -52), T / 2 * (1 + 2 ** -52), T, 8 * dt0] + [T / 2 + k * 1e-3 * dt0 for k in range(-20, 21)]
    ts += [T / 2 + k * 1e-8 * dt0 for k in range(-5, 6)]
    want = [O.compute_cfl(fo, to, t) for t in ts]
    assert max(want) > 1e6 * dt0
    ctx = m.default_context()
    try:
        for cand in (1, 0):
            ctx.set_option(OPT_CAND, cand)
            phi = tcase.engine_field(m)
            terms = tcase.engine_terms(m, phi)
            got = [m.compute_cfl(terms, phi, t) for t in ts]
            bad = [(t, g, w) for t, g, w in zip(ts, got, want) if g != w]
            assert not bad, (cand, bad[:4])
        lines = []
        for dt_max in (dt0, math.inf):
            t_o, n_o, a = run_oracle(O, tcase, "RK3", 0.0, 8 * dt0, dt_max)
            outs = []
            for cand in (1, 0):
                ctx.set_option(OPT_CAND, cand)
                outs.append(run(m, tcase, "RK3", 0.0, 8 * dt0, dt_max))
            assert outs[0][:2] == outs[1][:2] == (t_o, n_o), (dt_max, outs[0][:2], outs[1][:2], t_o, n_o)
            assert np.array_equal(outs[0][2], outs[1][2]), (dt_max, rel(outs[0][2], outs[1][2]))
            d, loc = rel(a, outs[0][2])
            assert d <= BAR_TILED["f64"], (dt_max, d, loc)
            lines.append(f"dt_max={'dt0' if dt_max == dt0 else 'inf'}: {n_o} steps, {d:.3e}")
        print(f"TSCALE candidates {name}: " + ", ".join(lines))
    finally:
        ctx.set_option(OPT_CAND, 1)


SHARED = {"3d": (40, 36, 32), "2d": (100, 70)}


@pytest.mark.gpu
@pytest.mark.parametrize("dim", list(SHARED))
@pytest.mark.parametrize("second", ["cos-T2", "unscaled"])
def test_one_field_two_factors(m, fast_oracle, dim, second):
    """One stored velocity (one MeshField, hence one CFL memo) in two AdvectionTerms: factors cos(pi t / T1) and cos(pi t / T2),
    which change sign at different times, or cos(pi t / T1) and none.  The CFL equals the oracle's bit for bit at every step of
    the loop, with and without dt_max, and the integrated state is within the BASELINE bar."""
    O = fast_oracle
    n = SHARED[dim]
    lc, hc, phi0, u, _, _ = H.small_problem(n)
    base = H.Case("shared", lc, hc, n, phi0, [dict(kind="advection", field=u), dict(kind="advection", field=u)], ("neumann",))
    dt0 = dt_half(O, base)
    T1, T2 = 6 * dt0, 4 * dt0
    spec = [dict(kind="advection", field=u, cos_period=T1), dict(kind="advection", field=u)]
    if second == "cos-T2":
        spec[1]["cos_period"] = T2
    case = H.Case("shared", lc, hc, n, phi0, spec, ("neumann",))

    def terms(m, phi):
        U = m.MeshField(u, phi.mesh)
        return (m.AdvectionTerm(m.TimeScaled(U, ("cos", T1))), m.AdvectionTerm(m.TimeScaled(U, ("cos", T2)) if second == "cos-T2" else U))

    fo, to = case.oracle_field(), case.oracle_terms()
    lines = []
    for dt_max in (dt0, math.inf):
        tf = 8 * dt0
        phi = case.engine_field(m)
        et = terms(m, phi)
        tc, steps = 0.0, 0
        while tc <= tf - np.spacing(abs(tc)):
            want = O.compute_cfl(fo, to, tc)
            got = m.compute_cfl(et, phi, tc)
            assert got == want, (dt_max, steps, tc, got, want)
            tc += min(dt_max, 0.5 * want, tf - tc)
            steps += 1
        t_o, n_o, a = run_oracle(O, case, "RK3", 0.0, tf, dt_max)
        assert n_o == steps
        out = run(m, case, "RK3", 0.0, tf, dt_max, terms=terms)
        assert out[:2] == (t_o, n_o)
        ran(out, "RK3", False, "two terms")
        d, loc = rel(a, out[2])
        assert d <= BAR_TILED["f64"], (dt_max, d, loc)
        lines.append(f"dt_max={'dt0' if dt_max == dt0 else 'inf'}: {n_o} steps, {d:.3e}")
    print(f"TSCALE shared field {dim} {second}: " + ", ".join(lines))


# ---- section 3: host-callable factor, zero factors, NaN factor -------------------------------------------------------
def _with_coef(m, term, coef):
    if isinstance(term, m.AdvectionTerm):
        return m.AdvectionTerm(coef, term.scheme)
    return m.NormalMotionTerm(coef) if isinstance(term, m.NormalMotionTerm) else m.CurvatureTerm(coef)


def host_terms(case, f=None):
    """`case`'s engine terms with every device factor ("cos", T) replaced by the host callable f, by default the same
    t -> cos(pi t / T) that lsm_api.cu evaluates (same operations, same libm)."""
    def cos_of(T):
        return lambda t: math.cos(math.pi * t / T)

    def mk(m, phi):
        return tuple(_with_coef(m, t, m.TimeScaled(t._coef().base, f or cos_of(t._coef().g[1]))) for t in case.engine_terms(m, phi))
    return mk


FAMILIES = {
    # name: (case factory, LSM_OPT_KERNEL values, x-pair kernel expected)
    "pair3d-adv-f64": (lambda: pair3d_case((72, 52, 37), "adv", "f64"), (0, 4), True),
    "pair3d-c5-f64": (lambda: pair3d_case((72, 52, 37), "normal_adv", "f64", ("symmetry",)), (0, 4), True),
    "pair3d-iso-sep-f32": (lambda: pair3d_case(ISO_N, "adv_sep", "f32", ("periodic",)), (0,), True),
    "pair2d-adv_curv-f64": (lambda: pair2d_case((256, 96), True, "f64", PAIR2D_BCS[3]), (2,), True),
    "pair2d-adv-f32": (lambda: pair2d_case((520, 70), False, "f32", ("periodic",)), (2,), True),
    "tiled-3d-three-f64": (lambda: tiled_case("B", "f64", "extrap", "three"), (3,), False),
    "tiled-2d-sep_upwind-f32": (lambda: tiled_case("C", "f32", "remap", "adv_sep_upwind"), (3,), False),
    "strict-3d-three-f64": (lambda: small_case((14, 12, 13), "three", "f64"), (1,), False),
    "strict-2d-adv_sep-f32": (lambda: small_case((26, 22), "adv_sep", "f32"), (1,), False),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FAMILIES))
def test_host_factor_equals_device_factor(m, fast_oracle, name):
    """TimeScaled(u, lambda t: cos(pi t / T)) runs the Python loop (lsm_stage with a host factor per stage); TimeScaled(u, ("cos",
    T)) runs lsm_integrate.  Through every reversal window, and without dt_max from 0 across T/2, both take the same steps and
    produce the same bits."""
    O = fast_oracle
    mk, kernels, pair = FAMILIES[name]
    case = mk()
    for integ, off in WINDOWS + (("RK3", None),):
        tcase, t0, tf, dt0 = window(O, case, bool(off))
        dt_max = math.inf if off is None else dt0
        for k in kernels:
            dev = run(m, tcase, integ, t0, tf, dt_max, kernel=k)
            host = run(m, tcase, integ, t0, tf, dt_max, kernel=k, terms=host_terms(tcase))
            for o in (dev, host):
                ran(o, integ, pair and k != 3 and k != 1, f"kernel {k}")
            assert dev[:2] == host[:2], (integ, off, k, dev[:2], host[:2])
            assert np.array_equal(dev[2], host[2]), (integ, off, k, rel(dev[2], host[2]))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FAMILIES))
def test_zero_factor_is_a_fixed_point(m, O, name):
    """A factor of exactly +0.0 or -0.0 (-0.0 sets the sign bit that the stencil choice reads, with a zero scale): the CFL is
    inf, so dt = min(dt_max, tf - t), and a ForwardEuler or RK2 step leaves the state bit-identical on every kernel family."""
    mk, kernels, pair = FAMILIES[name]
    case = mk()
    dt0 = dt_half(O, case)
    tcase = timed(case, 1.0)
    for zero in (0.0, -0.0):
        f = lambda t, z=zero: z
        phi = tcase.engine_field(m)
        assert m.compute_cfl(host_terms(tcase, f)(m, phi), phi, 0.3) == math.inf
        for integ in ("FE", "RK2"):
            for k in kernels:
                out = run(m, tcase, integ, 0.0, 2 * dt0, dt0, kernel=k, terms=host_terms(tcase, f))
                ran(out, integ, pair and k not in (1, 3), f"kernel {k}")
                assert out[:2] == (2 * dt0, 2), out[:2]
                assert np.array_equal(out[2], tcase.phi0), (zero, integ, k, rel(tcase.phi0, out[2]))


@pytest.mark.gpu
def test_nan_factor_raises(m):
    """A factor that is NaN: compute_cfl and integrate raise CFLError and leave the state and the time as they were, also when
    the CFL candidates of the field were built by earlier requests, for a stored, a separable and a constant coefficient, and
    for the device factor cos(pi t / 0) (0/0 at t = 0)."""
    cases = [H.c3_enright(24), H.c3_enright(24, separable=True), small_case((26, 22), "normal_const", "f64"),
             small_case((26, 22), "curv", "f32")]
    for case in cases:
        tcase = timed(case, 1.0)
        phi = tcase.engine_field(m)
        et = host_terms(tcase, lambda t: math.nan if t >= 1.0 else math.cos(t))(m, phi)
        for t in (0.1, 0.2, 0.3, 0.4):           # the second request of a stored or separable field builds its candidates
            assert math.isfinite(m.compute_cfl(et, phi, t))
        with pytest.raises(m.CFLError):
            m.compute_cfl(et, phi, 1.0)
        eq = m.LevelSetEquation(terms=et, ic=phi, t=1.0, integrator=m.RK3())
        with pytest.raises(m.CFLError):
            m.integrate(eq, 1.5)
        assert eq.t == 1.0 and np.array_equal(eq.state.peek(), tcase.phi0)
        dev = timed(case, 0.0)
        phi = dev.engine_field(m)
        et = dev.engine_terms(m, phi)
        with pytest.raises(m.CFLError):
            m.compute_cfl(et, phi, 0.0)
        eq = m.LevelSetEquation(terms=et, ic=phi, integrator=m.RK3())
        with pytest.raises(m.CFLError):
            m.integrate(eq, 0.5)
        assert eq.t == 0.0 and np.array_equal(eq.state.peek(), dev.phi0)


# ---- section 4: whole periods --------------------------------------------------------------------------------------------
def single_vortex(n=512, T=0.5):
    """The single vortex: u = (-sin^2(pi x) sin(2 pi y), sin^2(pi y) sin(2 pi x)) cos(pi t / T) on [0, 1]^2, a disk of radius
    0.15 at (0.5, 0.75); the velocity vanishes on the boundary (Neumann)."""
    lc, hc, nn = (0, 0), (1, 1), (n, n)
    x, y = H.coords(lc, hc, nn)
    phi = np.hypot(x - 0.5, y - 0.75) - 0.15
    u = np.stack([H.bcast(-np.sin(np.pi * x) ** 2 * np.sin(2 * np.pi * y), nn), H.bcast(np.sin(np.pi * y) ** 2 * np.sin(2 * np.pi * x), nn)], axis=0)
    return H.Case("vortex", lc, hc, nn, H.bcast(phi, nn), [dict(kind="advection", field=u, cos_period=T)], ("neumann",))


PERIODS = {
    "enright-96-stored": lambda: H.c3_enright(96, period=0.5),
    "enright-96-separable": lambda: H.c3_enright(96, separable=True, period=0.5),
    "vortex-512": lambda: single_vortex(512, 0.5),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PERIODS))
def test_full_period_against_the_oracle(m, fast_oracle, name):
    """From t = 0 to T = 0.5, dt_max = dt0, RK3, Float64, default kernels (the x-pair kernels): the BASELINE bar, the sign and
    cut-cell classification of the oracle, and the device's level-set integrals of the engine's state equal to the NumPy
    restatement on the oracle's state within 1e-9 relative.  Prints the observed difference and the change of the area or volume
    over the period (the shape comes back)."""
    O = fast_oracle
    case = PERIODS[name]()
    T = case.terms[0]["cos_period"]
    dt0 = dt_half(O, case)
    t_o, n_o, a = run_oracle(O, case, "RK3", 0.0, T, dt0)
    out = run(m, case, "RK3", 0.0, T, dt0)
    assert out[:2] == (t_o, n_o)
    ran(out, "RK3", True, name)
    d = H.check_parity(a, out[2], 1e-10)
    h = [(case.hc[k] - case.lc[k]) / (case.n[k] - 1) for k in range(len(case.n))]
    g = case.engine_grid(m)
    got = m.level_set_integrals(m.MeshField(out[2], g))
    want = IR.integrals(a, case.lc, h)
    for k, what in enumerate(("inside", "interface")):
        assert abs(got[k] - want[k]) <= 1e-9 * abs(want[k]), (what, got[k], want[k])
    start = m.level_set_integrals(m.MeshField(case.phi0, g))
    what = "area" if len(case.n) == 2 else "volume"
    print(f"TSCALE full period {name}: {n_o} RK3 steps, max-abs diff {d:.3e} (bar 1e-10), {what} {start.inside:.6e} -> "
          f"{got.inside:.6e} ({(got.inside - start.inside) / start.inside:+.3e} relative)")
