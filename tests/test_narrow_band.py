"""Narrow-band fields (lsm_field_set_band) on the device against the NumPy restatement of the band rules and a masked oracle step.

Every comparison with the oracle runs one step at a time and advances the oracle with the band the device reports for that step
(lsm_field_band before the step), so that a last-bit difference between the two sides cannot move a brick in or out of the band.
"""
import ctypes as C

import numpy as np
import pytest

import helpers as H
import narrow_band_ref as NB

pytestmark = pytest.mark.gpu

OPT_KERNEL = 0
BCS = {"periodic": ("periodic",), "neumann": ("neumann",), "extrap2": ("extrap", 2), "symmetry": ("symmetry",)}
DTYPES = {"f64": np.float64, "f32": np.float32}
BAR_STRICT = {"f64": 1e-13, "f32": 2e-6}          # strict kernel vs oracle where pow() is involved (test_tiled_multitile.py)
BAR_TILED = {"f64": 1e-10, "f32": 1e-4}


@pytest.fixture(scope="module")
def m():
    import lsm_b200
    return lsm_b200


@pytest.fixture
def kernel(m):
    ctx = m.default_context()
    yield lambda k: ctx.set_option(OPT_KERNEL, k)
    ctx.set_option(OPT_KERNEL, 0)


def corner_case(n, bc, dtype, terms="adv_weno"):
    """A sphere near the low corner of an anisotropic box (so that some bricks are frozen), stored coefficients of every kind."""
    N = len(n)
    lc, hc, _, u, v, b = H.small_problem(n)
    X = H.coords(lc, hc, n)
    phi = H.bcast(np.sqrt(sum((x + 0.55) ** 2 for x in X)) - 0.3, n)
    sets = H.small_termsets(u, v, b, N)
    return H.Case(terms, lc, hc, n, phi, sets[terms], bc, dtype)


def periodic_axes(case):
    fo = case.oracle_field()
    return [fo.bc[d][0][0] == 0 for d in range(fo.ndim)]          # BC_PERIODIC == 0


def fetch(phi):
    info = phi.band_info()
    return info["states"], (info["core"], info["active"], info["shell"])


def check_band(phi, case, w):
    st, counts = fetch(phi)
    ref = NB.band_states(phi.peek(), phi.mesh.meshsize(), w, periodic_axes(case))
    assert np.array_equal(st, ref), np.argwhere(st != ref)[:5]
    assert counts == (int((ref == 3).sum()), int((ref >= 2).sum()), int((ref == 1).sum()))
    return st


def engine_step(m, phi, terms, integ, tc, dt):
    import lsm_b200.api as A
    low = A._Lowered(terms, phi, tc)
    lib = m._lib
    lib.check(lib.lib().lsm_advance(phi._context().handle, H.INTEG[integ], phi.device(), low.arr, len(terms), float(tc), float(dt)))
    phi._mark_device_advanced()


def band_run(m, O, case, integ, steps, w, check_states=False):
    """`steps` steps of the band field and of the masked oracle; returns (oracle state, engine state, initial state, ever-active)."""
    fo, to = case.oracle_field(), case.oracle_terms()
    phi = m.NarrowBandMeshField(case.engine_field(m), halfwidth=w)
    terms = case.engine_terms(m, phi)
    dt = 0.5 * O.compute_cfl(fo, to, 0.0)
    ever = np.zeros(case.n, dtype=bool)
    tc = 0.0
    for _ in range(steps):
        st = check_band(phi, case, w) if check_states else fetch(phi)[0]
        act = NB.node_mask(st, case.n)
        ever |= act
        NB.masked_step(O, fo, H.INTEG[integ], to, tc, dt, act)
        engine_step(m, phi, terms, integ, tc, dt)
        tc += dt
    if check_states:
        check_band(phi, case, w)
    return fo.vals, phi.peek().copy(), case.phi0, ever


# ---- band states: the device against the restatement -------------------------------------------------------------------
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("bc", BCS)
@pytest.mark.parametrize("n", [(100, 70), (513, 40), (70, 52, 45), (97, 40, 33)])
def test_band_states_match_the_restatement(m, O, n, bc, dt):
    case = corner_case(n, BCS[bc], DTYPES[dt])
    band_run(m, O, case, "RK3", 3, 3.0, check_states=True)


# ---- the strict kernel: the masked oracle, bit for bit where IEEE arithmetic is all that is involved ---------------------
STRICT = [(n, t, i, bc) for n in [(100, 52), (70, 40, 36)] for t in ("adv_weno", "adv_upwind", "normal", "curv", "eik_live", "three")
          for i in ("FE", "RK2", "RK3") for bc in BCS]


@pytest.mark.parametrize("n,terms,integ,bc", STRICT)
def test_strict_kernel_equals_masked_oracle(m, O, kernel, n, terms, integ, bc):
    kernel(1)
    case = corner_case(n, BCS[bc], np.float64, terms)
    a, b, p0, ever = band_run(m, O, case, integ, 3, 2.0)
    if "curv" in terms or "three" in terms:
        assert np.abs(a - b).max() <= BAR_STRICT["f64"]
    else:
        assert np.array_equal(a, b)
    assert np.array_equal(b[~ever], p0[~ever])


# ---- the tiled kernel after 50 RK3 steps ---------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("n,terms,bc", [((100, 70), "adv_weno", "periodic"), ((100, 70), "three", "neumann"),
                                        ((70, 52, 45), "adv_weno", "neumann"), ((70, 52, 45), "normal_adv", "symmetry"),
                                        ((97, 40, 33), "adv_curvc", "extrap2")])
def test_tiled_kernel_against_masked_oracle(m, O, kernel, n, terms, bc, dt):
    kernel(3)
    case = corner_case(n, BCS[bc], DTYPES[dt], terms)
    a, b, p0, ever = band_run(m, O, case, "RK3", 50, 3.0)
    scale = max(1.0, float(np.abs(a).max()))
    assert np.abs(a.astype(np.float64) - b.astype(np.float64)).max() / scale <= BAR_TILED[dt]
    assert np.array_equal(b[~ever], p0[~ever]), "nodes that were never active changed"
    assert (~ever).any(), "the case has no frozen nodes"


# ---- an all-core band is the dense field ---------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [3, 1])
@pytest.mark.parametrize("integ", ["FE", "RK2", "RK3"])
@pytest.mark.parametrize("n", [(100, 70), (70, 52, 45)])
def test_all_core_band_equals_dense(m, kernel, n, integ, k):
    kernel(k)
    case = corner_case(n, BCS["neumann"], np.float64, "normal_adv")
    tf = 1e-2
    dense = H.run_engine(m, case, integ, tf)
    phi = m.NarrowBandMeshField(case.engine_field(m), halfwidth=1e6)
    eq = m.LevelSetEquation(terms=case.engine_terms(m, phi), ic=phi, integrator=getattr(m, {"FE": "ForwardEuler"}.get(integ, integ))(0.5))
    assert isinstance(eq.state, m.NarrowBandMeshField)
    m.integrate(eq, tf)
    info = eq.state.band_info()
    assert info["core"] == info["states"].size
    assert eq.steps_taken == dense.steps_taken and eq.t == dense.t
    assert np.array_equal(eq.state.peek(), dense.state.peek())


# ---- rebuilds --------------------------------------------------------------------------------------------------------------
def test_full_scans(m, O):
    ctx = m.default_context()
    case = corner_case((70, 52, 45), BCS["neumann"], np.float64, "adv_weno")
    phi = m.NarrowBandMeshField(case.engine_field(m), halfwidth=3)
    eq = m.LevelSetEquation(terms=case.engine_terms(m, phi), ic=phi, integrator=m.RK3())
    dt0 = 0.5 * O.compute_cfl(case.oracle_field(), case.oracle_terms(), 0.0)
    ctx.reset_counters()
    m.integrate(eq, 20 * dt0 * (1 - 1e-12))
    c = ctx.counters()
    assert eq.steps_taken == 20 and c["band_full_scans"] == 1 and c["resident_steps"] == 0
    check_band(eq.state, case, 3)
    assert ctx.counters()["band_full_scans"] == 1, "a query after band steps rescans only the active bricks"
    state = eq.state
    # every other write to phi costs a full scan at the next step, whose band is the restatement's
    lib = m._lib
    moved = np.asfortranarray(np.roll(case.phi0, 20, axis=0))

    def upload():
        state.vals[...] = moved

    def fill():
        lib.check(lib.lib().lsm_field_fill_shape(state.device(), lib.SHAPE_SPHERE, (C.c_double * 4)(-0.6, -0.6, -0.6, 0.3), 4))
        state._mark_device_advanced()

    def redistance():
        m.redistance(state)

    writes = [upload, fill, redistance]
    for k, write in enumerate(writes):
        write()
        before = ctx.counters()["band_full_scans"]
        m.integrate(eq, eq.t + dt0 * (1 - 1e-12))
        assert ctx.counters()["band_full_scans"] == before + 1, k
        check_band(state, case, 3)
        assert ctx.counters()["band_full_scans"] == before + 1, k


# ---- agreement with the dense field (the reference's narrow-band-vs-full-grid check) ----------------------------------------
def rotation_case(n):
    lc, hc, nn = (-1, -1, -1), (1, 1, 1), (n, n, n)
    x, y, z = H.coords(lc, hc, nn)
    phi = np.sqrt((x - 0.5) ** 2 + y * y + z * z) - 0.25
    u = np.stack([H.bcast(-y, nn), H.bcast(x, nn), np.zeros(nn)], axis=0)
    return H.Case("rotation", lc, hc, nn, phi, [dict(kind="advection", field=u)], ("neumann",))


# max |phi_band - phi_dense| where |phi_dense| <= 2h, and the relative difference of the level-set integrals.  Measured on a B200:
# rotation 1.1e-10 and 3.1e-12, Enright 2.9e-11 and 2.3e-12 (84 and 100 of 256 bricks active after 100 steps)
AGREE_BAR = {"rotation": (1e-9, 1e-10), "enright": (1e-9, 1e-10)}


@pytest.mark.parametrize("name", ["rotation", "enright"])
def test_band_agrees_with_dense(m, O, name):
    case = rotation_case(128) if name == "rotation" else H.c3_enright(128)
    dt0 = 0.5 * O.compute_cfl(case.oracle_field(), case.oracle_terms(), 0.0)
    tf = 100 * dt0 * (1 - 1e-12)
    dense = H.run_engine(m, case, "RK3", tf)
    phi = m.NarrowBandMeshField(case.engine_field(m), halfwidth=3)
    eq = m.LevelSetEquation(terms=case.engine_terms(m, phi), ic=phi, integrator=m.RK3())
    m.integrate(eq, tf)
    assert eq.steps_taken == dense.steps_taken == 100
    a, b = dense.state.peek(), eq.state.peek()
    h = case.oracle_field().meshsize()[0]
    near = np.abs(a) <= 2 * h
    d = float(np.abs(a - b)[near].max())
    ia, ib = m.level_set_integrals(dense.state), m.level_set_integrals(eq.state)
    rel = max(abs(ia.inside - ib.inside) / ia.inside, abs(ia.interface - ib.interface) / ia.interface)
    info = eq.state.band_info()
    print(f"\n{name} 128^3, 100 RK3 steps, halfwidth 3: max|phi_band - phi_dense| (|phi_dense| <= 2h) = {d:.3e}, "
          f"integrals rel. diff = {rel:.3e} (inside {ia.inside:.9f} / {ib.inside:.9f}, interface {ia.interface:.9f} / "
          f"{ib.interface:.9f}), active bricks {info['active']} / {info['states'].size}")
    assert d <= AGREE_BAR[name][0] and rel <= AGREE_BAR[name][1]


# ---- refusals and the Python path --------------------------------------------------------------------------------------------
def test_refusals(m):
    lib = m._lib
    L = lib.lib()
    g2 = m.CartesianGrid((0, 0), (1, 1), (40, 40))
    phi = m.MeshField(np.zeros((40, 40)), g2, bc=m.NeumannBC())
    h = phi.device()
    for w in (-1.0, float("nan"), float("inf")):
        assert L.lsm_field_set_band(h, w) == lib.ERR_ARG
    counts = (C.c_int64 * 3)()
    assert L.lsm_field_band(h, counts, None) == lib.ERR_ARG          # no band
    g1 = m.CartesianGrid((0,), (1,), (40,))
    assert L.lsm_field_set_band(m.MeshField(np.zeros(40), g1).device(), 3.0) == lib.ERR_UNSUPPORTED
    vec = m.MeshField(np.zeros((2, 40, 40)), g2)
    assert L.lsm_field_set_band(vec.device(), 3.0) == lib.ERR_UNSUPPORTED
    with pytest.raises(m.LSMError):
        m.NarrowBandMeshField(vec)
    band = m.NarrowBandMeshField(phi, halfwidth=2)
    eq = m.LevelSetEquation(terms=(m.AdvectionTerm((1.0, 0.5)),), ic=band, integrator=m.SemiImplicit())
    with pytest.raises(m.LSMError) as e:
        m.integrate(eq, 0.01)
    assert e.value.code == lib.ERR_UNSUPPORTED
    assert L.lsm_field_set_band(band.device(), 0.0) == lib.OK           # off again: a dense field
    assert L.lsm_field_band(band.device(), counts, None) == lib.ERR_ARG


def test_python_copy_keeps_the_band(m, O):
    case = corner_case((100, 70), BCS["periodic"], np.float64, "adv_weno")
    phi = m.NarrowBandMeshField(case.engine_field(m), halfwidth=2.5)
    eq = m.LevelSetEquation(terms=case.engine_terms(m, phi), ic=phi, integrator=m.RK2())
    m.integrate(eq, 0.05)
    c = eq.state.copy()
    assert isinstance(c, m.NarrowBandMeshField) and c.halfwidth == 2.5
    assert np.array_equal(c.peek(), eq.state.peek())
    check_band(c, case, 2.5)
    assert eq.state.band_info()["active"] < eq.state.band_info()["states"].size
