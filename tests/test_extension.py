"""Closest-point extension (lsm_extend_closest_point, extend_closest_point).

Without a GPU: the NumPy restatement (extension_ref.py) against hand-computed 1-D and 2-D values, its value at the closest point
in every region of Ericson's routine and on degenerate triangles (a linear F comes back as the linear function at the point, a
constant F exactly), its points against redistance_ref's bit for bit, and the argument checks of the C ABI that need no device.
On the GPU: the device F equals the restatement bit for bit over dimensions, dtypes (mixed too), bands, odd sizes, anisotropic and
mirrored grids, the Zalesak disk, exact zeros, NaN nodes in phi and NaN in F, and a field without an interface; redistance=True
writes lsm_redistance's phi; a constant F is kept; second-order accuracy on a sphere; determinism; asynchrony; invalidation of the
CFL cache; the prehook; error codes."""
import ctypes as C
import math

import numpy as np
import pytest

import extension_ref as E
import redistance_ref as R
from zero_set_helpers import BAND_CASES, CASES, bits_equal, grid_h, m, on_device, sphere, zalesak  # noqa: F401 (m is a fixture)


def same(a, b):
    """Bit-equal, except that any NaN matches any NaN (the payload of a NaN computed from a NaN in F is not part of the contract)."""
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype != b.dtype or a.shape != b.shape or not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    v = ~np.isnan(a)
    return bits_equal(a[v], b[v])


def smooth(n, lc, h):
    """A smooth F on the grid: g(x) = sin(3 x1) + x2^2 - 0.5 x3 (fewer terms in 1-D / 2-D)."""
    x = R.node_coords(n, lc, h)
    return g_of(x)


def g_of(x):
    out = np.sin(3.0 * x[..., 0])
    if x.shape[-1] > 1:
        out = out + x[..., 1] ** 2
    if x.shape[-1] > 2:
        out = out - 0.5 * x[..., 2]
    return out


# ================================================================================================
# the restatement (no GPU)
# ================================================================================================
def test_1d_hand_computed():
    phi = np.array([-1.0, 3.0, 2.0, -0.5, np.nan, 1.0, 0.0, 4.0])
    F = np.array([0.0, 4.0, 8.0, 16.0, 32.0, 64.0, 128.0, 256.0])
    # nodes at 1.0, 1.5, ..., 4.5.  Crossings and their values: 1.125 (t = 0.25: 0 + 0.25 * 4 = 1), 2.4 (t = 0.8: 8 + 0.8 * 8),
    # 4.0 twice (cell 5, t = 1: 64 + 1 * 64 = 128; cell 6, t = -0: 128)
    out, phi_out, nb = E.extend(F, phi, [1.0], [0.5], band=3)
    want = [1.0, 1.0, 8.0 + 0.8 * 8.0, 8.0 + 0.8 * 8.0, 32.0, 128.0, 128.0, 128.0]
    assert np.array_equal(out, want)              # the NaN node keeps its F
    assert nb == 8 and bits_equal(phi_out, phi)
    out1, _, nb1 = E.extend(F, phi, [1.0], [0.5], band=1)
    assert nb1 == 7 and bits_equal(out1, out)


def test_2d_hand_computed():
    # phi = -1 on the column i1 = 0 and +1 on i1 = 1: the interface is x1 = 0.5, cut into segments by the triangulation's diagonals
    phi = np.array([[-1.0, -1.0, -1.0], [1.0, 1.0, 1.0]])
    F = 10.0 * np.arange(3.0)[None, :] + 100.0 * np.arange(2.0)[:, None]          # F[i1, i2] = 100 i1 + 10 i2
    # vertices: (0.5, j) on the edge (0, j)-(1, j), F = 10 j + 50; (0.5, j + 0.5) on the diagonal (0, j)-(1, j + 1), F = 10 j + 55.
    # Node (i1, j) has closest point (0.5, j), a vertex, so it gets 10 j + 50 exactly.
    out, _, nb = E.extend(F, phi, [0.0, 0.0], [1.0, 1.0])
    assert nb == 6
    assert np.array_equal(out, np.array([[50.0, 60.0, 70.0]] * 2))
    # an oblique straight interface: the mesh is exact, so a linear F comes back as F at the orthogonal projection
    n, lc, h = (23, 19), (-1.0, -0.8), (2.0 / 22, 1.6 / 18)
    x = R.node_coords(n, lc, h)
    nrm = np.array([0.6, 0.8])
    phi = x @ nrm - 0.1
    lin = lambda y: 0.3 + 2.0 * y[..., 0] - 1.5 * y[..., 1]
    out, _, _ = E.extend(lin(x), phi, lc, h)
    proj = x - (x @ nrm - 0.1)[..., None] * nrm
    inside = np.all((proj >= np.array(lc) + 1e-12) & (proj <= np.array(lc) - 1e-12 + np.array(h) * (np.array(n) - 1)), axis=-1)
    near = inside & (np.abs(phi) < 3 * min(h))                          # band nodes hold their exact closest point
    assert near.sum() > 100
    assert np.allclose(out[near], lin(proj)[near], rtol=0, atol=1e-13)


def _regions(A, B, Cc, q):
    """For each closest point q in triangle (A, B, Cc): 'vertex' / 'edge' / 'face' from its barycentric weights."""
    G = np.stack([B - A, Cc - A], axis=1)
    uv = np.linalg.lstsq(G, (q - A).T, rcond=None)[0].T
    w = np.stack([1 - uv[:, 0] - uv[:, 1], uv[:, 0], uv[:, 1]], axis=1)
    return np.abs(w) < 1e-12


def test_value_in_every_region_of_ericson():
    rng = np.random.default_rng(7)
    A, B, Cc = np.array([0.0, 0.0, 0.0]), np.array([1.0, 0.1, 0.2]), np.array([0.3, 0.9, -0.1])
    p = rng.uniform(-1.0, 2.0, (3000, 3))
    bc = lambda z: np.broadcast_to(z, p.shape)
    lin = lambda y: 0.7 - 1.3 * y[..., 0] + 0.4 * y[..., 1] + 2.1 * y[..., 2]
    f = [np.full(len(p), lin(v)) for v in (A, B, Cc)]
    q, fq = E.closest_triangle(p, bc(A), bc(B), bc(Cc), *f)
    assert bits_equal(q, R.closest_triangle(p, bc(A), bc(B), bc(Cc)))       # the point is redistance_ref's
    assert np.allclose(fq, lin(q), rtol=0, atol=1e-14)                      # a linear F: the linear function at the point
    zero = _regions(A, B, Cc, q)
    nz = zero.sum(1)
    for k in range(3):
        at_vertex = (nz == 2) & ~zero[:, k]
        on_edge = (nz == 1) & zero[:, k]
        assert at_vertex.sum() > 0 and on_edge.sum() > 0
        assert np.array_equal(fq[at_vertex], f[k][at_vertex])             # vertex regions return the vertex value itself
    assert np.sum(nz == 0) > 0, "the face region"
    const = np.full(len(p), -3.7)
    _, fc = E.closest_triangle(p, bc(A), bc(B), bc(Cc), const, const, const)
    assert np.all(fc == -3.7)                                               # a constant F exactly, in every region
    # 2-D segments: both end regions, the interior, and a segment that is a point
    x = rng.uniform(-1, 2, (500, 2))
    lin2 = lambda y: 1.5 - 0.25 * y[..., 0] + 0.75 * y[..., 1]
    for a, b in ((np.array([0.1, -0.2]), np.array([0.9, 0.4])), (np.array([0.3, 0.3]), np.array([0.3, 0.3]))):
        a2, b2 = np.broadcast_to(a, x.shape), np.broadcast_to(b, x.shape)
        q2, f2 = E.closest_segment(x, a2, b2, np.full(len(x), lin2(a)), np.full(len(x), lin2(b)))
        assert bits_equal(q2, R.closest_segment(x, a2, b2))
        assert np.allclose(f2, lin2(q2), rtol=0, atol=1e-14)
        assert np.array_equal(f2[np.all(q2 == a, axis=-1)], np.full(np.sum(np.all(q2 == a, axis=-1)), lin2(a)))
        const = np.full(len(x), 1.5)
        assert np.all(E.closest_segment(x, a2, b2, const, const)[1] == 1.5)


@pytest.mark.parametrize("kind", ["a_eq_b", "a_eq_c", "b_eq_c", "point"])
def test_value_on_degenerate_triangles(kind):
    rng = np.random.default_rng(3)
    a, e = np.array([0.2, -0.1, 0.3]), np.array([0.7, 0.4, -0.2])
    a, b, c = {"a_eq_b": (a, a, e), "a_eq_c": (a, e, a), "b_eq_c": (a, e, e), "point": (a, a, a)}[kind]
    p = rng.uniform(-1.0, 2.0, (400, 3))
    bc = lambda z: np.broadcast_to(z, p.shape)
    lin = lambda y: -0.4 + 0.9 * y[..., 0] + 1.7 * y[..., 1] - 0.6 * y[..., 2]
    f = [np.full(len(p), lin(v)) for v in (a, b, c)]
    q, fq = E.closest_triangle(p, bc(a), bc(b), bc(c), *f)
    assert bits_equal(q, R.closest_triangle(p, bc(a), bc(b), bc(c)))
    assert not np.any(np.isnan(fq))
    assert np.allclose(fq, lin(q), rtol=0, atol=1e-14)
    const = np.full(len(p), 2.25)
    assert np.all(E.closest_triangle(p, bc(a), bc(b), bc(c), const, const, const)[1] == 2.25)


@pytest.mark.parametrize("name", list(BAND_CASES))
def test_points_are_redistance_ref_points(name):
    phi, lc, h = BAND_CASES[name]
    F = smooth(phi.shape, lc, h)
    V, cell = R.primitives(phi, lc, h)
    V2, cell2, FV = E.primitives(phi, F, lc, h)
    assert bits_equal(V, V2) and np.array_equal(cell, cell2) and FV.shape == V.shape[:2]
    for band in (1, 3):
        P, val, is_band = E.band_phase(phi, F, lc, h, band)
        P0, is_band0 = R.band_phase(phi, lc, h, band)
        assert bits_equal(P, P0) and np.array_equal(is_band, is_band0)
        assert np.array_equal(np.isnan(val), np.isnan(P[..., 0]))
        Pf, valf = E.propagate(P, val, lc, h)
        assert bits_equal(Pf, R.propagate(P0, lc, h))
    out, phi_out, nb = E.extend(F, phi, lc, h, redistance=True)
    want, nb0 = R.redistance(phi, lc, h)
    assert nb == nb0 and bits_equal(phi_out, want)
    # near the interface F is F at a point within about h of the node's exact closest point: close to F at the node itself
    near = np.abs(want) < 0.5 * min(abs(v) for v in h)
    assert np.abs(out - F)[near].max() < 4 * max(abs(v) for v in h)


def test_constant_and_without_interface():
    phi, h = sphere((14, 13, 15), r=0.3)
    lc = (-0.5,) * 3
    for dtype in (np.float64, np.float32):
        F = np.full(phi.shape, 0.37, dtype=dtype)
        out, _, nb = E.extend(F, phi, lc, h)
        assert nb > 0 and bits_equal(out, F)
    F = smooth(phi.shape, lc, h)
    out, phi_out, nb = E.extend(F, phi + 2.0, lc, h, redistance=True)
    assert nb == 0 and bits_equal(out, F) and bits_equal(phi_out, phi + 2.0)


def test_abi_argument_checks_without_a_device(m):
    lib, L = m._lib.lib(), m._lib
    nb = C.c_int64(-1)
    assert lib.lsm_extend_closest_point(None, None, None, 0, 0, C.byref(nb)) == L.ERR_ARG and "band" in L.last_error()
    assert lib.lsm_extend_closest_point(None, None, None, -2, 1, None) == L.ERR_ARG
    assert lib.lsm_extend_closest_point(None, None, None, 3, 0, None) == L.ERR_ARG and "null" in L.last_error()
    # F is phi is refused before either handle is looked at (a zeroed host buffer stands in for the handles)
    buf = C.create_string_buffer(256)
    h = C.cast(buf, C.c_void_p)
    assert lib.lsm_extend_closest_point(h, h, h, 3, 0, None) == L.ERR_ARG and "must not be phi" in L.last_error()
    assert nb.value == -1


# ================================================================================================
# device == restatement, bit for bit
# ================================================================================================
def _run(m, F, phi, band, redistance=0):
    """lsm_extend_closest_point through the C ABI with the band-node count; returns (F, phi, band nodes)."""
    ctx = phi._context()
    nb = C.c_int64(-1)
    m._lib.check(m._lib.lib().lsm_extend_closest_point(ctx.handle, F.device(), phi.device(), band, redistance, C.byref(nb)))
    F._mark_device_advanced()
    phi._mark_device_advanced()
    return np.array(F.peek()), np.array(phi.peek()), nb.value


def _f_case(name, vals, lc, hc):
    h = grid_h(lc, hc, vals.shape)
    F = smooth(vals.shape, lc, h)
    if name == "3d_zeros_nan":                # NaN in F as well as in phi
        F[10:13, 4:6, 9] = np.nan
        F[20, 3:5, 14:16] = np.nan
    return F, h


DTYPES = {"f64": (np.float64, np.float64), "f32": (np.float32, np.float32), "phi64_F32": (np.float64, np.float32),
          "phi32_F64": (np.float32, np.float64)}


@pytest.mark.gpu
@pytest.mark.parametrize("band", [3, 1])
@pytest.mark.parametrize("dt", list(DTYPES))
@pytest.mark.parametrize("name", list(CASES))
def test_device_equals_restatement(m, name, dt, band):
    pd, fd = DTYPES[dt]
    vals, lc, hc = CASES[name]
    vals = vals.astype(pd)
    F, h = _f_case(name, vals, lc, hc)
    F = F.astype(fd)
    got, phi_got, nb = _run(m, on_device(m, F, lc, hc, fd), on_device(m, vals, lc, hc, pd), band)
    want, _, nb_want = E.extend(F, vals, lc, h, band)
    assert nb == nb_want
    assert same(got, want)
    assert bits_equal(phi_got, vals)                  # phi is not written without redistance
    if name == "3d_all_positive":
        assert nb == 0 and bits_equal(got, F)


@pytest.mark.gpu
@pytest.mark.parametrize("band", [2, 5])
def test_device_equals_restatement_wider_bands(m, band):
    for name in ("1d", "2d_odd_aniso", "3d_notched_sphere"):
        vals, lc, hc = CASES[name]
        F, h = _f_case(name, vals, lc, hc)
        got, _, nb = _run(m, on_device(m, F, lc, hc, np.float64), on_device(m, vals, lc, hc, np.float64), band)
        want, _, nb_want = E.extend(F, vals, lc, h, band)
        assert nb == nb_want and same(got, want), name


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_zalesak_disk_equals_restatement(m, dtype):
    phi, g = zalesak(m, 101, dtype)
    before = np.array(phi.peek())
    F0 = smooth(g.n, g.lc, g.meshsize()).astype(dtype)
    F = m.MeshField(np.asfortranarray(F0), g)
    assert m.extend_closest_point(F, phi) is F
    want, _, _ = E.extend(F0, before, g.lc, g.meshsize())
    assert bits_equal(np.array(F.peek()), want) and bits_equal(np.array(phi.peek()), before)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["2d_mirrored", "3d_odd_aniso", "3d_zeros_nan"])
def test_redistance_flag_writes_lsm_redistance_phi(m, name):
    vals, lc, hc = CASES[name]
    F, _ = _f_case(name, vals, lc, hc)
    f1, phi1, nb1 = _run(m, on_device(m, F, lc, hc, np.float64), on_device(m, vals, lc, hc, np.float64), 3, redistance=1)
    f0, phi0, nb0 = _run(m, on_device(m, F, lc, hc, np.float64), on_device(m, vals, lc, hc, np.float64), 3, redistance=0)
    ref = on_device(m, vals, lc, hc, np.float64)
    m.redistance(ref)
    assert bits_equal(phi1, np.array(ref.peek()))     # phi is lsm_redistance's, bit for bit
    assert same(f1, f0) and nb1 == nb0 and bits_equal(phi0, vals)


@pytest.mark.gpu
def test_constant_F_is_kept(m):
    for name in ("2d_odd_aniso", "3d_notched_sphere", "3d_zeros_nan"):
        vals, lc, hc = CASES[name]
        for dtype in (np.float64, np.float32):
            F0 = np.full(vals.shape, -1.25, dtype=dtype)
            F = on_device(m, F0, lc, hc, dtype)
            m.extend_closest_point(F, on_device(m, vals, lc, hc, np.float64), redistance=True)
            assert bits_equal(np.array(F.peek()), F0), name


# ================================================================================================
# accuracy, determinism, asynchrony, invalidation, prehook, errors
# ================================================================================================
@pytest.mark.gpu
def test_second_order_on_a_sphere(m):
    c, r0 = np.array([0.02, -0.01, 0.0]), 0.3
    errs = []
    for n in (64, 128):
        g = m.CartesianGrid((-0.5,) * 3, (0.5,) * 3, (n, n, n))
        x = R.node_coords(g.n, g.lc, g.meshsize())
        rel = x - c
        r = np.sqrt((rel[..., 0] ** 2 + rel[..., 1] ** 2) + rel[..., 2] ** 2)
        phi = m.MeshField(np.asfortranarray(r * r - r0 * r0), g)
        F = m.MeshField(np.asfortranarray(g_of(x)), g)
        m.extend_closest_point(F, phi)
        exact = g_of(c + r0 * rel / r[..., None])                       # g at the exact closest point of the sphere
        # the error grows with the distance d to the interface (facet normals are O(h) off, so the closest point moves by about
        # d * O(h) along the surface); within a fixed multiple of h it is second order.  The restatement gives orders 1.99, 1.96
        # and 1.74 within h, 2h and 3h: at 3h the 128^3 band edge is still pre-asymptotic.
        near = np.abs(r - r0) < 2 * g.meshsize(1)
        errs.append(float(np.abs(np.array(F.peek()) - exact)[near].max()))
    order = math.log2(errs[0] / errs[1])
    print("max |F - g(closest point)| within 2h:", errs, "order", order)
    assert order > 1.8, errs                 # the restatement: 2.98e-3 and 7.68e-4, order 1.96


@pytest.mark.gpu
def test_deterministic_and_asynchronous(m):
    vals, lc, hc = CASES["3d_notched_sphere"]
    F0, _ = _f_case("3d_notched_sphere", vals, lc, hc)
    ctx = m.default_context()
    fa, fb = on_device(m, F0, lc, hc, np.float64), on_device(m, F0, lc, hc, np.float64)
    pa, pb = on_device(m, vals, lc, hc, np.float64), on_device(m, vals, lc, hc, np.float64)
    for f in (fa, fb, pa, pb):
        f.device()
    ctx.reset_counters()
    m.extend_closest_point(fa, pa, redistance=True)
    c = ctx.counters()
    assert c["d2h_bytes"] == 0 and c["h2d_bytes"] == 0
    assert c["kernel_launches"] == 5 + len(R.flood_steps(vals.shape))     # flag, 2 cell passes, pick, flooding, write
    nb = C.c_int64(-1)
    m._lib.check(m._lib.lib().lsm_extend_closest_point(ctx.handle, fb.device(), pb.device(), 3, 1, C.byref(nb)))
    fb._mark_device_advanced()
    pb._mark_device_advanced()
    assert ctx.counters()["d2h_bytes"] == 8 and nb.value > 0          # one 8-byte copy of the band-node count
    assert bits_equal(np.array(fa.peek()), np.array(fb.peek())) and bits_equal(np.array(pa.peek()), np.array(pb.peek()))


@pytest.mark.gpu
def test_cfl_cache_sees_new_values(m):
    g = m.CartesianGrid((-1.0, -1.0), (1.0, 1.0), (65, 61))
    x = R.node_coords(g.n, g.lc, g.meshsize())
    phi = m.MeshField(np.asfortranarray(np.hypot(x[..., 0], x[..., 1]) - 0.5), g, bc=m.NeumannBC())
    speed = m.MeshField(np.asfortranarray(3.0 * (x[..., 0] ** 2 + x[..., 1] ** 2) - 0.2 + x[..., 0]), g)
    terms = (m.NormalMotionTerm(speed),)
    dt0 = m.compute_cfl(terms, phi, 0.0)
    m.compute_cfl(terms, phi, 0.0)           # served from the cache
    m.extend_closest_point(speed, phi)
    fresh = m.MeshField(np.array(speed.peek(), order="F"), g)
    dt1 = m.compute_cfl(terms, phi, 0.0)
    assert dt1 == m.compute_cfl((m.NormalMotionTerm(fresh),), phi, 0.0) and dt1 != dt0


@pytest.mark.gpu
def test_prehook_equals_explicit_loop(m):
    g = m.CartesianGrid((-0.5,) * 3, (0.5,) * 3, (40, 38, 42))
    x = R.node_coords(g.n, g.lc, g.meshsize())
    r = np.sqrt(((x[..., 0] - 0.02) ** 2 + (x[..., 1] + 0.01) ** 2) + x[..., 2] ** 2)
    ic = m.MeshField(np.asfortranarray(r * r - 0.09), g, bc=m.NeumannBC())
    ctx = m.default_context()
    speeds = [m.MeshField(np.asfortranarray(0.5 + 0.3 * x[..., 0] - 0.2 * x[..., 2]), g, bc=m.NeumannBC()) for _ in range(2)]
    eqs = [m.LevelSetEquation(terms=(m.NormalMotionTerm(v),), ic=ic, integrator=m.RK3()) for v in speeds]
    tf = 0.05
    for e, v in zip(eqs, speeds):
        e.state.device()
        v.device()
    ctx.reset_counters()
    m.integrate(eqs[0], tf, prehook=lambda ls: m.extend_closest_point(speeds[0], ls.state, redistance=True))
    c = ctx.counters()
    assert c["h2d_bytes"] == 0                                         # neither field left the device
    e, v = eqs[1], speeds[1]
    phi, tc, steps = e.state, 0.0, 0
    while tc <= tf - float(np.spacing(abs(tc))):
        m.extend_closest_point(v, phi, redistance=True)
        dt = min(math.inf, e.integrator.cfl * m.compute_cfl(e.terms, phi, tc), tf - tc)
        m.api._advance(e.integrator, phi, e.terms, tc, dt)
        tc += dt
        steps += 1
    assert steps == eqs[0].steps_taken >= 3
    assert bits_equal(np.array(eqs[0].state.peek()), np.array(phi.peek()))
    assert bits_equal(np.array(speeds[0].peek()), np.array(v.peek()))


@pytest.mark.gpu
def test_error_codes(m):
    lib, L = m._lib.lib(), m._lib
    fresh = m.Context(0)
    try:
        g = m.CartesianGrid((0, 0), (1, 1), (9, 8))
        sc = m.MeshField(np.zeros((9, 8)) - 1, g, ctx=fresh)
        F = m.MeshField(np.ones((9, 8)), g, ctx=fresh)
        vec = m.MeshField(np.zeros((2, 9, 8)), g, ctx=fresh)
        assert lib.lsm_extend_closest_point(fresh.handle, vec.device(), sc.device(), 3, 0, None) == L.ERR_ARG
        assert lib.lsm_extend_closest_point(fresh.handle, F.device(), vec.device(), 3, 0, None) == L.ERR_ARG
        sep = m.SeparableVelocity(g, (1.0, 1.0), [[np.ones(9), np.ones(8)], [np.ones(9), np.ones(8)]], ctx=fresh)
        assert lib.lsm_extend_closest_point(fresh.handle, sep.device(), sc.device(), 3, 0, None) == L.ERR_ARG
        thin_g = m.CartesianGrid((0, 0), (1, 1), (9, 1))
        thin, thin_f = (m.MeshField(np.zeros((9, 1)), thin_g, ctx=fresh) for _ in range(2))
        assert lib.lsm_extend_closest_point(fresh.handle, thin_f.device(), thin.device(), 3, 0, None) == L.ERR_ARG
        for other in (m.CartesianGrid((0, 0), (1, 1), (9, 9)), m.CartesianGrid((0, 0.5), (1, 1.5), (9, 8)),
                      m.CartesianGrid((0, 0), (1, 2), (9, 8)), m.CartesianGrid((0, 0, 0), (1, 1, 1), (9, 8, 2))):
            mis = m.MeshField(np.ones(other.n), other, ctx=fresh)              # another n, lc, h or dimension
            assert lib.lsm_extend_closest_point(fresh.handle, mis.device(), sc.device(), 3, 0, None) == L.ERR_ARG
            assert "same grid" in L.last_error()
        assert lib.lsm_extend_closest_point(fresh.handle, sc.device(), sc.device(), 3, 0, None) == L.ERR_ARG
        assert lib.lsm_extend_closest_point(fresh.handle, F.device(), sc.device(), 0, 0, None) == L.ERR_ARG
        other_ctx = m.MeshField(np.ones((9, 8)), g)
        assert lib.lsm_extend_closest_point(fresh.handle, other_ctx.device(), sc.device(), 3, 0, None) == L.ERR_ARG
        assert lib.lsm_extend_closest_point(fresh.handle, F.device(), sc.device(), 3, 0, None) == L.OK
        with pytest.raises(m.LSMError):
            m.extend_closest_point(F, sc, band=0)
        del vec, sep, thin, thin_f, sc, F, mis
    finally:
        fresh.close()

