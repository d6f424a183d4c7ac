"""Closest-point redistancing (lsm_redistance, redistance).

Without a GPU: the NumPy restatement (redistance_ref.py) against hand-computed 1-D distances, its closest-point routines against
dense sampling in every region of Ericson's algorithm and on degenerate triangles, the band guarantee against brute force over the
whole mesh, the propagated distances against brute force, classification (with the subnormal raise), and the argument checks of
the C ABI that need no device.  On the GPU: the device result equals the restatement bit for bit over dimensions, dtypes, odd
sizes, anisotropic and mirrored grids, bands, kinked shapes, exact zeros, NaN nodes and a field without an interface; second-order
accuracy on a sphere; the interface shift; determinism; asynchrony; invalidation of the CFL cache; the prehook; error codes.  On
2 GPUs: every single-rank zero-level-set entry point refuses a slab-decomposed field."""
import ctypes as C
import math

import numpy as np
import pytest

import redistance_ref as R
from zero_set_helpers import BAND_CASES, CASES, bits_equal, grid_h, m, on_device, sphere, zalesak  # noqa: F401 (m is a fixture)


# ================================================================================================
# the restatement (no GPU)
# ================================================================================================
def test_1d_hand_computed():
    phi = np.array([-1.0, 3.0, 2.0, -0.5, np.nan, 1.0, 0.0, 4.0])
    # nodes at 1.0, 1.5, ..., 4.5; crossings (extraction): 1.125 (cell 0), 2.4 (cell 2), 4.0 twice (cells 5 and 6)
    out, nb = R.redistance(phi, [1.0], [0.5], band=3)
    want = [-0.125, 0.375, 0.4, -0.1, np.nan, 0.5, -0.0, 0.5]
    assert np.allclose(out, want, rtol=0, atol=1e-15, equal_nan=True)
    assert out[0] == -0.125 and out[1] == 0.375 and out[5] == 0.5 and out[7] == 0.5       # dyadic: exact
    assert out[6] == 0.0 and np.signbit(out[6])                                           # s = 0 is inside: -0.0
    assert nb == 8                                    # every node is within 3 cells of a crossing (the NaN node keeps NaN)
    out1, nb1 = R.redistance(phi, [1.0], [0.5], band=1)
    # band 1: node i sees cells i-1..i; node 4 sees only cells 3 and 4, which touch the NaN node and hold nothing
    assert nb1 == 7 and bits_equal(out1, out)


def _tri_samples(a, b, c, k=300):
    u, v = np.meshgrid(np.linspace(0, 1, k + 1), np.linspace(0, 1, k + 1))
    m = u + v <= 1
    u, v = u[m], v[m]
    return a + u[:, None] * (b - a) + v[:, None] * (c - a)


def test_closest_point_segment_and_triangle_against_sampling():
    rng = np.random.default_rng(7)
    # segments (2-D), points around them
    a, b = np.array([0.1, -0.2]), np.array([0.9, 0.4])
    S = a + np.linspace(0, 1, 20001)[:, None] * (b - a)
    x = rng.uniform(-1, 2, (500, 2))
    q = R.closest_segment(x, np.broadcast_to(a, x.shape), np.broadcast_to(b, x.shape))
    dmin = np.sqrt(((x[:, None, :] - S[None]) ** 2).sum(-1)).min(1)
    d = R.dist(x, q)
    assert np.all(d <= dmin + 1e-12) and np.all(d >= dmin - 1e-4)
    # a triangle in 3-D and points in every Voronoi region of Ericson's algorithm (3 vertices, 3 edges, the face)
    A, B, Cc = np.array([0.0, 0.0, 0.0]), np.array([1.0, 0.1, 0.2]), np.array([0.3, 0.9, -0.1])
    T = _tri_samples(A, B, Cc)
    p = rng.uniform(-1.0, 2.0, (3000, 3))
    bc = lambda z: np.broadcast_to(z, p.shape)
    q = R.closest_triangle(p, bc(A), bc(B), bc(Cc))
    d = R.dist(p, q)
    dmin = np.concatenate([np.sqrt(((p[i:i + 200, None, :] - T[None]) ** 2).sum(-1)).min(1) for i in range(0, len(p), 200)])
    assert np.all(d <= dmin + 1e-12) and np.all(d >= dmin - 5e-3)
    # which region each answer came from: a vertex, an edge interior, or the face interior
    G = np.stack([B - A, Cc - A], axis=1)
    uv = np.linalg.lstsq(G, (q - A).T, rcond=None)[0].T
    w = np.stack([1 - uv[:, 0] - uv[:, 1], uv[:, 0], uv[:, 1]], axis=1)
    assert np.all(w > -1e-12) and np.allclose(A + uv @ G.T, q, atol=1e-12)        # every answer lies in the triangle
    zero = np.abs(w) < 1e-12
    nz = zero.sum(1)
    assert all(np.sum((nz == 2) & ~zero[:, k]) > 0 for k in range(3)), "every vertex region"
    assert all(np.sum((nz == 1) & zero[:, k]) > 0 for k in range(3)), "every edge region"
    assert np.sum(nz == 0) > 0, "the face region"


@pytest.mark.parametrize("kind", ["a_eq_b", "a_eq_c", "b_eq_c", "point"])
def test_closest_point_on_degenerate_triangles(kind):
    # the mesh's degenerate triangles have coincident vertices: exact zeros at nodes put two crossings on the same node
    rng = np.random.default_rng(3)
    a, e = np.array([0.2, -0.1, 0.3]), np.array([0.7, 0.4, -0.2])
    a, b, c = {"a_eq_b": (a, a, e), "a_eq_c": (a, e, a), "b_eq_c": (a, e, e), "point": (a, a, a)}[kind]
    p = rng.uniform(-1.0, 2.0, (400, 3))
    bc = lambda z: np.broadcast_to(z, p.shape)
    q = R.closest_triangle(p, bc(a), bc(b), bc(c))
    assert not np.any(np.isnan(q))
    S = np.concatenate([u + np.linspace(0, 1, 4001)[:, None] * (v - u) for u, v in ((a, b), (a, c), (b, c))])
    dmin = np.sqrt(((p[:, None, :] - S[None]) ** 2).sum(-1)).min(1)
    d = R.dist(p, q)
    assert np.all(d <= dmin + 1e-12) and np.all(d >= dmin - 1e-3)


@pytest.mark.parametrize("name", list(BAND_CASES))
def test_band_guarantee_against_brute_force(name):
    phi, lc, h = BAND_CASES[name]
    bf = R.brute_force(phi, lc, h)
    x = R.node_coords(phi.shape, lc, h)
    hmin = min(abs(v) for v in h)
    for band in (1, 3):
        P, is_band = R.band_phase(phi, lc, h, band)
        d = R.dist(x, P)
        sure = is_band & (d < band * hmin)
        assert sure.sum() > 0.5 * np.sum(np.abs(phi) < 0.5 * band * hmin)
        assert np.array_equal(d[sure], bf[sure]), "a band node closer than band * min h holds the minimum over the whole mesh"
        assert np.all(np.isnan(d[~is_band]))


@pytest.mark.parametrize("name", list(BAND_CASES))
def test_propagated_distances_against_brute_force(name):
    phi, lc, h = BAND_CASES[name]
    bf = R.brute_force(phi, lc, h)
    out, nb = R.redistance(phi, lc, h, band=3)
    a = np.abs(out)
    # a distance to a point on the mesh is never below the distance to the mesh, up to the rounding of the closest points
    # (coordinates are O(1): a few ulps of 0.5)
    assert np.all(a >= bf - 1e-15)
    # observed on these four grids: 0.56 .. 0.70 of the nodes bit-equal to brute force, 0.85 .. 0.98 within 0.01 h of it, and
    # at most 0.09 h above it; jump flooding hands far nodes a point that was closest to a neighbour, not to them
    hmin = min(abs(v) for v in h)
    assert np.mean(a == bf) > 0.5, np.mean(a == bf)
    assert np.mean(a - bf < 1e-2 * hmin) > 0.8, np.mean(a - bf < 1e-2 * hmin)
    assert np.max(a - bf) < 0.15 * hmin
    assert np.array_equal(out <= 0, phi <= 0)


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_classification_kept_with_subnormal_raise(dtype):
    tiny = {np.float64: 1e-300, np.float32: 1e-30}[dtype]
    phi = np.array([-1.0, tiny, 2.0], dtype=dtype)      # t = -1 / (-1 - tiny) rounds to 1: the crossing sits on node 1
    out, _ = R.redistance(phi, [0.0], [1.0])
    assert out[0] == -1.0 and out[1] == np.finfo(dtype).smallest_subnormal and out[2] == 1.0
    assert out.dtype == dtype
    # exact zeros and NaN nodes on a 3-D sphere
    q, h = sphere((14, 13, 15), r=0.3)
    q = (np.round(q * 16) / 16).astype(dtype)
    q[2:4, 5, 6] = np.nan
    out, _ = R.redistance(q, (-0.5,) * 3, h)
    assert np.array_equal(np.isnan(out), np.isnan(q))
    v = ~np.isnan(q)
    assert np.array_equal(out[v] <= 0, q[v] <= 0)


def test_without_interface_nothing_changes():
    phi, h = sphere((9, 8, 7))
    out, nb = R.redistance(phi + 2.0, (-0.5,) * 3, h)
    assert nb == 0 and bits_equal(out, phi + 2.0)


def test_abi_argument_checks_without_a_device(m):
    lib, L = m._lib.lib(), m._lib
    nb = C.c_int64(-1)
    assert lib.lsm_redistance(None, None, 0, C.byref(nb)) == L.ERR_ARG and "band" in L.last_error()
    assert lib.lsm_redistance(None, None, -2, None) == L.ERR_ARG
    assert lib.lsm_redistance(None, None, 3, None) == L.ERR_ARG and "null" in L.last_error()
    assert nb.value == -1


# ================================================================================================
# device == restatement, bit for bit
# ================================================================================================
def _run(m, phi, band):
    """lsm_redistance through the C ABI with the band-node count; returns (values, band nodes)."""
    ctx = phi._context()
    nb = C.c_int64(-1)
    m._lib.check(m._lib.lib().lsm_redistance(ctx.handle, phi.device(), band, C.byref(nb)))
    phi._mark_device_advanced()
    return np.array(phi.peek()), nb.value


@pytest.mark.gpu
@pytest.mark.parametrize("band", [3, 1])
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("name", list(CASES))
def test_device_equals_restatement(m, name, dtype, band):
    vals, lc, hc = CASES[name]
    vals = vals.astype(dtype)
    h = grid_h(lc, hc, vals.shape)
    got, nb = _run(m, on_device(m, vals, lc, hc, dtype), band)
    want, nb_want = R.redistance(vals, lc, h, band)
    assert nb == nb_want
    assert bits_equal(got, want)
    if name == "3d_all_positive":
        assert nb == 0 and bits_equal(got, vals)


@pytest.mark.gpu
@pytest.mark.parametrize("band", [2, 5])
def test_device_equals_restatement_wider_bands(m, band):
    for name in ("2d_odd_aniso", "3d_notched_sphere"):
        vals, lc, hc = CASES[name]
        got, nb = _run(m, on_device(m, vals, lc, hc, np.float64), band)
        want, nb_want = R.redistance(vals, lc, grid_h(lc, hc, vals.shape), band)
        assert nb == nb_want and bits_equal(got, want), name


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_zalesak_disk_equals_restatement(m, dtype):
    phi, g = zalesak(m, 101, dtype)
    before = np.array(phi.peek())
    m.redistance(phi)
    want, _ = R.redistance(before, g.lc, g.meshsize(), 3)
    assert bits_equal(np.array(phi.peek()), want)


# ================================================================================================
# accuracy, interface shift, determinism, asynchrony, invalidation, prehook, errors
# ================================================================================================
@pytest.mark.gpu
def test_second_order_on_a_sphere(m):
    errs = []
    for n in (64, 128):
        g = m.CartesianGrid((-0.5,) * 3, (0.5,) * 3, (n, n, n))
        x = R.node_coords(g.n, g.lc, g.meshsize())
        r = np.sqrt(((x[..., 0] - 0.02) ** 2 + (x[..., 1] + 0.01) ** 2) + x[..., 2] ** 2)
        exact = r - 0.3
        phi = m.MeshField(np.asfortranarray(r * r - 0.09), g)        # same zero level set, far from a distance
        m.redistance(phi)
        near = np.abs(exact) < 3 * g.meshsize(1)
        errs.append(float(np.abs(phi.peek() - exact)[near].max()))
    order = math.log2(errs[0] / errs[1])
    print("max error within 3h:", errs, "order", order)
    assert order > 1.8, errs                 # measured on a B200: 3.1e-4 and 7.7e-5, order 2.02


def mesh_shift(before, after):
    """Largest distance from a vertex of `after` to the mesh `before` (InterfaceMesh pairs; closest points over the 32 primitives
    nearest by centroid, so the figure is an upper bound)."""
    from scipy.spatial import cKDTree
    V = before.vertices[before.faces.astype(np.int64)]
    cent = V.mean(axis=1)
    k = min(32, len(V))
    _, j = cKDTree(cent).query(after.vertices, k=k)
    j = j.reshape(len(after.vertices), k)
    X = np.repeat(after.vertices[:, None, :], k, axis=1)
    q = R.closest_point(X, V[j])
    return float(np.nanmin(R.dist(X, q), axis=1).max())


@pytest.mark.gpu
def test_interface_shift(m):
    g = m.CartesianGrid((-0.5,) * 3, (0.5,) * 3, (48, 50, 46))
    x = R.node_coords(g.n, g.lc, g.meshsize())
    r = np.sqrt(((x[..., 0] - 0.02) ** 2 + (x[..., 1] + 0.01) ** 2) + x[..., 2] ** 2)
    z, gz = zalesak(m, 128)
    # measured on a B200: 0.013 h on the sphere, 0.11 h on the Zalesak disk, at the corners of its slot (where the distance to the
    # linear interface is not linear along an edge, so its zero crossing moves)
    cases = [(m.MeshField(np.asfortranarray(r * r - 0.09), g), min(g.meshsize()), 0.025), (z, min(gz.meshsize()), 0.15)]
    for phi, h, bound in cases:
        before = m.extract_interface(phi)
        m.redistance(phi)
        shift = mesh_shift(before, m.extract_interface(phi))
        print("interface shift / h:", shift / h)
        assert shift < bound * h, shift / h


@pytest.mark.gpu
def test_deterministic_and_asynchronous(m):
    vals, lc, hc = CASES["3d_notched_sphere"]
    ctx = m.default_context()
    a = on_device(m, vals, lc, hc, np.float64)
    b = on_device(m, vals, lc, hc, np.float64)
    a.device(), b.device()
    ctx.reset_counters()
    m.redistance(a)
    c = ctx.counters()
    assert c["d2h_bytes"] == 0 and c["h2d_bytes"] == 0
    assert c["kernel_launches"] == 5 + len(R.flood_steps(vals.shape))     # flag, 2 cell passes, pick, flooding, write
    nb = C.c_int64(-1)
    m._lib.check(m._lib.lib().lsm_redistance(ctx.handle, b.device(), 3, C.byref(nb)))
    b._mark_device_advanced()
    assert ctx.counters()["d2h_bytes"] == 8 and nb.value > 0          # one 8-byte copy of the band-node count
    assert bits_equal(np.array(a.peek()), np.array(b.peek()))
    again = m.redistance(a)                  # redistancing a distance field is not the identity bit for bit, but close
    assert again is a


@pytest.mark.gpu
def test_cfl_cache_sees_new_values(m):
    g = m.CartesianGrid((-1.0, -1.0), (1.0, 1.0), (65, 61))
    x = R.node_coords(g.n, g.lc, g.meshsize())
    phi = m.MeshField(np.asfortranarray(np.hypot(x[..., 0], x[..., 1]) - 0.5), g, bc=m.NeumannBC())
    speed = m.MeshField(np.asfortranarray(3.0 * (x[..., 0] ** 2 + x[..., 1] ** 2) - 0.2), g)
    terms = (m.NormalMotionTerm(speed),)
    dt0 = m.compute_cfl(terms, phi, 0.0)
    m.compute_cfl(terms, phi, 0.0)           # served from the cache
    m.redistance(speed)
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
    eqs = [m.LevelSetEquation(terms=(m.AdvectionTerm((0.3, -0.2, 0.5), m.WENO5()),), ic=ic, integrator=m.RK3()) for _ in range(2)]
    tf = 0.05
    for e in eqs:
        e.state.device()
    ctx.reset_counters()
    m.integrate(eqs[0], tf, prehook=lambda ls: m.redistance(ls.state))
    c = ctx.counters()
    assert c["d2h_bytes"] < 64 * max(1, eqs[0].steps_taken) and c["h2d_bytes"] == 0      # the field never left the device
    e = eqs[1]
    phi, tc, steps = e.state, 0.0, 0
    while tc <= tf - float(np.spacing(abs(tc))):
        m.redistance(phi)
        dt = min(math.inf, e.integrator.cfl * m.compute_cfl(e.terms, phi, tc), tf - tc)
        m.api._advance(e.integrator, phi, e.terms, tc, dt)
        tc += dt
        steps += 1
    assert steps == eqs[0].steps_taken >= 3
    assert bits_equal(np.array(eqs[0].state.peek()), np.array(phi.peek()))


@pytest.mark.gpu
def test_error_codes(m):
    lib, L = m._lib.lib(), m._lib
    fresh = m.Context(0)
    try:
        g = m.CartesianGrid((0, 0), (1, 1), (9, 8))
        vec = m.MeshField(np.zeros((2, 9, 8)), g, ctx=fresh)
        assert lib.lsm_redistance(fresh.handle, vec.device(), 3, None) == L.ERR_ARG
        sep = m.SeparableVelocity(g, (1.0, 1.0), [[np.ones(9), np.ones(8)], [np.ones(9), np.ones(8)]], ctx=fresh)
        assert lib.lsm_redistance(fresh.handle, sep.device(), 3, None) == L.ERR_ARG
        thin = m.MeshField(np.zeros((9, 1)), m.CartesianGrid((0, 0), (1, 1), (9, 1)), ctx=fresh)
        assert lib.lsm_redistance(fresh.handle, thin.device(), 3, None) == L.ERR_ARG
        sc = m.MeshField(np.zeros((9, 8)) - 1, g, ctx=fresh)
        assert lib.lsm_redistance(fresh.handle, sc.device(), 0, None) == L.ERR_ARG
        assert lib.lsm_redistance(m.default_context().handle, sc.device(), 3, None) == L.ERR_ARG      # another context
        assert lib.lsm_redistance(fresh.handle, sc.device(), 3, None) == L.OK
        with pytest.raises(m.LSMError):
            m.redistance(sc, band=0)
        del vec, sep, thin, sc
    finally:
        fresh.close()


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["redistance", "extend_closest_point", "redistance_cubic", "interpolate_cubic"])
def test_slab_decomposition_is_refused(m, entry):
    """The single-rank zero-level-set operations refuse a slab-decomposed field with the header's wording."""
    n = C.c_int32(0)
    m._lib.lib().lsm_device_count(C.byref(n))
    if n.value < 2:
        pytest.skip("needs 2 GPUs")
    lib = m._lib.lib()
    mc = m.MultiContext([0, 1])
    try:
        ctx = mc.ranks[0]
        phi, _ = sphere((20, 18, 24))
        f = on_device(m, phi, (-0.5,) * 3, (0.5,) * 3, np.float64, ctx=ctx)
        F = on_device(m, np.ones(phi.shape), (-0.5,) * 3, (0.5,) * 3, np.float64, ctx=ctx)
        Y = np.zeros((1, 3))
        call = {
            "redistance": lambda: lib.lsm_redistance(ctx.handle, f.device(), 3, None),
            "extend_closest_point": lambda: lib.lsm_extend_closest_point(ctx.handle, F.device(), f.device(), 3, 0, None),
            "redistance_cubic": lambda: lib.lsm_redistance_cubic(ctx.handle, f.device(), 3, None, None),
            "interpolate_cubic": lambda: lib.lsm_interpolate_cubic(ctx.handle, f.device(), 1, C.cast(Y.ctypes.data, C.POINTER(C.c_double)),
                                                                   None, None, None),
        }[entry]
        assert call() == m._lib.ERR_UNSUPPORTED
        assert "slab decomposition is not supported" in m._lib.last_error()
        del f, F
    finally:
        mc.close()
