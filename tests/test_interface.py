"""Zero-level-set extraction (lsm_interface_extract / lsm_interface_fetch / lsm_multi_interface_extract, extract_interface,
merge_interfaces, extract_interface_multi).

Without a GPU: the NumPy restatement of the contract (interface_ref.py) against hand-computed answers for single simplices, the
closed-surface properties of its meshes (edge use, orientation, Euler characteristic, second-order area and volume), the weld,
and the argument checks of the C ABI that need no device.  On the GPU: the device mesh equals the restatement bit for bit over
dimensions, dtypes, odd sizes, anisotropic and mirrored grids, kinked shapes, exact zeros, NaN nodes and empty results; it is
deterministic; the accounting shows that only the mesh leaves the device; error codes; and the 2-GPU weld equals 1 GPU."""
import ctypes as C
import itertools
import math

import numpy as np
import pytest

import helpers as H
import interface_ref as R
from zero_set_helpers import m, on_device, sphere, torus  # noqa: F401 (m is a fixture)


def grid_values(lc, hc, n):
    h = [(hc[d] - lc[d]) / (n[d] - 1) for d in range(len(n))]
    return H.coords(lc, hc, n), h


# ================================================================================================
# the restatement against hand-computed answers (no GPU)
# ================================================================================================
def test_1d_crossings():
    phi = np.array([-1.0, 3.0, 2.0, -0.5, np.nan, 1.0, 0.0, 4.0])
    X, F, K = R.extract(phi, [1.0], [0.5])
    # (0,1): t = -1 / (-1 - 3) = 0.25;  (2,3): t = 2 / 2.5 = 0.8;  (3,4), (4,5): NaN;  0 is inside: (5,6): t = 1 / (1 - 0) = 1,
    # (6,7): t = 0 / (0 - 4) = 0 — both on node 6, two vertices of two edges
    assert K.tolist() == [0, 2, 5, 6]
    assert X[:, 0].tolist() == [1.0 + 0.25 * 0.5, 1.0 + 2.8 * 0.5, 4.0, 4.0]
    assert F.tolist() == [[0], [1], [2], [3]]


def _simplex_geometry(N, p, inside, h):
    """Chain vertex positions (scaled by h), node values with the given inside mask (distinct magnitudes), the gradient of their
    linear interpolant, and the crossing point of every chain edge."""
    w = R.chain(N, p)
    P = np.array([[((wk >> d) & 1) * h[d] for d in range(N)] for wk in w], dtype=np.float64)
    s = np.array([-(1.0 + 0.3 * k) if (inside >> k) & 1 else 1.0 + 0.7 * k for k in range(N + 1)])
    g = np.linalg.solve(P[1:] - P[0], s[1:] - s[0])
    cross = {}
    for x, y in itertools.combinations(range(N + 1), 2):
        if (s[x] <= 0) != (s[y] <= 0):
            t = s[x] / (s[x] - s[y])
            cross[(x, y)] = P[x] + t * (P[y] - P[x])
    return cross, g


@pytest.mark.parametrize("h", [(1.0, 1.0), (0.5, 2.0), (-0.5, 2.0)], ids=["unit", "aniso", "mirrored"])
def test_triangle_all_inside_masks(h):
    hsign = -1 if h[0] * h[1] < 0 else 1
    for p in range(2):
        for mask in range(8):
            prims = R.simplex_primitives(2, p, mask, hsign)
            assert len(prims) == (0 if mask in (0, 7) else 1), (p, mask)
            if not prims:
                continue
            cross, g = _simplex_geometry(2, p, mask, h)
            (e0, e1), = prims
            assert {e0, e1} <= set(cross) and e0 != e1
            d = cross[e1] - cross[e0]
            assert np.dot((-d[1], d[0]), g) < 0, (p, mask)     # the inside (smaller s) lies on the left
    # by hand: w = (0, 1, 3) for p = 0 (+), w = (0, 2, 3) for p = 1 (-)
    assert R.simplex_primitives(2, 0, 0b001) == [((0, 1), (0, 2))]
    assert R.simplex_primitives(2, 1, 0b001) == [((0, 2), (0, 1))]
    assert R.simplex_primitives(2, 0, 0b110) == [((0, 2), (0, 1))]      # lone outside vertex w_0
    assert R.simplex_primitives(2, 0, 0b010) == [((1, 2), (0, 1))]      # w_1 = (1, 0) inside, left of (1, .5) -> (.5, 0)


@pytest.mark.parametrize("h", [(1.0, 1.0, 1.0), (0.5, 2.0, 0.75), (0.5, -2.0, 0.75)], ids=["unit", "aniso", "mirrored"])
def test_tetrahedron_all_inside_masks(h):
    hsign = -1 if h[0] * h[1] * h[2] < 0 else 1
    for p in range(6):
        for mask in range(16):
            k = bin(mask).count("1")
            prims = R.simplex_primitives(3, p, mask, hsign)
            assert len(prims) == {0: 0, 1: 1, 2: 2, 3: 1, 4: 0}[k], (p, mask)
            cross, g = _simplex_geometry(3, p, mask, h)
            assert sorted({e for t in prims for e in t}) == sorted(cross)    # every cut edge is used, nothing else
            for tri in prims:
                a, b, c = (cross[e] for e in tri)
                assert np.dot(np.cross(b - a, c - a), g) > 0, (p, mask, tri)      # normal toward s > 0
            if k == 2:
                (t0, t1) = prims
                assert t0[0] == t1[0] and len(set(t0) & set(t1)) == 2     # quad split along its diagonal (ac, bd)
    # by hand, p = 0 (w = 0, 1, 3, 7, even): inside {w_0}, {w_0, w_1}; p = 1 (odd) reverses the same masks
    assert R.simplex_primitives(3, 0, 0b0001) == [((0, 1), (0, 2), (0, 3))]
    assert R.simplex_primitives(3, 1, 0b0001) == [((0, 1), (0, 3), (0, 2))]
    assert R.simplex_primitives(3, 0, 0b0011) == [((0, 2), (0, 3), (1, 3)), ((0, 2), (1, 3), (1, 2))]
    assert R.simplex_primitives(3, 1, 0b0011) == [((0, 2), (1, 3), (0, 3)), ((0, 2), (1, 2), (1, 3))]
    assert R.simplex_primitives(3, 0, 0b1110) == [((0, 1), (0, 3), (0, 2))]      # lone outside vertex w_0


def _closed_surface(X, F, chi):
    cu, cd = R.edge_counts(F)
    assert np.all(cu == 2), "every edge is used by exactly two triangles"
    assert np.all(cd == 1), "every directed edge is used once (consistent orientation)"
    assert len(np.unique(F)) == len(X)
    assert R.euler_characteristic(X, F) == chi


@pytest.mark.parametrize("shape", ["sphere", "torus"])
def test_closed_surfaces_converge_at_second_order(shape):
    errs = []
    for n in (24, 48):
        if shape == "sphere":
            phi, h = sphere((n, n, n), r=0.3507, c=(0.0, 0.0, 0.0))
            A0, V0, chi = 4 * math.pi * 0.3507 ** 2, 4 / 3 * math.pi * 0.3507 ** 3, 2
        else:
            phi, h = torus((n, n, n), R0=0.3, r=0.12)
            A0, V0, chi = 4 * math.pi ** 2 * 0.3 * 0.12, 2 * math.pi ** 2 * 0.3 * 0.12 ** 2, 0
        X, F, K = R.extract(phi, (-0.5,) * 3, h)
        _closed_surface(X, F, chi)
        assert np.all(np.diff(K) > 0)
        errs.append((abs(R.area(X, F) / A0 - 1), abs(R.enclosed_volume(X, F) / V0 - 1)))
    for k in range(2):
        assert errs[1][k] < errs[0][k] / 3.0, errs      # second order: a factor of about 4 per halving of h
    if shape == "sphere":
        assert errs[0][0] < 5e-3 and errs[1][0] < 1.2e-3 and errs[0][1] < 9e-3 and errs[1][1] < 2.2e-3, errs


def test_circle_is_a_closed_counterclockwise_curve():
    (x, y), h = grid_values((-1, -1), (1, 1), (41, 37))
    phi = np.hypot(x - 0.1, y + 0.05) - 0.6
    X, F, K = R.extract(phi, (-1, -1), h)
    deg = np.bincount(F.ravel(), minlength=len(X))
    assert np.all(deg == 2)
    assert np.all(np.bincount(F[:, 0], minlength=len(X)) == 1)       # one outgoing and one incoming segment per vertex
    assert abs(R.signed_area_2d(X, F) / (math.pi * 0.36) - 1) < 1e-2


def test_merge_interfaces_welds_overlapping_pieces(m):
    a = m.InterfaceMesh(np.array([[0.0, 0.0], [1.0, 0.0], [2.0, 0.0]]), np.array([[0, 1], [1, 2]], np.int32), np.array([3, 5, 9]))
    b = m.InterfaceMesh(np.array([[2.0, 0.0], [3.0, 1.0]]), np.array([[0, 1]], np.int32), np.array([9, 12]))
    w = m.merge_interfaces([a, b])
    assert w.keys.tolist() == [3, 5, 9, 12]
    assert w.vertices.tolist() == [[0, 0], [1, 0], [2, 0], [3, 1]]
    assert w.faces.tolist() == [[0, 1], [1, 2], [2, 3]] and w.faces.dtype == np.int32
    # slab pieces of the restatement (each box = the rank's planes + the next rank's first plane) weld to the whole mesh
    phi, h = sphere((20, 18, 23), r=0.3, c=(0.02, -0.03, 0.01))
    whole = R.extract(phi, (-0.5,) * 3, h)
    pieces = []
    for first, count in ((0, 8), (8, 7), (15, 8)):
        top = min(first + count + 1, 23)
        X, F, K = R.extract(phi[..., first:top], (-0.5,) * 3, h, first_last=first, nglob_last=23)
        pieces.append(m.InterfaceMesh(X, F, K))
    assert len(pieces[0].keys) + len(pieces[1].keys) + len(pieces[2].keys) > len(whole[2])     # the slab planes are shared
    w = m.merge_interfaces(pieces)
    for got, want in zip((w.vertices, w.faces, w.keys), whole):
        assert got.dtype == want.dtype and np.array_equal(got, want)


def test_abi_argument_checks_without_a_device(m):
    lib = m._lib.lib()
    nv, nf = C.c_int64(-1), C.c_int64(-1)
    assert lib.lsm_interface_extract(None, None, 0.0, C.byref(nv), C.byref(nf)) == m._lib.ERR_ARG
    assert lib.lsm_interface_fetch(None, None, None, None) == m._lib.ERR_ARG
    assert lib.lsm_multi_interface_extract(0, None, None, 0.0, None, None) == m._lib.ERR_ARG
    with pytest.raises(ValueError):
        m.merge_interfaces([])


# ================================================================================================
# device mesh == restatement, bit for bit
# ================================================================================================
def _same(got, want):
    X, F, K = want
    assert got.vertices.dtype == np.float64 and got.faces.dtype == np.int32 and got.keys.dtype == np.int64
    assert got.vertices.shape == X.shape and got.faces.shape == F.shape and got.keys.shape == K.shape
    assert np.array_equal(got.keys, K)
    assert np.array_equal(got.vertices.view(np.int64), X.view(np.int64))        # bits, so that -0.0 != 0.0 would show
    assert np.array_equal(got.faces, F)


def _cases():
    out = {}
    x = np.linspace(-1, 1, 37)
    v1 = np.sin(7 * x) + 0.1
    v1[5] = 0.0
    v1[20] = np.nan
    out["1d"] = (v1, (-1.0,), (1.0,), 0.0)
    (gx, gy), _ = grid_values((-1, -1.5), (1.2, 1.5), (37, 53))
    out["2d_circle_level"] = (np.hypot(gx - 0.1, gy), (-1, -1.5), (1.2, 1.5), 0.55)
    z = H.c2_zalesak_curvature(61)
    out["2d_zalesak"] = (z.phi0, z.lc, z.hc, 0.0)
    phi, _ = sphere((37, 53, 29), r=0.33, lc=(-0.5, -0.6, -0.4), hc=(0.55, 0.6, 0.45), c=(0.03, -0.02, 0.01))
    out["3d_odd_aniso_level"] = (phi, (-0.5, -0.6, -0.4), (0.55, 0.6, 0.45), -0.021)
    out["3d_mirrored"] = (phi, (0.55, -0.6, -0.4), (-0.5, 0.6, 0.45), 0.0)
    (x3, y3, z3), _ = grid_values((-0.5,) * 3, (0.5,) * 3, (33, 31, 35))
    ball = np.sqrt((x3 * x3 + y3 * y3) + z3 * z3) - 0.35
    slot = np.maximum(np.maximum(np.abs(x3) - 0.06, np.abs(y3 + 0.25) - 0.25), np.abs(z3) - 0.5)
    out["3d_notched_sphere"] = (np.maximum(ball, -slot), (-0.5,) * 3, (0.5,) * 3, 0.0)
    q = np.round(ball * 16) / 16            # many exact zeros at nodes, and NaN nodes
    q[3:6, 10:12, 4] = np.nan
    q[16, 16, 20:23] = np.nan
    out["3d_zeros_nan"] = (q, (-0.5,) * 3, (0.5,) * 3, 0.0)
    out["3d_empty"] = (ball + 2.0, (-0.5,) * 3, (0.5,) * 3, 0.0)
    return out


CASES = _cases()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("name", list(CASES))
def test_device_mesh_equals_restatement(m, name, dtype):
    vals, lc, hc, level = CASES[name]
    phi = on_device(m, vals, lc, hc, dtype)
    h = [(hc[d] - lc[d]) / (vals.shape[d] - 1) for d in range(vals.ndim)]
    got = m.extract_interface(phi, level)
    want = R.extract(vals.astype(dtype), lc, h, level)
    _same(got, want)
    if name == "3d_empty":
        assert len(got.keys) == 0 and len(got.faces) == 0
    if name in ("3d_odd_aniso_level", "3d_notched_sphere"):
        _closed_surface(want[0], want[1], 2)
    again = m.extract_interface(phi, level)
    for a, b in zip(got, again):
        assert np.array_equal(a, b)              # order does not depend on scheduling


@pytest.mark.gpu
def test_empty_fetch_with_null_arrays(m):
    phi = on_device(m, np.ones((9, 7)), (0, 0), (1, 1), np.float64)
    lib, ctx = m._lib.lib(), m.default_context()
    nv, nf = C.c_int64(-1), C.c_int64(-1)
    m._lib.check(lib.lsm_interface_extract(ctx.handle, phi.device(), 0.0, C.byref(nv), C.byref(nf)))
    assert nv.value == 0 and nf.value == 0
    m._lib.check(lib.lsm_interface_fetch(ctx.handle, None, None, None))


@pytest.mark.gpu
def test_device_expression_torus(m):
    g = m.CartesianGrid((-0.5,) * 3, (0.5,) * 3, (40, 42, 38))
    phi = m.MeshField.from_expr(g, "sqrt((sqrt(x1*x1 + x2*x2) - 0.3)*(sqrt(x1*x1 + x2*x2) - 0.3) + x3*x3) - 0.12")
    got = m.extract_interface(phi)
    want = R.extract(phi.peek(), g.lc, [g.meshsize(d + 1) for d in range(3)])
    _same(got, want)
    _closed_surface(want[0], want[1], 0)


@pytest.mark.gpu
def test_c3_state_after_integration(m):
    case = H.c3_enright(128)
    phi = case.engine_field(m)
    eq = m.LevelSetEquation(terms=case.engine_terms(m, phi), ic=phi, integrator=m.RK3())
    m.integrate(eq, 4.5 * 0.5 * m.compute_cfl(eq.terms, eq.state, 0.0))
    assert eq.steps_taken >= 4
    got = m.extract_interface(eq)
    h = [(case.hc[d] - case.lc[d]) / (case.n[d] - 1) for d in range(3)]
    want = R.extract(eq.state.peek(), case.lc, h)
    _same(got, want)
    _closed_surface(want[0], want[1], 2)


@pytest.mark.gpu
def test_only_the_mesh_leaves_the_device(m):
    ctx = m.default_context()
    g = m.CartesianGrid((-0.5,) * 3, (0.5,) * 3, (512, 512, 512))
    phi = m.MeshField.from_shape(g, "sphere", (0.0, 0.0, 0.0, 0.35))
    phi.device()
    ctx.reset_counters()
    mesh = m.extract_interface(phi)
    c = ctx.counters()
    mesh_bytes = mesh.vertices.nbytes + mesh.keys.nbytes + mesh.faces.nbytes
    assert c["d2h_bytes"] == 16 + mesh_bytes
    assert c["d2h_bytes"] < 512 ** 3 * 8 / 10
    assert c["kernel_launches"] == 4
    _closed_surface(mesh.vertices, mesh.faces, 2)
    assert abs(R.area(mesh.vertices, mesh.faces) / (4 * math.pi * 0.35 ** 2) - 1) < 1e-4
    del phi


@pytest.mark.gpu
def test_error_codes(m):
    lib, L = m._lib.lib(), m._lib
    fresh = m.Context(0)
    try:
        assert lib.lsm_interface_fetch(fresh.handle, None, None, None) == L.ERR_ARG          # nothing extracted yet
        assert "no interface" in L.last_error()
        nv, nf = C.c_int64(), C.c_int64()
        g = m.CartesianGrid((0, 0), (1, 1), (9, 8))
        vec = m.MeshField(np.zeros((2, 9, 8)), g, ctx=fresh)
        assert lib.lsm_interface_extract(fresh.handle, vec.device(), 0.0, C.byref(nv), C.byref(nf)) == L.ERR_ARG
        sep = m.SeparableVelocity(g, (1.0, 1.0), [[np.ones(9), np.ones(8)], [np.ones(9), np.ones(8)]], ctx=fresh)
        assert lib.lsm_interface_extract(fresh.handle, sep.device(), 0.0, C.byref(nv), C.byref(nf)) == L.ERR_ARG
        sc = m.MeshField(np.zeros((9, 8)) - 1, g, ctx=fresh)
        assert lib.lsm_interface_extract(fresh.handle, sc.device(), float("nan"), C.byref(nv), C.byref(nf)) == L.ERR_ARG
        assert lib.lsm_interface_extract(fresh.handle, sc.device(), float("inf"), C.byref(nv), C.byref(nf)) == L.ERR_ARG
        thin = m.MeshField(np.zeros((9, 1)), m.CartesianGrid((0, 0), (1, 1), (9, 1)), ctx=fresh)
        assert lib.lsm_interface_extract(fresh.handle, thin.device(), 0.0, C.byref(nv), C.byref(nf)) == L.ERR_ARG
        assert lib.lsm_interface_fetch(fresh.handle, None, None, None) == L.ERR_ARG          # a failed extraction leaves nothing
        assert lib.lsm_interface_extract(fresh.handle, sc.device(), 0.0, C.byref(nv), C.byref(nf)) == L.OK
        assert lib.lsm_interface_fetch(fresh.handle, None, None, None) == L.OK               # all inside: empty mesh
        del vec, sep, sc, thin
    finally:
        fresh.close()


# ================================================================================================
# two GPUs: the welded pieces equal the 1-GPU mesh bit for bit
# ================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("periodic", [False, True], ids=["neumann", "periodic_last_axis"])
def test_multi_gpu_weld_equals_single_gpu(m, periodic):
    n = C.c_int32(0)
    m._lib.lib().lsm_device_count(C.byref(n))
    if n.value < 2:
        pytest.skip("needs 2 GPUs")
    mc = m.MultiContext([0, 1])
    solo = m.Context(0)
    try:
        shape = (30, 26, 41)
        lc, hc = (-0.5,) * 3, (0.5,) * 3
        # the sphere crosses the slab boundary (plane 20 of 41); with the periodic axis it also crosses the seam
        c = (0.05, -0.02, 0.45 if periodic else 0.02)
        phi0, _ = sphere(shape, r=0.3, c=c)
        bc = (m.NeumannBC(), m.NeumannBC(), m.PeriodicBC() if periodic else m.NeumannBC())
        eqs = []
        for ctx in mc.ranks:
            f = on_device(m, phi0, lc, hc, np.float64, ctx=ctx, bc=bc)
            eqs.append(m.LevelSetEquation(terms=(m.AdvectionTerm((0.3, -0.2, 0.5), m.WENO5()),), ic=f, integrator=m.RK3()))
        m.integrate_multi(mc, eqs, 0.02)
        for fresh_upload in (False, True):
            if fresh_upload:                   # new values, stale ghost planes: the extraction exchanges them first
                vals = -m.MultiContext.gather([e.state for e in eqs])
                for e in eqs:
                    e.state.vals[...] = vals[..., e.state._first:e.state._first + e.state._count]
            glob = m.MultiContext.gather([e.state for e in eqs])
            got = m.extract_interface_multi(mc, [e.state for e in eqs])
            ref = m.extract_interface(on_device(m, glob, lc, hc, np.float64, ctx=solo, bc=bc))
            for a, b in zip(got, ref):
                assert a.dtype == b.dtype and np.array_equal(a, b)
            assert len(ref.faces) > 1000
    finally:
        mc.close()
        solo.close()
