"""The cubic interpolant (lsm_interpolate_cubic, interpolate) and cubic closest-point redistancing (lsm_redistance_cubic,
redistance(order=3)).

Without a GPU: the NumPy restatement (cubic_ref.py) reproduces tensor-cubic polynomials, their gradients and Hessians, node values
exactly, and gives NaN outside the box; refined points satisfy the KKT conditions; refined 2-D distances match a brute-force
distance to the sampled cubic zero set; a plane gives its exact distance; each fallback rule; the C ABI's argument checks.  On the
GPU: both entry points equal the restatement bit for bit over dimensions, dtypes, odd, anisotropic and mirrored grids, cell and
box faces, outside points, bands, n_d = 4, NaN nodes, no interface, the Zalesak disk and the fallback count; third-order accuracy
on a sphere; determinism; asynchrony; the CFL cache; the prehook; error codes."""
import ctypes as C
import itertools
import math

import numpy as np
import pytest

import cubic_ref as CR
import redistance_ref as R
from zero_set_helpers import bits_equal, grid_h, m, on_device, zalesak  # noqa: F401 (m is a fixture)


def same_values(a, b):
    """bit for bit where a value is a number, NaN at the same places (the payload of a computed NaN differs between the device and
    NumPy on the host)"""
    a, b = np.asarray(a), np.asarray(b)
    nan = np.isnan(a)
    return a.shape == b.shape and np.array_equal(nan, np.isnan(b)) and bits_equal(a[~nan], b[~nan])


def tensor_cubic(C3, X):
    """sum_{ijk} C[i,j,k] x^i y^j z^k (degrees <= 3 per axis; N = C3.ndim), its gradient and its Hessian at X (..., N)."""
    N = C3.ndim
    pw = lambda v, e, k: (math.perm(e, k) * v ** (e - k)) if e >= k else np.zeros_like(v)
    val, g, H = np.zeros(X.shape[:-1]), np.zeros(X.shape), np.zeros(X.shape + (N,))
    for ex in itertools.product(range(4), repeat=N):
        c = C3[ex]
        term = lambda ks: c * np.prod([pw(X[..., d], ex[d], ks[d]) for d in range(N)], axis=0)
        val += term([0] * N)
        for d in range(N):
            k = [0] * N
            k[d] = 1
            g[..., d] += term(k)
            for e in range(N):
                k2 = [0] * N
                k2[d] += 1
                k2[e] += 1
                H[..., d, e] += term(k2)
    return val, g, H


# ================================================================================================
# the restatement (no GPU)
# ================================================================================================
@pytest.mark.parametrize("N", [1, 2, 3])
def test_reproduces_tensor_cubic_polynomials(N):
    rng = np.random.default_rng(N)
    n = (7, 6, 8)[:N]
    lc, h = (-0.4, 0.3, -0.2)[:N], (0.15, -0.12, 0.11)[:N]          # one mirrored axis
    C3 = rng.uniform(-1, 1, (4,) * N)
    phi = tensor_cubic(C3, R.node_coords(n, lc, h))[0]
    # interior points, points on cell faces, on box faces and in the one-sided boundary cells
    U = rng.uniform(0, 1, (3000, N)) * (np.array(n) - 1)
    U[:300] = np.round(U[:300] * 2) / 2
    U[300:600, 0] = 0.0
    U[600:900, -1] = n[-1] - 1
    U[900:1200] = rng.uniform(0, 1, (300, N))
    Y = np.array(lc) + U * np.array(h)
    P, g, H = CR.evaluate(phi, lc, h, Y)
    v, gv, Hv = tensor_cubic(C3, Y)
    assert np.abs(P - v).max() <= 1e-12
    assert np.abs(g - gv).max() <= 1e-12
    assert np.abs(H - Hv).max() <= 1e-12
    assert np.array_equal(H, np.swapaxes(H, 1, 2))


def test_node_values_exact_and_outside_nan():
    rng = np.random.default_rng(5)
    n, lc, h = (6, 5, 7), (-0.5, 1.0, 0.25), (0.125, -0.25, 0.0625)      # dyadic: node coordinates map to integer u exactly
    phi = rng.normal(size=n)
    X = R.node_coords(n, lc, h).reshape(-1, 3)
    P, g, H = CR.evaluate(phi, lc, h, X)
    assert np.array_equal(P, phi.reshape(-1))
    assert np.all(np.isfinite(g)) and np.all(np.isfinite(H))
    out = np.array([[-0.5 - 1e-12, 1.0, 0.25], [0.2, 1.0 + 1e-9, 0.25], [0.0, 0.0, 0.25 + 6 * 0.0625 + 1e-12], [np.nan, 0.0, 0.5]])
    P, g, H = CR.evaluate(phi, lc, h, out)
    assert np.all(np.isnan(P)) and np.all(np.isnan(g)) and np.all(np.isnan(H))
    phi[2, 2, 3] = np.nan                                                 # a NaN node poisons every stencil that holds it
    P, _, _ = CR.evaluate(phi, lc, h, np.array([[-0.5 + 2.3 * 0.125, 1.0 - 2.5 * 0.25, 0.25 + 3.1 * 0.0625]]))
    assert np.isnan(P[0])


def ellipse2d(n=(41, 37), lc=(-1.0, -0.9), hc=(1.0, 0.9)):
    """An ellipse whose axes are not grid lines: the interpolant is only continuous across cell faces, so a closest point on a face
    (every node on a symmetry axis that is a grid line has one) can make Newton alternate between two patches and fall back."""
    h = grid_h(lc, hc, n)
    x = R.node_coords(n, lc, h)
    return np.sqrt(((x[..., 0] - 0.013) / 0.7) ** 2 + ((x[..., 1] + 0.021) / 0.45) ** 2) - 1.0, lc, h


def test_refined_points_satisfy_kkt():
    phi, lc, h = ellipse2d()
    P, _ = R.band_phase(phi, lc, h, 3)
    x = R.node_coords(phi.shape, lc, h)
    has = ~np.isnan(P[..., 0])
    y, fell, iters = CR.refine(phi, lc, h, x[has], P[has])
    ok = ~fell
    assert ok.mean() > 0.99 and iters[ok].max() <= 8
    v, g, _ = CR.evaluate(phi, lc, h, y[ok])
    assert np.abs(v).max() <= 1e-12
    d = x[has][ok] - y[ok]
    cross = d[:, 0] * g[:, 1] - d[:, 1] * g[:, 0]
    assert np.all(np.abs(cross) <= 1e-9 * np.hypot(d[:, 0], d[:, 1]) * np.hypot(g[:, 0], g[:, 1]) + 1e-15)


def test_2d_distances_match_brute_force_on_the_cubic_zero_set():
    phi, lc, h = ellipse2d((29, 27))
    out, nb, nf = CR.redistance_cubic(phi, lc, h, band=3)
    # the zero set of the interpolant, sampled at h/64 along both axes of every cut cell, crossings located by bisection
    k = 64
    pts = []
    n = phi.shape
    for i, j in itertools.product(range(n[0] - 1), range(n[1] - 1)):
        c = phi[i:i + 2, j:j + 2]
        if not (c.min() <= 0.05 and c.max() >= -0.05):
            continue
        t = np.arange(k + 1) / k
        for axis in (0, 1):
            a, b = np.meshgrid(t, t, indexing="ij")
            u = np.stack([i + (a if axis == 0 else b), j + (b if axis == 0 else a)], -1).reshape(k + 1, k + 1, 2)
            Y = np.array(lc) + u * np.array(h)
            v = CR.evaluate(phi, lc, h, Y.reshape(-1, 2))[0].reshape(k + 1, k + 1)
            s = np.nonzero(np.sign(v[:, :-1]) != np.sign(v[:, 1:]))
            lo, hi = Y[s[0], s[1]], Y[s[0], s[1] + 1]
            for _ in range(40):
                mid = 0.5 * (lo + hi)
                vm = CR.evaluate(phi, lc, h, mid)[0]
                vl = CR.evaluate(phi, lc, h, lo)[0]
                left = np.sign(vm) == np.sign(vl)
                lo = np.where(left[:, None], mid, lo)
                hi = np.where(left[:, None], hi, mid)
            pts.append(0.5 * (lo + hi))
    Z = np.concatenate(pts)
    x = R.node_coords(n, lc, h).reshape(-1, 2)
    near = np.abs(phi.reshape(-1)) < 2 * min(h)
    bf = np.array([np.sqrt(((Z - p) ** 2).sum(1)).min() for p in x[near]])
    got = np.abs(out.reshape(-1)[near])
    # the samples are at most s = h/64 sqrt(2) apart along the curve, so brute force overestimates a distance d by about
    # (s/2)^2 / (2 d): the refined distance is never above it, and below it by no more than that
    assert nf == 0
    assert np.all(got <= bf + 1e-12)
    s = min(h) / 64 * math.sqrt(2)
    assert np.all(bf - got <= (s / 2) ** 2 / got)


def test_plane_gives_the_exact_distance():
    n, lc, h = (9, 10, 8), (-0.5, -0.5, -0.5), (0.125, 0.125, 0.125)
    x = R.node_coords(n, lc, h)
    nrm = np.array([0.36, 0.48, 0.8])
    phi = ((nrm[0] * x[..., 0] + nrm[1] * x[..., 1]) + nrm[2] * x[..., 2]) - 0.03
    exact = phi / np.linalg.norm(nrm)
    out, nb, nf = CR.redistance_cubic(phi, lc, h, band=3)
    # where the foot of the perpendicular lies outside the box, Newton leaves the box and the node keeps the distance to the
    # clipped linear mesh; everywhere else the distance is exact
    foot = x - (exact / np.linalg.norm(nrm))[..., None] * nrm
    inbox = np.all((foot > -0.5) & (foot < np.array([0.5, 0.625, 0.375])), axis=-1)
    assert nb > 0 and 0 < nf < np.sum(~inbox) + 1
    assert np.abs(out - exact)[inbox].max() <= 1e-15


def test_no_fallback_near_a_sphere():
    # Every node within 3h of an exact-distance sphere is refined.  The fallbacks (90 of 110 592 nodes, the nearest 4h from the
    # interface) are far nodes whose flooded seed lies more than 2h from their cubic closest point (40), or where Newton alternates
    # for 20 iterations between two patches across a cell face, where the interpolant is only continuous (50).  On coarser grids
    # that can happen within 3h too (2 nodes at 32^3 and at 40^3).  The device equals this restatement bit for bit
    # (test_redistance_cubic_equals_restatement), and test_third_order_on_a_sphere checks the same on the device at 64^3 and 128^3.
    n = 48
    lc, h = (-0.5,) * 3, [1.0 / (n - 1)] * 3
    x = R.node_coords((n,) * 3, lc, h)
    exact = np.sqrt(((x[..., 0] - 0.02) ** 2 + (x[..., 1] + 0.01) ** 2) + x[..., 2] ** 2) - 0.3
    P, _ = R.band_phase(exact, lc, h, 3)
    P = R.propagate(P, lc, h)
    y, fell, iters = CR.refine(exact, lc, h, x.reshape(-1, 3), P.reshape(-1, 3))
    near = (np.abs(exact) < 3 * h[0]).reshape(-1)
    assert near.sum() > 1000 and not np.any(fell & near)
    assert iters[near].max() <= 6


def test_fallback_rules():
    n, lc, h = (12, 12), (0.0, 0.0), (0.1, 0.1)
    x = R.node_coords(n, lc, h)
    plane = x[..., 0] - 0.55
    X, Y0 = np.array([[0.3, 0.4]]), np.array([[0.55, 0.4]])
    y, fell, _ = CR.refine(plane, lc, h, X, Y0)                         # the seed is the answer: converges, no fallback
    assert not fell[0] and np.abs(y - [[0.55, 0.4]]).max() <= 1e-15
    # a far seed: Newton moves more than 2 max h from it
    y, fell, _ = CR.refine(plane, lc, h, X, np.array([[0.55, 0.9]]))
    assert fell[0] and np.array_equal(y, [[0.55, 0.9]])
    # NaN in the stencil
    q = plane.copy()
    q[6, 4] = np.nan
    y, fell, _ = CR.refine(q, lc, h, X, Y0)
    assert fell[0] and np.array_equal(y, Y0)
    # a flat patch: grad P = 0 at the seed
    flat = np.where(x[..., 0] < 0.85, 0.0, x[..., 0] - 0.85)
    y, fell, _ = CR.refine(flat, lc, h, X, np.array([[0.3, 0.4]]))
    assert fell[0]
    # and through the whole pipeline: a NaN node makes its neighbours fall back, they keep the linear distance
    phi, lc2, h2 = ellipse2d((25, 23))
    phi[12, 4] = np.nan
    out, nb, nf = CR.redistance_cubic(phi, lc2, h2, band=3)
    lin, _ = R.redistance(phi, lc2, h2, 3)
    assert nf > 0 and np.isnan(out[12, 4])
    v = ~np.isnan(phi)
    assert np.array_equal(out[v] <= 0, phi[v] <= 0) and np.array_equal(np.isnan(out), np.isnan(lin))


def test_abi_argument_checks_without_a_device(m):
    lib, L = m._lib.lib(), m._lib
    nb, nf = C.c_int64(-1), C.c_int64(-1)
    assert lib.lsm_redistance_cubic(None, None, 0, C.byref(nb), C.byref(nf)) == L.ERR_ARG and "band" in L.last_error()
    assert lib.lsm_redistance_cubic(None, None, 3, None, None) == L.ERR_ARG and "null" in L.last_error()
    assert nb.value == -1 and nf.value == -1
    assert lib.lsm_interpolate_cubic(None, None, 1, None, None, None, None) == L.ERR_ARG and "null" in L.last_error()
    with pytest.raises(ValueError):
        m.redistance(None, order=2)


# ================================================================================================
# device == restatement, bit for bit
# ================================================================================================
def _cases():
    out = {}
    x = np.linspace(-1, 1, 37)
    v1 = np.sin(7 * x) + 0.1
    v1[5] = 0.0
    v1[20] = np.nan
    out["1d"] = (v1, (-1.0,), (1.0,))
    h2 = grid_h((-1, -1.5), (1.2, 1.5), (37, 53))
    x2 = R.node_coords((37, 53), (-1, -1.5), h2)
    out["2d_odd_aniso"] = (np.hypot(x2[..., 0] - 0.1, x2[..., 1]) ** 2 - 0.55 ** 2 + 0.1 * np.sin(3 * x2[..., 1]), (-1, -1.5), (1.2, 1.5))
    out["2d_mirrored"] = (np.hypot(x2[..., 0] - 0.1, x2[..., 1]) - 0.55, (1.2, -1.5), (-1, 1.5))
    h3 = grid_h((-0.5, -0.6, -0.4), (0.55, 0.6, 0.45), (29, 33, 23))
    x3 = R.node_coords((29, 33, 23), (-0.5, -0.6, -0.4), h3)
    phi = np.sqrt(((x3[..., 0] - 0.03) ** 2 + (x3[..., 1] + 0.02) ** 2) + (x3[..., 2] - 0.01) ** 2) - 0.33
    out["3d_odd_aniso"] = (phi * (1.5 + phi), (-0.5, -0.6, -0.4), (0.55, 0.6, 0.45))
    out["3d_mirrored"] = (phi, (0.55, -0.6, -0.4), (-0.5, 0.6, 0.45))
    g = R.node_coords((27, 25, 29), (-0.5,) * 3, grid_h((-0.5,) * 3, (0.5,) * 3, (27, 25, 29)))
    ball = np.sqrt((g[..., 0] ** 2 + g[..., 1] ** 2) + g[..., 2] ** 2) - 0.35
    q = ball.copy()
    q[3:6, 10:12, 4] = np.nan
    q[13, 13, 20:23] = np.nan
    out["3d_nan"] = (q, (-0.5,) * 3, (0.5,) * 3)
    out["3d_all_positive"] = (ball + 2.0, (-0.5,) * 3, (0.5,) * 3)
    h4 = grid_h((-1, -1, -1), (1, 1, 1), (4, 5, 4))
    x4 = R.node_coords((4, 5, 4), (-1, -1, -1), h4)
    out["3d_n4"] = (((x4[..., 0] ** 2 + x4[..., 1] ** 2) + x4[..., 2] ** 2) - 0.6, (-1, -1, -1), (1, 1, 1))
    return out


CASES = _cases()


def _points(vals, lc, hc, seed):
    """points inside the box, on cell faces (half-integer and integer u), on box faces, and outside"""
    rng = np.random.default_rng(seed)
    n = np.array(vals.shape)
    N = len(n)
    h = np.array(grid_h(lc, hc, vals.shape))
    U = rng.uniform(0, 1, (400, N)) * (n - 1)
    U[:60, 0] = np.floor(U[:60, 0])
    U[60:100] = np.round(U[60:100])
    U[100:130, -1] = 0.0
    U[130:160, 0] = n[0] - 1
    U[160:200] = rng.uniform(-0.6, 0, (40, N))
    U[200:220, -1] = n[-1] - 1 + 0.3
    return np.array(lc) + U * h


def _interp(m, phi, Y):
    N = Y.shape[1]
    n = len(Y)
    val, grad, hess = np.empty(n), np.empty((n, N)), np.empty((n, N, N))
    p = lambda a: C.cast(a.ctypes.data, C.POINTER(C.c_double))
    m._lib.check(m._lib.lib().lsm_interpolate_cubic(phi._context().handle, phi.device(), n, p(np.ascontiguousarray(Y)), p(val), p(grad), p(hess)))
    return val, grad, hess


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("name", list(CASES))
def test_interpolate_equals_restatement(m, name, dtype):
    vals, lc, hc = CASES[name]
    vals = vals.astype(dtype)
    Y = _points(vals, lc, hc, len(name))
    got = _interp(m, on_device(m, vals, lc, hc, dtype), Y)
    want = CR.evaluate(vals, lc, grid_h(lc, hc, vals.shape), Y)
    for a, b in zip(got, want):
        assert same_values(a, b)
    assert np.all(np.isnan(got[0][160:220]))
    res = m.interpolate(on_device(m, vals, lc, hc, dtype), Y)                  # the Python wrapper, and NULL outputs
    assert all(same_values(a, b) for a, b in zip(res, want))
    ph = on_device(m, vals, lc, hc, dtype)
    v = np.empty(len(Y))
    m._lib.check(m._lib.lib().lsm_interpolate_cubic(ph._context().handle, ph.device(), len(Y),
                                                    C.cast(np.ascontiguousarray(Y).ctypes.data, C.POINTER(C.c_double)),
                                                    C.cast(v.ctypes.data, C.POINTER(C.c_double)), None, None))
    assert same_values(v, want[0])


def _run(m, phi, band):
    ctx = phi._context()
    nb, nf = C.c_int64(-1), C.c_int64(-1)
    m._lib.check(m._lib.lib().lsm_redistance_cubic(ctx.handle, phi.device(), band, C.byref(nb), C.byref(nf)))
    phi._mark_device_advanced()
    return np.array(phi.peek()), nb.value, nf.value


@pytest.mark.gpu
@pytest.mark.parametrize("band", [3, 1, 5])
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("name", list(CASES))
def test_redistance_cubic_equals_restatement(m, name, dtype, band):
    vals, lc, hc = CASES[name]
    vals = vals.astype(dtype)
    got, nb, nf = _run(m, on_device(m, vals, lc, hc, dtype), band)
    want, nb_want, nf_want = CR.redistance_cubic(vals, lc, grid_h(lc, hc, vals.shape), band)
    assert (nb, nf) == (nb_want, nf_want)
    assert bits_equal(got, want)
    if name == "3d_all_positive":
        assert nb == 0 and nf == 0 and bits_equal(got, vals)
    if name == "3d_nan":
        assert nf > 0                                                          # stencils holding a NaN node fall back


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
def test_zalesak_disk_equals_restatement(m, dtype):
    phi, g = zalesak(m, 101, dtype)
    before = np.array(phi.peek())
    got, nb, nf = _run(m, phi, 3)
    want, nb_want, nf_want = CR.redistance_cubic(before, g.lc, g.meshsize(), 3)
    assert (nb, nf) == (nb_want, nf_want)
    assert bits_equal(got, want)
    assert np.array_equal(got <= 0, before <= 0)


# ================================================================================================
# accuracy, determinism, asynchrony, invalidation, prehook, errors
# ================================================================================================
@pytest.mark.gpu
def test_third_order_on_a_sphere(m):
    errs, errs1 = [], []
    for n in (64, 128):
        g = m.CartesianGrid((-0.5,) * 3, (0.5,) * 3, (n, n, n))
        x = R.node_coords(g.n, g.lc, g.meshsize())
        exact = np.sqrt(((x[..., 0] - 0.02) ** 2 + (x[..., 1] + 0.01) ** 2) + x[..., 2] ** 2) - 0.3
        near = np.abs(exact) < 3 * g.meshsize(1)
        phi = m.MeshField(np.asfortranarray(exact), g)
        got, nb, nf = _run(m, phi, 3)
        errs.append(float(np.abs(got - exact)[near].max()))
        lin = np.array(m.redistance(m.MeshField(np.asfortranarray(exact), g)).peek())
        errs1.append(float(np.abs(lin - exact)[near].max()))
        print(f"n = {n}: max error within 3h, order 3 {errs[-1]:.3e}, order 1 {errs1[-1]:.3e}; fallbacks {nf} of {lin.size}")
        # a node that falls back gets order 1's value bit for bit, a refined one (almost surely) does not: no fallback within 3h.
        # The count comes from far nodes (measured on a B200: 213 of 262 144 nodes at 64^3, 3332 of 2 097 152 at 128^3):
        # test_no_fallback_near_a_sphere checks the same per node with the restatement and says why they fall back
        assert not np.any((got == lin) & near)
        assert nf < 1e-2 * lin.size
    order = math.log2(errs[0] / errs[1])
    print("observed order", order)
    assert order >= 3.0, errs                # measured on a B200: 2.76e-7 and 1.66e-8, order 4.06; order 1: 3.07e-4, 7.68e-5
    assert errs[1] * 20 <= errs1[1], (errs, errs1)


@pytest.mark.gpu
def test_deterministic_and_asynchronous(m):
    vals, lc, hc = CASES["3d_odd_aniso"]
    ctx = m.default_context()
    a = on_device(m, vals, lc, hc, np.float64)
    b = on_device(m, vals, lc, hc, np.float64)
    a.device(), b.device()
    ctx.reset_counters()
    assert m.redistance(a, order=3) is a
    c = ctx.counters()
    assert c["d2h_bytes"] == 0 and c["h2d_bytes"] == 0
    assert c["kernel_launches"] == 6 + len(R.flood_steps(vals.shape))     # flag, 2 cell passes, pick, flooding, refine, write
    nb, nf = C.c_int64(-1), C.c_int64(-1)
    m._lib.check(m._lib.lib().lsm_redistance_cubic(ctx.handle, b.device(), 3, C.byref(nb), C.byref(nf)))
    b._mark_device_advanced()
    assert ctx.counters()["d2h_bytes"] == 16 and nb.value > 0 and nf.value >= 0     # one 16-byte copy of the two counts
    assert bits_equal(np.array(a.peek()), np.array(b.peek()))
    with pytest.raises(ValueError):
        m.redistance(a, order=2)


@pytest.mark.gpu
def test_cfl_cache_sees_new_values(m):
    g = m.CartesianGrid((-1.0, -1.0), (1.0, 1.0), (65, 61))
    x = R.node_coords(g.n, g.lc, g.meshsize())
    phi = m.MeshField(np.asfortranarray(np.hypot(x[..., 0], x[..., 1]) - 0.5), g, bc=m.NeumannBC())
    speed = m.MeshField(np.asfortranarray(3.0 * (x[..., 0] ** 2 + x[..., 1] ** 2) - 0.2), g)
    terms = (m.NormalMotionTerm(speed),)
    dt0 = m.compute_cfl(terms, phi, 0.0)
    m.compute_cfl(terms, phi, 0.0)
    m.redistance(speed, order=3)
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
    m.integrate(eqs[0], tf, prehook=lambda ls: m.redistance(ls.state, order=3))
    c = ctx.counters()
    assert c["d2h_bytes"] < 64 * max(1, eqs[0].steps_taken) and c["h2d_bytes"] == 0
    e = eqs[1]
    phi, tc, steps = e.state, 0.0, 0
    while tc <= tf - float(np.spacing(abs(tc))):
        m.redistance(phi, order=3)
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
        pt = np.array([[0.5, 0.5]])
        pp = C.cast(pt.ctypes.data, C.POINTER(C.c_double))
        vec = m.MeshField(np.zeros((2, 9, 8)), g, ctx=fresh)
        assert lib.lsm_redistance_cubic(fresh.handle, vec.device(), 3, None, None) == L.ERR_ARG
        assert lib.lsm_interpolate_cubic(fresh.handle, vec.device(), 1, pp, None, None, None) == L.ERR_ARG
        sep = m.SeparableVelocity(g, (1.0, 1.0), [[np.ones(9), np.ones(8)], [np.ones(9), np.ones(8)]], ctx=fresh)
        assert lib.lsm_redistance_cubic(fresh.handle, sep.device(), 3, None, None) == L.ERR_ARG
        thin = m.MeshField(np.zeros((9, 3)) - 1, m.CartesianGrid((0, 0), (1, 1), (9, 3)), ctx=fresh)
        assert lib.lsm_redistance_cubic(fresh.handle, thin.device(), 3, None, None) == L.ERR_ARG and "4 nodes" in L.last_error()
        assert lib.lsm_interpolate_cubic(fresh.handle, thin.device(), 1, pp, None, None, None) == L.ERR_ARG
        assert lib.lsm_redistance(fresh.handle, thin.device(), 3, None) == L.OK           # order 1 only needs 2 nodes
        sc = m.MeshField(np.zeros((9, 8)) - 1, g, ctx=fresh)
        assert lib.lsm_redistance_cubic(fresh.handle, sc.device(), 0, None, None) == L.ERR_ARG
        assert lib.lsm_redistance_cubic(m.default_context().handle, sc.device(), 3, None, None) == L.ERR_ARG
        assert lib.lsm_interpolate_cubic(fresh.handle, sc.device(), -1, pp, None, None, None) == L.ERR_ARG
        assert lib.lsm_interpolate_cubic(fresh.handle, sc.device(), 1, None, None, None, None) == L.ERR_ARG
        assert lib.lsm_interpolate_cubic(fresh.handle, sc.device(), 0, None, None, None, None) == L.OK
        assert lib.lsm_redistance_cubic(fresh.handle, sc.device(), 3, None, None) == L.OK
        with pytest.raises(m.LSMError):
            m.redistance(sc, band=0, order=3)
        with pytest.raises(ValueError):
            m.interpolate(sc, np.zeros((3, 3)))
        del vec, sep, thin, sc
    finally:
        fresh.close()

