"""Level-set integrals (lsm_level_set_integrals / lsm_multi_level_set_integrals, level_set_integrals, level_set_integrals_multi).

Without a GPU: the NumPy restatement of the contract (integrals_ref.py) against exact answers for a plane through a box with a linear
F (every output, 1-D to 3-D, anisotropic and mirrored grids, a plane of exact zeros at nodes), against the measure of
interface_ref.extract's mesh, and against the exact area / volume of a circle, a sphere and the Zalesak disk as the grid is refined;
edge cases; the argument checks of the C ABI that need no device.  On the GPU: the device equals the restatement to rounding over
dimensions, dtypes of phi and F, odd sizes, mirrored grids, NaN nodes, exact zeros, level != 0, F == phi and empty fields; repeated
calls are bitwise equal; the interface measure equals that of extract_interface's mesh; error codes, launches and D2H bytes; and on
two GPUs the slab-decomposed call equals the single-GPU call bit for bit."""
import ctypes as C
import itertools
import math

import numpy as np
import pytest

import integrals_ref as R
import redistance_ref as RR
from zero_set_helpers import CASES, m, on_device, sphere, zalesak  # noqa: F401 (m is a fixture)


def _rel(a, b):
    return abs(a - b) / max(abs(b), 1e-300)


# ================================================================================================
# the restatement against exact answers (no GPU)
# ================================================================================================
def _box_halfspace(lo, hi, nrm, c, a0, a):
    """Exact |{n.x <= c} cap box|, the measure of {n.x = c} cap box and the integrals of F = a0 + a.x over both, from a
    triangulation of the polytope (F is linear, so a simplex contributes its volume times F at its centroid)."""
    from scipy.spatial import Delaunay
    N = len(lo)
    F = lambda x: a0 + np.dot(a, x)
    corners = [np.array(v, dtype=float) for v in itertools.product(*zip(lo, hi))]
    g = lambda v: np.dot(nrm, v) - c
    cuts = []
    for v, w in itertools.combinations(corners, 2):
        if np.count_nonzero(v != w) == 1 and g(v) * g(w) < 0:
            cuts.append(v + g(v) / (g(v) - g(w)) * (w - v))
    pts = np.array([v for v in corners if g(v) <= 0] + cuts)
    if N == 1:
        x0, x1 = pts.min(), pts.max()
        return x1 - x0, float(len(cuts)), (x1 - x0) * F([(x0 + x1) / 2]), sum(F(p) for p in cuts)
    vol = fvol = 0.0
    for simp in Delaunay(pts).simplices:
        P = pts[simp]
        v = abs(np.linalg.det(P[1:] - P[0])) / math.factorial(N)
        vol += v
        fvol += v * F(P.mean(axis=0))
    cuts = np.array(cuts)
    if N == 2:
        L = np.linalg.norm(cuts[1] - cuts[0])
        return vol, L, fvol, L * F(cuts.mean(axis=0))
    ctr = cuts.mean(axis=0)
    e1 = cuts[0] - ctr
    e1 /= np.linalg.norm(e1)
    e2 = np.cross(nrm / np.linalg.norm(nrm), e1)
    order = np.argsort(np.arctan2((cuts - ctr) @ e2, (cuts - ctr) @ e1))
    poly = cuts[order]
    area = farea = 0.0
    for k in range(len(poly)):
        A = 0.5 * np.linalg.norm(np.cross(poly[k] - ctr, poly[(k + 1) % len(poly)] - ctr))
        area += A
        farea += A * F((ctr + poly[k] + poly[(k + 1) % len(poly)]) / 3)
    return vol, area, fvol, farea


PLANES = {
    "1d": ((-1.0,), (1.3,), (17,), (1.0,), 0.2117),
    "1d_mirrored": ((1.3,), (-1.0,), (17,), (1.0,), 0.2117),
    "2d_aniso": ((-1.0, -0.5), (1.2, 0.8), (13, 17), (0.6, 0.8), 0.1731),
    "2d_mirrored": ((1.2, -0.5), (-1.0, 0.8), (13, 17), (0.6, -0.8), 0.1731),
    "3d_aniso": ((-0.5, -0.6, -0.4), (0.55, 0.6, 0.45), (9, 11, 7), (0.48, 0.6, 0.64), 0.0513),
    "3d_mirrored": ((0.55, -0.6, 0.45), (-0.5, 0.6, -0.4), (9, 11, 7), (0.48, -0.6, 0.64), -0.0713),
}


def _plane_field(lc, hc, n, nrm, c, a0, a):
    h = [(hc[d] - lc[d]) / (n[d] - 1) for d in range(len(n))]
    x = RR.node_coords(n, lc, h)
    phi = x[..., 0] * nrm[0]
    F = a0 + x[..., 0] * a[0]
    for d in range(1, len(n)):
        phi = phi + x[..., d] * nrm[d]
        F = F + x[..., d] * a[d]
    return phi - c, F, h


@pytest.mark.parametrize("name", list(PLANES))
def test_plane_with_linear_F_is_exact(name):
    lc, hc, n, nrm, c = PLANES[name]
    N = len(n)
    a0, a = 1.7, (0.9, -1.3, 0.4)[:N]
    phi, F, h = _plane_field(lc, hc, n, nrm, c, a0, a)
    got = R.integrals(phi, lc, h, F=F)
    lo, hi = [min(p, q) for p, q in zip(lc, hc)], [max(p, q) for p, q in zip(lc, hc)]
    want = _box_halfspace(lo, hi, np.array(nrm), c, a0, np.array(a))
    for q in range(4):
        assert _rel(got[q], want[q]) < 1e-12, (q, got, want)
    # level shifts the plane: phi - level = n.x - (c + level)
    got = R.integrals(phi, lc, h, level=0.05, F=F)
    want = _box_halfspace(lo, hi, np.array(nrm), c + 0.05, a0, np.array(a))
    for q in range(4):
        assert _rel(got[q], want[q]) < 1e-12, (q, got, want)


@pytest.mark.parametrize("N", [2, 3])
def test_plane_of_exact_zeros_is_counted_once(N):
    lc, hc, n = (-0.5, -0.6, -0.4)[:N], (0.55, 0.6, 0.45)[:N], (9, 11, 13)[:N]
    h = [(hc[d] - lc[d]) / (n[d] - 1) for d in range(N)]
    x = RR.node_coords(n, lc, h)
    zk = lc[-1] + 5 * h[-1]
    phi = x[..., -1] - zk
    assert np.count_nonzero(phi == 0) == np.prod(n[:-1])           # a whole lattice plane of exact zeros
    a0, a = 0.3, np.array((0.5, -0.25, 0.75)[:N])
    F = a0 + x @ a
    vol, area, fvol, farea = R.integrals(phi, lc, h, F=F)
    base = np.prod([hc[d] - lc[d] for d in range(N - 1)])
    ctr = np.array([(lc[d] + hc[d]) / 2 for d in range(N - 1)])
    assert _rel(vol, base * (zk - lc[-1])) < 1e-12
    assert _rel(area, base) < 1e-12
    assert _rel(fvol, base * (zk - lc[-1]) * (a0 + ctr @ a[:-1] + a[-1] * (lc[-1] + zk) / 2)) < 1e-12
    assert _rel(farea, base * (a0 + ctr @ a[:-1] + a[-1] * zk)) < 1e-12


@pytest.mark.parametrize("name", ["2d_odd_aniso", "2d_mirrored", "3d_odd_aniso", "3d_mirrored", "3d_notched_sphere", "3d_zeros_nan"])
def test_interface_agrees_with_the_extracted_mesh(name):
    vals, lc, hc = CASES[name]
    h = [(hc[d] - lc[d]) / (vals.shape[d] - 1) for d in range(vals.ndim)]
    F = 2.0 + np.cos(np.arange(vals.size, dtype=np.float64).reshape(vals.shape) * 0.37)
    for level in (0.0, 0.013):
        _, area, _, farea = R.integrals(vals, lc, h, level, F)
        marea, mfarea = R.mesh_integrals(vals, lc, h, level, F)
        assert _rel(area, marea) < 1e-13 and _rel(farea, mfarea) < 1e-13


def _order(e0, e1):
    return math.log2(e0 / e1)


def test_convergence_sphere_circle_zalesak():
    r3, errs3 = 0.35, []
    for n in (24, 48):
        phi, h = sphere((n, n, n), r=r3, c=(0.013, -0.007, 0.004))
        vol, area, _, _ = R.integrals(phi, (-0.5,) * 3, h)
        errs3.append((abs(vol / (4 / 3 * math.pi * r3 ** 3) - 1), abs(area / (4 * math.pi * r3 ** 2) - 1)))
    r2, errs2, errsz = 0.37, [], []
    w, rz = 0.025, 0.15
    zal = math.pi * rz ** 2 - (2 * w * 0.1 + w * math.sqrt(rz ** 2 - w ** 2) + rz ** 2 * math.asin(w / rz))
    for n in (64, 128, 256):
        h = [2.0 / (n - 1)] * 2
        x = RR.node_coords((n, n), (-1.0, -1.0), h)
        phi = np.sqrt((x[..., 0] - 0.031) ** 2 + (x[..., 1] + 0.017) ** 2) - r2
        vol, area, _, _ = R.integrals(phi, (-1.0, -1.0), h)
        errs2.append((abs(vol / (math.pi * r2 ** 2) - 1), abs(area / (2 * math.pi * r2) - 1)))
        # the Zalesak disk of zero_set_helpers.zalesak, on the unit square (disk minus slot, as the device builds it)
        hz = [1.0 / (n - 1)] * 2
        xz = RR.node_coords((n, n), (0.0, 0.0), hz)
        disk = np.sqrt((xz[..., 0] - 0.5) ** 2 + (xz[..., 1] - 0.75) ** 2) - rz
        slot = np.maximum(np.abs(xz[..., 0] - 0.5) - 0.05 / 2, np.abs(xz[..., 1] - 0.725) - 0.25 / 2)
        vz, _, _, _ = R.integrals(np.maximum(disk, -slot), (0.0, 0.0), hz)
        errsz.append(abs(vz / zal - 1))
    # second order for the smooth shapes (observed about 2.0 for each), first order at least for the slot's corners
    for k in range(2):
        assert _order(errs3[0][k], errs3[1][k]) > 1.6, errs3
        assert _order(errs2[0][k], errs2[1][k]) > 1.6 and _order(errs2[1][k], errs2[2][k]) > 1.6, errs2
    assert errs3[1][0] < 2e-3 and errs3[1][1] < 2e-3 and errs2[2][0] < 1e-4 and errs2[2][1] < 1e-4, (errs3, errs2)
    assert errsz[2] < errsz[0] / 3 and errsz[2] < 2e-3, errsz


def test_edge_cases():
    vals, lc, hc = CASES["3d_odd_aniso"]
    h = [(hc[d] - lc[d]) / (vals.shape[d] - 1) for d in range(3)]
    box = abs(np.prod([hc[d] - lc[d] for d in range(3)]))
    F = np.full(vals.shape, 3.0)
    assert R.integrals(np.abs(vals) + 1.0, lc, h, F=F) == (0.0, 0.0, 0.0, 0.0)                 # empty
    vol, area, fvol, farea = R.integrals(-np.abs(vals) - 1.0, lc, h, F=F)                         # fully inside
    assert _rel(vol, box) < 1e-13 and area == 0.0 and _rel(fvol, 3.0 * box) < 1e-13 and farea == 0.0
    assert all(math.isnan(v) for v in R.integrals(vals, lc, h)[2:])                              # no F
    # a NaN node drops exactly the simplices it touches: the region shrinks, nothing becomes NaN
    q = vals.copy()
    q[10, 12, 8] = np.nan
    got, ref = R.integrals(q, lc, h, F=F), R.integrals(vals, lc, h, F=F)
    assert all(np.isfinite(got)) and got[0] < ref[0]
    # a NaN in F propagates
    Fn = F.copy()
    Fn[14, 16, 11] = np.nan
    assert math.isnan(R.integrals(vals, lc, h, F=Fn)[2])
    # level != 0 moves the interface outward
    assert R.integrals(vals, lc, h, level=0.01)[0] > ref[0]


def test_abi_argument_checks_without_a_device(m):
    lib = m._lib.lib()
    out = (C.c_double * 4)()
    assert lib.lsm_level_set_integrals(None, None, None, 0.0, out) == m._lib.ERR_ARG
    assert lib.lsm_multi_level_set_integrals(0, None, None, None, 0.0, out) == m._lib.ERR_ARG
    assert lib.lsm_multi_level_set_integrals(1, None, None, None, 0.0, None) == m._lib.ERR_ARG


# ================================================================================================
# the device against the restatement
# ================================================================================================
def _Fvals(shape):
    idx = np.indices(shape).astype(np.float64)
    return 2.0 + np.sin(0.3 * idx[0]) + (0.1 * idx[-1]) ** 2


def _dev_cases():
    out = {k: (v, lc, hc, 0.0) for k, v_ in CASES.items() for (v, lc, hc) in [v_]}
    v, lc, hc = CASES["3d_odd_aniso"]
    out["3d_level"] = (v, lc, hc, -0.021)
    v, lc, hc = CASES["2d_odd_aniso"]
    out["2d_level"] = (v, lc, hc, 0.05)
    return out


DEV = _dev_cases()


def _check(got, want, scale, with_F):
    for q in range(4 if with_F else 2):
        assert abs(got[q] - want[q]) <= 1e-13 * max(scale[q], 1e-300), (q, got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("fdt", [None, np.float64, np.float32, "phi"], ids=["noF", "F64", "F32", "Fphi"])
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("name", list(DEV))
def test_device_equals_restatement(m, name, dtype, fdt):
    vals, lc, hc, level = DEV[name]
    h = [(hc[d] - lc[d]) / (vals.shape[d] - 1) for d in range(vals.ndim)]
    phi = on_device(m, vals, lc, hc, dtype)
    pv = vals.astype(dtype)
    if fdt is None:
        F, Fv = None, None
    elif fdt == "phi":
        F, Fv = phi, pv
    else:
        Fv = _Fvals(vals.shape).astype(fdt)
        F = on_device(m, Fv, lc, hc, fdt)
    got = m.level_set_integrals(phi, F, level)
    want = R.integrals(pv, lc, h, level, Fv)
    _check(got, want, R.scales(pv, lc, h, level, Fv), F is not None)
    if F is None:
        assert got.F_inside is None and got.F_interface is None
    again = m.level_set_integrals(phi, F, level)
    assert tuple(got) == tuple(again)                      # bitwise: the order does not depend on scheduling
    if name == "3d_all_positive":
        assert got.inside == 0.0 and got.interface == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["2d_odd_aniso", "3d_odd_aniso", "3d_notched_sphere", "3d_zeros_nan"])
def test_interface_equals_the_extracted_mesh(m, name):
    vals, lc, hc = CASES[name]
    phi = on_device(m, vals, lc, hc, np.float64)
    mesh = m.extract_interface(phi)
    N = vals.ndim
    meas = R._measure([mesh.vertices[mesh.faces[:, j]] for j in range(N)], N).sum()
    assert _rel(m.level_set_integrals(phi).interface, meas) < 1e-13


@pytest.mark.gpu
def test_zalesak_disk_on_the_device(m):
    phi, g = zalesak(m, 201)
    w, rz = 0.025, 0.15
    exact = math.pi * rz ** 2 - (2 * w * 0.1 + w * math.sqrt(rz ** 2 - w ** 2) + rz ** 2 * math.asin(w / rz))
    got = m.level_set_integrals(phi)
    want = R.integrals(phi.peek(), g.lc, [g.meshsize(d + 1) for d in range(2)])
    assert _rel(got.inside, want[0]) < 1e-13 and _rel(got.inside, exact) < 2e-3


@pytest.mark.gpu
def test_error_codes_and_counters(m):
    lib, L = m._lib.lib(), m._lib
    fresh = m.Context(0)
    try:
        out = (C.c_double * 4)()
        g = m.CartesianGrid((0, 0), (1, 1), (9, 8))
        sc = m.MeshField(np.zeros((9, 8)) - 1, g, ctx=fresh)
        vec = m.MeshField(np.zeros((2, 9, 8)), g, ctx=fresh)
        assert lib.lsm_level_set_integrals(fresh.handle, vec.device(), None, 0.0, out) == L.ERR_ARG
        assert lib.lsm_level_set_integrals(fresh.handle, sc.device(), vec.device(), 0.0, out) == L.ERR_ARG
        other = m.MeshField(np.zeros((9, 8)), m.CartesianGrid((0, 0), (1, 2), (9, 8)), ctx=fresh)
        assert lib.lsm_level_set_integrals(fresh.handle, sc.device(), other.device(), 0.0, out) == L.ERR_ARG
        assert "F and phi must be on the same grid (n, lc and h)" in L.last_error()
        assert lib.lsm_level_set_integrals(fresh.handle, sc.device(), None, float("nan"), out) == L.ERR_ARG
        assert lib.lsm_level_set_integrals(fresh.handle, sc.device(), None, 0.0, None) == L.ERR_ARG
        thin = m.MeshField(np.zeros((9, 1)), m.CartesianGrid((0, 0), (1, 1), (9, 1)), ctx=fresh)
        assert lib.lsm_level_set_integrals(fresh.handle, thin.device(), None, 0.0, out) == L.ERR_ARG
        fresh.reset_counters()
        assert lib.lsm_level_set_integrals(fresh.handle, sc.device(), sc.device(), 0.0, out) == L.OK
        c = fresh.counters()
        assert c["kernel_launches"] == 2 and c["d2h_bytes"] == 32 and c["h2d_bytes"] == 0
        assert abs(out[0] - 1.0) < 1e-14 and out[1] == 0.0 and abs(out[2] + 1.0) < 1e-14
        del vec, sc, other, thin
    finally:
        fresh.close()


@pytest.mark.gpu
def test_extraction_is_left_alone(m):
    vals, lc, hc = CASES["3d_odd_aniso"]
    phi = on_device(m, vals, lc, hc, np.float64)
    mesh = m.extract_interface(phi)
    m.level_set_integrals(phi, phi)
    again = m.api._fetch_interface(m.default_context(), 3, len(mesh.keys), len(mesh.faces))
    for a, b in zip(mesh, again):
        assert np.array_equal(a, b)


# ================================================================================================
# two GPUs: the slab-decomposed call equals the single-GPU call bit for bit
# ================================================================================================
def _two_gpus(m):
    n = C.c_int32(0)
    m._lib.lib().lsm_device_count(C.byref(n))
    if n.value < 2:
        pytest.skip("needs 2 GPUs")


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["3d_uneven_F", "2d_along_y", "3d_periodic", "3d_stale"])
def test_multi_gpu_equals_single_gpu(m, case):
    _two_gpus(m)
    mc = m.MultiContext([0, 1])
    solo = m.Context(0)
    try:
        if case.startswith("2d"):
            shape, lc, hc = (37, 53), (-1.0, -1.5), (1.2, 1.5)
            h = [(hc[d] - lc[d]) / (shape[d] - 1) for d in range(2)]
            x = RR.node_coords(shape, lc, h)
            phi0 = np.hypot(x[..., 0] - 0.1, x[..., 1] - 0.05) - 0.55
        else:
            shape, lc, hc = (30, 26, 41), (-0.5,) * 3, (0.5,) * 3       # 41 planes: 21 + 20, the sphere crosses the slab boundary
            phi0, _ = sphere(shape, r=0.3, c=(0.05, -0.02, 0.45 if case == "3d_periodic" else 0.02))
        bc = m.PeriodicBC() if case == "3d_periodic" else m.NeumannBC()
        Fv = _Fvals(shape)
        phis = [on_device(m, phi0, lc, hc, np.float64, ctx=c, bc=bc) for c in mc.ranks]
        Fs = [on_device(m, Fv, lc, hc, np.float32, ctx=c, bc=bc) for c in mc.ranks] if case != "2d_along_y" else None
        if case == "3d_stale":                # new values after upload: the ghost planes are stale when the call is made
            for p in phis:
                p.device()
            for p in phis:
                p.vals[...] = -phi0[..., p._first:p._first + p._count] + 0.01
            phi0 = 0.01 - phi0
        got = m.level_set_integrals_multi(mc, phis, Fs)
        one = on_device(m, phi0, lc, hc, np.float64, ctx=solo, bc=bc)
        F1 = None if Fs is None else on_device(m, Fv, lc, hc, np.float32, ctx=solo, bc=bc)
        ref = m.level_set_integrals(one, F1)
        assert np.array_equal(np.array(tuple(got), dtype=object) == None, np.array(tuple(ref), dtype=object) == None)  # noqa: E711
        for a, b in zip(got, ref):
            assert (a is None and b is None) or np.float64(a).tobytes() == np.float64(b).tobytes(), (got, ref)
        assert ref.interface > 0
    finally:
        mc.close()
        solo.close()
