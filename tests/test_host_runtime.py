"""The host runtime's shared field checks and boundary-condition overrides, through the C ABI.

- lsm_max_abs_diff refuses fields of another shape or dimension, even with as many nodes.
- A temporary boundary condition (LinearExtrapolationBC for lsm_perimeter, phi's BCs on F for lsm_extend_along_normals) is gone
  once the call returns, on the field and on the stage buffers created during the call.
- Every entry point on the shared checks refuses a field of another context, a separable field, a field with the wrong number of
  components and a field of another shape with LSM_ERR_ARG, before any device work."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


class Runtime:
    """Two contexts on device 0 and the fields made on them (destroyed with the fixture)."""

    def __init__(self):
        import lsm_b200
        self.L = lsm_b200._lib
        self.lib = self.L.lib()
        self.ctx = [self._ctx(), self._ctx()]
        self.fields = []

    def _ctx(self):
        h = C.c_void_p()
        self.ok(self.lib.lsm_ctx_create(0, C.byref(h)))
        return h

    def ok(self, rc):
        assert rc == self.L.OK, (rc, self.L.last_error())

    def field(self, n, ncomp=1, vals=None, ctx=0, bc=None):
        """A Float64 field of context `ctx` holding vals (default 0), x fastest; bc: one lsm_bc kind/P pair for every side."""
        h = C.c_void_p()
        self.ok(self.lib.lsm_field_create(self.ctx[ctx], len(n), (C.c_int32 * len(n))(*n), self.L.F64, ncomp, None, None,
                                          C.byref(h)))
        self.fields.append(h)
        self.upload(h, np.zeros(int(np.prod(n)) * ncomp) if vals is None else vals)
        if bc is not None:
            self.set_bc(h, len(n), bc)
        return h

    def separable(self, n, ctx=0):
        h = C.c_void_p()
        nd = len(n)
        tabs = np.ones(nd * sum(n))
        self.ok(self.lib.lsm_field_create_separable(self.ctx[ctx], nd, (C.c_int32 * nd)(*n), None, None, (C.c_double * nd)(*[1.0] * nd),
                                                    tabs.ctypes.data_as(C.POINTER(C.c_double)), C.byref(h)))
        self.fields.append(h)
        return h

    def upload(self, h, vals):
        vals = np.ascontiguousarray(vals, dtype=np.float64)
        self.ok(self.lib.lsm_field_upload(h, vals.ctypes.data))

    def set_bc(self, h, ndim, bc):
        arr = (self.L.lsm_bc * (2 * ndim))()
        for s in arr:
            s.kind, s.P = bc
        self.ok(self.lib.lsm_field_set_bc(h, arr))

    def getindex(self, h, idx):
        """(status, values) of 1-based 2-D indices."""
        flat = np.asarray(idx, dtype=np.int32).ravel()
        out = (C.c_double * len(idx))()
        rc = self.lib.lsm_field_getindex(h, flat.ctypes.data_as(C.POINTER(C.c_int32)), len(idx), out)
        return rc, list(out)

    def close(self):
        for h in self.fields:
            self.lib.lsm_field_destroy(h)
        for c in self.ctx:
            self.lib.lsm_ctx_destroy(c)


@pytest.fixture(scope="module")
def rt():
    r = Runtime()
    yield r
    r.close()


def circle(n, r=0.3):
    """Signed distance to a circle on [0, 1]^2, x fastest."""
    x = np.linspace(0.0, 1.0, n[0])[:, None]
    y = np.linspace(0.0, 1.0, n[1])[None, :]
    return (np.sqrt((x - 0.52) ** 2 + (y - 0.47) ** 2) - r).ravel(order="F")


def test_max_abs_diff_refuses_fields_of_another_shape(rt):
    L, lib = rt.L, rt.lib
    d = C.c_double(-1.0)
    a, b = rt.field((10, 20), vals=np.arange(200.0)), rt.field((10, 20), vals=np.arange(200.0) + 0.5)
    rt.ok(lib.lsm_max_abs_diff(rt.ctx[0], a, b, C.byref(d)))
    assert d.value == 0.5
    for x, y in (((10, 20), (20, 10)), ((4, 50), (200,))):
        fa, fb = rt.field(x), rt.field(y)
        assert lib.lsm_max_abs_diff(rt.ctx[0], fa, fb, C.byref(d)) == L.ERR_ARG, (x, y)
        assert "shape" in L.last_error()


def test_perimeter_leaves_a_field_without_boundary_conditions(rt):
    L, lib = rt.L, rt.lib
    n = (16, 16)
    phi = rt.field(n, vals=circle(n))
    p = C.c_double()
    rt.ok(lib.lsm_perimeter(rt.ctx[0], phi, C.byref(p)))
    assert p.value > 0
    assert rt.getindex(phi, [(1, 1)])[0] == L.OK
    assert rt.getindex(phi, [(0, 1)])[0] == L.ERR_BC


def test_extend_along_normals_restores_the_boundary_conditions_of_F_and_its_stage_buffer(rt):
    L, lib = rt.L, rt.lib
    n = (16, 16)
    phi = rt.field(n, vals=circle(n), bc=(L.BC_EXTRAP, 0))           # Neumann
    F_per = rt.field(n, vals=circle(n), bc=(L.BC_PERIODIC, 0))
    F_none = rt.field(n, vals=circle(n))
    vals = np.arange(n[0] * n[1], dtype=np.float64) * 1.25 + 3.0     # distinct, x fastest
    ghost = [(0, 5), (n[0] + 1, 5), (7, 0), (7, n[1] + 1)]

    def node(i, j):
        return vals[(i - 1) + n[0] * (j - 1)]

    def periodic(i, m):                                               # node m duplicates node 1 (boundaryconditions.jl:107-119)
        return i + (m - 1) if i < 1 else i - (m - 1) if i > m else i

    want = [node(periodic(i, n[0]), periodic(j, n[1])) for i, j in ghost]
    assert want != [node(min(max(i, 1), n[0]), min(max(j, 1), n[1])) for i, j in ghost]    # not what Neumann would give
    for F, has_bc in ((F_per, True), (F_none, False)):
        rt.ok(lib.lsm_extend_along_normals(rt.ctx[0], F, phi, 3, 0.45, None, 1.5, 1e-14))
        buf = C.c_void_p()
        rt.ok(lib.lsm_field_stage_buffer(F, 1, C.byref(buf)))         # made by the extension's stages
        for h in (F, buf):
            rt.upload(h, vals)
            rc, got = rt.getindex(h, ghost)
            if has_bc:
                assert rc == L.OK and got == want
            else:
                assert rc == L.ERR_BC


def test_entry_points_refuse_unsuitable_fields(rt):
    """Each entry point on the shared checks, with one argument replaced by an unsuitable field: status LSM_ERR_ARG."""
    L, lib = rt.L, rt.lib
    n, other = (8, 8), (8, 16)
    A, B = rt.field(n, vals=circle(n)), rt.field(n, vals=circle(n))
    P = rt.field(n, vals=circle(n), bc=(L.BC_EXTRAP, 0))
    V = rt.field(n, ncomp=2)
    bad = {
        "context": rt.field(n, vals=circle(n), ctx=1),
        "separable": rt.separable(n),
        "components": rt.field(n, ncomp=2),
        "shape": rt.field(other, vals=circle(other)),
    }
    bad_vector = {"context": rt.field(n, ncomp=2, ctx=1), "separable": bad["separable"], "components": A,
                  "shape": rt.field(other, ncomp=2)}
    S = rt.separable(n)
    d = C.c_double()
    out4 = (C.c_double * 4)()
    buf = C.c_void_p()
    idx = (C.c_int32 * 2)(1, 1)

    def normal_term(coef):
        t = (L.lsm_term * 1)()
        t[0].kind, t[0].coef_kind, t[0].tscale_kind, t[0].field = L.TERM_NORMAL, L.COEF_FIELD, L.TS_NONE, coef.value
        return t

    def advection_const():
        t = (L.lsm_term * 1)()
        t[0].kind, t[0].scheme, t[0].coef_kind, t[0].tscale_kind = L.TERM_ADVECTION, L.WENO5, L.COEF_CONST, L.TS_NONE
        t[0].cval[0] = t[0].cval[1] = 1.0
        return t

    c0 = rt.ctx[0]
    calls = {   # name: (call with the unsuitable field x, kinds of unsuitable field it takes)
        "check_level_set (lsm_redistance)": (lambda x: lib.lsm_redistance(c0, x, 3, None), ("context", "separable", "components")),
        "check_state (lsm_compute_cfl)": (lambda x: lib.lsm_compute_cfl(c0, x, advection_const(), 1, 0.0, None, C.byref(d)),
                                          ("context", "separable", "components")),
        "lsm_volume": (lambda x: lib.lsm_volume(c0, x, C.byref(d)), ("context", "separable", "components")),
        "lsm_perimeter": (lambda x: lib.lsm_perimeter(c0, x, C.byref(d)), ("context", "separable", "components")),
        "lsm_extend_along_normals F": (lambda x: lib.lsm_extend_along_normals(c0, x, P, 1, 0.45, None, 1.5, 1e-14), tuple(bad)),
        "lsm_extend_along_normals phi": (lambda x: lib.lsm_extend_along_normals(c0, B, x, 1, 0.45, None, 1.5, 1e-14), tuple(bad)),
        "lsm_field_csg src": (lambda x: lib.lsm_field_csg(c0, B, x, 0), tuple(bad)),
        "lsm_field_csg dst": (lambda x: lib.lsm_field_csg(c0, x, None, 3), ("context", "separable", "components")),
        "lsm_eikonal_s0 dst": (lambda x: lib.lsm_eikonal_s0(x, A), tuple(bad)),
        "lsm_eikonal_s0 phi0": (lambda x: lib.lsm_eikonal_s0(B, x), tuple(bad)),
        "lsm_max_abs_diff": (lambda x: lib.lsm_max_abs_diff(c0, A, x, C.byref(d)), tuple(bad)),
        "lsm_field_getindex": (lambda x: lib.lsm_field_getindex(x, idx, 1, C.byref(d)), ("separable", "components")),
        "lsm_field_stage_buffer": (lambda x: lib.lsm_field_stage_buffer(x, 1, C.byref(buf)), ("separable", "components")),
        "make_term_dev (normal-motion coefficient)": (lambda x: lib.lsm_compute_cfl(c0, P, normal_term(x), 1, 0.0, None, C.byref(d)),
                                                      tuple(bad)),
        "lsm_field_copy src": (lambda x: lib.lsm_field_copy(B, x), tuple(bad)),
        "lsm_field_copy dst": (lambda x: lib.lsm_field_copy(x, A), tuple(bad)),
        "check_same_grid (lsm_extend_closest_point)": (lambda x: lib.lsm_extend_closest_point(c0, x, A, 3, 0, None), tuple(bad)),
        "check_same_grid (lsm_level_set_integrals)": (lambda x: lib.lsm_level_set_integrals(c0, A, x, 0.0, out4), tuple(bad)),
    }
    refused = []
    for name, (call, kinds) in calls.items():
        for k in kinds:
            refused.append((name, k, call(bad[k]), L.last_error()))
    for k in bad_vector:     # lsm_field_fill_separable wants a stored vector field of the separable field's shape
        refused.append(("lsm_field_fill_separable dst", k, lib.lsm_field_fill_separable(bad_vector[k], S), L.last_error()))
    wrong = [r for r in refused if r[2] != L.ERR_ARG]
    assert not wrong, wrong
    # the same calls with suitable fields pass the checks
    rt.ok(lib.lsm_field_fill_separable(V, S))
    rt.ok(lib.lsm_field_copy(B, A))
    rt.ok(lib.lsm_max_abs_diff(c0, A, B, C.byref(d)))
    assert d.value == 0.0
