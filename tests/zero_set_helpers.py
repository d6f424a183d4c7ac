"""Helpers shared by the tests of the zero-level-set operations (test_interface.py, test_redistance.py, test_extension.py and
test_redistance_cubic.py): the module fixture, grids, analytic level sets, bit comparison, device fields, and the redistancing
cases that the extension reuses."""
import numpy as np
import pytest

import redistance_ref as R


@pytest.fixture(scope="module")
def m():
    import lsm_b200
    return lsm_b200


def grid_h(lc, hc, n):
    return [(hc[d] - lc[d]) / (n[d] - 1) for d in range(len(n))]


def sphere(n, r=0.3, lc=(-0.5,) * 3, hc=(0.5,) * 3, c=(0.02, -0.01, 0.0)):
    h = grid_h(lc, hc, n)
    x = R.node_coords(n, lc, h)
    return np.sqrt(((x[..., 0] - c[0]) ** 2 + (x[..., 1] - c[1]) ** 2) + (x[..., 2] - c[2]) ** 2) - r, h


def torus(n, R0=0.28, r=0.11):
    lc, hc = (-0.5,) * 3, (0.5,) * 3
    h = grid_h(lc, hc, n)
    x = R.node_coords(n, lc, h)
    return np.sqrt((np.sqrt(x[..., 0] ** 2 + x[..., 1] ** 2) - R0) ** 2 + x[..., 2] ** 2) - r, h


def bits_equal(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return (a.dtype == b.dtype and a.shape == b.shape
            and np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8)))


def zalesak(m, n, dtype=np.float64):
    """The Zalesak disk of docs/src/example-zalesak.md built on the device: a disk minus a slot."""
    g = m.CartesianGrid((0.0, 0.0), (1.0, 1.0), (n, n))
    disk = m.MeshField.from_shape(g, "sphere", (0.5, 0.75, 0.15), dtype=dtype)
    slot = m.MeshField.from_shape(g, "box", (0.5, 0.725, 0.05, 0.25), dtype=dtype)
    return m.setdiff_(disk, slot), g


def on_device(m, vals, lc, hc, dtype, ctx=None, bc=None):
    """A MeshField holding vals (rounded to dtype) on the grid from lc to hc."""
    return m.MeshField(np.asfortranarray(np.asarray(vals).astype(dtype)), m.CartesianGrid(lc, hc, np.shape(vals)), bc=bc, ctx=ctx)


def _cases():
    out = {}
    x = np.linspace(-1, 1, 37)
    v1 = np.sin(7 * x) + 0.1
    v1[5] = 0.0
    v1[20] = np.nan
    out["1d"] = (v1, (-1.0,), (1.0,))
    h2 = grid_h((-1, -1.5), (1.2, 1.5), (37, 53))
    x2 = R.node_coords((37, 53), (-1, -1.5), h2)
    out["2d_odd_aniso"] = (np.hypot(x2[..., 0] - 0.1, x2[..., 1]) ** 2 - 0.55 ** 2, (-1, -1.5), (1.2, 1.5))
    out["2d_mirrored"] = (np.hypot(x2[..., 0] - 0.1, x2[..., 1]) - 0.55, (1.2, -1.5), (-1, 1.5))
    phi, _ = sphere((29, 33, 23), r=0.33, lc=(-0.5, -0.6, -0.4), hc=(0.55, 0.6, 0.45), c=(0.03, -0.02, 0.01))
    out["3d_odd_aniso"] = (phi * (1.5 + phi), (-0.5, -0.6, -0.4), (0.55, 0.6, 0.45))
    out["3d_mirrored"] = (phi, (0.55, -0.6, -0.4), (-0.5, 0.6, 0.45))
    h3 = grid_h((-0.5,) * 3, (0.5,) * 3, (27, 25, 29))
    x3 = R.node_coords((27, 25, 29), (-0.5,) * 3, h3)
    ball = np.sqrt((x3[..., 0] ** 2 + x3[..., 1] ** 2) + x3[..., 2] ** 2) - 0.35
    slot = np.maximum(np.maximum(np.abs(x3[..., 0]) - 0.06, np.abs(x3[..., 1] + 0.25) - 0.25), np.abs(x3[..., 2]) - 0.5)
    out["3d_notched_sphere"] = (np.maximum(ball, -slot), (-0.5,) * 3, (0.5,) * 3)
    q = np.round(ball * 16) / 16            # many exact zeros at nodes, and NaN nodes
    q[3:6, 10:12, 4] = np.nan
    q[13, 13, 20:23] = np.nan
    out["3d_zeros_nan"] = (q, (-0.5,) * 3, (0.5,) * 3)
    out["3d_all_positive"] = (ball + 2.0, (-0.5,) * 3, (0.5,) * 3)
    return out


# (values, lc, hc) of the device-equals-restatement tests of lsm_redistance and lsm_extend_closest_point
CASES = _cases()


def _band_cases():
    out = {}
    phi, h = sphere((16, 17, 15), r=0.27)
    out["sphere"] = (phi, (-0.5,) * 3, h)
    phi, h = torus((20, 20, 14))
    out["torus"] = (phi, (-0.5,) * 3, h)
    lc, hc = (-0.5, -0.6, -0.4), (0.55, 0.6, 0.45)
    phi, h = sphere((15, 26, 11), r=0.3, lc=lc, hc=hc)
    out["aniso"] = (phi, lc, h)
    lc, hc = (0.55, -0.6, -0.4), (-0.5, 0.6, 0.45)
    phi, h = sphere((15, 19, 13), r=0.3, lc=lc, hc=hc)
    out["mirrored"] = (phi, lc, h)
    return out


# (values, lc, h) of the brute-force checks of the restatement's band scan, propagation and extension
BAND_CASES = _band_cases()
