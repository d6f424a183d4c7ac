"""The fused RK-stage kernels of csrc/lsm_tiled.cu against the CPU oracle on grids of many tiles.

A block of the tiled kernel owns a 32 x 16 x-y tile and reads a 3-node halo; a tile whose halo lies inside the grid copies
it plainly (cp.async, or TMA in 3-D when rows are a multiple of 16 bytes), every other tile resolves ghosts, and in 3-D the
z march is split into chunks of 32 planes.  The small grids of test_gpu_parity.py are one tile wide, so only these shapes
reach interior tiles, tile seams, the TMA fill and the chunk starts with every term list and boundary condition:

  A = 72 x 52 x 70: 3 x 4 tiles (the last 8 wide and 4 high), plain-copy tiles at x0 = 32, y0 = 16 and 32, TMA in both
      dtypes, z chunks of 32, 32 and 6 planes;
  B = 71 x 40 x 45: no TMA (rows of 568 / 284 bytes), so the interior tile takes the cp.async plain copy; chunks 32, 13;
  C = 100 x 70: 4 x 5 tiles, partial at the far edges, with interior tiles.

test_shapes_cover_the_tile_geometry re-derives these facts from the constants of launch_tiled, so a retuned tile makes it
say which claim no longer holds.  Every difference is measured relative to max(1, max|phi|) of the oracle's state.
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import helpers as H

OPT_KERNEL = 0
TESTS = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(TESTS)
CSRC = os.path.join(REPO, "levelsetmethods.jl_b200", "csrc")

# ---- tile geometry: launch_tiled and TileGeom in csrc/lsm_tiled.cu, HAL in csrc/lsm_tile_util.cuh ----------------------
TX, TY, NY, XL, HAL = 32, 8, 2, 4, 3
TYNY = TY * NY                       # tile height
W = TX + 2 * XL                      # width of a staged row: x0 - XL .. x0 + TX + XL - 1


def z_chunk(nz):
    """Planes per block of the 3-D z march (launch_tiled's cz)."""
    return 64 if nz >= 128 else (32 if nz >= 32 else nz)


def tma_fill(n, itemsize):
    """launch_tiled builds TMA maps for 3-D grids whose rows are a multiple of 16 bytes and that have at least 32^3 nodes."""
    return len(n) == 3 and (n[0] * itemsize) % 16 == 0 and int(np.prod(n)) >= 32 ** 3


def tile_starts(n, t):
    return list(range(0, n, t))


def plain_tiles(n):
    """(x0, y0) of the tiles whose staged rows and halo rows all lie inside the grid (the kernel's xy_in)."""
    return [(x0, y0) for x0 in tile_starts(n[0], TX) for y0 in tile_starts(n[1], TYNY)
            if x0 - XL >= 0 and x0 - XL + W <= n[0] and y0 - HAL >= 0 and y0 + TYNY + HAL <= n[1]]


def z_chunks(nz):
    cz = z_chunk(nz)
    return [min(cz, nz - z0) for z0 in range(0, nz, cz)]


SHAPES = {"A": (72, 52, 70), "B": (71, 40, 45), "C": (100, 70)}


def test_shapes_cover_the_tile_geometry():
    src = open(os.path.join(CSRC, "lsm_tiled.cu")).read()
    util = open(os.path.join(CSRC, "lsm_tile_util.cuh")).read()
    defs = {k: int(v) for k, v in re.findall(r"#define (LSM_TX|LSM_TY|LSM_NY) (\d+)", src)}
    assert defs == {"LSM_TX": TX, "LSM_TY": TY, "LSM_NY": NY}, f"tile retuned to {defs}: re-derive SHAPES"
    assert re.search(rf"static constexpr int XL = {XL};", src) and re.search(rf"constexpr int HAL = {HAL};", util), "halo retuned"
    assert "cz = nr >= 128 ? 64 : (nr >= 32 ? 32 : nr);" in src, "z chunking changed: update z_chunk and SHAPES"
    assert "(v.n[0] * sizeof(T)) % 16 == 0 && (long)v.n[0] * v.n[1] * v.n[2] >= 32L * 32 * 32" in src, "TMA rule changed"
    A, B, C = SHAPES["A"], SHAPES["B"], SHAPES["C"]
    assert tile_starts(A[0], TX) == [0, 32, 64] and A[0] - 64 == 8
    assert tile_starts(A[1], TYNY) == [0, 16, 32, 48] and A[1] - 48 == 4
    assert plain_tiles(A) == [(32, 16), (32, 32)]
    assert tma_fill(A, 8) and tma_fill(A, 4)
    assert z_chunks(A[2]) == [32, 32, 6]
    assert not tma_fill(B, 8) and not tma_fill(B, 4)
    assert plain_tiles(B) == [(32, 16)]
    assert z_chunks(B[2]) == [32, 13]
    assert len(tile_starts(C[0], TX)) == 4 and C[0] % TX and len(tile_starts(C[1], TYNY)) == 5 and C[1] % TYNY
    assert len(plain_tiles(C)) == 6


# ---- the matrix ------------------------------------------------------------------------------------------------------
# two BC sets: index maps only (mixed per axis, and per side along y on every third term set), and one in which every term
# set has ExtrapolationBC(1), (2) or (3) on some side, so that it runs the REMAP = false instantiation
BCSETS = {
    "remap": ((("periodic",), ("neumann",), ("symmetry",)), (("symmetry",), ("neumann",))),
    "extrap": ((("extrap", 3), ("neumann",), ("extrap", 1), ("periodic",), ("extrap", 2)), (("extrap", 3), ("symmetry",))),
}
# a Float32 state with Float64 stored coefficients: read from global memory, not staged (coef_f64)
MIXED = ("mixed_weno", "mixed_upwind", "mixed_normal", "mixed_curv")


def _termsets(n):
    lc, hc, phi, u, v, b = H.small_problem(n)
    ts = H.small_termsets(u, v, b, len(n))
    # four terms: 3 + 3 + 1 aux tiles, + phi^n in RK3 stages 2-3 = 8, the most the tiled kernel stages; a stored b makes
    # it 9, so those stages take the strict kernel while stage 1 stays tiled
    four = [dict(kind="advection", field=u), dict(kind="advection", field=u, scheme="upwind"), dict(kind="normal", field=v)]
    ts["aux8"] = four + [dict(kind="curvature", const=-0.02)]
    ts["aux9"] = four + [dict(kind="curvature", field=b)]
    ts["mixed_weno"] = [dict(kind="advection", field=u, field_dtype=np.float64)]
    ts["mixed_upwind"] = [dict(kind="advection", field=u, scheme="upwind", field_dtype=np.float64)]
    ts["mixed_normal"] = [dict(kind="normal", field=v, field_dtype=np.float64)]
    ts["mixed_curv"] = [dict(kind="curvature", field=b, field_dtype=np.float64)]
    return lc, hc, phi, ts


TERMSETS = [t for t in _termsets((8, 8))[3] if t not in MIXED]
ALL_TERMSETS = TERMSETS + list(MIXED)

_CASES = {}


def _case(shape, bcset, termset, dtype):
    n = SHAPES[shape]
    if n not in _CASES:
        _CASES.clear()                       # one shape's arrays at a time
        _CASES[n] = _termsets(n)
    lc, hc, phi, ts = _CASES[n]
    bcs, split = BCSETS[bcset]
    bc = H.small_bc(ALL_TERMSETS.index(termset), len(n), bcs, split)
    return H.Case(termset, lc, hc, n, phi, ts[termset], bc, dtype)


DTYPES = {"f64": np.float64, "f32": np.float32}
MATRIX = [(s, dt, bs, t) for s in SHAPES for dt in DTYPES for bs in BCSETS for t in TERMSETS]
MATRIX += [(s, "f32", bs, t) for s in ("A", "C") for bs in BCSETS for t in MIXED]
INTEGS = ("FE", "RK2", "RK3")


def _integrators(shape, dt, bcset, termset):
    if shape == "A" and dt == "f64":
        return INTEGS
    k = ALL_TERMSETS.index(termset) + list(BCSETS).index(bcset) + list(DTYPES).index(dt) + list(SHAPES).index(shape)
    return (INTEGS[k % 3],)


def _specialised(shape, dt, bcset, termset):
    """Whether the default selection leaves the tiled kernel: for the 3-D x-pair kernels (csrc/lsm_pair3d.cu: index-map BCs,
    rows a multiple of 16 bytes, WENO5 advection by a stored velocity of the state's dtype; in Float64 also the frozen eikonal
    term and normal motion + advection) or the 2-D resident kernel (lsm_api.cu resident_eligible)."""
    n = SHAPES[shape]
    if bcset != "remap":
        return False
    if len(n) == 2:
        return termset == "adv_weno"
    if (n[0] * np.dtype(DTYPES[dt]).itemsize) % 16:
        return False
    return termset == "adv_weno" or (dt == "f64" and termset in ("eik_frozen", "normal_adv"))


# bars, relative to max(1, max|phi|): the strict kernel is the reference's operation order; the tiled kernels restructure
# the arithmetic (FMA contraction, one reciprocal per WENO5 evaluation ...) and are held to the BASELINE bar after 4 steps,
# and to rounding level after one ForwardEuler step, where an error at a tile seam has not spread yet
BAR_STRICT = {"f64": 1e-13, "f32": 2e-6}
BAR_TILED = {"f64": 1e-10, "f32": 1e-4}
BAR_ONE_STEP = {"f64": 1e-12, "f32": 1e-5}


def where(idx, n):
    """Which seams of the tiled kernel the node idx (0-based) lies on."""
    tags = []
    if any(min(i, n[d] - 1 - i) < HAL for d, i in enumerate(idx)):
        tags.append("within 3 nodes of a face")
    if idx[0] % TX < HAL or idx[0] % TX >= TX - HAL:
        tags.append("on an x tile seam")
    if idx[1] % TYNY < HAL or idx[1] % TYNY >= TYNY - HAL:
        tags.append("on a y tile seam")
    if len(n) == 3:
        cz = z_chunk(n[2])
        z0 = idx[2] // cz * cz
        if idx[2] - z0 < HAL or min(z0 + cz, n[2]) - 1 - idx[2] < HAL:
            tags.append("on the first or last planes of a z chunk")
    return f"worst node {tuple(int(i) for i in idx)}: " + (", ".join(tags) or "inside a tile")


def rel_diff(a, b, scale):
    """(max |a - b| / scale, location of the worst node); a NaN counts as the worst."""
    d = np.abs(a.astype(np.float64) - b.astype(np.float64))
    worst = np.unravel_index(np.argmax(np.where(np.isnan(d), np.inf, d)), d.shape)
    return float(np.max(d)) / scale, where(worst, a.shape)


@pytest.fixture(scope="module")
def m():
    import lsm_b200
    return lsm_b200


@pytest.fixture(scope="module")
def fast_oracle(O):
    O.set_threads(O.max_threads())
    return O


def run_kernel(m, case, integ, tf, kernel):
    """Integrate through LSM_OPT_KERNEL = kernel (1 strict, 3 tiled only, 0 default); return (t, steps, state, counters)."""
    ctx = m.default_context()
    ctx.set_option(OPT_KERNEL, kernel)
    try:
        ctx.reset_counters()
        eq = H.run_engine(m, case, integ, tf)
        return eq.t, eq.steps_taken, eq.state.peek().copy(), ctx.counters()
    finally:
        ctx.set_option(OPT_KERNEL, 0)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,dt,bcset,termset", MATRIX, ids=["-".join(c) for c in MATRIX])
def test_multitile_vs_oracle(m, fast_oracle, shape, dt, bcset, termset):
    """Strict (1), tiled-only (3) and default (0) kernels against the oracle: 4 steps of each integrator the case runs, and one
    ForwardEuler step.  Where the default selection keeps the tiled kernel it must equal kernel 3 bit for bit."""
    O = fast_oracle
    case = _case(shape, bcset, termset, DTYPES[dt])
    special = _specialised(shape, dt, bcset, termset)
    name = f"{shape}-{dt}-{bcset}-{termset}"
    lines = []
    for integ, steps in [(i, 4) for i in _integrators(shape, dt, bcset, termset)] + [("FE", 1)]:
        a, t_o, n_o, tf = H.run_oracle(O, case, integ, steps=steps)
        assert n_o == steps or "cos" in termset
        scale = max(1.0, float(np.abs(a).max()))
        outs = {k: run_kernel(m, case, integ, tf, k) for k in (1, 3, 0)}
        bars = {1: BAR_STRICT[dt], 3: BAR_TILED[dt], 0: BAR_TILED[dt]} if steps > 1 else \
               {1: BAR_STRICT[dt], 3: BAR_ONE_STEP[dt], 0: BAR_ONE_STEP[dt]}
        rel = {}
        for k, (t, n, phi, c) in outs.items():
            assert (t, n) == (t_o, n_o), (name, integ, k, t, n, t_o, n_o)
            rel[k], loc = rel_diff(a, phi, scale)
            assert rel[k] <= bars[k], f"{name} {integ} x{steps}, kernel {k}: {rel[k]:.3e} > {bars[k]:.0e} ({loc})"
        c3, c0 = outs[3][3], outs[0][3]
        assert c3["pair_launches"] == 0 and c3["resident_steps"] == 0, ("kernel 3 left the tiled kernel", name, integ)
        if special:
            assert c0["pair_launches"] > 0 or c0["resident_steps"] > 0, ("default selection", name, integ)
        else:
            assert c0["pair_launches"] == 0 and c0["resident_steps"] == 0, ("default selection", name, integ)
            assert np.array_equal(outs[0][2], outs[3][2]), (name, integ, "default kernel differs from kernel 3", rel_diff(outs[0][2], outs[3][2], scale))
        lines.append(f"PARITY multitile {name} {integ} {n_o} step{'s' if n_o > 1 else ''}: strict {rel[1]:.3e} (bar {bars[1]:.0e}) "
                     f"tiled {rel[3]:.3e} default {rel[0]:.3e} (bar {bars[3]:.0e})")
    print("\n".join(lines))


# ---- TMA fill vs cp.async fill ---------------------------------------------------------------------------------------
TMA_CASES = [("f64", "remap", "curv"), ("f64", "extrap", "three"), ("f64", "extrap", "adv_curvf"),
             ("f32", "remap", "three"), ("f32", "extrap", "curv_const")]


def tiled_states(m):
    """RK3, 4 steps of the TMA_CASES on shape A through the tiled kernel alone."""
    out = {}
    for dt, bcset, termset in TMA_CASES:
        case = _case("A", bcset, termset, DTYPES[dt])
        phi = case.engine_field(m)
        tf = 4 * 0.5 * m.compute_cfl(case.engine_terms(m, phi), phi, 0.0) * (1 - 1e-12)
        t, n, state, _ = run_kernel(m, case, "RK3", tf, 3)
        out[f"{dt}-{bcset}-{termset}"] = state
        out[f"{dt}-{bcset}-{termset}-t-steps"] = np.array([t, n])
    return out


def _write_tiled_states(path):
    """Entry point of the child process of test_tma_and_cp_async_fills_agree."""
    import lsm_b200
    np.savez(path, **tiled_states(lsm_b200))


@pytest.mark.gpu
def test_tma_and_cp_async_fills_agree(m, tmp_path):
    """The TMA fill of plain-copy tiles (and of the aux tiles) and the cp.async fill that LSM_B200_NO_TMA=1 selects move the
    same values, so the states must be bit-identical.  The variable is read once per process, hence the child process."""
    here = tiled_states(m)
    out = tmp_path / "no_tma.npz"
    code = (f"import sys; sys.path[:0] = {[REPO, os.path.join(REPO, 'oracle'), TESTS]!r}; "
            f"import test_tiled_multitile as T; T._write_tiled_states(sys.argv[1])")
    flags = [f for f, on in (("-I", sys.flags.isolated), ("-E", sys.flags.ignore_environment), ("-s", sys.flags.no_user_site)) if on]
    r = subprocess.run([sys.executable, *flags, "-c", code, str(out)], cwd=REPO, env=dict(os.environ, LSM_B200_NO_TMA="1"),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    there = np.load(out)
    assert sorted(there.files) == sorted(here)
    for k, v in here.items():
        assert np.array_equal(v, there[k]), (k, float(np.abs(v.astype(np.float64) - there[k].astype(np.float64)).max()))


# ---- extend_along_normals (its stages run the tiled kernel's upwind term with skip_zero_u) ---------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(DTYPES))
def test_extend_along_normals_multitile(m, fast_oracle, dt):
    """test_extend_along_normals on shape A: default band mask and an explicit mask, strict and default kernels, same bars."""
    O, dtype = fast_oracle, DTYPES[dt]
    n = SHAPES["A"]
    lc, hc = (-1.0, -1.0, -1.0), (1.0, 1.1, 1.2)
    X = H.coords(lc, hc, n)
    r = np.sqrt(sum(x * x for x in X))
    phi0 = H.bcast((r - 0.5) * (1 + 0.2 * X[0]), n).astype(dtype)
    F0 = H.bcast(np.sin(3 * X[0]) + X[1] ** 2, n).astype(dtype)
    mask = np.asfortranarray(np.abs(phi0) < 0.08)
    ctx = m.default_context()
    try:
        for frozen in (None, mask):
            for bc in (None, "neumann"):
                fo = O.Field(phi0.copy(order="F"), lc, hc, bc=None if bc is None else O.NEUMANN)
                Fo = O.extend_along_normals(F0.copy(order="F"), fo, nb_iters=12, frozen=frozen)
                for kernel in (1, 0):
                    ctx.set_option(OPT_KERNEL, kernel)
                    g = m.CartesianGrid(lc, hc, n)
                    phi = m.MeshField(phi0.copy(order="F"), g, bc=None if bc is None else m.NeumannBC())
                    F = m.MeshField(F0.copy(order="F"), g)
                    m.extend_along_normals(F, phi, nb_iters=12, frozen=frozen)
                    d = np.abs(F.peek().astype(np.float64) - Fo.astype(np.float64))
                    tol = (1e-13 if kernel == 1 else 1e-11) if dtype == np.float64 else 2e-5
                    worst = np.unravel_index(np.argmax(np.where(np.isnan(d), np.inf, d)), d.shape)
                    assert d.max() <= tol, (frozen is not None, bc, kernel, float(d.max()), where(worst, n))
                    if frozen is not None:
                        assert np.array_equal(F.peek()[mask], F0[mask])
                    print(f"PARITY multitile extend_along_normals A-{dt} mask={frozen is not None} bc={bc} kernel {kernel}: "
                          f"{float(d.max()):.3e} (bar {tol:.0e})")
    finally:
        ctx.set_option(OPT_KERNEL, 0)
