#!/usr/bin/env python
"""tools/extension_bench.py — closest-point extension on the device (extend_closest_point, lsm_extend_closest_point, band 3) against
the PDE extension extend_along_normals(nb_iters=50) on the same Float64 states, with F = g(x) = sin(3 x1) + x2^2 - 0.5 x3:

  sphere  a 512^3 sphere of radius 0.35 on [-0.5, 0.5]^3, generated on the device (lsm_field_fill_shape), NeumannBC;
  c3      bench.py's C3 state (Enright sphere, WENO5 + TVD-RK3, NeumannBC) after --c3-steps RK3 steps.

Time: CUDA events on the library's stream around each call, the median of --reps after --warmup calls, for
extend_closest_point, extend_closest_point(redistance=True), redistance alone and extend_along_normals(nb_iters=50) (each call
works on the output of the previous one).  Accuracy, from one call of each method on copies of F and phi: max and 99th percentile
of |F - g(p)| over the nodes within 3 h of the interface, where p is the exact closest point on the sphere, and on C3 (whose exact
interface is not known) the closest point on the extract_interface mesh over the 8 primitives nearest by centroid.  --profile:
mean CUDA time per kernel of extend_closest_point(redistance=True) under torch.profiler, in a separate run.  The card's name and
power limit are read in the same run.  One JSON line per state.

    python tools/extension_bench.py [--n 512] [--c3-steps 20] [--reps 10] [--warmup 2] [--profile]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

from redistance_bench import timed      # noqa: E402


def g(x0, x1, x2):
    return (np.sin(3.0 * x0) + x1 ** 2) - 0.5 * x2


def axes(mesh):
    return [mesh.lc[d] + np.arange(mesh.n[d], dtype=np.float64) * mesh.meshsize(d + 1) for d in range(3)]


def g_field(m, mesh, ctx):
    x = axes(mesh)
    vals = np.asfortranarray(g(x[0][:, None, None], x[1][None, :, None], x[2][None, None, :]))
    return m.MeshField(vals, mesh, bc=m.NeumannBC(), ctx=ctx)


def node_xyz(mesh, lin):
    i = np.unravel_index(lin, tuple(mesh.n), order="F")
    x = axes(mesh)
    return np.stack([x[d][i[d]] for d in range(3)], axis=-1)


def sphere_targets(mesh, r0):
    """(linear indices of the nodes within 3 h of the sphere, g at their exact closest points)."""
    x = axes(mesh)
    r = np.sqrt((x[0][:, None, None] ** 2 + x[1][None, :, None] ** 2) + x[2][None, None, :] ** 2)
    lin = np.nonzero((np.abs(r - r0) < 3 * mesh.meshsize(1)).ravel(order="F"))[0]
    del r
    X = node_xyz(mesh, lin)
    P = r0 * X / np.linalg.norm(X, axis=1)[:, None]
    return lin, g(P[:, 0], P[:, 1], P[:, 2])


def mesh_targets(m, phi, k=8, chunk=1 << 17):
    """(linear indices of the nodes within 3 h of phi's mesh, g at their closest points on it over the k primitives nearest by
    centroid)."""
    import redistance_ref as R
    from scipy.spatial import cKDTree
    mesh = phi.mesh
    work = phi.copy()
    m.redistance(work)
    lin = np.nonzero((np.abs(np.asarray(work.peek())) < 3 * mesh.meshsize(1)).ravel(order="F"))[0]
    del work
    im = m.extract_interface(phi)
    V = im.vertices[im.faces.astype(np.int64)]
    tree = cKDTree(V.mean(axis=1))
    out = np.empty(len(lin))
    for b in range(0, len(lin), chunk):
        X = node_xyz(mesh, lin[b:b + chunk])
        _, j = tree.query(X, k=k)
        Xk = np.repeat(X[:, None, :], k, axis=1)
        Q = R.closest_point(Xk, V[j])
        best = np.nanargmin(R.dist(Xk, Q), axis=1)
        P = Q[np.arange(len(X)), best]
        out[b:b + chunk] = g(P[:, 0], P[:, 1], P[:, 2])
    return lin, out


def error(F, lin, want):
    e = np.abs(np.asarray(F.peek()).ravel(order="F")[lin] - want)
    return {"max": float(e.max()), "p99": float(np.percentile(e, 99))}


def measure(m, ctx, phi, F, targets, reps, warmup):
    lib = m._lib.lib()
    nb = C.c_int64()
    Fw, pw = F.copy(), phi.copy()
    m._lib.check(lib.lsm_extend_closest_point(ctx.handle, Fw.device(), pw.device(), 3, 0, C.byref(nb)))
    cp_ms, cp_min = timed(ctx, lambda: m.extend_closest_point(Fw, pw), reps, warmup)
    cpr_ms, cpr_min = timed(ctx, lambda: m.extend_closest_point(Fw, pw, redistance=True), reps, warmup)
    pw = phi.copy()
    red_ms, red_min = timed(ctx, lambda: m.redistance(pw), reps, warmup)
    Fw, pw = F.copy(), phi.copy()
    pde_ms, pde_min = timed(ctx, lambda: m.extend_along_normals(Fw, pw, nb_iters=50), reps, warmup)
    del Fw, pw
    lin, want = targets
    Fw = F.copy()
    m.extend_closest_point(Fw, phi.copy())
    cp_err = error(Fw, lin, want)
    Fw = F.copy()
    m.extend_along_normals(Fw, phi.copy(), nb_iters=50)
    pde_err = error(Fw, lin, want)
    del Fw
    return {"nodes": list(phi.mesh.n), "band_nodes": int(nb.value), "nodes_within_3h": int(len(lin)),
            "extend_closest_point_ms": cp_ms, "extend_closest_point_ms_min": cp_min,
            "extend_closest_point_redistance_ms": cpr_ms, "extend_closest_point_redistance_ms_min": cpr_min,
            "redistance_ms": red_ms, "redistance_ms_min": red_min,
            "extend_along_normals50_ms": pde_ms, "extend_along_normals50_ms_min": pde_min,
            "err_extend_closest_point": cp_err, "err_extend_along_normals50": pde_err}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--c3-steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--profile", action="store_true", help="only the sphere, under torch.profiler: mean CUDA time per kernel (a separate run)")
    args = ap.parse_args()
    import lsm_b200 as m
    import bench
    from expr_bench import card

    ctx = m.default_context()
    name, limit = card(ctx.device)
    n = args.n
    grid = m.CartesianGrid((-0.5,) * 3, (0.5,) * 3, (n, n, n))
    phi = m.MeshField.from_shape(grid, "sphere", (0.0, 0.0, 0.0, 0.35), bc=m.NeumannBC(), ctx=ctx)
    F = g_field(m, phi.mesh, ctx)
    if args.profile:
        import torch
        from torch.profiler import ProfilerActivity, profile
        m.extend_closest_point(F, phi, redistance=True)
        ctx.sync()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.reps):
                m.extend_closest_point(F, phi, redistance=True)
            ctx.sync()
        torch.cuda.synchronize()
        kern = {e.key[:60]: {"calls": e.count, "mean_us": e.device_time} for e in prof.key_averages() if "redist" in e.key}
        print(json.dumps({"state": f"sphere r=0.35, {n}^3, Float64 (profiled)", "card": name, "power_limit": limit, "kernels": kern}), flush=True)
        return
    res = measure(m, ctx, phi, F, sphere_targets(phi.mesh, 0.35), args.reps, args.warmup)
    print(json.dumps({"state": f"sphere r=0.35, {n}^3, Float64", "card": name, "power_limit": limit, **res}), flush=True)
    del phi, F

    _, phi, vel, terms = bench.build_c3(m, ctx, n, 1)
    low = m.api._Lowered(terms, phi, 0.0)
    t_out, st = C.c_double(), C.c_int64()
    m._lib.check(m._lib.lib().lsm_integrate(ctx.handle, m._lib.RK3, 0.5, phi.device(), low.arr, len(terms), 0.0, 1e9, float("inf"),
                                            args.c3_steps, C.byref(t_out), C.byref(st)))
    phi._mark_device_advanced()
    F = g_field(m, phi.mesh, ctx)
    res = measure(m, ctx, phi, F, mesh_targets(m, phi), args.reps, args.warmup)
    print(json.dumps({"state": f"C3 after {st.value} RK3 steps, {n}^3, Float64", "card": name, "power_limit": limit, **res}), flush=True)


if __name__ == "__main__":
    main()
