#!/usr/bin/env python
"""tools/redistance_bench.py — closest-point redistancing on the device (redistance, lsm_redistance, band 3; and order=3,
lsm_redistance_cubic, with its fallback count) against the PDE reinitialisation eikonal_reinitialize(iterations=20) on the same
Float64 states:

  sphere  a 512^3 sphere of radius 0.35 on [-0.5, 0.5]^3, generated on the device (lsm_field_fill_shape), NeumannBC;
  c3      bench.py's C3 state (Enright sphere, WENO5 + TVD-RK3, NeumannBC) after --c3-steps RK3 steps.

Time: CUDA events on the library's stream around each call, the median of --reps after --warmup calls (each call works on the
output of the previous one; the working set, 8.6 GB of scratch at 512^3, is far larger than the L2).  Quality, from one call
on a copy of the state: the mean Newton iterations of order 3 within 3h (newton_iterations: the NumPy restatement of the device's
arithmetic on a sample of the state's nodes), the interface shift (the largest distance from a vertex of extract_interface after the call to the mesh
before, over the 8 primitives nearest by centroid: an upper bound) and max | |grad phi| - 1 | over the nodes with |phi| < 3 h whose
second differences are below 0.5 / h on every axis (centred differences; away from kinks).  --profile: mean CUDA time per kernel of
redistance and of redistance(order=3) under torch.profiler, in a separate run.  The card's name and power limit are read in the same run.  One JSON line per
state.

    python tools/redistance_bench.py [--n 512] [--c3-steps 20] [--reps 10] [--warmup 2] [--profile]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)


def timed(ctx, fn, reps, warmup):
    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(reps):
        ctx.event_record(0)
        fn()
        ctx.event_record(1)
        ms.append(ctx.event_elapsed_ms(0, 1))
    return statistics.median(ms), min(ms)


def mesh_shift(before, after, k=8, chunk=1 << 17):
    import redistance_ref as R
    from scipy.spatial import cKDTree
    V = before.vertices[before.faces.astype(np.int64)]
    tree = cKDTree(V.mean(axis=1))
    worst = 0.0
    for b in range(0, len(after.vertices), chunk):
        X = after.vertices[b:b + chunk]
        _, j = tree.query(X, k=k)
        Xk = np.repeat(X[:, None, :], k, axis=1)
        d = np.nanmin(R.dist(Xk, R.closest_point(Xk, V[j])), axis=1)
        worst = max(worst, float(d.max()))
    return worst


def gradient_error(phi_vals, h):
    """max | |grad phi| - 1 | over smooth nodes with |phi| < 3 h (interior nodes, centred differences)."""
    f = np.asarray(phi_vals, dtype=np.float64)
    n = f.shape
    flat = f.ravel(order="F")
    inner = np.zeros(n, bool)
    inner[1:-1, 1:-1, 1:-1] = True
    lin = np.nonzero((inner & (np.abs(f) < 3 * h)).ravel(order="F"))[0]
    strides = (1, n[0], n[0] * n[1])
    g2 = np.zeros(len(lin))
    smooth = np.ones(len(lin), bool)
    for s in strides:
        fp, fm, f0 = flat[lin + s], flat[lin - s], flat[lin]
        g2 += ((fp - fm) / (2 * h)) ** 2
        smooth &= np.abs(fp - 2 * f0 + fm) / h < 0.5
    err = np.abs(np.sqrt(g2[smooth]) - 1.0)
    return float(err.max()), float(np.percentile(err, 99)), int(smooth.sum())


def quality(m, phi, fn):
    work = phi.copy()
    before = m.extract_interface(work)
    fn(work)
    after = m.extract_interface(work)
    h = work.mesh.meshsize(1)
    gmax, g99, nodes = gradient_error(work.peek(), h)
    out = {"shift_over_h": mesh_shift(before, after) / h, "grad_err_max": gmax, "grad_err_p99": g99, "grad_nodes": nodes}
    del work
    return out


def newton_iterations(phi, mesh, sample=20000, k=16, seed=0):
    """Newton iterations of redistance(order=3) within 3h, from tests/cubic_ref.py (the device's arithmetic) on the same state: up
    to `sample` random nodes whose distance to the extracted mesh is below 3h, seeded with their closest point on that mesh (the
    band scan's point; the first primitive in mesh order among equally close ones, over the k nearest by centroid).  Returns
    (mean iterations of the converged nodes, nodes that fell back, nodes sampled)."""
    import cubic_ref as CR
    import redistance_ref as R
    from scipy.spatial import cKDTree
    vals = np.asarray(phi.peek())
    g = phi.mesh
    h, lc = g.meshsize(), g.lc
    h3 = 3 * min(abs(v) for v in h)
    cand = np.flatnonzero(np.abs(vals) < 2 * h3)
    cand = np.random.default_rng(seed).permutation(cand)[:4 * sample]
    idx = np.stack(np.unravel_index(cand, vals.shape), axis=-1)
    x = np.stack([float(lc[d]) + idx[:, d].astype(np.float64) * float(h[d]) for d in range(vals.ndim)], axis=-1)
    V = mesh.vertices[mesh.faces.astype(np.int64)]
    _, j = cKDTree(V.mean(axis=1)).query(x, k=k)
    j = np.sort(j.reshape(len(x), k), axis=1)
    X = np.repeat(x[:, None, :], k, axis=1)
    q = R.closest_point(X, V[j])
    d = R.dist(X, q)
    best = np.argmin(d, axis=1)
    dmin = d[np.arange(len(x)), best]
    keep = np.flatnonzero(dmin < h3)[:sample]
    y, fell, iters = CR.refine(vals, lc, h, x[keep], q[keep, best[keep]])
    return float(iters[~fell].mean()), int(fell.sum()), int(len(keep))


def measure(m, ctx, phi, reps, warmup):
    lib = m._lib.lib()
    nb = C.c_int64()
    work = phi.copy()
    m._lib.check(lib.lsm_redistance(ctx.handle, work.device(), 3, C.byref(nb)))
    work = phi.copy()
    red_ms, red_min = timed(ctx, lambda: m.redistance(work, band=3), reps, warmup)
    work = phi.copy()
    nf = C.c_int64()
    m._lib.check(lib.lsm_redistance_cubic(ctx.handle, work.device(), 3, None, C.byref(nf)))     # fallbacks on the state itself
    work = phi.copy()
    cub_ms, cub_min = timed(ctx, lambda: m.redistance(work, band=3, order=3), reps, warmup)
    work = phi.copy()
    eik_ms, eik_min = timed(ctx, lambda: m.eikonal_reinitialize(work, iterations=20), reps, warmup)
    del work
    it, it_fell, it_nodes = newton_iterations(phi, m.extract_interface(phi))
    return {"nodes": list(phi.mesh.n), "band_nodes": int(nb.value), "newton_iters_3h": it, "newton_fallbacks_3h": it_fell,
            "newton_sampled_3h": it_nodes,
            "redistance_ms": red_ms, "redistance_ms_min": red_min, "cubic_ms": cub_ms, "cubic_ms_min": cub_min,
            "cubic_fallbacks": int(nf.value), "eikonal20_ms": eik_ms, "eikonal20_ms_min": eik_min,
            "redistance": quality(m, phi, lambda f: m.redistance(f, band=3)),
            "cubic": quality(m, phi, lambda f: m.redistance(f, band=3, order=3)),
            "eikonal20": quality(m, phi, lambda f: m.eikonal_reinitialize(f, iterations=20))}


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
    g = m.CartesianGrid((-0.5,) * 3, (0.5,) * 3, (n, n, n))
    phi = m.MeshField.from_shape(g, "sphere", (0.0, 0.0, 0.0, 0.35), bc=m.NeumannBC(), ctx=ctx)
    if args.profile:
        import torch
        from torch.profiler import ProfilerActivity, profile
        cub = phi.copy()                       # each order works on its own output, as in the timed runs
        m.redistance(phi)
        m.redistance(cub, order=3)
        ctx.sync()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.reps):
                m.redistance(phi)
                m.redistance(cub, order=3)
            ctx.sync()
        torch.cuda.synchronize()
        kern = {e.key[:70]: {"calls": e.count, "mean_us": e.device_time} for e in prof.key_averages() if "redist" in e.key or "refine" in e.key}
        print(json.dumps({"state": f"sphere r=0.35, {n}^3, Float64 (profiled)", "card": name, "power_limit": limit, "kernels": kern}), flush=True)
        return
    res = measure(m, ctx, phi, args.reps, args.warmup)
    print(json.dumps({"state": f"sphere r=0.35, {n}^3, Float64", "card": name, "power_limit": limit, **res}), flush=True)
    del phi

    grid, phi, vel, terms = bench.build_c3(m, ctx, n, 1)
    low = m.api._Lowered(terms, phi, 0.0)
    t_out, st = C.c_double(), C.c_int64()
    m._lib.check(m._lib.lib().lsm_integrate(ctx.handle, m._lib.RK3, 0.5, phi.device(), low.arr, len(terms), 0.0, 1e9, float("inf"),
                                            args.c3_steps, C.byref(t_out), C.byref(st)))
    phi._mark_device_advanced()
    res = measure(m, ctx, phi, args.reps, args.warmup)
    print(json.dumps({"state": f"C3 after {st.value} RK3 steps, {n}^3, Float64", "card": name, "power_limit": limit, **res}), flush=True)


if __name__ == "__main__":
    main()
