#!/usr/bin/env python
"""tools/interface_bench.py — zero-level-set extraction on the device (lsm_interface_extract + lsm_interface_fetch) against
downloading the field (lsm_field_download, values(phi)) and extracting on the host with the NumPy restatement
(tests/interface_ref.py), on two Float64 states:

  sphere  a 512^3 sphere of radius 0.35 on [-0.5, 0.5]^3, generated on the device (lsm_field_fill_shape);
  c3      bench.py's C3 state (Enright sphere, WENO5 + TVD-RK3, NeumannBC) after --c3-steps RK3 steps.

extract: CUDA events on the library's stream around lsm_interface_extract (it ends with the emit kernels enqueued; the stop event
follows them).  fetch: a host clock around lsm_interface_fetch (blocking, pageable host arrays).  Both after --warmup calls; the
median of --reps.  download and the host restatement: a host clock, once (with --ref).  The device mesh is compared with the host
one bit for bit.  Also printed: the shape-only estimates (mesh bytes, the compulsory read of phi at 6450 GB/s, DESIGN.md §6) and
the card's name and power limit, read in the same run.  One JSON line per state.

    python tools/interface_bench.py [--n 512] [--c3-steps 20] [--reps 20] [--warmup 3] [--ref] [--profile]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

HBM_GBPS = 6450.0      # streaming read rate measured in DESIGN.md §6


def measure(m, ctx, phi, reps, warmup, ref):
    lib, L = m._lib.lib(), m._lib
    dev = phi.device()
    nv, nf = C.c_int64(), C.c_int64()
    for _ in range(warmup):
        mesh = m.extract_interface(phi)
    ext, fet = [], []
    for _ in range(reps):
        ctx.event_record(0)
        L.check(lib.lsm_interface_extract(ctx.handle, dev, 0.0, C.byref(nv), C.byref(nf)))
        ctx.event_record(1)
        ext.append(ctx.event_elapsed_ms(0, 1))
        t0 = time.perf_counter()
        mesh = m.api._fetch_interface(ctx, phi.ndim, nv.value, nf.value)
        fet.append((time.perf_counter() - t0) * 1e3)
    ctx.reset_counters()
    mesh = m.extract_interface(phi)
    c = ctx.counters()
    n = phi.mesh.n
    field_bytes = int(np.prod(n)) * phi.valtype.itemsize
    mesh_bytes = mesh.vertices.nbytes + mesh.keys.nbytes + mesh.faces.nbytes
    out = {"nodes": list(n), "nverts": int(nv.value), "nprims": int(nf.value), "mesh_MB": mesh_bytes / 1e6, "field_MB": field_bytes / 1e6,
           "extract_ms": statistics.median(ext), "extract_ms_min": min(ext), "fetch_ms": statistics.median(fet),
           "kernel_launches": c["kernel_launches"], "d2h_bytes_extract_fetch": c["d2h_bytes"],
           "compulsory_read_ms": field_bytes / (HBM_GBPS * 1e9) * 1e3}
    if ref:
        import interface_ref as R
        t0 = time.perf_counter()
        host = np.empty(phi._shape, dtype=phi.valtype, order="F")
        L.check(lib.lsm_field_download(dev, host.ctypes.data))
        out["download_ms"] = (time.perf_counter() - t0) * 1e3
        t0 = time.perf_counter()
        g = phi.mesh
        X, F, K = R.extract(host, g.lc, g.meshsize())
        out["host_restatement_s"] = time.perf_counter() - t0
        out["bitwise_equal_to_host"] = bool(np.array_equal(mesh.keys, K) and np.array_equal(mesh.faces, F)
                                            and np.array_equal(mesh.vertices.view(np.int64), X.view(np.int64)))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--c3-steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--ref", action="store_true", help="also time the download + host restatement and compare the meshes")
    ap.add_argument("--profile", action="store_true", help="only the sphere, under torch.profiler: mean CUDA time per kernel (a separate run)")
    args = ap.parse_args()
    import lsm_b200 as m
    import bench
    from expr_bench import card

    ctx = m.default_context()
    name, limit = card(ctx.device)
    n = args.n
    g = m.CartesianGrid((-0.5,) * 3, (0.5,) * 3, (n, n, n))
    phi = m.MeshField.from_shape(g, "sphere", (0.0, 0.0, 0.0, 0.35), ctx=ctx)
    if args.profile:
        import torch
        from torch.profiler import ProfilerActivity, profile
        measure(m, ctx, phi, 1, args.warmup, False)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            measure(m, ctx, phi, args.reps, 0, False)
        torch.cuda.synchronize()
        kern = {e.key: {"calls": e.count, "mean_us": e.device_time}
                for e in prof.key_averages() if "iface" in e.key}
        print(json.dumps({"state": f"sphere r=0.35, {n}^3, Float64 (profiled)", "card": name, "power_limit": limit, "kernels": kern}), flush=True)
        return
    res = measure(m, ctx, phi, args.reps, args.warmup, args.ref)
    print(json.dumps({"state": f"sphere r=0.35, {n}^3, Float64", "card": name, "power_limit": limit, **res}), flush=True)
    del phi

    grid, phi, vel, terms = bench.build_c3(m, ctx, n, 1)
    eq = m.LevelSetEquation(terms=terms, ic=phi, integrator=m.RK3())
    low = m.api._Lowered(terms, phi, 0.0)
    t_out, st = C.c_double(), C.c_int64()
    m._lib.check(m._lib.lib().lsm_integrate(ctx.handle, m._lib.RK3, 0.5, phi.device(), low.arr, len(terms), 0.0, 1e9, float("inf"),
                                            args.c3_steps, C.byref(t_out), C.byref(st)))
    phi._mark_device_advanced()
    res = measure(m, ctx, phi, args.reps, args.warmup, args.ref)
    print(json.dumps({"state": f"C3 after {st.value} RK3 steps, {n}^3, Float64", "card": name, "power_limit": limit, **res}), flush=True)
    del eq


if __name__ == "__main__":
    main()
