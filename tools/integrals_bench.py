#!/usr/bin/env python
"""tools/integrals_bench.py — level-set integrals on the device (level_set_integrals, lsm_level_set_integrals) next to the smoothed
volume and perimeter sums (lsm_volume, lsm_perimeter) on the same Float64 states:

  sphere  a 512^3 sphere of radius 0.35 on [-0.5, 0.5]^3, generated on the device (lsm_field_fill_shape), NeumannBC;
  c3      bench.py's C3 state (Enright sphere, WENO5 + TVD-RK3, NeumannBC) after --c3-steps RK3 steps.

Time: CUDA events on the library's stream around each call (each call ends in its own synchronisation and D2H copy), the median of
--reps after --warmup calls, for level_set_integrals without F and with F = x1 (generated on the device), volume and perimeter, in
the same run.  Bandwidth: the compulsory bytes (8 per node for phi, 8 more for F) over the median time, also as a fraction of the
7.7 TB/s of the HGX B200 data sheet.  Accuracy (sphere only): the errors of the volume and area against 4/3 pi r^3 and 4 pi r^2 for
n = 64 .. --n, from level_set_integrals and from volume / perimeter.  The card's name and power limit are read in the same run.  One
JSON line per state, then one for the accuracy table.

    python tools/integrals_bench.py [--n 512] [--c3-steps 20] [--reps 10] [--warmup 2]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

from redistance_bench import timed      # noqa: E402

HBM_TBS = 7.7


def measure(m, ctx, phi, reps, warmup):
    F = m.MeshField.from_shape(phi.mesh, "plane", (1.0, 0.0, 0.0, 0.0), bc=m.NeumannBC(), ctx=ctx)     # F = x1
    F.device()
    nodes = math.prod(phi.mesh.n)
    res = {"nodes": list(phi.mesh.n)}
    for key, fn, nbytes in (("integrals", lambda: m.level_set_integrals(phi), 8 * nodes),
                            ("integrals_F", lambda: m.level_set_integrals(phi, F), 16 * nodes),
                            ("volume", lambda: m.volume(phi), 8 * nodes),
                            ("perimeter", lambda: m.perimeter(phi), 8 * nodes)):
        med, lo = timed(ctx, fn, reps, warmup)
        res[f"{key}_ms"], res[f"{key}_ms_min"] = med, lo
        res[f"{key}_GBps"] = nbytes / (med * 1e-3) / 1e9
        res[f"{key}_frac_hbm"] = nbytes / (med * 1e-3) / (HBM_TBS * 1e12)
    r = m.level_set_integrals(phi, F)
    res.update(inside=r.inside, interface=r.interface, x1_inside=r.F_inside, x1_interface=r.F_interface,
               volume=m.volume(phi), perimeter=m.perimeter(phi))
    ctx.reset_counters()
    m.level_set_integrals(phi, F)
    c = ctx.counters()
    res.update(launches=c["kernel_launches"], d2h_bytes=c["d2h_bytes"])
    del F
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--c3-steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    import lsm_b200 as m
    import bench
    from expr_bench import card

    ctx = m.default_context()
    name, limit = card(ctx.device)
    n, r0 = args.n, 0.35
    grid = m.CartesianGrid((-0.5,) * 3, (0.5,) * 3, (n, n, n))
    phi = m.MeshField.from_shape(grid, "sphere", (0.0, 0.0, 0.0, r0), bc=m.NeumannBC(), ctx=ctx)
    res = measure(m, ctx, phi, args.reps, args.warmup)
    print(json.dumps({"state": f"sphere r={r0}, {n}^3, Float64", "card": name, "power_limit": limit, **res}), flush=True)
    del phi

    _, phi, vel, terms = bench.build_c3(m, ctx, n, 1)
    low = m.api._Lowered(terms, phi, 0.0)
    t_out, st = C.c_double(), C.c_int64()
    m._lib.check(m._lib.lib().lsm_integrate(ctx.handle, m._lib.RK3, 0.5, phi.device(), low.arr, len(terms), 0.0, 1e9, float("inf"),
                                            args.c3_steps, C.byref(t_out), C.byref(st)))
    phi._mark_device_advanced()
    del vel, terms, low
    res = measure(m, ctx, phi, args.reps, args.warmup)
    print(json.dumps({"state": f"C3 after {st.value} RK3 steps, {n}^3, Float64", "card": name, "power_limit": limit, **res}), flush=True)
    del phi

    V0, A0 = 4.0 / 3.0 * math.pi * r0 ** 3, 4.0 * math.pi * r0 ** 2
    rows = []
    k = 64
    while k <= n:
        g = m.CartesianGrid((-0.5,) * 3, (0.5,) * 3, (k, k, k))
        phi = m.MeshField.from_shape(g, "sphere", (0.0, 0.0, 0.0, r0), bc=m.NeumannBC(), ctx=ctx)
        r = m.level_set_integrals(phi)
        rows.append({"n": k, "integrals_volume_err": r.inside / V0 - 1, "integrals_area_err": r.interface / A0 - 1,
                     "volume_err": m.volume(phi) / V0 - 1, "perimeter_err": m.perimeter(phi) / A0 - 1})
        del phi
        k *= 2
    print(json.dumps({"state": f"sphere r={r0} accuracy, Float64", "card": name, "power_limit": limit, "rows": rows}), flush=True)


if __name__ == "__main__":
    main()
