#!/usr/bin/env python
"""tools/expr_bench.py — one time-dependent velocity given three ways, on C3 (Enright sphere, Float64, WENO5 + TVD-RK3, NeumannBC):

  stored  the stored Float64 velocity x cos(pi t / 3) (TimeScaled; bench.py's headline path, CFL from the candidate nodes);
  expr    the same velocity as a time-dependent DeviceExpr, materialised on the device at the CFL and stage times by the generated
          kernel, which also reduces the CFL maximum;
  host    the same velocity as a Python callable f(x, t), evaluated with NumPy and uploaded at every CFL and stage time (the
          path every f(x, t) coefficient took before DeviceExpr), on a smaller grid it can finish.

stored and expr: CUDA events on the library's stream around one lsm_integrate call of --steps RK3 steps (the call ends in a stream
sync), after --warmup steps.  host: a host clock around integrate() (blocking).  Prints one JSON line: ms per RK3 step of each
path, the NVRTC compile time of the three expressions, launch counters of the expr run, and the card's name and power limit read
in the same run.

    python tools/expr_bench.py [--n 512] [--steps 20] [--warmup 3] [--host-n 128] [--host-steps 3]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

ENRIGHT = ("2.0*sin(pi*x1)*sin(pi*x1)*sin(2.0*pi*x2)*sin(2.0*pi*x3)*cos(pi*t/3.0)",
           "-sin(2.0*pi*x1)*sin(pi*x2)*sin(pi*x2)*sin(2.0*pi*x3)*cos(pi*t/3.0)",
           "-sin(2.0*pi*x1)*sin(2.0*pi*x2)*sin(pi*x3)*sin(pi*x3)*cos(pi*t/3.0)")


def enright_callable(x, t):
    s, c = np.sin, np.cos(np.pi * t / 3.0)
    return (2.0 * s(np.pi * x[0]) * s(np.pi * x[0]) * s(2.0 * np.pi * x[1]) * s(2.0 * np.pi * x[2]) * c,
            -s(2.0 * np.pi * x[0]) * s(np.pi * x[1]) * s(np.pi * x[1]) * s(2.0 * np.pi * x[2]) * c,
            -s(2.0 * np.pi * x[0]) * s(2.0 * np.pi * x[1]) * s(np.pi * x[2]) * s(np.pi * x[2]) * c)


def card(device):
    """Name and power limit of the card, read with a query (no setting is changed)."""
    try:
        out = subprocess.run(["nvidia-smi", f"--id={device}", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, limit = [s.strip() for s in out.split(",")[:2]]
        return name, limit
    except (OSError, IndexError, ValueError, subprocess.TimeoutExpired):
        return None, None


def device_ms(m, ctx, phi, terms, steps, warmup):
    """ms per RK3 step of `steps` steps in one lsm_integrate call (CUDA events), after `warmup` steps; plus the counters."""
    lib, L = m._lib.lib(), m._lib
    low = m.api._Lowered(terms, phi, 0.0)
    dev = phi.device()

    def go(k, t0):
        t_out, st = C.c_double(), C.c_int64()
        L.check(lib.lsm_integrate(ctx.handle, L.RK3, 0.5, dev, low.arr, len(terms), t0, 1e9, float("inf"), k, C.byref(t_out), C.byref(st)))
        assert st.value == k
        return t_out.value

    t = go(warmup, 0.0)
    ctx.reset_counters()
    ctx.event_record(0)
    go(steps, t)
    ctx.event_record(1)
    ms = ctx.event_elapsed_ms(0, 1)
    phi._mark_device_advanced()
    return ms / steps, ctx.counters()


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--host-n", type=int, default=128)
    ap.add_argument("--host-steps", type=int, default=3)
    args = ap.parse_args()
    import lsm_b200 as m
    import bench

    ctx = m.default_context()
    name, limit = card(ctx.device)
    out = {"workload": f"C3 Enright sphere, {args.n}^3, Float64, WENO5 + TVD-RK3, NeumannBC, velocity x cos(pi t/3)",
           "card": name, "power_limit": limit, "n": args.n, "steps": args.steps, "warmup": args.warmup}

    # stored: bench.py's configuration
    grid, phi, vel, terms = bench.build_c3(m, ctx, args.n, 1)
    out["stored_ms_per_step"], _ = device_ms(m, ctx, phi, terms, args.steps, args.warmup)
    del vel, terms

    # expr: the same velocity written as expressions; the first DeviceExpr of the process compiles them
    t0 = time.perf_counter()
    expr = m.DeviceExpr(ENRIGHT)
    out["nvrtc_compile_s"] = time.perf_counter() - t0
    phi2 = m.MeshField.from_shape(grid, "sphere", (0.35, 0.35, 0.35, 0.15), bc=m.NeumannBC(), ctx=ctx)
    ms, c = device_ms(m, ctx, phi2, (m.AdvectionTerm(expr, m.WENO5()),), args.steps, args.warmup)
    out["expr_ms_per_step"] = ms
    out["expr_counters"] = {k: c[k] for k in ("kernel_launches", "stage_launches", "cfl_passes", "d2h_bytes", "h2d_bytes")}
    d = C.c_double()
    m._lib.check(m._lib.lib().lsm_max_abs_diff(ctx.handle, phi.device(), phi2.device(), C.byref(d)))
    out["max_abs_diff_stored_vs_expr"] = d.value
    del phi, phi2

    # host callable on a grid it can finish, and the expr path on the same grid for comparison
    hn = args.host_n
    hgrid = m.CartesianGrid((0, 0, 0), (1, 1, 1), (hn, hn, hn))
    hres = {"n": hn, "steps": args.host_steps}
    for label, coef in (("host", enright_callable), ("expr", expr)):
        phi = m.MeshField.from_shape(hgrid, "sphere", (0.35, 0.35, 0.35, 0.15), bc=m.NeumannBC(), ctx=ctx)
        eq = m.LevelSetEquation(terms=(m.AdvectionTerm(coef, m.WENO5()),), ic=phi, integrator=m.RK3())
        dt0 = 0.5 * m.compute_cfl(eq.terms, eq.state, 0.0)
        m.integrate(eq, dt0 * (1 - 1e-12), dt0)                      # one warm-up step
        # dt_max = dt0: |cos(pi t / 3)| only shrinks on [0, 3/2], so every step is exactly dt0
        t0 = time.perf_counter()
        m.integrate(eq, dt0 * (1 + args.host_steps) * (1 - 1e-12), dt0)
        ctx.sync()
        sec = time.perf_counter() - t0
        assert eq.steps_taken == args.host_steps, eq.steps_taken
        hres[f"{label}_ms_per_step"] = sec * 1e3 / args.host_steps
    out["host_grid"] = hres
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
