#!/usr/bin/env python
"""tools/semi_implicit_bench.py — the semi-implicit advection integrator (SemiImplicit, LSM_SEMI_IMPLICIT, cfl 2, one Jacobi sweep per
launch) against TVD-RK3 (cfl 0.5) with WENO5 and with Upwind, Float64, on:

  rot2048  a circle in the rigid rotation (-2 pi y, 2 pi x) on [-1, 1]^2, 2048^2 nodes, NeumannBC, stored velocity;
  c3_256, c3_512  bench.py's C3 (Enright sphere, stored velocity x cos(pi t / 3), NeumannBC) at 256^3 and 512^3.

For each case and integrator the same simulated time S = --steps semi-implicit steps (S = steps x 2 x dt_cfl at t = 0) is run with
integrate() after one warm-up step, timed with CUDA events on the library's stream: time per step and per unit of simulated time.
Bytes per step are the compulsory HBM traffic computed from shapes (8 bytes per node and value): RK3 3 stages x (phi, N velocity
components, one more read for stages 2-3, one write); semi-implicit: the right-hand side (phi, N components, one write) and every
sweep launch (r, x, N components, one write), times the number of sweeps k.  The card's name and power limit
are read in the same run.  One JSON line per case.

    python tools/semi_implicit_bench.py [--steps 8] [--cases rot2048,c3_256,c3_512]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
        return [s.strip() for s in out.split(",")]
    except Exception as e:       # the measurement itself needs the GPU; the card query is informational
        return [f"unknown ({e})"]


def make_case(m, name):
    if name == "rot2048":
        n = 2048
        grid = m.CartesianGrid((-1.0, -1.0), (1.0, 1.0), (n, n))
        X = grid.coords()
        phi0 = np.broadcast_to(np.sqrt((X[0] - 0.4) ** 2 + X[1] ** 2) - 0.3, grid.n).astype(np.float64)
        u = np.stack([np.broadcast_to(-2 * np.pi * X[1], grid.n), np.broadcast_to(2 * np.pi * X[0], grid.n)]).astype(np.float64)
        vel = m.MeshField(u, grid)

        def build(scheme):
            phi = m.MeshField(phi0.copy(), grid, bc=m.NeumannBC())
            return phi, (m.AdvectionTerm(vel, scheme),)
        return build, grid.n
    import helpers as H
    case = H.c3_enright(int(name.split("_")[1]))
    u = case.terms[0]["field"]
    grid = m.CartesianGrid(case.lc, case.hc, case.n)
    vel = m.TimeScaled(m.MeshField(u, grid), ("cos", case.terms[0]["cos_period"]))

    def build(scheme):
        phi = m.MeshField(np.asarray(case.phi0, dtype=np.float64).copy(), grid, bc=m.NeumannBC())
        return phi, (m.AdvectionTerm(vel, scheme),)
    return build, case.n


def run(m, ctx, build, integ, scheme, S):
    phi, terms = build(scheme)
    eq = m.LevelSetEquation(terms=terms, ic=phi, integrator=integ)
    dt_cfl = m.compute_cfl(terms, eq.state, 0.0)
    m.integrate(eq, integ.cfl * dt_cfl)                  # warm-up: one step
    t0 = eq.t
    ctx.reset_counters()
    L = m._lib
    L.check(L.lib().lsm_event_record(ctx.handle, 0))
    m.integrate(eq, t0 + S)
    L.check(L.lib().lsm_event_record(ctx.handle, 1))
    ms = C.c_double()
    L.check(L.lib().lsm_event_elapsed_ms(ctx.handle, 0, 1, C.byref(ms)))
    c = ctx.counters()
    return ms.value, eq.steps_taken, c


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--cases", default="rot2048,c3_256,c3_512")
    a = ap.parse_args()
    import lsm_b200 as m
    ctx = m.default_context()
    info = card()
    for name in a.cases.split(","):
        build, n = make_case(m, name)
        N, nodes = len(n), math.prod(n)
        phi, terms = build(m.WENO5())
        S = a.steps * 2.0 * m.compute_cfl(terms, phi, 0.0)
        res = {"case": name, "n": list(n), "card": info, "sim_time": S}
        for label, integ, scheme in (("semi_implicit", m.SemiImplicit(2.0), m.Upwind()),
                                     ("rk3_weno5", m.RK3(0.5), m.WENO5()), ("rk3_upwind", m.RK3(0.5), m.Upwind())):
            ms, steps, c = run(m, ctx, build, integ, scheme, S)
            if label == "semi_implicit":
                k = c["jacobi_sweeps"] / max(steps, 1)
                launches = math.ceil(k)
                bytes_step = 8 * nodes * ((N + 2) + launches * (N + 3))
                extra = {"sweeps_per_step": k, "sweep_launches_per_step": launches}
            else:
                bytes_step = 8 * nodes * 3 * (N + 3)
                extra = {}
            res[label] = {"steps": steps, "ms_total": ms, "ms_per_step": ms / steps, "ms_per_unit_time": ms / S,
                          "bytes_per_step": bytes_step, "GBps": bytes_step * steps / (ms * 1e-3) / 1e9, **extra}
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
