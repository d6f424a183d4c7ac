#!/usr/bin/env python
"""tools/narrow_band_bench.py — RK3 steps of a narrow-band field (NarrowBandMeshField, lsm_field_set_band) against the dense field.

Workload: bench.py's C3 (Enright sphere r = 0.15, stored Float64 velocity x cos(pi t / 3), WENO5, NeumannBC, every field generated
on the device) at --n nodes per axis (512 and 1024 by default), halfwidth --halfwidth.  For each size:

  * dense (LSM_OPT_KERNEL = 0: the x-pair kernel) and band: ms per RK3 step over --steps steps at t = 0, and again after both have
    advanced --advance more steps (the interface stretches);
  * the active and shell brick fractions at both points;
  * the band's rebuild and shell copy per step: the band step minus its stage kernels (LSM_OPT_TIME_STAGES) in a separate window;
  * the exit-at-once blocks: ms per step of a band with no core brick (phi = 1 everywhere), where every list kernel and every stage
    launch runs only blocks that exit at once.

Steps are timed with CUDA events on the library's stream around lsm_integrate(max_steps = K) after a warm-up window.  The card's
name and power limit are read in the same run.  One JSON line per size.

    python tools/narrow_band_bench.py [--n 512,1024] [--steps 20] [--advance 1000] [--halfwidth 3]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    return [s.strip() for s in out.split(",")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", default="512,1024")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--advance", type=int, default=1000)
    ap.add_argument("--halfwidth", type=float, default=3.0)
    args = ap.parse_args()

    import bench
    import lsm_b200 as m
    import lsm_b200.api as A
    L, lib = m._lib, m._lib.lib()
    ctx = m.Context(0)
    m.set_default_context(ctx)
    name, plimit, maxclk = card()

    def steps(phi, terms, t, k):
        """k RK3 steps from t through lsm_integrate; returns (ms per step, time reached)."""
        low = A._Lowered(terms, phi, t)
        t_out, n = C.c_double(), C.c_int64()
        ctx.event_record(0)
        L.check(lib.lsm_integrate(ctx.handle, L.RK3, 0.5, phi.device(), low.arr, len(terms), float(t), 1e9, float("inf"), k,
                                  C.byref(t_out), C.byref(n)))
        ctx.event_record(1)
        assert n.value == k
        phi._mark_device_advanced()
        return ctx.event_elapsed_ms(0, 1) / k, t_out.value

    def fractions(phi):
        i = phi.band_info()
        return {"active": i["active"] / i["states"].size, "shell": i["shell"] / i["states"].size, "bricks": int(i["states"].size)}

    for n in [int(s) for s in args.n.split(",")]:
        grid, dense, vel, terms = bench.build_c3(m, ctx, n, 1)
        band = m.NarrowBandMeshField(dense, halfwidth=args.halfwidth)
        rec = {"n": n, "halfwidth": args.halfwidth, "gpu": name, "power_limit": plimit, "clocks_max_sm": maxclk, "steps": args.steps}
        t = {"dense": 0.0, "band": 0.0}
        for when in ("t0", "later"):
            if when == "later":
                for key, f in (("dense", dense), ("band", band)):
                    _, t[key] = steps(f, terms, t[key], args.advance)
            row = {"band_fractions": fractions(band)}
            for key, f in (("dense", dense), ("band", band)):
                _, t[key] = steps(f, terms, t[key], args.warmup)
                row[f"{key}_ms"], t[key] = steps(f, terms, t[key], args.steps)
            ctx.set_option(L.OPT_TIME_STAGES, 1)
            ctx.reset_counters()
            ms, t["band"] = steps(band, terms, t["band"], args.steps)
            c = ctx.counters()
            ctx.set_option(L.OPT_TIME_STAGES, 0)
            stage_ms = c["sum_stage_ms"] / args.steps
            row.update(band_timed_ms=ms, band_stage_kernels_ms=stage_ms, band_rebuild_copy_cfl_ms=ms - stage_ms, t=dict(t))
            rec[when] = row
        del band, dense
        empty = m.NarrowBandMeshField(m.MeshField.from_shape(grid, "const", (1.0,), bc=m.NeumannBC(), ctx=ctx), halfwidth=args.halfwidth)
        assert empty.band_info()["active"] == 0
        te = 0.0
        _, te = steps(empty, terms, te, args.warmup)
        rec["empty_band_ms"], te = steps(empty, terms, te, args.steps)
        del empty, vel
        print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
