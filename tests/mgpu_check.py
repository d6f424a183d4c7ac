"""Multi-GPU decomposition-invariance check (SURVEY.md §8e), run under torchrun on N >= 2 GPUs:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tests/mgpu_check.py

For every configuration the slab-decomposed run (NCCL halo exchange, interior/boundary overlap) must
equal the single-GPU run BIT FOR BIT and match the CPU oracle within 1e-10.  Exit code 0 = pass.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def main():
    import torch
    import torch.distributed as dist
    import lsm_b200 as m
    import helpers as H

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = m.Context.from_torch_distributed(local)
    solo = m.Context(local) if rank == 0 else None

    def periodic_z(case):
        case.bc = (("neumann",), ("extrap", 2), ("periodic",))
        return case

    nz = 16 * world + 5
    # every slab keeps >= 8 planes so that ranks and the 1-GPU comparison run select the same (tiled) kernels;
    # thinner slabs fall back to the strict kernel, which is bit-equal to the oracle but not to the tiled kernel
    nc = max(24, 10 * world)
    cases = []
    c = H.c3_enright(nc); cases.append(("C3 WENO5 advection x cos (CFL candidates), Neumann", c, "RK3", 8))
    c = H.c5_normal_advection(nc); cases.append(("C5 normal motion + advection", c, "RK3", 6))
    c = H.c4_eikonal(nc); cases.append(("C4 eikonal RK2", c, "RK2", 6))
    # 2-D, decomposed along y: on 2 ranks every slab is large enough for the 2-D x-pair kernel (rows arrive through the halo rows)
    c = H.c2_zalesak_curvature(768); cases.append(("C2 2-D Zalesak advection + curvature", c, "RK3", 5))
    # uneven slabs + periodic wrap across ranks (node n duplicates node 1) + extrapolation in y
    lc, hc, n = (-1, -1, -1), (1, 1, 1), (20, 18, nz)
    X = H.coords(lc, hc, n)
    phi = np.sqrt((X[0] - 0.2) ** 2 + X[1] ** 2 + X[2] ** 2) - 0.5
    u = np.stack([H.bcast(0.3 + 0 * X[0], n), H.bcast(-0.2 + 0.1 * X[1], n), H.bcast(1.0 + 0.2 * np.sin(X[0]), n)], axis=0)
    cases.append(("advection, periodic z across ranks", periodic_z(H.Case("pz", lc, hc, n, phi, [dict(kind="advection", field=u)], None)), "RK3", 10))
    cases.append(("FE upwind, periodic z", periodic_z(H.Case("pz2", lc, hc, n, phi, [dict(kind="advection", field=u, scheme="upwind")], None)), "FE", 5))

    ok = True
    for name, case, integ, steps in cases:
        mk = {"RK3": m.RK3, "RK2": m.RK2, "FE": m.ForwardEuler}[integ]
        for overlap in (1, 0):
            ctx.set_option(m._lib.OPT_OVERLAP, overlap)
            phi_f = case.engine_field(m, ctx=ctx)
            eq = m.LevelSetEquation(terms=case.engine_terms(m, phi_f, ctx=ctx), ic=phi_f, integrator=mk())
            dt0 = 0.5 * m.compute_cfl(eq.terms, eq.state, 0.0)
            tf = dt0 * steps * (1 - 1e-12)
            m.integrate(eq, tf)
            mine = np.ascontiguousarray(eq.state.peek())
            parts = [None] * world
            dist.gather_object((eq.state.local_range, mine), parts if rank == 0 else None, dst=0)
            if rank == 0:
                full = np.concatenate([p[1] for p in sorted(parts, key=lambda q: q[0][0])], axis=-1)
                m.set_default_context(solo)
                phi_s = case.engine_field(m, ctx=solo)
                eq_s = m.LevelSetEquation(terms=case.engine_terms(m, phi_s, ctx=solo), ic=phi_s, integrator=mk())
                m.integrate(eq_s, tf)
                single = eq_s.state.peek()
                import oracle as O
                fo = case.oracle_field()
                O.set_threads(8)
                O.integrate(fo, {"RK3": O.RK3, "RK2": O.RK2, "FE": O.FE}[integ], case.oracle_terms(), tf)
                bit = np.array_equal(full, single)
                d = float(np.abs(full - fo.vals).max())
                good = bit and d <= 1e-10 and eq.steps_taken == eq_s.steps_taken
                ok &= good
                print(f"[{'ok' if good else 'FAIL'}] {name} ({world} ranks, overlap={overlap}): bitwise == 1-GPU: {bit}; "
                      f"max-abs vs oracle {d:.2e}; steps {eq.steps_taken}", flush=True)
    # ---- "next" rows on a decomposed field: device volume / perimeter (all-reduced), set operations, velocity extension
    m.set_default_context(ctx)
    n3 = (nc, nc + 2, 16 * world + 3)
    lc3, hc3 = (-1, -1, -1), (1, 1, 1)
    X = H.coords(lc3, hc3, n3)
    a0 = H.bcast(np.sqrt((X[0] - 0.1) ** 2 + X[1] ** 2 + X[2] ** 2) - 0.6, n3)
    b0 = H.bcast(np.maximum(np.abs(X[0]), np.maximum(np.abs(X[1]), np.abs(X[2] - 0.2))) - 0.45, n3)
    F0 = H.bcast(np.sin(2 * X[0]) + X[1] * X[2], n3)

    def run_next(c):
        g = m.CartesianGrid(lc3, hc3, n3)
        a = m.MeshField(a0.copy(order="F"), g, bc=m.NeumannBC(), ctx=c)
        b = m.MeshField(b0.copy(order="F"), g, ctx=c)
        m.setdiff_(a, b)
        vol, per = m.volume(a), m.perimeter(a)
        F = m.MeshField(F0.copy(order="F"), g, ctx=c)
        m.extend_along_normals(F, a, nb_iters=10)
        return vol, per, np.ascontiguousarray(a.peek()), np.ascontiguousarray(F.peek()), a.local_range

    vol, per, av, Fv, rng = run_next(ctx)
    parts = [None] * world
    dist.gather_object((rng, av, Fv), parts if rank == 0 else None, dst=0)
    if rank == 0:
        parts.sort(key=lambda q: q[0][0])
        a_full = np.concatenate([p[1] for p in parts], axis=-1)
        F_full = np.concatenate([p[2] for p in parts], axis=-1)
        m.set_default_context(solo)
        vol1, per1, a1, F1, _ = run_next(solo)
        good = (np.array_equal(a_full, a1) and abs(vol - vol1) <= 1e-12 * abs(vol1) and abs(per - per1) <= 1e-12 * abs(per1)
                and float(np.abs(F_full - F1).max()) <= 1e-12)
        ok &= good
        print(f"[{'ok' if good else 'FAIL'}] setdiff! + volume/perimeter + extend_along_normals! ({world} ranks): CSG bitwise {np.array_equal(a_full, a1)}; "
              f"volume {vol:.15g} vs {vol1:.15g}; perimeter {per:.15g} vs {per1:.15g}; extension max-abs diff {float(np.abs(F_full - F1).max()):.2e}", flush=True)
    res = [ok]
    dist.broadcast_object_list(res, src=0)
    if rank == 0:
        c = ctx.counters()
        print(f"halo bytes sent by rank 0: {c['halo_bytes_sent']}", flush=True)
        print("ALL OK" if res[0] else "FAILED", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if res[0] else 1)


if __name__ == "__main__":
    main()
