#!/usr/bin/env python
"""bench.py — cell-updates/s per RK3 step of the dense-grid hot path (BASELINE.json metric).

Workload (N = 1): BASELINE.json configs[2] "C3": 3-D sphere SDF in the Enright/LeVeque deformation
velocity (stored Float64 velocity field x cos(pi t / 3)), 512^3 nodes, WENO5 + TVD-RK3, NeumannBC.
One bench "step" = one RK3 step of integrate! = CFL reduction + 3 fused stage kernels.
N > 1: the same workload weak-scaled — every rank owns a 512 x 512 x 512 slab of a 512 x 512 x (512 N)
grid of cubic cells, 3-plane halos exchanged over NCCL each stage ("scaling": "weak").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--n 512] [--impl reference] [--dump-outputs DIR]
    torchrun --nproc-per-node N ... bench.py --gpus N ...

Prints ONE JSON line (rank 0).  `value` = device-timed (CUDA events on the library's compute stream,
max over ranks) with inputs resident in HBM; `e2e` = same metric through the public API with pinned
HOST buffers (H2D of phi, K steps, D2H of phi inside the timed region); `roofline` = the fused stage
kernel against the measured HBM copy bandwidth; `cpu_baseline` = the CPU oracle (a C++ restatement of
the reference — Julia is not installed) on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "cell-updates/s per RK3 step (3D WENO5 advection, Float64)"
UNIT = "cell-updates/s"
PERIOD = 3.0
B_ALG = 136.0          # bytes per cell-update, 3-D f64 RK3 advection with a stored velocity: (8 + 3N) * s (SURVEY.md §8d)
CPU_SAMPLE_N = 128     # cpu_baseline leg of the main line: the same configuration on a 128^3 grid (~0.12 s per RK3 step on 16 cores)
REF_SAMPLE_N = 256     # --impl reference: a 256^3 grid (~1 s per RK3 step on 16 cores; 512^3 would take ~8 s per step)
DUMP_NODES = 1 << 20   # --dump-outputs: nodes of the final level set written (8 MB of values + 8 MB of indices in float64)
DUMP_SEED = 0


def enright_tables(n, nz_glob, lz):
    """Per-axis factors of the C3 velocity on an n x n x nz_glob grid on (0,0,0)..(1,1,lz) (tests/helpers.py:enright_tables):
    u_d = ((s_d X_d[i]) Y_d[j]) Z_d[k]."""
    x = np.arange(n) * (1.0 / (n - 1))
    z = np.arange(nz_glob) * (lz / (nz_glob - 1))
    s2 = lambda a: np.sin(np.pi * a) ** 2
    s1 = lambda a: np.sin(2 * np.pi * a)
    return (2.0, -1.0, -1.0), [[s2(x), s1(x), s1(z)], [s1(x), s2(x), s1(z)], [s1(x), s1(x), s2(z)]]


def build_c3(m, ctx, n, G):
    """C3 with every field generated on the device (lsm_field_fill_shape / lsm_field_fill_separable): phi0 = |x - 0.35| - 0.15,
    stored Float64 Enright velocity x cos(pi t / 3).  N ranks: an n x n x (n N) grid of cubic cells, one n^3 slab per rank."""
    # cubic cells at every N: the domain is (0,0,0)..(1,1,lz) with lz = (nz - 1) h_x, so that h_z == h_x exactly (the isotropic-mesh
    # instantiation of the stage kernel runs at N > 1 as it does at N = 1)
    nz = n * G
    hx = 1.0 / (n - 1)
    lz = (nz - 1) * hx
    for _ in range(8):
        if lz / (nz - 1) == hx:
            break
        lz = float(np.nextafter(lz, lz + 1 if lz / (nz - 1) < hx else lz - 1))
    grid = m.CartesianGrid((0, 0, 0), (1, 1, lz), (n, n, nz))
    phi = m.MeshField.from_shape(grid, "sphere", (0.35, 0.35, 0.35, 0.15), bc=m.NeumannBC(), ctx=ctx)
    sc, tabs = enright_tables(n, nz, lz)
    vel = m.MeshField.from_separable(m.SeparableVelocity(grid, sc, tabs, ctx=ctx), ctx=ctx)
    terms = (m.AdvectionTerm(m.TimeScaled(vel, ("cos", PERIOD)), m.WENO5()),)
    return grid, phi, vel, terms


def build_c5(m, ctx, n, nz=None):
    """BASELINE.json configs[4] "C5" on the n^3 grid on (-1,-1,-1)..(1,1,1): phi0 = |x - (0.3,0,0)| - 0.4, NormalMotionTerm(v = 0.2
    stored scalar field) + AdvectionTerm(u = (-y, x, 0) stored field), all generated on the device.  nz != n (experiments: the slab
    shape of an 8-GPU run on fewer GPUs) keeps the cells cubic by shortening the domain along z."""
    nz = nz or n
    h = 2.0 / (n - 1)
    grid = m.CartesianGrid((-1, -1, -1), (1, 1, 1 if nz == n else -1 + (nz - 1) * h), (n, n, nz))
    phi = m.MeshField.from_shape(grid, "sphere", (0.3, 0.0, 0.0 if nz == n else -1 + 0.5 * (nz - 1) * h, 0.4), bc=m.NeumannBC(), ctx=ctx)
    x = -1.0 + np.arange(n) * (2.0 / (n - 1))
    one, onez = np.ones(n), np.ones(nz)
    rot = m.SeparableVelocity(grid, (-1.0, 1.0, 0.0), [[one, x, onez], [x, one, onez], [one, one, onez]], ctx=ctx)
    vel = m.MeshField.from_separable(rot, ctx=ctx)
    spd = m.MeshField.from_shape(grid, "const", (0.2,), ctx=ctx)
    return grid, phi, (m.NormalMotionTerm(spd), m.AdvectionTerm(vel, m.WENO5()))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={device}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.count(",") >= 8]
        os.unlink(self.f.name)
        if not rows:
            return out
        sm = sorted(float(r[1]) for r in rows)
        out["sm_mhz"] = sm[len(sm) // 2]
        out["sm_max_mhz"] = float(rows[0][2])
        out["power_w_max"] = max(float(r[3]) for r in rows)
        out["samples"] = len(rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for i, nm in enumerate(names):
            if any(r[5 + i].strip().lower().startswith("active") for r in rows):
                out["reasons"].append(nm)
        return out


def hbm_peak():
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(pk["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """dram bytes per stage-kernel launch from the committed ncu capture, if any (profiles/traffic.json)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["c3_stage_dram_bytes_per_launch"]
    except Exception:
        return None


def cpu_leg(steps, warmup, threads, n=CPU_SAMPLE_N):
    """The CPU oracle on an n^3 grid of the same configuration; returns (updates/s, seconds/step)."""
    import oracle as O
    import helpers as H
    O.set_threads(threads)
    case = H.c3_enright(n, period=PERIOD)
    f, terms = case.oracle_field(), case.oracle_terms()
    nodes = n ** 3
    t = 0.0
    for _ in range(warmup):
        dt = 0.5 * O.compute_cfl(f, terms, t)
        O.advance(f, O.RK3, terms, t, dt); t += dt
    t0 = time.perf_counter()
    for _ in range(steps):
        dt = 0.5 * O.compute_cfl(f, terms, t)
        O.advance(f, O.RK3, terms, t, dt); t += dt
    sec = time.perf_counter() - t0
    return nodes * steps / sec, sec / steps


def host_threads():
    """Threads the CPU legs use: every core this process may run on (torchrun exports OMP_NUM_THREADS=1, which would
    otherwise silently serialise the reference arm under N > 1)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the path.  The reference is 100 % Julia
    and Julia is not in this image, so this is the oracle port (kind "port") with all host threads."""
    if rank != 0:
        return
    threads = host_threads()
    v, sps = cpu_leg(args.steps, max(args.warmup, 1), threads, REF_SAMPLE_N)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"C3 Enright sphere, {REF_SAMPLE_N}^3 sample of the 512^3 config, WENO5+RK3, NeumannBC, stored velocity x cos(pi t/3)"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{REF_SAMPLE_N}^3 grid, {args.steps} RK3 steps, OpenMP over the slowest axis; C++ restatement of the "
                                   "reference (oracle/), not Julia — the reference's hot loop itself is serial"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def timed_steps(m, ctx, eq, steps, warmup, dist, barrier, time_stages=True):
    """`warmup` untimed RK3 steps, then `steps` steps bracketed by CUDA events on the library's compute stream; returns
    (ms, counters).  The whole loop runs inside lsm_integrate: 3 fused stage kernels per step, the CFL maximum of the time-scaled
    velocity evaluated on the host from its candidate nodes (no reduction pass / D2H / sync per step)."""
    import ctypes as C
    lib, L = m._lib.lib(), m._lib
    low = m.api._Lowered(eq.terms, eq.state, 0.0)
    dev = eq.state.device()

    def go(k, t0):
        t_out, st = C.c_double(), C.c_int64()
        L.check(lib.lsm_integrate(ctx.handle, L.RK3, 0.5, dev, low.arr, len(eq.terms), t0, 1e9, float("inf"), k, C.byref(t_out), C.byref(st)))
        assert st.value == k
        return t_out.value

    t = go(warmup, 0.0)
    if time_stages:
        ctx.set_option(L.OPT_TIME_STAGES, 1)
    barrier()
    ctx.reset_counters()
    ctx.event_record(0)
    t = go(steps, t)
    ctx.event_record(1)
    ms = ctx.event_elapsed_ms(0, 1)
    barrier()
    cnt = ctx.counters()
    ctx.set_option(L.OPT_TIME_STAGES, 0)
    eq.t = t                                  # lsm_integrate was called directly: record the time integrate! would have left
    if dist is not None:
        import torch
        tt = torch.tensor([ms], dtype=torch.float64, device=f"cuda:{ctx.device}")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    return ms, cnt, low


def dump_outputs(out_dir, eq):
    """--dump-outputs: what a caller of the timed path receives after its last step, i.e. the level set and the final time.
    The level set is written at DUMP_NODES nodes drawn with a fixed seed (all of them on a smaller grid), with their
    column-major flat indices, so that two builds run with the same arguments can be compared output for output."""
    phi = eq.state.peek().ravel(order="F")
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(phi.size, min(DUMP_NODES, phi.size), replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "phi_sample.npy"), phi[idx].astype(np.float64))
    np.save(os.path.join(out_dir, "phi_sample_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "t.npy"), np.array([eq.t], dtype=np.float64))


def invariance_check(m, ctx, dist, rank, world, local):
    """SURVEY.md §8(e): the slab-decomposed result must equal the 1-GPU result BITWISE.  Small C3 instance (96 x 80 x 24 N nodes,
    6 RK3 steps, periodic in the decomposed axis so that the wrap-around exchange is covered too): every rank integrates its slab,
    rank 0 also integrates the whole grid alone on a single-rank context and compares with the gathered slabs."""
    import torch
    n0, n1, nz = 96, 80, 24 * world
    bc = (m.NeumannBC(), m.NeumannBC(), m.PeriodicBC())

    def run(c):
        grid = m.CartesianGrid((0, 0, 0), (1, 1, 1), (n0, n1, nz))
        phi = m.MeshField.from_shape(grid, "sphere", (0.4, 0.45, 0.5, 0.2), bc=bc, ctx=c)
        x, y, z = [np.arange(k) / (k - 1) for k in (n0, n1, nz)]
        s2 = lambda a: np.sin(np.pi * a) ** 2 + 0.05
        s1 = lambda a: np.sin(2 * np.pi * a) + 0.05
        sep = m.SeparableVelocity(grid, (2.0, -1.0, -1.0), [[s2(x), s1(y), s1(z)], [s1(x), s2(y), s1(z)], [s1(x), s1(y), s2(z)]], ctx=c)
        vel = m.MeshField.from_separable(sep, ctx=c)
        eq = m.LevelSetEquation(terms=(m.AdvectionTerm(m.TimeScaled(vel, ("cos", PERIOD)), m.WENO5()),), ic=phi, integrator=m.RK3())
        dt = 0.5 * m.compute_cfl(eq.terms, eq.state, 0.0)
        m.integrate(eq, 6 * dt * (1 - 1e-12))
        return eq.steps_taken, np.ascontiguousarray(np.moveaxis(eq.state.peek(), -1, 0))      # planes first

    steps, mine = run(ctx)
    parts = [torch.empty((24,) + mine.shape[1:], dtype=torch.float64, device=f"cuda:{local}") for _ in range(world)]
    dist.all_gather(parts, torch.from_numpy(mine).to(f"cuda:{local}"))
    out = None
    if rank == 0:
        single = m.Context(local)
        s1, whole = run(single)
        got = torch.cat(parts, 0).cpu().numpy()
        out = {"bitwise": bool(s1 == steps and np.array_equal(got, whole)), "max_abs_diff": float(np.abs(got - whole).max()),
               "grid": [n0, n1, nz], "steps": int(steps), "bc": "Neumann x Neumann x Periodic(decomposed axis)"}
        single.close()
    dist.barrier()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--n", "--size", dest="n", type=int, default=0,
                    help="nodes per axis (c3: per GPU, default 512; c5: global, default 1024); use --size under torchrun, whose own parser\n"
                         "rejects --n as an ambiguous abbreviation of --nnodes / --nproc-per-node")
    ap.add_argument("--nz", type=int, default=0, help="c5 only (experiments): global node count along the decomposed axis, default = size")
    ap.add_argument("--workload", default="c3", choices=["c3", "c5"],
                    help="c3 = headline (weak-scaled Enright advection); c5 = BASELINE configs[4], strong-scaled 1024^3 normal motion + advection")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kernel", type=int, default=0, help="0 auto, 1 strict generic, 2 tiled / x-pair, 3 tiled only, 4 x-pair with exact epsilon maximum")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="N > 1: skip the C5 1024^3 strong-scaling attachment and the invariance check")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a seeded sample of the final level set and the "
                                                         "final time to DIR/*.npy (float64); single GPU only")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (args.impl == "reference" or world > 1):
        raise SystemExit("--dump-outputs writes the outputs of the single-GPU device path (--impl ours, --gpus 1)")
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    # stdout carries exactly ONE JSON line: NCCL prints its version banner to stdout at NCCL_DEBUG >= VERSION (WARN included),
    # so send NCCL's debug output to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

    import lsm_b200 as m
    import ctypes as C
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        ctx = m.Context.from_torch_distributed(local)
    else:
        ctx = m.Context(local)
    m.set_default_context(ctx)
    ctx.set_option(m._lib.OPT_KERNEL, args.kernel)
    lib, L = m._lib.lib(), m._lib

    def barrier():
        ctx.sync()
        if dist is not None:
            dist.barrier()

    G = world
    c5 = args.workload == "c5"
    n = args.n or (1024 if c5 else 512)
    invariance = None
    if G > 1 and not args.no_extras:
        invariance = invariance_check(m, ctx, dist, rank, world, local)
    if c5:
        grid, phi, terms = build_c5(m, ctx, n, args.nz or None)
        nz = args.nz or n
        args.no_e2e = True
        args.no_cpu = True
    else:
        grid, phi, vel, terms = build_c3(m, ctx, n, G)
        nz = n * G
    z_first, nz_loc = ctx.slab(nz) if G > 1 else (0, nz)
    nodes_total = n * n * nz
    balg = 160.0 if c5 else B_ALG
    eq = m.LevelSetEquation(terms=terms, ic=phi, integrator=m.RK3())

    # ---- warm-up, then the device-timed region -------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None      # samples clocks from the warm-up on (all of it is under load)
    if sampler:
        time.sleep(0.4)                                       # let nvidia-smi start sampling
    ms, cnt, low = timed_steps(m, ctx, eq, args.steps, args.warmup, dist, barrier)
    clocks = sampler.stop() if sampler else None
    value = nodes_total * args.steps / (ms * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, eq)              # before the e2e leg, which integrates the same state again from phi0

    # ---- e2e: the public API with pinned HOST buffers ------------------------------------------------------------------
    # cold  = what a first integrate! sees: H2D of phi AND of the stored velocity (AoS -> SoA on the device), K steps, D2H of phi
    # warm  = a repeated integrate! on the same equation: the velocity's device mirror is current, only phi travels
    e2e = None
    if not args.no_e2e:
        state = eq.state
        host_phi0 = phi.peek().copy(order="F")             # D2H of the device-generated fields (outside the timed regions)
        host_u = vel.vals                                  # host AoS array (N, n, n, nz_loc); marks the device mirror stale
        host = state.vals
        for arr in (host, host_u):
            L.check(lib.lsm_host_register(arr.ctypes.data, arr.nbytes))
        res = {}
        for mode in ("cold", "warm"):
            host[...] = host_phi0
            if mode == "cold":
                vel.vals                                   # the caller touched the velocity: upload it again
            eq.t = 0.0
            barrier()
            w0 = time.perf_counter()
            state.vals                                     # host copy is the fresh one -> integrate! uploads it
            low2 = m.api._Lowered(eq.terms, state, 0.0)    # H2D of the velocity when stale (pinned)
            dev2 = state.device()                          # H2D of phi (pinned)
            t_out, st = C.c_double(), C.c_int64()
            L.check(lib.lsm_integrate(ctx.handle, L.RK3, 0.5, dev2, low2.arr, len(eq.terms), 0.0, 1e9, float("inf"), args.steps, C.byref(t_out), C.byref(st)))
            state._mark_device_advanced()
            out = state.peek()                             # D2H of phi (pinned)
            chk = float(out[0, 0, 0])
            barrier()
            w = time.perf_counter() - w0
            if dist is not None:
                import torch
                tt = torch.tensor([w], dtype=torch.float64, device=f"cuda:{local}")
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                w = float(tt.item())
            res[mode] = (nodes_total * args.steps / w, chk)
        for arr in (host, host_u):
            L.check(lib.lsm_host_unregister(arr.ctypes.data))
        e2e = {"value": res["cold"][0], "unit": UNIT,
               "h2d_bytes_per_step": (host.nbytes + host_u.nbytes) * G / args.steps, "d2h_bytes_per_step": host.nbytes * G / args.steps,
               "call": f"one integrate! of {args.steps} RK3 steps on host MeshFields: H2D of phi and of the stored velocity from pinned host memory, "
                       "steps, D2H of phi (what the first integrate! of a session sees)",
               "warm": {"value": res["warm"][0], "h2d_bytes_per_step": host.nbytes * G / args.steps,
                        "call": "the same call again: the velocity's device mirror is current (cached per host array), only phi travels — "
                                "what every later integrate! on the same equation sees, in Python and in the Julia glue"},
               "check": res["cold"][1]}
        assert res["cold"][1] == res["warm"][1]

    # ---- N > 1: the north-star multi-GPU target, C5 1024^3 STRONG-scaled over the same ranks ------------------------------
    c5_strong = None
    if G > 1 and not c5 and not args.no_extras:
        del eq, phi, vel, terms
        n5, k5 = 1024, 6
        g5, p5, t5 = build_c5(m, ctx, n5)
        eq5 = m.LevelSetEquation(terms=t5, ic=p5, integrator=m.RK3())
        ms5, cnt5, _ = timed_steps(m, ctx, eq5, k5, 2, dist, barrier)
        st5 = cnt5["sum_stage_ms"] / max(cnt5["timed_stages"], 1)
        del eq5, p5, t5
        c5_strong = {"workload": "C5 NormalMotionTerm(v field) + AdvectionTerm(u field) 1024^3 Float64, slab-decomposed, NCCL halo exchange",
                     "value": n5 ** 3 * k5 / (ms5 * 1e-3), "unit": UNIT, "ms_per_step": ms5 / k5, "steps": k5, "n_gpus": G,
                     "stage_ms": st5, "roofline_frac_per_gpu": (160.0 / 3.0) * (n5 ** 3 / G) / (st5 * 1e-3) / 1e9 / hbm_peak()[0]}
        if rank == 0:        # the 1-GPU time of the same problem, measured now on GPU 0 alone (60 GB of fields), gives the efficiency
            single = m.Context(local)
            g1, p1, t1 = build_c5(m, single, n5)
            eq1 = m.LevelSetEquation(terms=t1, ic=p1, integrator=m.RK3())
            ms1, _, _ = timed_steps(m, single, eq1, k5, 2, None, single.sync)
            del eq1, p1, t1
            single.close()
            c5_strong["single_gpu_ms_per_step"] = ms1 / k5
            c5_strong["parallel_efficiency"] = (ms1 / k5) / (G * ms5 / k5)
        dist.barrier()

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peak, peak_src = hbm_peak()
    stage_ms = cnt["sum_stage_ms"] / max(cnt["timed_stages"], 1)
    bytes_per_launch = (balg / 3.0) * (n * n * nz_loc)           # average over the 3 stage launches of a step (c3: 40+48+48 B/node)
    achieved = bytes_per_launch / (stage_ms * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": G, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if c5 else "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": (f"C5 NormalMotionTerm(v field) + AdvectionTerm(u field), {n}^3 global (BASELINE.json configs[4]), WENO5 + TVD-RK3, "
                                "NeumannBC, slab-decomposed with NCCL halo exchange" if c5 else
                                f"C3 Enright sphere {n}x{n}x{nz} (BASELINE.json configs[2]; {n}^3 per GPU), WENO5 + TVD-RK3, NeumannBC, "
                                "stored Float64 velocity field x cos(pi t/3), CFL step recomputed every step (exact, from the velocity's candidate nodes)"),
                   "grid": [n, n, nz], "parallelism": f"slab{G}" if G > 1 else "single",
                   "l2": "inputs larger than L2 (each field >= 1 GB per GPU)",
                   "kernel": ["auto (x-pair kernel, 20-bit epsilon maximum)", "strict-generic", "tiled / x-pair", "tiled", "x-pair, exact epsilon maximum"][args.kernel],
                   "fields": "generated on the device (lsm_field_fill_shape / lsm_field_fill_separable)"},
        "clocks": clocks,
        "gpu_launches": int(cnt["kernel_launches"]),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": ncu_traffic(), "peak_source": peak_src,
                     "kernel": "fused RK stage (stencil + Hamiltonian + RK combination)",
                     "algorithmic_bytes_per_launch": bytes_per_launch, "avg_launch_ms": stage_ms,
                     "launches_timed": int(cnt["timed_stages"]),
                     "frac_of_nominal_8TBs": achieved / 8000.0,      # SURVEY.md §8(d): reported against both the measured and the nominal roof
                     "co_bound": "FP64 issue: a DP instruction holds the SMSP dispatch port 2 cycles (tools/issue_model.cu); "
                                 "18.3 T lane-ops/s measured (tools/fp64_peak.cu); see DESIGN.md §4.1"},
        "e2e": e2e,
    }
    if invariance is not None:
        line["invariance"] = invariance
    if c5_strong is not None:
        line["c5_strong"] = c5_strong
    if G == 1 and not args.no_cpu:
        thr = host_threads()
        v_all, _ = cpu_leg(3, 1, thr)
        v_one, _ = cpu_leg(1, 0, 1)
        line["cpu_baseline"] = {"value": v_all, "unit": UNIT, "cores": thr, "kind": "port",
                                "sample": f"C3 on a {CPU_SAMPLE_N}^3 grid, 3 RK3 steps, OpenMP x{thr}; 1 thread (the reference's hot loop "
                                          f"is serial): {v_one:.4g} updates/s. C++ restatement of the reference, not Julia (not installed)"}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
