"""Per-step time and stage-kernel time (CUDA events) of C3 at 512^3 for a dtype, and the CFL reduction passes of the timed steps."""
import os, sys, ctypes as C
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np, lsm_b200 as m, helpers as H
L = m._lib
dt = np.float32 if len(sys.argv) > 1 and sys.argv[1] == "f32" else np.float64
ctx = m.default_context()
case = H.c3_enright(512, dt)
phi = case.engine_field(m); terms = case.engine_terms(m, phi)
eq = m.LevelSetEquation(terms=terms, ic=phi, integrator=m.RK3())
low = m.api._Lowered(eq.terms, eq.state, 0.0); dev = eq.state.device(); lib = L.lib()
def go(k, t0):
    t_out, n = C.c_double(), C.c_int64()
    L.check(lib.lsm_integrate(ctx.handle, 2, 0.5, dev, low.arr, 1, t0, 1e9, float("inf"), k, C.byref(t_out), C.byref(n)))
    return t_out.value
t = go(3, 0.0)
ctx.set_option(L.OPT_TIME_STAGES, 1)
ctx.reset_counters(); ctx.event_record(0); t = go(10, t); ctx.event_record(1)
ms = ctx.event_elapsed_ms(0, 1); c = ctx.counters()
print(np.dtype(dt).name, "ms/step", round(ms / 10, 3), "sum stage ms/step", round(c["sum_stage_ms"] / 10, 3), "cfl passes", c["cfl_passes"], flush=True)
