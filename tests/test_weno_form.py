"""The completed-square form of the WENO5 smoothness indicators in the default mode of the 3-D x-pair kernel
(csrc/lsm_pair_common.cuh: weno_core_de).  The weights depend only on ratios of b1..b3, so the kernel evaluates
(3/16) b_k as a square plus a non-negative rest, with eps scaled by 3/16 as well:

    (3/16) b1 = (e1 - 11/8 e2)^2 + 39/64 e2^2 + eps'
    (3/16) b2 = (e2 - 5/8 e3)^2  + 39/64 e3^2 + eps'
    (3/16) b3 = (e4 - 11/8 e3)^2 + 39/64 e3^2 + eps'        eps' = (3/16) eps

and G1 = 5/6 e2 - 1/3 e1 as 3/8 e2 - 1/3 (e1 - 11/8 e2).  The CPU tests check the identity exactly and restate both
forms in Float64 with correctly rounded fma; the GPU test checks that the kernel's eps' is scaled with the b_k.
"""
import math
import random
from fractions import Fraction as Fr

import numpy as np
import pytest

import helpers as H

# weno_constants() (csrc/lsm_kernels.h) and the scaled eps constants weno_regs<false> derives from them
C133, C56, CM13, E6, FL = 13.0 / 3.0, 5.0 / 6.0, -1.0 / 3.0, 4.0e-6, 1.0e-70
E6S, FLS = E6 * 0.1875, FL * 0.1875
DYADIC = {"11/8": (1.375, Fr(11, 8)), "5/8": (0.625, Fr(5, 8)), "39/64": (0.609375, Fr(39, 64)),
          "3/8": (0.375, Fr(3, 8)), "3/16": (0.1875, Fr(3, 16))}


def fma(a, b, c):
    """Correctly rounded a * b + c (IEEE fma) for finite operands; NaN / Inf propagate as in hardware."""
    if not (math.isfinite(a) and math.isfinite(b) and math.isfinite(c)):
        return a * b + c
    return float(Fr(a) * Fr(b) + Fr(c))


def stencil_e(d):
    return d[1] - d[0], d[2] - d[1], d[3] - d[2], d[4] - d[3]


def absmax(d):
    m = d[0]
    for x in d[1:]:
        m = x if abs(x) > abs(m) else m
    return m


def core_old(d):
    """The exact-mode evaluation (weno5_up of lsm_tile_util.cuh) with an exact quotient: (b1, b2, b3), h * weno."""
    e1, e2, e3, e4 = stencil_e(d)
    m = absmax(d)
    eps = fma(E6, m * m, FL)
    t1a, t1b, t1c = e2 - e1, e3 - e2, e4 - e3
    t2a, t2b, t2c = fma(3.0, e2, -e1), e2 + e3, fma(-3.0, e3, e4)
    b = (fma(t2a, t2a, fma(C133, t1a * t1a, eps)), fma(t2b, t2b, fma(C133, t1b * t1b, eps)),
         fma(t2c, t2c, fma(C133, t1c * t1c, eps)))
    G1 = fma(C56, e2, CM13 * e1)
    return b, _finish(d, b, G1, e2, e3, e4)


def core_new(d):
    """The default-mode evaluation of weno_core_de (exact maximum, to isolate the form): (3/16) (b1, b2, b3), h * weno."""
    e1, e2, e3, e4 = stencil_e(d)
    m = absmax(d)
    eps = fma(E6S, m * m, FLS)
    X1, X2, X3 = fma(-1.375, e2, e1), fma(-0.625, e3, e2), fma(-1.375, e3, e4)
    F2, F3 = fma(0.609375, e2 * e2, eps), fma(0.609375, e3 * e3, eps)
    b = (fma(X1, X1, F2), fma(X2, X2, F3), fma(X3, X3, F3))
    G1 = fma(0.375, e2, CM13 * X1)
    return b, _finish(d, b, G1, e2, e3, e4)


def _finish(d, b, G1, e2, e3, e4):
    b1, b2, b3 = b
    p12, p13, p23 = b1 * b2, b1 * b3, b2 * b3
    w1, w2, w3 = p23 * p23, p13 * p13, p12 * p12
    den = fma(3.0, w3, fma(6.0, w2, w1))
    G2, G3 = fma(2.0, e3, e2), fma(2.0, e3, -0.5 * e4)
    num = fma(w3, G3, fma(w2, G2, w1 * G1))
    return fma(num, 1.0 / den, d[2])


def test_coefficients_are_dyadic():
    """Every coefficient of the form is exact in binary, so it is an instruction immediate and carries no rounding."""
    for name, (x, f) in DYADIC.items():
        assert Fr(x) == f, name


@pytest.mark.parametrize("side", ["minus", "plus"])
def test_identity_exact(side):
    """(3/16) b_k of the reference equals the completed square for every k, in exact arithmetic, on random integer samples of
    either upwind side (the plus-biased side evaluates the reversed first differences, i.e. negated second differences)."""
    rng = random.Random(20261020 + (side == "plus"))
    for trial in range(2000):
        span = 10 ** rng.randint(0, 12)
        phi = [rng.randint(-span, span) for _ in range(7)]
        if side == "minus":
            d = [Fr(phi[k + 1] - phi[k]) for k in range(5)]
        else:
            d = [Fr(phi[6 - k] - phi[5 - k]) for k in range(5)]
        e1, e2, e3, e4 = stencil_e(d)
        eps = Fr(rng.randint(0, span)) / 7
        b_ref = (Fr(13, 3) * (e2 - e1) ** 2 + (3 * e2 - e1) ** 2 + eps,
                 Fr(13, 3) * (e3 - e2) ** 2 + (e2 + e3) ** 2 + eps,
                 Fr(13, 3) * (e4 - e3) ** 2 + (e4 - 3 * e3) ** 2 + eps)
        eps_s = Fr(3, 16) * eps
        b_sq = ((e1 - Fr(11, 8) * e2) ** 2 + Fr(39, 64) * e2 ** 2 + eps_s,
                (e2 - Fr(5, 8) * e3) ** 2 + Fr(39, 64) * e3 ** 2 + eps_s,
                (e4 - Fr(11, 8) * e3) ** 2 + Fr(39, 64) * e3 ** 2 + eps_s)
        for k in range(3):
            assert Fr(3, 16) * b_ref[k] == b_sq[k], (side, trial, k)
        assert Fr(5, 6) * e2 - Fr(1, 3) * e1 == Fr(3, 8) * e2 - Fr(1, 3) * (e1 - Fr(11, 8) * e2)


def _samples():
    """Adversarial first-difference stencils: flat, linear (rounding-level second differences), kinked, smooth, random, at
    magnitudes 1e-30 .. 1e3."""
    rng = np.random.default_rng(7)
    out = []
    for scale in (1e-30, 1e-20, 1e-12, 1e-6, 1e-2, 1.0, 1e3):
        for _ in range(40):
            c = scale * rng.uniform(-1, 1)
            out.append(("flat", [c] * 5))
            x0, s = rng.uniform(-3, 3), scale * rng.uniform(-1, 1)
            phi = [s * (x0 + k) for k in range(6)]
            out.append(("linear", [phi[k + 1] - phi[k] for k in range(5)]))
            k0, a, b = rng.uniform(0, 5), scale * rng.uniform(-1, 1), scale * rng.uniform(-1, 1)
            phi = [a * (k - k0) if k < k0 else b * (k - k0) for k in range(6)]
            out.append(("kink", [phi[k + 1] - phi[k] for k in range(5)]))
            h, x = 10 ** rng.uniform(-3, -1), rng.uniform(0, 6)
            phi = [scale * math.sin(x + k * h) for k in range(6)]
            out.append(("smooth", [phi[k + 1] - phi[k] for k in range(5)]))
            out.append(("random", list(scale * rng.uniform(-1, 1, 5))))
            out.append(("noisy-linear", list(s * (1 + 1e-3 * rng.uniform(-1, 1, 5)))))
    return out


def test_float64_restatement_matches_old_form():
    """Both forms in Float64, correctly rounded fma, the same exact eps maximum: the scaled indicators agree with 3/16 of the old
    ones to a few ulp (every term is non-negative: no cancellation), and the result agrees to a few ulp of the stencil scale.
    Flat stencils give exactly d2.  Below |d| ~ 1e-25 the products w_k G_k of either form are subnormal (the weights are
    ~b^4 and b >= eps' >= 1.9e-71), so there the quotient is only good to the subnormal spacing over the smallest denominator:
    `tiny`, an absolute ~6e-39, far below anything a level set resolves."""
    tiny = 16 * 2.0 ** -1074 / FLS ** 4
    worst_b, worst_w = 0.0, 0.0
    for kind, d in _samples():
        d = [float(x) for x in d]
        bo, wo = core_old(d)
        bn, wn = core_new(d)
        for k in range(3):
            assert bn[k] > 0
            rel = abs(bn[k] - 0.1875 * bo[k]) / (0.1875 * bo[k])
            worst_b = max(worst_b, rel)
            assert rel <= 4e-15, (kind, d, k, rel)
        if kind == "flat":
            assert wn == d[2] and wo == d[2], (d, wn, wo)
        scale = max(abs(x) for x in d)
        excess = abs(wn - wo) - tiny
        if excess > 0:
            worst_w = max(worst_w, excess / scale)
            assert excess <= 2e-15 * scale, (kind, d, wn, wo)
    print(f"worst relative b difference {worst_b:.2e}, worst result difference beyond `tiny` {worst_w:.2e} of max|d|")


def test_nan_propagates():
    for pos in range(5):
        d = [0.1, 0.2, 0.25, 0.27, 0.3]
        d[pos] = float("nan")
        assert math.isnan(core_new(d)[1]) and math.isnan(core_old(d)[1])


# ---- on the device --------------------------------------------------------------------------------------------------------
OPT_KERNEL = 0


def _near_eps_case(two_terms):
    """A linear field plus noise of 3e-4 h on an isotropic 64 x 48 x 40 grid: away from the Neumann boundary layer the
    smoothness indicators are a few times eps, so the weights depend on eps at first order."""
    n = (64, 48, 40)
    h = 1.0 / 63
    lc, hc = (0, 0, 0), tuple(h * (k - 1) for k in n)
    x, y, z = H.coords(lc, hc, n)
    rng = np.random.default_rng(11)
    phi = H.bcast(0.6 * x - 0.5 * y + 0.4 * z - 0.1, n) + 3e-4 * h * rng.uniform(-1, 1, n)
    u = np.stack([H.bcast(np.full((1, 1, 1), c), n) for c in (0.7, -0.5, 0.3)], axis=0)
    terms = [dict(kind="advection", field=u)]
    if two_terms:
        terms.insert(0, dict(kind="normal", field=H.bcast(0.2 + 0.1 * np.sin(5 * x) * np.cos(3 * y) - 0.05 * z, n)))
    return H.Case("eps", lc, hc, n, phi, terms, ("neumann",), np.float64), u, h


@pytest.mark.gpu
@pytest.mark.parametrize("two_terms", [False, True], ids=["advection", "normal+advection"])
def test_default_mode_eps_scaling(two_terms):
    """One ForwardEuler step where the weights depend on eps at first order, default mode (20-bit eps maximum) against the
    exact mode (LSM_OPT_KERNEL = 4).  The 20-bit maximum changes eps by a relative delta <= 2^-19, each b_k by at most that,
    each normalised weight by <= 4 delta (w ~ 1/b^2, then normalised), so the WENO value of a dimension moves by at most
    4 delta max|q_k| with q = (G1, G2/6, G3/3), |q_k| <= 7/6 max|e|; the step scales that by dt sum_d |u_d| / h.  An eps'
    that is not scaled with the b_k moves the weights by O(1) here, over 1e4 times this bound."""
    import lsm_b200 as m
    case, u, h = _near_eps_case(two_terms)
    ctx = m.default_context()
    outs = []
    try:
        for kernel in (0, 4):
            ctx.set_option(OPT_KERNEL, kernel)
            ctx.reset_counters()
            phi = case.engine_field(m)
            eq = m.LevelSetEquation(terms=case.engine_terms(m, phi), ic=phi, integrator=m.ForwardEuler())
            dt = 0.5 * m.compute_cfl(eq.terms, eq.state, 0.0)
            m.integrate(eq, dt * (1 - 1e-12))
            assert eq.steps_taken == 1 and ctx.counters()["pair_launches"] > 0
            outs.append((eq.t, eq.state.peek().copy()))
    finally:
        ctx.set_option(OPT_KERNEL, 0)
    assert outs[0][0] == outs[1][0]
    # max|e| away from the boundary layer (there the mirrored kink makes b >> eps and the eps sensitivity vanishes)
    p = case.phi0
    emax = max(np.abs(np.diff(p, 2, axis=a)[3:-3, 3:-3, 3:-3]).max() for a in range(3))
    delta = 2.0 ** -19
    cfl_sum = sum(abs(float(u[d].flat[0])) for d in range(3)) / h
    tol = dt * cfl_sum * (4 * delta * 7 / 6 * emax) * 2 + 8 * np.finfo(np.float64).eps * np.abs(p).max()
    diff = float(np.abs(outs[0][1] - outs[1][1]).max())
    print(f"eps-scaling {'two terms' if two_terms else 'advection'}: max |mode 0 - mode 4| {diff:.3e}, bound {tol:.3e}")
    assert 0 < diff <= tol, (diff, tol)
