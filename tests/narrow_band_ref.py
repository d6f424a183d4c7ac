"""NumPy restatement of the narrow-band rules of include/lsm_b200.h (lsm_field_set_band) and of a band step on the oracle.

Written from the header's definitions, set by set: N(b) is built per axis as a Python set and the shell is the union of N(a) over
the active bricks a (a scatter), where the device gathers through the inverse neighbourhood.
"""
import numpy as np

BRICK = (32, 16, 16)


def brick_counts(n):
    return tuple(-(-n[d] // BRICK[d]) for d in range(len(n)))


def axis_neighbours(b, n, B, periodic):
    """R_d(b) on an axis of n nodes in bricks of B nodes."""
    nb = -(-n // B)
    r = {k for k in (b - 1, b, b + 1) if 0 <= k < nb}
    if periodic:
        holds = lambda k, nodes: any(k * B <= i < min(n, (k + 1) * B) for i in nodes)
        brick_of = lambda i: i // B
        if holds(b, [i for i in (0, 1, 2) if 0 <= i < n]):
            r |= {brick_of(i) for i in (n - 4, n - 3, n - 2) if 0 <= i < n}
        if holds(b, [i for i in (n - 3, n - 2, n - 1) if 0 <= i < n]):
            r |= {brick_of(i) for i in (1, 2, 3) if 0 <= i < n}
    return r


def neighbourhood(b, n, periodic):
    """N(b): the product over axes of R_d(b_d); b and the result are brick coordinate tuples."""
    sets = [sorted(axis_neighbours(b[d], n[d], BRICK[d], periodic[d])) for d in range(len(n))]
    out = [()]
    for s in sets:
        out = [o + (k,) for o in out for k in s]
    return out


def gamma(halfwidth, h):
    return halfwidth * min(abs(x) for x in h)


def core_flags(phi, h, halfwidth):
    """Per brick: holds a node with !(|phi| > gamma) (|phi| <= gamma or NaN)."""
    g = gamma(halfwidth, h)
    near = ~(np.abs(phi.astype(np.float64)) > g)
    nb = brick_counts(phi.shape)
    core = np.zeros(nb, dtype=bool)
    for b in np.ndindex(*nb):
        sl = tuple(slice(b[d] * BRICK[d], (b[d] + 1) * BRICK[d]) for d in range(phi.ndim))
        core[b] = near[sl].any()
    return core


def band_states(phi, h, halfwidth, periodic):
    """One byte per brick (array of brick coordinates): 0 frozen, 1 shell, 2 active, 3 active and core."""
    n = phi.shape
    core = core_flags(phi, h, halfwidth)
    nb = core.shape
    active = np.zeros(nb, dtype=bool)
    for b in np.ndindex(*nb):
        active[b] = any(core[k] for k in neighbourhood(b, n, periodic))
    shell = np.zeros(nb, dtype=bool)
    for a in zip(*np.nonzero(active)):
        for k in neighbourhood(tuple(int(x) for x in a), n, periodic):
            shell[k] = True
    shell &= ~active
    states = np.zeros(nb, dtype=np.uint8)
    states[shell] = 1
    states[active] = 2
    states[active & core] = 3
    return states


def node_mask(states, n):
    """Per node: lies in an active brick."""
    act = states >= 2
    for d in range(len(n)):
        act = np.repeat(act, BRICK[d], axis=d)
    return act[tuple(slice(0, n[d]) for d in range(len(n)))]


def masked_step(O, fo, integrator, terms, tc, dt, active):
    """One band step on the oracle: O.stage for every stage, after which every node outside `active` of phi and of both stage
    buffers is reset to phi^n (the dense step in which those nodes hold phi^n at every stage)."""
    pn = fo.vals.copy(order="F")
    b1, b2 = pn.copy(order="F"), pn.copy(order="F")
    off = ~active
    for s in range(1, O.nstages(integrator) + 1):
        O.stage(fo, integrator, s, b1, b2, terms, tc, dt)
        for a in (fo.vals, b1, b2):
            a[off] = pn[off]
