"""The narrow-band rules of include/lsm_b200.h on hand-built cases, through the NumPy restatement (no GPU needed)."""
import numpy as np

import helpers as H
import narrow_band_ref as NB


def test_partial_bricks_are_ordinary_bricks():
    n = (70, 40, 20)                            # 3 x 3 x 2 bricks: the last ones 6, 8 and 4 nodes deep
    phi = np.full(n, 5.0)
    phi[69, 39, 19] = 0.0                       # the far corner node, alone in its partial brick
    st = NB.band_states(phi, (1.0, 1.0, 1.0), 1.0, (False,) * 3)
    assert st.shape == (3, 3, 2)
    assert st[2, 2, 1] == 3 and (st == 3).sum() == 1
    assert (st >= 2).sum() == 2 * 2 * 2          # N of the corner brick: {1, 2} on every axis
    assert (st == 1).sum() == 3 * 3 * 2 - 8      # everything else lies in N of an active brick


def test_periodic_wrap_partners_at_513():
    assert NB.axis_neighbours(0, 513, 32, True) == {0, 1, 15}          # nodes n-4..n-2 = 509..511 lie in brick 15
    assert NB.axis_neighbours(16, 513, 32, True) == {15, 16, 0}        # the one-node last brick wraps to brick 0
    assert NB.axis_neighbours(15, 513, 32, True) == {14, 15, 16, 0}    # brick 15 holds nodes n-3, n-2
    assert NB.axis_neighbours(14, 513, 32, True) == {13, 14, 15}
    assert NB.axis_neighbours(0, 513, 16, True) == {0, 1, 31}
    assert NB.axis_neighbours(32, 513, 16, True) == {31, 32, 0}
    assert NB.axis_neighbours(0, 513, 32, False) == {0, 1}
    # a core brick at x = 0: the bricks whose N holds it are active; the last brick (one node) is active, its own wrap partner
    # brick 15 too, and the shell is what their neighbourhoods reach beyond
    phi = np.full((513, 20), 5.0)
    phi[1, 5] = 0.0
    st = NB.band_states(phi, (1.0, 1.0), 1.0, (True, False))
    act = sorted({int(b) for b in np.nonzero(st[:, 0] >= 2)[0]})
    assert act == [0, 1, 15, 16]
    assert sorted(int(b) for b in np.nonzero(st[:, 0] == 1)[0]) == [2, 14]


def test_nan_makes_a_brick_core():
    phi = np.full((64, 32), 5.0)
    phi[40, 20] = np.nan
    st = NB.band_states(phi, (0.1, 0.1), 3.0, (False, False))
    assert st[1, 1] == 3 and (st == 3).sum() == 1


def test_no_node_within_gamma_leaves_every_brick_frozen():
    phi = np.full((64, 48, 20), 1.0)
    phi[3, 3, 3] = 0.31                         # gamma = 3 * 0.1 = 0.3 (the smallest |h| counts)
    st = NB.band_states(phi, (0.2, -0.1, 0.3), 3.0, (False,) * 3)
    assert not st.any()
    phi[3, 3, 3] = 0.3
    assert NB.band_states(phi, (0.2, -0.1, 0.3), 3.0, (False,) * 3)[0, 0, 0] == 3


def test_infinite_halfwidth_masked_step_is_the_dense_step(O):
    """Every brick is core when w is infinite, so the masked oracle integration equals the dense one bit for bit."""
    n = (70, 40)
    for integ in ("FE", "RK2", "RK3"):
        for name, case in H.small_cases(n)[:4]:
            fo, fd = case.oracle_field(), case.oracle_field()
            to, td = case.oracle_terms(), case.oracle_terms()
            dt = 0.5 * O.compute_cfl(fo, to, 0.0)
            tc = 0.0
            for _ in range(3):
                st = NB.band_states(fo.vals, fo.meshsize(), np.inf, [b[0][0] == O.PERIODIC[0] for b in fo.bc])
                assert (st == 3).all()
                NB.masked_step(O, fo, H.INTEG[integ], to, tc, dt, NB.node_mask(st, n))
                O.advance(fd, H.INTEG[integ], td, tc, dt)
                tc += dt
            assert np.array_equal(fo.vals, fd.vals), (integ, name)
