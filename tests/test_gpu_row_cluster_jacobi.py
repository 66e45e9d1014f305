"""The Jacobi stage of the largest register-cached charge blocks (at least 40 rows of R) runs spread over a 4-CTA thread-block
cluster by row blocks (jacobi_rows_cluster_kernel).  At the cfg2 shape (L=20, chi=100) the saturated gate decompositions have
such blocks; these tests check that they take that path and that the headline evaluation still reproduces its golden."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cfg2_eval():
    import bench
    import optimalcontrolmps_b200 as oc
    from conftest import load_golden
    from optimalcontrolmps_b200.states import ground_state
    L, d = bench.CFG["L"], bench.CFG["d"]
    st = oc.BH_tDMRG(oc.BoseHubbard(L, d), bench.CFG["J"], bench.CFG["tstep"], oc.Args("Cutoff=", bench.CFG["cutoff"], "Maxm=", bench.CFG["maxm"]))
    psi_i = ground_state(L, d, bench.CFG["Npart"], bench.CFG["U_i"])
    psi_f = ground_state(L, d, bench.CFG["Npart"], bench.CFG["U_f"])
    basis, c, _ = bench.make_problem_host(0)
    z = load_golden("golden_cfg2_eval.npz")
    assert np.allclose(c, z["c"])
    lib = oc._lib.load()
    counters = (ctypes.c_ulonglong * 2)()

    def single():
        g = oc.OptimalControl(psi_f, psi_i, st, basis, bench.CFG["gamma"])
        g.setThreadCount(2)
        grad = np.array(g.getAnalyticGradient(list(c), True))
        cost = g.getCost(list(c), False)
        return g, cost, grad

    lib.ocmps_debug_row_cluster(counters, 1)
    g1, cost1, grad1 = single()
    lib.ocmps_debug_row_cluster(counters, 0)
    used = (int(counters[0]), int(counters[1]))
    g2, cost2, grad2 = single()
    gb = oc.OptimalControl(psi_f, psi_i, st, basis, bench.CFG["gamma"])
    (cost_b, grad_b), = oc.batch_cost_gradient([gb], [list(c)])
    return dict(z=z, used=used, runs=[(g1, cost1, grad1), (g2, cost2, grad2)], batch=(cost_b, np.array(grad_b)))


def test_large_blocks_take_the_cluster_path(cfg2_eval):
    blocks, sweeps = cfg2_eval["used"]
    assert blocks > 0
    assert 2 * blocks <= sweeps <= 60 * blocks          # Jacobi converges in a handful of sweeps (limit 60)


def test_single_evaluation_matches_golden(cfg2_eval):
    z = cfg2_eval["z"]
    g, cost, grad = cfg2_eval["runs"][0]
    assert abs(cost - float(z["cost"])) / abs(float(z["cost"])) < 1e-9
    assert np.max(np.abs(grad - z["grad"])) / np.max(np.abs(z["grad"])) < 1e-7
    assert np.array_equal(g.psi_t.bond_dims(), z["psi_dims"])
    assert np.array_equal(g.xi_t.bond_dims(), z["xi_dims"])


def test_single_evaluation_is_deterministic(cfg2_eval):
    (g1, c1, d1), (g2, c2, d2) = cfg2_eval["runs"]
    assert c1 == c2
    assert np.array_equal(d1, d2)
    assert np.array_equal(g1.psi_t.bond_dims(), g2.psi_t.bond_dims())


def test_single_evaluation_agrees_with_batched(cfg2_eval):
    _, cost, grad = cfg2_eval["runs"][0]
    cost_b, grad_b = cfg2_eval["batch"]
    assert abs(cost - cost_b) / abs(cost_b) < 1e-12
    assert np.max(np.abs(grad - grad_b)) / np.max(np.abs(grad_b)) < 1e-11
