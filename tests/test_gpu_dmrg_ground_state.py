"""Two-site DMRG ground states on the device (``ocmps_ground_state_dmrg`` / ``InitializeStateDMRG``, the algorithm of the reference's
include/InitializeState.hpp:18-117): against exact diagonalisation, the oracle's DMRG, the shipped fixtures and the imaginary-time
generator; the returned energy against two independent evaluations; the cfg5 chain; determinism, re-entrancy, error paths, and a
GROUP cost + gradient started from the DMRG states."""
import threading

import numpy as np
import pytest

from conftest import to_host, to_oracle

pytestmark = pytest.mark.gpu

J = 1.0


def _oc():
    import optimalcontrolmps_b200 as oc
    return oc


def _dmrg(L, d, Np, U, maxm, cutoff, nsweeps=10, chi_cap=None, ctx=None):
    oc = _oc()
    return oc.InitializeStateDMRG(oc.BoseHubbard(L, d), Np, J, U, maxm, cutoff, nsweeps=nsweeps, ctx=ctx, chi_cap=chi_cap,
                                  return_info=True)


def _check_state(psi, Np):
    got = to_oracle(psi.download())
    assert got.check_charges() == 0.0 and int(got.q[-1][0]) == Np
    assert abs(psi.norm() - 1.0) < 1e-12
    return got


def _device_energy(psi, U):
    """-J sum 2 Re<a+_i a_i+1> + U/2 sum <n_i(n_i-1)> from the device's two-point functions and site expectations."""
    oc = _oc()
    store = oc.SliceStore(psi.ctx, psi.L, psi.D, psi.chi_cap, 1)
    store.put(0, psi)
    rho = store.correlationMatrix(0, "Adag", "A")
    nn1 = store.expectationValues(("N(N-1)",))[0, :, 0]
    hop = sum(2.0 * rho[i, i + 1].real for i in range(psi.L - 1))
    return -J * hop + 0.5 * U * float(np.sum(nn1))


@pytest.mark.parametrize("L,U", [(L, U) for L in (2, 3, 5, 8) for U in (2.5, 50.0)])
def test_against_exact_diagonalisation(L, U):
    """Nothing of weight is truncated: cutoff 1e-16 (ITensor's smallest).  A cutoff of 1e-12 is not enough for that -- on the
    Mott side (U=50) the Schmidt weights just above 1e-12 carry 1e-10 of the energy (5.8e-10 relative at L=5), in the oracle's
    DMRG exactly as here; test_against_oracle_dmrg pins that case against the oracle."""
    from oracle import bh_mps as ob, ground_state as og
    d = 4
    ed = og.ground_state_ed(L, d + 1, L, J, U)
    e_ed = og.mps_energy(ed, J, U)
    psi, e, sweeps = _dmrg(L, d, L, U, 256, 1e-16)
    print(f"L={L} U={U}: E_ED {e_ed:.15f} sweeps {[f'{x:.15f}' for x in sweeps]}")
    got = _check_state(psi, L)
    assert abs(e - e_ed) <= 1e-11 * abs(e_ed)
    assert 1.0 - abs(ob.overlap(ed, got)) ** 2 <= 1e-10


@pytest.mark.parametrize("L,U,maxm,cutoff", [(8, 2.5, 40, 1e-9), (8, 50.0, 40, 1e-9), (5, 50.0, 256, 1e-12), (8, 50.0, 256, 1e-12)])
def test_against_oracle_dmrg(L, U, maxm, cutoff):
    from oracle import ground_state as og
    d = 4
    ref = og.ground_state_dmrg(L, d + 1, L, J, U, maxm_schedule=tuple(min(m, maxm) for m in (10, 20, 50, maxm)), cutoff=cutoff,
                               nsweeps=10)
    psi, e, sweeps = _dmrg(L, d, L, U, maxm, cutoff)
    # the oracle's .energy is its last Ritz value, taken before the final truncation; the device returns both that value (the
    # last sweep energy) and <psi|H|psi> of the truncated state it hands back (5.7e-8 apart at U=50, cutoff 1e-9)
    assert abs(sweeps[-1] - ref.energy) <= 1e-10 * abs(ref.energy)
    e_ref = og.mps_energy(ref, J, U)
    assert abs(e - e_ref) <= 1e-10 * abs(e_ref)
    assert psi.bond_dims() == ref.bond_dims()


@pytest.fixture(scope="module")
def cfg2_states():
    from optimalcontrolmps_b200.states import DATA_DIR
    import os
    out = {}
    for U in (2.5, 50.0):
        psi, e, sweeps = _dmrg(20, 5, 20, U, 100, 1e-8)
        meta = np.load(os.path.join(DATA_DIR, f"bh_L20_d5_N20_U{U:g}.npz"))["meta"]
        out[U] = (psi, e, sweeps, float(meta[7]))
    return out


@pytest.mark.parametrize("U", [2.5, 50.0])
def test_against_cfg2_fixture_and_tebd(cfg2_states, U):
    oc = _oc()
    from optimalcontrolmps_b200.states import ground_state
    from oracle import bh_mps as ob
    psi, e, sweeps, e_fix = cfg2_states[U]
    print(f"U={U}: E {e:.15f} fixture {e_fix:.15f} sweeps {[f'{x:.15f}' for x in sweeps]} dims {psi.bond_dims()}")
    got = _check_state(psi, 20)
    assert abs(e - e_fix) <= 1e-8 * abs(e)
    assert 1.0 - abs(ob.overlap(to_oracle(ground_state(20, 5, 20, U)), got)) ** 2 <= 1e-6
    _, e_tebd, _ = oc.InitializeState(oc.BoseHubbard(20, 5), 20, J, U, 100, 1e-8, return_info=True)
    assert e < e_tebd


@pytest.mark.parametrize("U", [2.5, 50.0])
def test_energy_is_the_energy_of_the_returned_state(cfg2_states, U):
    from oracle import ground_state as og
    psi, e, _, _ = cfg2_states[U]
    assert abs(og.mps_energy(to_oracle(psi.download()), J, U) - e) <= 1e-10 * abs(e)
    assert abs(_device_energy(psi, U) - e) <= 1e-10 * abs(e)


def test_cfg5_chain():
    from oracle import ground_state as og
    L, d, U = 50, 5, 2.5
    psi, e, sweeps = _dmrg(L, d, L, U, 256, 1e-10)
    print(f"cfg5: E {e:.15f} sweeps {[f'{x:.15f}' for x in sweeps]} dims {psi.bond_dims()}")
    assert max(psi.bond_dims()) > 112                        # the bulk decompositions take the cluster kernels
    _check_state(psi, L)
    assert abs(og.mps_energy(to_oracle(psi.download()), J, U) - e) <= 1e-10 * abs(e)
    assert abs(_device_energy(psi, U) - e) <= 1e-10 * abs(e)
    tail = sweeps[3:]                                        # from the sweep that reaches maxm on
    assert np.all(np.diff(tail) <= 1e-10 * abs(e))


def _flat(h):
    return np.concatenate([a.ravel() for a in h.A])


def test_bit_identical_and_reentrant():
    oc = _oc()
    ctx = oc.Context.default()
    a1, e1, s1 = _dmrg(20, 5, 20, 2.5, 100, 1e-8, ctx=ctx)
    a2, e2, s2 = _dmrg(20, 5, 20, 2.5, 100, 1e-8, ctx=ctx)
    b1, f1, _ = _dmrg(20, 5, 20, 50.0, 100, 1e-8, ctx=ctx)
    h1, h2 = a1.download(), a2.download()
    assert e1 == e2 and np.array_equal(s1, s2) and h1.bond_dims() == h2.bond_dims()
    assert np.array_equal(_flat(h1), _flat(h2))
    par = {}

    def run(U):
        par[U] = _dmrg(20, 5, 20, U, 100, 1e-8, ctx=ctx)

    ths = [threading.Thread(target=run, args=(U,)) for U in (2.5, 50.0)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    for U, (ref, eref) in ((2.5, (h1, e1)), (50.0, (b1.download(), f1))):
        got = par[U][0].download()
        assert par[U][1] == eref and got.bond_dims() == ref.bond_dims()
        assert np.array_equal(_flat(got), _flat(ref))


def test_usable_as_input_of_a_group_evaluation(cfg2_states):
    oc = _oc()
    from oracle import bh_mps as ob, optimal_control as oo
    L, d, ts, cutoff, maxm, gamma, N, M = 20, 5, 0.01, 1e-8, 100, 1e-6, 20, 4
    psi_i = to_oracle(cfg2_states[2.5][0].download())
    psi_f = to_oracle(cfg2_states[50.0][0].download())
    u0 = list(np.linspace(2.5, 50.0, N))
    T = (N - 1) * ts
    basis = oc.ControlBasisFactory.buildChoppedSineBasis(u0, ts, T, M)
    c = list(0.5 * np.sin(np.arange(1, M + 1)))
    st = oc.BH_tDMRG(oc.BoseHubbard(L, d), J, ts, oc.Args("Cutoff=", cutoff, "Maxm=", maxm))
    g = oc.OptimalControl(to_host(psi_f), to_host(psi_i), st, basis, gamma)
    grad = np.array(g.getAnalyticGradient(c, True))
    cost = g.getCost(c, False)
    ref_basis = oo.ControlBasis(list(basis._u0), list(basis._S), basis._f.tolist())
    ref = oo.OptimalControl(psi_f, psi_i, ob.BHStepper(L, d + 1, J, ts, ob.TruncArgs(cutoff=cutoff, maxm=maxm)), basis=ref_basis,
                            gamma=gamma)
    grad_ref = np.array(ref.getAnalyticGradient(c, True))
    cost_ref = ref.getCost(c, False)
    assert abs(cost - cost_ref) / abs(cost_ref) < 1e-9
    assert np.max(np.abs(grad - grad_ref)) / np.max(np.abs(grad_ref)) < 1e-7
    assert np.array_equal(g.psi_t.bond_dims(), np.array([p.bond_dims() for p in ref.psi_t]))


def test_error_paths_leave_no_stale_status():
    oc = _oc()
    ctx = oc.Context.default()
    lib = ctx.lib
    L, D = 6, 5
    out = oc.DeviceMPS(ctx, L, D, 20)
    e = np.zeros(1)
    sw = np.zeros(4)
    pd = lambda a: a.ctypes.data_as(__import__("ctypes").POINTER(__import__("ctypes").c_double))
    assert lib.ocmps_ground_state_dmrg(ctx.h, L, D, L, J, 2.5, 21, 1e-9, 4, out.h, pd(e), pd(sw)) == -3     # CAPACITY
    assert lib.ocmps_ground_state_dmrg(ctx.h, L, D, L + 1, J, 2.5, 20, 1e-9, 4, out.h, pd(e), pd(sw)) == -1  # INVALID
    assert lib.ocmps_ground_state_dmrg(ctx.h, L + 1, D, L, J, 2.5, 20, 1e-9, 4, out.h, pd(e), pd(sw)) == -1  # shape
    assert lib.ocmps_ground_state_dmrg(ctx.h, L, D - 1, L, J, 2.5, 20, 1e-9, 4, out.h, pd(e), pd(sw)) == -1  # shape
    assert lib.ocmps_ground_state_dmrg(ctx.h, L, D, L, J, 2.5, 20, 1e-9, 0, out.h, pd(e), pd(sw)) == -1     # nsweeps
    # the next call on the same workspace runs clean
    assert lib.ocmps_ground_state_dmrg(ctx.h, L, D, L, J, 2.5, 20, 1e-9, 4, out.h, pd(e), pd(sw)) == 0
    from oracle import ground_state as og
    assert abs(og.mps_energy(to_oracle(out.download()), J, 2.5) - e[0]) <= 1e-10 * abs(e[0])
