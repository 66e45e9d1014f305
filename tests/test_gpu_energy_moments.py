"""Energy moments of resident slices (``ocmps_store_energy_moments``, ``SliceStore.energyMoments`` / ``energies``, ``energy``,
``OptimalControl.getEnergyForAllT`` / ``getEnergyVarianceForAllT``): <psi|psi>, <psi|H-c|psi> and <psi|(H-c)^2|psi> of the
Bose-Hubbard Hamiltonian H(U) against exact diagonalisation and the dense MPO contraction of _energy_reference; eigenstates; the slices of a ramp;
agreement between the layers; batch independence, determinism and re-entrancy; the cfg5 size; error paths."""
import ctypes as C
import threading

import numpy as np
import pytest

from _energy_reference import mps_energy_moments as ref_moments
from conftest import golden_state, load_golden, random_symmetric_mps, to_host, to_oracle

pytestmark = pytest.mark.gpu

J = 1.0


def _oc():
    import optimalcontrolmps_b200 as oc
    return oc


def _store(states, cap=None, ctx=None):
    """Slice store holding the oracle MPS `states` (one per slot)."""
    oc = _oc()
    ctx = ctx or oc.Context.default()
    L, D = states[0].L, states[0].D
    cap = cap or max(max(s.bond_dims()) for s in states)
    store = oc.SliceStore(ctx, L, D, cap, len(states))
    m = oc.DeviceMPS(ctx, L, D, cap)
    for z, s in enumerate(states):
        m.upload(to_host(s))
        store.put(z, m)
    return store


def _exact(psi, U, c):
    from oracle import ground_state as og
    L, D = psi.L, psi.D
    H, states = og.bh_hamiltonian_sector(L, D, int(psi.q[-1][0]), J, U)
    v = psi.to_dense().ravel()
    x = v[[np.ravel_multi_index(s, (D,) * L) for s in states]]
    hx = H @ x - c * x
    return np.vdot(x, x).real, np.vdot(x, hx).real, np.vdot(hx, hx).real


def _close(got, ref, tol):
    return abs(got - ref) <= tol * max(abs(ref), 1.0)


def _dmrg(L, d, U, maxm, cutoff, chi_cap=None):
    oc = _oc()
    return oc.InitializeStateDMRG(oc.BoseHubbard(L, d), L, J, U, maxm, cutoff, chi_cap=chi_cap)


# ---- 1. exact values ----
@pytest.mark.parametrize("L", [3, 5, 8])
def test_against_exact_diagonalisation(L):
    from oracle import ground_state as og
    D = 5
    states = [random_symmetric_mps(L, D, L, 16, 100 + L), random_symmetric_mps(L, D, L, 9, 200 + L)]
    states[1].A[L // 2] = 0.6 * states[1].A[L // 2]                         # norm != 1: the moments are raw
    states.append(og.ground_state_ed(L, D, L, J, 7.0))                       # an eigenstate of H(7), measured at other U
    U = np.array([3.7, 50.0, 2.5])
    store = _store(states)
    for shift in (None, np.array([-2.3, 11.0, -4.0])):
        n, h1, h2 = store.energyMoments(J, U, shift=shift)
        n4, g1, g2 = store.energyMoments(J, U, shift=shift, second_moment=False)
        assert np.all(np.isnan(g2))
        for z, s in enumerate(states):
            ref = _exact(s, U[z], 0.0 if shift is None else shift[z])
            assert _close(n[z], ref[0], 1e-12) and _close(h1[z], ref[1], 1e-12) and _close(h2[z], ref[2], 1e-12), (z, n[z], h1[z], h2[z], ref)
            assert _close(n4[z], ref[0], 1e-12) and _close(g1[z], ref[1], 1e-12)


# ---- 2. eigenstates ----
@pytest.mark.parametrize("L,U", [(3, 2.5), (5, 2.5), (5, 50.0)])
def test_exact_eigenstates_have_no_variance(L, U):
    from oracle import ground_state as og
    oc = _oc()
    psi = og.ground_state_ed(L, 5, L, J, U)
    E, var = _store([psi]).energies(J, U, variance=True)
    e_ed = og.mps_energy(psi, J, U)
    assert abs(E[0] - e_ed) <= 1e-12 * abs(e_ed)
    assert abs(var[0]) <= 1e-12 * E[0] ** 2
    dev = oc.DeviceMPS(oc.Context.default(), L, 5, max(psi.bond_dims()))
    dev.upload(to_host(psi))
    e1, v1 = oc.energy(dev, J, U, variance=True)
    assert e1 == E[0] and v1 == var[0]
    assert oc.energy(dev, J, U) == E[0]


def test_dmrg_states():
    oc = _oc()
    psi = _dmrg(8, 4, 2.5, 256, 1e-16)
    E, var = oc.energy(psi, J, 2.5, variance=True)
    print(f"L=8 DMRG cutoff 1e-16: E {E:.15f} var {var:.3e}")
    assert var <= 1e-10 * E * E
    v = {}
    for maxm in (20, 100):
        E, v[maxm] = oc.energy(_dmrg(20, 5, 2.5, maxm, 1e-10, chi_cap=maxm), J, 2.5, variance=True)
        print(f"L=20 U=2.5 maxm {maxm}: E {E:.15f} var {v[maxm]:.3e}")
    assert v[20] > v[100] > 0.0


# ---- 3. the slices of a ramp ----
@pytest.fixture(scope="module")
def cfg1():
    """cfg1 (the reference's README input: L=5, d=4, Nt=201, GRAPE) propagated on the device and by the oracle."""
    oc = _oc()
    from oracle import bh_mps as ob, optimal_control as oo
    z = load_golden("golden_cfg1.npz")
    L, d, Np, J_, cs, ce, T, ts, cutoff, maxm, M, gamma, N = z["params"]
    L, d, N, maxm = int(L), int(d), int(N), int(maxm)
    init, target = golden_state(z, "init"), golden_state(z, "target")
    u = np.array(z["u"])
    st = oc.BH_tDMRG(oc.BoseHubbard(L, d), J_, ts, oc.Args("Cutoff=", cutoff, "Maxm=", maxm))
    g = oc.OptimalControl(to_host(target), to_host(init), st, N, float(gamma))
    ref = oo.OptimalControl(target, init, ob.BHStepper(L, d + 1, J_, ts, ob.TruncArgs(cutoff=cutoff, maxm=maxm)), N=N, gamma=gamma)
    ref.calcPsi(list(u))
    return dict(g=g, st=st, ref=ref, u=u, N=N, L=L, J=float(J_))


def test_ramp_slices_against_oracle(cfg1):
    g, ref, u = cfg1["g"], cfg1["ref"], cfg1["u"]
    E = np.array(g.getEnergyForAllT(list(u), True))
    var = np.array(g.getEnergyVarianceForAllT(list(u), False))
    E2, var2 = g.psi_t.energies(cfg1["J"], u, variance=True)
    assert np.array_equal(E, E2) and np.array_equal(var, var2)
    for i, p in enumerate(ref.psi_t):
        n, h1, _ = ref_moments(p, cfg1["J"], u[i])
        e_ref = h1 / n
        n2, g1, g2 = ref_moments(p, cfg1["J"], u[i], shift=e_ref)
        v_ref = g2 / n2 - (g1 / n2) ** 2
        assert abs(E[i] - e_ref) <= 1e-10 * abs(e_ref), (i, E[i], e_ref)
        assert abs(var[i] - v_ref) <= 1e-8 * e_ref ** 2, (i, var[i], v_ref)
    print(f"E(t=0) {E[0]:.12f}  E(T) {E[-1]:.12f}  max var {var.max():.3e}")


def test_ramp_slices_against_two_point_composition(cfg1):
    g, u, L, J_ = cfg1["g"], cfg1["u"], cfg1["L"], cfg1["J"]
    g.getEnergyForAllT(list(u), True)
    store = g.psi_t
    n, h1, _ = store.energyMoments(J_, u, second_moment=False)
    nn1, nrm = store.expectationValues(("N(N-1)",), return_norm=True)
    for i in range(cfg1["N"]):
        rho = store.correlationMatrix(i, "Adag", "A")
        comp = -J_ * sum(2.0 * rho[j, j + 1].real for j in range(L - 1)) + 0.5 * u[i] * float(np.sum(nn1[i, :, 0]))
        assert abs(h1[i] - comp) <= 1e-11 * abs(comp), (i, h1[i], comp)
        assert abs(n[i] - nrm[i, 0]) <= 1e-13


# ---- 4. the layers agree ----
def test_layers_grape(cfg1):
    g, u, J_ = cfg1["g"], cfg1["u"], cfg1["J"]
    E = g.getEnergyForAllT(list(u), True)
    assert np.array_equal(E, g.psi_t.energies(J_, u))
    dims = g.psi_t.bond_dims().copy()
    # new_control=False: the control passed sets U, the cached psi (propagated under u) is kept
    u2 = u + 1.5
    E2 = g.getEnergyForAllT(list(u2), False)
    assert np.array_equal(g.psi_t.bond_dims(), dims)
    assert np.array_equal(E2, g.psi_t.energies(J_, u2))
    assert not np.array_equal(E2, E)
    V2 = g.getEnergyVarianceForAllT(list(u2), False)
    assert np.array_equal(V2, g.psi_t.energies(J_, u2, variance=True)[1])
    # new_control=True re-propagates under the control passed
    E3 = g.getEnergyForAllT(list(u2), True)
    assert not np.array_equal(g.psi_t.bond_dims(), dims) or not np.array_equal(E3, E2)
    assert np.array_equal(E3, g.psi_t.energies(J_, u2))
    g.getEnergyForAllT(list(u), True)                                        # leave the fixture as it was


def test_layers_group():
    oc = _oc()
    from optimalcontrolmps_b200.states import ground_state
    L, d, ts, N, M = 8, 4, 0.01, 41, 4
    u0 = list(np.linspace(2.5, 50.0, N))
    basis = oc.ControlBasisFactory.buildChoppedSineBasis(u0, ts, (N - 1) * ts, M)
    st = oc.BH_tDMRG(oc.BoseHubbard(L, d), J, ts, oc.Args("Cutoff=", 1e-8, "Maxm=", 60))
    assert st.getJ() == J
    g = oc.OptimalControl(ground_state(L, d, L, 50.0), ground_state(L, d, L, 2.5), st, basis, 1e-6)
    c = list(0.5 * np.sin(np.arange(1, M + 1)))
    E = g.getEnergyForAllT(c, True)
    u = np.array(basis.convertControl(c))
    assert np.array_equal(E, g.psi_t.energies(J, u))
    fid = g.getFidelityForAllT(c, False)                                     # the slices are those getFidelityForAllT sees
    c2 = list(np.array(c) + 0.3)
    E2 = g.getEnergyForAllT(c2, False)                                       # GROUP: new_control=False keeps the cached u too
    assert np.array_equal(E2, E)
    assert g.getFidelityForAllT(c2, False) == fid
    V = g.getEnergyVarianceForAllT(c, True)
    assert np.array_equal(V, g.psi_t.energies(J, u, variance=True)[1])


# ---- 5. batch independence, determinism, re-entrancy ----
@pytest.fixture(scope="module")
def cfg2():
    """The psi slices of bench.py's cfg2 evaluation: L=20 fixtures, seeded GROUP control, 201 slices at chi=100."""
    import bench
    oc = _oc()
    from optimalcontrolmps_b200.states import ground_state
    CFG = bench.CFG
    st = oc.BH_tDMRG(oc.BoseHubbard(CFG["L"], CFG["d"]), CFG["J"], CFG["tstep"], oc.Args("Cutoff=", CFG["cutoff"], "Maxm=", CFG["maxm"]))
    basis, c, u = bench.make_problem_host(0)
    g = oc.OptimalControl(ground_state(CFG["L"], CFG["d"], CFG["Npart"], CFG["U_f"]),
                          ground_state(CFG["L"], CFG["d"], CFG["Npart"], CFG["U_i"]), st, basis, CFG["gamma"])
    g.getFidelityForAllT(list(c), True)
    return dict(g=g, u=np.array(basis.convertControl(list(c), False)), J=CFG["J"])


def test_batch_independence_and_determinism(cfg2):
    store, u, J_ = cfg2["g"].psi_t, cfg2["u"], cfg2["J"]
    nt = store.nslots
    assert nt == 201 and store.chi_cap == 100
    shift = -20.0 + 0.01 * np.arange(nt)
    full = np.stack(store.energyMoments(J_, u, shift=shift))                 # 16 channels: several chunks at chi=100
    for i in range(nt):
        one = np.stack(store.energyMoments(J_, u[i], first=i, count=1, shift=shift[i]))
        assert np.array_equal(one[:, 0], full[:, i]), i
    full4 = np.stack(store.energyMoments(J_, u, shift=shift, second_moment=False))
    for i in (0, 57, 200):
        one = np.stack(store.energyMoments(J_, u[i], first=i, count=1, shift=shift[i], second_moment=False))
        assert np.array_equal(one[:2, 0], full4[:2, i])
    again = np.stack(store.energyMoments(J_, u, shift=shift))
    assert np.array_equal(again, full)
    assert np.max(np.abs(full4[0] - full[0]) / np.abs(full[0])) <= 1e-14
    assert np.max(np.abs(full4[1] - full[1]) / np.abs(full[1])) <= 1e-14
    res = {}

    def run(k, sm):
        res[k] = np.stack(store.energyMoments(J_, u, shift=shift, second_moment=sm))

    ths = [threading.Thread(target=run, args=(0, True)), threading.Thread(target=run, args=(1, False))]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    assert np.array_equal(res[0], full)
    assert np.array_equal(res[1][:2], full4[:2])
    E, var = store.energies(J_, u, variance=True)
    print(f"cfg2: E(0) {E[0]:.10f} E(T) {E[-1]:.10f} var(T) {var[-1]:.4e}")
    assert np.all(var > 0.0)


# ---- 6. the cfg5 size ----
def test_cfg5_ground_state():
    oc = _oc()
    from oracle import ground_state as og
    L, U = 50, 2.5
    psi = _dmrg(L, 5, U, 256, 1e-10)
    assert max(psi.bond_dims()) > 128
    store = oc.SliceStore(psi.ctx, L, 6, psi.chi_cap, 7)                      # 7 copies: 16-channel chunks of 5 at chi=256
    for z in range(7):
        store.put(z, psi)
    E, var = store.energies(J, U, variance=True)
    assert np.all(E == E[0]) and np.all(var == var[0])
    e_ref = og.mps_energy(to_oracle(psi.download()), J, U)
    assert abs(E[0] - e_ref) <= 1e-10 * abs(e_ref)
    e50, v50 = oc.energy(_dmrg(L, 5, U, 50, 1e-10, chi_cap=50), J, U, variance=True)
    print(f"cfg5: E {E[0]:.12f} var {var[0]:.3e}; maxm 50: E {e50:.12f} var {v50:.3e}")
    assert 0.0 <= var[0] < 0.1 * v50


# ---- 7. error paths ----
def test_error_paths():
    oc = _oc()
    ctx = oc.Context.default()
    lib = ctx.lib
    psi = random_symmetric_mps(5, 5, 5, 10, 3)
    store = _store([psi, psi], ctx=ctx)
    pd = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    U = np.array([2.5, 3.0])
    sh = np.array([0.0, 1.0])
    out = np.zeros(6)
    f = lib.ocmps_store_energy_moments
    assert f(None, 0, 2, J, pd(U), None, 1, pd(out)) == -1
    assert f(store.h, 0, 2, J, None, None, 1, pd(out)) == -1
    assert f(store.h, 0, 2, J, pd(U), None, 1, None) == -1
    assert f(store.h, -1, 1, J, pd(U), None, 1, pd(out)) == -1
    assert f(store.h, 1, 2, J, pd(U), None, 1, pd(out)) == -1
    assert f(store.h, 0, 0, J, pd(U), None, 1, pd(out)) == -1
    assert f(store.h, 0, 2, J, pd(U), None, 2, pd(out)) == -1
    assert f(store.h, 0, 2, float("nan"), pd(U), None, 1, pd(out)) == -1
    assert f(store.h, 0, 2, J, pd(np.array([2.5, np.inf])), None, 1, pd(out)) == -1
    assert f(store.h, 0, 2, J, pd(U), pd(np.array([0.0, np.nan])), 1, pd(out)) == -1
    with pytest.raises(oc.OcmpsError):
        store.energyMoments(J, 2.5, first=1, count=5)
    # the next call on the workspace runs clean
    assert f(store.h, 0, 2, J, pd(U), pd(sh), 1, pd(out)) == 0
    for z in range(2):
        ref = ref_moments(psi, J, U[z], shift=sh[z])
        assert all(_close(out[3 * z + k], ref[k], 1e-12) for k in range(3))


# ---- 4b. the C++ layer on the same kind of problem, against the oracle ----
def test_cpp_energy(tmp_path):
    import os
    import struct
    import subprocess
    from conftest import ROOT
    from oracle import bh_mps as ob, optimal_control as oo
    binary = os.path.join(ROOT, "cpp", "tests", "test_energy")
    if not os.path.exists(binary):
        subprocess.run(["make", "-C", os.path.join(ROOT, "cpp")], check=True)
    z = load_golden("golden_L6_maxm.npz")
    L, d, Np, J_, cs, ce, T, ts, cutoff, maxm, M, gamma, N = z["params"]
    L, d, N, maxm = int(L), int(d), int(N), max(int(maxm), 0)                # (-1 in the goldens: no Maxm)
    init, target = golden_state(z, "init"), golden_state(z, "target")
    cap = max([maxm] + init.bond_dims() + target.bond_dims()) if maxm > 0 else min((d + 1) ** (L // 2), 256)
    u = np.array(z["u"], dtype=np.float64)
    ref = oo.OptimalControl(target, init, ob.BHStepper(L, d + 1, J_, ts, ob.TruncArgs(cutoff=cutoff, maxm=maxm or None)), N=N,
                            gamma=gamma)
    ref.calcPsi(list(u))
    E, var = [], []
    for i, p in enumerate(ref.psi_t):
        n, h1, _ = ref_moments(p, J_, u[i])
        n2, g1, g2 = ref_moments(p, J_, u[i], shift=h1 / n)
        E.append(h1 / n)
        var.append(g2 / n2 - (g1 / n2) ** 2)
    n, h1, _ = ref_moments(init, J_, cs)
    n2, g1, g2 = ref_moments(init, J_, cs, shift=h1 / n)

    def w_vec(f, a, dt=np.float64):
        a = np.ascontiguousarray(a, dtype=dt).ravel()
        f.write(struct.pack("<i", a.size))
        f.write(a.tobytes())

    def w_state(f, psi):
        w_vec(f, psi.bond_dims(), np.int32)
        w_vec(f, np.concatenate(psi.q), np.int32)
        w_vec(f, np.concatenate([a.ravel() for a in psi.A]).view(np.float64))

    path = tmp_path / "energy.bin"
    with open(path, "wb") as f:
        f.write(struct.pack("<5i", L, d, N, maxm, int(cap)))
        f.write(struct.pack("<5d", J_, ts, cutoff, gamma, cs))
        w_state(f, init)
        w_state(f, target)
        w_vec(f, u); w_vec(f, E); w_vec(f, var)
        f.write(struct.pack("<2d", h1 / n, g2 / n2 - (g1 / n2) ** 2))
    res = subprocess.run([binary, str(path)], capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
    print(res.stdout)
    print(res.stderr)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "PASSED" in res.stdout
