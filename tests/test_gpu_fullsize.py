"""GPU tests at BASELINE.json's full cfg2 shape (L=20, D=6, chi=100) through size-independent properties:
norm preservation, charge conservation, forward/backward consistency of divT, bond dimensions capped at
Maxm, and agreement with the oracle on a short horizon that the oracle finishes in seconds."""
import numpy as np
import pytest

from conftest import to_host, to_oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cfg2():
    import optimalcontrolmps_b200 as oc
    from optimalcontrolmps_b200.states import ground_state
    L, d = 20, 5
    st = oc.BH_tDMRG(oc.BoseHubbard(L, d), 1.0, 1e-2, oc.Args("Cutoff=", 1e-8, "Maxm=", 100))
    return oc, st, ground_state(L, d, 20, 2.5), ground_state(L, d, 20, 50.0)


def test_short_horizon_matches_oracle(cfg2):
    oc, st, psi_i, psi_f = cfg2
    from oracle import bh_mps as ob, optimal_control as oo
    N = 6
    u = list(np.linspace(2.5, 12.0, N))
    so = ob.BHStepper(20, 6, 1.0, 1e-2, ob.TruncArgs(cutoff=1e-8, maxm=100))
    o = oo.OptimalControl(to_oracle(psi_f), to_oracle(psi_i), so, N=N, gamma=1e-6)
    g = oc.OptimalControl(psi_f, psi_i, st, N, 1e-6)
    g.setThreadCount(2)
    co, cg = o.getCost(u), g.getCost(u)
    assert abs(co - cg) / abs(co) < 1e-9
    go, gg = np.array(o.getAnalyticGradient(u)), np.array(g.getAnalyticGradient(u))
    assert np.max(np.abs(go - gg)) / np.max(np.abs(go)) < 1e-7
    assert np.array_equal(g.psi_t.bond_dims(), np.array([p.bond_dims() for p in o.psi_t]))
    assert np.array_equal(g.xi_t.bond_dims(), np.array([p.bond_dims() for p in o.xi_t]))


def test_fast_ramp_properties(cfg2):
    """A steep ramp saturates chi=100 within ~60 steps; check invariants on the saturated states."""
    oc, st, psi_i, psi_f = cfg2
    from oracle import bh_mps as ob
    N = 64
    u = list(np.linspace(2.5, 50.0, N))
    g = oc.OptimalControl(psi_f, psi_i, st, N, 1e-6)
    g.setThreadCount(2)
    grad = np.array(g.getAnalyticGradient(u))
    cost = g.getCost(u, False)
    assert np.all(np.isfinite(grad)) and np.isfinite(cost) and 0.0 <= cost <= 0.6
    dims = g.psi_t.bond_dims()
    assert dims.max() == 100                                    # Maxm binds
    assert np.all(dims <= 100) and np.all(dims[:, 0] == 1) and np.all(dims[:, -1] == 1)
    last = g.psi_t.get(N - 1)
    assert abs(last.norm() - 1.0) < 1e-12                       # normalised after every step (src/BH_tDMRG.cpp:228)
    assert abs(oc.overlapC(last, last) - 1.0) < 1e-10           # canonical form: <psi|psi> = |centre|^2
    h = to_oracle(last.download())
    assert h.check_charges() == 0.0                             # boson number conserved exactly
    assert int(h.q[-1][0]) == 20
    fid = np.array(g.getFidelityForAllT(u, False))
    assert np.all(fid >= -1e-12) and np.all(fid <= 1 + 1e-12)
    assert abs(0.5 * (1 - fid[-1]) + g._calcRegularization(u) - cost) < 1e-12
    # one more step of the saturated state agrees with the oracle (identical truncation decisions at chi=100)
    so = ob.BHStepper(20, 6, 1.0, 1e-2, ob.TruncArgs(cutoff=1e-8, maxm=100))
    po = h.copy()
    so.step(po, 30.0, 31.0, True)
    st.step(last, 30.0, 31.0, True)
    got = to_oracle(last.download())
    assert got.bond_dims() == po.bond_dims()
    assert abs(abs(ob.overlap(po, got)) - 1.0) < 1e-10


def test_large_blocks_beyond_shared_memory():
    """Bond dimension 160 (> 128): charge blocks that do not fit the 200 KB shared-memory tile take the global-memory
    variant of the block kernel, rows longer than 128 take the non-cached rotation path.  A random number-conserving
    MPS has flat spectra, so Maxm binds at every bond and every block is large."""
    import optimalcontrolmps_b200 as oc
    from oracle import bh_mps as ob
    from conftest import random_symmetric_mps
    L, d, Np, chi = 10, 5, 10, 160
    psi = random_symmetric_mps(L, d + 1, Np, chi, seed=5)
    assert max(psi.bond_dims()) > 128
    so = ob.BHStepper(L, d + 1, 1.0, 1e-2, ob.TruncArgs(cutoff=1e-10, maxm=chi))
    st = oc.BH_tDMRG(oc.BoseHubbard(L, d), 1.0, 1e-2, oc.Args("Cutoff=", 1e-10, "Maxm=", chi))
    dev = st.to_device(to_host(psi))
    po = psi.copy()
    for k in range(2):
        so.step(po, 3.0 + k, 4.0 + k, True)
        st.step(dev, 3.0 + k, 4.0 + k, True)
        got = to_oracle(dev.download())
        assert got.bond_dims() == po.bond_dims()
        assert abs(abs(ob.overlap(po, got)) - 1.0) < 1e-10
        assert got.check_charges() == 0.0
    # K|psi> needs bonds of 2*chi = 320 inside: also through the global-memory variant
    kg = to_oracle(st.exactApplyMPO(dev).download())
    ko = ob.apply_K(po, ob.TruncArgs(cutoff=1e-10, maxm=chi))
    assert kg.bond_dims() == ko.bond_dims()
    assert abs(kg.norm() - ko.norm()) < 1e-9 * ko.norm()
    assert abs(abs(ob.overlap(ko, kg)) / (ko.norm() * kg.norm()) - 1.0) < 1e-9


def test_cfg2_full_evaluation_matches_golden(cfg2):
    """The complete headline workload (400 Trotter steps at chi=100, Nt=201 MPO overlaps, GROUP M=10) against the oracle's
    golden evaluation (tests/golden/make_golden_cfg2.py): cost 1e-9, gradient 1e-7, identical bond dimensions of every slice."""
    import os
    from conftest import GOLDEN
    path = os.path.join(GOLDEN, "golden_cfg2_eval.npz")
    if not os.path.exists(path):
        pytest.skip("golden_cfg2_eval.npz not generated")
    import bench
    oc, st, psi_i, psi_f = cfg2
    z = np.load(path)
    basis, c, u = bench.make_problem_host(0)
    assert np.allclose(c, z["c"]) and np.allclose(u, z["u"])
    g = oc.OptimalControl(psi_f, psi_i, st, basis, bench.CFG["gamma"])
    g.setThreadCount(2)
    grad = np.array(g.getAnalyticGradient(list(c), True))
    cost = g.getCost(list(c), False)
    assert abs(cost - float(z["cost"])) / abs(float(z["cost"])) < 1e-9
    assert np.max(np.abs(grad - z["grad"])) / np.max(np.abs(z["grad"])) < 1e-7
    fid = np.array(g.getFidelityForAllT(list(c), False))
    assert np.max(np.abs(fid - z["fidelities"])) < 1e-9
    assert np.max(np.abs(g.divT - z["divT"])) / np.max(np.abs(z["divT"])) < 1e-7
    assert np.array_equal(g.psi_t.bond_dims(), z["psi_dims"])
    assert np.array_equal(g.xi_t.bond_dims(), z["xi_dims"])


def test_bench_dump_outputs_match_golden(tmp_path):
    """bench.py --dump-outputs writes what its last timed evaluation computed.  At the default seed that is the evaluation of
    golden_cfg2_eval.npz: cost and fidelities 1e-9, gradient and divT 1e-7, every bond dimension, and the cost of the JSON line."""
    import json
    import os
    import subprocess
    import sys
    from conftest import ROOT, load_golden
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--batch", "1", "--hessian-nt", "0",
           "--cfg1", "0", "--cfg5", "0", "--cfg4-seeds", "0", "--no-cpu-baseline", "--dump-outputs", str(out)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["steps"] == 1
    d = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert sorted(d) == ["cost", "divT", "fidelities", "gradient", "psi_bond_dims", "xi_bond_dims"]
    assert all(a.dtype == np.float64 for a in d.values())
    z = load_golden("golden_cfg2_eval.npz")
    assert d["cost"][0] == line["result"]["cost"]
    assert abs(d["cost"][0] - float(z["cost"])) / abs(float(z["cost"])) < 1e-9
    assert np.max(np.abs(d["gradient"] - z["grad"])) / np.max(np.abs(z["grad"])) < 1e-7
    divT = d["divT"][:, 0] + 1j * d["divT"][:, 1]
    assert np.max(np.abs(divT - z["divT"])) / np.max(np.abs(z["divT"])) < 1e-7
    assert np.max(np.abs(d["fidelities"] - z["fidelities"])) < 1e-9
    assert np.array_equal(d["psi_bond_dims"], z["psi_dims"])
    assert np.array_equal(d["xi_bond_dims"], z["xi_dims"])


@pytest.mark.parametrize("L,Np,chi,cutoff", [(30, 30, 150, 1e-8), (50, 50, 256, 1e-10)])
def test_cfg4_cfg5_shapes_one_step(L, Np, chi, cutoff):
    """BASELINE.json configs[3] (L=30, chi=150) and configs[4] (L=50, chi=256, Cutoff 1e-10) at their full shapes: one forward
    and one backward Trotter step of a random number-conserving MPS (every bond saturated) against the oracle."""
    import optimalcontrolmps_b200 as oc
    from oracle import bh_mps as ob
    from conftest import random_symmetric_mps
    d = 5
    psi = random_symmetric_mps(L, d + 1, Np, chi, seed=L)
    assert max(psi.bond_dims()) == chi
    so = ob.BHStepper(L, d + 1, 1.0, 1e-2, ob.TruncArgs(cutoff=cutoff, maxm=chi))
    st = oc.BH_tDMRG(oc.BoseHubbard(L, d), 1.0, 1e-2, oc.Args("Cutoff=", cutoff, "Maxm=", chi))
    dev = st.to_device(to_host(psi))
    po = psi.copy()
    for (a, b, fwd) in [(3.0, 4.0, True), (4.0, 3.5, False)]:
        so.step(po, a, b, fwd)
        st.step(dev, a, b, fwd)
        got = to_oracle(dev.download())
        assert got.bond_dims() == po.bond_dims()
        assert abs(abs(ob.overlap(po, got)) - 1.0) < 1e-9
        assert abs(dev.norm() - 1.0) < 1e-12
    assert got.check_charges() == 0.0
