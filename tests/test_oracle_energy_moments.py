"""The reference energy moments of the tests (``_energy_reference.mps_energy_moments``: the dense W and W x W transfer chains of the
Bose-Hubbard MPO) against the exact sector Hamiltonian applied to the dense state vector."""
import numpy as np
import pytest

from _energy_reference import mps_energy_moments as ref_moments
from conftest import random_symmetric_mps


def _exact(psi, J, U, c):
    from oracle import ground_state as og
    L, D = psi.L, psi.D
    Np = int(psi.q[-1][0])
    H, states = og.bh_hamiltonian_sector(L, D, Np, J, U)
    v = psi.to_dense().ravel()
    x = v[[np.ravel_multi_index(s, (D,) * L) for s in states]]
    hx = H @ x - c * x
    return np.vdot(x, x).real, np.vdot(x, hx).real, np.vdot(hx, hx).real


@pytest.mark.parametrize("L,D,chi,seed", [(2, 4, 4, 1), (3, 5, 6, 2), (5, 5, 12, 3), (6, 5, 12, 7), (6, 6, 20, 11)])
@pytest.mark.parametrize("U,c", [(3.7, 0.0), (3.7, -2.3), (50.0, 12.5)])
def test_against_sector_hamiltonian(L, D, chi, seed, U, c):
    from oracle import ground_state as og
    psi = random_symmetric_mps(L, D, L, chi, seed)
    psi.A[0] = 1.7 * psi.A[0]                                   # a norm other than 1: the moments are raw
    got = ref_moments(psi, 0.9, U, shift=c)
    ref = _exact(psi, 0.9, U, c)
    for g, r in zip(got, ref):
        assert abs(g - r) <= 1e-12 * max(abs(r), 1.0), (got, ref)


def test_energy_matches_mps_energy():
    from oracle import ground_state as og
    psi = random_symmetric_mps(5, 5, 5, 12, 4)
    n, h1, _ = ref_moments(psi, 1.0, 2.5)
    assert abs(h1 / n - og.mps_energy(psi, 1.0, 2.5)) <= 1e-13 * abs(h1 / n)


def test_ground_state_has_zero_variance():
    from oracle import ground_state as og
    U = 4.0
    psi = og.ground_state_ed(4, 5, 4, 1.0, U)
    n, h1, _ = ref_moments(psi, 1.0, U)
    E = h1 / n
    n2, g1, g2 = ref_moments(psi, 1.0, U, shift=E)
    assert abs(g1 / n2) <= 1e-12 * abs(E)
    assert g2 / n2 - (g1 / n2) ** 2 <= 1e-12 * E * E
