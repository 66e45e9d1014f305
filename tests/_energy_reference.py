"""Reference energy moments for the tests: the dense W and W x W transfer chains of the Bose-Hubbard MPO on the oracle's MPS
containers (NumPy only; the device computes the same chains in ``ocmps_store_energy_moments``)."""
import numpy as np


def mps_energy_moments(psi, J, U, shift=0.0):
    """Raw moments (<psi|psi>, <psi|H-c|psi>, <psi|(H-c)^2|psi>) of H(U) - c, c = shift.  W is the bond-dimension-4 MPO of
    ``oracle.ground_state._bh_mpo`` (states 3 = nothing placed yet, 1 / 2 = a / adag placed, 0 = done) with the on-site entry
    W[3,0] = K - (c/L) I; the 16 channels (a,b) of W x W apply W[a,a'] W[b,b'].  Any gauge; nothing is divided by the norm."""
    from oracle.bh_mps import boson_ops
    L, D = psi.L, psi.D
    op = boson_ops(D)
    I, A, Ad, K = op["Id"], op["A"], op["Adag"], 0.5 * U * op["N(N-1)"]
    W = np.zeros((4, 4, D, D))
    W[0, 0] = I
    W[3, 3] = I
    W[3, 0] = K - (shift / L) * I
    W[3, 1] = -J * A
    W[3, 2] = -J * Ad
    W[1, 0] = Ad
    W[2, 0] = A
    W2 = np.einsum("abts,cdsu->acbdtu", W, W).reshape(16, 16, D, D)
    E = np.zeros((16, 1, 1), dtype=complex)
    E[15] = 1.0
    for a in psi.A:
        T = np.einsum("wxl,lsr->wxsr", E, a)               # E_w . B
        Tp = np.einsum("wvts,wxsr->vxtr", W2, T)           # channel mixing on the physical index
        E = np.einsum("xtR,vxtr->vRr", a.conj(), Tp)       # A^H . T'
    return E[15, 0, 0].real, E[3, 0, 0].real, E[0, 0, 0].real
