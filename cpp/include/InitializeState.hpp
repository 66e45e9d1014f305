// Bose-Hubbard ground states for psi_init / psi_target: the two overloads of the reference's include/InitializeState.hpp:18-117.
// The reference sets up the Hamiltonian as an AutoMPO and runs ITensor's DMRG (10 sweeps, maxm 10,20,50,100,200 or
// 10,20,50,maxBondDim, cutoff 1e-9 or `threshold`); here the device engine's Trotter-step kernels run in imaginary time from the
// same product state with the same bond-dimension schedule (ocmps_ground_state).  Energies agree with DMRG to ~1e-6 relative,
// fidelities to ~1e-6 (tools/gpu_ground_state.py).  `silent` is accepted for source compatibility (nothing is printed).
#ifndef OCMPS_INITIALIZESTATE_HPP
#define OCMPS_INITIALIZESTATE_HPP
#include <algorithm>
#include "itensor/all.h"

namespace itensor {

inline IQMPS InitializeState(const SiteSet& sites, const int Npart, const double J, const double U, const int maxBondDim,
                             const double threshold, bool silent = true) {
  (void)silent;
  const int L = sites.N(), D = sites.D();
  long long full = 1;
  for (int i = 0; i < L / 2 && full < 4096; ++i) full *= D;
  const int cap = (int)std::min<long long>(maxBondDim, full);
  IQMPS psi(L, D, cap);
  ocmps_check(ocmps_ground_state(default_context(), L, D, Npart, J, U, cap, threshold, 0.0, psi.handle(), nullptr, nullptr), "ocmps_ground_state");
  return psi;
}

inline IQMPS InitializeState(const SiteSet& sites, const int Npart, const double J, const double U, bool silent = true) {
  return InitializeState(sites, Npart, J, U, 200, 1E-9, silent);          // :52-54
}

// The same ground state by two-site DMRG on the device, the algorithm of the reference (10 sweeps, maxm 10, 20, 50, maxBondDim,
// cutoff `threshold`; no noise term): ocmps_ground_state_dmrg.
inline IQMPS InitializeStateDMRG(const SiteSet& sites, const int Npart, const double J, const double U, const int maxBondDim,
                                 const double threshold, bool silent = true) {
  (void)silent;
  const int L = sites.N(), D = sites.D();
  long long full = 1;
  for (int i = 0; i < L / 2 && full < 4096; ++i) full *= D;
  const int cap = (int)std::min<long long>(maxBondDim, full);
  IQMPS psi(L, D, cap);
  ocmps_check(ocmps_ground_state_dmrg(default_context(), L, D, Npart, J, U, cap, threshold, 10, psi.handle(), nullptr, nullptr),
              "ocmps_ground_state_dmrg");
  return psi;
}

inline IQMPS InitializeStateDMRG(const SiteSet& sites, const int Npart, const double J, const double U, bool silent = true) {
  return InitializeStateDMRG(sites, Npart, J, U, 200, 1E-9, silent);
}

}  // namespace itensor
#endif
