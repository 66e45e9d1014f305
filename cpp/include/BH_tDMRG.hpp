// tDMRG propagator of the Bose-Hubbard model on the GPU; public interface of the reference's
// include/BH_tDMRG.hpp:16-40.  prop = exp(-i H_U(to) dt/2) exp(-i H_J dt) exp(-i H_U(from) dt/2).
#ifndef OCMPS_BH_TDMRG_HPP
#define OCMPS_BH_TDMRG_HPP
#include <memory>
#include "itensor/all.h"

using namespace itensor;

class BH_tDMRG {
  struct Holder { ocmps_stepper* h = nullptr; ~Holder() { if (h) ocmps_stepper_destroy(h); } };
  std::shared_ptr<Holder> p_;          // copies of a stepper share the immutable device gates (step is const / re-entrant)
  SiteSet sites_;
  Args args_;
  double J_ = 1.0, tstep_ = 0.0;
  int cap_ = 0;
 public:
  BH_tDMRG() {}
  // chi_cap: allocated bond capacity; defaults to Maxm (or min(D^(L/2), 256) when Maxm is not given)
  BH_tDMRG(const SiteSet& sites, const double J, const double tstep, const Args& args, int chi_cap = 0);
  void setTstep(const double tstep_);
  void step(IQMPS& psi, const double from, const double to, bool propagateForward = true) const;
  IQMPO propagatorDeriv(const double& control_n) const;
  double getTstep() const;
  Args getArgs() const;
  double getJ() const { return J_; }
  // GPU-side accessors used by OptimalControl
  ocmps_stepper* handle() const { return p_ ? p_->h : nullptr; }
  int capacity() const { return cap_; }
  const SiteSet& sites() const { return sites_; }
};
#endif
