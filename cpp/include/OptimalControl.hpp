// OptimalControl<TimeStepper>: cost / gradient / Hessian of the state-transfer fidelity with the reference's
// public interface (include/OptimalControl.hpp:52-75) and new_control caching semantics.  psi_t, xi_t and
// xiHlist are slice stores resident in HBM instead of host vectors of IQMPS.
#ifndef OCMPS_OPTIMALCONTROL_HPP
#define OCMPS_OPTIMALCONTROL_HPP
#include <complex>
#include <memory>
#include <vector>
#include "itensor/all.h"
#include "ControlBasis.hpp"

using namespace itensor;
using stdvec = std::vector<double>;
using rowmat = std::vector<std::vector<double>>;

template <class TimeStepper>
class OptimalControl {
  struct Store { ocmps_store* h = nullptr; ~Store() { if (h) ocmps_store_destroy(h); } };
  TimeStepper timeStepper;
  ControlBasis basis;
  double gamma, tstep;
  size_t N, M, threadCount;
  IQMPS psi_target, psi_init;
  std::shared_ptr<Store> psi_t, xi_t, xiHlist;
  std::vector<Cplx> divT, fidOvl;
  bool GRAPE, BFGS, calculatedXi;

  void init(IQMPS& target, IQMPS& init);
  std::shared_ptr<Store> newStore() const;
  void calcPsi(const stdvec& control);
  void calcXi(const stdvec& control);
  void calcDivT(const stdvec& control);
  void calcPsiXiDivT(const stdvec& control);
  Cplx overlapFactor();
  double calcCost(const stdvec& control, const bool new_control = true);
  double calcRegularization(const stdvec& control) const;
  stdvec calcRegularizationGrad(const stdvec& control) const;
  rowmat calcRegularizationHessian(const stdvec& control) const;
  stdvec calcFidelityGrad(const stdvec& control, const bool new_control = true);
  stdvec calcAnalyticGradient(const stdvec& control, const bool new_control = true);
  rowmat calcHessian(const stdvec& control, const bool new_control = true);
  stdvec calcFidelityForAllT(const stdvec& control, const bool new_control = true);
  void calcEnergyForAllT(const stdvec& control, const bool new_control, bool variance, stdvec& E, stdvec& var);

 public:
  // psi_t / xi_t / xiHlist live in device stores owned by this object; a copy would have to duplicate gigabytes of
  // slices to keep the reference's value semantics (every copy of the reference's class is deep), so copies are
  // disabled instead of silently aliasing the caches of two objects.  Moves are fine.
  OptimalControl(const OptimalControl&) = delete;
  OptimalControl& operator=(const OptimalControl&) = delete;
  OptimalControl(OptimalControl&&) = default;
  // GRAPE constructor
  OptimalControl(IQMPS& psi_target, IQMPS& psi_init, TimeStepper& timeStepper, size_t N, double gamma, bool BFGS = false);
  // GROUP constructor
  OptimalControl(IQMPS& psi_target, IQMPS& psi_init, TimeStepper& timeStepper, ControlBasis& basis, double gamma, bool BFGS = false);

  std::vector<IQMPS> getPsit() const;
  size_t getM() const;
  size_t getN() const;
  stdvec getControl(const stdvec& control);
  stdvec getTimeAxis() const;
  void setGamma(double newgamma);
  void setThreadCount(const size_t newThreadCount);
  void setGRAPE(const bool useGRAPE);
  void setBFGS(const bool useBFGS);
  bool useBFGS() const;

  void propagatePsi(const stdvec& control);
  double getCost(const stdvec& control, const bool new_control = true);
  stdvec getAnalyticGradient(const stdvec& control, const bool new_control = true);
  rowmat getHessian(const stdvec& control, const bool new_control = true);
  stdvec getFidelityForAllT(const stdvec& control, const bool new_control = true);
  // <psi_i|H(u_i)|psi_i> / <psi_i|psi_i> on the psi slices (the excess energy along the ramp) and its variance <H^2> - <H>^2;
  // J from the stepper, caching as getFidelityForAllT (new_control = false keeps the slices, the control only sets u_i)
  stdvec getEnergyForAllT(const stdvec& control, const bool new_control = true);
  stdvec getEnergyVarianceForAllT(const stdvec& control, const bool new_control = true);
  rowmat getControlJacobian() const;
};
#endif
