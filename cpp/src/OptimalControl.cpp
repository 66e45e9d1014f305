// OptimalControl<TimeStepper> on resident slice stores.  State machine, formulas and call order follow the
// reference's src/OptimalControl.cpp (line numbers cited per method); every MPS operation is a libocmps call.
#include "OptimalControl.hpp"
#include "BH_tDMRG.hpp"

#include <algorithm>
#include <cmath>
#include <stdexcept>

template <class TS>
std::shared_ptr<typename OptimalControl<TS>::Store> OptimalControl<TS>::newStore() const {
  auto s = std::make_shared<Store>();
  const SiteSet& sites = timeStepper.sites();
  ocmps_check(ocmps_store_create(default_context(), sites.N(), sites.D(), timeStepper.capacity(), (int)N, &s->h), "ocmps_store_create");
  return s;
}

template <class TS>
void OptimalControl<TS>::init(IQMPS& target, IQMPS& init) {
  calculatedXi = false;
  threadCount = 1;
  psi_target = target.withCapacity(timeStepper.capacity());      // both states are copied into the object (:20-24)
  psi_init = init.withCapacity(timeStepper.capacity());
  psi_t = newStore();
  divT.assign(N, Cplx(0.0, 0.0));
  if (!BFGS) xi_t = newStore();                                   // BFGS mode does not keep xi / K.xi (:22-26)
}

template <class TS>
OptimalControl<TS>::OptimalControl(IQMPS& target, IQMPS& initial, TS& stepper, size_t N_, double gamma_, bool BFGS_)
    : timeStepper(stepper), gamma(gamma_), tstep(stepper.getTstep()), N(N_), M(0), BFGS(BFGS_) {
  GRAPE = true;                                                   // no ControlBasis -> GRAPE (:13-16)
  init(target, initial);
}

template <class TS>
OptimalControl<TS>::OptimalControl(IQMPS& target, IQMPS& initial, TS& stepper, ControlBasis& basis_, double gamma_, bool BFGS_)
    : timeStepper(stepper), basis(basis_), gamma(gamma_), tstep(stepper.getTstep()), N(basis_.getN()), M(basis_.getM()), BFGS(BFGS_) {
  GRAPE = false;                                                  // GROUP (:37-41)
  init(target, initial);
}

template <class TS> void OptimalControl<TS>::setThreadCount(const size_t n) {
  if (n < 1) throw std::invalid_argument("Mininum threadCount is 1.");       // :56
  threadCount = n;
}
template <class TS> void OptimalControl<TS>::setGRAPE(const bool g) { GRAPE = g; calculatedXi = false; }
template <class TS> void OptimalControl<TS>::setBFGS(const bool useBFGS_) {
  BFGS = useBFGS_;
  calculatedXi = false;
  if (BFGS) { xi_t.reset(); xiHlist.reset(); } else { xi_t = newStore(); }    // :70-85
}
template <class TS> bool OptimalControl<TS>::useBFGS() const { return BFGS; }
template <class TS> size_t OptimalControl<TS>::getM() const { return M; }
template <class TS> size_t OptimalControl<TS>::getN() const { return N; }
template <class TS> void OptimalControl<TS>::setGamma(double g) { gamma = g; }
template <class TS> stdvec OptimalControl<TS>::getControl(const stdvec& c) { return GRAPE ? c : basis.convertControl(c); }

template <class TS> std::vector<IQMPS> OptimalControl<TS>::getPsit() const {
  std::vector<IQMPS> out;
  const SiteSet& sites = timeStepper.sites();
  for (size_t i = 0; i < N; ++i) {
    IQMPS m(sites.N(), sites.D(), timeStepper.capacity());
    ocmps_check(ocmps_store_get(psi_t->h, (int)i, m.handle()), "ocmps_store_get");
    out.push_back(std::move(m));
  }
  return out;
}

template <class TS> stdvec OptimalControl<TS>::getTimeAxis() const {            // :188-201
  stdvec t;
  const double dt = timeStepper.getTstep();
  for (double x = 0; std::fabs(x - N * dt) > 1e-2 * dt; x += dt) t.push_back(x);
  return t;
}

// ---- regularisation (:89-143) ----
template <class TS> double OptimalControl<TS>::calcRegularization(const stdvec& u) const {
  double acc = 0;
  for (size_t i = 0; i + 1 < N; ++i) { const double d = u[i + 1] - u[i]; acc += d * d / tstep; }
  return gamma / 2.0 * acc;
}
template <class TS> stdvec OptimalControl<TS>::calcRegularizationGrad(const stdvec& u) const {
  stdvec g;
  g.reserve(N);
  g.push_back(-gamma * (-5.0 * u[1] + 4.0 * u[2] - u[3] + 2.0 * u[0]) / tstep);
  for (size_t i = 1; i + 1 < N; ++i) g.push_back(-gamma * (u[i + 1] + u[i - 1] - 2.0 * u[i]) / tstep);
  g.push_back(-gamma * (-5.0 * u[N - 2] + 4.0 * u[N - 3] - u[N - 4] + 2.0 * u[N - 1]) / tstep);
  return g;
}
template <class TS> rowmat OptimalControl<TS>::calcRegularizationHessian(const stdvec&) const {
  rowmat H(N, stdvec(N, 0.0));
  const double w = gamma / tstep;
  for (size_t i = 1; i + 1 < N; ++i) { H[i][i - 1] = -w; H[i][i + 1] = -w; H[i][i] = 2.0 * w; }
  H[1][0] = 0;
  H[N - 2][N - 1] = 0;
  return H;
}

// ---- sweeps (:376-438) ----
template <class TS> void OptimalControl<TS>::calcPsi(const stdvec& u) {
  ocmps_check(ocmps_forward_sweep(timeStepper.handle(), psi_init.handle(), u.data(), (int)N, psi_t->h), "ocmps_forward_sweep");
  calculatedXi = false;
}
template <class TS> void OptimalControl<TS>::calcXi(const stdvec& u) {
  ocmps_check(ocmps_backward_sweep(timeStepper.handle(), psi_target.handle(), u.data(), (int)N, xi_t->h), "ocmps_backward_sweep");
  calculatedXi = true;
}
template <class TS> void OptimalControl<TS>::calcDivT(const stdvec&) {
  ocmps_check(ocmps_store_divT(xi_t->h, psi_t->h, (int)N, reinterpret_cast<double*>(divT.data())), "ocmps_store_divT");
}
template <class TS> void OptimalControl<TS>::calcPsiXiDivT(const stdvec& u) {
  if (threadCount > 1) {          // the reference's two threads (:424-430) become two CUDA streams
    ocmps_check(ocmps_sweep_pair(timeStepper.handle(), psi_init.handle(), psi_target.handle(), u.data(), (int)N, psi_t->h, xi_t->h),
                "ocmps_sweep_pair");
    calculatedXi = true;
  } else {
    calcPsi(u);
    calcXi(u);
  }
  calcDivT(u);
}
template <class TS> Cplx OptimalControl<TS>::overlapFactor() {                  // overlapC(psi_t.back(), psi_target) (:242)
  fidOvl.assign(N, Cplx(0.0, 0.0));
  ocmps_check(ocmps_store_overlaps(psi_t->h, psi_target.handle(), (int)N, reinterpret_cast<double*>(fidOvl.data())), "ocmps_store_overlaps");
  return std::conj(fidOvl.back());
}

// ---- cost (:441-453) ----
template <class TS> double OptimalControl<TS>::calcCost(const stdvec& u, const bool new_control) {
  if (new_control) { calculatedXi = false; calcPsi(u); }
  overlapFactor();
  const Cplx o = fidOvl.back();
  return 0.5 * (1.0 - (o.real() * o.real() + o.imag() * o.imag())) + calcRegularization(u);
}

// ---- gradient (:205-249, :457-467) ----
template <class TS> stdvec OptimalControl<TS>::calcFidelityGrad(const stdvec& u, const bool new_control) {
  if (new_control) {
    calculatedXi = false;
    if (BFGS) calcPsi(u); else calcPsiXiDivT(u);
  }
  if (BFGS) {
    ocmps_check(ocmps_backward_sweep_divT(timeStepper.handle(), psi_target.handle(), u.data(), (int)N, psi_t->h,
                                          reinterpret_cast<double*>(divT.data())), "ocmps_backward_sweep_divT");
  } else if (!calculatedXi) {
    calcXi(u);
    calcDivT(u);
  }
  const Cplx of = overlapFactor();
  stdvec g(N);
  for (size_t i = 0; i < N; ++i) g[i] = tstep * (divT[i] * of * Cplx_i).real();
  return g;
}
template <class TS> stdvec OptimalControl<TS>::calcAnalyticGradient(const stdvec& u, const bool new_control) {
  stdvec g = calcFidelityGrad(u, new_control);
  const stdvec r = calcRegularizationGrad(u);
  for (size_t i = 0; i < N; ++i) g[i] += r[i];
  return g;
}

// ---- Hessian (:252-372) ----
template <class TS> rowmat OptimalControl<TS>::calcHessian(const stdvec& u, const bool new_control) {
  if (BFGS) throw std::logic_error("getHessian is undefined in BFGS mode");
  // prerequisites (:284-303) and rows (:305-335) as one event-ordered schedule on the GPU; the cache flags end up as the
  // reference leaves them
  const bool do_psi = new_control, do_xi = new_control || !calculatedXi;
  rowmat H = calcRegularizationHessian(u);
  if (!xiHlist) xiHlist = newStore();
  std::vector<int> rows;
  for (size_t r = 1; r + 1 < N; ++r) rows.push_back((int)r);
  std::vector<Cplx> ovl(N * N, Cplx(0.0, 0.0));
  std::vector<double> norms(N, 0.0);
  fidOvl.assign(N, Cplx(0.0, 0.0));
  const int chains = (int)std::max<size_t>(1, std::min<size_t>(64, 16 * threadCount));   // rows in flight (chi=100: 48 -> 8.84 s, 64 -> 8.43 s); the engine also bounds it by the free memory
  ocmps_check(ocmps_hessian_eval(timeStepper.handle(), psi_init.handle(), psi_target.handle(), u.data(), (int)N, psi_t->h, xi_t->h,
                                 xiHlist->h, rows.data(), (int)rows.size(), chains, do_psi ? 1 : 0, do_xi ? 1 : 0,
                                 reinterpret_cast<double*>(divT.data()), reinterpret_cast<double*>(fidOvl.data()),
                                 reinterpret_cast<double*>(ovl.data()), norms.data()), "ocmps_hessian_eval");
  calculatedXi = true;
  const Cplx of = std::conj(fidOvl[N - 1]);                                                                   // :297
  const double ts2 = tstep * tstep;
  for (int r : rows) {
    H[r][r] += ts2 * ((of * ovl[r * N + r]).real() - (divT[r] * std::conj(divT[r])).real());                  // :260-264
    for (size_t j = r + 1; j + 1 < N; ++j) {
      const double v = ts2 * ((of * ovl[r * N + j] * norms[r]).real() - (divT[r] * std::conj(divT[j])).real());  // :272-277
      H[r][j] += v;
      H[j][r] += v;
    }
  }
  return H;
}

template <class TS> stdvec OptimalControl<TS>::calcFidelityForAllT(const stdvec& u, const bool new_control) {   // :471-491
  if (new_control) { calculatedXi = false; calcPsi(u); }
  overlapFactor();
  stdvec f(N);
  for (size_t i = 0; i < N; ++i) f[i] = std::norm(fidOvl[i]);
  return f;
}

template <class TS>
void OptimalControl<TS>::calcEnergyForAllT(const stdvec& u, const bool new_control, bool variance, stdvec& E, stdvec& var) {
  if (new_control) { calculatedXi = false; calcPsi(u); }
  std::vector<double> m(3 * N, 0.0);
  ocmps_check(ocmps_store_energy_moments(psi_t->h, 0, (int)N, timeStepper.getJ(), u.data(), nullptr, 0, m.data()), "ocmps_store_energy_moments");
  E.assign(N, 0.0);
  for (size_t i = 0; i < N; ++i) E[i] = m[3 * i + 1] / m[3 * i];
  if (!variance) return;
  ocmps_check(ocmps_store_energy_moments(psi_t->h, 0, (int)N, timeStepper.getJ(), u.data(), E.data(), 1, m.data()), "ocmps_store_energy_moments");
  var.assign(N, 0.0);
  for (size_t i = 0; i < N; ++i) {
    const double h1 = m[3 * i + 1] / m[3 * i];
    var[i] = m[3 * i + 2] / m[3 * i] - h1 * h1;
  }
}

// ---- public API (:495-589) ----
template <class TS> void OptimalControl<TS>::propagatePsi(const stdvec& c) { calcPsi(GRAPE ? c : basis.convertControl(c)); }
template <class TS> double OptimalControl<TS>::getCost(const stdvec& c, const bool nc) {
  return GRAPE ? calcCost(c, nc) : calcCost(basis.convertControl(c, nc), nc);
}
template <class TS> stdvec OptimalControl<TS>::getAnalyticGradient(const stdvec& c, const bool nc) {
  if (GRAPE) return calcAnalyticGradient(c, nc);
  return basis.convertGradient(calcAnalyticGradient(basis.convertControl(c, nc), nc));
}
template <class TS> rowmat OptimalControl<TS>::getHessian(const stdvec& c, const bool nc) {
  if (GRAPE) return calcHessian(c, nc);
  return basis.convertHessian(calcHessian(basis.convertControl(c, nc), nc));
}
template <class TS> stdvec OptimalControl<TS>::getFidelityForAllT(const stdvec& c, const bool nc) {
  return GRAPE ? calcFidelityForAllT(c, nc) : calcFidelityForAllT(basis.convertControl(c, nc), nc);
}
template <class TS> stdvec OptimalControl<TS>::getEnergyForAllT(const stdvec& c, const bool nc) {
  stdvec E, var;
  calcEnergyForAllT(GRAPE ? c : basis.convertControl(c, nc), nc, false, E, var);
  return E;
}
template <class TS> stdvec OptimalControl<TS>::getEnergyVarianceForAllT(const stdvec& c, const bool nc) {
  stdvec E, var;
  calcEnergyForAllT(GRAPE ? c : basis.convertControl(c, nc), nc, true, E, var);
  return var;
}
template <class TS> rowmat OptimalControl<TS>::getControlJacobian() const {
  if (!GRAPE) return basis.getControlJacobian();
  rowmat J(N, stdvec(N, 0.0));
  for (size_t i = 0; i < N; ++i) J[i][i] = 1;
  return J;
}

template class OptimalControl<BH_tDMRG>;
