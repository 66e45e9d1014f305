// Observables of the reference's include/correlations.hpp that are diagonal in the boson number, on the device engine:
//   expectationValue(sites, psi, opname, i)  (:99-107)   and   expectationValues(sites, psi, opname)  (:109-117)
// with opname "N", "N(N-1)" or "NN" (include/BH_sites.h:129-171).  The value is <psi|O_i|psi>, not divided by the norm,
// as in the reference.  The state is copied into a one-slot slice store and evaluated by the batched transfer-matrix
// chain (ocmps_store_site_expectations); that chain needs the orthogonality centre at site 1, which every state that
// went through BH_tDMRG::step has -- any other gauge is detected and reported.
// entanglementEntropy(sites, psi) (:119-148) is provided as well (gauge moves of the engine, spectrum per bond), and so are
// the two-point functions correlationFunction (:10-55), correlationMatrix (:57-80) and correlationTerm (:82-97) with every
// operator name of include/BH_sites.h ("N", "A", "Adag", "N(N-1)", "NN", "Id"): one batched transfer-matrix pass on the GPU
// (ocmps_store_correlations).  correlationMatrix returns a plain L x L matrix of Cplx instead of an ITensor.
#ifndef OCMPS_CORRELATIONS_HPP
#define OCMPS_CORRELATIONS_HPP

#include <algorithm>
#include <cmath>
#include <complex>
#include <stdexcept>
#include <string>
#include <vector>

#include "itensor/all.h"

namespace ocmps_detail {
inline std::vector<double> site_op_diagonal(const std::string& opname, int D) {
  std::vector<double> v(D);
  for (int n = 0; n < D; ++n) {
    if (opname == "N") v[n] = n;
    else if (opname == "N(N-1)") v[n] = n * (n - 1.0);
    else if (opname == "NN") v[n] = (double)n * n;
    else if (opname == "Id") v[n] = 1.0;
    else throw std::invalid_argument("correlations.hpp: operator '" + opname + "' is not diagonal in the boson number");
  }
  return v;
}
}  // namespace ocmps_detail

inline std::vector<itensor::Cplx> expectationValues(itensor::SiteSet const& sites, itensor::IQMPS& psi, std::string const& opname) {
  using namespace itensor;
  const int L = psi.N(), D = psi.D();
  (void)sites;
  ocmps_store* store = nullptr;
  ocmps_check(ocmps_store_create(default_context(), L, D, psi.capacity(), 1, &store), "ocmps_store_create");
  std::vector<double> out(L), nrm(L);
  const std::vector<double> diag = ocmps_detail::site_op_diagonal(opname, D);
  int rc = ocmps_store_put(store, 0, psi.handle());
  if (!rc) rc = ocmps_store_site_expectations(store, 0, 1, diag.data(), 1, out.data(), nrm.data());
  ocmps_store_destroy(store);
  ocmps_check(rc, "ocmps_store_site_expectations");
  for (int j = 1; j < L; ++j)
    if (std::fabs(nrm[j] - nrm[0]) > 1e-9 * std::fabs(nrm[0]))
      throw std::runtime_error("expectationValues: the orthogonality centre of psi is not at site 1");
  std::vector<Cplx> res(L);
  for (int j = 0; j < L; ++j) res[j] = Cplx(out[j], 0.0);
  return res;
}

inline itensor::Cplx expectationValue(itensor::SiteSet const& sites, itensor::IQMPS& psi, std::string const& opname, int i) {
  return expectationValues(sites, psi, opname).at(i - 1);       // sites are 1-based in the reference
}

namespace ocmps_detail {
// <t|Op|s> as a real D x D matrix, row-major (include/BH_sites.h:129-171; "Id" is the true identity)
inline std::vector<double> site_op_matrix(const std::string& opname, int D) {
  std::vector<double> m((size_t)D * D, 0.0);
  if (opname == "A") { for (int j = 1; j < D; ++j) m[(size_t)(j - 1) * D + j] = std::sqrt((double)j); return m; }          // <j-1|A|j>
  if (opname == "Adag") { for (int j = 1; j < D; ++j) m[(size_t)j * D + (j - 1)] = std::sqrt((double)j); return m; }       // <j|Adag|j-1>
  const std::vector<double> d = site_op_diagonal(opname, D);
  for (int n = 0; n < D; ++n) m[(size_t)n * D + n] = d[n];
  return m;
}
inline std::vector<double> matmul(const std::vector<double>& a, const std::vector<double>& b, int D) {
  std::vector<double> c((size_t)D * D, 0.0);
  for (int i = 0; i < D; ++i) for (int k = 0; k < D; ++k) for (int j = 0; j < D; ++j) c[(size_t)i * D + j] += a[(size_t)i * D + k] * b[(size_t)k * D + j];
  return c;
}
// values of a list of (i, j) requests (1-based sites) for one operator pair
inline std::vector<itensor::Cplx> correlations(itensor::IQMPS& psi, std::string const& opname1, std::string const& opname2,
                                               const std::vector<std::pair<int, int>>& req) {
  using namespace itensor;
  const int L = psi.N(), D = psi.D();
  const std::vector<double> o1 = site_op_matrix(opname1, D), o2 = site_op_matrix(opname2, D), o12 = matmul(o1, o2, D);
  std::vector<double> table;
  table.insert(table.end(), o1.begin(), o1.end());
  table.insert(table.end(), o2.begin(), o2.end());
  table.insert(table.end(), o12.begin(), o12.end());
  std::vector<int> entries;
  for (auto& r : req) {
    if (r.first < 1 || r.first > L || r.second < 1 || r.second > L) throw std::invalid_argument("correlationFunction: site out of range");
    if (r.first == r.second) { entries.insert(entries.end(), {r.first - 1, 2, -1, 0}); }
    else { entries.insert(entries.end(), {r.first - 1, 0, r.second - 1, 1}); }
  }
  ocmps_store* store = nullptr;
  ocmps_check(ocmps_store_create(default_context(), L, D, psi.capacity(), 1, &store), "ocmps_store_create");
  std::vector<Cplx> out(req.size());
  int rc = ocmps_store_put(store, 0, psi.handle());
  if (!rc) rc = ocmps_store_correlations(store, 0, table.data(), 3, entries.data(), (int)req.size(), reinterpret_cast<double*>(out.data()));
  ocmps_store_destroy(store);
  ocmps_check(rc, "ocmps_store_correlations");
  return out;
}
}  // namespace ocmps_detail

// <psi| Op1_i Op2_j |psi>, sites 1-based (:10-55); for i == j the product Op1.Op2 on that site, whose real part the reference returns
inline itensor::Cplx correlationFunction(itensor::SiteSet const& sites, itensor::IQMPS& psi, std::string const& opname1, int i,
                                         std::string const& opname2, int j) {
  (void)sites;
  const itensor::Cplx v = ocmps_detail::correlations(psi, opname1, opname2, {{i, j}})[0];
  return i == j ? itensor::Cplx(v.real(), 0.0) : v;
}

using CorrMatrix = std::vector<std::vector<itensor::Cplx>>;
inline CorrMatrix correlationMatrix(itensor::SiteSet const& sites, itensor::IQMPS& psi, std::string const& opname1, std::string const& opname2) {
  (void)sites;
  const int L = psi.N();
  std::vector<std::pair<int, int>> req;
  for (int i = 1; i <= L; ++i) for (int j = i; j <= L; ++j) req.push_back({i, j});
  const std::vector<itensor::Cplx> v = ocmps_detail::correlations(psi, opname1, opname2, req);
  CorrMatrix rho(L, std::vector<itensor::Cplx>(L));
  for (size_t k = 0; k < req.size(); ++k) {
    const int i = req[k].first - 1, j = req[k].second - 1;
    if (i == j) rho[i][i] = itensor::Cplx(v[k].real(), 0.0);
    else { rho[i][j] = v[k]; rho[j][i] = std::conj(v[k]); }
  }
  return rho;
}

// largest eigenvalue of the (Hermitian) correlation matrix (:82-97): cyclic Jacobi on the L x L matrix, host side
inline double correlationTerm(itensor::SiteSet const& sites, itensor::IQMPS& psi, std::string const& opname1, std::string const& opname2) {
  CorrMatrix a = correlationMatrix(sites, psi, opname1, opname2);
  const int n = (int)a.size();
  for (int sweep = 0; sweep < 60; ++sweep) {
    double off = 0.0;
    for (int p = 0; p < n; ++p) for (int q = p + 1; q < n; ++q) off += std::norm(a[p][q]);
    if (off < 1e-28) break;
    for (int p = 0; p < n; ++p)
      for (int q = p + 1; q < n; ++q) {
        const itensor::Cplx apq = a[p][q];
        const double g = std::abs(apq);
        if (g < 1e-300) continue;
        const itensor::Cplx ph = apq / g;                         // a_pq = g e^{i phi}
        const double app = a[p][p].real(), aqq = a[q][q].real();
        const double zeta = (aqq - app) / (2.0 * g);
        const double t = (zeta >= 0 ? 1.0 : -1.0) / (std::fabs(zeta) + std::sqrt(1.0 + zeta * zeta));
        const double c = 1.0 / std::sqrt(1.0 + t * t), s = t * c;
        for (int k = 0; k < n; ++k) {                              // columns p, q
          const itensor::Cplx akp = a[k][p], akq = a[k][q];
          a[k][p] = c * akp - s * std::conj(ph) * akq;
          a[k][q] = s * ph * akp + c * akq;
        }
        for (int k = 0; k < n; ++k) {                              // rows p, q
          const itensor::Cplx apk = a[p][k], aqk = a[q][k];
          a[p][k] = c * apk - s * ph * aqk;
          a[q][k] = s * std::conj(ph) * apk + c * aqk;
        }
      }
  }
  double best = a[0][0].real();
  for (int i = 1; i < n; ++i) best = std::max(best, a[i][i].real());
  return best;
}

inline std::vector<double> entanglementEntropy(itensor::SiteSet const& sites, itensor::IQMPS& psi) {
  using namespace itensor;
  const int L = psi.N(), D = psi.D();
  (void)sites;
  ocmps_store* store = nullptr;
  ocmps_check(ocmps_store_create(default_context(), L, D, psi.capacity(), 1, &store), "ocmps_store_create");
  std::vector<double> S(L > 1 ? L - 1 : 0);
  int rc = ocmps_store_put(store, 0, psi.handle());
  if (!rc && L > 1) rc = ocmps_store_entanglement_entropy(store, 0, 1, S.data());
  ocmps_store_destroy(store);
  ocmps_check(rc, "ocmps_store_entanglement_entropy");
  return S;
}

// Energy <psi|H|psi> / <psi|psi> of H = -J sum (a_i adag_{i+1} + h.c.) + U/2 sum n_i(n_i-1) (include/InitializeState.hpp:41-50) and
// its variance <H^2> - <H>^2 (zero on an eigenstate), by the transfer-matrix chain of the MPO on the device.  Any gauge.
namespace ocmps_detail {
inline void energy_moments(itensor::IQMPS& psi, double J, double U, const double* shift, int second_moment, double* m) {
  using namespace itensor;
  ocmps_store* store = nullptr;
  ocmps_check(ocmps_store_create(default_context(), psi.N(), psi.D(), psi.capacity(), 1, &store), "ocmps_store_create");
  int rc = ocmps_store_put(store, 0, psi.handle());
  if (!rc) rc = ocmps_store_energy_moments(store, 0, 1, J, &U, shift, second_moment, m);
  ocmps_store_destroy(store);
  ocmps_check(rc, "ocmps_store_energy_moments");
}
}  // namespace ocmps_detail

inline double energy(itensor::SiteSet const& sites, itensor::IQMPS& psi, double J, double U) {
  (void)sites;
  double m[3] = {0.0, 0.0, 0.0};
  ocmps_detail::energy_moments(psi, J, U, nullptr, 0, m);
  return m[1] / m[0];
}

inline double energyVariance(itensor::SiteSet const& sites, itensor::IQMPS& psi, double J, double U) {
  const double E = energy(sites, psi, J, U);
  double m[3] = {0.0, 0.0, 0.0};
  ocmps_detail::energy_moments(psi, J, U, &E, 1, m);
  const double h1 = m[1] / m[0];
  return m[2] / m[0] - h1 * h1;
}

#endif
