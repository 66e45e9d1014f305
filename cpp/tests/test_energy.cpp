// Energy along a ramp through the C++ layer: reads a problem + the oracle's expected values written by
// tests/test_gpu_energy_moments.py (binary, little endian), evaluates OptimalControl::getEnergyForAllT /
// getEnergyVarianceForAllT (GRAPE) and energy / energyVariance of correlations.hpp.  Exit code 0 = all checks pass.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <fstream>
#include <vector>

#include "correlations.hpp"
#include "BH_tDMRG.hpp"
#include "OptimalControl.hpp"

static std::ifstream in;
static int failures = 0;

template <typename T> T rd() { T v; in.read(reinterpret_cast<char*>(&v), sizeof(T)); return v; }
static std::vector<double> rdvec() { int n = rd<int>(); std::vector<double> v(n); in.read(reinterpret_cast<char*>(v.data()), 8 * n); return v; }
static std::vector<int> rdivec() { int n = rd<int>(); std::vector<int> v(n); in.read(reinterpret_cast<char*>(v.data()), 4 * n); return v; }

static IQMPS rdstate(int L, int D, int cap) {
  std::vector<int> dims = rdivec(), q = rdivec();
  std::vector<double> t = rdvec();
  std::vector<Cplx> tc(t.size() / 2);
  for (size_t i = 0; i < tc.size(); ++i) tc[i] = Cplx(t[2 * i], t[2 * i + 1]);
  return IQMPS(L, D, cap, dims, q, tc);
}

// max_i |a_i - b_i| / scale_i
static double err(const std::vector<double>& a, const std::vector<double>& b, const std::vector<double>& scale) {
  double e = 0;
  for (size_t i = 0; i < a.size(); ++i) e = std::max(e, std::fabs(a[i] - b[i]) / scale[i]);
  return a.size() == b.size() ? e : INFINITY;
}
static void check(bool ok, const char* what, double val) {
  printf("%-52s %s (%.3e)\n", what, ok ? "ok" : "FAIL", val);
  if (!ok) ++failures;
}

int main(int argc, char** argv) {
  if (argc < 2) { fprintf(stderr, "usage: test_energy problem.bin\n"); return 2; }
  in.open(argv[1], std::ios::binary);
  if (!in) { fprintf(stderr, "cannot open %s\n", argv[1]); return 2; }
  const int L = rd<int>(), d = rd<int>(), N = rd<int>(), maxm = rd<int>(), cap = rd<int>();
  const double J = rd<double>(), tstep = rd<double>(), cutoff = rd<double>(), gamma = rd<double>(), U0 = rd<double>();
  auto sites = BoseHubbard(L, d);
  IQMPS psi_i = rdstate(L, d + 1, cap), psi_f = rdstate(L, d + 1, cap);
  const std::vector<double> u = rdvec(), E_ref = rdvec(), var_ref = rdvec();
  const double e0_ref = rd<double>(), v0_ref = rd<double>();
  if (!in) { fprintf(stderr, "truncated problem file\n"); return 2; }

  auto stepper = maxm > 0 ? BH_tDMRG(sites, J, tstep, {"Cutoff=", cutoff, "Maxm=", maxm}, cap) : BH_tDMRG(sites, J, tstep, {"Cutoff=", cutoff}, cap);
  check(stepper.getJ() == J, "BH_tDMRG::getJ", std::fabs(stepper.getJ() - J));
  OptimalControl<BH_tDMRG> OC(psi_f, psi_i, stepper, (size_t)N, gamma);
  std::vector<double> escale(N), vscale(N);
  for (int i = 0; i < N; ++i) { escale[i] = std::fabs(E_ref[i]); vscale[i] = E_ref[i] * E_ref[i]; }
  const std::vector<double> E = OC.getEnergyForAllT(u, true);
  check(err(E, E_ref, escale) < 1e-10, "getEnergyForAllT (new_control=true)", err(E, E_ref, escale));
  const std::vector<double> var = OC.getEnergyVarianceForAllT(u, false);
  check(err(var, var_ref, vscale) < 1e-8, "getEnergyVarianceForAllT (new_control=false)", err(var, var_ref, vscale));
  // new_control=false keeps the slices; the control passed only sets U
  std::vector<double> u2(u);
  for (double& x : u2) x += 1.0;
  const std::vector<double> E2 = OC.getEnergyForAllT(u2, false);
  const std::vector<double> E2b = OC.getEnergyForAllT(u2, false);
  check(E2 == E2b && E2 != E, "getEnergyForAllT(u2, false): U from the control", 0.0);
  const double e0 = energy(sites, psi_i, J, U0), v0 = energyVariance(sites, psi_i, J, U0);
  check(std::fabs(e0 - e0_ref) < 1e-12 * std::fabs(e0_ref), "energy(sites, psi_init, J, U)", std::fabs(e0 - e0_ref) / std::fabs(e0_ref));
  check(std::fabs(v0 - v0_ref) < 1e-10 * e0_ref * e0_ref, "energyVariance(sites, psi_init, J, U)", std::fabs(v0 - v0_ref) / (e0_ref * e0_ref));
  printf(failures ? "FAILED (%d)\n" : "PASSED\n", failures);
  return failures ? 1 : 0;
}
