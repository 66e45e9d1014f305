/* ocmps.h -- C ABI of libocmps: the B200-native Bose-Hubbard tDMRG / optimal-control engine.
 *
 * The reference (fskovbo/OptimalControlMPS) has no FFI: its hot path is the C++ classes
 * BH_tDMRG (include/BH_tDMRG.hpp:16-40) and OptimalControl<TimeStepper>
 * (include/OptimalControl.hpp:17-76) calling ITensor on the CPU.  This header is the boundary a
 * maintainer binds instead of ITensor: every entry point below names the reference call it
 * replaces.  Plain C types only; opaque handles; caller-owned host buffers; library-owned device
 * memory; every function returns 0 on success and a negative code on failure, with the message
 * available from ocmps_last_error().  There is no CPU fallback: without a CUDA device
 * ocmps_ctx_create fails.
 *
 * Conventions
 *   L      chain length, sites are 0-based in this API (the reference is 1-based)
 *   D      local dimension = reference "d"+1 (include/BH_sites.h:73-91)
 *   MPS    site tensor j is a row-major complex128 array A[l][s][r] (chi_j x D x chi_{j+1});
 *          `tensors` is the concatenation over sites; `bond_dims` has L+1 entries;
 *          `charges` is the concatenation over the L+1 bonds of the boson number to the left of
 *          each bond index (the QN labels of ITensor's IQIndex, include/BH_sites.h:78-88).
 *   complex numbers cross the ABI as interleaved (re, im) doubles.
 */
#ifndef OCMPS_H
#define OCMPS_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ocmps_ctx ocmps_ctx;           /* one per GPU */
typedef struct ocmps_mps ocmps_mps;           /* device-resident MPS (replaces itensor::IQMPS) */
typedef struct ocmps_stepper ocmps_stepper;   /* replaces class BH_tDMRG */
typedef struct ocmps_store ocmps_store;       /* Nt time slices resident in HBM (replaces std::vector<IQMPS> psi_t / xi_t / xiHlist,
                                                 include/OptimalControl.hpp:26-28) */

#define OCMPS_OK 0
#define OCMPS_ERR_INVALID (-1)
#define OCMPS_ERR_CUDA (-2)
#define OCMPS_ERR_CAPACITY (-3)
#define OCMPS_ERR_NUMERIC (-4)

const char* ocmps_last_error(void);
int ocmps_version(void);
/* number of CUDA kernels launched by this library so far (bench.py reports it as gpu_launches) */
long long ocmps_launch_count(void);
/* measurement aid (bench.py): CUDA-event timing of the dominant kernel (the block SVD) on its own stream.
 * read -> out4 = { total ms inside the kernel, launches, block-summed algorithmic flops, dense-formula flops } */
int ocmps_profile_enable(int on);
int ocmps_profile_read(double* out4);

/* ---- context ---- */
int ocmps_ctx_create(int device, ocmps_ctx** out);
int ocmps_ctx_destroy(ocmps_ctx* ctx);
int ocmps_ctx_synchronize(ocmps_ctx* ctx);
/* frees the idle per-chain workspaces the library keeps between calls (they are re-created on demand) */
int ocmps_ctx_trim(ocmps_ctx* ctx);
/* measurement aid (bench.py): a pair of CUDA events on the library's own stream; stop returns the milliseconds between them */
int ocmps_timer_start(ocmps_ctx* ctx);
int ocmps_timer_stop(ocmps_ctx* ctx, double* ms);

/* ---- MPS container (itensor::IQMPS in the reference's signatures) ---- */
int ocmps_mps_create(ocmps_ctx* ctx, int L, int D, int chi_cap, ocmps_mps** out);
int ocmps_mps_destroy(ocmps_mps* mps);
int ocmps_mps_upload(ocmps_mps* mps, const int* bond_dims, const int* charges, const double* tensors, int llim, int rlim);
/* sizes needed by download: number of complex elements and number of charge labels */
int ocmps_mps_sizes(ocmps_mps* mps, long long* n_elems, long long* n_charges);
int ocmps_mps_download(ocmps_mps* mps, int* bond_dims, int* charges, double* tensors, int* llim, int* rlim);
int ocmps_mps_bond_dims(ocmps_mps* mps, int* bond_dims);       /* linkInd(psi,b).m(), main/AnalyzeBondDim.cpp:140 */
int ocmps_mps_copy(ocmps_mps* dst, ocmps_mps* src);            /* IQMPS copy, e.g. src/OptimalControl.cpp:379-380 */
/* psi.position(1): moves the orthogonality centre to site 1 with the engine's gauge moves, starting from the limits given at
 * upload (llim = 0, rlim = L+1: no site assumed orthogonal).  step / sweeps / apply_K require the centre at site 1. */
int ocmps_mps_position1(ocmps_mps* mps);
int ocmps_mps_norm(ocmps_mps* mps, double* out);               /* itensor::norm(psi), src/OptimalControl.cpp:257 */
/* overlapC(a,b) = <a|b> (first argument conjugated), src/OptimalControl.cpp:242,261,272,450 */
int ocmps_overlap(ocmps_mps* a, ocmps_mps* b, double* re_im);
/* overlapC(a, propDeriv, b) = <a|K|b>, K = sum_j 1/2 n_j(n_j-1), src/OptimalControl.cpp:220,227,417 */
int ocmps_overlap_K(ocmps_mps* a, ocmps_mps* b, double* re_im);

/* ---- time stepper (class BH_tDMRG) ----
 * cutoff < 0 / maxm <= 0 mean "key not given" (ITensor defaults 1e-16 / 5000, tests/CostTests.cpp:41).
 * chi_cap is the allocated bond capacity; a truncation that keeps more raises OCMPS_ERR_CAPACITY.
 * rel_cutoff selects ITensor's DoRelCutoff for the Cutoff rule. */
int ocmps_stepper_create(ocmps_ctx* ctx, int L, int D, double J, double tstep, double cutoff, int maxm, int chi_cap,
                         int rel_cutoff, ocmps_stepper** out);                 /* BH_tDMRG::BH_tDMRG, src/BH_tDMRG.cpp:3-15 */
int ocmps_stepper_destroy(ocmps_stepper* st);
int ocmps_stepper_set_tstep(ocmps_stepper* st, double tstep);                    /* BH_tDMRG::setTstep :61-65 */
double ocmps_stepper_get_tstep(ocmps_stepper* st);                                /* BH_tDMRG::getTstep :68-71 */
/* BH_tDMRG::step(psi, from, to, propagateForward), src/BH_tDMRG.cpp:111-125 (in place) */
int ocmps_step(ocmps_stepper* st, ocmps_mps* psi, double from, double to, int forward);
/* exactApplyMPO(stepper.propagatorDeriv(u), psi, stepper.getArgs()), src/OptimalControl.cpp:256,302,362 */
int ocmps_apply_K(ocmps_stepper* st, ocmps_mps* in, ocmps_mps* out);
/* the op list one step executes (for tests): writes up to `cap` quadruples (kind, a, b, c); returns the count */
int ocmps_stepper_schedule(ocmps_stepper* st, int* quads, int cap);
/* the two-site J gate exp(-+ i tstep h) as D^2 x D^2 interleaved complex (BondGate, src/BH_tDMRG.cpp:35-36) */
int ocmps_stepper_gate(ocmps_stepper* st, int forward, double* out);

/* InitializeState(sites, Npart, J, U[, maxBondDim, threshold]) (include/InitializeState.hpp:18-117): Bose-Hubbard ground state
 * H = -J sum (a_i adag_{i+1} + h.c.) + U/2 sum n_i(n_i-1) with Npart <= L bosons, produced on the device by imaginary-time evolution
 * with the Trotter-step kernels (the reference uses ITensor's DMRG; same start state :24-38, same bond-dimension schedule
 * 10, 20, 50, maxm :52-54, cutoff = threshold).  tau_final <= 0 selects 2e-3.  `out` must have capacity >= maxm; it ends
 * normalised with its orthogonality centre at site 1.  energy / steps may be NULL. */
int ocmps_ground_state(ocmps_ctx* ctx, int L, int D, int Npart, double J, double U, int maxm, double cutoff, double tau_final,
                       ocmps_mps* out, double* energy, int* steps);
/* The same ground state by two-site DMRG on the device, as the reference computes it (include/InitializeState.hpp:18-117:
 * `nsweeps` sweeps, maxm 10, 20, 50, maxm, cutoff; no noise term): the same start state, a Lanczos solve with 4 Krylov vectors
 * at every bond, the engine's truncating decomposition.  `out` must have capacity >= maxm (maxm < 1 selects the capacity); it
 * ends normalised with its orthogonality centre at site 1.  `energy` (may be NULL) is <psi|H|psi> of the returned state;
 * `sweep_energies` (nsweeps entries, or NULL) the last Ritz value of every sweep. */
int ocmps_ground_state_dmrg(ocmps_ctx* ctx, int L, int D, int Npart, double J, double U, int maxm, double cutoff, int nsweeps,
                            ocmps_mps* out, double* energy, double* sweep_energies);

/* ---- resident slice stores and sweeps (OptimalControl::calcPsi / calcXi / calcDivT) ---- */
int ocmps_store_create(ocmps_ctx* ctx, int L, int D, int chi_cap, int nslots, ocmps_store** out);
int ocmps_store_destroy(ocmps_store* store);
int ocmps_store_get(ocmps_store* store, int slot, ocmps_mps* out);            /* psi_t[slot] -> mps */
int ocmps_store_put(ocmps_store* store, int slot, ocmps_mps* in);
int ocmps_store_bond_dims(ocmps_store* store, int* out /* nslots*(L+1) */);
/* calcPsi (src/OptimalControl.cpp:376-390): store[0]=psi_init, store[i+1]=step(store[i],u[i],u[i+1],fwd) */
int ocmps_forward_sweep(ocmps_stepper* st, ocmps_mps* psi_init, const double* u, int Nt, ocmps_store* psi_store);
/* calcXi (:393-407): store[Nt-1]=psi_target, store[i-1]=step(store[i],u[i],u[i-1],bwd) */
int ocmps_backward_sweep(ocmps_stepper* st, ocmps_mps* psi_target, const double* u, int Nt, ocmps_store* xi_store);
/* both sweeps enqueued on two streams (the reference's two std::threads, :424-430) */
int ocmps_sweep_pair(ocmps_stepper* st, ocmps_mps* psi_init, ocmps_mps* psi_target, const double* u, int Nt,
                     ocmps_store* psi_store, ocmps_store* xi_store);
/* batches of independent controls (north_star; SeedGenerator fan-out of main/OptimizeRamp.cpp:60,83): `nchains` sweeps, chain c
 * starts from starts[c], runs forward (forward[c]=1, like calcPsi) or backward (like calcXi) under the controls
 * u[c*Nt .. c*Nt+Nt) and fills stores[c]; every chain has its own stream, one synchronisation at the end */
int ocmps_sweep_batch(ocmps_stepper* st, int nchains, ocmps_mps** starts, const int* forward, const double* u, int Nt,
                      ocmps_store** stores);
/* BFGS branch (:217-229): xi is propagated backwards without being stored, divT filled on the fly */
int ocmps_backward_sweep_divT(ocmps_stepper* st, ocmps_mps* psi_target, const double* u, int Nt, ocmps_store* psi_store,
                              double* divT /* 2*Nt */);
/* out[i] = <bra|store[i]> for all slots (calcFidelityForAllT :471-491, calcCost :450) */
int ocmps_store_overlaps(ocmps_store* store, ocmps_mps* bra, int Nt, double* out /* 2*Nt */);
/* divT[i] = <xi_i|K|psi_i> (calcDivT :410-419) */
int ocmps_store_divT(ocmps_store* xi_store, ocmps_store* psi_store, int Nt, double* out /* 2*Nt */);
/* Observables on resident slices (include/correlations.hpp:99-117 expectationValue / expectationValues; used per slice at
 * main/OptimizeRamp.cpp:144-158): out[((z*L + j)*nops + k] = <psi_z| O_k at site j |psi_z> for the slices first..first+count-1,
 * every site j and `nops` (1..7) site operators that are diagonal in the boson number, given by their diagonals
 * op_diag[k*D + n] (N: n; N(N-1): n(n-1); NN: n^2 -- include/BH_sites.h:129-171).  Not divided by the norm, like the reference.
 * The slices must have their orthogonality centre at site 1 (every slice written by the sweeps has); norm2 (may be NULL)
 * receives <psi_z|psi_z> as seen from every site, count*L values that all equal the norm when that holds. */
int ocmps_store_site_expectations(ocmps_store* store, int first, int count, const double* op_diag, int nops,
                                  double* out /* count*L*nops */, double* norm2 /* count*L or NULL */);
/* Two-point functions on a resident slice (include/correlations.hpp:10-55 correlationFunction, :57-80 correlationMatrix; used per
 * slice at main/AnalyzeQuench.cpp:143-144): out[z] = <psi| O_a(site_a) O_b(site_b) |psi> for `nentries` entries of four ints
 * (site_a, op_a, site_b, op_b): sites 0-based and distinct, op_x an index into op_table (nops real D x D matrices, row-major
 * O[t*D + s] = <t|O|s>, e.g. A: <j-1|A|j> = sqrt(j), include/BH_sites.h:129-171); site_b = -1 for a single operator (the caller
 * multiplies two operators that sit on the same site, :17-24).  Not divided by the norm.  Any gauge. */
int ocmps_store_correlations(ocmps_store* store, int slot, const double* op_table, int nops, const int* entries, int nentries,
                             double* out /* 2*nentries */);
/* Entanglement entropy of every bond (include/correlations.hpp:119-148: psi.position(i), SVD of the two-site wavefunction,
 * S = -sum_{p > 1e-12} p ln p over the density-matrix eigenvalues): out[z*(L-1) + (i-1)] for bond i = 1..L-1 of the slices
 * first..first+count-1.  Works on a copy (the store is not modified); slices must have their centre at site 1. */
int ocmps_store_entanglement_entropy(ocmps_store* store, int first, int count, double* out /* count*(L-1) */);
/* Energy moments of the slices first..first+count-1 under H(U_z) - c_z, H(U) = -J sum (a_i adag_{i+1} + h.c.) + U/2 sum n_i(n_i-1)
 * (the Hamiltonian of include/InitializeState.hpp:41-50 and of the stepper at control value U):
 * out[3z+0] = <psi|psi>,  out[3z+1] = <psi|H-c|psi>,  out[3z+2] = <psi|(H-c)^2|psi>  (raw, not divided by the norm).
 * U: count values (the control value of each slice); shift: count values or NULL (c = 0).
 * second_moment = 0 runs the 4-channel chain of the MPO and leaves out[3z+2] untouched; 1 runs the 16-channel chain of its
 * square (about 4x the work).  Any gauge.  A slice's results do not depend on the other slices of the call. */
int ocmps_store_energy_moments(ocmps_store* store, int first, int count, double J, const double* U, const double* shift,
                               int second_moment, double* out /* 3*count */);
/* xiHlist[i] = exactApplyMPO(K, xi_t[i], args) for all i (:300-303) */
int ocmps_store_apply_K(ocmps_stepper* st, ocmps_store* in, int Nt, ocmps_store* out);
/* calcHessianRow (:252-279) for `nrows` rows listed in `rows`: for every row r the raw ingredients are returned,
 *   ovl[r*Nt + j] = <xiH_j | psiH_r(t_j)>  (j = r .. Nt-2), norm[r] = ||K psi_r||;
 * the caller assembles H (it also needs divT and the regularisation).  `nchains` independent rows are in flight at once. */
int ocmps_hessian_rows(ocmps_stepper* st, ocmps_store* psi_store, ocmps_store* xiH_store, const double* u, int Nt,
                       const int* rows, int nrows, int nchains, double* ovl /* 2*Nt*Nt */, double* norms /* Nt */);

/* calcHessian_parallel (src/OptimalControl.cpp:282-338) as ONE schedule: the prerequisites of :284-303 -- psi sweep (do_psi),
 * xi sweep (do_xi), divT, xiHlist_i = exactApplyMPO(K, xi_i) -- and the rows of :305-335 are enqueued together and ordered by
 * events: row r starts as soon as psi_r exists, K.xi follows the xi sweep slice by slice, and a row's overlaps with xiHlist wait
 * for that store without stalling the row.  do_psi / do_xi = 0 reuse the slices already in psi_store / xi_store (the
 * new_control = false and calculatedXi cases of :284-294).  Outputs: divT[i] = <xi_i|K|psi_i>, fid[i] = <target|psi_i>
 * (overlapFactor :297 is conj(fid[Nt-1])), and ovl / norms as in ocmps_hessian_rows. */
int ocmps_hessian_eval(ocmps_stepper* st, ocmps_mps* psi_init, ocmps_mps* psi_target, const double* u, int Nt,
                       ocmps_store* psi_store, ocmps_store* xi_store, ocmps_store* xiH_store, const int* rows, int nrows,
                       int nchains, int do_psi, int do_xi, double* divT /* 2*Nt */, double* fid /* 2*Nt */,
                       double* ovl /* 2*Nt*Nt */, double* norms /* Nt */);

#ifdef __cplusplus
}
#endif
#endif /* OCMPS_H */
