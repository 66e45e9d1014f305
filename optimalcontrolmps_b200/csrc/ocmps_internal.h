// Internal declarations shared by the CUDA translation units of libocmps.
// Device-resident "descriptors" drive every kernel: bond dimensions are decided on the GPU
// (truncation), so kernels are launched on capacity-sized grids and read the actual problem
// sizes from device memory.  No host synchronisation happens inside a Trotter step.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

typedef double2 cplx;

#define OCMPS_MAX_L 64      // chain length limit (pointer tables passed by value)
#define OCMPS_MAX_D 8       // local Hilbert space dimension limit
#define OCMPS_MAX_Q 256     // charges (boson number left of a bond) must be < OCMPS_MAX_Q
#define OCMPS_MAX_BLK 128   // max charge blocks per decomposition

// status bits written by kernels into Ctx::d_status
#define OCMPS_ST_CAPACITY   1   // kept bond dimension exceeds the allocated capacity
#define OCMPS_ST_NOCONV     2   // Jacobi did not converge within the sweep limit
#define OCMPS_ST_CHARGE     4   // charge label outside [0, OCMPS_MAX_Q)
#define OCMPS_ST_TOOMANYBLK 8

struct GemmDesc {           // C(MxN) = op(A) * op(B), row-major complex128
  const cplx* A; const cplx* B; cplx* C;
  int M, N, K;
  int lda, ldb, ldc;
  int opA, opB;             // 0: as stored, 1: conjugate transpose
  int pad;
};

struct DecompBlock {
  int q;                    // charge of the block
  int nv, len;              // number of vectors to orthogonalise, their length
  int vec_off, comp_off;    // offsets into vec_idx / comp_idx
  int ws_off;               // element offset into the vector workspace (nv*len elements)
  int p_off;                // offset into P / pos
  int pad;
};

struct DecompWork {
  int n, m, ld;             // matrix X is n x m, leading dimension ld
  int mode;                 // 0: vectors are columns (isometry n x k); 1: vectors are rows (isometry k x m)
  int nblocks, nvtot, newdim;
  int pad0;
  double scale;             // factor applied to the centre-carrying factor (1/norm for gate decompositions)
  DecompBlock blk[OCMPS_MAX_BLK];
};

struct TruncParams {
  double cutoff;            // ITensor "Cutoff"
  int maxm, minm;
  int rel_cutoff;           // ITensor doRelCutoff
  int cap;                  // capacity of the new bond
  int normalize;            // divide the centre-carrying factor by its Frobenius norm (src/BH_tDMRG.cpp:183-184)
};

// Everything that changes from one Trotter step to the next lives in device memory, so that the kernel sequence
// of a step has constant arguments and can be replayed as a CUDA graph.
struct StepParams {
  double u1r[OCMPS_MAX_D], u1i[OCMPS_MAX_D];   // exp(-i/4 U_from tstep n(n-1))   (src/BH_tDMRG.cpp:84-88)
  double u2r[OCMPS_MAX_D], u2i[OCMPS_MAX_D];   // ... U_to
  const cplx* G;                               // forward or backward J gate
  cplx* slot_data; int* slot_dims; int* slot_q; // destination slice of the store (or null)
};

struct SitePtrs { cplx* p[OCMPS_MAX_L]; };
struct SiteOffs { long long o[OCMPS_MAX_L + 1]; };

// diagonal on-site phases around the J gate: [0] in on site 1, [1] in on site 2, [2] out on site 1, [3] out on site 2
struct Phases { double re[4][OCMPS_MAX_D]; double im[4][OCMPS_MAX_D]; };

#include <atomic>
extern std::atomic<long long> g_ocmps_launches;   // kernels launched so far (bench.py reports it)

void debug_jacobi_counters(unsigned long long* out, bool reset);
void debug_row_cluster_counters(unsigned long long* out, bool reset);
void profile_enable(bool on);
bool profile_is_on();
void profile_read(double* out);

// ---- kernels (launchers) ----
void launch_zgemm(const GemmDesc* d_descs, int batch, int maxM, int maxN, cudaStream_t s);

enum DecompKind { DK_GATE_LEFT = 0, DK_GATE_RIGHT = 1, DK_ORTH_LEFT = 2, DK_ORTH_RIGHT = 3 };

struct DecompArgs {
  int kind;                 // DecompKind
  int D;
  const int* dimL;          // pointer to the dimension of the left bond of X
  const int* dimR;          // ... right bond of X
  const int* qL;            // charges of the left bond
  const int* qR;            // charges of the right bond
  int* dimNew;              // bond whose dimension / charges are (re)written
  int* qNew;
  const cplx* X;            // matrix to decompose
  cplx* iso;                // isometry output
  cplx* partner;            // gate kinds: the other site tensor; orth kinds: the carry matrix C
  const cplx* nb_in;        // orth kinds: neighbouring site tensor (input)
  cplx* nb_out;             // orth kinds: neighbouring site tensor (output)
  const int* dimNb;         // orth kinds: far bond dimension of the neighbour
  const int* qNb;           // orth kinds: charges of that far bond; if set, build_factors pushes the carry matrix into
                            // the neighbour itself (sector by sector) and no GEMM follows; nullptr: caller runs descs[1]
};

struct DecompBuffers {
  DecompWork* dw;
  int* vec_idx; int* comp_idx;   // sorted index lists
  int* vecq;                      // charge per entry of P
  double* P;                      // squared norms of all vectors
  int* pos;                       // new bond index of each vector (-1: dropped)
  cplx* ywork;                    // region A: right vectors Z block after block; region B (+ywork_half): scratch
  long long ywork_half;
  double* scratch_d;              // 8*NV_MAX doubles (global-memory fallback of the block kernel)
  GemmDesc* descs;                // [1] neighbour gemm of gauge moves, [2] two-site merge
  double* partial;                // norm partial sums
  int* status;
};

void launch_decomp_setup(const DecompArgs& a, const DecompBuffers& b, cudaStream_t s);
// second stream + events for the cluster chain of a decomposition (qr_big -> jacobi_big beside QR -> rotations), see decomp.cu
struct SvdFork { cudaStream_t stream = nullptr; cudaEvent_t ev_fork = nullptr, ev_first = nullptr, ev_join = nullptr; };
void launch_jacobi_blocks(const DecompArgs& a, const DecompBuffers& b, int nblk_launch, size_t smem_limit, bool need_global,
                          bool long_rows, double rank_tol, int max_rows, int capV, int capC, bool spread_rows, cudaStream_t s,
                          const SvdFork* fork = nullptr);
void launch_spectrum_entropy(const DecompBuffers& b, double* out, cudaStream_t s);
void launch_truncate(const DecompArgs& a, const DecompBuffers& b, const TruncParams& tp, cudaStream_t s);
void launch_build_factors(const DecompArgs& a, const DecompBuffers& b, int cap_k, int cap_vec, int cap_comp, cudaStream_t s);

// merge setup: fills desc for theta = A1 (chil*D x chim) * A2 (chim x D*chir)
void launch_merge_setup(GemmDesc* d, const cplx* A1, const cplx* A2, cplx* theta, const int* dimL, const int* dimM,
                        const int* dimR, int D, cudaStream_t s);
// gate_kind: 0 = U(from) then J, 1 = same plus the lonely U(to) on the second site, 2 = J then U(to)
void launch_merge_gate(const cplx* A1, const cplx* A2, cplx* theta, const int* dimL, const int* dimM, const int* dimR,
                       const int* qL, const int* qM, const int* qR, int D, const StepParams* sp, int gate_kind, int maxL, int maxR,
                       cudaStream_t s);
void launch_gate_apply(cplx* theta, const int* dimL, const int* dimR, const int* qL, const int* qR, int D, const StepParams* sp,
                       int gate_kind, int maxL, int maxR, cudaStream_t s);
void launch_site_phase(cplx* A, const int* dimL, const int* dimR, int D, const StepParams* sp, int which, int max_elems, cudaStream_t s);
void launch_set_step_params(const StepParams& hp, StepParams* dst, cudaStream_t s);
// pack the work MPS into the store slot named by *sp (data, dims and charge labels)
void launch_pack_to_slot(SitePtrs src, SiteOffs offs, const int* dims, const int* q, int L, int D, int cap, int max_site_elems,
                         const StepParams* sp, int* status, cudaStream_t s);
void launch_norm_only(const cplx* x, const int* dimL, const int* dimR, int D, double* partial, double* out, int max_elems,
                      cudaStream_t s);
void launch_normalize_site(cplx* x, const int* dimL, const int* dimR, int D, double* partial, int max_elems, cudaStream_t s);

// packed copies between a work MPS (per-site pointers) and a store slot
// (status: device status word of the caller's workspace, or nullptr -- a bulk copy that fails then traps)
void launch_pack_copy(SitePtrs src, cplx* dst_base, SiteOffs offs, const int* dims, int L, int D, int max_site_elems, int* status,
                      cudaStream_t s);
void launch_unpack_copy(const cplx* src_base, SitePtrs dst, SiteOffs offs, const int* dims, int L, int D, int max_site_elems, int* status,
                        cudaStream_t s);

// overlaps (transfer matrices).  One "pair" per batch entry.
struct OvlSide {              // how to find site tensors / dims of batch entry z
  const cplx* base;           // store base (or nullptr when ptrs are used)
  long long slot_stride;      // elements between slots
  SiteOffs offs;              // site offsets within a slot
  SitePtrs ptrs;              // per-site pointers for a work MPS (batch 1)
  const int* dims;            // dims base
  int dims_stride;            // ints between slots' dims arrays
  int use_ptrs;
  int slot0;                  // first slot of the batch
};
void launch_overlap_plan(GemmDesc* descs, const OvlSide& bra, const OvlSide& ket, int site, int batch, int D, int withK,
                         cplx* E_in, cplx* E_out, cplx* T, long long e_stride, long long t_stride, cudaStream_t s);
void launch_overlap_init(cplx* E, long long e_stride, int batch, int withK, cudaStream_t s);
constexpr int OCMPS_EXPECT_MAX_OPS = 8;   // site operators per call of the expectation-value chain (slot 0 = identity)
void launch_overlap_local_expect(const GemmDesc* descs, const OvlSide& bra, int site, int batch, int D, const double* ops, int nops,
                                 double* out, int L, cudaStream_t s);
void launch_overlap_kfix(cplx* T, long long t_stride, const GemmDesc* descs, int batch, int D, int max_elems, cudaStream_t s);
void launch_overlap_site_op(cplx* T, long long t_stride, const GemmDesc* descs, int batch, int D, const double* op_table, const int* sel,
                            int max_elems, cudaStream_t s);
void launch_overlap_final(const cplx* E, long long e_stride, int batch, int withK, cplx* out, cudaStream_t s);
// nch environment channels; the E' gemms read Tmix (pass T for no channel mixing).  launch_overlap_plan is nch = withK ? 2 : 1.
void launch_overlap_plan_channels(GemmDesc* descs, const OvlSide& bra, const OvlSide& ket, int site, int batch, int D, int nch,
                                  cplx* E_in, cplx* E_out, cplx* T, const cplx* Tmix, long long e_stride, long long t_stride,
                                  cudaStream_t s);

// Energy moments of H(U) - c with the bond-dimension-4 MPO W of the Bose-Hubbard chain (MPO states 3 = nothing placed, 1 / 2 =
// a / adag placed, 0 = done): W[0,0] = W[3,3] = I, W[3,0] = U/2 N(N-1) - c/L, W[3,1] = -J A, W[3,2] = -J Adag, W[1,0] = Adag,
// W[2,0] = A.  A transition src -> dst of the channel chain applies coef * F1 F2 (F2 = I for the 4 channels of W; the 16
// channels (a,b) of W x W apply W[a,a'] W[b,b']).
enum { ENERGY_F_ID = 0, ENERGY_F_A = 1, ENERGY_F_ADAG = 2, ENERGY_F_ONSITE = 3 };
constexpr int ENERGY_MAX_TRANS = 49;
struct EnergyTable {
  int nch, nt;                                   // channels (4 or 16), transitions (7 or 49), sorted by dst
  int src[ENERGY_MAX_TRANS], dst[ENERGY_MAX_TRANS];
  int f1[ENERGY_MAX_TRANS], f2[ENERGY_MAX_TRANS];
  double coef[ENERGY_MAX_TRANS];
  double A[OCMPS_MAX_D * OCMPS_MAX_D], Adag[OCMPS_MAX_D * OCMPS_MAX_D];   // <t|a|s>, <t|adag|s>, row-major D x D
};
void launch_energy_init(cplx* E, long long e_stride, int batch, int nch, cudaStream_t s);
// uc: per batch entry (U_z, c_z / L); max_cols: capacity bound of aL * bR
void launch_energy_mix(const cplx* T, cplx* Tmix, long long t_stride, const GemmDesc* descs, int batch, int D, const double* uc,
                       const EnergyTable& tab, int max_cols, cudaStream_t s);
void launch_energy_final(const cplx* E, long long e_stride, int batch, int nch, double* out, cudaStream_t s);

// ---- two-site DMRG (dmrg.cu) ----
constexpr int DMRG_KRYLOV = 4;      // Lanczos vectors per bond
struct KrylovState {                // device-resident state of the Lanczos solve of one bond
  double alpha[DMRG_KRYLOV], beta[DMRG_KRYLOV];
  double y[DMRG_KRYLOV];            // Ritz vector in the Krylov basis
  double ritz;                      // lowest Ritz value
  int nk;                           // Krylov vectors in use
  int stop;                         // breakdown: the remaining Krylov launches of this bond do nothing
};
// W = H_eff V on the two-site tensor of bonds dimL / dimR: environments EL (left bond) and ER (right bond), three channels at
// stride estride each; Y, Z: scratch of 3 x ystride elements each; descs: 6 GemmDesc
void launch_heff(GemmDesc* descs, const cplx* V, cplx* W, cplx* Y, cplx* Z, long long ystride, const cplx* EL, const cplx* ER,
                 long long estride, const int* dimL, const int* dimR, const int* qL, const int* qR, int D, double J, double U,
                 const KrylovState* ks, int capL, int capR, cudaStream_t s);
// environment of bond j+1 from bond j (side 0, A = left isometry of site j) or of bond j from bond j+1 (side 1, A = right
// isometry of site j); dimL / dimR are bonds j, j+1; T, T2: scratch of 3 x tstride elements each; descs: 6 GemmDesc
void launch_env_update(GemmDesc* descs, int side, const cplx* A, const cplx* Ein, cplx* Eout, cplx* T, cplx* T2, long long tstride,
                       long long estride, const int* dimL, const int* dimR, int D, double J, double U, int capL, int capR,
                       cudaStream_t s);
// Lanczos steps on two-site vectors of bonds dimL / dimR; partial: (DMRG_KRYLOV + 1) x 128 x 2 doubles; ks = nullptr in
// krylov_dot: run even after a breakdown
void launch_krylov_dot(const cplx* V, long long vstride, int nvec, const cplx* w, const int* dimL, const int* dimR, int D,
                       const KrylovState* ks, double* partial, cudaStream_t s);
void launch_krylov_init(const cplx* X, cplx* V0, const int* dimL, const int* dimR, int D, KrylovState* ks, const double* partial,
                        int max_elems, cudaStream_t s);
void launch_krylov_alpha(const cplx* V, long long vstride, int it, cplx* w, const int* dimL, const int* dimR, int D, KrylovState* ks,
                         const double* partial, int max_elems, cudaStream_t s);
void launch_krylov_reorth(const cplx* V, long long vstride, int nvec, cplx* w, const int* dimL, const int* dimR, int D,
                          const KrylovState* ks, const double* partial, int max_elems, cudaStream_t s);
void launch_krylov_next(cplx* V, long long vstride, int it, const cplx* w, const int* dimL, const int* dimR, int D, KrylovState* ks,
                        const double* partial, int max_elems, cudaStream_t s);
void launch_krylov_ritz(KrylovState* ks, cudaStream_t s);
void launch_krylov_combine(const cplx* V, long long vstride, cplx* X, const int* dimL, const int* dimR, int D, const KrylovState* ks,
                           int max_elems, cudaStream_t s);
void launch_krylov_scale(cplx* X, const int* dimL, const int* dimR, int D, const double* partial, int max_elems, cudaStream_t s);
void launch_partial_total(const double* partial, double* out, cudaStream_t s);   // real part of the first dot product

// K|psi>: builds the bond-dimension-2chi tensors
void launch_applyK_expand(const cplx* A, cplx* B, const int* dimL_in, const int* dimR_in, const int* qL_in, const int* qR_in,
                          int* dimL_out, int* dimR_out, int* qL_out, int* qR_out, int D, int site, int L, int max_elems,
                          cudaStream_t s);
