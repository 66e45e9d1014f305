// Truncated decompositions of the engine: charge-blocked, QR-preconditioned one-sided Jacobi SVD in
// shared memory.
//
// The reference truncates with ITensor's denmatDecomp (eigen-decomposition of the two-site reduced
// density matrix, i.e. the Gram matrix theta.theta^H) per particle-number block, followed by a
// global sort of all eigenvalues and the Cutoff/Maxm rule (SURVEY.md appendix A.2/A.3), and moves the
// orthogonality centre with block SVDs (A.4).  The eigenvalues of the Gram matrix are the squared
// singular values of theta and its eigenvectors are the singular vectors, so each charge block
// M (len x nv, columns = the vectors to orthogonalise) is decomposed as M = U D Z directly:
//   1. Householder QR with column pivoting, M P = Q R, in shared memory (rank revealing; k <= min(len, nv))
//      -- jacobi_blocks_kernel, step code in qr_step_cached;
//   2. Hestenes one-sided Jacobi on the k rows of R (Drmac-Veselic preconditioning: 6-7 sweeps instead of
//      the ~20 plain cyclic Jacobi needs on these strongly graded spectra): pairs of rows are rotated
//      until every Gram entry <r_p|r_q> vanishes; one half-warp per pair, dot products by shuffles;
//      the Gram diagonal (squared norms) is the spectrum the truncation rule sees
//      -- jacobi_rot_kernel (rows register resident, jacobi_sweep_blocked) for blocks with at most 64 rows of R,
//      (jacobi_rows_cluster_kernel: the same spread over a 4-CTA cluster by row blocks from 40 rows of R on, for calls with one or two chains),
//      the generic loops at the end of jacobi_blocks_kernel otherwise;
//   3. global truncation over all blocks (truncate_kernel);
//   4. only the kept left vectors are formed, u_j = M z_j^H / |M z_j^H| (build_factors_kernel; for gauge moves it
//      also pushes the carry matrix into the neighbouring site tensor).
// One CTA per block in 1 and 2.  Both are bound by instruction issue and dependent latency on that one SM (see
// profiles/r01_kernel_shares.md), so the code is specialised at compile time on the block shape wherever it is hot.
#include <cstdio>
#include <cstdlib>
#include "ocmps_internal.h"

// development counters: [0] sum of sweeps, [1] blocks, [2] max sweeps, [3] sweeps of blocks with nv >= 64, [4] such blocks,
// [5] QR clocks, [6] Jacobi clocks, [7] total clocks of those blocks
__device__ unsigned long long g_jac_dbg[8];
// algorithmic flops of the decompositions (SURVEY 8d): [0] block-summed, [1] dense formula
__device__ double g_jac_flops[2];

namespace {

constexpr int JAC_THREADS = 512;
constexpr int JAC_EPL = 8;                // elements per lane cached in registers (rows up to 16*8 = 128 long)
constexpr int JAC_NV_SMEM = 512;          // cached norms in shared memory for blocks with at most this many vectors
constexpr int JAC_MAX_SWEEPS = 60;
constexpr int JAC_BLOCKED_ROWS = 64;      // 4 rows per warp, JAC_THREADS / 32 warps
constexpr double JAC_TOL2 = 1e-28;        // rotate while |<p|q>|^2 > tol^2 <p|p><q|q>, tol = 1e-14
constexpr double DEFLATE_REL = 1e-30;     // vectors below this fraction of the block's weight are numerically zero
constexpr int NV_MAX = 2048;              // max number of vectors in one decomposition
// cluster kernel for large blocks (jacobi_big_kernel)
constexpr int BJ_C = 8;                   // CTAs per cluster
constexpr int BJ_TPP = 4;                 // lanes per pair
constexpr int BJ_MAX_ROWS = 256;          // rows of R
constexpr int BJ_SLOTS = BJ_MAX_ROWS / 2; // pair slots
constexpr int BJ_THREADS = BJ_SLOTS * BJ_TPP;      // 512
constexpr int BJ_MAX_EPL = 8;             // columns per lane: slices of up to 32 columns, rows of R up to 256 long
constexpr int BJ_MIN_CAP = 112;           // launched when the capacities allow blocks with at least this many rows

// Gram-matrix path of the gate decompositions (gram_chol_block)
__host__ __device__ __forceinline__ int gc_ldy(int len) { int l = (len + 3) & ~3; if ((l & 7) == 0) l += 4; return l; }   // = 4 (mod 8): conflict-free fragment loads
__host__ __device__ __forceinline__ int gc_ldg(int nvp) { return nvp | 1; }
__device__ __forceinline__ void gc_dmma(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}
constexpr int GC_MIN_RANK = 48;           // blocks with fewer vectors or shorter vectors than this keep the Householder QR
constexpr int GC_MAX_NV = 96;             // 12 x 12 tiles: at most 5 of the 78 upper tiles per warp (their accumulators live in registers)
constexpr int GC_TILES_PER_WARP = ((GC_MAX_NV / 8) * (GC_MAX_NV / 8 + 1) / 2 + 512 / 32 - 1) / (512 / 32);

// ------------------------------------------------------------------------------------------------
// setup: charges of rows / columns, block table, sorted index lists
// ------------------------------------------------------------------------------------------------
struct Geometry { int n, m, mode; };

__device__ __forceinline__ Geometry geometry(const DecompArgs& a, int chiL, int chiR) {
  Geometry g;
  switch (a.kind) {
    case DK_GATE_LEFT:  g.n = chiL * a.D; g.m = a.D * chiR; g.mode = 0; break;
    case DK_GATE_RIGHT: g.n = chiL * a.D; g.m = a.D * chiR; g.mode = 1; break;
    case DK_ORTH_LEFT:  g.n = chiL * a.D; g.m = chiR;       g.mode = 0; break;
    default:            g.n = chiL;       g.m = a.D * chiR; g.mode = 1; break;
  }
  return g;
}
// Block table and index lists of one decomposition.  Bond charges are kept sorted ascending by the engine
// (upload sorts, truncation emits sorted labels), so the members of a charge bin are a handful of contiguous
// index ranges and every list entry can be placed independently: rank within the bin = (ranges of smaller s)
// + offset inside its own range.  comp_blk / comp_rank live behind comp_idx, vec_blk / vec_rank behind vec_idx
// (3 * NV_MAX ints each).
constexpr int SETUP_THREADS = 1024;
constexpr int QT = OCMPS_MAX_Q + 2 * OCMPS_MAX_D + 2;     // charge tables with room for q +- s

__global__ void __launch_bounds__(SETUP_THREADS) decomp_setup_kernel(DecompArgs a, DecompBuffers b) {
  __shared__ int startL[QT + 1], startR[QT + 1];          // first bond index with charge >= c (c shifted by OCMPS_MAX_D)
  __shared__ int cnt_v[OCMPS_MAX_Q], cnt_c[OCMPS_MAX_Q], off_v[OCMPS_MAX_Q], off_c[OCMPS_MAX_Q], blk_of_q[OCMPS_MAX_Q];
  __shared__ int s_bad;
  const int chiL = *a.dimL, chiR = *a.dimR, D = a.D;
  const Geometry g = geometry(a, chiL, chiR);
  const int tid = threadIdx.x;
  const int Drow = (a.kind == DK_ORTH_RIGHT) ? 1 : D;     // rows are (l, t): charge qL[l] + t
  const int Dcol = (a.kind == DK_ORTH_LEFT) ? 1 : D;      // cols are (t, r): charge qR[r] - t
  int* comp_blk = b.comp_idx + NV_MAX;
  int* comp_rank = b.comp_idx + 2 * NV_MAX;
  int* vec_blk = b.vec_idx + NV_MAX;
  int* vec_rank = b.vec_idx + 2 * NV_MAX;
  const int SH = OCMPS_MAX_D;                             // table shift so that q - t >= -D is addressable
  if (tid == 0) s_bad = 0;
  __syncthreads();
  // start tables from the sorted labels: startX[c + SH] = first index whose charge is >= c
  for (int i = tid; i <= chiL; i += SETUP_THREADS) {
    const int lo = (i == 0) ? -SH : a.qL[i - 1] + 1;
    const int hi = (i == chiL) ? QT - SH : a.qL[i];
    if (i < chiL && (hi < 0 || hi >= OCMPS_MAX_Q || hi + 1 < lo)) s_bad = 1;       // out of range or not sorted
    for (int c = lo; c <= hi && c + SH <= QT; ++c) startL[c + SH] = i;
  }
  for (int i = tid; i <= chiR; i += SETUP_THREADS) {
    const int lo = (i == 0) ? -SH : a.qR[i - 1] + 1;
    const int hi = (i == chiR) ? QT - SH : a.qR[i];
    if (i < chiR && (hi < 0 || hi >= OCMPS_MAX_Q || hi + 1 < lo)) s_bad = 1;
    for (int c = lo; c <= hi && c + SH <= QT; ++c) startR[c + SH] = i;
  }
  __syncthreads();
  if (s_bad) { if (tid == 0) atomicOr(b.status, OCMPS_ST_CHARGE); }
#define CNTL(c) (((c) + SH < 0 || (c) + SH >= QT) ? 0 : startL[(c) + SH + 1] - startL[(c) + SH])
#define CNTR(c) (((c) + SH < 0 || (c) + SH >= QT) ? 0 : startR[(c) + SH + 1] - startR[(c) + SH])
  if (tid < OCMPS_MAX_Q) {
    const int q = tid;
    int nr = 0, nc = 0;
    for (int t = 0; t < Drow; ++t) nr += CNTL(q - t);
    for (int t = 0; t < Dcol; ++t) nc += CNTR(q + t);
    cnt_v[q] = g.mode == 0 ? nc : nr;
    cnt_c[q] = g.mode == 0 ? nr : nc;
  }
  __syncthreads();
  // block charges lie between the smallest and the largest row charge (labels are sorted): only that range is scanned
  int c_lo = chiL > 0 ? a.qL[0] : 0, c_hi = chiL > 0 ? a.qL[chiL - 1] + Drow - 1 : -1;
  c_lo = c_lo < 0 ? 0 : c_lo;
  c_hi = c_hi >= OCMPS_MAX_Q ? OCMPS_MAX_Q - 1 : c_hi;
  if (tid < OCMPS_MAX_Q && (tid < c_lo || tid > c_hi)) blk_of_q[tid] = -1;
  if (tid == 0) {
    DecompWork* w = b.dw;
    int nb = 0, ov = 0, oc = 0, ows = 0;
    for (int c = c_lo; c <= c_hi; ++c) {
      int bid = -1;
      if (cnt_v[c] > 0 && cnt_c[c] > 0) {
        if (nb < OCMPS_MAX_BLK) {
          bid = nb;
          off_v[c] = ov; off_c[c] = oc;
          DecompBlock B;
          B.q = c; B.nv = cnt_v[c]; B.len = cnt_c[c];
          B.vec_off = ov; B.comp_off = oc; B.ws_off = ows; B.p_off = ov; B.pad = 0;
          w->blk[nb] = B;
          {   // workspace of the block: nv*len for the vectors, or (rows of R) x (row stride padded to 16) if larger
            const int nvq = cnt_v[c], lenq = cnt_c[c];
            const int padded = (nvq < lenq ? nvq : lenq) * (((nvq + 15) >> 4) << 4);
            ows += nvq * lenq > padded ? nvq * lenq : padded;
          }
          ov += cnt_v[c]; oc += cnt_c[c];
          ++nb;
        } else {
          atomicOr(b.status, OCMPS_ST_TOOMANYBLK);
        }
      }
      blk_of_q[c] = bid;
    }
    w->n = g.n; w->m = g.m; w->ld = g.m; w->mode = g.mode;
    w->nblocks = nb; w->nvtot = ov; w->newdim = 0; w->scale = 1.0;
  }
  __syncthreads();
  // rows: index i = l * Drow + t
  for (int i = tid; i < g.n; i += SETUP_THREADS) {
    const int l = i / Drow, t = i % Drow;
    const int q = a.qL[l] + t;
    int bid = -1, rank = 0;
    if (q >= 0 && q < OCMPS_MAX_Q) {
      bid = blk_of_q[q];
      for (int tt = 0; tt < t; ++tt) rank += CNTL(q - tt);
      rank += l - startL[q - t + SH];
    }
    if (g.mode == 0) {                                   // rows are components
      comp_blk[i] = bid; comp_rank[i] = rank;
      if (bid >= 0) b.comp_idx[off_c[q] + rank] = i;
    } else {                                             // rows are vectors
      vec_blk[i] = bid; vec_rank[i] = rank;
      if (bid >= 0) { b.vec_idx[off_v[q] + rank] = i; b.vecq[off_v[q] + rank] = q; }
    }
  }
  // cols: index j = t * chiR + r
  for (int j = tid; j < g.m; j += SETUP_THREADS) {
    const int t = (Dcol == 1) ? 0 : j / chiR, r = (Dcol == 1) ? j : j % chiR;
    const int q = a.qR[r] - t;
    int bid = -1, rank = 0;
    if (q >= 0 && q < OCMPS_MAX_Q) {
      bid = blk_of_q[q];
      for (int tt = 0; tt < t; ++tt) rank += CNTR(q + tt);
      rank += r - startR[q + t + SH];
    }
    if (g.mode == 0) {                                   // cols are vectors
      vec_blk[j] = bid; vec_rank[j] = rank;
      if (bid >= 0) { b.vec_idx[off_v[q] + rank] = j; b.vecq[off_v[q] + rank] = q; }
    } else {
      comp_blk[j] = bid; comp_rank[j] = rank;
      if (bid >= 0) b.comp_idx[off_c[q] + rank] = j;
    }
  }
#undef CNTL
#undef CNTR
}

// ------------------------------------------------------------------------------------------------
// QR-preconditioned one-sided Jacobi on one charge block per CTA
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double half_sum(double v) {
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// One plane rotation of the rows a, b (16*EPL long, one half-warp, EPL elements per lane) that annihilates <a|b>.
// na, nb are the cached squared norms.  All 32 lanes must call (shuffles); `act` is uniform per half-warp.
template <int EPL>
__device__ __forceinline__ void jac_rotate(cplx (&ra)[EPL], cplx (&rb)[EPL], double& na, double& nb, bool act, double thr,
                                           int hl, int* s_rot, int* s_big) {
  double c0r = 0.0, c0i = 0.0, c1r = 0.0, c1i = 0.0;
#pragma unroll
  for (int e = 0; e < EPL; ++e) {
    const double pr = ra[e].x * rb[e].x + ra[e].y * rb[e].y;      // conj(a) * b
    const double pi = ra[e].x * rb[e].y - ra[e].y * rb[e].x;
    if (e & 1) { c1r += pr; c1i += pi; } else { c0r += pr; c0i += pi; }
  }
  const double cre = half_sum(c0r + c1r), cim = half_sum(c0i + c1i);
  if (!act) return;
  const double aa = na, bb = nb;
  const double c2 = cre * cre + cim * cim;
  if (aa <= thr || bb <= thr) {
    if (aa <= thr && aa > 0.0) {
#pragma unroll
      for (int e = 0; e < EPL; ++e) ra[e] = make_double2(0.0, 0.0);
      na = 0.0;
    }
    if (bb <= thr && bb > 0.0) {
#pragma unroll
      for (int e = 0; e < EPL; ++e) rb[e] = make_double2(0.0, 0.0);
      nb = 0.0;
    }
  } else if (c2 > JAC_TOL2 * aa * bb) {
    // tan 2theta = |c| / d with d = (b - a)/2.  With h = sqrt(d^2 + |c|^2), s = |d| + h and w = 1/sqrt(2 h s):
    // cos = s w, sigma = sin e^{i phi} = +-w c, tan(theta) |c| = |c|^2 / s = |c|^2 w^2 2h  (two rsqrt, no division)
    const double dd = 0.5 * (bb - aa);
    const double xh = dd * dd + c2;
    const double ih = rsqrt(xh);
    const double h = xh * ih;
    const double sdh = fabs(dd) + h;
    const double w = rsqrt(2.0 * h * sdh);
    const double cs = sdh * w;
    const double sgw = dd >= 0.0 ? w : -w;
    const double sr = sgw * cre, si = sgw * cim;
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
      const cplx u = ra[e], v = rb[e];
      ra[e] = make_double2(cs * u.x - (sr * v.x + si * v.y), cs * u.y - (sr * v.y - si * v.x));   // cs a - conj(sigma) b
      rb[e] = make_double2(cs * v.x + (sr * u.x - si * u.y), cs * v.y + (sr * u.y + si * u.x));   // sigma a + cs b
    }
    const double trr = c2 * (sgw * w) * (2.0 * h);
    const double a1 = aa - trr, b1 = bb + trr;
    na = a1 > 0.0 ? a1 : 0.0;
    nb = b1 > 0.0 ? b1 : 0.0;
    if (hl == 0) {
      *s_rot = 1;
      if (c2 > 1e-16 * aa * bb) *s_big = 1;                // an off-diagonal above 1e-8 (relative) was seen
    }
  }
}

// One sweep over all pairs of the keff <= 64 rows of Z (row stride ldz = 16*EPL, zero padded), rows held in registers.
//
// A round of the plain scheme moves every row through the 128 B/clk shared-memory crossbar twice and ends in a CTA
// barrier, which together cost more than the dot -> angle -> rotation latency chain itself.  Here the rows are grouped
// in blocks of two and a WARP owns a pair of blocks (one row of each per half-warp): the four cross pairs are done in
// two rounds with a register shuffle in between, and the block-level round-robin is mapped onto the warps such that
// every warp keeps one of its two blocks from one block round to the next (warp s plays block pair s in even block
// rounds and s-1 in odd ones).  Per rotation round that is half a row stored and half a row loaded per half-warp
// instead of two and two, and one CTA barrier per two rounds.  The pairs inside a block are done first.
template <int EPL>
__device__ __forceinline__ void jacobi_sweep_blocked(cplx* __restrict__ Z, int keff, double* __restrict__ nrm, double thr, int* s_rot, int* s_big) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, half = lane >> 4, hl = lane & 15;
  constexpr int ldz = 16 * EPL;
  const int nb = (keff + 1) >> 1;            // blocks of two rows
  const int nbp = (nb + 1) & ~1;             // padded to an even count
  const int nslots = nbp >> 1, mm = nbp - 1;
  cplx ra[EPL], rb[EPL];
  double na = 0.0, nbn = 0.0;
  auto load_row = [&](cplx (&r)[EPL], double& n, int row) {
    const cplx* z = Z + (row >= 0 ? row : 0) * ldz + hl;
#pragma unroll
    for (int e = 0; e < EPL; ++e) r[e] = row >= 0 ? z[16 * e] : make_double2(0.0, 0.0);
    n = row >= 0 ? nrm[row] : 0.0;
  };
  auto store_row = [&](const cplx (&r)[EPL], double n, int row) {
    if (row < 0) return;
    cplx* z = Z + row * ldz + hl;
#pragma unroll
    for (int e = 0; e < EPL; ++e) z[16 * e] = r[e];
    if (hl == 0) nrm[row] = n;
  };
  {   // pairs inside the blocks: half-warp i takes block i
    const int i = 2 * warp + half;
    const int x = 2 * i < keff ? 2 * i : -1, y = 2 * i + 1 < keff ? 2 * i + 1 : -1;
    load_row(ra, na, x);
    load_row(rb, nbn, y);
    jac_rotate<EPL>(ra, rb, na, nbn, x >= 0 && y >= 0, thr, hl, s_rot, s_big);
    store_row(ra, na, x);
    store_row(rb, nbn, y);
  }
  __syncthreads();
  auto blocks_of = [&](int R, int& P, int& Q) {
    P = -1; Q = -1;
    if (warp >= nslots) return;
    const int k = (R & 1) ? (warp == 0 ? nslots - 1 : warp - 1) : warp;
    int p = R + k; if (p >= mm) p -= mm;
    int q = R - k; if (q < 0) q += mm;
    if (k == 0) q = nbp - 1;
    P = p < nb ? p : -1;
    Q = q < nb ? q : -1;
  };
  int hbA = -1, hbB = -1;          // blocks in the A / B registers of this warp
  int rowA = -1, rowB = -1;        // rows in the A / B registers of this half-warp
  int P, Q;
  blocks_of(0, P, Q);
  for (int R = 0; R < nbp - 1; ++R) {
    if (P != hbA) { rowA = (P >= 0 && 2 * P + half < keff) ? 2 * P + half : -1; load_row(ra, na, rowA); }
    if (Q != hbB) { rowB = (Q >= 0 && 2 * Q + half < keff) ? 2 * Q + half : -1; load_row(rb, nbn, rowB); }
    hbA = P; hbB = Q;
    jac_rotate<EPL>(ra, rb, na, nbn, rowA >= 0 && rowB >= 0, thr, hl, s_rot, s_big);
    // the two halves swap their B rows: (a0,b0)(a1,b1) -> (a0,b1)(a1,b0)
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
      rb[e].x = __shfl_xor_sync(0xffffffffu, rb[e].x, 16);
      rb[e].y = __shfl_xor_sync(0xffffffffu, rb[e].y, 16);
    }
    nbn = __shfl_xor_sync(0xffffffffu, nbn, 16);
    rowB = __shfl_xor_sync(0xffffffffu, rowB, 16);
    jac_rotate<EPL>(ra, rb, na, nbn, rowA >= 0 && rowB >= 0, thr, hl, s_rot, s_big);
    // blocks of the next block round, named such that the block that stays keeps its registers
    int NP = -1, NQ = -1;
    if (R + 1 < nbp - 1) {
      blocks_of(R + 1, NP, NQ);
      if ((NP >= 0 && NP == hbB) || (NQ >= 0 && NQ == hbA)) { const int t = NP; NP = NQ; NQ = t; }
    }
    if (hbA != NP) store_row(ra, na, rowA);
    if (hbB != NQ) store_row(rb, nbn, rowB);
    P = NP; Q = NQ;
    __syncthreads();
  }
}

// Householder QR with column pivoting of one block whose vectors have at most 16*EPL components (rows of Y, stride
// len), one half-warp per vector and EPL components per lane at the fixed positions c = hl + 16 e.  A step is bound by
// instruction issue, not by arithmetic, so everything is specialised at compile time: EPL (addresses are immediates)
// and E0 = j / 16, the first chunk of 16 components that still takes part (chunks above the diagonal are not touched;
// inside the chunk of the diagonal the reflector is zero above it, so those lanes compute y -= f * 0).
//  * The reflector is built from the exact norm of the pivot vector; the downdated norms only select pivots.
//  * The dot products use the raw pivot vector and are corrected for the replaced diagonal element afterwards, so
//    the reflector scalars (two dependent rsqrt) and the first dot product are independent chains.
//  * The pivot of step j+1: every half-warp leaves the best (norm bits | 2047 - position) key of the vectors it
//    updated in s_cand; a step starts with two REDUX over the 32 candidates.
struct QrState {
  cplx* Y;
  int nv, len;
  double rtol_abs;
  double *ncur, *nnext, *nrmref, *rdr, *rdi;
  short *perm, *pcur, *pnext;
  unsigned long long (*s_cand)[32];
};

// One step; false when the numerical rank is reached (nothing was changed then).
template <int EPL, int E0>
__device__ __forceinline__ bool qr_step_cached(const QrState& q, int j) {
  constexpr unsigned long long KEY_POS = 2047ull;
  constexpr int nwarps = JAC_THREADS / 32;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, half = lane >> 4, hl = lane & 15;
  const int len = q.len, nv = q.nv;
  int bpos;
  {
    const unsigned long long kk = q.s_cand[j & 1][lane];
    const unsigned khi = (unsigned)(kk >> 32);
    const unsigned mhi = __reduce_max_sync(0xffffffffu, khi);
    const unsigned mlo = __reduce_max_sync(0xffffffffu, khi == mhi ? (unsigned)kk : 0u);
    bpos = (int)(KEY_POS - (unsigned long long)(mlo & 2047u));
  }
  const int pv = q.pcur[bpos];             // physical slot of the pivot vector
  const int pj = q.pcur[j];
  const cplx* x = q.Y + pv * len;
  const cplx alpha = x[j];
  cplx xv[EPL];
  double sq0 = 0.0, sq1 = 0.0;
#pragma unroll
  for (int e = E0; e < EPL; ++e) {
    const int c = hl + 16 * e;
    const bool in = (e > E0 || c >= j) && (e < EPL - 1 || c < len);
    xv[e] = x[in ? c : j];
    if (!in) xv[e] = make_double2(0.0, 0.0);
    const double q2 = xv[e].x * xv[e].x + xv[e].y * xv[e].y;
    if ((e - E0) & 1) sq1 += q2; else sq0 += q2;
  }
  const double best = half_sum(sq0 + sq1);             // exact |x[j..len)|^2, bitwise identical in every half-warp
  if (!(best > q.rtol_abs)) return false;              // numerical rank reached: the trailing block is negligible
  const double inx = rsqrt(best), normx = best * inx;
  const double a2 = alpha.x * alpha.x + alpha.y * alpha.y;
  const double ia = a2 > 0.0 ? rsqrt(a2) : 0.0, aabs = a2 * ia;
  const double phr = a2 > 0.0 ? alpha.x * ia : 1.0, phi = a2 > 0.0 ? alpha.y * ia : 0.0;
  const double dr = phr * normx, di = phi * normx;     // v0 - alpha
  const double v0r = alpha.x + dr, v0i = alpha.y + di;
  const double rb = rsqrt(normx * (normx + aabs));
  const double beta = rb * rb;
  if (tid == 0) { q.rdr[j] = -dr; q.rdi[j] = -di; q.perm[j] = (short)pv; }   // R_jj; final position j
  unsigned long long cand = 0ull;
  for (int ib = j + 1 + 2 * warp; ib < nv; ib += 2 * nwarps) {
    const int i = ib + half;
    const bool act = i < nv;
    const int phys = act ? (i == bpos ? pj : (int)q.pcur[i]) : pv;
    cplx* y = q.Y + phys * len;
    const cplx yj = y[j];
    const double told = q.ncur[phys], tref = q.nrmref[phys];
    cplx yv[EPL];
    double w0r = 0.0, w0i = 0.0, w1r = 0.0, w1i = 0.0;
#pragma unroll
    for (int e = E0; e < EPL; ++e) {
      const int c = hl + 16 * e;
      if (e < EPL - 1) yv[e] = y[c];
      else { yv[e] = y[c < len ? c : j]; if (c >= len) yv[e] = make_double2(0.0, 0.0); }
      const double pr = xv[e].x * yv[e].x + xv[e].y * yv[e].y;      // conj(x) * y
      const double pi = xv[e].x * yv[e].y - xv[e].y * yv[e].x;
      if ((e - E0) & 1) { w1r += pr; w1i += pi; } else { w0r += pr; w0i += pi; }
    }
    double wr = half_sum(w0r + w1r), wi = half_sum(w0i + w1i);
    wr += dr * yj.x + di * yj.y;                           // + conj(v0 - alpha) * y_j
    wi += dr * yj.y - di * yj.x;
    const double fr = beta * wr, fi = beta * wi;
#pragma unroll
    for (int e = E0; e < EPL; ++e) {
      const int c = hl + 16 * e;
      cplx yy = yv[e];
      yy.x -= fr * xv[e].x - fi * xv[e].y;
      yy.y -= fr * xv[e].y + fi * xv[e].x;
      yv[e] = yy;
      if (act && (e < EPL - 1 || c < len)) y[c] = yy;
    }
    // the diagonal component sees v0 instead of alpha: its owner lane overwrites what the loop stored
    const double yjr = yj.x - (fr * v0r - fi * v0i), yji = yj.y - (fr * v0i + fi * v0r);
    if (act && hl == (j & 15)) y[j] = make_double2(yjr, yji);
    const double rji2 = yjr * yjr + yji * yji;
    double tnew = told - rji2;
    const bool redo = act && !(tnew > 1.5e-8 * tref);
    if (__any_sync(0xffffffffu, redo)) {                   // rare: exact trailing norm
      double tail = 0.0;
#pragma unroll
      for (int e = E0; e < EPL; ++e) {
        const int c = hl + 16 * e;
        if (e > E0 || c > j) tail += yv[e].x * yv[e].x + yv[e].y * yv[e].y;
      }
      tail = half_sum(tail);
      if (redo) { tnew = tail; if (hl == 0) q.nrmref[phys] = tail; }
    }
    if (act) {
      tnew = tnew > 0.0 ? tnew : 0.0;
      if (hl == 0) { q.nnext[phys] = tnew; q.pnext[i] = (short)phys; }
      const unsigned long long kv = ((unsigned long long)__double_as_longlong(tnew) & ~KEY_POS) | (KEY_POS - (unsigned long long)i);
      cand = kv > cand ? kv : cand;
    }
  }
  if (hl == 0) q.s_cand[(j + 1) & 1][2 * warp + half] = cand;
  return true;
}

// Returns the numerical rank; q.ncur / q.pcur are left pointing at the final trailing norms / position -> slot map.
template <int EPL>
__device__ __forceinline__ int qr_pivoted_cached(QrState& q) {
  constexpr unsigned long long KEY_POS = 2047ull;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int kmax = q.nv < q.len ? q.nv : q.len;
  if (warp == 0) {
    unsigned long long k = 0ull;
    for (int v = lane; v < q.nv; v += 32) {
      const unsigned long long kv = ((unsigned long long)__double_as_longlong(q.ncur[v]) & ~KEY_POS) | (KEY_POS - (unsigned long long)v);
      k = kv > k ? kv : k;
    }
    q.s_cand[0][lane] = k;
  }
  __syncthreads();
  int keff = 0;
  for (int j = 0; j < kmax; ++j) {
    bool ok = false;
    switch (j >> 4) {
      case 0: ok = qr_step_cached<EPL, 0>(q, j); break;
      case 1: if constexpr (EPL > 1) ok = qr_step_cached<EPL, 1>(q, j); break;
      case 2: if constexpr (EPL > 2) ok = qr_step_cached<EPL, 2>(q, j); break;
      case 3: if constexpr (EPL > 3) ok = qr_step_cached<EPL, 3>(q, j); break;
      case 4: if constexpr (EPL > 4) ok = qr_step_cached<EPL, 4>(q, j); break;
      case 5: if constexpr (EPL > 5) ok = qr_step_cached<EPL, 5>(q, j); break;
      case 6: if constexpr (EPL > 6) ok = qr_step_cached<EPL, 6>(q, j); break;
      default: if constexpr (EPL > 7) ok = qr_step_cached<EPL, 7>(q, j); break;
    }
    if (!ok) break;
    keff = j + 1;
    __syncthreads();
    { double* t = q.ncur; q.ncur = q.nnext; q.nnext = t; short* u = q.pcur; q.pcur = q.pnext; q.pnext = u; }
  }
  return keff;
}

// SMEM: the block lives in shared memory (else in the global scratch); CACHED: rows are at most 16*JAC_EPL long and a
// pair's elements stay in registers between the dot product and the rotation.  A block is handled by exactly one
// instantiation; splitting them keeps the hot loop of the common case small enough for the instruction caches.
// the small work arrays of gram_chol_block are the caller's: its QR path does not run on a block that function finishes
struct GramScratch {
  short *posof, *order, *posphys;          // GC_MAX_NV entries each
  double* rdiag;                           // 2 * GC_MAX_NV
  int* rowoff;                             // GC_MAX_NV
  unsigned long long (*cand)[32];          // [2][32]
};
__device__ bool gram_chol_block(const DecompArgs& a, const DecompBuffers& b, const DecompWork* w, const DecompBlock& B, unsigned char* smem_raw,
                                int gc_elems, double rank_tol, const GramScratch& gs);

template <bool SMEM, bool CACHED>
__global__ void __launch_bounds__(JAC_THREADS) jacobi_blocks_kernel(DecompArgs a, DecompBuffers b, int smem_elems, double rank_tol, int big_on) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_rot, s_keff, s_big;
  __shared__ unsigned long long s_key[3];       // pivot keys of the QR steps j, j+1 and the one being reset (generic path)
  __shared__ unsigned long long s_cand[2][32];  // per half-warp pivot candidates of the steps j, j+1 (cached path)
  __shared__ double s_F;
  __shared__ double s_nrm[JAC_NV_SMEM], s_nrm2[JAC_NV_SMEM], s_nrmref[JAC_NV_SMEM];
  __shared__ double s_rdr[JAC_NV_SMEM], s_rdi[JAC_NV_SMEM];   // diagonal of R
  __shared__ short s_perm[JAC_NV_SMEM], s_permA[JAC_NV_SMEM], s_permB[JAC_NV_SMEM];
  const DecompWork* w = b.dw;
  // the grid is sized from the largest charge seen at upload time: a block table that outgrew it must not go unnoticed
  if (blockIdx.x == 0 && threadIdx.x == 0 && w->nblocks > (int)gridDim.x) atomicOr(b.status, OCMPS_ST_TOOMANYBLK);
  if ((int)blockIdx.x >= w->nblocks) return;
  const DecompBlock B = w->blk[blockIdx.x];
  const int nv = B.nv, len = B.len, ld = w->ld, mode = w->mode;
  const bool fits = nv * len <= smem_elems && nv <= JAC_NV_SMEM;
  // register-cached variant: rows of R at most 16*JAC_EPL long, stored with a zero-padded stride of 16*ceil(nv/16)
  const int ldpad = ((nv + 15) >> 4) << 4;
  const bool can_cache = nv <= 16 * JAC_EPL && (nv < len ? nv : len) * ldpad <= smem_elems;
  if (fits != SMEM || (SMEM && can_cache != CACHED)) return;   // another instantiation handles this block
  const int gram_on = big_on & 2;
  big_on &= 1;
  if (big_on && !(SMEM && CACHED) && nv <= BJ_MAX_ROWS && len <= BJ_MAX_ROWS) return;   // taken by qr_big_kernel (cluster)
  if constexpr (SMEM && CACHED) {
    // gate decompositions: Gram matrix (DMMA) + pivoted Cholesky instead of the Householder QR below (gram_chol_block)
    if (gram_on) {
      const GramScratch gs{s_perm, s_permA, s_permB, s_nrm, reinterpret_cast<int*>(s_nrm2), s_cand};
      if (gram_chol_block(a, b, w, B, smem_raw, smem_elems, rank_tol, gs)) return;
      __syncthreads();
    }
  }
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = JAC_THREADS / 32;
  const int half = lane >> 4, hl = lane & 15;
  cplx* Ya = b.ywork + B.ws_off;                       // region A: final Z (k x nv, physical vector order)
  cplx* Yb = b.ywork + b.ywork_half + B.ws_off;        // region B: transposition scratch
  cplx* Y = SMEM ? reinterpret_cast<cplx*>(smem_raw) : Ya;
  double* nrm = SMEM ? s_nrm : (b.P + B.p_off);        // the fallback keeps its cached norms in global memory
  double* rdr = SMEM ? s_rdr : (b.scratch_d + 2 * B.p_off);
  double* rdi = rdr + (SMEM ? JAC_NV_SMEM : nv);
  if (SMEM) rdi = s_rdi;
  short* perm = SMEM ? s_perm : reinterpret_cast<short*>(b.scratch_d + 4 * NV_MAX) + B.p_off;            // final order
  short* permA = SMEM ? s_permA : reinterpret_cast<short*>(b.scratch_d + 5 * NV_MAX) + B.p_off;          // ping-pong
  short* permB = SMEM ? s_permB : reinterpret_cast<short*>(b.scratch_d + 6 * NV_MAX) + B.p_off;
  double* nrm2 = SMEM ? s_nrm2 : (b.scratch_d + 2 * NV_MAX + B.p_off);
  double* nrmref = SMEM ? s_nrmref : (b.scratch_d + 3 * NV_MAX + B.p_off);
  const int* vidx = b.vec_idx + B.vec_off;
  const int* cidx = b.comp_idx + B.comp_off;

  const long long t_start = clock64();
  // ---- phase 0: gather the block, Y[v][c] = component c of vector v ----
  if (mode == 0) {   // vectors are columns of X: consecutive threads take consecutive vectors (coalesced over columns)
    for (int e = tid; e < nv * len; e += JAC_THREADS) {
      int c = e / nv, v = e % nv;
      Y[v * len + c] = a.X[(size_t)cidx[c] * ld + vidx[v]];
    }
  } else {
    for (int e = tid; e < nv * len; e += JAC_THREADS) {
      int v = e / len, c = e % len;
      Y[v * len + c] = a.X[(size_t)vidx[v] * ld + cidx[c]];
    }
  }
  __syncthreads();
  for (int v = warp; v < nv; v += nwarps) {
    const cplx* y = Y + v * len;
    double s = 0.0;
    for (int c = lane; c < len; c += 32) { cplx u = y[c]; s += u.x * u.x + u.y * u.y; }
    s = warp_sum(s);
    if (lane == 0) { nrm[v] = s; nrmref[v] = s; perm[v] = (short)v; permA[v] = (short)v; }
  }
  __syncthreads();
  if (tid == 0) {
    double t = 0.0;
    for (int v = 0; v < nv; ++v) t += nrm[v];
    s_F = t;
    s_keff = 0;
  }
  __syncthreads();
  const double F = s_F;
  const double rtol_abs = F * rank_tol;

  const long long t_qr0 = clock64();
  // ---- phase 1: Householder QR with column pivoting, in place; R's strict upper part and rdiag remain ----
  // One barrier per step: the trailing norms and the position->slot map are double buffered, so the updates of
  // step j (written to the "next" copies) cannot disturb a warp that is still reading the pivot of step j.
  // Trailing norms are downdated (|y|^2 -= |r_ji|^2) and recomputed exactly only when cancellation has eaten
  // half of the digits since the last exact value (the LAPACK xGEQP3 safeguard); they only SELECT the pivot, the
  // reflector is built from the exact norm of the pivot vector.  The pivot of step j+1 is found while step j
  // updates the norms: every update does an atomicMax on a (norm bits | position) key.
  const int kmax = nv < len ? nv : len;
  int keff = 0;
  double* ncur = nrm;  double* nnext = nrm2;
  short* pcur = permA; short* pnext = permB;
  constexpr unsigned long long KEY_POS = 2047ull;        // low 11 bits: 2047 - position (ties -> smaller position)
  const bool qr_cached = CACHED && len <= 16 * JAC_EPL;
  if (qr_cached) {
    QrState q;
    q.Y = Y; q.nv = nv; q.len = len; q.rtol_abs = rtol_abs;
    q.ncur = ncur; q.nnext = nnext; q.nrmref = nrmref; q.rdr = rdr; q.rdi = rdi;
    q.perm = perm; q.pcur = pcur; q.pnext = pnext; q.s_cand = s_cand;
    switch ((len + 15) >> 4) {
      case 1: keff = qr_pivoted_cached<1>(q); break;
      case 2: keff = qr_pivoted_cached<2>(q); break;
      case 3: keff = qr_pivoted_cached<3>(q); break;
      case 4: keff = qr_pivoted_cached<4>(q); break;
      case 5: keff = qr_pivoted_cached<5>(q); break;
      case 6: keff = qr_pivoted_cached<6>(q); break;
      case 7: keff = qr_pivoted_cached<7>(q); break;
      default: keff = qr_pivoted_cached<8>(q); break;
    }
    ncur = q.ncur; nnext = q.nnext; pcur = q.pcur; pnext = q.pnext;
  }
  if (tid < 3) s_key[tid] = 0ull;
  __syncthreads();
  for (int v = tid; v < nv; v += JAC_THREADS)
    atomicMax(&s_key[0], ((unsigned long long)__double_as_longlong(nrm[v]) & ~KEY_POS) | (KEY_POS - (unsigned long long)v));
  __syncthreads();
  for (int j = 0; j < (qr_cached ? 0 : kmax); ++j) {
    const int bpos = (int)(KEY_POS - (s_key[j % 3] & KEY_POS));
    if (tid == 0) s_key[(j + 2) % 3] = 0ull;   // read last in step j-1, written next in step j+1
    const int pv = pcur[bpos];             // physical slot of the pivot vector
    const int pj = pcur[j];
    const cplx* x = Y + pv * len;          // Householder vector: x[j..len), with x[j] replaced by v0
    unsigned long long* knext = &s_key[(j + 1) % 3];
    {
    // generic path: every warp computes the exact norm of the pivot vector
    double sq = 0.0;
    for (int c = j + lane; c < len; c += 32) { const cplx u = x[c]; sq += u.x * u.x + u.y * u.y; }
    const double best = warp_sum(sq);
    if (!(best > rtol_abs)) break;
    keff = j + 1;
    const cplx alpha = x[j];
    const double inx = rsqrt(best), normx = best * inx;
    const double a2 = alpha.x * alpha.x + alpha.y * alpha.y;
    const double ia = a2 > 0.0 ? rsqrt(a2) : 0.0, aabs = a2 * ia;
    const double phr = a2 > 0.0 ? alpha.x * ia : 1.0, phi = a2 > 0.0 ? alpha.y * ia : 0.0;
    const double v0r = alpha.x + phr * normx, v0i = alpha.y + phi * normx;
    const double rb = rsqrt(normx * (normx + aabs));
    const double beta = rb * rb;
    if (tid == 0) { rdr[j] = -phr * normx; rdi[j] = -phi * normx; perm[j] = (short)pv; }   // R_jj; final position j
    for (int ib = j + 1 + 2 * warp; ib < nv; ib += 2 * nwarps) {
      const int i = ib + half;
      const bool act = i < nv;
      const int phys = act ? (i == bpos ? pj : (int)pcur[i]) : pv;
      cplx* y = Y + phys * len;
      double wr = 0.0, wi = 0.0;
      if (act) {
        for (int c = j + hl; c < len; c += 16) {
          cplx vv = x[c];
          if (c == j) { vv.x = v0r; vv.y = v0i; }
          const cplx yy = y[c];
          wr += vv.x * yy.x + vv.y * yy.y;      // conj(v) * y
          wi += vv.x * yy.y - vv.y * yy.x;
        }
      }
      wr = half_sum(wr); wi = half_sum(wi);
      double rji2 = 0.0;
      if (act) {
        const double fr = beta * wr, fi = beta * wi;
        for (int c = j + hl; c < len; c += 16) {
          cplx vv = x[c];
          if (c == j) { vv.x = v0r; vv.y = v0i; }
          cplx yy = y[c];
          yy.x -= fr * vv.x - fi * vv.y;
          yy.y -= fr * vv.y + fi * vv.x;
          y[c] = yy;
          if (c == j) rji2 = yy.x * yy.x + yy.y * yy.y;
        }
      }
      rji2 = __shfl_sync(0xffffffffu, rji2, lane & 16);        // component j is owned by lane 0 of the half-warp
      double tnew = 0.0;
      bool redo = false;
      if (act) {
        tnew = ncur[phys] - rji2;
        redo = !(tnew > 1.5e-8 * nrmref[phys]);
      }
      if (__any_sync(0xffffffffu, redo)) {     // rare: exact trailing norm
        double tail = 0.0;
        if (act && redo) for (int c = j + 1 + hl; c < len; c += 16) { const cplx yy = y[c]; tail += yy.x * yy.x + yy.y * yy.y; }
        tail = half_sum(tail);
        if (act && redo) { tnew = tail; if (hl == 0) nrmref[phys] = tail; }
      }
      if (act && hl == 0) {
        tnew = tnew > 0.0 ? tnew : 0.0;
        nnext[phys] = tnew; pnext[i] = (short)phys;
        atomicMax(knext, ((unsigned long long)__double_as_longlong(tnew) & ~KEY_POS) | (KEY_POS - (unsigned long long)i));
      }
    }
    }
    __syncthreads();
    { double* t = ncur; ncur = nnext; nnext = t; short* u = pcur; pcur = pnext; pnext = u; }
  }
  for (int i = keff + tid; i < nv; i += JAC_THREADS) perm[i] = pcur[i];     // positions past the numerical rank
  __syncthreads();
  if (tid == 0) s_keff = keff;

  // ---- phase 2: R (keff x nv, position order) -> row-major scratch -> back as the Jacobi working set ----
  const int ldz = CACHED ? ldpad : nv;            // row stride of the Jacobi working set (padding is zero)
  for (int e = tid; e < keff * ldz; e += JAC_THREADS) {
    const int c = e / ldz, i = e % ldz;
    cplx v = make_double2(0.0, 0.0);
    if (i == c) v = make_double2(rdr[c], rdi[c]);
    else if (i > c && i < nv) v = Y[(int)perm[i] * len + c];
    Yb[e] = v;
  }
  __syncthreads();
  {
    // hand-over: blocks whose R has at most JAC_BLOCKED_ROWS rows are finished by jacobi_rot_kernel (register-resident
    // rows; a kernel of its own so that its register allocation is not shared with the QR phase)
    double* hF = b.scratch_d + 7 * NV_MAX;
    int* hK = reinterpret_cast<int*>(b.scratch_d + 7 * NV_MAX + OCMPS_MAX_BLK);
    // blocks with more rows (or longer rows) than that go to the cluster kernel jacobi_big_kernel when it is launched
    // (big_on): R distributed by columns over a thread-block cluster, up to 256 rows of up to 256 columns
    int* hB = hK + OCMPS_MAX_BLK;
    int* hS = hB + OCMPS_MAX_BLK;
    const bool handover_small = CACHED && keff <= JAC_BLOCKED_ROWS;
    const bool handover_big = !handover_small && big_on && keff <= BJ_MAX_ROWS && nv <= BJ_MAX_ROWS;
    const bool handover = handover_small || handover_big;
    if (tid == 0) {
      hF[blockIdx.x] = F;
      hK[blockIdx.x] = handover_small ? keff : -1;
      hB[blockIdx.x] = handover_big ? keff : -1;
      hS[blockIdx.x] = ldz;
    }
    if (handover) {
      short* gperm = reinterpret_cast<short*>(b.scratch_d + 4 * NV_MAX) + B.p_off;
      for (int i = tid; i < nv; i += JAC_THREADS) gperm[i] = perm[i];
      if (tid == 0) {
        const double nn = (double)len, mmv = (double)nv;
        atomicAdd(&g_jac_flops[0], 8.0 * nn * nn * mmv + (56.0 / 3.0) * nn * nn * nn);
        if (blockIdx.x == 0) {
          const double dn = mode == 0 ? (double)w->n : (double)w->m, dm = mode == 0 ? (double)w->m : (double)w->n;
          atomicAdd(&g_jac_flops[1], 8.0 * dn * dn * dm + (56.0 / 3.0) * dn * dn * dn);
        }
        if (nv >= 64) {
          const long long t_now = clock64();
          atomicAdd(&g_jac_dbg[5], (unsigned long long)(t_now - t_qr0));
          atomicAdd(&g_jac_dbg[7], (unsigned long long)(t_now - t_start));
        }
      }
      return;
    }
  }
  cplx* Z = SMEM ? Y : Yb;
  if (SMEM) {
    for (int e = tid; e < keff * ldz; e += JAC_THREADS) Z[e] = Yb[e];
    __syncthreads();
  }

  const long long t_jac0 = clock64();
  // ---- phase 3: one-sided Jacobi on the keff rows of R (length nv each) ----
  const int npad = (keff + 1) & ~1;
  const int npairs = npad / 2;
  const double thr = F * DEFLATE_REL;
  constexpr bool cached = CACHED;
  const int epl = (nv + 15) >> 4;                  // elements per lane of a row
  bool converged = false;
  for (int sweep = 0; sweep < JAC_MAX_SWEEPS && !converged; ++sweep) {
    for (int v = warp; v < keff; v += nwarps) {        // exact Gram diagonal at the start of every sweep
      const cplx* y = Z + v * ldz;
      double s = 0.0;
      for (int c = lane; c < nv; c += 32) { cplx u = y[c]; s += u.x * u.x + u.y * u.y; }
      s = warp_sum(s);
      if (lane == 0) nrm[v] = s;
    }
    if (tid == 0) { s_rot = 0; s_big = 0; }
    __syncthreads();
    if (keff < 2) break;
    for (int r = 0; r < npad - 1; ++r) {
      for (int kb = 2 * warp; kb < npairs; kb += 2 * nwarps) {     // warp-uniform trip count
        const int k = kb + half;
        // round-robin pairing without integer division: p = (r + k) mod (npad-1), q = (r - k) mod (npad-1); r, k < npad-1
        int p = r + k; if (p >= npad - 1) p -= npad - 1;
        int q = r - k; if (q < 0) q += npad - 1;
        if (k == 0) q = npad - 1;
        const bool act = (k < npairs) && p < keff && q < keff;
        if (p > q) { int tmp = p; p = q; q = tmp; }
        cplx* yp = Z + (act ? p : 0) * ldz;
        cplx* yq = Z + (act ? q : 0) * ldz;
        double cre = 0.0, cim = 0.0;
        cplx ru[JAC_EPL], rv[JAC_EPL];                 // the pair's elements stay in registers between dot and update
        if (act) {
          if (cached) {
            // epl = ceil(nv / 16) is uniform: the guards below are branches, so unused slots issue nothing
            // (the FP64 pipe, 2 cycles per warp instruction and 23 cycles of latency, is what bounds a round)
            double c0r = 0.0, c0i = 0.0, c1r = 0.0, c1i = 0.0;
#pragma unroll
            for (int e = 0; e < JAC_EPL; ++e) {
              if (e >= epl) break;
              const int c = hl + 16 * e;
              ru[e] = yp[c]; rv[e] = yq[c];                       // the padding of a row is zero
              const double pr = ru[e].x * rv[e].x + ru[e].y * rv[e].y;      // conj(u) * v
              const double pi = ru[e].x * rv[e].y - ru[e].y * rv[e].x;
              if (e & 1) { c1r += pr; c1i += pi; } else { c0r += pr; c0i += pi; }
            }
            cre = c0r + c1r; cim = c0i + c1i;
          } else {
            for (int c = hl; c < nv; c += 16) {
              cplx u = yp[c], v = yq[c];
              cre += u.x * v.x + u.y * v.y;
              cim += u.x * v.y - u.y * v.x;
            }
          }
        }
        cre = half_sum(cre); cim = half_sum(cim);
        if (!act) continue;
        const double aa = nrm[p], bb = nrm[q];
        const double c2 = cre * cre + cim * cim;
        if (aa <= thr || bb <= thr) {
          if (aa <= thr && aa > 0.0) { for (int c = hl; c < nv; c += 16) yp[c] = make_double2(0.0, 0.0); if (hl == 0) nrm[p] = 0.0; }
          if (bb <= thr && bb > 0.0) { for (int c = hl; c < nv; c += 16) yq[c] = make_double2(0.0, 0.0); if (hl == 0) nrm[q] = 0.0; }
        } else if (c2 > JAC_TOL2 * aa * bb) {
          // rotation angle theta: tan 2theta = |c| / d, d = (b - a)/2.  Two reciprocal square roots give
          // cos and sin without a division: cos^2 = (1 + |cos 2theta|)/2, sin = sin 2theta / (2 cos).
          const double inv_r = rsqrt(c2);
          const double rr = c2 * inv_r;                         // |c|
          const double dd = 0.5 * (bb - aa);
          const double ih = rsqrt(dd * dd + c2);
          const double cs2 = 0.5 + 0.5 * fabs(dd) * ih;
          const double ics = rsqrt(cs2);
          const double cs = cs2 * ics;
          const double snm = 0.5 * rr * ih * ics;
          const double sn = dd >= 0.0 ? snm : -snm;
          const double phr = cre * inv_r, phi = cim * inv_r;    // e^{i phi} = c / |c|, absorbed into vector q
          if (cached) {
#pragma unroll
            for (int e = 0; e < JAC_EPL; ++e) {
              if (e >= epl) break;
              const int c = hl + 16 * e;
              const double vx = phr * rv[e].x + phi * rv[e].y, vy = phr * rv[e].y - phi * rv[e].x;
              yp[c] = make_double2(cs * ru[e].x - sn * vx, cs * ru[e].y - sn * vy);
              yq[c] = make_double2(sn * ru[e].x + cs * vx, sn * ru[e].y + cs * vy);
            }
          } else {
            for (int c = hl; c < nv; c += 16) {
              const cplx u = yp[c], v = yq[c];
              const double vx = phr * v.x + phi * v.y, vy = phr * v.y - phi * v.x;
              yp[c] = make_double2(cs * u.x - sn * vx, cs * u.y - sn * vy);
              yq[c] = make_double2(sn * u.x + cs * vx, sn * u.y + cs * vy);
            }
          }
          if (hl == 0) {
            const double trr = sn * ics * rr;                   // tan(theta) |c|
            const double na = aa - trr, nb = bb + trr;
            nrm[p] = na > 0.0 ? na : 0.0;
            nrm[q] = nb > 0.0 ? nb : 0.0;
            s_rot = 1;
            if (c2 > 1e-16 * aa * bb) s_big = 1;                // an off-diagonal above 1e-8 (relative) was seen
          }
        }
      }
      __syncthreads();
    }
    // quadratic convergence: if every rotated pair had |<p|q>| < 1e-8 |p||q|, the residuals are now ~1e-16
    converged = (s_rot == 0) || (s_big == 0);
    if (tid == 0) { atomicAdd(&g_jac_dbg[0], 1ull); atomicMax(&g_jac_dbg[2], (unsigned long long)(sweep + 1)); if (nv >= 64) atomicAdd(&g_jac_dbg[3], 1ull); if (nv >= 64 && sweep == 0) atomicAdd(&g_jac_dbg[4], 1ull); }
    __syncthreads();
    if (!converged && sweep == JAC_MAX_SWEEPS - 1 && tid == 0) atomicOr(b.status, OCMPS_ST_NOCONV);
  }
  if (tid == 0) {
    atomicAdd(&g_jac_dbg[1], 1ull);
    // SURVEY 8d: F_gram = 8 n^2 m, F_evd = 56/3 n^3 with n the side that is orthogonalised (here per charge block)
    const double nn = (double)len, mm = (double)nv;
    atomicAdd(&g_jac_flops[0], 8.0 * nn * nn * mm + (56.0 / 3.0) * nn * nn * nn);
    if (blockIdx.x == 0) {
      const double dn = mode == 0 ? (double)w->n : (double)w->m, dm = mode == 0 ? (double)w->m : (double)w->n;
      atomicAdd(&g_jac_flops[1], 8.0 * dn * dn * dm + (56.0 / 3.0) * dn * dn * dn);
    }
  }

  // ---- phase 4: spectrum + normalised right vectors Z[j][physical vector] ----
  __syncthreads();
  const long long t_jac1 = clock64();
#ifdef OCMPS_JAC_TRACE
  if (tid == 0 && nv >= 24)
    printf("JT kind %d blk %d nv %d len %d keff %d qr %lld jac %lld tot %lld\n", a.kind, (int)blockIdx.x, nv, len, s_keff,
           t_jac0 - t_qr0, t_jac1 - t_jac0, t_jac1 - t_start);
#endif
  if (tid == 0 && nv >= 64) {
    atomicAdd(&g_jac_dbg[5], (unsigned long long)(t_jac0 - t_qr0));
    atomicAdd(&g_jac_dbg[6], (unsigned long long)(t_jac1 - t_jac0));
    atomicAdd(&g_jac_dbg[7], (unsigned long long)(t_jac1 - t_start));
  }
  for (int v = warp; v < nv; v += nwarps) {
    if (v < keff) {
      const cplx* y = Z + v * ldz;
      double s = 0.0;
      for (int c = lane; c < nv; c += 32) { cplx u = y[c]; s += u.x * u.x + u.y * u.y; }
      s = warp_sum(s);
      const double inv = s > 0.0 ? rsqrt(s) : 0.0;
      for (int c = lane; c < nv; c += 32) {
        cplx u = y[c];
        Ya[v * nv + (int)perm[c]] = make_double2(u.x * inv, u.y * inv);
      }
      __syncwarp();
      if (lane == 0) b.P[B.p_off + v] = s;
    } else if (lane == 0) {
      b.P[B.p_off + v] = 0.0;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Gate decompositions, first half: Gram matrix on the FP64 tensor cores + pivoted Cholesky (instead of the Householder QR)
// ------------------------------------------------------------------------------------------------
// The reference truncates with denmatDecomp, i.e. it diagonalises the Gram matrix theta.theta^H of every charge block
// (SURVEY A.2); a spectrum that is exact relative to the block's weight (absolute accuracy ~1e-16 F) is therefore all
// the reference itself has.  For the gate decompositions the triangular factor the Jacobi rotations work on is obtained
// the same way here: G = <v_i|v_j> of the block's vectors is accumulated with DMMA (mma.sync m8n8k4.f64, 4 real products
// per complex k4-step) straight from the gathered block in shared memory, and a Cholesky factorisation with diagonal
// pivoting G = R^H R yields the same R (rows in pivot order, trailing weight test on the pivot) the Householder QR with
// column pivoting would: 62 left-looking steps of one barrier each (every warp finds the pivot redundantly from the running
// diagonal; four lanes per vector form its entry of the new row of R from the earlier rows, which are kept in the dead rows of G)
// instead of 62 Householder steps of ~4 kclk.  The centre moves (psi.position(), Cutoff 1e-16) keep the QR: their
// rank decisions sit at the rounding level of a Gram matrix.  The code is a branch of jacobi_blocks_kernel<true, true> (a kernel of
// its own cost a launch per decomposition and a third of the throughput of 48 concurrent chains: every CTA of these kernels
// needs a whole SM); a block it cannot take -- more than 96 vectors, more than JAC_BLOCKED_ROWS rows of R -- falls through to the QR.
// Opt-in (OCMPS_GRAM=1): parity-green on the whole GPU suite, but not faster than the QR where it matters (see launch_jacobi_blocks).
// Returns true if the block was finished (R, permutation and hand-over entries written), false if it has to take the QR path:
// more than GC_MAX_NV vectors, a shape that does not fit the shared memory of this launch, or more than JAC_BLOCKED_ROWS rows of R.
__device__ bool gram_chol_block(const DecompArgs& a, const DecompBuffers& b, const DecompWork* w, const DecompBlock& B, unsigned char* smem_raw,
                                int gc_elems, double rank_tol, const GramScratch& gs) {
  short* const s_posof = gs.posof; short* const s_order = gs.order; short* const s_posphys = gs.posphys;
  double* const s_rdiag = gs.rdiag;
  int* const s_rowoff = gs.rowoff;
  unsigned long long (*const s_cand)[32] = gs.cand;
  const int nv = B.nv, len = B.len, ld = w->ld, mode = w->mode;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double* hF = b.scratch_d + 7 * NV_MAX;
  int* hK = reinterpret_cast<int*>(b.scratch_d + 7 * NV_MAX + OCMPS_MAX_BLK);
  int* hB = hK + OCMPS_MAX_BLK;
  int* hS = hB + OCMPS_MAX_BLK;
  const int nvp = (nv + 7) & ~7, ldy = gc_ldy(len), ldg = gc_ldg(nvp);
  // Small blocks stay with the QR: its steps are cheaper there (measured: with every block on this path 48 concurrent chains lose a
  // fifth of their throughput and the L=5 configuration 8 %), and only the largest blocks of a decomposition set its latency.
  if (nv > GC_MAX_NV || (nv < len ? nv : len) < GC_MIN_RANK || nvp * ldy > gc_elems || nvp * ldg > gc_elems) return false;
  const long long t_start = clock64();
  cplx* Y = reinterpret_cast<cplx*>(smem_raw);         // gathered block, Y[v][c], rows padded to nvp, components to a multiple of 4
  cplx* G = Y;                                          // the Gram matrix takes the place of the block once it is accumulated
  const int* vidx = b.vec_idx + B.vec_off;
  const int* cidx = b.comp_idx + B.comp_off;
  const int len4 = (len + 3) & ~3;
  for (int e = tid; e < nvp * ldy; e += JAC_THREADS) Y[e] = make_double2(0.0, 0.0);
  __syncthreads();
  if (mode == 0) {
    for (int e = tid; e < nv * len; e += JAC_THREADS) {
      const int c = e / nv, v = e % nv;
      Y[v * ldy + c] = a.X[(size_t)cidx[c] * ld + vidx[v]];
    }
  } else {
    for (int e = tid; e < nv * len; e += JAC_THREADS) {
      const int v = e / len, c = e % len;
      Y[v * ldy + c] = a.X[(size_t)vidx[v] * ld + cidx[c]];
    }
  }
  for (int i = tid; i < GC_MAX_NV; i += JAC_THREADS) s_posof[i] = -1;
  __syncthreads();
  // ---- Gram matrix, upper triangle of 8x8 tiles; the accumulators stay in registers until every warp is done with Y ----
  const int nt = nvp >> 3, ntiles = nt * (nt + 1) / 2;
  const int g = lane >> 2, t = lane & 3;
  double acc[GC_TILES_PER_WARP][4];
  auto tile_of = [&](int e, int& ti, int& tj) { ti = 0; while (e >= nt - ti) { e -= nt - ti; ++ti; } tj = ti + e; };
#pragma unroll
  for (int sl = 0; sl < GC_TILES_PER_WARP; ++sl) {
    acc[sl][0] = acc[sl][1] = acc[sl][2] = acc[sl][3] = 0.0;
    const int e = warp + (JAC_THREADS / 32) * sl;
    if (e < ntiles) {
      int ti, tj;
      tile_of(e, ti, tj);
      const cplx* ya = Y + (ti * 8 + g) * ldy + t;
      const cplx* yb = Y + (tj * 8 + g) * ldy + t;
      double cr0 = 0.0, cr1 = 0.0, ci0 = 0.0, ci1 = 0.0;
      for (int k4 = 0; k4 < len4; k4 += 4) {
        const cplx av = ya[k4], bv = yb[k4];
        gc_dmma(cr0, cr1, av.x, bv.x);                 // Re: yr yr' + yi yi'
        gc_dmma(cr0, cr1, av.y, bv.y);
        gc_dmma(ci0, ci1, av.x, bv.y);                 // Im: yr yi' - yi yr'
        gc_dmma(ci0, ci1, -av.y, bv.x);
      }
      acc[sl][0] = cr0; acc[sl][1] = cr1; acc[sl][2] = ci0; acc[sl][3] = ci1;
    }
  }
  __syncthreads();
#pragma unroll
  for (int sl = 0; sl < GC_TILES_PER_WARP; ++sl) {
    const int e = warp + (JAC_THREADS / 32) * sl;
    if (e < ntiles) {
      int ti, tj;
      tile_of(e, ti, tj);
      cplx* gp = G + (ti * 8 + g) * ldg + tj * 8 + 2 * t;
      gp[0] = make_double2(acc[sl][0], acc[sl][2]);
      gp[1] = make_double2(acc[sl][1], acc[sl][3]);
    }
  }
  __syncthreads();
  // block weight F = trace(G): the same bits in every warp (fixed order)
  double F;
  {
    double part = 0.0;
    for (int i = lane; i < nv; i += 32) part += G[i * ldg + i].x;
    F = warp_sum(part);
  }
  const double rtol_abs = F * (rank_tol > 1e-15 ? rank_tol : 1e-15);      // a Gram matrix resolves nothing below ~1e-16 F
  const long long t_qr0 = clock64();
  // ---- Cholesky with diagonal pivoting, left-looking; vectors keep their physical index ----
  // Step j: every warp finds the pivot p (largest remaining diagonal) redundantly; row j of R,
  //   r_j[c] = (G[p][c] - sum_{m<j} conj(R[m][p]) R[m][c]) / sqrt(d_p)     for the vectors c still in play,
  // is computed by four lanes per vector (every fourth earlier row each) and stored IN the row p of G: that row and the
  // column p are dead from now on (G itself is never updated, only the diagonal d is downdated), and what later steps
  // need of G -- row / column p' of the vectors still in play -- lives in rows that have not been overwritten.
  constexpr unsigned long long KEY_POS = 2047ull;
  const int kmax = nv < len ? nv : len;
  double* dgl = s_rdiag + GC_MAX_NV;                     // running diagonal d[i] (second half of s_rdiag)
  const int col = tid >> 2, sub = tid & 3;               // vector of this lane group, its share of the earlier rows
  const bool has_cols = warp * 8 < nv;                   // (warp uniform) warps without vectors only follow the pivots
  bool alive = col < nv;
  double dcol = 0.0;
  auto key_of = [&](double dd, int i) -> unsigned long long {
    return dd > 0.0 ? (((unsigned long long)__double_as_longlong(dd) & ~KEY_POS) | (KEY_POS - (unsigned long long)i)) : 0ull;
  };
  // pivot candidates: the best (diagonal bits | 2047 - index) key of every warp's vectors, double buffered over the steps
  auto publish = [&](int buf, unsigned long long key) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { const unsigned long long k2 = __shfl_xor_sync(0xffffffffu, key, o); key = k2 > key ? k2 : key; }
    if (lane == 0) s_cand[buf][warp] = key;
  };
  if (alive && sub == 0) { dcol = G[col * ldg + col].x; dgl[col] = dcol; }
  if (has_cols) publish(0, (alive && sub == 0) ? key_of(dcol, col) : 0ull);
  else if (lane == 0) { s_cand[0][warp] = 0ull; s_cand[1][warp] = 0ull; }
  __syncthreads();
  int keff = 0;
#ifdef OCMPS_JAC_TRACE
  long long tg[7] = {0, 0, 0, 0, 0, 0, 0};
  long long tgl = clock64();
#define GC_MARK(i) { const long long tn = clock64(); tg[i] += tn - tgl; tgl = tn; }
#else
#define GC_MARK(i)
#endif
  for (int j = 0; j < kmax; ++j) {
    unsigned long long key = lane < JAC_THREADS / 32 ? s_cand[j & 1][lane] : 0ull;
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) { const unsigned long long k2 = __shfl_xor_sync(0xffffffffu, key, o); key = k2 > key ? k2 : key; }
    key = __shfl_sync(0xffffffffu, key, 0);
    GC_MARK(5)
    if (key == 0ull) break;
    const int p = (int)(KEY_POS - (key & KEY_POS));
    const double dp = dgl[p];
    if (!(dp > rtol_abs)) break;                        // numerical rank reached (uniform: every warp sees the same bits)
    keff = j + 1;
    GC_MARK(6)
    if (tid == 0) { s_order[j] = (short)p; s_rowoff[j] = p * ldg; s_posof[p] = (short)j; }
    GC_MARK(0)
    if (has_cols) {
      const double inv = rsqrt(dp);
      if (tid == 0) s_rdiag[j] = dp * inv;
      if (col == p) alive = false;
      GC_MARK(1)
      double sr = 0.0, si = 0.0;
      if (alive) {
        // four earlier rows in flight per lane (the loads of one row depend on nothing but the row offset)
        for (int m = sub; m < j; m += 16) {
          cplx x[4], y[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int mm = m + 4 * q;
            x[q] = make_double2(0.0, 0.0); y[q] = make_double2(0.0, 0.0);
            if (mm < j) { const cplx* rrow = G + s_rowoff[mm]; x[q] = rrow[p]; y[q] = rrow[col]; }
          }
          double ar = 0.0, ai = 0.0, br = 0.0, bi = 0.0;
          ar += x[0].x * y[0].x + x[0].y * y[0].y;  ai += x[0].x * y[0].y - x[0].y * y[0].x;     // conj(R[m][p]) R[m][c]
          br += x[1].x * y[1].x + x[1].y * y[1].y;  bi += x[1].x * y[1].y - x[1].y * y[1].x;
          ar += x[2].x * y[2].x + x[2].y * y[2].y;  ai += x[2].x * y[2].y - x[2].y * y[2].x;
          br += x[3].x * y[3].x + x[3].y * y[3].y;  bi += x[3].x * y[3].y - x[3].y * y[3].x;
          sr += ar + br; si += ai + bi;
        }
      }
      sr += __shfl_xor_sync(0xffffffffu, sr, 1); si += __shfl_xor_sync(0xffffffffu, si, 1);
      sr += __shfl_xor_sync(0xffffffffu, sr, 2); si += __shfl_xor_sync(0xffffffffu, si, 2);
      GC_MARK(2)
      unsigned long long mykey = 0ull;
      if (alive && sub == 0) {
        const cplx gv = col > p ? G[p * ldg + col] : G[col * ldg + p];
        const double gr = gv.x, gi = col > p ? gv.y : -gv.y;
        const double rr = (gr - sr) * inv, ri = (gi - si) * inv;
        G[p * ldg + col] = make_double2(rr, ri);
        const double dn = dcol - (rr * rr + ri * ri);
        dcol = dn > 0.0 ? dn : 0.0;
        dgl[col] = dcol;
        mykey = key_of(dcol, col);
      }
      publish((j + 1) & 1, mykey);
      GC_MARK(3)
    }
    __syncthreads();
    GC_MARK(4)
  }
  __syncthreads();
#ifdef OCMPS_JAC_TRACE
  if (tid == 0 && nv >= 64 && keff > 0)
    printf("JTC nv %d keff %d per step: candidates %lld diagonal %lld bookkeeping %lld rsqrt %lld dot+reduce %lld tail+publish %lld barrier %lld\n", nv, keff,
           tg[5] / keff, tg[6] / keff, tg[0] / keff, tg[1] / keff, tg[2] / keff, tg[3] / keff, tg[4] / keff);
#endif
  if (keff > JAC_BLOCKED_ROWS) return false;            // more rows than the register-resident rotations take: the QR path redoes the block
  // positions: picked vectors in pivot order, then the rest in index order
  if (tid == 0) {
    for (int j = 0; j < keff; ++j) s_posphys[j] = s_order[j];
    int q = keff;
    for (int i = 0; i < nv; ++i) if (s_posof[i] < 0) s_posphys[q++] = (short)i;
  }
  __syncthreads();
  // ---- R (keff x nv, position order, zero-padded stride) -> the Jacobi working set ----
  const int ldz = ((nv + 15) >> 4) << 4;
  cplx* Yb = b.ywork + b.ywork_half + B.ws_off;
  for (int e = tid; e < keff * ldz; e += JAC_THREADS) {
    const int c = e / ldz, pos = e % ldz;
    cplx v = make_double2(0.0, 0.0);
    if (pos == c) v = make_double2(s_rdiag[c], 0.0);
    else if (pos > c && pos < nv) v = G[(int)s_order[c] * ldg + (int)s_posphys[pos]];
    Yb[e] = v;
  }
  short* gperm = reinterpret_cast<short*>(b.scratch_d + 4 * NV_MAX) + B.p_off;
  for (int i = tid; i < nv; i += JAC_THREADS) gperm[i] = s_posphys[i];
  if (tid == 0) {
    hF[blockIdx.x] = F;
    hK[blockIdx.x] = keff;
    hB[blockIdx.x] = -1;
    hS[blockIdx.x] = ldz;
    const double nn = (double)len, mmv = (double)nv;
    atomicAdd(&g_jac_flops[0], 8.0 * nn * nn * mmv + (56.0 / 3.0) * nn * nn * nn);
    if (blockIdx.x == 0) {
      const double dn = mode == 0 ? (double)w->n : (double)w->m, dm = mode == 0 ? (double)w->m : (double)w->n;
      atomicAdd(&g_jac_flops[1], 8.0 * dn * dn * dm + (56.0 / 3.0) * dn * dn * dn);
    }
    if (nv >= 64) {
      const long long t_now = clock64();
      atomicAdd(&g_jac_dbg[5], (unsigned long long)(t_now - t_qr0));
      atomicAdd(&g_jac_dbg[7], (unsigned long long)(t_now - t_start));
#ifdef OCMPS_JAC_TRACE
      printf("JTG kind %d blk %d nv %d len %d keff %d gather+gram %lld cholesky+out %lld\n", a.kind, (int)blockIdx.x, nv, len, keff,
             (long long)(t_qr0 - t_start), (long long)(t_now - t_qr0));
#endif
    }
  }
  return true;
}

// Rows of R handed over for the register-resident second stage by jacobi_blocks_kernel<true, true>, or -1 if the block is not
// finished by that stage.  Only blocks of the register-cached first stage hand over to it; the hand-over entries of the others
// may still be in the making on the cluster stream (launch_jacobi_blocks), so they are told apart by their shape.
__device__ __forceinline__ int rot_handover_rows(const DecompBuffers& b, int blk, int smem_elems) {
  const DecompWork* w = b.dw;
  if (blk >= w->nblocks) return -1;
  const int nv0 = w->blk[blk].nv, len0 = w->blk[blk].len;
  const bool fits = nv0 * len0 <= smem_elems && nv0 <= JAC_NV_SMEM;
  const int ldpad = ((nv0 + 15) >> 4) << 4;
  const bool can_cache = nv0 <= 16 * JAC_EPL && (nv0 < len0 ? nv0 : len0) * ldpad <= smem_elems;
  if (!(fits && can_cache)) return -1;
  return reinterpret_cast<const int*>(b.scratch_d + 7 * NV_MAX + OCMPS_MAX_BLK)[blk];
}

// Second half of the block decomposition for the blocks handed over by jacobi_blocks_kernel<true, true>: one-sided
// Jacobi on the rows of R with the rows held in registers (jacobi_sweep_blocked), then spectrum and right vectors.
// One CTA of JAC_THREADS per block (block `blk`, keff rows of R).
__device__ __forceinline__ void jacobi_rot_block(const DecompArgs& a, const DecompBuffers& b, int blk, int keff, unsigned char* smem_raw) {
  __shared__ int s_rot, s_big;
  __shared__ double s_nrm[JAC_BLOCKED_ROWS];
  const DecompWork* w = b.dw;
  const DecompBlock B = w->blk[blk];
  const int nv = B.nv;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = JAC_THREADS / 32;
  const int epl = (nv + 15) >> 4, ldz = epl << 4;
  const double F = (b.scratch_d + 7 * NV_MAX)[blk];
  const double thr = F * DEFLATE_REL;
  const short* perm = reinterpret_cast<const short*>(b.scratch_d + 4 * NV_MAX) + B.p_off;
  cplx* Ya = b.ywork + B.ws_off;
  const cplx* Yb = b.ywork + b.ywork_half + B.ws_off;
  cplx* Z = reinterpret_cast<cplx*>(smem_raw);
  double* nrm = s_nrm;
  const long long t_jac0 = clock64();
  for (int e = tid; e < keff * ldz; e += JAC_THREADS) Z[e] = Yb[e];
  __syncthreads();
  bool converged = false;
  for (int sweep = 0; sweep < JAC_MAX_SWEEPS && !converged; ++sweep) {
    for (int v = warp; v < keff; v += nwarps) {        // exact Gram diagonal at the start of every sweep
      const cplx* y = Z + v * ldz;
      double s = 0.0;
      for (int c = lane; c < nv; c += 32) { cplx u = y[c]; s += u.x * u.x + u.y * u.y; }
      s = warp_sum(s);
      if (lane == 0) nrm[v] = s;
    }
    if (tid == 0) { s_rot = 0; s_big = 0; }
    __syncthreads();
    if (keff < 2) break;
    switch (epl) {
      case 1: jacobi_sweep_blocked<1>(Z, keff, nrm, thr, &s_rot, &s_big); break;
      case 2: jacobi_sweep_blocked<2>(Z, keff, nrm, thr, &s_rot, &s_big); break;
      case 3: jacobi_sweep_blocked<3>(Z, keff, nrm, thr, &s_rot, &s_big); break;
      case 4: jacobi_sweep_blocked<4>(Z, keff, nrm, thr, &s_rot, &s_big); break;
      case 5: jacobi_sweep_blocked<5>(Z, keff, nrm, thr, &s_rot, &s_big); break;
      case 6: jacobi_sweep_blocked<6>(Z, keff, nrm, thr, &s_rot, &s_big); break;
      case 7: jacobi_sweep_blocked<7>(Z, keff, nrm, thr, &s_rot, &s_big); break;
      default: jacobi_sweep_blocked<8>(Z, keff, nrm, thr, &s_rot, &s_big); break;
    }
    // quadratic convergence: if every rotated pair had |<p|q>| < 1e-8 |p||q|, the residuals are now ~1e-16
    converged = (s_rot == 0) || (s_big == 0);
    if (tid == 0) { atomicAdd(&g_jac_dbg[0], 1ull); atomicMax(&g_jac_dbg[2], (unsigned long long)(sweep + 1)); if (nv >= 64) atomicAdd(&g_jac_dbg[3], 1ull); if (nv >= 64 && sweep == 0) atomicAdd(&g_jac_dbg[4], 1ull); }
    __syncthreads();
    if (!converged && sweep == JAC_MAX_SWEEPS - 1 && tid == 0) atomicOr(b.status, OCMPS_ST_NOCONV);
  }
  __syncthreads();
  const long long t_jac1 = clock64();
  if (tid == 0) {
    atomicAdd(&g_jac_dbg[1], 1ull);
    if (nv >= 64) {
      atomicAdd(&g_jac_dbg[6], (unsigned long long)(t_jac1 - t_jac0));
      atomicAdd(&g_jac_dbg[7], (unsigned long long)(t_jac1 - t_jac0));
    }
#ifdef OCMPS_JAC_TRACE
    if (nv >= 24) printf("JT2 kind %d blk %d nv %d keff %d jac %lld\n", a.kind, blk, nv, keff, t_jac1 - t_jac0);
#endif
  }
  // spectrum + normalised right vectors Z[j][physical vector]
  for (int v = warp; v < nv; v += nwarps) {
    if (v < keff) {
      const cplx* y = Z + v * ldz;
      double s = 0.0;
      for (int c = lane; c < nv; c += 32) { cplx u = y[c]; s += u.x * u.x + u.y * u.y; }
      s = warp_sum(s);
      const double inv = s > 0.0 ? rsqrt(s) : 0.0;
      for (int c = lane; c < nv; c += 32) {
        cplx u = y[c];
        Ya[v * nv + (int)perm[c]] = make_double2(u.x * inv, u.y * inv);
      }
      if (lane == 0) b.P[B.p_off + v] = s;
    } else if (lane == 0) {
      b.P[B.p_off + v] = 0.0;
    }
  }
}

__global__ void __launch_bounds__(JAC_THREADS) jacobi_rot_kernel(DecompArgs a, DecompBuffers b, int smem_elems) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int keff = rot_handover_rows(b, (int)blockIdx.x, smem_elems);
  if (keff < 0) return;                                   // not handed over to this stage
  jacobi_rot_block(a, b, (int)blockIdx.x, keff, smem_raw);
}

// ------------------------------------------------------------------------------------------------
// Large blocks: one-sided Jacobi on the rows of R distributed over a thread-block cluster
// ------------------------------------------------------------------------------------------------
// A block with more than 64 rows of R (chi_cap >= ~110: K|psi> with its 2 chi bonds, the chi = 150 / 256 configurations) does not
// fit the register-resident kernel, and from 200 KB on not even one SM's shared memory: the generic loops then stream every
// pair of rows through L2 in every round (measured: 11 ms per decomposition at chi = 256).  Here the COLUMNS of R are split over
// the BJ_C = 8 CTAs of a cluster: every CTA keeps all rows (up to 256) of its slice (up to 32 columns, 128 KB) in shared memory.
// A round: partial dot products of the slice (4 lanes per pair, <= 8 columns per lane) -> one exchange of the 16-byte partials
// through distributed shared memory (st.async carries data + mbarrier complete_tx in one message; double buffered) -> every CTA
// sums the partials in rank order, so all CTAs compute bitwise identical angles, norms and convergence flags and never have
// to agree on anything else -> rotation of the slice.  Exact squared norms at the start of a sweep go through the same exchange.
// For blocks that FIT one SM this layout is no faster than jacobi_rot_kernel (profiles/r02_cluster_jacobi.md); it is the
// path for the blocks that do not.
namespace clus {
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ unsigned mapa(unsigned addr, unsigned rank) {
  unsigned r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_async_v2(unsigned raddr, double a, double b, unsigned rmbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f64 [%0], {%1, %2}, [%3];" ::"r"(raddr), "d"(a), "d"(b), "r"(rmbar) : "memory");
}
__device__ __forceinline__ void mbar_init(unsigned mbar, unsigned count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_expect(unsigned mbar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned mbar, unsigned parity) {
  asm volatile(
      "{\n.reg .pred p;\nWAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}\n" ::"r"(mbar), "r"(parity) : "memory");
}
__device__ __forceinline__ void cluster_sync() { asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;\n" ::: "memory"); }
__device__ __forceinline__ unsigned cluster_rank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
}  // namespace clus

// ------------------------------------------------------------------------------------------------
// Large blocks, first half: Householder QR with column pivoting, the VECTORS distributed over the cluster
// ------------------------------------------------------------------------------------------------
// CTA r of the 8 owns the vectors [r wv, (r+1) wv), wv = ceil(nv / 8) <= 32, each up to 256 components long, in shared memory
// (<= 128 KB), one half-warp per vector.  A step: (1) every CTA's best pivot candidate -- (norm bits | position) keys as in the
// single-CTA kernel -- is exchanged through distributed shared memory, so all CTAs pick the same pivot; (2) the pivot vector is
// pulled from its owner's shared memory (ld.shared::cluster) into every CTA; (3) every CTA forms the reflector from the exact
// pivot norm (bitwise the same everywhere), applies it to the vectors it owns and downdates their norms with the xGEQP3
// safeguard.  Position bookkeeping, R's diagonal and the rank test are replicated, so nothing else has to be agreed on.
// At the end every CTA writes the columns of R that belong to its vectors; jacobi_big_kernel takes over.
struct QbShared {
  unsigned long long key[2][BJ_C][2];     // exchanged candidates (double buffered), [buffer][source rank][key, unused]
  unsigned long long mbar[2];
  unsigned long long best;                // local candidate of the step (atomicMax)
  double red[BJ_THREADS / 32];
  double ncur[32], nref[32];              // trailing norms of the owned vectors (downdated / last exact value)
  double rdr[BJ_MAX_ROWS], rdi[BJ_MAX_ROWS];
  short pos2phys[BJ_MAX_ROWS], posof[BJ_MAX_ROWS];
  double F;
};

__device__ __forceinline__ void st_async_b64x2(unsigned raddr, unsigned long long a, unsigned long long b, unsigned rmbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.b64 [%0], {%1, %2}, [%3];" ::"r"(raddr), "l"(a), "l"(b), "r"(rmbar) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(unsigned mbar, unsigned parity) {
  asm volatile(
      "{\n.reg .pred p;\nWAITC_%=:\n"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONEC_%=;\nbra WAITC_%=;\nDONEC_%=:\n}\n" ::"r"(mbar), "r"(parity) : "memory");
}
// every CTA contributes one 64-bit value; afterwards out[r] holds the value of rank r in every CTA.  Called by all threads after
// a __syncthreads() that ordered the CTA's shared-memory writes of the step (they are released to the cluster here).
__device__ __forceinline__ void qb_allgather(QbShared& sh, unsigned& xcount, unsigned rank, unsigned long long mine, unsigned long long (&out)[BJ_C]) {
  const unsigned b = xcount & 1u, par = (xcount >> 1) & 1u;
  ++xcount;
  const unsigned mb = clus::smem_u32(&sh.mbar[b]);
  if (threadIdx.x == 0) {
    sh.key[b][rank][0] = mine;
    asm volatile("fence.acq_rel.cluster;" ::: "memory");       // the vectors updated in this step are visible to remote loads
    const unsigned la = clus::smem_u32(&sh.key[b][rank][0]);
#pragma unroll
    for (unsigned p = 1; p < (unsigned)BJ_C; ++p) {
      const unsigned peer = (rank + p) % BJ_C;
      st_async_b64x2(clus::mapa(la, peer), mine, 0ull, clus::mapa(mb, peer));
    }
  }
  mbar_wait_cluster(mb, par);
  if (threadIdx.x == 0) clus::mbar_expect(mb, (unsigned)((BJ_C - 1) * 16));
  __syncthreads();                                               // (own value written by thread 0)
#pragma unroll
  for (int r = 0; r < BJ_C; ++r) out[r] = sh.key[b][r][0];
}

__global__ void __launch_bounds__(BJ_THREADS) qr_big_kernel(DecompArgs a, DecompBuffers b, int smem_elems, double rank_tol) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ QbShared sh;
  constexpr unsigned long long KEY_POS = 2047ull;
  const DecompWork* w = b.dw;
  const int blk = blockIdx.x / BJ_C;
  if (blk >= w->nblocks) return;
  const DecompBlock B = w->blk[blk];
  const int nv = B.nv, len = B.len, ld = w->ld, mode = w->mode;
  {   // the same routing test as jacobi_blocks_kernel: only the blocks its register-cached instantiation does not take
    const bool fits = nv * len <= smem_elems && nv <= JAC_NV_SMEM;
    const int ldpad = ((nv + 15) >> 4) << 4;
    const bool can_cache = nv <= 16 * JAC_EPL && (nv < len ? nv : len) * ldpad <= smem_elems;
    if ((fits && can_cache) || nv > BJ_MAX_ROWS || len > BJ_MAX_ROWS) return;
  }
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, half = lane >> 4, hl = lane & 15;
  const unsigned rank = clus::cluster_rank();
  const int wv = (nv + BJ_C - 1) / BJ_C;                     // vectors per CTA
  const int v0 = (int)rank * wv;
  const int nown = max(0, min(nv, v0 + wv) - v0);
  cplx* Yv = reinterpret_cast<cplx*>(smem_raw);              // [owned vector][component], row stride len
  cplx* xp = Yv + (size_t)32 * BJ_MAX_ROWS;                  // pivot vector of the step
  const int* vidx = b.vec_idx + B.vec_off;
  const int* cidx = b.comp_idx + B.comp_off;
  cplx* Yb = b.ywork + b.ywork_half + B.ws_off;
  unsigned xcount = 0;
  if (tid == 0) {
    clus::mbar_init(clus::smem_u32(&sh.mbar[0]), 1);
    clus::mbar_init(clus::smem_u32(&sh.mbar[1]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    clus::mbar_expect(clus::smem_u32(&sh.mbar[0]), (unsigned)((BJ_C - 1) * 16));
    clus::mbar_expect(clus::smem_u32(&sh.mbar[1]), (unsigned)((BJ_C - 1) * 16));
  }
  // gather the owned vectors
  if (mode == 0) {
    for (int e = tid; e < nown * len; e += BJ_THREADS) {
      const int c = e / nown, vl = e % nown;
      Yv[vl * len + c] = a.X[(size_t)cidx[c] * ld + vidx[v0 + vl]];
    }
  } else {
    for (int e = tid; e < nown * len; e += BJ_THREADS) {
      const int vl = e / len, c = e % len;
      Yv[vl * len + c] = a.X[(size_t)vidx[v0 + vl] * ld + cidx[c]];
    }
  }
  for (int i = tid; i < nv; i += BJ_THREADS) { sh.pos2phys[i] = (short)i; sh.posof[i] = (short)i; }
  __syncthreads();
  const int hv = 2 * warp + half;                            // the owned vector of this half-warp
  {
    double sq = 0.0;
    if (hv < nown) for (int c = hl; c < len; c += 16) { const cplx u = Yv[hv * len + c]; sq += u.x * u.x + u.y * u.y; }
    sq = half_sum(sq);
    if (hv < nown && hl == 0) { sh.ncur[hv] = sq; sh.nref[hv] = sq; }
  }
  __syncthreads();
  clus::cluster_sync();
  {   // block weight F: sum of all initial norms, rank order
    double part = 0.0;
    for (int i = 0; i < nown; ++i) part += sh.ncur[i];
    unsigned long long all[BJ_C];
    qb_allgather(sh, xcount, rank, (unsigned long long)__double_as_longlong(part), all);
    double F = 0.0;
#pragma unroll
    for (int r = 0; r < BJ_C; ++r) F += __longlong_as_double((long long)all[r]);
    if (tid == 0) sh.F = F;
    __syncthreads();
  }
  const double F = sh.F;
  const double rtol_abs = F * rank_tol;
  const int kmax = nv < len ? nv : len;
  int keff = 0;
  const long long t_qr0 = clock64();
#ifdef OCMPS_JAC_TRACE
  long long tp[4] = {0, 0, 0, 0};
  long long tl = clock64();
#define QB_MARK(i) { const long long tn = clock64(); tp[i] += tn - tl; tl = tn; }
#else
#define QB_MARK(i)
#endif
  for (int j = 0; j < kmax; ++j) {
    // (1) pivot: local candidate among the owned vectors that are still in play, then the cluster-wide maximum
    if (tid == 0) sh.best = 0ull;
    __syncthreads();
    if (hv < nown && hl == 0) {
      const int pos = sh.posof[v0 + hv];
      if (pos >= j) atomicMax(&sh.best, ((unsigned long long)__double_as_longlong(sh.ncur[hv]) & ~KEY_POS) | (KEY_POS - (unsigned long long)pos));
    }
    __syncthreads();
    unsigned long long all[BJ_C];
    qb_allgather(sh, xcount, rank, sh.best, all);
    unsigned long long gbest = 0ull;
#pragma unroll
    for (int r = 0; r < BJ_C; ++r) gbest = all[r] > gbest ? all[r] : gbest;
    const int bpos = (int)(KEY_POS - (gbest & KEY_POS));
    const int pv = sh.pos2phys[bpos], pj = sh.pos2phys[j];
    QB_MARK(0)
    // (2) pull the pivot vector (components j .. len-1) from its owner
    {
      const unsigned owner = (unsigned)(pv / wv);
      const cplx* src = Yv + (size_t)(pv - (int)owner * wv) * len;
      if (owner == rank) {
        for (int c = j + tid; c < len; c += BJ_THREADS) xp[c] = src[c];
      } else {
        const unsigned base = clus::mapa(clus::smem_u32(src), owner);
        for (int c = j + tid; c < len; c += BJ_THREADS) {
          double xr, xi;
          asm volatile("ld.shared::cluster.v2.f64 {%0, %1}, [%2];" : "=d"(xr), "=d"(xi) : "r"(base + (unsigned)c * 16u) : "memory");
          xp[c] = make_double2(xr, xi);
        }
      }
    }
    __syncthreads();
    QB_MARK(1)
    // (3) exact norm of the pivot vector, the same bits in every CTA (fixed reduction order)
    {
      double sq = 0.0;
      for (int c = j + tid; c < len; c += BJ_THREADS) { const cplx u = xp[c]; sq += u.x * u.x + u.y * u.y; }
      sq = warp_sum(sq);
      if (lane == 0) sh.red[warp] = sq;
    }
    __syncthreads();
    double best = 0.0;
#pragma unroll
    for (int i = 0; i < BJ_THREADS / 32; ++i) best += sh.red[i];
    if (!(best > rtol_abs)) break;                              // numerical rank reached (uniform over the cluster)
    keff = j + 1;
    const cplx alpha = xp[j];
    const double inx = rsqrt(best), normx = best * inx;
    const double a2 = alpha.x * alpha.x + alpha.y * alpha.y;
    const double ia = a2 > 0.0 ? rsqrt(a2) : 0.0, aabs = a2 * ia;
    const double phr = a2 > 0.0 ? alpha.x * ia : 1.0, phi = a2 > 0.0 ? alpha.y * ia : 0.0;
    const double v0r = alpha.x + phr * normx, v0i = alpha.y + phi * normx;
    const double rb = rsqrt(normx * (normx + aabs));
    const double beta = rb * rb;
    if (tid == 0) {
      sh.rdr[j] = -phr * normx; sh.rdi[j] = -phi * normx;       // R_jj
      sh.pos2phys[bpos] = (short)pj; sh.pos2phys[j] = (short)pv;
      sh.posof[pj] = (short)bpos; sh.posof[pv] = (short)j;
    }
    __syncthreads();
    QB_MARK(2)
    // (4) reflector on the owned vectors that are still in play (all 32 lanes take part in the shuffles; `act` is per half-warp)
    {
      const int pos = hv < nown ? (int)sh.posof[v0 + hv] : -1;
      const bool act = pos > j;
      cplx* y = Yv + (size_t)(act ? hv : 0) * len;
      double wr = 0.0, wi = 0.0;
      if (act) {
        for (int c = j + hl; c < len; c += 16) {
          cplx vv = xp[c];
          if (c == j) { vv.x = v0r; vv.y = v0i; }
          const cplx yy = y[c];
          wr += vv.x * yy.x + vv.y * yy.y;      // conj(v) * y
          wi += vv.x * yy.y - vv.y * yy.x;
        }
      }
      wr = half_sum(wr); wi = half_sum(wi);
      double rji2 = 0.0;
      if (act) {
        const double fr = beta * wr, fi = beta * wi;
        for (int c = j + hl; c < len; c += 16) {
          cplx vv = xp[c];
          if (c == j) { vv.x = v0r; vv.y = v0i; }
          cplx yy = y[c];
          yy.x -= fr * vv.x - fi * vv.y;
          yy.y -= fr * vv.y + fi * vv.x;
          y[c] = yy;
          if (c == j) rji2 = yy.x * yy.x + yy.y * yy.y;
        }
      }
      rji2 = __shfl_sync(0xffffffffu, rji2, lane & 16);          // component j is owned by lane 0 of the half-warp
      double tnew = 0.0;
      bool redo = false;
      if (act) {
        tnew = sh.ncur[hv] - rji2;
        redo = !(tnew > 1.5e-8 * sh.nref[hv]);
      }
      if (__any_sync(0xffffffffu, redo)) {                        // rare: exact trailing norm (xGEQP3 safeguard)
        double tail = 0.0;
        if (act && redo) for (int c = j + 1 + hl; c < len; c += 16) { const cplx yy = y[c]; tail += yy.x * yy.x + yy.y * yy.y; }
        tail = half_sum(tail);
        if (act && redo) { tnew = tail; if (hl == 0) sh.nref[hv] = tail; }
      }
      if (act && hl == 0) sh.ncur[hv] = tnew > 0.0 ? tnew : 0.0;
    }
    __syncthreads();
    QB_MARK(3)
  }
#ifdef OCMPS_JAC_TRACE
  if (tid == 0 && rank == 0 && nv >= 24)
    printf("JTQ kind %d blk %d nv %d len %d keff %d qr %lld : exchange %lld pull %lld norm+scalars %lld update %lld\n", a.kind, blk, nv, len, keff,
           (long long)(clock64() - t_qr0), tp[0], tp[1], tp[2], tp[3]);
#endif
  // R (keff x nv, position order, row stride nv) -> global scratch; every CTA writes the columns of its vectors
  const int ldz = nv;
  for (int vl = warp; vl < nown; vl += BJ_THREADS / 32) {
    const int i = sh.posof[v0 + vl];
    const cplx* y = Yv + (size_t)vl * len;
    for (int c = lane; c < keff; c += 32) {
      cplx v = make_double2(0.0, 0.0);
      if (c < i) v = y[c];
      else if (c == i) v = make_double2(sh.rdr[c], sh.rdi[c]);
      Yb[(size_t)c * ldz + i] = v;
    }
  }
  if (rank == 0) {
    short* gperm = reinterpret_cast<short*>(b.scratch_d + 4 * NV_MAX) + B.p_off;
    for (int i = tid; i < nv; i += BJ_THREADS) gperm[i] = sh.pos2phys[i];
    if (tid == 0) {
      double* hF = b.scratch_d + 7 * NV_MAX;
      int* hK = reinterpret_cast<int*>(b.scratch_d + 7 * NV_MAX + OCMPS_MAX_BLK);
      hF[blk] = F;
      hK[blk] = -1;
      if (nv >= 64) { const long long t_now = clock64(); atomicAdd(&g_jac_dbg[5], (unsigned long long)(t_now - t_qr0)); atomicAdd(&g_jac_dbg[7], (unsigned long long)(t_now - t_qr0)); }
      hK[OCMPS_MAX_BLK + blk] = keff;
      hK[2 * OCMPS_MAX_BLK + blk] = ldz;
      const double nn = (double)len, mmv = (double)nv;
      atomicAdd(&g_jac_flops[0], 8.0 * nn * nn * mmv + (56.0 / 3.0) * nn * nn * nn);
      if (blk == 0) {
        const double dn = mode == 0 ? (double)w->n : (double)w->m, dm = mode == 0 ? (double)w->m : (double)w->n;
        atomicAdd(&g_jac_flops[1], 8.0 * dn * dn * dm + (56.0 / 3.0) * dn * dn * dn);
      }
    }
  }
  clus::cluster_sync();                                   // no CTA may exit while a peer can still read its vectors
}

struct BjShared {
  double2 xbuf[2][BJ_C][BJ_SLOTS];        // partials of the exchange in flight (double buffered), [buffer][source rank][slot]
  unsigned long long mbar[2];
  double nrm[BJ_MAX_ROWS];
  int rot, big;
};

// all-CTAs sum of one (x, y) pair per active slot; every lane of a slot gets the sum (lanes other than the first pass anything).
// Called by ALL threads; nslots (the same in every CTA) is the number of slots that take part.
__device__ __forceinline__ double2 bj_exchange(BjShared& sh, unsigned& xcount, unsigned rank, int nslots, int slot, int lane, double x, double y) {
  const unsigned b = xcount & 1u, par = (xcount >> 1) & 1u;
  ++xcount;
  const unsigned mb = clus::smem_u32(&sh.mbar[b]);
  if (lane == 0 && slot < nslots) {
    sh.xbuf[b][rank][slot] = make_double2(x, y);
    const unsigned la = clus::smem_u32(&sh.xbuf[b][rank][slot]);
#pragma unroll
    for (unsigned p = 1; p < (unsigned)BJ_C; ++p) {
      const unsigned peer = (rank + p) % BJ_C;
      clus::st_async_v2(clus::mapa(la, peer), x, y, clus::mapa(mb, peer));
    }
  }
  clus::mbar_wait(mb, par);
  if (threadIdx.x == 0) clus::mbar_expect(mb, (unsigned)((BJ_C - 1) * nslots * 16));      // re-arm for the exchange after the next
  __syncwarp();                                                                             // (own partial: written by lane 0 of the slot)
  double sx = 0.0, sy = 0.0;
  if (slot < nslots) {
#pragma unroll
    for (int r = 0; r < BJ_C; ++r) { const double2 v = sh.xbuf[b][r][slot]; sx += v.x; sy += v.y; }
  }
  return make_double2(sx, sy);
}

// TPP lanes per pair (8 while the block has at most 128 rows: 64 pair slots x 8 lanes; 4 beyond that), EPL columns per lane
template <int TPP, int EPL>
__device__ void bj_run(DecompBuffers& b, const DecompBlock& B, int keff, int ldz, double F, cplx* __restrict__ Rs, BjShared& sh) {
  const int tid = threadIdx.x, slot = tid / TPP, lane = tid % TPP;
  const unsigned rank = clus::cluster_rank();
  const int nv = B.nv;
  const int w = (nv + BJ_C - 1) / BJ_C;                // columns of this CTA's slice: [c0, c0 + w) clipped to nv
  const int c0 = (int)rank * w;
  // row stride of the slice in shared memory, = 4 (mod 8) complex numbers: the lanes of a pair read 16 B each from consecutive
  // addresses, the pairs of a warp sit in consecutive rows, and a stride of 0 (mod 128 B) would put them all on the same banks
  constexpr int WP = (TPP * EPL) % 8 == 0 ? TPP * EPL + 4 : ((TPP * EPL) % 8 == 4 ? TPP * EPL : TPP * EPL + (12 - (TPP * EPL) % 8) % 8);
  const cplx* Yb = b.ywork + b.ywork_half + B.ws_off;
  cplx* Ya = b.ywork + B.ws_off;
  const short* perm = reinterpret_cast<const short*>(b.scratch_d + 4 * NV_MAX) + B.p_off;
  const double thr = F * DEFLATE_REL;
  unsigned xcount = 0;
  for (int e = tid; e < keff * WP; e += BJ_THREADS) {  // slice of R -> shared memory (zero padded)
    const int r = e / WP, cl = e % WP, c = c0 + cl;
    Rs[e] = (cl < w && c < nv) ? Yb[(size_t)r * ldz + c] : make_double2(0.0, 0.0);
  }
  __syncthreads();
  const int npad = (keff + 1) & ~1, nslots = npad >> 1, mm = npad - 1;
  cplx ra[EPL], rb[EPL];
  auto load_row = [&](cplx (&r)[EPL], int row) {
    const cplx* z = Rs + (row >= 0 ? row : 0) * WP + lane;
#pragma unroll
    for (int e = 0; e < EPL; ++e) r[e] = row >= 0 ? z[TPP * e] : make_double2(0.0, 0.0);
  };
  auto store_row = [&](const cplx (&r)[EPL], int row) {
    if (row < 0) return;
    cplx* z = Rs + row * WP + lane;
#pragma unroll
    for (int e = 0; e < EPL; ++e) z[TPP * e] = r[e];
  };
  auto lanes_sum = [&](double v) {
#pragma unroll
    for (int o = TPP / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
  };
  auto exact_norms = [&]() {                           // slot s takes rows 2s and 2s+1
    const int x = 2 * slot < keff ? 2 * slot : -1, y = 2 * slot + 1 < keff ? 2 * slot + 1 : -1;
    load_row(ra, x);
    load_row(rb, y);
    double sa = 0.0, sb = 0.0;
#pragma unroll
    for (int e = 0; e < EPL; ++e) { sa += ra[e].x * ra[e].x + ra[e].y * ra[e].y; sb += rb[e].x * rb[e].x + rb[e].y * rb[e].y; }
    sa = lanes_sum(sa); sb = lanes_sum(sb);
    const double2 t = bj_exchange(sh, xcount, rank, nslots, slot, lane, sa, sb);
    if (lane == 0) { if (x >= 0) sh.nrm[x] = t.x; if (y >= 0) sh.nrm[y] = t.y; }
  };
  bool converged = keff < 2;
#ifdef OCMPS_JAC_TRACE
  long long tq[3] = {0, 0, 0};
  long long tql = clock64();
  int nrounds = 0;
#define BJ_MARK(i) { const long long tn = clock64(); tq[i] += tn - tql; tql = tn; }
#else
#define BJ_MARK(i)
#endif
  for (int sweep = 0; sweep < JAC_MAX_SWEEPS && !converged; ++sweep) {
    exact_norms();
    if (tid == 0) { sh.rot = 0; sh.big = 0; }
    __syncthreads();
    for (int R = 0; R < npad - 1; ++R) {
      // round-robin pairing: slot k plays p = (R + k) mod (npad-1) against q = (R - k) mod (npad-1); slot 0 plays the fixed row
      int p = -1, q = -1;
      if (slot < nslots) {
        p = R + slot; if (p >= mm) p -= mm;
        q = R - slot; if (q < 0) q += mm;
        if (slot == 0) q = npad - 1;
        if (p > q) { const int t = p; p = q; q = t; }
        if (q >= keff) { p = -1; q = -1; }
      }
      const bool act = p >= 0;
      load_row(ra, p);
      load_row(rb, q);
      const double aa = act ? sh.nrm[p] : 0.0, bb = act ? sh.nrm[q] : 0.0;
      double c0r = 0.0, c0i = 0.0, c1r = 0.0, c1i = 0.0;
#pragma unroll
      for (int e = 0; e < EPL; ++e) {
        const double pr = ra[e].x * rb[e].x + ra[e].y * rb[e].y;      // conj(a) * b
        const double pi = ra[e].x * rb[e].y - ra[e].y * rb[e].x;
        if (e & 1) { c1r += pr; c1i += pi; } else { c0r += pr; c0i += pi; }
      }
      const double pre = lanes_sum(c0r + c1r), pim = lanes_sum(c0i + c1i);
      BJ_MARK(0)
      const double2 cc = bj_exchange(sh, xcount, rank, nslots, slot, lane, pre, pim);
      BJ_MARK(1)
      if (act) {
        const double cre = cc.x, cim = cc.y;
        const double c2 = cre * cre + cim * cim;
        if (aa <= thr || bb <= thr) {
          if (aa <= thr && aa > 0.0) {
#pragma unroll
            for (int e = 0; e < EPL; ++e) ra[e] = make_double2(0.0, 0.0);
            store_row(ra, p);
            if (lane == 0) sh.nrm[p] = 0.0;
          }
          if (bb <= thr && bb > 0.0) {
#pragma unroll
            for (int e = 0; e < EPL; ++e) rb[e] = make_double2(0.0, 0.0);
            store_row(rb, q);
            if (lane == 0) sh.nrm[q] = 0.0;
          }
        } else if (c2 > JAC_TOL2 * aa * bb) {
          // same angle formulas as jac_rotate (two rsqrt, no division)
          const double dd = 0.5 * (bb - aa);
          const double xh = dd * dd + c2;
          const double ih = rsqrt(xh);
          const double h = xh * ih;
          const double sdh = fabs(dd) + h;
          const double wv = rsqrt(2.0 * h * sdh);
          const double cs = sdh * wv;
          const double sgw = dd >= 0.0 ? wv : -wv;
          const double sr = sgw * cre, si = sgw * cim;
#pragma unroll
          for (int e = 0; e < EPL; ++e) {
            const cplx u = ra[e], v = rb[e];
            ra[e] = make_double2(cs * u.x - (sr * v.x + si * v.y), cs * u.y - (sr * v.y - si * v.x));   // cs a - conj(sigma) b
            rb[e] = make_double2(cs * v.x + (sr * u.x - si * u.y), cs * v.y + (sr * u.y + si * u.x));   // sigma a + cs b
          }
          store_row(ra, p);
          store_row(rb, q);
          if (lane == 0) {
            const double trr = c2 * (sgw * wv) * (2.0 * h);
            const double a1 = aa - trr, b1 = bb + trr;
            sh.nrm[p] = a1 > 0.0 ? a1 : 0.0;
            sh.nrm[q] = b1 > 0.0 ? b1 : 0.0;
            sh.rot = 1;
            if (c2 > 1e-16 * aa * bb) sh.big = 1;
          }
        }
      }
      __syncthreads();
      BJ_MARK(2)
#ifdef OCMPS_JAC_TRACE
      ++nrounds;
#endif
    }
    converged = (sh.rot == 0) || (sh.big == 0);
    __syncthreads();
    if (!converged && sweep == JAC_MAX_SWEEPS - 1 && tid == 0 && rank == 0) atomicOr(b.status, OCMPS_ST_NOCONV);
    if (tid == 0 && rank == 0) { atomicAdd(&g_jac_dbg[0], 1ull); atomicMax(&g_jac_dbg[2], (unsigned long long)(sweep + 1)); if (nv >= 64) atomicAdd(&g_jac_dbg[3], 1ull); if (nv >= 64 && sweep == 0) atomicAdd(&g_jac_dbg[4], 1ull); }
  }
#ifdef OCMPS_JAC_TRACE
  if (tid == 0 && rank == 0 && nv >= 24 && nrounds > 0)
    printf("JTB nv %d keff %d EPL %d rounds %d per round: load+dot %lld exchange %lld rotate+sync %lld\n", nv, keff, EPL, nrounds, tq[0] / nrounds, tq[1] / nrounds,
           tq[2] / nrounds);
#endif
  // spectrum + normalised right vectors Z[j][physical vector]: every CTA writes its columns
  exact_norms();
  __syncthreads();
  for (int v = slot; v < nv; v += BJ_THREADS / TPP) {
    if (v < keff) {
      const double sq = sh.nrm[v];
      const double inv = sq > 0.0 ? rsqrt(sq) : 0.0;
      for (int cl = lane; cl < w; cl += TPP) {
        const int c = c0 + cl;
        if (c < nv) { const cplx u = Rs[v * WP + cl]; Ya[(size_t)v * nv + (int)perm[c]] = make_double2(u.x * inv, u.y * inv); }
      }
      if (lane == 0 && rank == 0) b.P[B.p_off + v] = sq;
    } else if (lane == 0 && rank == 0) {
      b.P[B.p_off + v] = 0.0;
    }
  }
}

__global__ void __launch_bounds__(BJ_THREADS) jacobi_big_kernel(DecompArgs a, DecompBuffers b) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ BjShared sh;
  const DecompWork* w = b.dw;
  const int blk = blockIdx.x / BJ_C;
  // (uniform over the cluster: all CTAs of a cluster see the same block and the same hand-over flag)
  if (blk >= w->nblocks) return;
  if (w->blk[blk].nv > BJ_MAX_ROWS || w->blk[blk].len > BJ_MAX_ROWS) return;   // finished by the generic first-stage variants
  const int* hK = reinterpret_cast<const int*>(b.scratch_d + 7 * NV_MAX + OCMPS_MAX_BLK);
  const int keff = hK[OCMPS_MAX_BLK + blk];
  if (keff < 0) return;                                  // not handed over to this kernel
  const int ldz = hK[2 * OCMPS_MAX_BLK + blk];
  const DecompBlock B = w->blk[blk];
  const double F = (b.scratch_d + 7 * NV_MAX)[blk];
  const int tid = threadIdx.x;
  const int nslots = ((keff + 1) & ~1) >> 1;
  if (tid == 0) {
    clus::mbar_init(clus::smem_u32(&sh.mbar[0]), 1);
    clus::mbar_init(clus::smem_u32(&sh.mbar[1]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    clus::mbar_expect(clus::smem_u32(&sh.mbar[0]), (unsigned)((BJ_C - 1) * nslots * 16));
    clus::mbar_expect(clus::smem_u32(&sh.mbar[1]), (unsigned)((BJ_C - 1) * nslots * 16));
  }
  __syncthreads();
  clus::cluster_sync();
  const long long t0 = clock64();
  cplx* Rs = reinterpret_cast<cplx*>(smem_raw);
  const int wcols = (B.nv + BJ_C - 1) / BJ_C;
  if (keff <= BJ_THREADS / 8 * 2) {                      // at most 128 rows: 8 lanes per pair, <= 4 columns per lane
    switch ((wcols + 7) / 8) {
      case 1: bj_run<8, 1>(b, B, keff, ldz, F, Rs, sh); break;
      case 2: bj_run<8, 2>(b, B, keff, ldz, F, Rs, sh); break;
      case 3: bj_run<8, 3>(b, B, keff, ldz, F, Rs, sh); break;
      default: bj_run<8, 4>(b, B, keff, ldz, F, Rs, sh); break;
    }
  } else {
    switch ((wcols + 3) / 4) {
      case 1: bj_run<4, 1>(b, B, keff, ldz, F, Rs, sh); break;
      case 2: bj_run<4, 2>(b, B, keff, ldz, F, Rs, sh); break;
      case 3: bj_run<4, 3>(b, B, keff, ldz, F, Rs, sh); break;
      case 4: bj_run<4, 4>(b, B, keff, ldz, F, Rs, sh); break;
      case 5: bj_run<4, 5>(b, B, keff, ldz, F, Rs, sh); break;
      case 6: bj_run<4, 6>(b, B, keff, ldz, F, Rs, sh); break;
      case 7: bj_run<4, 7>(b, B, keff, ldz, F, Rs, sh); break;
      default: bj_run<4, 8>(b, B, keff, ldz, F, Rs, sh); break;
    }
  }
  clus::cluster_sync();                                   // no CTA may exit while a peer can still send to it
  if (tid == 0 && clus::cluster_rank() == 0) {
    atomicAdd(&g_jac_dbg[1], 1ull);
    const long long t1 = clock64();
    if (B.nv >= 64) { atomicAdd(&g_jac_dbg[6], (unsigned long long)(t1 - t0)); atomicAdd(&g_jac_dbg[7], (unsigned long long)(t1 - t0)); }
#ifdef OCMPS_JAC_TRACE
    if (B.nv >= 24) printf("JT3 kind %d blk %d nv %d keff %d jac %lld\n", a.kind, blk, B.nv, keff, (long long)(t1 - t0));
#endif
  }
}

// ------------------------------------------------------------------------------------------------
// Register-cached blocks with many rows of R: row-block parallel Jacobi on a cluster of RC_C CTAs
// ------------------------------------------------------------------------------------------------
// The largest block of a saturated gate decomposition (nv ~ 80, ~62 rows of R) sets the latency of the whole decomposition, and
// on one SM a rotation round of jacobi_sweep_blocked is bound by that SM's instruction issue (16 warps, 4 per scheduler), not by
// the round's dependent chain (profiles/r02_cluster_jacobi.md).  Here the rows are split into RC_NBLK = 2 RC_C row blocks of
// rb = ceil(keff / RC_NBLK) <= 8 rows and every CTA of the cluster holds two of them, so dot products and rotations stay local
// and every SM carries a quarter of the issue load.  A sweep = the pairs inside every row block, then RC_NBLK - 1 block rounds
// of a round-robin tournament over the row blocks; in a block round a CTA does the rb x rb cross pairs of its two blocks in rb
// rotation rounds (one half-warp per row of the first block, rows of the second one passed on through shared memory).
// Between block rounds every CTA pulls the two blocks of its next pairing from the CTAs that held them (ld.shared::cluster,
// double-buffered, one cluster barrier per block round).  The round-robin does not let a CTA keep one of its blocks in every
// transition, so both are always pulled (the one it keeps from itself); that is ~2 x 10 KB per CTA per block round.
// The stop flags are OR-reduced over the cluster once per sweep, so every CTA applies the same stop rule and the result is
// deterministic (fixed pair order); it is not bitwise that of jacobi_rot_kernel (the rotation order differs).
constexpr int RC_C = 4;                                    // CTAs per cluster
constexpr int RC_NBLK = 2 * RC_C;                          // row blocks of the tournament
constexpr int RC_ROWS = JAC_BLOCKED_ROWS / RC_NBLK;        // rows per row block, at most
constexpr int RC_WORK_THREADS = 16 * RC_ROWS;              // one half-warp per row of a block
// blocks with at least this many rows of R take the cluster path (K_CL); smaller ones stay with jacobi_rot_block on one SM
constexpr int RC_MIN_ROWS = 40;

__device__ unsigned long long g_rc_dbg[2];                 // development counters: [0] blocks finished on the cluster path, [1] their sweeps

struct RcShared {
  double nrm[2][2][RC_ROWS];       // cached squared norms: [buffer][block of this CTA][row]
  int flags[2][RC_C];              // per sweep parity and rank: rotated | (rotated above 1e-8) << 1
  int rot, big;
};

// the two row blocks CTA s plays in block round R (round-robin over RC_NBLK blocks with RC_C pair slots)
__device__ __forceinline__ void rc_blocks(int R, int s, int& P, int& Q) {
  constexpr int mm = RC_NBLK - 1;
  int p = R + s; if (p >= mm) p -= mm;
  int q = R - s; if (q < 0) q += mm;
  if (s == 0) q = RC_NBLK - 1;
  P = p; Q = q;
}

__device__ __forceinline__ void rc_bar() { asm volatile("bar.sync 1, %0;" ::"n"(RC_WORK_THREADS) : "memory"); }

// One block round of the RC_WORK_THREADS working threads: (intra: the pairs inside both blocks first) the rb x rb cross pairs of
// block 0 (rows Z0, norms n0, global rows base0 + i) and block 1.  Rows past keff are zero padding and take no part.
template <int EPL>
__device__ __forceinline__ void rc_block_round(cplx* __restrict__ Z0, cplx* __restrict__ Z1, double* n0, double* n1, int rb, int base0, int base1,
                                               int keff, double thr, bool intra, int* s_rot, int* s_big) {
  constexpr int ldz = 16 * EPL;
  const int tid = threadIdx.x, hl = tid & 15, h = tid >> 4;
  cplx ra[EPL], rb_[EPL];
  double na = 0.0, nb = 0.0;
  auto load_row = [&](cplx (&r)[EPL], double& n, const cplx* Z, const double* nz, int row) {
    const cplx* z = Z + (row >= 0 ? row : 0) * ldz + hl;
#pragma unroll
    for (int e = 0; e < EPL; ++e) r[e] = row >= 0 ? z[16 * e] : make_double2(0.0, 0.0);
    n = row >= 0 ? nz[row] : 0.0;
  };
  auto store_row = [&](const cplx (&r)[EPL], double n, cplx* Z, double* nz, int row) {
    cplx* z = Z + row * ldz + hl;
#pragma unroll
    for (int e = 0; e < EPL; ++e) z[16 * e] = r[e];
    if (hl == 0) nz[row] = n;
  };
  if (intra) {   // half-warps [0, RC_ROWS/2) take the pairs of block 0, the others those of block 1; round-robin over rbp rows
    const int X = h / (RC_ROWS / 2), j = h % (RC_ROWS / 2);
    cplx* Z = X ? Z1 : Z0;
    double* nz = X ? n1 : n0;
    const int base = X ? base1 : base0;
    const int rbp = (rb + 1) & ~1, m = rbp - 1;
    for (int r = 0; r < m; ++r) {
      int p = r + j; if (p >= m) p -= m;
      int q = r - j; if (q < 0) q += m;
      if (j == 0) q = m;
      const bool act = 2 * j < rbp && p < rb && q < rb && base + p < keff && base + q < keff;
      load_row(ra, na, Z, nz, act ? p : -1);
      load_row(rb_, nb, Z, nz, act ? q : -1);
      jac_rotate<EPL>(ra, rb_, na, nb, act, thr, hl, s_rot, s_big);
      if (act) { store_row(ra, na, Z, nz, p); store_row(rb_, nb, Z, nz, q); }
      rc_bar();
    }
  }
  // cross pairs: half-warp h keeps row h of block 0 in registers and meets row (h + t) mod rb of block 1 in round t
  const bool has_a = h < rb && base0 + h < keff;
  load_row(ra, na, Z0, n0, has_a ? h : -1);
  for (int t = 0; t < rb; ++t) {
    int jb = h + t; if (jb >= rb) jb -= rb;
    const bool act = has_a && base1 + jb < keff;
    load_row(rb_, nb, Z1, n1, act ? jb : -1);
    jac_rotate<EPL>(ra, rb_, na, nb, act, thr, hl, s_rot, s_big);
    if (act) store_row(rb_, nb, Z1, n1, jb);
    rc_bar();
  }
  if (has_a) store_row(ra, na, Z0, n0, h);
}

template <int EPL>
__device__ __forceinline__ void rc_run(const DecompArgs& a, const DecompBuffers& b, int blk, int keff, unsigned rank, cplx* __restrict__ Zs, RcShared& sh) {
  constexpr int ldz = 16 * EPL;
  constexpr int BLK = RC_ROWS * ldz;                     // elements of one row block in a buffer
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = JAC_THREADS / 32;
  const DecompBlock B = b.dw->blk[blk];
  const int nv = B.nv;
  const int rb = (keff + RC_NBLK - 1) / RC_NBLK;
  const double F = (b.scratch_d + 7 * NV_MAX)[blk];
  const double thr = F * DEFLATE_REL;
  const cplx* Yb = b.ywork + b.ywork_half + B.ws_off;   // R, keff rows of stride ldz (the padding of a row is zero)
  auto zb = [&](int buf, int k) { return Zs + (2 * buf + k) * BLK; };
  const long long t_jac0 = clock64();
  int P, Q;
  rc_blocks(0, (int)rank, P, Q);
  for (int e = tid; e < 2 * BLK; e += JAC_THREADS) {
    const int k = e / BLK, r = (e % BLK) / ldz, c = e % ldz;
    const int row = (k ? Q : P) * rb + r;
    Zs[e] = (r < rb && row < keff) ? Yb[row * ldz + c] : make_double2(0.0, 0.0);
  }
  __syncthreads();
  int cur = 0;
  bool done = false;
#ifdef OCMPS_JAC_TRACE
  long long t_work = 0, t_xchg = 0;
  int nrounds = 0, nxchg = 0;
#endif
  for (int sweep = 0; sweep < JAC_MAX_SWEEPS && !done; ++sweep) {
    for (int lr = warp; lr < 2 * RC_ROWS; lr += nwarps) {     // exact Gram diagonal at the start of every sweep
      const int k = lr / RC_ROWS, r = lr % RC_ROWS;
      const cplx* y = zb(cur, k) + r * ldz;
      double s = 0.0;
      for (int c = lane; c < nv; c += 32) { const cplx u = y[c]; s += u.x * u.x + u.y * u.y; }
      s = warp_sum(s);
      if (lane == 0) sh.nrm[cur][k][r] = s;                   // (zero for padding rows)
    }
    if (tid == 0) { sh.rot = 0; sh.big = 0; }
    __syncthreads();
    for (int R = 0; R < RC_NBLK - 1; ++R) {
#ifdef OCMPS_JAC_TRACE
      const long long tw0 = clock64();
#endif
      if (tid < RC_WORK_THREADS) rc_block_round<EPL>(zb(cur, 0), zb(cur, 1), sh.nrm[cur][0], sh.nrm[cur][1], rb, P * rb, Q * rb, keff, thr, R == 0, &sh.rot, &sh.big);
      __syncthreads();
#ifdef OCMPS_JAC_TRACE
      const long long tw1 = clock64();
      t_work += tw1 - tw0;
      nrounds += rb + (R == 0 ? ((rb + 1) & ~1) - 1 : 0);
#endif
      const bool last = R == RC_NBLK - 2;
      if (last && tid < RC_C) {     // this CTA's flags into slot `rank` of every CTA (released by the cluster barrier)
        const int f = (sh.rot ? 1 : 0) | (sh.big ? 2 : 0);
        asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(clus::mapa(clus::smem_u32(&sh.flags[sweep & 1][rank]), (unsigned)tid)), "r"(f) : "memory");
      }
      clus::cluster_sync();
      if (last) {
        int any = 0;
#pragma unroll
        for (int r = 0; r < RC_C; ++r) any |= sh.flags[sweep & 1][r];
        // quadratic convergence: if every rotated pair had |<p|q>| < 1e-8 |p||q|, the residuals are now ~1e-16
        done = !(any & 1) || !(any & 2);
        if (tid == 0 && rank == 0) {
          atomicAdd(&g_jac_dbg[0], 1ull); atomicMax(&g_jac_dbg[2], (unsigned long long)(sweep + 1)); atomicAdd(&g_rc_dbg[1], 1ull);
          if (nv >= 64) atomicAdd(&g_jac_dbg[3], 1ull);
          if (nv >= 64 && sweep == 0) atomicAdd(&g_jac_dbg[4], 1ull);
          if (!done && sweep == JAC_MAX_SWEEPS - 1) atomicOr(b.status, OCMPS_ST_NOCONV);
        }
        if (done || sweep == JAC_MAX_SWEEPS - 1) break;
      }
      // pull the two blocks of the next pairing (round 0 of the next sweep after the last round) from the CTAs that hold them
      // (the one this CTA keeps from itself)
      int NP, NQ;
      rc_blocks(last ? 0 : R + 1, (int)rank, NP, NQ);
      unsigned src0 = 0, src1 = 0, nsrc0 = 0, nsrc1 = 0;       // shared::cluster addresses of their rows / norms
      for (int s = 0; s < RC_C; ++s) {
        int p, q;
        rc_blocks(R, s, p, q);
        const unsigned zp = clus::mapa(clus::smem_u32(zb(cur, 0)), (unsigned)s), zq = clus::mapa(clus::smem_u32(zb(cur, 1)), (unsigned)s);
        const unsigned np = clus::mapa(clus::smem_u32(sh.nrm[cur][0]), (unsigned)s), nq = clus::mapa(clus::smem_u32(sh.nrm[cur][1]), (unsigned)s);
        if (p == NP) { src0 = zp; nsrc0 = np; }
        if (q == NP) { src0 = zq; nsrc0 = nq; }
        if (p == NQ) { src1 = zp; nsrc1 = np; }
        if (q == NQ) { src1 = zq; nsrc1 = nq; }
      }
      for (int e = tid; e < 2 * rb * ldz; e += JAC_THREADS) {
        const int k = e >= rb * ldz, o = e - k * rb * ldz;
        double xr, xi;
        asm volatile("ld.shared::cluster.v2.f64 {%0, %1}, [%2];" : "=d"(xr), "=d"(xi) : "r"((k ? src1 : src0) + (unsigned)o * 16u) : "memory");
        zb(cur ^ 1, k)[o] = make_double2(xr, xi);
      }
      if (tid < 2 * RC_ROWS) {
        const int k = tid / RC_ROWS, r = tid % RC_ROWS;
        double x;
        asm volatile("ld.shared::cluster.f64 %0, [%1];" : "=d"(x) : "r"((k ? nsrc1 : nsrc0) + (unsigned)r * 8u) : "memory");
        sh.nrm[cur ^ 1][k][r] = x;
      }
      __syncthreads();
#ifdef OCMPS_JAC_TRACE
      t_xchg += clock64() - tw1;
      ++nxchg;
#endif
      cur ^= 1; P = NP; Q = NQ;
    }
  }
  const long long t_jac1 = clock64();
  // spectrum + normalised right vectors Z[j][physical vector]: every CTA writes the rows it holds
  const short* perm = reinterpret_cast<const short*>(b.scratch_d + 4 * NV_MAX) + B.p_off;
  cplx* Ya = b.ywork + B.ws_off;
  for (int lr = warp; lr < 2 * RC_ROWS; lr += nwarps) {
    const int k = lr / RC_ROWS, r = lr % RC_ROWS, v = (k ? Q : P) * rb + r;
    if (r >= rb || v >= keff) continue;
    const cplx* y = zb(cur, k) + r * ldz;
    double s = 0.0;
    for (int c = lane; c < nv; c += 32) { const cplx u = y[c]; s += u.x * u.x + u.y * u.y; }
    s = warp_sum(s);
    const double inv = s > 0.0 ? rsqrt(s) : 0.0;
    for (int c = lane; c < nv; c += 32) {
      const cplx u = y[c];
      Ya[v * nv + (int)perm[c]] = make_double2(u.x * inv, u.y * inv);
    }
    if (lane == 0) b.P[B.p_off + v] = s;
  }
  if (rank == 0) for (int v = keff + tid; v < nv; v += JAC_THREADS) b.P[B.p_off + v] = 0.0;
  if (tid == 0 && rank == 0) {
    atomicAdd(&g_jac_dbg[1], 1ull);
    atomicAdd(&g_rc_dbg[0], 1ull);
    if (nv >= 64) {
      atomicAdd(&g_jac_dbg[6], (unsigned long long)(t_jac1 - t_jac0));
      atomicAdd(&g_jac_dbg[7], (unsigned long long)(t_jac1 - t_jac0));
    }
#ifdef OCMPS_JAC_TRACE
    if (nv >= 24)
      printf("JTR kind %d blk %d nv %d keff %d rb %d jac %lld : rotation rounds %d, %lld clk per round; block exchanges %d, %lld clk each\n", a.kind, blk, nv,
             keff, rb, t_jac1 - t_jac0, nrounds, nrounds ? t_work / nrounds : 0ll, nxchg, nxchg ? t_xchg / nxchg : 0ll);
#endif
  }
  // (no DSMEM access follows the last cluster barrier: a CTA may leave while its peers write their rows)
}

// Second stage of the register-cached blocks, one cluster of RC_C CTAs per block: blocks with at least RC_MIN_ROWS rows of R are
// spread over the cluster (rc_run), smaller ones are finished by rank 0 alone (jacobi_rot_block) while the other ranks leave.
__global__ void __launch_bounds__(JAC_THREADS) jacobi_rows_cluster_kernel(DecompArgs a, DecompBuffers b, int smem_elems) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ RcShared sh;
  const int blk = (int)blockIdx.x / RC_C;
  const unsigned rank = clus::cluster_rank();
  const int keff = rot_handover_rows(b, blk, smem_elems);   // (uniform over the cluster)
  if (keff < 0) return;
  if (keff < RC_MIN_ROWS) {
    if (rank == 0) jacobi_rot_block(a, b, blk, keff, smem_raw);
    return;
  }
  cplx* Zs = reinterpret_cast<cplx*>(smem_raw);
  switch ((b.dw->blk[blk].nv + 15) >> 4) {
    case 1: rc_run<1>(a, b, blk, keff, rank, Zs, sh); break;
    case 2: rc_run<2>(a, b, blk, keff, rank, Zs, sh); break;
    case 3: rc_run<3>(a, b, blk, keff, rank, Zs, sh); break;
    case 4: rc_run<4>(a, b, blk, keff, rank, Zs, sh); break;
    case 5: rc_run<5>(a, b, blk, keff, rank, Zs, sh); break;
    case 6: rc_run<6>(a, b, blk, keff, rank, Zs, sh); break;
    case 7: rc_run<7>(a, b, blk, keff, rank, Zs, sh); break;
    default: rc_run<8>(a, b, blk, keff, rank, Zs, sh); break;
  }
}

// ------------------------------------------------------------------------------------------------
// global truncation (ITensor truncate(), SURVEY A.3) + new bond bookkeeping + follow-up descriptor
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) truncate_kernel(DecompArgs a, DecompBuffers b, TruncParams tp) {
  // Only the non-zero weights take part (rows past a block's numerical rank report 0 and can never be kept); they are
  // compacted first, so the two O(n^2 / threads) ranking loops run over the candidates only.
  __shared__ double cP[NV_MAX];           // candidate weights, compact
  __shared__ double sSorted[NV_MAX];      // descending; then overwritten by its suffix sums
  __shared__ short cQ[NV_MAX], cI[NV_MAX], cI2[NV_MAX];   // charge, original index, kept candidates before
  __shared__ unsigned char sKeep[NV_MAX];
  __shared__ int sBlkOff[OCMPS_MAX_BLK + 1];
  __shared__ double sWarp[32];
  __shared__ int sWarpCnt[33];
  __shared__ double s_docut, s_kept;
  __shared__ int s_nfinal;
  DecompWork* w = b.dw;
  const int nv = w->nvtot;
  const int nblocks = w->nblocks;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < nblocks; i += blockDim.x) sBlkOff[i] = w->blk[i].p_off;
  if (tid == 0) { s_nfinal = 0; s_docut = 0.0; }
  // ---- compaction (order preserving): thread t owns entries 2t, 2t+1 ----
  const int i0 = 2 * tid, i1 = i0 + 1;
  const double p0 = i0 < nv ? b.P[i0] : 0.0, p1 = i1 < nv ? b.P[i1] : 0.0;
  const int f0 = p0 > 0.0, f1 = p1 > 0.0;
  int incl = f0 + f1;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int up = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += up; }
  if (lane == 31) sWarpCnt[warp + 1] = incl;
  if (tid == 0) sWarpCnt[0] = 0;
  __syncthreads();
  if (warp == 0) {
    int v = sWarpCnt[lane + 1];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int up = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += up; }
    sWarpCnt[lane + 1] = v;
  }
  __syncthreads();
  const int nnz = sWarpCnt[32];
  {
    int k = sWarpCnt[warp] + incl - f0 - f1;
    if (f0) { cP[k] = p0; cQ[k] = (short)b.vecq[i0]; cI[k] = (short)i0; ++k; }
    if (f1) { cP[k] = p1; cQ[k] = (short)b.vecq[i1]; cI[k] = (short)i1; }
  }
  __syncthreads();
  // ---- descending rank of every candidate: tpe (1..8) threads share the comparisons of one candidate ----
  {
    int tpe = 1;
    while (tpe < 8 && nnz * tpe * 2 <= (int)blockDim.x) tpe *= 2;
    const int sub = tid & (tpe - 1);
    for (int k0 = 0; k0 < nnz; k0 += (int)blockDim.x / tpe) {        // uniform trip count (shuffles inside)
      const int k = k0 + tid / tpe;
      const bool in = k < nnz;
      const double pk = in ? cP[k] : 0.0;
      int rank = 0;
      if (in)
        for (int j = sub; j < nnz; j += tpe) {
          const double pj = cP[j];
          rank += (pj > pk) || (pj == pk && j < k);
        }
      for (int o = 1; o < tpe; o <<= 1) rank += __shfl_xor_sync(0xffffffffu, rank, o);
      if (in && sub == 0) sSorted[rank] = pk;
    }
  }
  __syncthreads();
  // ---- suffix sums Suf[n] = sum_{i >= n} sorted[i] (ITensor accumulates them in `truncerr` walking up from the small
  // end); block-wide scan, thread t owns the two entries 2t, 2t+1 counted from the END of the candidate list ----
  const int origm = nv;                                    // ITensor's count includes the zero weights
  const int e0 = nnz - 1 - 2 * tid, e1 = e0 - 1;           // e0 > e1
  const double v0 = e0 >= 0 ? sSorted[e0] : 0.0, v1 = e1 >= 0 ? sSorted[e1] : 0.0;
  {
    double run = v0 + v1;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const double up = __shfl_up_sync(0xffffffffu, run, o); if (lane >= o) run += up; }
    if (lane == 31) sWarp[warp] = run;
    __syncthreads();
    if (warp == 0) {
      double ws = sWarp[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const double up = __shfl_up_sync(0xffffffffu, ws, o); if (lane >= o) ws += up; }
      sWarp[lane] = ws;
    }
    __syncthreads();
    const double base = warp > 0 ? sWarp[warp - 1] : 0.0;
    const double inc = base + run;
    if (e0 >= 0) sSorted[e0] = inc - v1;                    // Suf[e0]
    if (e1 >= 0) sSorted[e1] = inc;                         // Suf[e1]
  }
  __syncthreads();
  {
    // final n = largest n <= min(maxm, origm) - 1 with (n < minm or Suf[n] >= cutoff * scale); Suf[n] = 0 for n >= nnz
    const double total_w = nnz > 0 ? sSorted[0] : 0.0;
    const double scale = tp.rel_cutoff ? (total_w == 0.0 ? 1.0 : total_w) : 1.0;
    const double cut = tp.cutoff * scale;
    const int nmax = (tp.maxm < origm ? tp.maxm : origm) - 1;
    int best = 0;
    if (cut <= 0.0) {
      best = nmax > 0 ? nmax : 0;
    } else {
      const int lim = nmax < nnz - 1 ? nmax : nnz - 1;
      for (int n = tid; n <= lim; n += blockDim.x)
        if (n < tp.minm || sSorted[n] >= cut) best = n > best ? n : best;
      if (tp.minm - 1 > best && tp.minm - 1 <= nmax) best = tp.minm - 1;
    }
    if (best > 0) atomicMax(&s_nfinal, best);
  }
  __syncthreads();
  {
    // docut = midpoint of the two sorted values that straddle the cut (+ the degeneracy bump); zeros beyond nnz
    const int m = s_nfinal + 1;
    if (tid == 0) { sWarp[0] = 0.0; sWarp[1] = 0.0; }
    __syncthreads();
    if (e0 == m) sWarp[0] = v0;
    if (e1 == m) sWarp[0] = v1;
    if (e0 == m - 1) sWarp[1] = v0;
    if (e1 == m - 1) sWarp[1] = v1;
    __syncthreads();
    if (tid == 0) {
      double docut = 0.0;
      if (origm == 1) {
        docut = sWarp[1] / 2.0;                             // m - 1 = 0: the only weight
      } else if (origm > 1 && m < origm) {
        const double pm = sWarp[0], pm1 = sWarp[1];
        docut = (pm + pm1) / 2.0;
        if (fabs(pm - pm1) < 1e-3 * pm1) docut += 1e-3 * pm1;
      }
      s_docut = docut;
    }
    __syncthreads();
  }
  const double docut = s_docut;
  // ---- kept flags and their running count.  Candidates are in block order and blocks in ascending charge order, so
  // the new index of a kept state = kept states before its charge run + its rank by weight inside the run ----
  {
    const int ka = 2 * tid, kb = ka + 1;
    const int fa = ka < nnz && cP[ka] > docut, fb = kb < nnz && cP[kb] > docut;
    if (ka < nnz) sKeep[ka] = (unsigned char)fa;
    if (kb < nnz) sKeep[kb] = (unsigned char)fb;
    int inc = fa + fb;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int up = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += up; }
    __syncthreads();                   // (sWarpCnt is free again)
    if (lane == 31) sWarpCnt[warp + 1] = inc;
    if (tid == 0) sWarpCnt[0] = 0;
    __syncthreads();
    if (warp == 0) {
      int v = sWarpCnt[lane + 1];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int up = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += up; }
      sWarpCnt[lane + 1] = v;
    }
    __syncthreads();
    const int base = sWarpCnt[warp] + inc - fa - fb;     // kept candidates before ka
    if (ka < nnz) cI2[ka] = (short)base;
    if (kb < nnz) cI2[kb] = (short)(base + fa);
  }
  __syncthreads();
  const int total = sWarpCnt[32];
  int* inv_blk = b.pos + NV_MAX;       // per new index: block id, vector-in-block
  int* inv_v = b.pos + 2 * NV_MAX;
  double part = 0.0;
  for (int k = tid; k < nnz; k += blockDim.x) {
    if (!sKeep[k]) continue;
    const int qk = cQ[k];
    const double pk = cP[k];
    int rank = 0, j = k - 1;
    for (; j >= 0 && cQ[j] == qk; --j) rank += sKeep[j] && cP[j] >= pk;        // ties: the earlier candidate first
    const int pos0 = cI2[j + 1];                                              // kept before the run of this charge
    for (j = k + 1; j < nnz && cQ[j] == qk; ++j) rank += sKeep[j] && cP[j] > pk;
    const int pos = pos0 + rank;
    if (pos < tp.cap) {
      const int i = cI[k];
      a.qNew[pos] = qk;
      int bi = 0;                      // block of vector i: scan the (short) block table
      while (bi + 1 < nblocks && sBlkOff[bi + 1] <= i) ++bi;
      inv_blk[pos] = bi;
      inv_v[pos] = i - sBlkOff[bi];
      part += pk;
    }
  }
  {
    // sum of the kept weights: fixed index pattern per thread, fixed-order tree
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    __syncthreads();
    if (lane == 0) sWarp[warp] = part;
    __syncthreads();
    if (tid == 0) {
      double t = 0.0;
      for (int i = 0; i < 32; ++i) t += sWarp[i];
      s_kept = t;
    }
    __syncthreads();
  }
  if (tid == 0) {
    int k = total;
    if (k == 0 && nv > 0) {            // zero tensor: keep one arbitrary state (the first vector of the first block)
      k = 1;
      a.qNew[0] = b.vecq[0];
      inv_blk[0] = 0;
      inv_v[0] = 0;
    }
    if (k > tp.cap) { atomicOr(b.status, OCMPS_ST_CAPACITY); k = tp.cap; }
    w->newdim = k;
    *a.dimNew = k;
    // Frobenius norm of the tensor that carries the centre = sqrt(sum of kept weights), fixed summation order
    const double kept = s_kept;
    double scale = 1.0;
    if (tp.normalize) {
      const double nrm = sqrt(kept);
      if (nrm > 1e-16) scale = 1.0 / nrm;      // src/BH_tDMRG.cpp:183-184
    }
    w->scale = scale;
    const int n = w->n, m = w->m;
    GemmDesc g1;
    g1.pad = 0;
    g1.A = g1.B = nullptr; g1.C = nullptr; g1.M = g1.N = g1.K = 0; g1.lda = g1.ldb = g1.ldc = 1; g1.opA = g1.opB = 0;
    if (a.kind == DK_ORTH_LEFT) {        // neighbour (k x D*chiFar) = C (k x m) . nb_in (m x D*chiFar)
      const int far = a.D * (*a.dimNb);
      g1.A = a.partner; g1.opA = 0; g1.lda = m;
      g1.B = a.nb_in; g1.opB = 0; g1.ldb = far;
      g1.C = a.nb_out; g1.ldc = far; g1.M = k; g1.N = far; g1.K = m;
    } else if (a.kind == DK_ORTH_RIGHT) { // neighbour (chiFar*D x k) = nb_in (chiFar*D x n) . C (n x k)
      const int far = a.D * (*a.dimNb);
      g1.A = a.nb_in; g1.opA = 0; g1.lda = n;
      g1.B = a.partner; g1.opB = 0; g1.ldb = k;
      g1.C = a.nb_out; g1.ldc = k; g1.M = far; g1.N = k; g1.K = n;
    }
    b.descs[1] = g1;
  }
}

// ------------------------------------------------------------------------------------------------
// assembly of the two factors, one CTA per kept state j:
//   isometry  u_j = M z_j^H / |M z_j^H|  (scattered into column / row j, zero outside the charge block)
//   partner   sigma_j z_j * scale         (the tensor that carries the orthogonality centre)
// ------------------------------------------------------------------------------------------------
constexpr int BUILD_THREADS = 512;
__global__ void __launch_bounds__(BUILD_THREADS) build_factors_kernel(DecompArgs a, DecompBuffers b) {
  extern __shared__ __align__(16) unsigned char bsm[];
  __shared__ double red[BUILD_THREADS / 32];
  __shared__ double s_inv;
  const DecompWork* w = b.dw;
  const int k = w->newdim;
  const int kk = blockIdx.x;
  if (kk >= k) return;
  const int n = w->n, m = w->m, ld = w->ld, mode = w->mode;
  const int* comp_blk = b.comp_idx + NV_MAX;
  const int* comp_rank = b.comp_idx + 2 * NV_MAX;
  const int* vec_blk = b.vec_idx + NV_MAX;
  const int* vec_rank = b.vec_idx + 2 * NV_MAX;
  const int bi = b.pos[NV_MAX + kk], j = b.pos[2 * NV_MAX + kk];
  const DecompBlock B = w->blk[bi];
  const int nv = B.nv, len = B.len;
  const cplx* Zj = b.ywork + B.ws_off + (size_t)j * nv;
  const double sigma = sqrt(b.P[B.p_off + j]) * w->scale;
  cplx* zs = reinterpret_cast<cplx*>(bsm);            // z_j (nv)
  cplx* out = zs + nv;                                // M z_j^H (len)
  int* vidx = reinterpret_cast<int*>(out + len);      // index lists of the block, staged: the loads of X below then
  int* cidx = vidx + nv;                              // depend on nothing but shared memory and can all be in flight
  const int tid = threadIdx.x, lane = tid & 31, wp = tid >> 5;
  constexpr int NW = BUILD_THREADS / 32;
  for (int v = tid; v < nv; v += BUILD_THREADS) { zs[v] = Zj[v]; vidx[v] = b.vec_idx[B.vec_off + v]; }
  for (int c = tid; c < len; c += BUILD_THREADS) cidx[c] = b.comp_idx[B.comp_off + c];
  __syncthreads();
  double part = 0.0;
  if (mode == 0) {
    // vectors are columns of X: one warp per output component, lanes stride over the (nearly contiguous) columns,
    // four independent loads per lane and pass
    for (int c = wp; c < len; c += NW) {
      const cplx* row = a.X + (size_t)cidx[c] * ld;
      double sr = 0.0, si = 0.0;
      for (int v0 = 0; v0 < nv; v0 += 128) {
        cplx x[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int v = v0 + lane + 32 * u;
          x[u] = make_double2(0.0, 0.0);
          if (v < nv) x[u] = row[vidx[v]];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int v = v0 + lane + 32 * u;
          if (v < nv) {
            const cplx z = zs[v];
            sr += x[u].x * z.x + x[u].y * z.y;          // x * conj(z)
            si += x[u].y * z.x - x[u].x * z.y;
          }
        }
      }
      sr = warp_sum(sr); si = warp_sum(si);
      if (lane == 0) { out[c] = make_double2(sr, si); part += sr * sr + si * si; }
    }
  } else {
    // vectors are rows of X: a warp takes 8 consecutive output components x 4 interleaved ranges of vectors
    // (consecutive lanes read consecutive columns), reduced over the ranges with two shuffles
    const int cl = lane & 7, g = lane >> 3;
    for (int c0 = 8 * wp; c0 < len; c0 += 8 * NW) {
      const int c = c0 + cl;
      const bool in = c < len;
      const cplx* colp = a.X + (in ? cidx[c] : 0);
      double sr = 0.0, si = 0.0;
      if (in) {
#pragma unroll 4
        for (int v = g; v < nv; v += 4) {
          const cplx x = colp[(size_t)vidx[v] * ld], z = zs[v];
          sr += x.x * z.x + x.y * z.y;
          si += x.y * z.x - x.x * z.y;
        }
      }
      sr += __shfl_xor_sync(0xffffffffu, sr, 8);  si += __shfl_xor_sync(0xffffffffu, si, 8);
      sr += __shfl_xor_sync(0xffffffffu, sr, 16); si += __shfl_xor_sync(0xffffffffu, si, 16);
      if (in && g == 0) { out[c] = make_double2(sr, si); part += sr * sr + si * si; }
    }
  }
  part = warp_sum(part);
  if ((tid & 31) == 0) red[tid >> 5] = part;
  __syncthreads();
  if (tid == 0) {
    double t = 0.0;
    for (int i = 0; i < BUILD_THREADS / 32; ++i) t += red[i];
    s_inv = t > 0.0 ? rsqrt(t) : 0.0;
  }
  __syncthreads();
  const double inv = s_inv;
  // isometry: element (component, kk); partner: element (vector, kk)
  const int ncomp = mode == 0 ? n : m, nvec = mode == 0 ? m : n;
  for (int c = tid; c < ncomp; c += BUILD_THREADS) {
    cplx v = make_double2(0.0, 0.0);
    if (comp_blk[c] == bi) { const cplx o = out[comp_rank[c]]; v = make_double2(o.x * inv, o.y * inv); }
    if (mode == 0) a.iso[(size_t)c * k + kk] = v; else a.iso[(size_t)kk * m + c] = v;
  }
  if (a.qNb != nullptr && (a.kind == DK_ORTH_LEFT || a.kind == DK_ORTH_RIGHT)) {
    // gauge push fused in: row / column kk of (carry matrix . neighbour).  The carry sigma_j z_j lives in one charge
    // sector, so for every far-bond index exactly one physical index of the neighbour contributes.
    const int D = a.D, chiFar = *a.dimNb, qj = B.q;
    if (a.kind == DK_ORTH_LEFT) {        // out[kk][s][r] = sum_v C[kk][v] nb[v][s][r],  s = qFar[r] - q_j
      const long long far = (long long)D * chiFar;
      for (int r = tid; r < chiFar; r += BUILD_THREADS) {
        const int sx = a.qNb[r] - qj;
        double ar = 0.0, ai = 0.0;
        if (sx >= 0 && sx < D) {
          const cplx* col = a.nb_in + (long long)sx * chiFar + r;
#pragma unroll 4
          for (int t = 0; t < nv; ++t) {
            const cplx z = zs[t], x = col[(long long)vidx[t] * far];
            ar += z.x * x.x - z.y * x.y;
            ai += z.x * x.y + z.y * x.x;
          }
        }
        for (int sp = 0; sp < D; ++sp)
          a.nb_out[(long long)kk * far + (long long)sp * chiFar + r] = sp == sx ? make_double2(ar * sigma, ai * sigma) : make_double2(0.0, 0.0);
      }
    } else {                             // out[l][s][kk] = sum_v nb[l][s][v] C[v][kk],  s = q_j - qFar[l]
      for (int l = tid; l < chiFar; l += BUILD_THREADS) {
        const int sx = qj - a.qNb[l];
        double ar = 0.0, ai = 0.0;
        if (sx >= 0 && sx < D) {
          const cplx* row = a.nb_in + ((long long)l * D + sx) * n;
#pragma unroll 4
          for (int t = 0; t < nv; ++t) {
            const cplx z = zs[t], x = row[vidx[t]];
            ar += z.x * x.x - z.y * x.y;
            ai += z.x * x.y + z.y * x.x;
          }
        }
        for (int sp = 0; sp < D; ++sp)
          a.nb_out[((long long)l * D + sp) * k + kk] = sp == sx ? make_double2(ar * sigma, ai * sigma) : make_double2(0.0, 0.0);
      }
    }
    return;
  }
  for (int v = tid; v < nvec; v += BUILD_THREADS) {
    cplx o = make_double2(0.0, 0.0);
    if (vec_blk[v] == bi) { const cplx z = zs[vec_rank[v]]; o = make_double2(z.x * sigma, z.y * sigma); }
    if (mode == 0) a.partner[(size_t)kk * m + v] = o; else a.partner[(size_t)v * k + kk] = o;
  }
}

// ------------------------------------------------------------------------------------------------
// Frobenius normalisation of one site tensor, deterministic two-stage reduction
// ------------------------------------------------------------------------------------------------
constexpr int NORM_CTAS = 32;
constexpr int NORM_THREADS = 256;

__device__ __forceinline__ void norm_partial_body(const cplx* x, long long count, double* partial) {
  __shared__ double red[NORM_THREADS];
  double s = 0.0;
  for (long long e = blockIdx.x * (long long)NORM_THREADS + threadIdx.x; e < count; e += (long long)NORM_CTAS * NORM_THREADS) {
    cplx u = x[e];
    s += u.x * u.x + u.y * u.y;
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = NORM_THREADS / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) partial[blockIdx.x] = red[0];
}
__device__ __forceinline__ double norm_total(const double* partial) {
  double s = 0.0;
  for (int i = 0; i < NORM_CTAS; ++i) s += partial[i];
  return s;
}
__global__ void __launch_bounds__(NORM_THREADS) norm_partial_site_kernel(const cplx* x, const int* dimL, const int* dimR, int D,
                                                                        double* partial) {
  norm_partial_body(x, (long long)(*dimL) * D * (*dimR), partial);
}
__global__ void scale_site_kernel(cplx* x, const int* dimL, const int* dimR, int D, const double* partial) {
  const double nrm = sqrt(norm_total(partial));
  if (!(nrm > 0.0)) return;
  const double inv = 1.0 / nrm;
  const long long count = (long long)(*dimL) * D * (*dimR);
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < count; e += (long long)gridDim.x * blockDim.x) {
    cplx u = x[e];
    x[e] = make_double2(u.x * inv, u.y * inv);
  }
}
__global__ void norm_finish_kernel(const double* partial, double* out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) *out = sqrt(norm_total(partial));
}

int grid_for(long long elems, int threads, int cap = 1184) {
  long long g = (elems + threads - 1) / threads;
  if (g < 1) g = 1;
  if (g > cap) g = cap;
  return (int)g;
}

}  // namespace

static bool g_jac_attr_set[64] = {false};

void debug_jacobi_counters(unsigned long long* out, bool reset) {
  cudaMemcpyFromSymbol(out, g_jac_dbg, sizeof(unsigned long long) * 8);
  if (reset) { unsigned long long z[8] = {0}; cudaMemcpyToSymbol(g_jac_dbg, z, sizeof(z)); }
}

void debug_row_cluster_counters(unsigned long long* out, bool reset) {
  cudaMemcpyFromSymbol(out, g_rc_dbg, sizeof(unsigned long long) * 2);
  if (reset) { unsigned long long z[2] = {0, 0}; cudaMemcpyToSymbol(g_rc_dbg, z, sizeof(z)); }
}

// von Neumann entropy of the spectrum the last decomposition left in b.P (include/correlations.hpp:119-148):
// S = -sum_{p > 1e-12} p ln p over the squared singular values of all charge blocks.  One CTA, fixed-order tree.
__global__ void __launch_bounds__(256) spectrum_entropy_kernel(DecompBuffers b, double* out) {
  __shared__ double red[256];
  const int nv = b.dw->nvtot;
  double acc = 0.0;
  for (int i = threadIdx.x; i < nv; i += 256) {
    const double p = b.P[i];
    if (p > 1e-12) acc -= p * log(p);
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = red[0];
}

void launch_spectrum_entropy(const DecompBuffers& b, double* out, cudaStream_t s) {
  spectrum_entropy_kernel<<<1, 256, 0, s>>>(b, out);
}

void launch_decomp_setup(const DecompArgs& a, const DecompBuffers& b, cudaStream_t s) {
  decomp_setup_kernel<<<1, SETUP_THREADS, 0, s>>>(a, b);
}

#include <vector>
#include <mutex>
static bool g_prof_on = false;
static std::vector<std::pair<cudaEvent_t, cudaEvent_t>> g_prof_events;
static size_t g_prof_used = 0;

bool profile_is_on() { return g_prof_on; }

void profile_enable(bool on) {
  g_prof_on = on;
  g_prof_used = 0;
  double z[2] = {0.0, 0.0};
  cudaMemcpyToSymbol(g_jac_flops, z, sizeof(z));
}
// out: [0] total ms inside the block-SVD kernel, [1] launches, [2] block-summed algorithmic flops, [3] dense-formula flops
void profile_read(double* out) {
  cudaDeviceSynchronize();
  double ms = 0.0;
  for (size_t i = 0; i < g_prof_used; ++i) {
    float t = 0.f;
    cudaEventElapsedTime(&t, g_prof_events[i].first, g_prof_events[i].second);
    ms += t;
  }
  double fl[2];
  cudaMemcpyFromSymbol(fl, g_jac_flops, sizeof(fl));
  out[0] = ms; out[1] = (double)g_prof_used; out[2] = fl[0]; out[3] = fl[1];
}

void launch_jacobi_blocks(const DecompArgs& a, const DecompBuffers& b, int nblk_launch, size_t smem_limit, bool need_global,
                          bool long_rows, double rank_tol, int max_rows, int capV, int capC, bool spread_rows, cudaStream_t s,
                          const SvdFork* fork) {
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (g_prof_on) {
    if (g_prof_used == g_prof_events.size()) {
      cudaEvent_t x, y;
      cudaEventCreate(&x); cudaEventCreate(&y);
      g_prof_events.push_back({x, y});
    }
    e0 = g_prof_events[g_prof_used].first; e1 = g_prof_events[g_prof_used].second;
    ++g_prof_used;
    cudaEventRecord(e0, s);
  }
  struct Tail { cudaEvent_t e; cudaStream_t s; ~Tail() { if (e) cudaEventRecord(e, s); } } tail{e1, s};
  int dev = 0;
  cudaGetDevice(&dev);
  static std::mutex attr_mu;
  if (dev < 64) {
  std::lock_guard<std::mutex> attr_lock(attr_mu);
  if (!g_jac_attr_set[dev]) {
    cudaFuncSetAttribute(jacobi_blocks_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(jacobi_blocks_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(build_factors_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    cudaFuncSetAttribute(jacobi_rot_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(JAC_BLOCKED_ROWS * 16 * JAC_EPL * sizeof(cplx)));
    cudaFuncSetAttribute(jacobi_rows_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(JAC_BLOCKED_ROWS * 16 * JAC_EPL * sizeof(cplx)));
    cudaFuncSetAttribute(jacobi_big_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(BJ_MAX_ROWS * (BJ_TPP * BJ_MAX_EPL + 4) * sizeof(cplx)));
    cudaFuncSetAttribute(qr_big_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((32 * BJ_MAX_ROWS + BJ_MAX_ROWS) * sizeof(cplx)));
    g_jac_attr_set[dev] = true;
  }
  }
  // Blocks beyond the register-resident rotation kernel (more than 64 rows of R, or rows longer than 128) exist only when the
  // capacities allow them; from chi_cap >= 112 on they are finished by the cluster kernel instead of the generic loops.
  static const bool big_env = [] { const char* e = getenv("OCMPS_BIG_CLUSTER"); return !(e && e[0] == '0'); }();
  int big_on = (big_env && max_rows >= BJ_MIN_CAP) ? 1 : 0;
  // OCMPS_GRAM=1: the large blocks of the gate decompositions get their triangular factor from the Gram matrix (DMMA) + pivoted
  // Cholesky inside the register-cached instantiation (flag bit 1 of big_on; gram_chol_block).  Off by default: measured on a B200
  // the single evaluation is the same within noise (0.862 vs 0.856 evaluations/s) while the 48 concurrent chains of a cfg3
  // Hessian lose a fifth of their throughput (10.8 s vs 8.8 s) -- profiles/r02_results.md.
  static const bool gram_env = [] { const char* e = getenv("OCMPS_GRAM"); return e && e[0] == '1'; }();
  if (gram_env && (a.kind == DK_GATE_LEFT || a.kind == DK_GATE_RIGHT)) big_on |= 2;
  // Two independent chains of kernels inside one decomposition: blocks that fit one SM (register-cached QR -> jacobi_rot_kernel) on
  // `s`, blocks that need a cluster (qr_big_kernel -> jacobi_big_kernel) on the fork stream.  jacobi_big_kernel also takes the blocks
  // the register-cached QR hands over with more than 64 rows of R, so it waits for that kernel as well.  (At chi = 256 the chains are
  // 156 + 173 us and 180 + 431 us long: 0.61 ms per decomposition side by side instead of 0.94 ms one after the other.)
  static const bool fork_env = [] { const char* e = getenv("OCMPS_SVD_FORK"); return !(e && e[0] == '0'); }();
  const bool forked = fork_env && (big_on & 1) && fork && fork->stream;
  cudaStream_t sb = forked ? fork->stream : s;
  if (forked) { cudaEventRecord(fork->ev_fork, s); cudaStreamWaitEvent(sb, fork->ev_fork, 0); }
  jacobi_blocks_kernel<true, true><<<nblk_launch, JAC_THREADS, smem_limit, s>>>(a, b, (int)(smem_limit / sizeof(cplx)), rank_tol, big_on);
  if (forked) cudaEventRecord(fork->ev_first, s);
  if (long_rows) jacobi_blocks_kernel<true, false><<<nblk_launch, JAC_THREADS, smem_limit, s>>>(a, b, (int)(smem_limit / sizeof(cplx)), rank_tol, big_on);
  if (need_global) jacobi_blocks_kernel<false, false><<<nblk_launch, JAC_THREADS, 0, s>>>(a, b, (int)(smem_limit / sizeof(cplx)), rank_tol, big_on);
  // (after ALL first-stage variants of its stream: each of them publishes the hand-over flag of the blocks it owns)
  if (big_on & 1) {      // cluster QR of the blocks the register-cached kernel does not take
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(nblk_launch * BJ_C, 1, 1);
    cfg.blockDim = dim3(BJ_THREADS, 1, 1);
    cfg.dynamicSmemBytes = (size_t)(32 * BJ_MAX_ROWS + BJ_MAX_ROWS) * sizeof(cplx);
    cfg.stream = sb;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = BJ_C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, qr_big_kernel, a, b, (int)(smem_limit / sizeof(cplx)), rank_tol);
  }
  if (spread_rows) {   // second stage of the register-cached blocks: one cluster per block, spread over it from RC_MIN_ROWS rows of R on
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(nblk_launch * RC_C, 1, 1);
    cfg.blockDim = dim3(JAC_THREADS, 1, 1);
    cfg.dynamicSmemBytes = (size_t)JAC_BLOCKED_ROWS * 16 * JAC_EPL * sizeof(cplx);
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = RC_C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, jacobi_rows_cluster_kernel, a, b, (int)(smem_limit / sizeof(cplx)));
  } else {
    jacobi_rot_kernel<<<nblk_launch, JAC_THREADS, JAC_BLOCKED_ROWS * 16 * JAC_EPL * sizeof(cplx), s>>>(a, b, (int)(smem_limit / sizeof(cplx)));
  }
  if (big_on & 1) {
    if (forked) cudaStreamWaitEvent(sb, fork->ev_first, 0);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(nblk_launch * BJ_C, 1, 1);
    cfg.blockDim = dim3(BJ_THREADS, 1, 1);
    cfg.dynamicSmemBytes = (size_t)BJ_MAX_ROWS * (BJ_TPP * BJ_MAX_EPL + 4) * sizeof(cplx);
    cfg.stream = sb;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = BJ_C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, jacobi_big_kernel, a, b);
    if (forked) { cudaEventRecord(fork->ev_join, sb); cudaStreamWaitEvent(s, fork->ev_join, 0); }
  }
}

void launch_truncate(const DecompArgs& a, const DecompBuffers& b, const TruncParams& tp, cudaStream_t s) {
  truncate_kernel<<<1, 1024, 0, s>>>(a, b, tp);
}

void launch_build_factors(const DecompArgs& a, const DecompBuffers& b, int cap_k, int cap_vec, int cap_comp, cudaStream_t s) {
  const size_t sm = (sizeof(cplx) + sizeof(int)) * (size_t)(cap_vec + cap_comp);
  build_factors_kernel<<<cap_k, BUILD_THREADS, sm, s>>>(a, b);
}

void launch_norm_only(const cplx* x, const int* dimL, const int* dimR, int D, double* partial, double* out, int max_elems,
                      cudaStream_t s) {
  (void)max_elems;
  norm_partial_site_kernel<<<NORM_CTAS, NORM_THREADS, 0, s>>>(x, dimL, dimR, D, partial);
  norm_finish_kernel<<<1, 32, 0, s>>>(partial, out);
}

void launch_normalize_site(cplx* x, const int* dimL, const int* dimR, int D, double* partial, int max_elems, cudaStream_t s) {
  norm_partial_site_kernel<<<NORM_CTAS, NORM_THREADS, 0, s>>>(x, dimL, dimR, D, partial);
  scale_site_kernel<<<grid_for(max_elems, 256), 256, 0, s>>>(x, dimL, dimR, D, partial);
}
