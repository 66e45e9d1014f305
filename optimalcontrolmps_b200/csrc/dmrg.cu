// Kernels of the two-site DMRG ground-state solver (ocmps_ground_state_dmrg in engine.cu).
//
// Two-site tensors theta[l, s1, s2, r] use the layout the gate decompositions read: a (chiL*D) x (D*chiR) row-major matrix.
// The Krylov vectors share it, so the Ritz vector is handed to the decomposition as it is.
//
// Environments are dense complex matrices, three per bond (the identity channel of the MPO is implicit because the sites
// between the environment and the centre are isometries):
//   left  bond b (sites < b):  [0] H_L, [1] -J a on site b-1, [2] -J a+ on site b-1         E[a', a] = <a'|O|a>
//   right bond b (sites >= b): [0] H_R, [1] a+ on site b,      [2] a on site b              S[b, b'] = <b'|O|b>  (transposed)
// so that H_eff theta = E_c . theta and theta . S_c are plain products on the first and last index of theta.
// All sizes are read from device memory (bond dimensions are decided on the GPU); reductions are two-stage with a fixed
// order, so every result is bit-identical from call to call.
#include <cmath>
#include "ocmps_internal.h"

namespace {

constexpr int KRY_CTAS = 128;
constexpr int KRY_THREADS = 256;
constexpr int KMAX = DMRG_KRYLOV;

int grid_for(long long elems, int threads, int cap = 1184) {
  long long g = (elems + threads - 1) / threads;
  if (g < 1) g = 1;
  if (g > cap) g = cap;
  return (int)g;
}

__device__ __forceinline__ bool ks_stopped(const KrylovState* ks) { return ks && ks->stop; }
__device__ __forceinline__ double kfac(double U, int n) { return 0.5 * U * (double)n * (double)(n - 1); }
__device__ __forceinline__ void cadd(cplx& acc, double f, cplx v) { acc.x += f * v.x; acc.y += f * v.y; }

// sum of the KRY_CTAS partials of dot product i, fixed order (every CTA that needs it recomputes it)
__device__ __forceinline__ void partial_sum(const double* partial, int i, double& re, double& im) {
  re = 0.0; im = 0.0;
  for (int c = 0; c < KRY_CTAS; ++c) { re += partial[(i * KRY_CTAS + c) * 2]; im += partial[(i * KRY_CTAS + c) * 2 + 1]; }
}

// ---- H_eff ----
// descs[c] = E_c (chiL x chiL) . theta (chiL x D*D*chiR) -> Y_c;  descs[3+c] = theta (chiL*D*D x chiR) . S_c -> Z_c.
// After a Krylov breakdown the products are empty (M = 0: every CTA of the GEMM exits at once).
__global__ void heff_setup_kernel(GemmDesc* descs, const cplx* V, cplx* Y, cplx* Z, long long ystride, const cplx* EL, const cplx* ER,
                                  long long estride, const int* dimL, const int* dimR, int D, const KrylovState* ks) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const int cl = *dimL, cr = *dimR, n1 = D * D * cr;
  const bool live = !ks_stopped(ks);
  for (int c = 0; c < 3; ++c) {
    GemmDesc g;
    g.pad = 0; g.opA = 0; g.opB = 0;
    g.A = EL + c * estride; g.lda = cl;
    g.B = V; g.ldb = n1;
    g.C = Y + c * ystride; g.ldc = n1;
    g.M = live ? cl : 0; g.N = n1; g.K = cl;
    descs[c] = g;
    g.A = V; g.lda = cr;
    g.B = ER + c * estride; g.ldb = cr;
    g.C = Z + c * ystride; g.ldc = cr;
    g.M = live ? cl * D * D : 0; g.N = cr; g.K = cr;
    descs[3 + c] = g;
  }
}

// W = H_eff V from the boundary products: on-site terms K on s1 and s2, the hopping inside theta, a+ / a on s1 after the
// left channels 1 / 2, -J a / -J a+ on s2 after the right channels 1 / 2.  Entries outside the charge sector
// qL[l] + s1 + s2 = qR[r] are written as exact zeros.  One thread per entry.
__global__ void __launch_bounds__(256) heff_combine_kernel(const cplx* __restrict__ V, const cplx* __restrict__ Y,
                                                           const cplx* __restrict__ Z, long long ystride, cplx* __restrict__ W,
                                                           const int* dimL, const int* dimR, const int* __restrict__ qL,
                                                           const int* __restrict__ qR, int D, double J, double U,
                                                           const KrylovState* ks) {
  if (ks_stopped(ks)) return;
  const int cl = *dimL, cr = *dimR;
  const long long total = (long long)cl * D * D * cr;
  const cplx *Y0 = Y, *Y1 = Y + ystride, *Y2 = Y + 2 * ystride;
  const cplx *Z0 = Z, *Z1 = Z + ystride, *Z2 = Z + 2 * ystride;
  const long long s1s = (long long)D * cr, s2s = cr;        // strides of s1, s2
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(e % cr);
    const int t2 = (int)((e / cr) % D);
    const int t1 = (int)((e / s1s) % D);
    const int l = (int)(e / (s1s * D));
    cplx acc = make_double2(0.0, 0.0);
    if (qL[l] + t1 + t2 == qR[r]) {
      acc = Y0[e];
      acc.x += Z0[e].x; acc.y += Z0[e].y;
      cadd(acc, kfac(U, t1) + kfac(U, t2), V[e]);
      if (t1 + 1 < D && t2 >= 1) cadd(acc, -J * sqrt((double)(t1 + 1) * t2), V[e + s1s - s2s]);     // a_1 a+_2
      if (t1 >= 1 && t2 + 1 < D) cadd(acc, -J * sqrt((double)t1 * (t2 + 1)), V[e - s1s + s2s]);     // a+_1 a_2
      if (t1 >= 1) cadd(acc, sqrt((double)t1), Y1[e - s1s]);                                         // a+_1 (-J a_left)
      if (t1 + 1 < D) cadd(acc, sqrt((double)(t1 + 1)), Y2[e + s1s]);                                // a_1 (-J a+_left)
      if (t2 + 1 < D) cadd(acc, -J * sqrt((double)(t2 + 1)), Z1[e + s2s]);                           // -J a_2 a+_right
      if (t2 >= 1) cadd(acc, -J * sqrt((double)t2), Z2[e - s2s]);                                    // -J a+_2 a_right
    }
    W[e] = acc;
  }
}

// ---- environment update ----
// side 0 (left, A = left isometry of site j):   T_c = E_c . A,  E'_c = A^H . T'_c
// side 1 (right, A = right isometry of site j): T_c = A . S_c,  S'_c = T'_c . A^H
// dimL / dimR: bonds j and j+1.  T' is written by env_combine_kernel between the two GEMMs.
__global__ void env_setup_kernel(GemmDesc* descs, int side, const cplx* A, const cplx* Ein, cplx* Eout, cplx* T, cplx* T2,
                                 long long tstride, long long estride, const int* dimL, const int* dimR, int D) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const int cl = *dimL, cr = *dimR;
  for (int c = 0; c < 3; ++c) {
    GemmDesc g, h;
    g.pad = h.pad = 0; g.opA = g.opB = h.opA = h.opB = 0;
    if (side == 0) {
      g.A = Ein + c * estride; g.lda = cl; g.B = A; g.ldb = D * cr; g.C = T + c * tstride; g.ldc = D * cr;
      g.M = cl; g.N = D * cr; g.K = cl;
      h.A = A; h.opA = 1; h.lda = cr; h.B = T2 + c * tstride; h.ldb = cr; h.C = Eout + c * estride; h.ldc = cr;
      h.M = cr; h.N = cr; h.K = cl * D;
    } else {
      g.A = A; g.lda = cr; g.B = Ein + c * estride; g.ldb = cr; g.C = T + c * tstride; g.ldc = cr;
      g.M = cl * D; g.N = cr; g.K = cr;
      h.A = T2 + c * tstride; h.lda = D * cr; h.B = A; h.opB = 1; h.ldb = D * cr; h.C = Eout + c * estride; h.ldc = cl;
      h.M = cl; h.N = cl; h.K = D * cr;
    }
    descs[c] = g;
    descs[3 + c] = h;
  }
}

// T'_c[row, t, col] from the three products T_c and the site tensor A (identity channel), one thread per entry:
//   left:  T'_0 = T_0 + a+ T_1 + a T_2 + K A,          T'_1 = -J a A,  T'_2 = -J a+ A
//   right: T'_0 = T_0 - J a T_1 - J a+ T_2 + K A,      T'_1 = a+ A,    T'_2 = a A
__global__ void __launch_bounds__(256) env_combine_kernel(int side, const cplx* __restrict__ A, const cplx* __restrict__ T,
                                                          cplx* __restrict__ T2, long long tstride, const int* dimL,
                                                          const int* dimR, int D, double J, double U) {
  const int cl = *dimL, cr = *dimR;
  const long long total = (long long)cl * D * cr;
  const cplx *T0 = T, *T1 = T + tstride, *Tb = T + 2 * tstride;
  cplx *O0 = T2, *O1 = T2 + tstride, *O2 = T2 + 2 * tstride;
  const double f1 = side == 0 ? 1.0 : -J;          // factor of the channel-1 / channel-2 terms of T'_0
  const double g1 = side == 0 ? -J : 1.0;          // factor of T'_1, T'_2
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int t = (int)((e / cr) % D);
    const double up = sqrt((double)(t + 1)), dn = sqrt((double)t);     // (a X)[t] = up X[t+1], (a+ X)[t] = dn X[t-1]
    const cplx a_up = t + 1 < D ? A[e + cr] : make_double2(0.0, 0.0);
    const cplx a_dn = t >= 1 ? A[e - cr] : make_double2(0.0, 0.0);
    cplx o0 = T0[e];
    cadd(o0, kfac(U, t), A[e]);
    if (side == 0) {
      if (t >= 1) cadd(o0, f1 * dn, T1[e - cr]);
      if (t + 1 < D) cadd(o0, f1 * up, Tb[e + cr]);
      O1[e] = make_double2(g1 * up * a_up.x, g1 * up * a_up.y);
      O2[e] = make_double2(g1 * dn * a_dn.x, g1 * dn * a_dn.y);
    } else {
      if (t + 1 < D) cadd(o0, f1 * up, T1[e + cr]);
      if (t >= 1) cadd(o0, f1 * dn, Tb[e - cr]);
      O1[e] = make_double2(g1 * dn * a_dn.x, g1 * dn * a_dn.y);
      O2[e] = make_double2(g1 * up * a_up.x, g1 * up * a_up.y);
    }
    O0[e] = o0;
  }
}

// ---- Lanczos ----
// partial[(i * KRY_CTAS + cta) * 2 + {0, 1}] = this CTA's share of <V_i | w> (re, im), i < nvec
__global__ void __launch_bounds__(KRY_THREADS) krylov_dot_kernel(const cplx* __restrict__ V, long long vstride, int nvec,
                                                                 const cplx* __restrict__ w, const int* dimL, const int* dimR, int D,
                                                                 const KrylovState* ks, double* __restrict__ partial) {
  if (ks_stopped(ks)) return;
  __shared__ double red[KRY_THREADS];
  const long long n = (long long)(*dimL) * D * D * (*dimR);
  double acc[2 * (KMAX + 1)];
#pragma unroll
  for (int i = 0; i < 2 * (KMAX + 1); ++i) acc[i] = 0.0;
  for (long long e = blockIdx.x * (long long)KRY_THREADS + threadIdx.x; e < n; e += (long long)KRY_CTAS * KRY_THREADS) {
    const cplx x = w[e];
#pragma unroll
    for (int i = 0; i < KMAX + 1; ++i) {
      if (i < nvec) {
        const cplx v = V[i * vstride + e];
        acc[2 * i] += v.x * x.x + v.y * x.y;
        acc[2 * i + 1] += v.x * x.y - v.y * x.x;
      }
    }
  }
  for (int k = 0; k < 2 * nvec; ++k) {
    red[threadIdx.x] = acc[k];
    __syncthreads();
    for (int o = KRY_THREADS / 2; o > 0; o >>= 1) {
      if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
      __syncthreads();
    }
    if (threadIdx.x == 0) partial[((k >> 1) * KRY_CTAS + blockIdx.x) * 2 + (k & 1)] = red[0];
    __syncthreads();
  }
}

// V_0 = X / |X| (partials of <X|X>); starts a new Krylov space
__global__ void krylov_init_kernel(const cplx* __restrict__ X, cplx* __restrict__ V0, const int* dimL, const int* dimR, int D,
                                   KrylovState* ks, const double* __restrict__ partial) {
  double nn, im;
  partial_sum(partial, 0, nn, im);
  const double inv = nn > 0.0 ? 1.0 / sqrt(nn) : 0.0;
  const long long n = (long long)(*dimL) * D * D * (*dimR);
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
    V0[e] = make_double2(X[e].x * inv, X[e].y * inv);
  if (blockIdx.x == 0 && threadIdx.x == 0) { ks->nk = 0; ks->stop = 0; }
}

// alpha_it = <V_it | w>;  w -= alpha_it V_it + beta_{it-1} V_{it-1}
__global__ void krylov_alpha_kernel(const cplx* __restrict__ V, long long vstride, int it, cplx* __restrict__ w, const int* dimL,
                                    const int* dimR, int D, KrylovState* ks, const double* __restrict__ partial) {
  if (ks->stop) return;
  double a, im;
  partial_sum(partial, 0, a, im);
  const double b = it > 0 ? ks->beta[it - 1] : 0.0;
  const cplx* v1 = V + it * vstride;
  const cplx* v0 = V + (it > 0 ? it - 1 : 0) * vstride;
  const long long n = (long long)(*dimL) * D * D * (*dimR);
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    cplx x = w[e];
    x.x -= a * v1[e].x + b * v0[e].x;
    x.y -= a * v1[e].y + b * v0[e].y;
    w[e] = x;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) { ks->alpha[it] = a; ks->nk = it + 1; }
}

// full reorthogonalisation: w -= sum_{i < nvec} <V_i | w> V_i
__global__ void krylov_reorth_kernel(const cplx* __restrict__ V, long long vstride, int nvec, cplx* __restrict__ w, const int* dimL,
                                     const int* dimR, int D, const KrylovState* ks, const double* __restrict__ partial) {
  if (ks->stop) return;
  double cr[KMAX + 1], ci[KMAX + 1];
  for (int i = 0; i < nvec; ++i) partial_sum(partial, i, cr[i], ci[i]);
  const long long n = (long long)(*dimL) * D * D * (*dimR);
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    cplx x = w[e];
    for (int i = 0; i < nvec; ++i) {
      const cplx v = V[i * vstride + e];
      x.x -= cr[i] * v.x - ci[i] * v.y;
      x.y -= cr[i] * v.y + ci[i] * v.x;
    }
    w[e] = x;
  }
}

// beta_it = |w|; V_{it+1} = w / beta_it, or a breakdown (beta <= 1e-12 |alpha_it|) that stops the Krylov space here
__global__ void krylov_next_kernel(cplx* __restrict__ V, long long vstride, int it, const cplx* __restrict__ w, const int* dimL,
                                   const int* dimR, int D, KrylovState* ks, const double* __restrict__ partial) {
  if (ks->stop) return;
  double nn, im;
  partial_sum(partial, 0, nn, im);
  const double b = sqrt(nn > 0.0 ? nn : 0.0);
  if (!(b > 1e-12 * fabs(ks->alpha[it]))) {        // every CTA takes the same decision
    if (blockIdx.x == 0 && threadIdx.x == 0) ks->stop = 1;
    return;
  }
  const double inv = 1.0 / b;
  cplx* vn = V + (it + 1) * vstride;
  const long long n = (long long)(*dimL) * D * D * (*dimR);
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
    vn[e] = make_double2(w[e].x * inv, w[e].y * inv);
  if (blockIdx.x == 0 && threadIdx.x == 0) ks->beta[it] = b;
}

// lowest eigenpair of the nk x nk tridiagonal matrix (cyclic Jacobi); the eigenvector is normalised with y[0] >= 0
__global__ void krylov_ritz_kernel(KrylovState* ks) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const int k = ks->nk;
  double A[KMAX][KMAX], Q[KMAX][KMAX];
  for (int i = 0; i < KMAX; ++i)
    for (int j = 0; j < KMAX; ++j) { A[i][j] = 0.0; Q[i][j] = i == j ? 1.0 : 0.0; }
  for (int i = 0; i < k; ++i) {
    A[i][i] = ks->alpha[i];
    if (i + 1 < k) { A[i][i + 1] = ks->beta[i]; A[i + 1][i] = ks->beta[i]; }
  }
  for (int sweep = 0; sweep < 64; ++sweep) {
    double off = 0.0;
    for (int p = 0; p < k; ++p)
      for (int q = p + 1; q < k; ++q) off += A[p][q] * A[p][q];
    if (off == 0.0) break;
    for (int p = 0; p < k; ++p)
      for (int q = p + 1; q < k; ++q) {
        if (A[p][q] == 0.0) continue;
        const double th = (A[q][q] - A[p][p]) / (2.0 * A[p][q]);
        const double t = (th >= 0.0 ? 1.0 : -1.0) / (fabs(th) + sqrt(th * th + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int r = 0; r < k; ++r) {              // columns p, q
          const double ap = A[r][p], aq = A[r][q];
          A[r][p] = c * ap - s * aq; A[r][q] = s * ap + c * aq;
        }
        for (int r = 0; r < k; ++r) {              // rows p, q
          const double ap = A[p][r], aq = A[q][r];
          A[p][r] = c * ap - s * aq; A[q][r] = s * ap + c * aq;
        }
        A[p][q] = A[q][p] = 0.0;
        for (int r = 0; r < k; ++r) {
          const double qp = Q[r][p], qq = Q[r][q];
          Q[r][p] = c * qp - s * qq; Q[r][q] = s * qp + c * qq;
        }
      }
  }
  int m = 0;
  for (int i = 1; i < k; ++i) if (A[i][i] < A[m][m]) m = i;
  double nrm = 0.0;
  for (int i = 0; i < k; ++i) nrm += Q[i][m] * Q[i][m];
  nrm = sqrt(nrm);
  const double sg = Q[0][m] < 0.0 ? -1.0 : 1.0;
  for (int i = 0; i < KMAX; ++i) ks->y[i] = i < k ? sg * Q[i][m] / nrm : 0.0;
  ks->ritz = A[m][m];
}

// X = sum_i y_i V_i
__global__ void krylov_combine_kernel(const cplx* __restrict__ V, long long vstride, cplx* __restrict__ X, const int* dimL,
                                      const int* dimR, int D, const KrylovState* ks) {
  const int k = ks->nk;
  double y[KMAX];
  for (int i = 0; i < KMAX; ++i) y[i] = ks->y[i];
  const long long n = (long long)(*dimL) * D * D * (*dimR);
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    cplx x = make_double2(0.0, 0.0);
    for (int i = 0; i < k; ++i) cadd(x, y[i], V[i * vstride + e]);
    X[e] = x;
  }
}

// X /= |X| (partials of <X|X>)
__global__ void krylov_scale_kernel(cplx* __restrict__ X, const int* dimL, const int* dimR, int D, const double* __restrict__ partial) {
  double nn, im;
  partial_sum(partial, 0, nn, im);
  if (!(nn > 0.0)) return;
  const double inv = 1.0 / sqrt(nn);
  const long long n = (long long)(*dimL) * D * D * (*dimR);
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
    X[e] = make_double2(X[e].x * inv, X[e].y * inv);
}

__global__ void partial_total_kernel(const double* partial, double* out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double re, im;
  partial_sum(partial, 0, re, im);
  *out = re;
}

}  // namespace

void launch_heff(GemmDesc* descs, const cplx* V, cplx* W, cplx* Y, cplx* Z, long long ystride, const cplx* EL, const cplx* ER,
                 long long estride, const int* dimL, const int* dimR, const int* qL, const int* qR, int D, double J, double U,
                 const KrylovState* ks, int capL, int capR, cudaStream_t s) {
  heff_setup_kernel<<<1, 32, 0, s>>>(descs, V, Y, Z, ystride, EL, ER, estride, dimL, dimR, D, ks);
  launch_zgemm(descs, 3, capL, D * D * capR, s);
  launch_zgemm(descs + 3, 3, capL * D * D, capR, s);
  heff_combine_kernel<<<grid_for((long long)capL * D * D * capR, 256), 256, 0, s>>>(V, Y, Z, ystride, W, dimL, dimR, qL, qR, D, J, U, ks);
}

void launch_env_update(GemmDesc* descs, int side, const cplx* A, const cplx* Ein, cplx* Eout, cplx* T, cplx* T2, long long tstride,
                       long long estride, const int* dimL, const int* dimR, int D, double J, double U, int capL, int capR,
                       cudaStream_t s) {
  env_setup_kernel<<<1, 32, 0, s>>>(descs, side, A, Ein, Eout, T, T2, tstride, estride, dimL, dimR, D);
  if (side == 0) launch_zgemm(descs, 3, capL, D * capR, s);
  else launch_zgemm(descs, 3, capL * D, capR, s);
  env_combine_kernel<<<grid_for((long long)capL * D * capR, 256), 256, 0, s>>>(side, A, T, T2, tstride, dimL, dimR, D, J, U);
  if (side == 0) launch_zgemm(descs + 3, 3, capR, capR, s);
  else launch_zgemm(descs + 3, 3, capL, capL, s);
}

void launch_krylov_dot(const cplx* V, long long vstride, int nvec, const cplx* w, const int* dimL, const int* dimR, int D,
                       const KrylovState* ks, double* partial, cudaStream_t s) {
  krylov_dot_kernel<<<KRY_CTAS, KRY_THREADS, 0, s>>>(V, vstride, nvec, w, dimL, dimR, D, ks, partial);
}
void launch_krylov_init(const cplx* X, cplx* V0, const int* dimL, const int* dimR, int D, KrylovState* ks, const double* partial,
                        int max_elems, cudaStream_t s) {
  krylov_init_kernel<<<grid_for(max_elems, 256), 256, 0, s>>>(X, V0, dimL, dimR, D, ks, partial);
}
void launch_krylov_alpha(const cplx* V, long long vstride, int it, cplx* w, const int* dimL, const int* dimR, int D, KrylovState* ks,
                         const double* partial, int max_elems, cudaStream_t s) {
  krylov_alpha_kernel<<<grid_for(max_elems, 256), 256, 0, s>>>(V, vstride, it, w, dimL, dimR, D, ks, partial);
}
void launch_krylov_reorth(const cplx* V, long long vstride, int nvec, cplx* w, const int* dimL, const int* dimR, int D,
                          const KrylovState* ks, const double* partial, int max_elems, cudaStream_t s) {
  krylov_reorth_kernel<<<grid_for(max_elems, 256), 256, 0, s>>>(V, vstride, nvec, w, dimL, dimR, D, ks, partial);
}
void launch_krylov_next(cplx* V, long long vstride, int it, const cplx* w, const int* dimL, const int* dimR, int D, KrylovState* ks,
                        const double* partial, int max_elems, cudaStream_t s) {
  krylov_next_kernel<<<grid_for(max_elems, 256), 256, 0, s>>>(V, vstride, it, w, dimL, dimR, D, ks, partial);
}
void launch_krylov_ritz(KrylovState* ks, cudaStream_t s) { krylov_ritz_kernel<<<1, 32, 0, s>>>(ks); }
void launch_krylov_combine(const cplx* V, long long vstride, cplx* X, const int* dimL, const int* dimR, int D, const KrylovState* ks,
                           int max_elems, cudaStream_t s) {
  krylov_combine_kernel<<<grid_for(max_elems, 256), 256, 0, s>>>(V, vstride, X, dimL, dimR, D, ks);
}
void launch_krylov_scale(cplx* X, const int* dimL, const int* dimR, int D, const double* partial, int max_elems, cudaStream_t s) {
  krylov_scale_kernel<<<grid_for(max_elems, 256), 256, 0, s>>>(X, dimL, dimR, D, partial);
}
void launch_partial_total(const double* partial, double* out, cudaStream_t s) { partial_total_kernel<<<1, 32, 0, s>>>(partial, out); }
