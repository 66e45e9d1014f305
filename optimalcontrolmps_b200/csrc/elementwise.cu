// Bandwidth-type kernels of the engine: Trotter gate application on the merged two-site tensor,
// diagonal on-site phases, slice-store copies, transfer-matrix planning / fix-ups, K|psi> expansion.
#include <algorithm>
#include <cstdlib>
#include <mutex>
#include "ocmps_internal.h"

namespace {

int grid_for(long long elems, int threads, int cap = 1184) {
  long long g = (elems + threads - 1) / threads;
  if (g < 1) g = 1;
  if (g > cap) g = cap;
  return (int)g;
}

__global__ void merge_setup_kernel(GemmDesc* d, const cplx* A1, const cplx* A2, cplx* theta, const int* dimL, const int* dimM,
                                   const int* dimR, int D) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  GemmDesc g;
  g.A = A1; g.B = A2; g.C = theta;
  g.M = (*dimL) * D; g.K = *dimM; g.N = D * (*dimR);
  g.lda = g.K; g.ldb = g.N; g.ldc = g.N;
  g.opA = g.opB = 0; g.pad = 0;
  *d = g;
}

// theta'[l,t1,t2,r] = o1[t1] o2[t2] sum_{s1,s2} G[(t1,t2),(s1,s2)] i1[s1] i2[s2] theta[l,s1,s2,r]
// (src/BH_tDMRG.cpp:150-159).  One thread per (l, r).  The gate conserves the boson number and theta[l,.,.,r]
// lives in the single sector s1 + s2 = qR[r] - qL[l], so only a (<= D) x (<= D) sub-block of the D^2 x D^2 gate
// acts: at most D inputs, D outputs, D^2 complex multiply-adds per thread instead of D^4.
template <int D>
__global__ void __launch_bounds__(128) gate_apply_kernel(cplx* __restrict__ theta, const int* dimL, const int* dimR,
                                                        const int* __restrict__ qL, const int* __restrict__ qR,
                                                        const StepParams* __restrict__ sp, int gate_kind) {
  extern __shared__ __align__(16) unsigned char gate_smem[];
  __shared__ Phases ph;
  cplx* W = reinterpret_cast<cplx*>(gate_smem);
  const int chiL = *dimL, chiR = *dimR;
  const cplx* __restrict__ G = sp->G;
  if (threadIdx.x < D) {                       // [0],[1]: phases before the J gate on site 1, 2; [2],[3]: after it
    const int n = threadIdx.x;
    const bool pre = gate_kind != 2;
    ph.re[0][n] = ph.re[1][n] = pre ? sp->u1r[n] : 1.0; ph.im[0][n] = ph.im[1][n] = pre ? sp->u1i[n] : 0.0;
    ph.re[2][n] = gate_kind == 2 ? sp->u2r[n] : 1.0;     ph.im[2][n] = gate_kind == 2 ? sp->u2i[n] : 0.0;
    ph.re[3][n] = gate_kind != 0 ? sp->u2r[n] : 1.0;     ph.im[3][n] = gate_kind != 0 ? sp->u2i[n] : 0.0;
  }
  __syncthreads();
  for (int e = threadIdx.x; e < D * D * D * D; e += blockDim.x) {
    const int row = e / (D * D), col = e % (D * D);
    const int t1 = row / D, t2 = row % D, s1 = col / D, s2 = col % D;
    double fr = ph.re[0][s1], fi = ph.im[0][s1];
    double xr = fr * ph.re[1][s2] - fi * ph.im[1][s2], xi = fr * ph.im[1][s2] + fi * ph.re[1][s2];
    fr = xr * ph.re[2][t1] - xi * ph.im[2][t1]; fi = xr * ph.im[2][t1] + xi * ph.re[2][t1];
    xr = fr * ph.re[3][t2] - fi * ph.im[3][t2]; xi = fr * ph.im[3][t2] + fi * ph.re[3][t2];
    const cplx g = G[e];
    W[e] = make_double2(g.x * xr - g.y * xi, g.x * xi + g.y * xr);
  }
  __syncthreads();
  const long long total = (long long)chiL * chiR;
  const long long rowstride = (long long)D * chiR;          // stride of s1 (elements)
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int l = (int)(e / chiR), r = (int)(e % chiR);
    const int N = qR[r] - qL[l];                           // bosons on the two sites
    if (N < 0 || N > 2 * (D - 1)) continue;                // no admissible (s1, s2): the entries are exact zeros
    const int lo = N - (D - 1) > 0 ? N - (D - 1) : 0, hi = N < D - 1 ? N : D - 1;
    cplx* base = theta + (long long)l * D * rowstride + r;
    cplx in[D];
#pragma unroll
    for (int k = 0; k < D; ++k) {
      const int s1 = lo + k;
      in[k] = make_double2(0.0, 0.0);
      if (s1 <= hi) in[k] = base[s1 * rowstride + (long long)(N - s1) * chiR];
    }
#pragma unroll
    for (int kt = 0; kt < D; ++kt) {
      const int t1 = lo + kt;
      if (t1 > hi) break;
      const int row = t1 * D + (N - t1);
      double ar = 0.0, ai = 0.0;
#pragma unroll
      for (int k = 0; k < D; ++k) {
        const int s1 = lo + k;
        if (s1 <= hi) {
          const cplx w = W[row * D * D + s1 * D + (N - s1)];
          ar += w.x * in[k].x - w.y * in[k].y;
          ai += w.x * in[k].y + w.y * in[k].x;
        }
      }
      base[t1 * rowstride + (long long)(N - t1) * chiR] = make_double2(ar, ai);
    }
  }
}

// Two-site merge and Trotter gate in one pass, sector by sector:
//   theta'[l,t1,t2,r] = sum_{s1+s2=N} W[(t1,t2),(s1,s2)] sum_{mid: q(mid) = qL[l]+s1} A1[l,s1,mid] A2[mid,s2,r],   N = qR[r] - qL[l]
// Only the charge-allowed entries of theta are computed and written (the decomposition that follows gathers exactly
// those); as a dense GEMM the merge would spend ~98 % of its multiply-adds on structural zeros.  The middle bond is
// sorted by charge, so the mids of one sector are a contiguous range.  Four lanes per (l, r), each taking every fourth
// mid (the kernel is a chain of L2 latencies, so the loop is kept short and many loads are in flight); a warp shares l:
// the A1 loads are broadcasts, the A2 loads are coalesced over 8 consecutive r.
template <int D>
__global__ void __launch_bounds__(128) merge_gate_kernel(const cplx* __restrict__ A1, const cplx* __restrict__ A2, cplx* __restrict__ theta,
                                                        const int* dimL, const int* dimM, const int* dimR,
                                                        const int* __restrict__ qL, const int* __restrict__ qM, const int* __restrict__ qR,
                                                        const StepParams* __restrict__ sp, int gate_kind) {
  __shared__ Phases ph;
  __shared__ int s_start[OCMPS_MAX_Q + 2];           // first mid whose charge is >= c
  const int chiL = *dimL, chiM = *dimM, chiR = *dimR;
  const cplx* __restrict__ G = sp->G;
  if (threadIdx.x < D) {                       // [0],[1]: phases before the J gate on site 1, 2; [2],[3]: after it
    const int n = threadIdx.x;
    const bool pre = gate_kind != 2;
    ph.re[0][n] = ph.re[1][n] = pre ? sp->u1r[n] : 1.0; ph.im[0][n] = ph.im[1][n] = pre ? sp->u1i[n] : 0.0;
    ph.re[2][n] = gate_kind == 2 ? sp->u2r[n] : 1.0;     ph.im[2][n] = gate_kind == 2 ? sp->u2i[n] : 0.0;
    ph.re[3][n] = gate_kind != 0 ? sp->u2r[n] : 1.0;     ph.im[3][n] = gate_kind != 0 ? sp->u2i[n] : 0.0;
  }
  for (int i = threadIdx.x; i <= chiM; i += blockDim.x) {
    int lo = (i == 0) ? 0 : qM[i - 1] + 1;
    int hi = (i == chiM) ? OCMPS_MAX_Q + 1 : qM[i];
    lo = lo < 0 ? 0 : lo;
    hi = hi > OCMPS_MAX_Q + 1 ? OCMPS_MAX_Q + 1 : hi;
    for (int c = lo; c <= hi; ++c) s_start[c] = i;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, g = lane >> 3;
  const int r = blockIdx.x * 8 + (lane & 7);
  const int l = blockIdx.y * 4 + (threadIdx.x >> 5);
  if (l >= chiL) return;                                   // (warp uniform)
  const bool rin = r < chiR;
  const int ql = qL[l];
  const int N = rin ? qR[r] - ql : -1;                     // bosons on the two sites
  const bool ok = rin && N >= 0 && N <= 2 * (D - 1);       // else no admissible (s1, s2): the entries are structural zeros
  const long long rowstride = (long long)D * chiR;         // stride of s1 in theta and of mid in A2 (elements)
  cplx in[D];
#pragma unroll
  for (int s1 = 0; s1 < D; ++s1) {
    in[s1] = make_double2(0.0, 0.0);
    const int c = ql + s1, s2 = N - s1;
    if (c < 0 || c > OCMPS_MAX_Q) continue;                // (uniform)
    const int m0 = s_start[c], m1 = s_start[c + 1];
    const bool act = ok && s2 >= 0 && s2 < D;
    const cplx* a1 = A1 + ((long long)l * D + s1) * chiM;
    const cplx* a2 = A2 + (act ? (long long)s2 * chiR + r : 0);
    double ar = 0.0, ai = 0.0;
#pragma unroll 4
    for (int mid = m0 + g; mid < m1; mid += 4) {
      const cplx x = a1[mid];
      cplx y = make_double2(0.0, 0.0);
      if (act) y = a2[(long long)mid * rowstride];
      ar += x.x * y.x - x.y * y.y;
      ai += x.x * y.y + x.y * y.x;
    }
    ar += __shfl_xor_sync(0xffffffffu, ar, 8);  ai += __shfl_xor_sync(0xffffffffu, ai, 8);
    ar += __shfl_xor_sync(0xffffffffu, ar, 16); ai += __shfl_xor_sync(0xffffffffu, ai, 16);
    if (act) {                                             // on-site phases before the hopping gate
      const double fr = ph.re[0][s1] * ph.re[1][s2] - ph.im[0][s1] * ph.im[1][s2];
      const double fi = ph.re[0][s1] * ph.im[1][s2] + ph.im[0][s1] * ph.re[1][s2];
      in[s1] = make_double2(ar * fr - ai * fi, ar * fi + ai * fr);
    }
  }
  if (!ok) return;
  cplx* base = theta + (long long)l * D * rowstride + r;
#pragma unroll
  for (int t1 = 0; t1 < D; ++t1) {
    const int t2 = N - t1;
    if (t2 < 0 || t2 >= D || (t1 & 3) != g) continue;      // the four lanes of an (l, r) share the outputs
    const cplx* Grow = G + (t1 * D + t2) * D * D;
    double ar = 0.0, ai = 0.0;
#pragma unroll
    for (int s1 = 0; s1 < D; ++s1) {
      const int s2 = N - s1;
      if (s2 >= 0 && s2 < D) {
        const cplx w = Grow[s1 * D + s2];
        ar += w.x * in[s1].x - w.y * in[s1].y;
        ai += w.x * in[s1].y + w.y * in[s1].x;
      }
    }
    const double fr = ph.re[2][t1] * ph.re[3][t2] - ph.im[2][t1] * ph.im[3][t2];     // on-site phases after it
    const double fi = ph.re[2][t1] * ph.im[3][t2] + ph.im[2][t1] * ph.re[3][t2];
    base[t1 * rowstride + (long long)t2 * chiR] = make_double2(ar * fr - ai * fi, ar * fi + ai * fr);
  }
}

__global__ void site_phase_kernel(cplx* A, const int* dimL, const int* dimR, int D, const StepParams* __restrict__ sp, int which) {
  const int chiL = *dimL, chiR = *dimR;
  const long long total = (long long)chiL * D * chiR;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int s = (int)((e / chiR) % D);
    const cplx u = A[e];
    const double pr = which == 0 ? sp->u1r[s] : sp->u2r[s], pi = which == 0 ? sp->u1i[s] : sp->u2i[s];
    A[e] = make_double2(u.x * pr - u.y * pi, u.x * pi + u.y * pr);
  }
}

__global__ void set_step_params_kernel(StepParams hp, StepParams* dst) {
  if (threadIdx.x == 0 && blockIdx.x == 0) *dst = hp;
}

// work MPS -> store slot named by *sp; blockIdx.y = site, the last y-slice copies dims and charge labels
__global__ void pack_to_slot_kernel(SitePtrs src, SiteOffs offs, const int* dims, const int* q, int L, int D, int cap,
                                    const StepParams* __restrict__ sp) {
  const int j = blockIdx.y;
  if (j < L) {
    const long long count = (long long)dims[j] * D * dims[j + 1];
    const cplx* s = src.p[j];
    cplx* d = sp->slot_data + offs.o[j];
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < count; e += (long long)gridDim.x * blockDim.x) d[e] = s[e];
  } else {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
    for (int b = tid; b <= L; b += nt) sp->slot_dims[b] = dims[b];
    for (int e = tid; e < (L + 1) * cap; e += nt) sp->slot_q[e] = q[e];
  }
}

__global__ void pack_copy_kernel(SitePtrs src, cplx* dst_base, SiteOffs offs, const int* dims, int D) {
  const int j = blockIdx.y;
  const long long count = (long long)dims[j] * D * dims[j + 1];
  const cplx* s = src.p[j];
  cplx* d = dst_base + offs.o[j];
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < count; e += (long long)gridDim.x * blockDim.x) d[e] = s[e];
}
__global__ void unpack_copy_kernel(const cplx* src_base, SitePtrs dst, SiteOffs offs, const int* dims, int D) {
  const int j = blockIdx.y;
  const long long count = (long long)dims[j] * D * dims[j + 1];
  const cplx* s = src_base + offs.o[j];
  cplx* d = dst.p[j];
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < count; e += (long long)gridDim.x * blockDim.x) d[e] = s[e];
}

// ---- slice store through the TMA unit ----
// A slice is L contiguous site tensors (up to 960 KB each at chi = 100): pure data movement, so no thread touches the data.
// One elected lane per CTA streams its share of a site through a ring of shared-memory stages with bulk asynchronous copies:
// global -> shared (cp.async.bulk ... mbarrier::complete_tx::bytes), then shared -> global (cp.async.bulk ... bulk_group) as soon as
// the stage has landed; a stage is reloaded once the store that reads it has drained (wait_group.read).  Site sizes are read from
// the device-resident bond dimensions like everywhere else; every piece is a multiple of 16 bytes (complex128) at a 16-byte
// aligned address.  mode 0: work MPS -> packed buffer, 1: packed buffer -> work MPS, 2: work MPS -> the store slot named by *sp
// (its last y-slice copies the bond dimensions and the charge labels with ordinary loads and stores).
namespace tma {
constexpr int CHUNK = 16384;            // bytes per bulk copy
constexpr int STAGES = 4;               // ring depth: 64 KB of shared memory per CTA
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned mbar, unsigned count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_expect(unsigned mbar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
// bounded wait: a copy that never completes sets the status word instead of hanging the device
__device__ __forceinline__ bool mbar_wait(unsigned mbar, unsigned parity) {
  for (int spin = 0; spin < (1 << 24); ++spin) {
    unsigned ok;
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(ok) : "r"(mbar), "r"(parity) : "memory");
    if (ok) return true;
  }
  return false;
}
__device__ __forceinline__ void load(unsigned dst_smem, const void* src, unsigned bytes, unsigned mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem), "l"(src), "r"(bytes), "r"(mbar) : "memory");
}
__device__ __forceinline__ void store(void* dst, unsigned src_smem, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src_smem), "r"(bytes) : "memory");
}
__device__ __forceinline__ void commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
}  // namespace tma

__global__ void __launch_bounds__(32) slice_copy_tma_kernel(SitePtrs work, cplx* packed, SiteOffs offs, const int* dims, const int* q, int L, int D,
                                                            int cap, const StepParams* __restrict__ sp, int mode, int* status) {
  extern __shared__ __align__(128) unsigned char stage_buf[];
  __shared__ __align__(8) unsigned long long mbar[tma::STAGES];
  const int j = blockIdx.y;
  if (j >= L) {                                            // (mode 2) bond dimensions and charge labels of the slot
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
    for (int b = tid; b <= L; b += nt) sp->slot_dims[b] = dims[b];
    for (int e = tid; e < (L + 1) * cap; e += nt) sp->slot_q[e] = q[e];
    return;
  }
  if (threadIdx.x != 0) return;
  const long long bytes = (long long)dims[j] * D * dims[j + 1] * (long long)sizeof(cplx);
  cplx* pk = (mode == 2 ? sp->slot_data : packed) + offs.o[j];
  const unsigned char* src = reinterpret_cast<const unsigned char*>(mode == 1 ? pk : work.p[j]);
  unsigned char* dst = reinterpret_cast<unsigned char*>(mode == 1 ? work.p[j] : pk);
  const long long nchunks = (bytes + tma::CHUNK - 1) / tma::CHUNK;
  const long long mine = nchunks > (long long)blockIdx.x ? (nchunks - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;    // chunks blockIdx.x, + gridDim.x, ...
  if (mine == 0) return;
  for (int i = 0; i < tma::STAGES; ++i) tma::mbar_init(tma::smem_u32(&mbar[i]), 1);
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  auto chunk_bytes = [&](long long i) -> unsigned {
    const long long c = blockIdx.x + i * (long long)gridDim.x;
    const long long rest = bytes - c * tma::CHUNK;
    return (unsigned)(rest < tma::CHUNK ? rest : tma::CHUNK);
  };
  auto issue_load = [&](long long i) {
    const int st = (int)(i % tma::STAGES);
    const long long c = blockIdx.x + i * (long long)gridDim.x;
    const unsigned nb = chunk_bytes(i);
    tma::mbar_expect(tma::smem_u32(&mbar[st]), nb);
    tma::load(tma::smem_u32(stage_buf + (size_t)st * tma::CHUNK), src + c * tma::CHUNK, nb, tma::smem_u32(&mbar[st]));
  };
  const long long pre = mine < tma::STAGES ? mine : tma::STAGES;
  for (long long i = 0; i < pre; ++i) issue_load(i);
  for (long long i = 0; i < mine; ++i) {
    const int st = (int)(i % tma::STAGES);
    if (!tma::mbar_wait(tma::smem_u32(&mbar[st]), (unsigned)((i / tma::STAGES) & 1))) { if (status) atomicOr(status, OCMPS_ST_NOCONV); else __trap(); break; }
    const long long c = blockIdx.x + i * (long long)gridDim.x;
    tma::store(dst + c * tma::CHUNK, tma::smem_u32(stage_buf + (size_t)st * tma::CHUNK), chunk_bytes(i));
    tma::commit();
    // the stage of chunk i-1 is reloaded (chunk i-1+STAGES) once the store of chunk i-1 has read it; the store of chunk i stays in flight
    if (i >= 1 && i - 1 + tma::STAGES < mine) {
      tma::wait_read<1>();
      issue_load(i - 1 + tma::STAGES);
    }
  }
  tma::wait_all();
}

// ---- overlaps ----
__device__ __forceinline__ const cplx* side_site(const OvlSide& s, int z, int site) {
  return s.use_ptrs ? s.ptrs.p[site] : s.base + (long long)(s.slot0 + z) * s.slot_stride + s.offs.o[site];
}
__device__ __forceinline__ const int* side_dims(const OvlSide& s, int z) {
  return s.dims + (long long)(s.use_ptrs ? 0 : (s.slot0 + z)) * s.dims_stride;
}

// Per batch entry z and site j: T = E . B_j   (nE*chiA x D*chiB')   and  E'_c = A_j^H . Tm_c  for c < nE, with nE environment
// channels stacked along M.  Tm is T itself, or a second buffer (same stride) that a channel-mixing kernel fills from T.
// descs layout: [0*batch + z] the T gemm, [(1+c)*batch + z] the E' gemms.
__global__ void overlap_plan_kernel(GemmDesc* descs, OvlSide bra, OvlSide ket, int site, int batch, int D, int nE, cplx* E_in,
                                    cplx* E_out, cplx* T, const cplx* Tm, long long e_stride, long long t_stride) {
  const int z = blockIdx.x * blockDim.x + threadIdx.x;
  if (z >= batch) return;
  const int* da = side_dims(bra, z);
  const int* db = side_dims(ket, z);
  const int aL = da[site], aR = da[site + 1], bL = db[site], bR = db[site + 1];
  const cplx* A = side_site(bra, z, site);
  const cplx* B = side_site(ket, z, site);
  cplx* Ei = E_in + z * e_stride;
  cplx* Eo = E_out + z * e_stride;
  cplx* Tz = T + z * t_stride;
  const cplx* Tmz = Tm + z * t_stride;
  GemmDesc g;
  g.pad = 0;
  // T (nE*aL x D*bR) = E (nE*aL x bL) . B (bL x D*bR)
  g.A = Ei; g.opA = 0; g.lda = bL;
  g.B = B; g.opB = 0; g.ldb = D * bR;
  g.C = Tz; g.ldc = D * bR; g.M = nE * aL; g.N = D * bR; g.K = bL;
  descs[z] = g;
  for (int c = 0; c < nE; ++c) {
    // E'_c (aR x bR) = A^H (aL*D x aR)^H . Tm_c (aL*D x bR)
    g.A = A; g.opA = 1; g.lda = aR;
    g.B = Tmz + (long long)c * aL * D * bR; g.opB = 0; g.ldb = bR;
    g.C = Eo + (long long)c * aR * bR; g.ldc = bR; g.M = aR; g.N = bR; g.K = aL * D;
    descs[(1 + c) * batch + z] = g;
  }
}

// Local expectation values on top of the transfer-matrix chain of <psi|psi> (include/correlations.hpp:99-117):
//   out[z][site][k] = sum_{l',s,r} conj(A[l',s,r]) T[l',s,r] op_k[s],   T = E_left . A  (the T gemm of this site)
// for diagonal site operators op_k (N, N(N-1), N^2 ... are all diagonal in the boson number).  Exact when the sites to
// the right of `site` are right-orthonormal, which is how the sweeps leave every slice (centre at site 1); k = 0 is
// reserved for the identity, so out[z][site][0] = <psi|psi> is the built-in check of that precondition.
// One CTA per batch entry; fixed-order tree reduction (deterministic).
constexpr int EXPECT_MAX_OPS = 8;
__global__ void __launch_bounds__(256) overlap_local_expect_kernel(const GemmDesc* __restrict__ descs, OvlSide bra, int site, int D,
                                                                   const double* __restrict__ ops, int nops, double* __restrict__ out,
                                                                   int L) {
  __shared__ double red[EXPECT_MAX_OPS][256];
  const int z = blockIdx.x;
  const GemmDesc g = descs[z];
  const int aL = g.M, N = g.N, bR = N / D;
  const cplx* __restrict__ T = g.C;
  const cplx* __restrict__ A = side_site(bra, z, site);
  double acc[EXPECT_MAX_OPS];
#pragma unroll
  for (int k = 0; k < EXPECT_MAX_OPS; ++k) acc[k] = 0.0;
  const long long total = (long long)aL * N;
  for (long long e = threadIdx.x; e < total; e += blockDim.x) {
    const int sx = (int)((e % N) / bR);
    const cplx a = A[e], t = T[e];
    const double w = a.x * t.x + a.y * t.y;          // Re(conj(a) t); the imaginary parts cancel in the sum
#pragma unroll
    for (int k = 0; k < EXPECT_MAX_OPS; ++k)
      if (k < nops) acc[k] += w * ops[k * D + sx];
  }
#pragma unroll
  for (int k = 0; k < EXPECT_MAX_OPS; ++k) red[k][threadIdx.x] = acc[k];
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o)
      for (int k = 0; k < nops; ++k) red[k][threadIdx.x] += red[k][threadIdx.x + o];
    __syncthreads();
  }
  if ((int)threadIdx.x < nops) out[((long long)z * L + site) * nops + threadIdx.x] = red[threadIdx.x][0];
}

__global__ void overlap_init_kernel(cplx* E, long long e_stride, int batch, int withK) {
  const int z = blockIdx.x * blockDim.x + threadIdx.x;
  if (z >= batch) return;
  E[z * e_stride] = make_double2(1.0, 0.0);
  if (withK) E[z * e_stride + 1] = make_double2(0.0, 0.0);
}

// T1 += k_s T0 with k_s = s(s-1)/2 (src/BH_tDMRG.cpp:10-14); T is [c][l][s][r]
__global__ void overlap_kfix_kernel(cplx* T, long long t_stride, const GemmDesc* descs, int D) {
  const int z = blockIdx.y;
  const GemmDesc g = descs[z];
  const int aL = g.M / 2, N = g.N;       // N = D*bR
  const int bR = N / D;
  cplx* T0 = T + z * t_stride;
  cplx* T1 = T0 + (long long)aL * N;
  const long long total = (long long)aL * N;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int s = (int)((e % N) / bR);
    const double k = 0.5 * s * (s - 1);
    if (k != 0.0) {
      cplx a = T0[e], b = T1[e];
      T1[e] = make_double2(b.x + k * a.x, b.y + k * a.y);
    }
  }
}

// Site operator on the physical index of T, in place, for the batch entries that have one at this site (sel[z] >= 0):
// T'[l][t][r] = sum_s O[t][s] T[l][s][r] with O = op_table[sel[z]] (D x D, real, row-major O[t][s] = <t|O|s>; the operators of
// include/BH_sites.h:129-171 -- N, A, Adag, N(N-1), NN, Id -- and their products).  One thread per (l, r).
__global__ void overlap_site_op_kernel(cplx* T, long long t_stride, const GemmDesc* descs, int D, const double* __restrict__ op_table,
                                       const int* __restrict__ sel) {
  const int z = blockIdx.y;
  const int op = sel[z];
  if (op < 0) return;
  const GemmDesc g = descs[z];
  const int aL = g.M, N = g.N, bR = N / D;
  const double* O = op_table + (size_t)op * D * D;
  cplx* Tz = T + z * t_stride;
  const long long total = (long long)aL * bR;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int l = (int)(e / bR), r = (int)(e % bR);
    cplx* col = Tz + (long long)l * N + r;
    cplx v[OCMPS_MAX_D];
    for (int sI = 0; sI < D; ++sI) v[sI] = col[(long long)sI * bR];
    for (int t = 0; t < D; ++t) {
      double ar = 0.0, ai = 0.0;
      for (int sI = 0; sI < D; ++sI) { const double o = O[t * D + sI]; ar += o * v[sI].x; ai += o * v[sI].y; }
      col[(long long)t * bR] = make_double2(ar, ai);
    }
  }
}

__global__ void overlap_final_kernel(const cplx* E, long long e_stride, int batch, int withK, cplx* out) {
  const int z = blockIdx.x * blockDim.x + threadIdx.x;
  if (z >= batch) return;
  out[z] = E[z * e_stride + (withK ? 1 : 0)];
}

// ---- energy moments: the transfer-matrix chain of <psi|W..W|psi> (4 channels) or <psi|(W x W)..(W x W)|psi> (16 channels) ----
// Left boundary: every channel 0 except the start channel nch-1 (MPO state 3, "nothing placed yet"), which is 1.
__global__ void energy_init_kernel(cplx* E, long long e_stride, int batch, int nch) {
  const int z = blockIdx.x * blockDim.x + threadIdx.x;
  if (z >= batch) return;
  for (int c = 0; c < nch; ++c) E[z * e_stride + c] = make_double2(c == nch - 1 ? 1.0 : 0.0, 0.0);
}

__device__ __forceinline__ double energy_factor(const EnergyTable& tab, int f, int t, int s, int D, double U, double cL) {
  switch (f) {
    case ENERGY_F_ID: return t == s ? 1.0 : 0.0;
    case ENERGY_F_A: return tab.A[t * D + s];
    case ENERGY_F_ADAG: return tab.Adag[t * D + s];
    default: return t == s ? 0.5 * U * t * (t - 1) - cL : 0.0;   // ENERGY_F_ONSITE
  }
}

// T'_v[l][t][r] = sum_{k: dst_k = v} sum_s O_k[t][s] T_{src_k}[l][s][r] for every target channel v, with the transition operators
// O_k = coef_k F1_k F2_k built per slice (its U_z, c_z / L) in shared memory.  T and T' are [c][l][s][r] with channel stride
// aL*D*bR.  One thread per (l, r) column; the table is sorted by target channel, so a target is accumulated in registers and
// written once, in a fixed order.
template <int D>
__global__ void __launch_bounds__(256) energy_mix_kernel(const cplx* __restrict__ T, cplx* __restrict__ Tm, long long t_stride,
                                                         const GemmDesc* __restrict__ descs, const double* __restrict__ uc,
                                                         const EnergyTable tab) {
  __shared__ double sO[ENERGY_MAX_TRANS * D * D];
  const int z = blockIdx.y;
  const double U = uc[2 * z], cL = uc[2 * z + 1];
  for (int i = threadIdx.x; i < tab.nt * D * D; i += blockDim.x) {
    const int k = i / (D * D), t = (i / D) % D, s = i % D;
    double acc = 0.0;
    for (int m = 0; m < D; ++m) acc += energy_factor(tab, tab.f1[k], t, m, D, U, cL) * energy_factor(tab, tab.f2[k], m, s, D, U, cL);
    sO[i] = tab.coef[k] * acc;
  }
  __syncthreads();
  const int nch = tab.nch;
  const GemmDesc g = descs[z];
  const int aL = g.M / nch, N = g.N, bR = N / D;
  const long long cs = (long long)aL * N;
  const cplx* __restrict__ Tz = T + z * t_stride;
  cplx* __restrict__ Tmz = Tm + z * t_stride;
  const long long total = (long long)aL * bR;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long off = (e / bR) * N + (e % bR);
    int k = 0;
    for (int v = 0; v < nch; ++v) {
      double ar[D], ai[D];
#pragma unroll
      for (int t = 0; t < D; ++t) { ar[t] = 0.0; ai[t] = 0.0; }
      for (; k < tab.nt && tab.dst[k] == v; ++k) {
        const cplx* col = Tz + tab.src[k] * cs + off;
        cplx x[D];
#pragma unroll
        for (int s = 0; s < D; ++s) x[s] = col[(long long)s * bR];
        const double* O = sO + k * D * D;
#pragma unroll
        for (int t = 0; t < D; ++t)
#pragma unroll
          for (int s = 0; s < D; ++s) { const double o = O[t * D + s]; ar[t] += o * x[s].x; ai[t] += o * x[s].y; }
      }
      cplx* out = Tmz + v * cs + off;
#pragma unroll
      for (int t = 0; t < D; ++t) out[(long long)t * bR] = make_double2(ar[t], ai[t]);
    }
  }
}

// Right boundary (1 x 1 per channel): out[3z] = <psi|psi>, out[3z+1] = <psi|H-c|psi>, out[3z+2] = <psi|(H-c)^2|psi> (16 channels;
// 0 with 4).  Channel (a, b) of the 16 is 4a+b; the end state is 0, so (3,3) carries the norm, (0,3) one factor of H-c, (0,0) two.
__global__ void energy_final_kernel(const cplx* E, long long e_stride, int batch, int nch, double* out) {
  const int z = blockIdx.x * blockDim.x + threadIdx.x;
  if (z >= batch) return;
  const cplx* Ez = E + z * e_stride;
  out[3 * z + 0] = Ez[nch - 1].x;
  out[3 * z + 1] = Ez[nch == 16 ? 3 : 0].x;
  out[3 * z + 2] = nch == 16 ? Ez[0].x : 0.0;
}

// ---- K|psi>: B[(l,a), s, (r,b)] = A[l,s,r] W[a,b,s], W = [[1,0],[k_s,1]], boundaries pick row 1 / column 0 ----
__global__ void applyK_expand_kernel(const cplx* A, cplx* B, const int* dimL_in, const int* dimR_in, const int* qL_in,
                                     const int* qR_in, int* dimL_out, int* dimR_out, int* qL_out, int* qR_out, int D, int site,
                                     int L) {
  const int chiL = *dimL_in, chiR = *dimR_in;
  const int nA = (site == 0) ? 1 : 2, nB = (site == L - 1) ? 1 : 2;
  const int oL = chiL * nA, oR = chiR * nB;
  const long long total = (long long)oL * D * oR;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int rb = (int)(e % oR);
    const int s = (int)((e / oR) % D);
    const int la = (int)(e / ((long long)oR * D));
    const int l = la / nA, a0 = la % nA, r = rb / nB, b0 = rb % nB;
    const int a = (site == 0) ? 1 : a0;            // left boundary: row 1
    const int b = (site == L - 1) ? 0 : b0;        // right boundary: column 0
    double w = 0.0;
    if (a == b) w = 1.0;
    else if (a == 1 && b == 0) w = 0.5 * s * (s - 1);
    const cplx u = A[((long long)l * D + s) * chiR + r];
    B[e] = make_double2(u.x * w, u.y * w);
  }
  if (blockIdx.x == 0) {
    // bookkeeping of the right bond (and the left bond on the first site)
    for (int i = threadIdx.x; i < oR; i += blockDim.x) qR_out[i] = qR_in[i / nB];
    if (site == 0) for (int i = threadIdx.x; i < oL; i += blockDim.x) qL_out[i] = qL_in[i / nA];
    if (threadIdx.x == 0) { *dimR_out = oR; if (site == 0) *dimL_out = oL; }
  }
}

}  // namespace

void launch_merge_setup(GemmDesc* d, const cplx* A1, const cplx* A2, cplx* theta, const int* dimL, const int* dimM,
                        const int* dimR, int D, cudaStream_t s) {
  merge_setup_kernel<<<1, 32, 0, s>>>(d, A1, A2, theta, dimL, dimM, dimR, D);
}

void launch_gate_apply(cplx* theta, const int* dimL, const int* dimR, const int* qL, const int* qR, int D, const StepParams* sp,
                       int gate_kind, int maxL, int maxR, cudaStream_t s) {
  const int grid = grid_for((long long)maxL * maxR, 128);
  const size_t sm = sizeof(cplx) * D * D * D * D;
  static bool attr8 = false;
  if (D == 8 && !attr8) {
    cudaFuncSetAttribute(gate_apply_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    attr8 = true;
  }
  switch (D) {
    case 2: gate_apply_kernel<2><<<grid, 128, sm, s>>>(theta, dimL, dimR, qL, qR, sp, gate_kind); break;
    case 3: gate_apply_kernel<3><<<grid, 128, sm, s>>>(theta, dimL, dimR, qL, qR, sp, gate_kind); break;
    case 4: gate_apply_kernel<4><<<grid, 128, sm, s>>>(theta, dimL, dimR, qL, qR, sp, gate_kind); break;
    case 5: gate_apply_kernel<5><<<grid, 128, sm, s>>>(theta, dimL, dimR, qL, qR, sp, gate_kind); break;
    case 6: gate_apply_kernel<6><<<grid, 128, sm, s>>>(theta, dimL, dimR, qL, qR, sp, gate_kind); break;
    case 7: gate_apply_kernel<7><<<grid, 128, sm, s>>>(theta, dimL, dimR, qL, qR, sp, gate_kind); break;
    case 8: gate_apply_kernel<8><<<grid, 128, sm, s>>>(theta, dimL, dimR, qL, qR, sp, gate_kind); break;
    default: break;
  }
}

void launch_merge_gate(const cplx* A1, const cplx* A2, cplx* theta, const int* dimL, const int* dimM, const int* dimR,
                       const int* qL, const int* qM, const int* qR, int D, const StepParams* sp, int gate_kind, int maxL, int maxR,
                       cudaStream_t s) {
  dim3 grid((maxR + 7) / 8, (maxL + 3) / 4);
  switch (D) {
    case 2: merge_gate_kernel<2><<<grid, 128, 0, s>>>(A1, A2, theta, dimL, dimM, dimR, qL, qM, qR, sp, gate_kind); break;
    case 3: merge_gate_kernel<3><<<grid, 128, 0, s>>>(A1, A2, theta, dimL, dimM, dimR, qL, qM, qR, sp, gate_kind); break;
    case 4: merge_gate_kernel<4><<<grid, 128, 0, s>>>(A1, A2, theta, dimL, dimM, dimR, qL, qM, qR, sp, gate_kind); break;
    case 5: merge_gate_kernel<5><<<grid, 128, 0, s>>>(A1, A2, theta, dimL, dimM, dimR, qL, qM, qR, sp, gate_kind); break;
    case 6: merge_gate_kernel<6><<<grid, 128, 0, s>>>(A1, A2, theta, dimL, dimM, dimR, qL, qM, qR, sp, gate_kind); break;
    case 7: merge_gate_kernel<7><<<grid, 128, 0, s>>>(A1, A2, theta, dimL, dimM, dimR, qL, qM, qR, sp, gate_kind); break;
    case 8: merge_gate_kernel<8><<<grid, 128, 0, s>>>(A1, A2, theta, dimL, dimM, dimR, qL, qM, qR, sp, gate_kind); break;
    default: break;
  }
}

void launch_site_phase(cplx* A, const int* dimL, const int* dimR, int D, const StepParams* sp, int which, int max_elems, cudaStream_t s) {
  site_phase_kernel<<<grid_for(max_elems, 256), 256, 0, s>>>(A, dimL, dimR, D, sp, which);
}

void launch_set_step_params(const StepParams& hp, StepParams* dst, cudaStream_t s) {
  set_step_params_kernel<<<1, 32, 0, s>>>(hp, dst);
}

// OCMPS_TMA_COPY=1 sends the slice store through the TMA unit (slice_copy_tma_kernel).  Measured on a B200 at the cfg2 shape
// (14.2 MB per slice, ncu gpu__time_duration): 8.9-9.3 us against 8.1-8.5 us of the plain load/store kernels below -- a copy
// this short is bound by its launch, the dependent loads of its sizes and one DRAM round trip, not by how the bytes are moved
// (profiles/r02_results.md) -- so the plain kernels stay the default.
static bool tma_copy_enabled() {
  static const bool on = [] { const char* e = getenv("OCMPS_TMA_COPY"); return e && e[0] == '1'; }();
  return on;
}
static void launch_slice_copy_tma(SitePtrs work, cplx* packed, SiteOffs offs, const int* dims, const int* q, int L, int D, int cap,
                                  int max_site_elems, const StepParams* sp, int mode, int* status, cudaStream_t s) {
  static std::once_flag once[64];
  int dev = 0;
  cudaGetDevice(&dev);
  std::call_once(once[dev & 63], [] {
    cudaFuncSetAttribute(slice_copy_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tma::CHUNK * tma::STAGES);
  });
  const long long max_chunks = ((long long)max_site_elems * (long long)sizeof(cplx) + tma::CHUNK - 1) / tma::CHUNK;
  // about two CTAs per SM over all sites, at least one chunk per CTA
  int gx = (int)std::min<long long>(std::max<long long>(max_chunks, 1), std::max(1, (2 * 148 + L - 1) / L));
  dim3 grid(gx, mode == 2 ? L + 1 : L);
  slice_copy_tma_kernel<<<grid, 32, tma::CHUNK * tma::STAGES, s>>>(work, packed, offs, dims, q, L, D, cap, sp, mode, status);
}

void launch_pack_to_slot(SitePtrs src, SiteOffs offs, const int* dims, const int* q, int L, int D, int cap, int max_site_elems,
                         const StepParams* sp, int* status, cudaStream_t s) {
  if (tma_copy_enabled()) { launch_slice_copy_tma(src, nullptr, offs, dims, q, L, D, cap, max_site_elems, sp, 2, status, s); return; }
  dim3 grid(grid_for(max_site_elems, 256, 64), L + 1);
  pack_to_slot_kernel<<<grid, 256, 0, s>>>(src, offs, dims, q, L, D, cap, sp);
}

void launch_pack_copy(SitePtrs src, cplx* dst_base, SiteOffs offs, const int* dims, int L, int D, int max_site_elems, int* status,
                      cudaStream_t s) {
  if (tma_copy_enabled()) { launch_slice_copy_tma(src, dst_base, offs, dims, nullptr, L, D, 0, max_site_elems, nullptr, 0, status, s); return; }
  dim3 grid(grid_for(max_site_elems, 256, 64), L);
  pack_copy_kernel<<<grid, 256, 0, s>>>(src, dst_base, offs, dims, D);
}
void launch_unpack_copy(const cplx* src_base, SitePtrs dst, SiteOffs offs, const int* dims, int L, int D, int max_site_elems, int* status,
                        cudaStream_t s) {
  if (tma_copy_enabled()) { launch_slice_copy_tma(dst, const_cast<cplx*>(src_base), offs, dims, nullptr, L, D, 0, max_site_elems, nullptr, 1, status, s); return; }
  dim3 grid(grid_for(max_site_elems, 256, 64), L);
  unpack_copy_kernel<<<grid, 256, 0, s>>>(src_base, dst, offs, dims, D);
}

void launch_overlap_plan(GemmDesc* descs, const OvlSide& bra, const OvlSide& ket, int site, int batch, int D, int withK,
                         cplx* E_in, cplx* E_out, cplx* T, long long e_stride, long long t_stride, cudaStream_t s) {
  overlap_plan_kernel<<<(batch + 63) / 64, 64, 0, s>>>(descs, bra, ket, site, batch, D, withK ? 2 : 1, E_in, E_out, T, T, e_stride,
                                                       t_stride);
}
void launch_overlap_plan_channels(GemmDesc* descs, const OvlSide& bra, const OvlSide& ket, int site, int batch, int D, int nch,
                                  cplx* E_in, cplx* E_out, cplx* T, const cplx* Tmix, long long e_stride, long long t_stride,
                                  cudaStream_t s) {
  overlap_plan_kernel<<<(batch + 63) / 64, 64, 0, s>>>(descs, bra, ket, site, batch, D, nch, E_in, E_out, T, Tmix, e_stride, t_stride);
}
void launch_energy_init(cplx* E, long long e_stride, int batch, int nch, cudaStream_t s) {
  energy_init_kernel<<<(batch + 63) / 64, 64, 0, s>>>(E, e_stride, batch, nch);
}
void launch_energy_mix(const cplx* T, cplx* Tmix, long long t_stride, const GemmDesc* descs, int batch, int D, const double* uc,
                       const EnergyTable& tab, int max_cols, cudaStream_t s) {
  const dim3 grid(grid_for(max_cols, 256, 128), batch);
  switch (D) {
    case 1: energy_mix_kernel<1><<<grid, 256, 0, s>>>(T, Tmix, t_stride, descs, uc, tab); break;
    case 2: energy_mix_kernel<2><<<grid, 256, 0, s>>>(T, Tmix, t_stride, descs, uc, tab); break;
    case 3: energy_mix_kernel<3><<<grid, 256, 0, s>>>(T, Tmix, t_stride, descs, uc, tab); break;
    case 4: energy_mix_kernel<4><<<grid, 256, 0, s>>>(T, Tmix, t_stride, descs, uc, tab); break;
    case 5: energy_mix_kernel<5><<<grid, 256, 0, s>>>(T, Tmix, t_stride, descs, uc, tab); break;
    case 6: energy_mix_kernel<6><<<grid, 256, 0, s>>>(T, Tmix, t_stride, descs, uc, tab); break;
    case 7: energy_mix_kernel<7><<<grid, 256, 0, s>>>(T, Tmix, t_stride, descs, uc, tab); break;
    default: energy_mix_kernel<8><<<grid, 256, 0, s>>>(T, Tmix, t_stride, descs, uc, tab); break;
  }
}
void launch_energy_final(const cplx* E, long long e_stride, int batch, int nch, double* out, cudaStream_t s) {
  energy_final_kernel<<<(batch + 63) / 64, 64, 0, s>>>(E, e_stride, batch, nch, out);
}
void launch_overlap_local_expect(const GemmDesc* descs, const OvlSide& bra, int site, int batch, int D, const double* ops, int nops,
                                 double* out, int L, cudaStream_t s) {
  overlap_local_expect_kernel<<<batch, 256, 0, s>>>(descs, bra, site, D, ops, nops, out, L);
}
void launch_overlap_init(cplx* E, long long e_stride, int batch, int withK, cudaStream_t s) {
  overlap_init_kernel<<<(batch + 63) / 64, 64, 0, s>>>(E, e_stride, batch, withK);
}
void launch_overlap_kfix(cplx* T, long long t_stride, const GemmDesc* descs, int batch, int D, int max_elems, cudaStream_t s) {
  dim3 grid(grid_for(max_elems, 256, 32), batch);
  overlap_kfix_kernel<<<grid, 256, 0, s>>>(T, t_stride, descs, D);
}
void launch_overlap_site_op(cplx* T, long long t_stride, const GemmDesc* descs, int batch, int D, const double* op_table, const int* sel,
                            int max_elems, cudaStream_t s) {
  int gx = (max_elems + 255) / 256;
  if (gx < 1) gx = 1;
  if (gx > 64) gx = 64;
  overlap_site_op_kernel<<<dim3(gx, batch), 256, 0, s>>>(T, t_stride, descs, D, op_table, sel);
}
void launch_overlap_final(const cplx* E, long long e_stride, int batch, int withK, cplx* out, cudaStream_t s) {
  overlap_final_kernel<<<(batch + 63) / 64, 64, 0, s>>>(E, e_stride, batch, withK, out);
}

void launch_applyK_expand(const cplx* A, cplx* B, const int* dimL_in, const int* dimR_in, const int* qL_in, const int* qR_in,
                          int* dimL_out, int* dimR_out, int* qL_out, int* qR_out, int D, int site, int L, int max_elems,
                          cudaStream_t s) {
  applyK_expand_kernel<<<grid_for(max_elems, 256), 256, 0, s>>>(A, B, dimL_in, dimR_in, qL_in, qR_in, dimL_out, dimR_out,
                                                                 qL_out, qR_out, D, site, L);
}
