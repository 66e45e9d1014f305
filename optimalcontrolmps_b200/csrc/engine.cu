// Host orchestration of libocmps and its C ABI (include/ocmps.h).
//
// A Trotter step is a fixed, data-independent list of operations (phase, two-site gate +
// truncating decomposition, gauge move, normalise) derived from the chain length exactly the
// way BH_tDMRG::doStep walks its gate list (reference src/BH_tDMRG.cpp:127-230, including
// ITensor's orthogonality-limit bookkeeping).  All data-dependent sizes stay on the GPU, so a
// whole sweep is enqueued without host synchronisation; independent chains (psi sweep, xi
// sweep, Hessian rows) run on their own streams.
#include <cmath>
#include <complex>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <algorithm>
#include <string>
#include <atomic>
#include <chrono>
#include <map>
#include <mutex>
#include <tuple>
#include <thread>
#include <vector>

#include "ocmps_internal.h"
#include "../../include/ocmps.h"

std::atomic<long long> g_ocmps_launches{0};

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define CK(call)                                                                                     \
  do {                                                                                               \
    cudaError_t e__ = (call);                                                                        \
    if (e__ != cudaSuccess)                                                                          \
      return fail(OCMPS_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));              \
  } while (0)

constexpr double MIN_CUT = 1e-16;   // ITensor default Cutoff (SURVEY A.3)
constexpr int MAX_M = 5000;         // ITensor default Maxm
constexpr int NV_MAX = 2048;        // must match decomp.cu
constexpr size_t JAC_SMEM_LIMIT = 200 * 1024;

struct Layout {
  int L = 0, D = 0, cap = 0;
  int capb[OCMPS_MAX_L + 1];
  SiteOffs offs;
  long long total = 0;
  int max_site_elems = 0;
  // mult = 2 for the intermediate K|psi> product whose bonds are twice those of a chi_cap MPS
  void init(int L_, int D_, int cap_, int mult = 1) {
    L = L_; D = D_; cap = cap_ * mult;
    for (int b = 0; b <= L; ++b) {
      int e = std::min(b, L - b);
      long long v = 1;
      for (int i = 0; i < e && v < cap_; ++i) v *= D;
      capb[b] = (int)std::min<long long>(v, cap_) * ((b == 0 || b == L) ? 1 : mult);
    }
    total = 0; max_site_elems = 0;
    for (int j = 0; j < L; ++j) {
      offs.o[j] = total;
      long long n = (long long)capb[j] * D * capb[j + 1];
      max_site_elems = std::max<long long>(max_site_elems, n);
      total += n;
    }
    offs.o[L] = total;
  }
};

}  // namespace

struct ocmps_ctx {
  int dev = 0;
  cudaStream_t stream0 = nullptr;
  // Everything below is shared by concurrent C-ABI calls (the reference steps one const BH_tDMRG from several
  // std::threads, src/OptimalControl.cpp:424-430) and guarded by `mu`.  A call checks workspaces out of the pool for its
  // duration (WsLease); a workspace -- stream, scratch buffers, step graphs, device status word -- is never shared
  // by two calls in flight.
  std::mutex mu;
  std::atomic<int> qmax{0};     // largest boson-number label uploaded so far: bounds the number of charge blocks
  std::vector<struct Workspace*> pool;
  std::vector<long long> dead_mps;   // serials of destroyed MPS: their step graphs are dropped when a workspace is next leased
  cudaEvent_t t0 = nullptr, t1 = nullptr;   // ocmps_timer_start / ocmps_timer_stop
};

struct ocmps_mps {
  ocmps_ctx* ctx = nullptr;
  Layout lay;
  cplx* arena[2] = {nullptr, nullptr};
  int cur[OCMPS_MAX_L];
  int* d_dims = nullptr;
  int* d_q = nullptr;       // (L+1) x cap
  int llim = 0, rlim = 2;
  long long serial = 0;     // unique id: key of the step graphs captured for this MPS (an address can be reused, a serial cannot)
  cplx* site(int j) const { return arena[cur[j]] + lay.offs.o[j]; }
  cplx* other(int j) const { return arena[1 - cur[j]] + lay.offs.o[j]; }
  int* dim(int b) const { return d_dims + b; }
  int* q(int b) const { return d_q + (size_t)b * lay.cap; }
  SitePtrs ptrs() const {
    SitePtrs p;
    for (int j = 0; j < lay.L; ++j) p.p[j] = site(j);
    return p;
  }
};

struct ocmps_store {
  ocmps_ctx* ctx = nullptr;
  Layout lay;
  int nslots = 0;
  cplx* data = nullptr;
  int* dims = nullptr;     // nslots x (L+1)
  int* q = nullptr;        // nslots x (L+1) x cap
};

namespace {

struct Op {
  int kind;    // 0 phase, 1 gate, 2 orth, 3 normalise
  int a, b, c; // phase: site(1-based), which(0: U1 / 1: U2), -; gate: i1, gate_kind(0 left,1 left+U2 on last,2 right), dir(0 left,1 right);
               // orth: bond b (sites b,b+1), dir; normalise: site
};

}  // namespace

struct Workspace {
  ocmps_ctx* ctx = nullptr;
  int L = 0, D = 0, cap = 0;
  bool busy = false;           // checked out by a call in flight (guarded by ctx->mu)
  size_t dead_seen = 0;        // prefix of ctx->dead_mps whose graphs have been dropped here
  int* d_status = nullptr;     // device status word of this workspace (kernels OR error bits into it)
  cplx* d_div = nullptr; int div_cap = 0;      // divT accumulator of the BFGS branch
  cudaStream_t stream = nullptr;
  cudaStream_t ovl = nullptr;                  // Hessian rows: batched overlaps of finished chunks run beside the chain
  cplx* theta = nullptr;
  cplx* cbuf = nullptr;
  DecompBuffers db;
  // Second set of decomposition buffers + side stream: the block table of decomposition n+1 only depends on bond
  // labels that are final once decomposition n has truncated, so it is built on `side` while n assembles its factors
  // (and, before a gate, while the two-site tensor is merged and the gate applied).  Consecutive decompositions of a
  // Trotter step alternate between db and db2.
  DecompBuffers db2;
  cudaStream_t side = nullptr;
  cudaEvent_t ev_trunc = nullptr, ev_setup = nullptr;
  // Third stream: inside one decomposition the blocks that fit one SM (QR -> register-resident rotations) and the blocks that
  // need a cluster (qr_big -> jacobi_big) are independent chains of kernels; the cluster chain runs on `side2` beside the other.
  SvdFork fork;
  // Second stage of the largest register-cached charge blocks spread over a thread-block cluster (jacobi_rows_cluster_kernel):
  // set per call by WsLease::acquire, for calls that run one or two chains.  With many chains in flight every SM is busy anyway
  // and four SMs per block would cost throughput, so those calls keep the one-SM kernel.
  bool spread_jacobi = true;
  // overlaps
  cplx* E[2] = {nullptr, nullptr};
  cplx* T = nullptr;
  GemmDesc* odescs = nullptr;
  cplx* d_out = nullptr;       // overlap results (device)
  int obatch = 0;
  long long e_stride = 0, t_stride = 0;
  // energy moments: nch-channel environments, T and the channel-mixed T' (kept apart from the overlap buffers, so that a
  // 16-channel pass does not grow what every overlap call of the workspace carries)
  struct EnergyBufs {
    cplx* E[2] = {nullptr, nullptr};
    cplx* T = nullptr;
    cplx* Tm = nullptr;
    GemmDesc* descs = nullptr;
    double* uc = nullptr;        // (U_z, c_z / L) per batch entry
    double* out = nullptr;       // 3 per batch entry
    long long e_elems = 0, t_elems = 0, ndescs = 0;   // allocated sizes (elements of each E / of T and of T')
    int batch = 0;
    long long e_stride = 0, t_stride = 0;             // of the current call
  } en;
  // work states
  ocmps_mps* work = nullptr;
  ocmps_mps* big = nullptr;    // 2*cap bonds, for K|psi>
  Workspace* bigws = nullptr;  // decomposition buffers for 2*cap
  double* d_norm = nullptr;    // scalar outputs
  StepParams* d_params = nullptr;   // per-step scalars and pointers (device), see StepParams
  ocmps_mps* tmpK = nullptr;        // K|xi_i> before it goes to its slot (ocmps_store_apply_K)
  ocmps_mps* psiH = nullptr;        // Hessian-row state of this chain
  ocmps_store* rowstore = nullptr;  // Hessian rows: the last few propagated slices, overlapped with xiH in one batched pass
  // CUDA graphs of one Trotter step (+ slice store), keyed by stepper serial, MPS serial, buffer parity, with/without
  // store, the block-grid bound (ctx->qmax) that the launches of the captured sequence were sized with, and spread_jacobi
  struct StepGraph { cudaGraphExec_t exec = nullptr; unsigned long long flips = 0; int launches = 0; int seen = 0; };
  std::map<std::tuple<long long, long long, unsigned long long, int, int, int>, StepGraph> graphs;
};

struct ocmps_stepper {
  ocmps_ctx* ctx = nullptr;
  int L = 0, D = 0, cap = 0;
  double J = 1.0, tstep = 0.0;
  bool has_cutoff = false, has_maxm = false;
  double cutoff = MIN_CUT;
  int maxm = MAX_M;
  int rel_cutoff = 0;
  cplx* d_G[2] = {nullptr, nullptr};     // [0] forward, [1] backward
  std::vector<std::complex<double>> h_G[2];
  std::vector<Op> ops;
  long long serial = 0;      // unique id (graph cache key)
  bool imag = false;         // imaginary-time evolution exp(-tau H) (ground-state generator): real gates, renormalised every step
};

namespace {

// ------------------------------------------------------------------------------------------------
// allocation helpers
// ------------------------------------------------------------------------------------------------
int alloc_mps(ocmps_ctx* ctx, int L, int D, int cap, ocmps_mps** out, int mult = 1) {
  if (L < 1 || L > OCMPS_MAX_L) return fail(OCMPS_ERR_INVALID, "L out of range [1,64]");
  if (D < 2 || D > OCMPS_MAX_D) return fail(OCMPS_ERR_INVALID, "D out of range [2,8]");
  if (cap < 1 || (long long)cap * mult * D > NV_MAX) return fail(OCMPS_ERR_INVALID, "chi_cap*D exceeds 2048");
  ocmps_mps* m = new ocmps_mps();
  m->ctx = ctx;
  m->lay.init(L, D, cap, mult);
  cap = m->lay.cap;
  CK(cudaSetDevice(ctx->dev));
  CK(cudaMalloc(&m->arena[0], sizeof(cplx) * m->lay.total));
  CK(cudaMalloc(&m->arena[1], sizeof(cplx) * m->lay.total));
  CK(cudaMalloc(&m->d_dims, sizeof(int) * (L + 1)));
  CK(cudaMalloc(&m->d_q, sizeof(int) * (size_t)(L + 1) * cap));
  CK(cudaMemset(m->d_dims, 0, sizeof(int) * (L + 1)));
  CK(cudaMemset(m->d_q, 0, sizeof(int) * (size_t)(L + 1) * cap));
  for (int j = 0; j < L; ++j) m->cur[j] = 0;
  { static std::atomic<long long> next_serial{1}; m->serial = next_serial++; }
  // the memsets above run on the legacy default stream, which does not order against the engine's non-blocking
  // streams: make sure they have landed before any chain touches the new buffers
  CK(cudaStreamSynchronize(cudaStreamLegacy));
  *out = m;
  return OCMPS_OK;
}

void free_mps(ocmps_mps* m) {
  if (!m) return;
  if (m->ctx) {      // step graphs captured for this MPS hold its buffer addresses: have every workspace drop them
    std::lock_guard<std::mutex> lock(m->ctx->mu);
    m->ctx->dead_mps.push_back(m->serial);
  }
  cudaFree(m->arena[0]); cudaFree(m->arena[1]); cudaFree(m->d_dims); cudaFree(m->d_q);
  delete m;
}

int alloc_ws(ocmps_ctx* ctx, int L, int D, int cap, bool with_work, Workspace** out, bool high_priority = false) {
  Workspace* w = new Workspace();
  w->ctx = ctx; w->L = L; w->D = D; w->cap = cap;
  CK(cudaSetDevice(ctx->dev));
  // The first two workspaces of a shape serve the psi / xi sweeps (leases hand out the lowest-numbered free workspaces):
  // their streams get the highest priority, so that the sweeps -- the critical path of a Hessian whose rows trail the psi
  // sweep -- are not queued behind the CTAs of dozens of row chains.  Kernel nodes of captured graphs inherit it.
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  const int prio = high_priority ? prio_hi : prio_lo;
  CK(cudaStreamCreateWithPriority(&w->stream, cudaStreamNonBlocking, prio));
  const size_t nD = (size_t)cap * D;
  CK(cudaMalloc(&w->theta, sizeof(cplx) * nD * nD));
  CK(cudaMalloc(&w->cbuf, sizeof(cplx) * (size_t)cap * cap));
  CK(cudaMalloc(&w->db.dw, sizeof(DecompWork)));
  CK(cudaMalloc(&w->db.vec_idx, sizeof(int) * 3 * NV_MAX));
  CK(cudaMalloc(&w->db.comp_idx, sizeof(int) * 3 * NV_MAX));
  CK(cudaMalloc(&w->db.vecq, sizeof(int) * NV_MAX));
  CK(cudaMalloc(&w->db.P, sizeof(double) * NV_MAX));
  CK(cudaMalloc(&w->db.pos, sizeof(int) * 3 * NV_MAX));
  // per block max(nv*len, rows*pad16(nv)) elements: sum_q <= cap*(D*cap) + cap*16*OCMPS_MAX_BLK
  const size_t ywhalf = nD * cap + (size_t)cap * 16 * OCMPS_MAX_BLK;
  CK(cudaMalloc(&w->db.ywork, sizeof(cplx) * 2 * ywhalf));
  w->db.ywork_half = (long long)ywhalf;
  CK(cudaMalloc(&w->db.scratch_d, sizeof(double) * 8 * NV_MAX));
  CK(cudaMalloc(&w->db.descs, sizeof(GemmDesc) * 4));
  CK(cudaMalloc(&w->db.partial, sizeof(double) * 64));
  CK(cudaMalloc(&w->d_norm, sizeof(double) * 4));
  CK(cudaMalloc(&w->d_params, sizeof(StepParams)));
  CK(cudaMalloc(&w->d_status, sizeof(int)));
  CK(cudaMemset(w->d_status, 0, sizeof(int)));
  w->db.status = w->d_status;
  w->db2 = w->db;                                     // shares status, partial; everything a decomposition writes is separate
  CK(cudaMalloc(&w->db2.dw, sizeof(DecompWork)));
  CK(cudaMalloc(&w->db2.vec_idx, sizeof(int) * 3 * NV_MAX));
  CK(cudaMalloc(&w->db2.comp_idx, sizeof(int) * 3 * NV_MAX));
  CK(cudaMalloc(&w->db2.vecq, sizeof(int) * NV_MAX));
  CK(cudaMalloc(&w->db2.P, sizeof(double) * NV_MAX));
  CK(cudaMalloc(&w->db2.pos, sizeof(int) * 3 * NV_MAX));
  CK(cudaMalloc(&w->db2.ywork, sizeof(cplx) * 2 * ywhalf));
  CK(cudaMalloc(&w->db2.scratch_d, sizeof(double) * 8 * NV_MAX));
  CK(cudaMalloc(&w->db2.descs, sizeof(GemmDesc) * 4));
  CK(cudaStreamCreateWithPriority(&w->side, cudaStreamNonBlocking, prio));
  CK(cudaEventCreateWithFlags(&w->ev_trunc, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&w->ev_setup, cudaEventDisableTiming));
  CK(cudaStreamCreateWithPriority(&w->fork.stream, cudaStreamNonBlocking, prio));
  CK(cudaEventCreateWithFlags(&w->fork.ev_fork, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&w->fork.ev_first, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&w->fork.ev_join, cudaEventDisableTiming));
  if (with_work) {
    int rc = alloc_mps(ctx, L, D, cap, &w->work);
    if (rc) return rc;
  }
  *out = w;
  return OCMPS_OK;
}

int ensure_overlap_bufs(Workspace* w, int batch, int capA, int capB) {
  const long long es = 2LL * capA * capB, ts = 2LL * capA * w->D * capB;
  if (w->obatch >= batch && w->e_stride >= es && w->t_stride >= ts) return OCMPS_OK;
  cudaFree(w->E[0]); cudaFree(w->E[1]); cudaFree(w->T); cudaFree(w->odescs); cudaFree(w->d_out);
  w->obatch = std::max(batch, w->obatch);
  w->e_stride = std::max(es, w->e_stride); w->t_stride = std::max(ts, w->t_stride);
  CK(cudaMalloc(&w->E[0], sizeof(cplx) * w->e_stride * w->obatch));
  CK(cudaMalloc(&w->E[1], sizeof(cplx) * w->e_stride * w->obatch));
  CK(cudaMalloc(&w->T, sizeof(cplx) * w->t_stride * w->obatch));
  CK(cudaMalloc(&w->odescs, sizeof(GemmDesc) * 3 * w->obatch));
  CK(cudaMalloc(&w->d_out, sizeof(cplx) * w->obatch));
  return OCMPS_OK;
}

// Energy-moment buffers for `batch` entries of nch channels at capacity cap (the workspace's stream is idle).  Sized in
// elements, so that the 4- and 16-channel passes, whose batches are cut to the same byte budget, share one allocation.
int ensure_energy_bufs(Workspace* w, int batch, int nch, int cap) {
  auto& b = w->en;
  const long long es = (long long)nch * cap * cap, ts = (long long)nch * cap * w->D * cap;
  b.e_stride = es; b.t_stride = ts;
  if (b.e_elems >= es * batch && b.t_elems >= ts * batch && b.ndescs >= (1LL + nch) * batch && b.batch >= batch) return OCMPS_OK;
  cudaFree(b.E[0]); cudaFree(b.E[1]); cudaFree(b.T); cudaFree(b.Tm); cudaFree(b.descs); cudaFree(b.uc); cudaFree(b.out);
  b.E[0] = b.E[1] = b.T = b.Tm = nullptr; b.descs = nullptr; b.uc = b.out = nullptr;
  b.e_elems = std::max(b.e_elems, es * batch); b.t_elems = std::max(b.t_elems, ts * batch);
  b.ndescs = std::max(b.ndescs, (1LL + nch) * batch); b.batch = std::max(b.batch, batch);
  CK(cudaMalloc(&b.E[0], sizeof(cplx) * b.e_elems));
  CK(cudaMalloc(&b.E[1], sizeof(cplx) * b.e_elems));
  CK(cudaMalloc(&b.T, sizeof(cplx) * b.t_elems));
  CK(cudaMalloc(&b.Tm, sizeof(cplx) * b.t_elems));
  CK(cudaMalloc(&b.descs, sizeof(GemmDesc) * b.ndescs));
  CK(cudaMalloc(&b.uc, sizeof(double) * 2 * b.batch));
  CK(cudaMalloc(&b.out, sizeof(double) * 3 * b.batch));
  return OCMPS_OK;
}

void free_ws(Workspace* w) {
  if (!w) return;
  cudaFree(w->theta); cudaFree(w->cbuf); cudaFree(w->db.dw); cudaFree(w->db.vec_idx); cudaFree(w->db.comp_idx);
  cudaFree(w->db.vecq); cudaFree(w->db.P); cudaFree(w->db.pos); cudaFree(w->db.ywork); cudaFree(w->db.descs);
  cudaFree(w->db.partial); cudaFree(w->d_norm); cudaFree(w->db.scratch_d); cudaFree(w->d_params);
  cudaFree(w->db2.dw); cudaFree(w->db2.vec_idx); cudaFree(w->db2.comp_idx); cudaFree(w->db2.vecq); cudaFree(w->db2.P);
  cudaFree(w->db2.pos); cudaFree(w->db2.ywork); cudaFree(w->db2.scratch_d); cudaFree(w->db2.descs);
  if (w->side) cudaStreamDestroy(w->side);
  if (w->fork.stream) cudaStreamDestroy(w->fork.stream);
  if (w->fork.ev_fork) cudaEventDestroy(w->fork.ev_fork);
  if (w->fork.ev_first) cudaEventDestroy(w->fork.ev_first);
  if (w->fork.ev_join) cudaEventDestroy(w->fork.ev_join);
  if (w->ev_trunc) cudaEventDestroy(w->ev_trunc);
  if (w->ev_setup) cudaEventDestroy(w->ev_setup);
  for (auto& kv : w->graphs) if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  if (w->psiH) w->psiH->ctx = nullptr;
  free_mps(w->psiH);
  if (w->tmpK) w->tmpK->ctx = nullptr;
  free_mps(w->tmpK);
  if (w->rowstore) { cudaFree(w->rowstore->data); cudaFree(w->rowstore->dims); cudaFree(w->rowstore->q); delete w->rowstore; }
  cudaFree(w->E[0]); cudaFree(w->E[1]); cudaFree(w->T); cudaFree(w->odescs); cudaFree(w->d_out);
  cudaFree(w->en.E[0]); cudaFree(w->en.E[1]); cudaFree(w->en.T); cudaFree(w->en.Tm); cudaFree(w->en.descs); cudaFree(w->en.uc);
  cudaFree(w->en.out);
  cudaFree(w->d_status); cudaFree(w->d_div);
  if (w->work) w->work->ctx = nullptr;      // (owned by the workspace, whose graphs are gone with it: no bookkeeping)
  if (w->big) w->big->ctx = nullptr;
  free_mps(w->work); free_mps(w->big);
  if (w->bigws) free_ws(w->bigws);
  if (w->stream) cudaStreamDestroy(w->stream);
  if (w->ovl) cudaStreamDestroy(w->ovl);
  delete w;
}

// Workspaces of one shape checked out of the context's pool for the duration of a C-ABI call.  Two calls in flight
// (different host threads, different MPS / stores) never share a workspace, so `step`, the sweeps and the overlaps are
// re-entrant on one const stepper like the reference's (src/BH_tDMRG.cpp:113-115).  The lowest-numbered free workspaces
// are taken first: a single-threaded caller always gets the same ones back, with their step graphs and Hessian buffers.
struct WsLease {
  ocmps_ctx* ctx = nullptr;
  std::vector<Workspace*> ws;
  WsLease() = default;
  WsLease(const WsLease&) = delete;
  WsLease& operator=(const WsLease&) = delete;
  ~WsLease() { release(); }
  void release() {
    if (!ctx || ws.empty()) return;
    std::lock_guard<std::mutex> lock(ctx->mu);
    for (Workspace* w : ws) w->busy = false;
    ws.clear();
  }
  int acquire(ocmps_ctx* c, int L, int D, int cap, int n) {
    ctx = c;
    std::lock_guard<std::mutex> lock(c->mu);
    for (Workspace* w : c->pool) {
      if ((int)ws.size() == n) break;
      if (!w->busy && w->L == L && w->D == D && w->cap == cap) { w->busy = true; ws.push_back(w); }
    }
    while ((int)ws.size() < n) {
      Workspace* w = nullptr;
      int same = 0;
      for (Workspace* o : c->pool) if (o->L == L && o->D == D && o->cap == cap) ++same;
      int rc = alloc_ws(c, L, D, cap, true, &w, same < 2);
      if (rc) return rc;
      w->busy = true;
      c->pool.push_back(w);
      ws.push_back(w);
    }
    for (Workspace* w : ws) w->spread_jacobi = n <= 2;
    for (Workspace* w : ws) {          // graphs of MPS destroyed since this workspace was last used
      if (w->dead_seen == c->dead_mps.size()) continue;
      if (!w->graphs.empty()) {
        std::vector<long long> dead(c->dead_mps.begin() + w->dead_seen, c->dead_mps.end());
        std::sort(dead.begin(), dead.end());
        for (auto it = w->graphs.begin(); it != w->graphs.end();) {
          if (std::binary_search(dead.begin(), dead.end(), std::get<1>(it->first))) {
            if (it->second.exec) cudaGraphExecDestroy(it->second.exec);
            it = w->graphs.erase(it);
          } else {
            ++it;
          }
        }
      }
      w->dead_seen = c->dead_mps.size();
    }
    return OCMPS_OK;
  }
  Workspace* operator[](int i) const { return ws[i]; }
  // waits for the leased streams and reports (and clears) what the kernels flagged
  int finish() {
    int st = 0;
    for (Workspace* w : ws) {
      CK(cudaStreamSynchronize(w->stream));
      int s1 = 0;
      CK(cudaMemcpy(&s1, w->d_status, sizeof(int), cudaMemcpyDeviceToHost));
      if (s1) { cudaMemset(w->d_status, 0, sizeof(int)); st |= s1; }
    }
    CK(cudaGetLastError());
    if (st) {
      std::string msg = "device status:";
      if (st & OCMPS_ST_CAPACITY) msg += " bond dimension exceeds chi_cap;";
      if (st & OCMPS_ST_NOCONV) msg += " Jacobi did not converge;";
      if (st & OCMPS_ST_CHARGE) msg += " charge label >= 256;";
      if (st & OCMPS_ST_TOOMANYBLK) msg += " more charge blocks than the launch was sized for;";
      return fail((st & OCMPS_ST_CAPACITY) ? OCMPS_ERR_CAPACITY : OCMPS_ERR_NUMERIC, msg);
    }
    return OCMPS_OK;
  }
};

// ------------------------------------------------------------------------------------------------
// gates (BondGate, SURVEY A.1) and the op schedule (src/BH_tDMRG.cpp:127-230)
// ------------------------------------------------------------------------------------------------
typedef std::complex<double> zc;

// exp(factor * h) by ITensor BondGate's Horner recursion; factor = -i tau for real time, -tau for imaginary time
std::vector<zc> bond_gate(int D, double J, double tau, bool imag = false) {
  const int n = D * D;
  std::vector<zc> h(n * n, 0.0), unit(n * n, 0.0), term, gate, x(n * n);
  // h[(t1,t2),(s1,s2)] = -J (A x Adag + Adag x A); <j-1|A|j> = sqrt(j)   (BH_sites.h:136-148)
  auto Aop = [&](int t, int s) { return (s == t + 1) ? std::sqrt((double)s) : 0.0; };
  auto Adop = [&](int t, int s) { return (t == s + 1) ? std::sqrt((double)t) : 0.0; };
  for (int t1 = 0; t1 < D; ++t1) for (int t2 = 0; t2 < D; ++t2)
    for (int s1 = 0; s1 < D; ++s1) for (int s2 = 0; s2 < D; ++s2)
      h[(t1 * D + t2) * n + s1 * D + s2] = -J * (Aop(t1, s1) * Adop(t2, s2) + Adop(t1, s1) * Aop(t2, s2));
  for (int i = 0; i < n; ++i) unit[i * n + i] = 1.0;
  for (int i = 0; i < n * n; ++i) x[i] = h[i] * (imag ? zc(-tau, 0.0) : zc(0.0, -tau));
  term = x;
  gate = unit;
  std::vector<zc> tmp(n * n);
  for (int ord = 100; ord >= 1; --ord) {       // Horner form of the Taylor series
    for (int i = 0; i < n * n; ++i) { term[i] /= (double)ord; gate[i] = unit[i] + term[i]; }
    for (int i = 0; i < n; ++i)
      for (int j = 0; j < n; ++j) {
        zc s = 0.0;
        for (int k = 0; k < n; ++k) s += gate[i * n + k] * x[k * n + j];
        tmp[i * n + j] = s;
      }
    term = tmp;
  }
  return gate;
}

struct Limits {
  int l = 0, r = 2;
  void touch(int i) { if (l > i - 1) l = i - 1; if (r < i + 1) r = i + 1; }
};

void emit_position(std::vector<Op>& ops, Limits& lim, int i, int L) {
  while (lim.l < i - 1) {
    if (lim.l < 0) lim.l = 0;
    ops.push_back({2, lim.l + 1, 0, 0});
    ++lim.l;
    if (lim.r < lim.l + 2) lim.r = lim.l + 2;
  }
  while (lim.r > i + 1) {
    if (lim.r > L + 1) lim.r = L + 1;
    ops.push_back({2, lim.r - 2, 1, 0});
    --lim.r;
    if (lim.l > lim.r - 2) lim.l = lim.r - 2;
  }
}

std::vector<Op> build_schedule(int L) {
  std::vector<Op> ops;
  std::vector<std::pair<int, int>> gates;
  for (int i = 1; i < L; i += 2) gates.push_back({i, i + 1});           // :28-38
  const int offset = (L % 2 == 0) ? 2 : 1;
  for (int i = L - offset; i >= 1; i -= 2) gates.push_back({i, i + 1}); // :45-57
  Limits lim;                       // centre at site 1
  if (L % 2 != 0) {                 // :133-136
    lim.touch(L);
    ops.push_back({0, L, 0, 0});
  }
  bool from_left = true;
  for (size_t gi = 0; gi < gates.size(); ++gi) {
    const int i1 = gates[gi].first, i2 = gates[gi].second;
    lim.touch(i1); lim.touch(i2);
    const int gk = from_left ? ((i2 == L && L % 2 == 0) ? 1 : 0) : 2;
    if (gi + 1 < gates.size()) {
      const int ni1 = gates[gi + 1].first, ni2 = gates[gi + 1].second;
      if (ni1 >= i2) {              // :173-188
        ops.push_back({1, i1, gk, 0});
        lim.l = i1;
        if (lim.r < i1 + 2) lim.r = i1 + 2;
        lim.touch(i1 + 1);
        emit_position(ops, lim, ni1, L);
      }
      if (ni1 < i2) {               // :189-199
        ops.push_back({1, i1, gk, 1});
        if (lim.l > i1 - 1) lim.l = i1 - 1;
        lim.r = i1 + 1;
        lim.touch(i1);
        emit_position(ops, lim, ni2, L);
      }
      if (i2 == ni1 || i1 == ni2) from_left = false;   // :200-204
    } else {                        // :206-218
      ops.push_back({1, i1, gk, 1});
      lim.l = i1 - 1;
      lim.r = i1 + 1;
      lim.touch(i1);
      emit_position(ops, lim, 1, L);
    }
  }
  lim.touch(1);
  ops.push_back({0, 1, 1, 0});      // :222-223
  ops.push_back({3, 1, 0, 0});      // :228
  return ops;
}

// ------------------------------------------------------------------------------------------------
// development trace (OCMPS_STEP_TRACE=1, plain launches): CUDA events between the phases of every decomposition
// ------------------------------------------------------------------------------------------------
struct StepTrace {
  bool on = false;
  std::vector<std::pair<int, cudaEvent_t>> marks;     // (phase that ENDS at this mark, event)
  void mark(int phase, cudaStream_t s) {
    if (!on) return;
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    cudaEventRecord(e, s);
    marks.push_back({phase, e});
  }
};
static StepTrace g_trace;
static bool step_trace_enabled() {
  static const bool v = [] { const char* e = getenv("OCMPS_STEP_TRACE"); return e && e[0] == '1'; }();
  return v;
}
enum { TR_START = 0, TR_MERGE, TR_SETUP, TR_SVD_GATE, TR_SVD_ORTH, TR_TRUNC, TR_BUILD, TR_OTHER, TR_NPHASE };

// ------------------------------------------------------------------------------------------------
// decomposition driver
// ------------------------------------------------------------------------------------------------
// setup -> QR + Jacobi per charge block -> global truncation -> assembly of isometry and centre factor
// `db`: buffer set to use; `setup_done`: the block table was already built on the side stream (the caller has made `s`
// wait for it); `next`: if given, the setup of the following decomposition (buffer set `db_next`) is started on the
// side stream as soon as this one has truncated.
void run_decomp(Workspace* ws, const DecompArgs& a, const TruncParams& tp, int capV, int capC, int capK, cudaStream_t s,
                DecompBuffers* dbp = nullptr, bool setup_done = false, const DecompArgs* next = nullptr, DecompBuffers* db_next = nullptr) {
  DecompBuffers& db = dbp ? *dbp : ws->db;
  if (!setup_done) { launch_decomp_setup(a, db, s); g_trace.mark(TR_SETUP, s); }
  // shared memory: the largest block has at most capV vectors of at most capC components
  size_t need = (size_t)capV * capC * sizeof(cplx);
  // the Jacobi working set stores its rows (<= min(capV, capC) of them) with a stride padded to a multiple of 16
  need = std::max(need, (size_t)std::min(capV, capC) * (size_t)(((capV + 15) / 16) * 16) * sizeof(cplx));
  size_t smem = std::min(need, JAC_SMEM_LIMIT);
  if (smem < 1024) smem = 1024;
  // blocks are labelled by a charge in [0, qmax + D): launch no more CTAs than that (surplus CTAs would still have to
  // wait for an SM with the full shared-memory carve-out and would serialise concurrent chains)
  int nblk = std::min(std::min(OCMPS_MAX_BLK, std::max(capV, capC) + a.D), ws->ctx->qmax.load() + a.D + 1);
  const bool need_global = need > JAC_SMEM_LIMIT;    // some block may not fit in shared memory
  // numerical-rank tolerance of the pivoted QR: the neglected weight stays >= 6 orders below the cutoff
  static const double rank_scale = [] { const char* e = getenv("OCMPS_RANK_TOL_SCALE"); return e ? atof(e) : 1e-6; }();
  double rank_tol = rank_scale * tp.cutoff;
  rank_tol = std::min(rank_scale * 1e-8, std::max(1e-30, rank_tol));
  const bool long_rows = capV > 128;                   // rows of R longer than the register-cached path handles
  const int max_rows = std::min(capV, capC);           // rows of R of the largest possible block
  launch_jacobi_blocks(a, db, nblk, smem, need_global, long_rows, rank_tol, max_rows, capV, capC, ws->spread_jacobi, s, &ws->fork);
  g_trace.mark((a.kind == DK_GATE_LEFT || a.kind == DK_GATE_RIGHT) ? TR_SVD_GATE : TR_SVD_ORTH, s);
  launch_truncate(a, db, tp, s);
  g_trace.mark(TR_TRUNC, s);
  if (next) {
    cudaEventRecord(ws->ev_trunc, s);
    cudaStreamWaitEvent(ws->side, ws->ev_trunc, 0);
    launch_decomp_setup(*next, *db_next, ws->side);
    cudaEventRecord(ws->ev_setup, ws->side);
  }
  launch_build_factors(a, db, capK, capV, capC, s);
  g_trace.mark(TR_BUILD, s);
  g_ocmps_launches += 5 + (need_global ? 1 : 0) + (long_rows ? 1 : 0);
}

void phases_of(int D, double U, double tstep, double* re, double* im, bool imag = false) {
  for (int n = 0; n < D; ++n) {
    if (imag) {                     // imaginary time: exp(-1/4 U tau n(n-1)), the same half-step split of the on-site term
      re[n] = std::exp(-0.25 * U * tstep * (double)n * (double)(n - 1));
      im[n] = 0.0;
      continue;
    }
    const double ang = -0.25 * U * tstep * (double)n * (double)(n - 1);   // src/BH_tDMRG.cpp:87-88
    re[n] = std::cos(ang);
    im[n] = std::sin(ang);
  }
}

// gauge pushes done inside build_factors (sector-wise) instead of a dense GEMM that follows it; OCMPS_FUSED_PUSH=0 restores the GEMM
static bool fused_push_enabled() {
  static const bool v = [] { const char* e = getenv("OCMPS_FUSED_PUSH"); return !(e && e[0] == '0'); }();
  return v;
}

// the kernel sequence of one Trotter step in place on `m` (all step-dependent values are read from ws->d_params)
void run_step_body(ocmps_stepper* st, ocmps_mps* m, Workspace* ws, cudaStream_t s, int op_begin = 0, int op_end = 1 << 30) {
  const int D = st->D;
  const Layout& lay = m->lay;
  const StepParams* sp = ws->d_params;
  TruncParams tpg{st->cutoff, st->maxm, 1, st->rel_cutoff, 0, 1};
  TruncParams tpo{MIN_CUT, MAX_M, 1, 0, 0, 0};

  // what decomp_setup_kernel reads of a decomposition op: kind and the labels of the two outer bonds
  auto setup_args = [&](const Op& op) {
    DecompArgs a;
    a.D = D;
    if (op.kind == 1) {
      const int bl = op.a - 1, br = op.a + 1;
      a.kind = op.c == 0 ? DK_GATE_LEFT : DK_GATE_RIGHT;
      a.dimL = m->dim(bl); a.dimR = m->dim(br); a.qL = m->q(bl); a.qR = m->q(br);
    } else {
      const int b = op.a;
      a.kind = op.b == 0 ? DK_ORTH_LEFT : DK_ORTH_RIGHT;
      const int lo = op.b == 0 ? b - 1 : b;
      a.dimL = m->dim(lo); a.dimR = m->dim(lo + 1); a.qL = m->q(lo); a.qR = m->q(lo + 1);
    }
    a.dimNew = nullptr; a.qNew = nullptr; a.X = nullptr; a.iso = nullptr; a.partner = nullptr;
    a.nb_in = nullptr; a.nb_out = nullptr; a.dimNb = nullptr; a.qNb = nullptr;
    return a;
  };
  const bool fused_push = fused_push_enabled();
  const int op_last = std::min((int)st->ops.size(), op_end);
  int ndec = 0;                    // decompositions issued so far: number n uses buffer set n & 1
  bool pre_setup = false;          // the setup of the next decomposition is already running on the side stream
  // issues decomposition `a` of op `oi`; looks ahead for the next decomposition op to start its setup early
  auto pipelined_decomp = [&](int oi, const DecompArgs& a, const TruncParams& tp, int capV, int capC, int capK) {
    DecompBuffers* dbc = (ndec & 1) ? &ws->db2 : &ws->db;
    DecompBuffers* dbn = (ndec & 1) ? &ws->db : &ws->db2;
    if (pre_setup) cudaStreamWaitEvent(s, ws->ev_setup, 0);
    int on = oi + 1;
    while (on < op_last && st->ops[on].kind != 1 && st->ops[on].kind != 2) ++on;
    DecompArgs an;
    const bool has_next = on < op_last;
    if (has_next) an = setup_args(st->ops[on]);
    run_decomp(ws, a, tp, capV, capC, capK, s, dbc, pre_setup, has_next ? &an : nullptr, dbn);
    pre_setup = has_next;
    ++ndec;
    return dbc;
  };

  for (int oi = op_begin; oi < (int)st->ops.size() && oi < op_end; ++oi) {
    const Op& op = st->ops[oi];
    if (op.kind == 0) {
      const int j = op.a - 1;
      launch_site_phase(m->site(j), m->dim(j), m->dim(j + 1), D, sp, op.b, lay.capb[j] * D * lay.capb[j + 1], s);
      g_ocmps_launches += 1;
    } else if (op.kind == 1) {
      const int j1 = op.a - 1, j2 = op.a;                 // 0-based sites
      const int bl = j1, bm = j1 + 1, br = j2 + 1;        // bonds
      // op.b: 0 = U(from) then J (:150), 1 = plus the lonely U(to) on the last site (:153-155), 2 = J then U(to) (:159)
      static const bool fused_merge = [] { const char* e = getenv("OCMPS_FUSED_MERGE"); return !(e && e[0] == '0'); }();
      if (fused_merge && D >= 2 && D <= 8) {
        launch_merge_gate(m->site(j1), m->site(j2), ws->theta, m->dim(bl), m->dim(bm), m->dim(br), m->q(bl), m->q(bm), m->q(br), D, sp,
                          op.b, lay.capb[bl], lay.capb[br], s);
        g_trace.mark(TR_MERGE, s);
        g_ocmps_launches -= 2;
      } else {
        launch_merge_setup(ws->db.descs + 2, m->site(j1), m->site(j2), ws->theta, m->dim(bl), m->dim(bm), m->dim(br), D, s);
        launch_zgemm(ws->db.descs + 2, 1, lay.capb[bl] * D, D * lay.capb[br], s);
        launch_gate_apply(ws->theta, m->dim(bl), m->dim(br), m->q(bl), m->q(br), D, sp, op.b, lay.capb[bl], lay.capb[br], s);
      }
      DecompArgs a;
      a.kind = op.c == 0 ? DK_GATE_LEFT : DK_GATE_RIGHT;
      a.D = D;
      a.dimL = m->dim(bl); a.dimR = m->dim(br); a.qL = m->q(bl); a.qR = m->q(br);
      a.dimNew = m->dim(bm); a.qNew = m->q(bm);
      a.X = ws->theta;
      a.iso = op.c == 0 ? m->other(j1) : m->other(j2);
      a.partner = op.c == 0 ? m->other(j2) : m->other(j1);
      a.nb_in = nullptr; a.nb_out = nullptr; a.dimNb = nullptr; a.qNb = nullptr;
      tpg.cap = lay.capb[bm];
      const int n_cap = lay.capb[bl] * D, m_cap = D * lay.capb[br];
      // vectors per block <= chi of their own side, components <= chi of the other side
      const int capV = op.c == 0 ? lay.capb[br] : lay.capb[bl];
      const int capC = op.c == 0 ? lay.capb[bl] : lay.capb[br];
      (void)n_cap; (void)m_cap;
      pipelined_decomp(oi, a, tpg, capV, capC, lay.capb[bm]);  // includes the normalisation of :183-184,195-196
      m->cur[j1] ^= 1; m->cur[j2] ^= 1;
      g_ocmps_launches += 3;
    } else if (op.kind == 2) {
      const int b = op.a;                                  // bond between sites b and b+1 (1-based) = bond index b
      DecompArgs a;
      a.D = D;
      a.dimNew = m->dim(b); a.qNew = m->q(b);
      a.partner = ws->cbuf;
      tpo.cap = lay.capb[b];
      if (op.b == 0) {            // left: SVD of site b (0-based b-1), S.V pushed into site b+1
        const int j = b - 1, jn = b;
        a.kind = DK_ORTH_LEFT;
        a.dimL = m->dim(b - 1); a.dimR = m->dim(b); a.qL = m->q(b - 1); a.qR = m->q(b);
        a.X = m->site(j); a.iso = m->other(j);
        a.nb_in = m->site(jn); a.nb_out = m->other(jn); a.dimNb = m->dim(b + 1);
        a.qNb = fused_push ? m->q(b + 1) : nullptr;
        DecompBuffers* dbc = pipelined_decomp(oi, a, tpo, lay.capb[b], lay.capb[b - 1], lay.capb[b]);
        if (!fused_push) launch_zgemm(dbc->descs + 1, 1, lay.capb[b], D * lay.capb[b + 1], s);
        m->cur[j] ^= 1; m->cur[jn] ^= 1;
      } else {                    // right: SVD of site b+1 (0-based b), U.S pushed into site b
        const int j = b, jn = b - 1;
        a.kind = DK_ORTH_RIGHT;
        a.dimL = m->dim(b); a.dimR = m->dim(b + 1); a.qL = m->q(b); a.qR = m->q(b + 1);
        a.X = m->site(j); a.iso = m->other(j);
        a.nb_in = m->site(jn); a.nb_out = m->other(jn); a.dimNb = m->dim(b - 1);
        a.qNb = fused_push ? m->q(b - 1) : nullptr;
        DecompBuffers* dbc = pipelined_decomp(oi, a, tpo, lay.capb[b], lay.capb[b + 1], lay.capb[b]);
        if (!fused_push) launch_zgemm(dbc->descs + 1, 1, lay.capb[b - 1] * D, lay.capb[b], s);
        m->cur[j] ^= 1; m->cur[jn] ^= 1;
      }
      g_ocmps_launches += fused_push ? 0 : 1;
    } else {
      const int j = op.a - 1;
      launch_normalize_site(m->site(j), m->dim(j), m->dim(j + 1), D, ws->db.partial, lay.capb[j] * D * lay.capb[j + 1], s);
      g_ocmps_launches += 2;
    }
  }
  if (op_end >= (int)st->ops.size()) { m->llim = 0; m->rlim = 2; }
}

void fill_step_params(ocmps_stepper* st, double from, double to, bool forward, ocmps_store* store, int slot, StepParams& hp) {
  phases_of(st->D, forward ? from : -from, st->tstep, hp.u1r, hp.u1i, st->imag);   // src/BH_tDMRG.cpp:116-123
  phases_of(st->D, forward ? to : -to, st->tstep, hp.u2r, hp.u2i, st->imag);
  hp.G = st->d_G[forward ? 0 : 1];
  hp.slot_data = nullptr; hp.slot_dims = nullptr; hp.slot_q = nullptr;
  if (store) {
    const Layout& lay = store->lay;
    hp.slot_data = store->data + (size_t)slot * lay.total;
    hp.slot_dims = store->dims + (size_t)slot * (lay.L + 1);
    hp.slot_q = store->q + (size_t)slot * (lay.L + 1) * lay.cap;
  }
}

static bool graphs_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("OCMPS_GRAPH"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}

// One Trotter step in place on `m` (and, if `store` is given, the copy of the result into `slot`), enqueued on `s`.
// The kernel sequence only depends on (stepper, MPS buffers, buffer parity): after one plain execution it is captured
// into a CUDA graph and replayed -- 1 graph launch + 1 parameter kernel instead of ~230 launches per step.
int step_enqueue(ocmps_stepper* st, ocmps_mps* m, Workspace* ws, double from, double to, bool forward, ocmps_store* store, int slot,
                 cudaStream_t s) {
  if (store) {
    const Layout& lay = store->lay;
    if (m->lay.L != lay.L || m->lay.D != lay.D || m->lay.cap != lay.cap) return fail(OCMPS_ERR_INVALID, "store/mps shape mismatch");
    if (slot < 0 || slot >= store->nslots) return fail(OCMPS_ERR_INVALID, "slot out of range");
  }
  StepParams hp;
  fill_step_params(st, from, to, forward, store, slot, hp);
  launch_set_step_params(hp, ws->d_params, s);
  g_ocmps_launches += 1;
  const Layout& lay = m->lay;
  auto body = [&]() {
    run_step_body(st, m, ws, s);
    if (store) {
      launch_pack_to_slot(m->ptrs(), lay.offs, m->d_dims, m->d_q, lay.L, lay.D, lay.cap, lay.max_site_elems, ws->d_params, ws->d_status, s);
      g_ocmps_launches += 1;
    }
  };
  if (step_trace_enabled()) {          // plain launches with an event after every phase; prints the phase sums of this step
    CK(cudaStreamSynchronize(s));
    g_trace.on = true;
    g_trace.marks.clear();
    g_trace.mark(TR_START, s);
    body();
    g_trace.mark(TR_OTHER, s);
    g_trace.on = false;
    CK(cudaStreamSynchronize(s));
    double sum[TR_NPHASE] = {0};
    int cnt[TR_NPHASE] = {0};
    for (size_t i = 1; i < g_trace.marks.size(); ++i) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, g_trace.marks[i - 1].second, g_trace.marks[i].second);
      sum[g_trace.marks[i].first] += ms;
      ++cnt[g_trace.marks[i].first];
    }
    float tot = 0.f;
    cudaEventElapsedTime(&tot, g_trace.marks.front().second, g_trace.marks.back().second);
    static const char* names[TR_NPHASE] = {"", "merge_gate", "setup", "svd(gate)", "svd(gauge)", "truncate", "build", "other"};
    fprintf(stderr, "[ocmps step] %.3f ms:", tot);
    for (int p = 1; p < TR_NPHASE; ++p) fprintf(stderr, " %s %dx %.3f |", names[p], cnt[p], sum[p]);
    fprintf(stderr, "\n");
    for (auto& m2 : g_trace.marks) cudaEventDestroy(m2.second);
    g_trace.marks.clear();
    return OCMPS_OK;
  }
  if (!graphs_enabled() || profile_is_on()) { body(); return OCMPS_OK; }   // event timing needs plain launches
  unsigned long long parity = 0;
  for (int j = 0; j < lay.L; ++j) parity |= (unsigned long long)(m->cur[j] & 1) << j;
  auto key = std::make_tuple(st->serial, m->serial, parity, store ? 1 : 0, ws->ctx->qmax.load(), ws->spread_jacobi ? 1 : 0);
  Workspace::StepGraph& g = ws->graphs[key];
  if (g.exec) {
    for (int j = 0; j < lay.L; ++j) m->cur[j] ^= (int)((g.flips >> j) & 1ull);
    m->llim = 0; m->rlim = 2;
    g_ocmps_launches += g.launches;
    CK(cudaGraphLaunch(g.exec, s));
    return OCMPS_OK;
  }
  if (g.seen == 0) {            // first use: plain launches (also sets the function attributes the kernels need)
    g.seen = 1;
    body();
    return OCMPS_OK;
  }
  if (ws->graphs.size() > 64) {   // stale entries (freed MPS buffers): start over
    for (auto& kv : ws->graphs) if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    ws->graphs.clear();
    Workspace::StepGraph& g2 = ws->graphs[key];
    g2.seen = 1;
    body();
    return OCMPS_OK;
  }
  const long long l0 = g_ocmps_launches;
  cudaGraph_t graph = nullptr;
  CK(cudaStreamBeginCapture(s, cudaStreamCaptureModeRelaxed));
  body();
  CK(cudaStreamEndCapture(s, &graph));
  unsigned long long after = 0;
  for (int j = 0; j < lay.L; ++j) after |= (unsigned long long)(m->cur[j] & 1) << j;
  g.flips = parity ^ after;
  g.launches = (int)(g_ocmps_launches - l0);
  CK(cudaGraphInstantiate(&g.exec, graph, 0));
  CK(cudaGraphDestroy(graph));
  CK(cudaGraphLaunch(g.exec, s));
  return OCMPS_OK;
}

// ------------------------------------------------------------------------------------------------
// copies
// ------------------------------------------------------------------------------------------------
int copy_mps_async(ocmps_mps* dst, ocmps_mps* src, cudaStream_t s) {
  if (dst->lay.L != src->lay.L || dst->lay.D != src->lay.D || dst->lay.cap != src->lay.cap)
    return fail(OCMPS_ERR_INVALID, "mps copy: shape mismatch");
  const Layout& lay = src->lay;
  launch_pack_copy(src->ptrs(), dst->arena[0], lay.offs, src->d_dims, lay.L, lay.D, lay.max_site_elems, nullptr, s);
  g_ocmps_launches += 1;
  for (int j = 0; j < lay.L; ++j) dst->cur[j] = 0;
  CK(cudaMemcpyAsync(dst->d_dims, src->d_dims, sizeof(int) * (lay.L + 1), cudaMemcpyDeviceToDevice, s));
  CK(cudaMemcpyAsync(dst->d_q, src->d_q, sizeof(int) * (size_t)(lay.L + 1) * lay.cap, cudaMemcpyDeviceToDevice, s));
  dst->llim = src->llim; dst->rlim = src->rlim;
  return OCMPS_OK;
}

int store_put_async(ocmps_store* st, int slot, ocmps_mps* m, cudaStream_t s) {
  const Layout& lay = st->lay;
  if (m->lay.L != lay.L || m->lay.D != lay.D || m->lay.cap != lay.cap) return fail(OCMPS_ERR_INVALID, "store/mps shape mismatch");
  if (slot < 0 || slot >= st->nslots) return fail(OCMPS_ERR_INVALID, "slot out of range");
  launch_pack_copy(m->ptrs(), st->data + (size_t)slot * lay.total, lay.offs, m->d_dims, lay.L, lay.D, lay.max_site_elems, nullptr, s);
  g_ocmps_launches += 1;
  CK(cudaMemcpyAsync(st->dims + (size_t)slot * (lay.L + 1), m->d_dims, sizeof(int) * (lay.L + 1), cudaMemcpyDeviceToDevice, s));
  CK(cudaMemcpyAsync(st->q + (size_t)slot * (lay.L + 1) * lay.cap, m->d_q, sizeof(int) * (size_t)(lay.L + 1) * lay.cap,
                     cudaMemcpyDeviceToDevice, s));
  return OCMPS_OK;
}

int store_get_async(ocmps_store* st, int slot, ocmps_mps* m, cudaStream_t s) {
  const Layout& lay = st->lay;
  if (m->lay.L != lay.L || m->lay.D != lay.D || m->lay.cap != lay.cap) return fail(OCMPS_ERR_INVALID, "store/mps shape mismatch");
  if (slot < 0 || slot >= st->nslots) return fail(OCMPS_ERR_INVALID, "slot out of range");
  for (int j = 0; j < lay.L; ++j) m->cur[j] = 0;
  const int* dims = st->dims + (size_t)slot * (lay.L + 1);
  launch_unpack_copy(st->data + (size_t)slot * lay.total, m->ptrs(), lay.offs, dims, lay.L, lay.D, lay.max_site_elems, nullptr, s);
  g_ocmps_launches += 1;
  CK(cudaMemcpyAsync(m->d_dims, dims, sizeof(int) * (lay.L + 1), cudaMemcpyDeviceToDevice, s));
  CK(cudaMemcpyAsync(m->d_q, st->q + (size_t)slot * (lay.L + 1) * lay.cap, sizeof(int) * (size_t)(lay.L + 1) * lay.cap,
                     cudaMemcpyDeviceToDevice, s));
  m->llim = 0; m->rlim = 2;
  return OCMPS_OK;
}

// ------------------------------------------------------------------------------------------------
// overlaps
// ------------------------------------------------------------------------------------------------
OvlSide side_of_mps(const ocmps_mps* m) {
  OvlSide s;
  s.base = nullptr; s.slot_stride = 0; s.offs = m->lay.offs; s.ptrs = m->ptrs();
  s.dims = m->d_dims; s.dims_stride = 0; s.use_ptrs = 1; s.slot0 = 0;
  return s;
}
OvlSide side_of_store(const ocmps_store* st, int slot0) {
  OvlSide s;
  s.base = st->data; s.slot_stride = st->lay.total; s.offs = st->lay.offs;
  for (int j = 0; j < OCMPS_MAX_L; ++j) s.ptrs.p[j] = nullptr;
  s.dims = st->dims; s.dims_stride = st->lay.L + 1; s.use_ptrs = 0; s.slot0 = slot0;
  return s;
}

// enqueue <bra_z|ket_z> (or <bra|K|ket>) for z < batch; results land in ws->d_out[z]
int overlaps_async(Workspace* ws, const OvlSide& bra, const Layout& la, const OvlSide& ket, const Layout& lb, int batch,
                   int withK, cudaStream_t s) {
  int rc = ensure_overlap_bufs(ws, batch, la.cap, lb.cap);
  if (rc) return rc;
  const int L = la.L, D = la.D;
  const int nE = withK ? 2 : 1;
  launch_overlap_init(ws->E[0], ws->e_stride, batch, withK, s);
  int cur = 0;
  for (int j = 0; j < L; ++j) {
    launch_overlap_plan(ws->odescs, bra, ket, j, batch, D, withK, ws->E[cur], ws->E[1 - cur], ws->T, ws->e_stride, ws->t_stride, s);
    launch_zgemm(ws->odescs, batch, nE * la.capb[j], D * lb.capb[j + 1], s);
    if (withK) launch_overlap_kfix(ws->T, ws->t_stride, ws->odescs, batch, D, la.capb[j] * D * lb.capb[j + 1], s);
    launch_zgemm(ws->odescs + batch, nE * batch, la.capb[j + 1], lb.capb[j + 1], s);
    cur = 1 - cur;
    g_ocmps_launches += 3 + withK;
  }
  launch_overlap_final(ws->E[cur], ws->e_stride, batch, withK, ws->d_out, s);
  g_ocmps_launches += 2;
  return OCMPS_OK;
}

// ------------------------------------------------------------------------------------------------
// K|psi> with compression (ITensor exactApplyMPO, SURVEY A.6)
// ------------------------------------------------------------------------------------------------
__global__ void copy_bookkeeping_kernel(const int* dims_in, const int* q_in, int qstride_in, int* dims_out, int* q_out,
                                        int qstride_out, int L, int cap_out, int* status) {
  for (int b = blockIdx.x; b <= L; b += gridDim.x) {
    int d = dims_in[b];
    if (d > cap_out) { if (threadIdx.x == 0) atomicOr(status, OCMPS_ST_CAPACITY); d = cap_out; }
    if (threadIdx.x == 0) dims_out[b] = d;
    for (int i = threadIdx.x; i < d; i += blockDim.x) q_out[(size_t)b * qstride_out + i] = q_in[(size_t)b * qstride_in + i];
  }
}

int apply_K_async(ocmps_stepper* st, Workspace* ws, ocmps_mps* in, ocmps_mps* out, cudaStream_t s) {
  const int L = st->L, D = st->D;
  const int cap2 = 2 * st->cap;
  if ((long long)cap2 * D > NV_MAX) return fail(OCMPS_ERR_INVALID, "apply_K: 2*chi_cap*D exceeds 2048");
  if (!ws->big) {
    int rc = alloc_mps(st->ctx, L, D, st->cap, &ws->big, 2);
    if (rc) return rc;
    rc = alloc_ws(st->ctx, L, D, cap2, false, &ws->bigws);
    if (rc) return rc;
    ws->bigws->db.status = ws->d_status;            // what its kernels flag is reported with the owning workspace
    ws->bigws->db2.status = ws->d_status;
  }
  ocmps_mps* big = ws->big;
  Workspace* bw = ws->bigws;
  bw->spread_jacobi = ws->spread_jacobi;
  const Layout& lb = big->lay;
  if (L == 1) return fail(OCMPS_ERR_INVALID, "apply_K needs L >= 2");
  for (int j = 0; j < L; ++j) big->cur[j] = 0;
  for (int j = 0; j < L; ++j) {
    launch_applyK_expand(in->site(j), big->site(j), in->dim(j), in->dim(j + 1), in->q(j), in->q(j + 1), big->dim(j), big->dim(j + 1),
                         big->q(j), big->q(j + 1), D, j, L, lb.capb[j] * D * lb.capb[j + 1], s);
  }
  g_ocmps_launches += L;
  // left-canonicalise the exact product (numerical-rank drops only)
  TruncParams tpl{MIN_CUT, MAX_M, 1, 1, 0, 0};
  for (int b = 1; b <= L - 1; ++b) {
    const int j = b - 1, jn = b;
    DecompArgs a;
    a.D = D; a.kind = DK_ORTH_LEFT;
    a.dimNew = big->dim(b); a.qNew = big->q(b); a.partner = bw->cbuf;
    a.dimL = big->dim(b - 1); a.dimR = big->dim(b); a.qL = big->q(b - 1); a.qR = big->q(b);
    a.X = big->site(j); a.iso = big->other(j);
    a.nb_in = big->site(jn); a.nb_out = big->other(jn); a.dimNb = big->dim(b + 1);
    a.qNb = fused_push_enabled() ? big->q(b + 1) : nullptr;
    tpl.cap = lb.capb[b];
    run_decomp(bw, a, tpl, lb.capb[b], lb.capb[b - 1], lb.capb[b], s);
    if (!a.qNb) launch_zgemm(bw->db.descs + 1, 1, lb.capb[b], D * lb.capb[b + 1], s);
    big->cur[j] ^= 1; big->cur[jn] ^= 1;
    g_ocmps_launches += 1;
  }
  // right-to-left compression with the stepper's Cutoff / Maxm (exactApplyMPO defaults: Cutoff 1e-13)
  TruncParams tpr{st->has_cutoff ? st->cutoff : 1e-13, st->has_maxm ? st->maxm : MAX_M, 1, st->rel_cutoff, 0, 0};
  for (int b = L - 1; b >= 1; --b) {
    const int j = b, jn = b - 1;
    DecompArgs a;
    a.D = D; a.kind = DK_ORTH_RIGHT;
    a.dimNew = big->dim(b); a.qNew = big->q(b); a.partner = bw->cbuf;
    a.dimL = big->dim(b); a.dimR = big->dim(b + 1); a.qL = big->q(b); a.qR = big->q(b + 1);
    a.X = big->site(j); a.iso = big->other(j);
    a.nb_in = big->site(jn); a.nb_out = big->other(jn); a.dimNb = big->dim(b - 1);
    a.qNb = fused_push_enabled() ? big->q(b - 1) : nullptr;
    tpr.cap = std::min(lb.capb[b], out->lay.capb[b]);
    run_decomp(bw, a, tpr, lb.capb[b], lb.capb[b + 1], tpr.cap, s);
    if (!a.qNb) launch_zgemm(bw->db.descs + 1, 1, lb.capb[b - 1] * D, lb.capb[b], s);
    big->cur[j] ^= 1; big->cur[jn] ^= 1;
    g_ocmps_launches += 1;
  }
  // compact into the chi_cap layout
  for (int j = 0; j < L; ++j) out->cur[j] = 0;
  copy_bookkeeping_kernel<<<L + 1, 128, 0, s>>>(big->d_dims, big->d_q, lb.cap, out->d_dims, out->d_q, out->lay.cap, L, out->lay.cap,
                                               ws->d_status);
  launch_pack_copy(big->ptrs(), out->arena[0], out->lay.offs, out->d_dims, L, D, out->lay.max_site_elems, ws->d_status, s);
  g_ocmps_launches += 2;
  out->llim = 0; out->rlim = 2;
  return OCMPS_OK;
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

const char* ocmps_last_error(void) { return g_err.c_str(); }
int ocmps_version(void) { return 100; }
long long ocmps_launch_count(void) { return g_ocmps_launches; }
int ocmps_profile_enable(int on) { profile_enable(on != 0); return OCMPS_OK; }
int ocmps_profile_read(double* out4) { if (!out4) return fail(OCMPS_ERR_INVALID, "null argument"); profile_read(out4); return OCMPS_OK; }

int ocmps_ctx_create(int device, ocmps_ctx** out) {
  if (!out) return fail(OCMPS_ERR_INVALID, "null out");
  // One hardware queue per chain stream where possible (default 8: chains on aliased queues serialise).  Only effective if
  // this is the first CUDA call of the process; a value set by the user is kept.
  setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) return fail(OCMPS_ERR_CUDA, "no CUDA device available (libocmps has no CPU fallback)");
  if (device < 0 || device >= n) return fail(OCMPS_ERR_INVALID, "device index out of range");
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return fail(OCMPS_ERR_CUDA, "libocmps is built for sm_100a (Blackwell) only");
  ocmps_ctx* c = new ocmps_ctx();
  c->dev = device;
  CK(cudaStreamCreateWithFlags(&c->stream0, cudaStreamNonBlocking));
  *out = c;
  return OCMPS_OK;
}

int ocmps_ctx_destroy(ocmps_ctx* ctx) {
  if (!ctx) return OCMPS_OK;
  cudaSetDevice(ctx->dev);
  cudaDeviceSynchronize();
  for (Workspace* w : ctx->pool) free_ws(w);
  if (ctx->t0) { cudaEventDestroy(ctx->t0); cudaEventDestroy(ctx->t1); }
  cudaStreamDestroy(ctx->stream0);
  delete ctx;
  return OCMPS_OK;
}

// Device-side stopwatch for bench.py: two CUDA events on the context's own stream.  Every entry point is synchronous, so the
// stream is idle when either event is recorded and the pair brackets all device work enqueued in between.
int ocmps_timer_start(ocmps_ctx* ctx) {
  if (!ctx) return fail(OCMPS_ERR_INVALID, "null argument");
  CK(cudaSetDevice(ctx->dev));
  if (!ctx->t0) { CK(cudaEventCreate(&ctx->t0)); CK(cudaEventCreate(&ctx->t1)); }
  CK(cudaEventRecord(ctx->t0, ctx->stream0));
  return OCMPS_OK;
}
int ocmps_timer_stop(ocmps_ctx* ctx, double* ms) {
  if (!ctx || !ms || !ctx->t0) return fail(OCMPS_ERR_INVALID, "timer not started");
  CK(cudaSetDevice(ctx->dev));
  CK(cudaEventRecord(ctx->t1, ctx->stream0));
  CK(cudaEventSynchronize(ctx->t1));
  float f = 0.f;
  CK(cudaEventElapsedTime(&f, ctx->t0, ctx->t1));
  *ms = (double)f;
  return OCMPS_OK;
}

// Releases the idle workspaces of the pool (streams, scratch, Hessian rings, step graphs).  They are re-created on demand;
// a long-lived process calls this between workloads of different shapes (bench.py does, before the chi=150 batch).
int ocmps_ctx_trim(ocmps_ctx* ctx) {
  if (!ctx) return fail(OCMPS_ERR_INVALID, "null argument");
  CK(cudaSetDevice(ctx->dev));
  std::vector<Workspace*> idle;
  {
    std::lock_guard<std::mutex> lock(ctx->mu);
    std::vector<Workspace*> keep;
    for (Workspace* w : ctx->pool) (w->busy ? keep : idle).push_back(w);
    ctx->pool.swap(keep);
  }
  for (Workspace* w : idle) { cudaStreamSynchronize(w->stream); if (w->ovl) cudaStreamSynchronize(w->ovl); free_ws(w); }
  return OCMPS_OK;
}

int ocmps_ctx_synchronize(ocmps_ctx* ctx) {
  if (!ctx) return fail(OCMPS_ERR_INVALID, "null argument");
  CK(cudaSetDevice(ctx->dev));
  CK(cudaDeviceSynchronize());      // every entry point is synchronous, so this only matters next to foreign CUDA work
  return OCMPS_OK;
}

// ---- MPS ----
int ocmps_mps_create(ocmps_ctx* ctx, int L, int D, int chi_cap, ocmps_mps** out) {
  if (!ctx || !out) return fail(OCMPS_ERR_INVALID, "null argument");
  return alloc_mps(ctx, L, D, chi_cap, out);
}
int ocmps_mps_destroy(ocmps_mps* mps) {
  if (mps) { cudaSetDevice(mps->ctx->dev); free_mps(mps); }
  return OCMPS_OK;
}

int ocmps_mps_upload(ocmps_mps* m, const int* bond_dims, const int* charges, const double* tensors, int llim, int rlim) {
  if (!m || !bond_dims || !charges || !tensors) return fail(OCMPS_ERR_INVALID, "null argument");
  const Layout& lay = m->lay;
  CK(cudaSetDevice(m->ctx->dev));
  for (int b = 0; b <= lay.L; ++b)
    if (bond_dims[b] < 1 || bond_dims[b] > lay.capb[b])
      return fail(OCMPS_ERR_CAPACITY, "upload: bond dimension " + std::to_string(bond_dims[b]) + " at bond " + std::to_string(b) +
                                          " exceeds capacity " + std::to_string(lay.capb[b]));
  if (bond_dims[0] != 1 || bond_dims[lay.L] != 1) return fail(OCMPS_ERR_INVALID, "upload: boundary bonds must have dimension 1");
  // The engine keeps bond charges sorted ascending (the block bookkeeping relies on it); a permutation of a
  // bond index is a gauge choice, so unsorted labels are sorted here, stably, together with the tensors.
  std::vector<std::vector<int>> perm(lay.L + 1);
  {
    size_t qo = 0;
    for (int b = 0; b <= lay.L; ++b) {
      const int nb = bond_dims[b];
      for (int i = 0; i < nb; ++i)
        if (charges[qo + i] < 0 || charges[qo + i] >= OCMPS_MAX_Q) return fail(OCMPS_ERR_INVALID, "upload: charge outside [0,256)");
      perm[b].resize(nb);
      for (int i = 0; i < nb; ++i) perm[b][i] = i;
      const int* qb = charges + qo;
      for (int i = 0; i < nb; ++i) {
        int seen = m->ctx->qmax.load();
        while (qb[i] > seen && !m->ctx->qmax.compare_exchange_weak(seen, qb[i])) {}
      }
      std::stable_sort(perm[b].begin(), perm[b].end(), [qb](int x, int y) { return qb[x] < qb[y]; });
      std::vector<int> sorted(nb);
      for (int i = 0; i < nb; ++i) sorted[i] = qb[perm[b][i]];
      CK(cudaMemcpy(m->q(b), sorted.data(), sizeof(int) * nb, cudaMemcpyHostToDevice));
      qo += nb;
    }
  }
  size_t off = 0;
  std::vector<zc> tmp;
  const zc* src = reinterpret_cast<const zc*>(tensors);
  for (int j = 0; j < lay.L; ++j) {
    m->cur[j] = 0;
    const int cl = bond_dims[j], cr = bond_dims[j + 1], D = lay.D;
    const size_t n = (size_t)cl * D * cr;
    tmp.resize(n);
    for (int l = 0; l < cl; ++l)
      for (int sI = 0; sI < D; ++sI) {
        const zc* in = src + off + ((size_t)perm[j][l] * D + sI) * cr;
        zc* out = tmp.data() + ((size_t)l * D + sI) * cr;
        for (int r = 0; r < cr; ++r) out[r] = in[perm[j + 1][r]];
      }
    CK(cudaMemcpy(m->site(j), tmp.data(), sizeof(cplx) * n, cudaMemcpyHostToDevice));
    off += n;
  }
  CK(cudaMemcpy(m->d_dims, bond_dims, sizeof(int) * (lay.L + 1), cudaMemcpyHostToDevice));
  m->llim = llim; m->rlim = rlim;
  return OCMPS_OK;
}

int ocmps_mps_bond_dims(ocmps_mps* m, int* bond_dims) {
  if (!m || !bond_dims) return fail(OCMPS_ERR_INVALID, "null argument");
  CK(cudaSetDevice(m->ctx->dev));
  CK(cudaMemcpy(bond_dims, m->d_dims, sizeof(int) * (m->lay.L + 1), cudaMemcpyDeviceToHost));
  return OCMPS_OK;
}

int ocmps_mps_sizes(ocmps_mps* m, long long* n_elems, long long* n_charges) {
  std::vector<int> d(m->lay.L + 1);
  int rc = ocmps_mps_bond_dims(m, d.data());
  if (rc) return rc;
  long long ne = 0, nq = 0;
  for (int j = 0; j < m->lay.L; ++j) ne += (long long)d[j] * m->lay.D * d[j + 1];
  for (int b = 0; b <= m->lay.L; ++b) nq += d[b];
  if (n_elems) *n_elems = ne;
  if (n_charges) *n_charges = nq;
  return OCMPS_OK;
}

int ocmps_mps_download(ocmps_mps* m, int* bond_dims, int* charges, double* tensors, int* llim, int* rlim) {
  if (!m || !bond_dims) return fail(OCMPS_ERR_INVALID, "null argument");
  int rc = ocmps_mps_bond_dims(m, bond_dims);
  if (rc) return rc;
  const Layout& lay = m->lay;
  size_t off = 0, qoff = 0;
  for (int j = 0; j < lay.L; ++j) {
    size_t n = (size_t)bond_dims[j] * lay.D * bond_dims[j + 1];
    if (tensors) CK(cudaMemcpy(tensors + 2 * off, m->site(j), sizeof(cplx) * n, cudaMemcpyDeviceToHost));
    off += n;
  }
  for (int b = 0; b <= lay.L; ++b) {
    if (charges) CK(cudaMemcpy(charges + qoff, m->q(b), sizeof(int) * bond_dims[b], cudaMemcpyDeviceToHost));
    qoff += bond_dims[b];
  }
  if (llim) *llim = m->llim;
  if (rlim) *rlim = m->rlim;
  return OCMPS_OK;
}

int ocmps_mps_copy(ocmps_mps* dst, ocmps_mps* src) {
  if (!dst || !src) return fail(OCMPS_ERR_INVALID, "null argument");
  CK(cudaSetDevice(src->ctx->dev));
  cudaStream_t s = nullptr;                   // a stream of its own: concurrent copies of different MPS do not queue up
  CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  int rc = copy_mps_async(dst, src, s);
  cudaError_t e = cudaStreamSynchronize(s);
  cudaStreamDestroy(s);
  if (rc) return rc;
  CK(e);
  return OCMPS_OK;
}

// psi.position(1) (ITensor MPS::position via orthMPS, SURVEY A.4) from the orthogonality limits the state was uploaded with:
// block-SVD gauge moves from site rlim-1 down to site 2 (Cutoff 1e-16, Maxm 5000: numerical-rank drops only), S.V pushed to the
// left.  Every other entry point that needs a gauge (step, sweeps, K|psi>) requires the centre at site 1 and says so; this is
// the call that establishes it for a state in any other gauge (llim = 0, rlim = L+1: nothing is assumed orthogonal).
int ocmps_mps_position1(ocmps_mps* m) {
  if (!m) return fail(OCMPS_ERR_INVALID, "null argument");
  const Layout& lay = m->lay;
  const int L = lay.L, D = lay.D;
  if (m->llim != 0) {
    // sites left of the centre are left-orthonormal by assumption; moving the centre to site 1 re-gauges them all
    if (m->llim < 0 || m->llim > L - 1) return fail(OCMPS_ERR_INVALID, "position: bad orthogonality limits");
  }
  int rlim = std::min(std::max(m->rlim, m->llim + 2), L + 1);
  if (rlim <= 2) { m->llim = 0; m->rlim = 2; return OCMPS_OK; }
  CK(cudaSetDevice(m->ctx->dev));
  WsLease lease;
  int rc = lease.acquire(m->ctx, L, D, lay.cap, 1);
  if (rc) return rc;
  Workspace* ws = lease[0];
  cudaStream_t s = ws->stream;
  TruncParams tpo{MIN_CUT, MAX_M, 1, 0, 0, 0};
  for (int b = rlim - 2; b >= 1; --b) {          // bond b joins sites b and b+1 (1-based): SVD of site b+1, U.S pushed into site b
    const int j = b, jn = b - 1;
    DecompArgs a;
    a.D = D; a.kind = DK_ORTH_RIGHT;
    a.dimNew = m->dim(b); a.qNew = m->q(b); a.partner = ws->cbuf;
    a.dimL = m->dim(b); a.dimR = m->dim(b + 1); a.qL = m->q(b); a.qR = m->q(b + 1);
    a.X = m->site(j); a.iso = m->other(j);
    a.nb_in = m->site(jn); a.nb_out = m->other(jn); a.dimNb = m->dim(b - 1);
    a.qNb = fused_push_enabled() ? m->q(b - 1) : nullptr;
    tpo.cap = lay.capb[b];
    run_decomp(ws, a, tpo, lay.capb[b], lay.capb[b + 1], lay.capb[b], s);
    if (!a.qNb) { launch_zgemm(ws->db.descs + 1, 1, lay.capb[b - 1] * D, lay.capb[b], s); g_ocmps_launches += 1; }
    m->cur[j] ^= 1; m->cur[jn] ^= 1;
  }
  m->llim = 0; m->rlim = 2;
  return lease.finish();
}

int ocmps_mps_norm(ocmps_mps* m, double* out) {
  if (!m || !out) return fail(OCMPS_ERR_INVALID, "null argument");
  if (m->llim + 2 != m->rlim) return fail(OCMPS_ERR_INVALID, "norm: MPS has no single orthogonality centre");
  CK(cudaSetDevice(m->ctx->dev));
  WsLease lease;
  int rc = lease.acquire(m->ctx, m->lay.L, m->lay.D, m->lay.cap, 1);
  if (rc) return rc;
  Workspace* ws = lease[0];
  const int j = m->llim;   // 0-based centre
  launch_norm_only(m->site(j), m->dim(j), m->dim(j + 1), m->lay.D, ws->db.partial, ws->d_norm, 0, ws->stream);
  g_ocmps_launches += 2;
  CK(cudaMemcpyAsync(out, ws->d_norm, sizeof(double), cudaMemcpyDeviceToHost, ws->stream));
  return lease.finish();
}

static int overlap_impl(ocmps_mps* a, ocmps_mps* b, double* re_im, int withK) {
  if (!a || !b || !re_im) return fail(OCMPS_ERR_INVALID, "null argument");
  if (a->lay.L != b->lay.L || a->lay.D != b->lay.D) return fail(OCMPS_ERR_INVALID, "overlap: shape mismatch");
  CK(cudaSetDevice(a->ctx->dev));
  WsLease lease;
  int rc = lease.acquire(a->ctx, a->lay.L, a->lay.D, a->lay.cap, 1);
  if (rc) return rc;
  Workspace* ws = lease[0];
  rc = overlaps_async(ws, side_of_mps(a), a->lay, side_of_mps(b), b->lay, 1, withK, ws->stream);
  if (rc) return rc;
  CK(cudaMemcpyAsync(re_im, ws->d_out, sizeof(cplx), cudaMemcpyDeviceToHost, ws->stream));
  return lease.finish();
}
int ocmps_overlap(ocmps_mps* a, ocmps_mps* b, double* re_im) { return overlap_impl(a, b, re_im, 0); }
int ocmps_overlap_K(ocmps_mps* a, ocmps_mps* b, double* re_im) { return overlap_impl(a, b, re_im, 1); }

// ---- stepper ----
int ocmps_stepper_set_tstep(ocmps_stepper* st, double tstep) {
  if (!st) return fail(OCMPS_ERR_INVALID, "null argument");
  CK(cudaSetDevice(st->ctx->dev));
  CK(cudaDeviceSynchronize());
  st->tstep = tstep;
  const int n = st->D * st->D;
  for (int dir = 0; dir < 2; ++dir) {
    st->h_G[dir] = bond_gate(st->D, st->J, dir == 0 ? tstep : -tstep, st->imag);
    if (!st->d_G[dir]) CK(cudaMalloc(&st->d_G[dir], sizeof(cplx) * n * n));
    CK(cudaMemcpy(st->d_G[dir], st->h_G[dir].data(), sizeof(cplx) * n * n, cudaMemcpyHostToDevice));
  }
  return OCMPS_OK;
}

int ocmps_stepper_create(ocmps_ctx* ctx, int L, int D, double J, double tstep, double cutoff, int maxm, int chi_cap, int rel_cutoff,
                         ocmps_stepper** out) {
  if (!ctx || !out) return fail(OCMPS_ERR_INVALID, "null argument");
  if (L < 2 || L > OCMPS_MAX_L) return fail(OCMPS_ERR_INVALID, "L out of range [2,64]");
  if (D < 2 || D > OCMPS_MAX_D) return fail(OCMPS_ERR_INVALID, "D out of range [2,8]");
  if (chi_cap < 1 || (long long)chi_cap * D > NV_MAX) return fail(OCMPS_ERR_INVALID, "chi_cap*D exceeds 2048");
  ocmps_stepper* st = new ocmps_stepper();
  st->ctx = ctx; st->L = L; st->D = D; st->J = J; st->cap = chi_cap;
  st->has_cutoff = cutoff >= 0.0; st->cutoff = st->has_cutoff ? cutoff : MIN_CUT;
  st->has_maxm = maxm > 0; st->maxm = st->has_maxm ? maxm : MAX_M;
  st->rel_cutoff = rel_cutoff ? 1 : 0;
  st->ops = build_schedule(L);
  { static std::atomic<long long> next_serial{1}; st->serial = next_serial++; }
  int rc = ocmps_stepper_set_tstep(st, tstep);
  if (rc) { delete st; return rc; }
  *out = st;
  return OCMPS_OK;
}

int ocmps_stepper_destroy(ocmps_stepper* st) {
  if (!st) return OCMPS_OK;
  cudaSetDevice(st->ctx->dev);
  cudaDeviceSynchronize();
  cudaFree(st->d_G[0]); cudaFree(st->d_G[1]);
  delete st;
  return OCMPS_OK;
}

double ocmps_stepper_get_tstep(ocmps_stepper* st) { return st ? st->tstep : 0.0; }

int ocmps_stepper_schedule(ocmps_stepper* st, int* quads, int cap) {
  if (!st) return fail(OCMPS_ERR_INVALID, "null argument");
  int n = (int)st->ops.size();
  for (int i = 0; i < n && i < cap; ++i) {
    quads[4 * i] = st->ops[i].kind; quads[4 * i + 1] = st->ops[i].a; quads[4 * i + 2] = st->ops[i].b; quads[4 * i + 3] = st->ops[i].c;
  }
  return n;
}

int ocmps_stepper_gate(ocmps_stepper* st, int forward, double* out) {
  if (!st || !out) return fail(OCMPS_ERR_INVALID, "null argument");
  const std::vector<zc>& g = st->h_G[forward ? 0 : 1];
  memcpy(out, g.data(), sizeof(zc) * g.size());
  return OCMPS_OK;
}

static int check_shapes(ocmps_stepper* st, const Layout& lay, const char* what) {
  if (lay.L != st->L || lay.D != st->D || lay.cap != st->cap)
    return fail(OCMPS_ERR_INVALID, std::string(what) + ": MPS/store shape (L, D, chi_cap) differs from the stepper's");
  return OCMPS_OK;
}

int ocmps_step(ocmps_stepper* st, ocmps_mps* psi, double from, double to, int forward) {
  if (!st || !psi) return fail(OCMPS_ERR_INVALID, "null argument");
  int rc = check_shapes(st, psi->lay, "step");
  if (rc) return rc;
  if (psi->llim != 0 || psi->rlim != 2) return fail(OCMPS_ERR_INVALID, "step: orthogonality centre must be at site 1");
  CK(cudaSetDevice(st->ctx->dev));
  WsLease lease;
  rc = lease.acquire(st->ctx, st->L, st->D, st->cap, 1);
  if (rc) return rc;
  Workspace* ws = lease[0];
  rc = step_enqueue(st, psi, ws, from, to, forward != 0, nullptr, 0, ws->stream);
  if (rc) { cudaStreamSynchronize(ws->stream); return rc; }
  return lease.finish();
}

int ocmps_debug_jacobi(unsigned long long* out, int reset) { cudaDeviceSynchronize(); debug_jacobi_counters(out, reset != 0); return 0; }
// out[0]: charge blocks whose Jacobi stage ran spread over a thread-block cluster (row-block path), out[1]: their sweeps
int ocmps_debug_row_cluster(unsigned long long* out2, int reset) { cudaDeviceSynchronize(); debug_row_cluster_counters(out2, reset != 0); return 0; }

// development aid: run ops [op_begin, op_end) of one step (not part of include/ocmps.h)
int ocmps_debug_run_ops(ocmps_stepper* st, ocmps_mps* psi, double from, double to, int forward, int op_begin, int op_end) {
  CK(cudaSetDevice(st->ctx->dev));
  WsLease lease;
  int rc = lease.acquire(st->ctx, st->L, st->D, st->cap, 1);
  if (rc) return rc;
  Workspace* ws = lease[0];
  { StepParams hp; fill_step_params(st, from, to, forward != 0, nullptr, 0, hp); launch_set_step_params(hp, ws->d_params, ws->stream); }
  run_step_body(st, psi, ws, ws->stream, op_begin, op_end);
  return lease.finish();
}

int ocmps_apply_K(ocmps_stepper* st, ocmps_mps* in, ocmps_mps* out) {
  if (!st || !in || !out) return fail(OCMPS_ERR_INVALID, "null argument");
  int rc = check_shapes(st, in->lay, "apply_K");
  if (rc) return rc;
  rc = check_shapes(st, out->lay, "apply_K");
  if (rc) return rc;
  CK(cudaSetDevice(st->ctx->dev));
  WsLease lease;
  rc = lease.acquire(st->ctx, st->L, st->D, st->cap, 1);
  if (rc) return rc;
  Workspace* ws = lease[0];
  rc = apply_K_async(st, ws, in, out, ws->stream);
  if (rc) { cudaStreamSynchronize(ws->stream); return rc; }
  return lease.finish();
}

// ---- stores ----
int ocmps_store_create(ocmps_ctx* ctx, int L, int D, int chi_cap, int nslots, ocmps_store** out) {
  if (!ctx || !out || nslots < 1) return fail(OCMPS_ERR_INVALID, "bad argument");
  if (L < 1 || L > OCMPS_MAX_L || D < 2 || D > OCMPS_MAX_D || chi_cap < 1) return fail(OCMPS_ERR_INVALID, "bad shape");
  ocmps_store* s = new ocmps_store();
  s->ctx = ctx; s->nslots = nslots;
  s->lay.init(L, D, chi_cap);
  CK(cudaSetDevice(ctx->dev));
  CK(cudaMalloc(&s->data, sizeof(cplx) * (size_t)s->lay.total * nslots));
  CK(cudaMalloc(&s->dims, sizeof(int) * (size_t)(L + 1) * nslots));
  CK(cudaMalloc(&s->q, sizeof(int) * (size_t)(L + 1) * chi_cap * nslots));
  CK(cudaMemset(s->dims, 0, sizeof(int) * (size_t)(L + 1) * nslots));
  CK(cudaStreamSynchronize(cudaStreamLegacy));
  *out = s;
  return OCMPS_OK;
}
int ocmps_store_destroy(ocmps_store* s) {
  if (!s) return OCMPS_OK;
  cudaSetDevice(s->ctx->dev);
  cudaDeviceSynchronize();
  cudaFree(s->data); cudaFree(s->dims); cudaFree(s->q);
  delete s;
  return OCMPS_OK;
}
int ocmps_store_get(ocmps_store* store, int slot, ocmps_mps* out) {
  if (!store || !out) return fail(OCMPS_ERR_INVALID, "null argument");
  CK(cudaSetDevice(store->ctx->dev));
  int rc = store_get_async(store, slot, out, store->ctx->stream0);
  if (rc) return rc;
  CK(cudaStreamSynchronize(store->ctx->stream0));
  return OCMPS_OK;
}
int ocmps_store_put(ocmps_store* store, int slot, ocmps_mps* in) {
  if (!store || !in) return fail(OCMPS_ERR_INVALID, "null argument");
  CK(cudaSetDevice(store->ctx->dev));
  int rc = store_put_async(store, slot, in, store->ctx->stream0);
  if (rc) return rc;
  CK(cudaStreamSynchronize(store->ctx->stream0));
  return OCMPS_OK;
}
int ocmps_store_bond_dims(ocmps_store* store, int* out) {
  if (!store || !out) return fail(OCMPS_ERR_INVALID, "null argument");
  CK(cudaSetDevice(store->ctx->dev));
  CK(cudaMemcpy(out, store->dims, sizeof(int) * (size_t)(store->lay.L + 1) * store->nslots, cudaMemcpyDeviceToHost));
  return OCMPS_OK;
}

// ---- sweeps ----
static int sweep_enqueue_init(ocmps_stepper* st, Workspace* ws, ocmps_mps* start, ocmps_store* store, int slot) {
  int rc = copy_mps_async(ws->work, start, ws->stream);
  if (rc) return rc;
  ws->work->llim = 0; ws->work->rlim = 2;
  if (store) return store_put_async(store, slot, ws->work, ws->stream);
  return OCMPS_OK;
}

static int sweep_args_ok(ocmps_stepper* st, ocmps_mps* start, const double* u, int Nt, ocmps_store* store) {
  if (!st || !start || !u || Nt < 2) return fail(OCMPS_ERR_INVALID, "bad argument");
  int rc = check_shapes(st, start->lay, "sweep");
  if (rc) return rc;
  if (start->llim != 0 || start->rlim != 2) return fail(OCMPS_ERR_INVALID, "sweep: orthogonality centre must be at site 1");
  if (store) {
    rc = check_shapes(st, store->lay, "sweep");
    if (rc) return rc;
    if (store->nslots < Nt) return fail(OCMPS_ERR_INVALID, "sweep: store has fewer slots than Nt");
  }
  return OCMPS_OK;
}

int ocmps_forward_sweep(ocmps_stepper* st, ocmps_mps* psi_init, const double* u, int Nt, ocmps_store* store) {
  int rc = sweep_args_ok(st, psi_init, u, Nt, store);
  if (rc) return rc;
  if (!store) return fail(OCMPS_ERR_INVALID, "null store");
  CK(cudaSetDevice(st->ctx->dev));
  WsLease lease;
  rc = lease.acquire(st->ctx, st->L, st->D, st->cap, 1);
  if (rc) return rc;
  Workspace* ws = lease[0];
  rc = sweep_enqueue_init(st, ws, psi_init, store, 0);
  for (int i = 0; i < Nt - 1 && !rc; ++i)
    rc = step_enqueue(st, ws->work, ws, u[i], u[i + 1], true, store, i + 1, ws->stream);
  if (rc) { cudaStreamSynchronize(ws->stream); return rc; }
  return lease.finish();
}

int ocmps_backward_sweep(ocmps_stepper* st, ocmps_mps* psi_target, const double* u, int Nt, ocmps_store* store) {
  int rc = sweep_args_ok(st, psi_target, u, Nt, store);
  if (rc) return rc;
  if (!store) return fail(OCMPS_ERR_INVALID, "null store");
  CK(cudaSetDevice(st->ctx->dev));
  WsLease lease;
  rc = lease.acquire(st->ctx, st->L, st->D, st->cap, 1);
  if (rc) return rc;
  Workspace* ws = lease[0];
  rc = sweep_enqueue_init(st, ws, psi_target, store, Nt - 1);
  for (int i = Nt - 1; i > 0 && !rc; --i)
    rc = step_enqueue(st, ws->work, ws, u[i], u[i - 1], false, store, i - 1, ws->stream);
  if (rc) { cudaStreamSynchronize(ws->stream); return rc; }
  return lease.finish();
}

int ocmps_sweep_pair(ocmps_stepper* st, ocmps_mps* psi_init, ocmps_mps* psi_target, const double* u, int Nt, ocmps_store* psi_store,
                     ocmps_store* xi_store) {
  int rc = sweep_args_ok(st, psi_init, u, Nt, psi_store);
  if (rc) return rc;
  rc = sweep_args_ok(st, psi_target, u, Nt, xi_store);
  if (rc) return rc;
  if (!psi_store || !xi_store) return fail(OCMPS_ERR_INVALID, "null store");
  CK(cudaSetDevice(st->ctx->dev));
  WsLease lease;
  rc = lease.acquire(st->ctx, st->L, st->D, st->cap, 2);
  if (rc) return rc;
  Workspace *wa = lease[0], *wb = lease[1];
  rc = sweep_enqueue_init(st, wa, psi_init, psi_store, 0);
  if (!rc) rc = sweep_enqueue_init(st, wb, psi_target, xi_store, Nt - 1);
  for (int k = 0; k < Nt - 1 && !rc; ++k) {      // interleave the two chains so both streams stay fed
    rc = step_enqueue(st, wa->work, wa, u[k], u[k + 1], true, psi_store, k + 1, wa->stream);
    if (rc) break;
    const int i = Nt - 1 - k;
    rc = step_enqueue(st, wb->work, wb, u[i], u[i - 1], false, xi_store, i - 1, wb->stream);
  }
  if (rc) { cudaStreamSynchronize(wa->stream); cudaStreamSynchronize(wb->stream); return rc; }
  return lease.finish();
}

int ocmps_sweep_batch(ocmps_stepper* st, int nchains, ocmps_mps** starts, const int* forward, const double* u, int Nt,
                      ocmps_store** stores) {
  if (!st || !starts || !forward || !u || !stores || nchains < 1) return fail(OCMPS_ERR_INVALID, "bad argument");
  int rc = OCMPS_OK;
  for (int c = 0; c < nchains; ++c) {
    rc = sweep_args_ok(st, starts[c], u + (size_t)c * Nt, Nt, stores[c]);
    if (rc) return rc;
    if (!stores[c]) return fail(OCMPS_ERR_INVALID, "null store");
  }
  CK(cudaSetDevice(st->ctx->dev));
  WsLease lease;
  rc = lease.acquire(st->ctx, st->L, st->D, st->cap, nchains);
  if (rc) return rc;
  const std::vector<Workspace*>& wss = lease.ws;
  for (int c = 0; c < nchains && !rc; ++c)
    rc = sweep_enqueue_init(st, wss[c], starts[c], stores[c], forward[c] ? 0 : Nt - 1);
  for (int k = 0; k < Nt - 1 && !rc; ++k) {          // all chains advance in lock step so every stream stays fed
    for (int c = 0; c < nchains; ++c) {
      const double* uc = u + (size_t)c * Nt;
      Workspace* ws = wss[c];
      if (forward[c]) {
        rc = step_enqueue(st, ws->work, ws, uc[k], uc[k + 1], true, stores[c], k + 1, ws->stream);
      } else {
        const int i = Nt - 1 - k;
        rc = step_enqueue(st, ws->work, ws, uc[i], uc[i - 1], false, stores[c], i - 1, ws->stream);
      }
      if (rc) break;
    }
  }
  if (rc) { for (Workspace* w : wss) cudaStreamSynchronize(w->stream); return rc; }
  return lease.finish();
}

int ocmps_backward_sweep_divT(ocmps_stepper* st, ocmps_mps* psi_target, const double* u, int Nt, ocmps_store* psi_store,
                              double* divT) {
  int rc = sweep_args_ok(st, psi_target, u, Nt, psi_store);
  if (rc) return rc;
  if (!psi_store || !divT) return fail(OCMPS_ERR_INVALID, "null argument");
  CK(cudaSetDevice(st->ctx->dev));
  WsLease lease;
  rc = lease.acquire(st->ctx, st->L, st->D, st->cap, 1);
  if (rc) return rc;
  Workspace* ws = lease[0];
  if (ws->div_cap < Nt) {                       // kept with the workspace: no allocation per call
    CK(cudaStreamSynchronize(ws->stream));
    cudaFree(ws->d_div); ws->d_div = nullptr; ws->div_cap = 0;
    CK(cudaMalloc(&ws->d_div, sizeof(cplx) * Nt));
    ws->div_cap = Nt;
  }
  cplx* d_div = ws->d_div;
  rc = sweep_enqueue_init(st, ws, psi_target, nullptr, 0);
  for (int i = Nt - 1; i >= 0 && !rc; --i) {
    rc = overlaps_async(ws, side_of_mps(ws->work), ws->work->lay, side_of_store(psi_store, i), psi_store->lay, 1, 1, ws->stream);
    if (rc) break;
    if (cudaMemcpyAsync(d_div + i, ws->d_out, sizeof(cplx), cudaMemcpyDeviceToDevice, ws->stream) != cudaSuccess) {
      rc = fail(OCMPS_ERR_CUDA, "cudaMemcpyAsync failed"); break;
    }
    if (i > 0) rc = step_enqueue(st, ws->work, ws, u[i], u[i - 1], false, nullptr, 0, ws->stream);
  }
  if (!rc && cudaMemcpyAsync(divT, d_div, sizeof(cplx) * Nt, cudaMemcpyDeviceToHost, ws->stream) != cudaSuccess)
    rc = fail(OCMPS_ERR_CUDA, "cudaMemcpyAsync failed");
  if (rc) { cudaStreamSynchronize(ws->stream); return rc; }
  return lease.finish();
}

static int store_overlaps_impl(ocmps_store* bra_store, ocmps_mps* bra, ocmps_store* ket, int Nt, int withK, double* out) {
  if (!ket || !out || Nt < 1 || Nt > ket->nslots) return fail(OCMPS_ERR_INVALID, "bad argument");
  ocmps_ctx* ctx = ket->ctx;
  CK(cudaSetDevice(ctx->dev));
  WsLease lease;
  int rc = lease.acquire(ctx, ket->lay.L, ket->lay.D, ket->lay.cap, 1);
  if (rc) return rc;
  Workspace* ws = lease[0];
  const int chunk = 64;
  for (int z0 = 0; z0 < Nt; z0 += chunk) {
    const int nb = std::min(chunk, Nt - z0);
    OvlSide sb = bra ? side_of_mps(bra) : side_of_store(bra_store, z0);
    const Layout& la = bra ? bra->lay : bra_store->lay;
    rc = overlaps_async(ws, sb, la, side_of_store(ket, z0), ket->lay, nb, withK, ws->stream);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out + 2 * z0, ws->d_out, sizeof(cplx) * nb, cudaMemcpyDeviceToHost, ws->stream));
    CK(cudaStreamSynchronize(ws->stream));
  }
  CK(cudaGetLastError());
  return OCMPS_OK;
}

int ocmps_store_overlaps(ocmps_store* store, ocmps_mps* bra, int Nt, double* out) {
  if (!bra) return fail(OCMPS_ERR_INVALID, "null bra");
  return store_overlaps_impl(nullptr, bra, store, Nt, 0, out);
}
int ocmps_store_divT(ocmps_store* xi_store, ocmps_store* psi_store, int Nt, double* out) {
  if (!xi_store) return fail(OCMPS_ERR_INVALID, "null store");
  return store_overlaps_impl(xi_store, nullptr, psi_store, Nt, 1, out);
}

// <psi_z| op_k at site j |psi_z> for the slices first .. first+count-1, all sites, `nops` diagonal site operators
// (include/correlations.hpp:99-117 `expectationValue(s)`: psi.position(j), local contraction -- here one pass of the
// transfer-matrix chain per slice, batched over the slices; see overlap_local_expect_kernel for the gauge precondition).
int ocmps_store_site_expectations(ocmps_store* store, int first, int count, const double* op_diag, int nops, double* out,
                                  double* norm2) {
  if (!store || !op_diag || !out || count < 1 || first < 0 || first + count > store->nslots)
    return fail(OCMPS_ERR_INVALID, "bad argument");
  if (nops < 1 || nops + 1 > OCMPS_EXPECT_MAX_OPS) return fail(OCMPS_ERR_INVALID, "site_expectations: 1..7 operators per call");
  ocmps_ctx* ctx = store->ctx;
  const Layout& lay = store->lay;
  const int L = lay.L, D = lay.D, nk = nops + 1;
  CK(cudaSetDevice(ctx->dev));
  WsLease lease;
  int rc = lease.acquire(ctx, L, D, lay.cap, 1);
  if (rc) return rc;
  Workspace* ws = lease[0];
  std::vector<double> h_ops((size_t)nk * D);
  for (int s = 0; s < D; ++s) h_ops[s] = 1.0;                               // slot 0: identity
  for (int k = 0; k < nops; ++k)
    for (int s = 0; s < D; ++s) h_ops[(size_t)(k + 1) * D + s] = op_diag[(size_t)k * D + s];
  const int chunk = 64;
  double *d_ops = nullptr, *d_res = nullptr;
  CK(cudaMalloc(&d_ops, sizeof(double) * h_ops.size()));
  CK(cudaMalloc(&d_res, sizeof(double) * (size_t)chunk * L * nk));
  CK(cudaMemcpy(d_ops, h_ops.data(), sizeof(double) * h_ops.size(), cudaMemcpyHostToDevice));
  std::vector<double> h_res((size_t)chunk * L * nk);
  cudaStream_t s = ws->stream;
  for (int z0 = 0; z0 < count && !rc; z0 += chunk) {
    const int nb = std::min(chunk, count - z0);
    const OvlSide side = side_of_store(store, first + z0);
    rc = ensure_overlap_bufs(ws, nb, lay.cap, lay.cap);
    if (rc) break;
    launch_overlap_init(ws->E[0], ws->e_stride, nb, 0, s);
    int cur = 0;
    for (int j = 0; j < L; ++j) {
      launch_overlap_plan(ws->odescs, side, side, j, nb, D, 0, ws->E[cur], ws->E[1 - cur], ws->T, ws->e_stride, ws->t_stride, s);
      launch_zgemm(ws->odescs, nb, lay.capb[j], D * lay.capb[j + 1], s);
      launch_overlap_local_expect(ws->odescs, side, j, nb, D, d_ops, nk, d_res, L, s);
      launch_zgemm(ws->odescs + nb, nb, lay.capb[j + 1], lay.capb[j + 1], s);
      cur = 1 - cur;
      g_ocmps_launches += 4;
    }
    g_ocmps_launches += 1;
    if (cudaMemcpyAsync(h_res.data(), d_res, sizeof(double) * (size_t)nb * L * nk, cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        cudaStreamSynchronize(s) != cudaSuccess) {
      rc = fail(OCMPS_ERR_CUDA, "site_expectations: copy failed");
      break;
    }
    for (int z = 0; z < nb; ++z)
      for (int j = 0; j < L; ++j) {
        const double* r = &h_res[((size_t)z * L + j) * nk];
        if (norm2) norm2[(size_t)(z0 + z) * L + j] = r[0];
        for (int k = 0; k < nops; ++k) out[((size_t)(z0 + z) * L + j) * nops + k] = r[k + 1];
      }
  }
  cudaFree(d_ops); cudaFree(d_res);
  if (rc) return rc;
  CK(cudaGetLastError());
  return OCMPS_OK;
}

// Two-point functions on a resident slice (include/correlations.hpp:10-55 correlationFunction, :57-80 correlationMatrix):
// out[z] = <psi| O_a(site_a) O_b(site_b) |psi> for `nentries` entries (site_a, op_a, site_b, op_b), sites 0-based, op_x an
// index into `op_table` (nops real D x D matrices <t|O|s>), site_b = -1 for a single operator.  All entries go through ONE
// batched pass of the <psi|psi> transfer-matrix chain with the operators applied to the physical index at their sites;
// number-changing operators (A, Adag) are fine, the intermediate transfer matrices then connect charge q with q +- 1.
// No gauge is assumed (the chain runs over all L sites), not divided by the norm (like the reference).
int ocmps_store_correlations(ocmps_store* store, int slot, const double* op_table, int nops, const int* entries, int nentries,
                             double* out) {
  if (!store || !op_table || !entries || !out || nops < 1 || nentries < 1 || slot < 0 || slot >= store->nslots)
    return fail(OCMPS_ERR_INVALID, "bad argument");
  ocmps_ctx* ctx = store->ctx;
  const Layout& lay = store->lay;
  const int L = lay.L, D = lay.D;
  for (int z = 0; z < nentries; ++z) {
    const int* e = entries + 4 * z;
    if (e[0] < 0 || e[0] >= L || e[1] < 0 || e[1] >= nops || e[2] >= L || (e[2] >= 0 && (e[3] < 0 || e[3] >= nops)) || e[2] == e[0])
      return fail(OCMPS_ERR_INVALID, "correlations: entry out of range (two operators on one site must be multiplied by the caller)");
  }
  CK(cudaSetDevice(ctx->dev));
  WsLease lease;
  int rc = lease.acquire(ctx, L, D, lay.cap, 1);
  if (rc) return rc;
  Workspace* ws = lease[0];
  cudaStream_t s = ws->stream;
  const int chunk = 128;
  double* d_ops = nullptr;
  int* d_sel = nullptr;
  CK(cudaMalloc(&d_ops, sizeof(double) * (size_t)nops * D * D));
  CK(cudaMalloc(&d_sel, sizeof(int) * (size_t)L * chunk));
  CK(cudaMemcpy(d_ops, op_table, sizeof(double) * (size_t)nops * D * D, cudaMemcpyHostToDevice));
  // every batch entry reads the same slice: strides 0
  OvlSide side = side_of_store(store, slot);
  side.slot_stride = 0;
  side.dims_stride = 0;
  side.base = store->data + (size_t)slot * lay.total;
  side.dims = store->dims + (size_t)slot * (L + 1);
  side.slot0 = 0;
  std::vector<int> h_sel((size_t)L * chunk);
  for (int z0 = 0; z0 < nentries && !rc; z0 += chunk) {
    const int nb = std::min(chunk, nentries - z0);
    rc = ensure_overlap_bufs(ws, nb, lay.cap, lay.cap);
    if (rc) break;
    for (int j = 0; j < L; ++j)
      for (int z = 0; z < nb; ++z) {
        const int* e = entries + 4 * (z0 + z);
        h_sel[(size_t)j * chunk + z] = e[0] == j ? e[1] : (e[2] == j ? e[3] : -1);
      }
    if (cudaMemcpyAsync(d_sel, h_sel.data(), sizeof(int) * h_sel.size(), cudaMemcpyHostToDevice, s) != cudaSuccess) { rc = fail(OCMPS_ERR_CUDA, "copy failed"); break; }
    launch_overlap_init(ws->E[0], ws->e_stride, nb, 0, s);
    int cur = 0;
    for (int j = 0; j < L; ++j) {
      launch_overlap_plan(ws->odescs, side, side, j, nb, D, 0, ws->E[cur], ws->E[1 - cur], ws->T, ws->e_stride, ws->t_stride, s);
      launch_zgemm(ws->odescs, nb, lay.capb[j], D * lay.capb[j + 1], s);
      launch_overlap_site_op(ws->T, ws->t_stride, ws->odescs, nb, D, d_ops, d_sel + (size_t)j * chunk, lay.capb[j] * lay.capb[j + 1], s);
      launch_zgemm(ws->odescs + nb, nb, lay.capb[j + 1], lay.capb[j + 1], s);
      cur = 1 - cur;
      g_ocmps_launches += 4;
    }
    launch_overlap_final(ws->E[cur], ws->e_stride, nb, 0, ws->d_out, s);
    g_ocmps_launches += 2;
    if (cudaMemcpyAsync(out + 2 * z0, ws->d_out, sizeof(cplx) * nb, cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        cudaStreamSynchronize(s) != cudaSuccess)
      rc = fail(OCMPS_ERR_CUDA, "correlations: copy failed");
  }
  cudaStreamSynchronize(s);
  cudaFree(d_ops); cudaFree(d_sel);
  if (rc) return rc;
  return lease.finish();
}

// Energy moments of resident slices under H(U_z) - c_z, the Hamiltonian of include/InitializeState.hpp:41-50 (and of the
// stepper at control value U): one transfer-matrix pass over all L sites per slice with the environments of the MPO channels
// (4 for W, 16 for W x W, see EnergyTable), batched over the slices.  Per site: T = E . B_j for all channels in one gemm per
// slice, the channel mixing on the physical index, then E'_v = A_j^H . T'_v.  No gauge is assumed; nothing is divided by the
// norm.  Slices are batched in chunks whose T and T' fit ENERGY_CHUNK_BYTES; every slice's reductions run in a fixed order
// that does not depend on the chunk, so a slice gives the same bits alone or in any batch.
constexpr long long ENERGY_CHUNK_BYTES = 1LL << 30;
constexpr int ENERGY_MAX_BATCH = 256;

static EnergyTable energy_table(int D, double J, int second_moment) {
  struct Entry { int a, b, f; double coef; };
  const Entry W[7] = {{0, 0, ENERGY_F_ID, 1.0},    {3, 3, ENERGY_F_ID, 1.0},  {3, 0, ENERGY_F_ONSITE, 1.0}, {3, 1, ENERGY_F_A, -J},
                      {3, 2, ENERGY_F_ADAG, -J},   {1, 0, ENERGY_F_ADAG, 1.0}, {2, 0, ENERGY_F_A, 1.0}};
  EnergyTable t;
  memset(&t, 0, sizeof(t));
  t.nch = second_moment ? 16 : 4;
  for (int s = 1; s < D; ++s) {
    t.A[(s - 1) * D + s] = std::sqrt((double)s);      // a|s> = sqrt(s) |s-1>
    t.Adag[s * D + (s - 1)] = std::sqrt((double)s);   // adag|s-1> = sqrt(s) |s>
  }
  std::vector<Entry> tr;                              // (src, dst, f1, coef) and f2 below
  std::vector<int> f2;
  for (int i = 0; i < 7; ++i) {
    if (!second_moment) { tr.push_back(W[i]); f2.push_back(ENERGY_F_ID); continue; }
    for (int k = 0; k < 7; ++k) {
      tr.push_back({4 * W[i].a + W[k].a, 4 * W[i].b + W[k].b, W[i].f, W[i].coef * W[k].coef});
      f2.push_back(W[k].f);
    }
  }
  std::vector<int> order(tr.size());
  for (size_t i = 0; i < order.size(); ++i) order[i] = (int)i;
  std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return tr[x].b < tr[y].b; });
  t.nt = (int)tr.size();
  for (int k = 0; k < t.nt; ++k) {
    const Entry& e = tr[order[k]];
    t.src[k] = e.a; t.dst[k] = e.b; t.f1[k] = e.f; t.f2[k] = f2[order[k]]; t.coef[k] = e.coef;
  }
  return t;
}

int ocmps_store_energy_moments(ocmps_store* store, int first, int count, double J, const double* U, const double* shift,
                               int second_moment, double* out) {
  if (!store || !U || !out || count < 1 || first < 0 || first > store->nslots - count || (second_moment != 0 && second_moment != 1))
    return fail(OCMPS_ERR_INVALID, "bad argument");
  if (!std::isfinite(J)) return fail(OCMPS_ERR_INVALID, "energy_moments: J is not finite");
  for (int z = 0; z < count; ++z)
    if (!std::isfinite(U[z]) || (shift && !std::isfinite(shift[z])))
      return fail(OCMPS_ERR_INVALID, "energy_moments: U or shift is not finite");
  ocmps_ctx* ctx = store->ctx;
  const Layout& lay = store->lay;
  const int L = lay.L, D = lay.D;
  const EnergyTable tab = energy_table(D, J, second_moment);
  const int nch = tab.nch;
  CK(cudaSetDevice(ctx->dev));
  WsLease lease;
  int rc = lease.acquire(ctx, L, D, lay.cap, 1);
  if (rc) return rc;
  Workspace* ws = lease[0];
  cudaStream_t s = ws->stream;
  const long long slice_bytes = 2LL * nch * lay.cap * D * lay.cap * (long long)sizeof(cplx);   // T and T'
  const int chunk = (int)std::max(1LL, std::min<long long>({(long long)ENERGY_MAX_BATCH, (long long)count, ENERGY_CHUNK_BYTES / slice_bytes}));
  CK(cudaStreamSynchronize(s));
  rc = ensure_energy_bufs(ws, chunk, nch, lay.cap);
  if (rc) return rc;
  const auto& b = ws->en;
  std::vector<double> h_uc(2 * (size_t)chunk), h_out(3 * (size_t)chunk);
  for (int z0 = 0; z0 < count && !rc; z0 += chunk) {
    const int nb = std::min(chunk, count - z0);
    for (int z = 0; z < nb; ++z) {
      h_uc[2 * z] = U[z0 + z];
      h_uc[2 * z + 1] = shift ? shift[z0 + z] / L : 0.0;
    }
    if (cudaMemcpyAsync(b.uc, h_uc.data(), sizeof(double) * 2 * nb, cudaMemcpyHostToDevice, s) != cudaSuccess) {
      rc = fail(OCMPS_ERR_CUDA, "energy_moments: copy failed"); break;
    }
    const OvlSide side = side_of_store(store, first + z0);
    launch_energy_init(b.E[0], b.e_stride, nb, nch, s);
    int cur = 0;
    for (int j = 0; j < L; ++j) {
      launch_overlap_plan_channels(b.descs, side, side, j, nb, D, nch, b.E[cur], b.E[1 - cur], b.T, b.Tm, b.e_stride, b.t_stride, s);
      launch_zgemm(b.descs, nb, nch * lay.capb[j], D * lay.capb[j + 1], s);
      launch_energy_mix(b.T, b.Tm, b.t_stride, b.descs, nb, D, b.uc, tab, lay.capb[j] * lay.capb[j + 1], s);
      launch_zgemm(b.descs + nb, nch * nb, lay.capb[j + 1], lay.capb[j + 1], s);
      cur = 1 - cur;
      g_ocmps_launches += 4;
    }
    launch_energy_final(b.E[cur], b.e_stride, nb, nch, b.out, s);
    g_ocmps_launches += 2;
    if (cudaMemcpyAsync(h_out.data(), b.out, sizeof(double) * 3 * nb, cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        cudaStreamSynchronize(s) != cudaSuccess) {
      rc = fail(OCMPS_ERR_CUDA, "energy_moments: copy failed"); break;
    }
    for (int z = 0; z < nb; ++z) {
      out[3 * (z0 + z) + 0] = h_out[3 * z + 0];
      out[3 * (z0 + z) + 1] = h_out[3 * z + 1];
      if (second_moment) out[3 * (z0 + z) + 2] = h_out[3 * z + 2];
    }
  }
  cudaStreamSynchronize(s);
  if (rc) return rc;
  return lease.finish();
}

// The start state of both ground-state generators, the reference's product state |0..0 1..1> (include/InitializeState.hpp:24-38):
// one boson on each of the last Npart sites.
static int upload_product_state(ocmps_mps* out, int L, int D, int Npart) {
  std::vector<int> dims(L + 1, 1), q(L + 1, 0);
  std::vector<double> t((size_t)2 * L * D, 0.0);
  int tot = 0;
  for (int j = 0; j < L; ++j) {
    const int occ = j >= L - Npart ? 1 : 0;
    t[((size_t)j * D + occ) * 2] = 1.0;
    tot += occ;
    q[j + 1] = tot;
  }
  return ocmps_mps_upload(out, dims.data(), q.data(), t.data(), 0, 2);
}

// Bose-Hubbard ground state on the device engine (the role of include/InitializeState.hpp:18-117 in the reference:
// psi_init / psi_target of every main program and test come from it).  The reference runs ITensor's DMRG; here the SAME
// Trotter-step kernels that do the real-time evolution run in imaginary time: gates exp(-tau h), on-site factors
// exp(-tau U/4 n(n-1)), renormalisation after every truncation (which the step does anyway).  Start: the reference's
// product state (one boson on each of the last Npart sites, :24-38).  tau is lowered in stages (0.1 -> tau_final) with the
// reference's bond-dimension schedule 10, 20, 50, maxm (:52-54); a stage ends when the energy
// <H> = -J sum <a+_i a_{i+1} + h.c.> + U/2 sum <n_i(n_i-1)> (two-point functions + site expectations on the device) has stopped
// moving.  The fixed point of a first-order Trotter splitting differs from the true ground state by O(tau) in the state and
// O(tau^2) in the energy; tau_final = 2e-3 gives energies good to ~1e-6 relative.  Result: normalised, centre at site 1.
int ocmps_ground_state(ocmps_ctx* ctx, int L, int D, int Npart, double J, double U, int maxm, double cutoff, double tau_final,
                       ocmps_mps* out, double* energy_out, int* steps_out) {
  if (!ctx || !out) return fail(OCMPS_ERR_INVALID, "null argument");
  if (L < 2 || Npart < 0 || Npart > L) return fail(OCMPS_ERR_INVALID, "ground_state: needs L >= 2 and 0 <= Npart <= L (the reference supports one boson per site at most in its initial guess)");
  if (out->lay.L != L || out->lay.D != D) return fail(OCMPS_ERR_INVALID, "ground_state: output MPS has another shape");
  if (maxm < 1) maxm = out->lay.cap;
  if (maxm > out->lay.cap) return fail(OCMPS_ERR_CAPACITY, "ground_state: maxm exceeds the capacity of the output MPS");
  if (!(tau_final > 0.0)) tau_final = 2e-3;
  if (cutoff < 0.0) cutoff = 1e-9;
  CK(cudaSetDevice(ctx->dev));
  const int cap = out->lay.cap;
  int rc = upload_product_state(out, L, D, Npart);
  if (rc) return rc;
  ocmps_store* tmp = nullptr;
  rc = ocmps_store_create(ctx, L, D, cap, 1, &tmp);
  if (rc) return rc;
  // operator table: 0 = Adag, 1 = A; entries (i, Adag, i+1, A)
  std::vector<double> ops((size_t)2 * D * D, 0.0);
  for (int j = 1; j < D; ++j) { ops[(size_t)j * D + (j - 1)] = std::sqrt((double)j); ops[(size_t)D * D + (size_t)(j - 1) * D + j] = std::sqrt((double)j); }
  std::vector<int> entries;
  for (int i = 0; i + 1 < L; ++i) { entries.push_back(i); entries.push_back(0); entries.push_back(i + 1); entries.push_back(1); }
  std::vector<double> corr((size_t)2 * (L - 1)), nn1(L), nrm(L), diag(D);
  for (int n = 0; n < D; ++n) diag[n] = (double)n * (n - 1);
  auto energy = [&](double& e) -> int {
    int r = ocmps_store_put(tmp, 0, out);
    if (!r) r = ocmps_store_correlations(tmp, 0, ops.data(), 2, entries.data(), L - 1, corr.data());
    if (!r) r = ocmps_store_site_expectations(tmp, 0, 1, diag.data(), 1, nn1.data(), nrm.data());
    if (r) return r;
    double hop = 0.0, on = 0.0;
    for (int i = 0; i + 1 < L; ++i) hop += corr[2 * i];
    for (int j = 0; j < L; ++j) on += nn1[j];
    e = (-2.0 * J * hop + 0.5 * U * on) / nrm[0];
    return OCMPS_OK;
  };
  const int sched[4] = {10, 20, 50, maxm};
  std::vector<double> taus;
  for (double tau : {0.1, 0.05, 0.02, 0.01, 0.005, 0.002, 0.001, 0.0005, 0.0002, 0.0001})
    if (tau > tau_final * 1.0001) taus.push_back(tau);
  taus.push_back(tau_final);
  int total_steps = 0;
  double e_prev = 0.0, e = 0.0;
  rc = energy(e_prev);
  for (size_t sg = 0; sg < taus.size() && !rc; ++sg) {
    const double tau = taus[sg];
    const int mm = std::min(maxm, sched[std::min<size_t>(sg, 3)]);
    ocmps_stepper* st = nullptr;
    rc = ocmps_stepper_create(ctx, L, D, J, tau, cutoff, mm, cap, 0, &st);
    if (rc) break;
    st->imag = true;
    rc = ocmps_stepper_set_tstep(st, tau);              // rebuilds the gates as exp(-tau h)
    const int check = 10, max_steps = 4000;
    const double tol = 1e-10 * std::max(1.0, tau / tau_final);
    int quiet = 0;
    for (int k = 0; k < max_steps && !rc; k += check) {
      {
        WsLease lease;
        rc = lease.acquire(ctx, L, D, cap, 1);
        if (rc) break;
        Workspace* ws = lease[0];
        for (int i = 0; i < check && !rc; ++i) rc = step_enqueue(st, out, ws, U, U, true, nullptr, 0, ws->stream);
        if (rc) { cudaStreamSynchronize(ws->stream); break; }
        rc = lease.finish();
        if (rc) break;
      }
      total_steps += check;
      rc = energy(e);
      if (rc) break;
      const bool still = std::fabs(e - e_prev) <= tol * std::max(1.0, std::fabs(e));
      e_prev = e;
      quiet = still ? quiet + 1 : 0;
      if (quiet >= 2) break;
    }
    ocmps_stepper_destroy(st);
  }
  ocmps_store_destroy(tmp);
  if (rc) return rc;
  if (energy_out) *energy_out = e_prev;
  if (steps_out) *steps_out = total_steps;
  return OCMPS_OK;
}

// Bose-Hubbard ground state by two-site DMRG on the device (the reference's InitializeState, include/InitializeState.hpp:18-117,
// runs ITensor's DMRG).  The algorithm is the oracle's ground_state_dmrg: the product start state of ocmps_ground_state, the
// bond-dimension-4 MPO of the chain, right environments first, then left->right and right->left half sweeps over the bonds.  At
// each bond: a Lanczos solve of H_eff theta (4 Krylov vectors, full reorthogonalisation, charge-allowed entries only), the gate
// decomposition with ITensor's truncation (cutoff, maxm of the sweep), the environment update.  Bond dimensions follow the
// reference's schedule 10, 20, 50, maxm.  There is no noise term (the reference adds none to its energy either; the oracle has
// none).  One sweep is enqueued without host synchronisation; the host reads the last Ritz value of every sweep.
int ocmps_ground_state_dmrg(ocmps_ctx* ctx, int L, int D, int Npart, double J, double U, int maxm, double cutoff, int nsweeps,
                            ocmps_mps* out, double* energy_out, double* sweep_energies) {
  if (!ctx || !out) return fail(OCMPS_ERR_INVALID, "null argument");
  if (L < 2 || Npart < 0 || Npart > L) return fail(OCMPS_ERR_INVALID, "ground_state_dmrg: needs L >= 2 and 0 <= Npart <= L (the reference supports one boson per site at most in its initial guess)");
  if (out->lay.L != L || out->lay.D != D) return fail(OCMPS_ERR_INVALID, "ground_state_dmrg: output MPS has another shape");
  if (nsweeps < 1) return fail(OCMPS_ERR_INVALID, "ground_state_dmrg: nsweeps must be >= 1");
  if (maxm < 1) maxm = out->lay.cap;
  if (maxm > out->lay.cap) return fail(OCMPS_ERR_CAPACITY, "ground_state_dmrg: maxm exceeds the capacity of the output MPS");
  if (cutoff < 0.0) cutoff = 1e-9;
  CK(cudaSetDevice(ctx->dev));
  int rc = upload_product_state(out, L, D, Npart);
  if (rc) return rc;
  ocmps_mps* m = out;
  const Layout& lay = m->lay;
  const int cap = lay.cap;
  WsLease lease;
  rc = lease.acquire(ctx, L, D, cap, 1);
  if (rc) return rc;
  Workspace* ws = lease[0];
  cudaStream_t s = ws->stream;

  // buffers of this call: environments (3 channels per bond and side), Krylov vectors V_0..V_3 + W, the Ritz vector X,
  // boundary products Y / Z of H_eff, products T / T' of the environment update
  long long vmax = 1, tmax = 1;
  for (int b = 0; b + 2 <= L; ++b) vmax = std::max(vmax, (long long)lay.capb[b] * D * D * lay.capb[b + 2]);
  for (int j = 0; j < L; ++j) tmax = std::max(tmax, (long long)lay.capb[j] * D * lay.capb[j + 1]);
  const long long estride = (long long)cap * cap;
  struct Bufs {
    cplx *EL = nullptr, *ER = nullptr, *V = nullptr, *X = nullptr, *Y = nullptr, *Z = nullptr, *T = nullptr, *T2 = nullptr;
    GemmDesc* descs = nullptr;
    KrylovState* ks = nullptr;
    double *partial = nullptr, *energies = nullptr;
    cudaStream_t s = nullptr;
    ~Bufs() {
      if (s) cudaStreamSynchronize(s);
      cudaFree(EL); cudaFree(ER); cudaFree(V); cudaFree(X); cudaFree(Y); cudaFree(Z); cudaFree(T); cudaFree(T2);
      cudaFree(descs); cudaFree(ks); cudaFree(partial); cudaFree(energies);
    }
  } B;
  B.s = s;
  const size_t env_bytes = sizeof(cplx) * (size_t)(L + 1) * 3 * estride;
  CK(cudaMalloc(&B.EL, env_bytes));
  CK(cudaMalloc(&B.ER, env_bytes));
  CK(cudaMalloc(&B.V, sizeof(cplx) * (size_t)(DMRG_KRYLOV + 1) * vmax));
  CK(cudaMalloc(&B.X, sizeof(cplx) * (size_t)vmax));
  CK(cudaMalloc(&B.Y, sizeof(cplx) * (size_t)3 * vmax));
  CK(cudaMalloc(&B.Z, sizeof(cplx) * (size_t)3 * vmax));
  CK(cudaMalloc(&B.T, sizeof(cplx) * (size_t)3 * tmax));
  CK(cudaMalloc(&B.T2, sizeof(cplx) * (size_t)3 * tmax));
  CK(cudaMalloc(&B.descs, sizeof(GemmDesc) * 13));
  CK(cudaMalloc(&B.ks, sizeof(KrylovState)));
  CK(cudaMalloc(&B.partial, sizeof(double) * 2 * 128 * (DMRG_KRYLOV + 1)));
  CK(cudaMalloc(&B.energies, sizeof(double) * (nsweeps + 1)));
  // the boundary environments (left of site 0, right of site L-1) are 1 x 1 and hold no term: zero
  CK(cudaMemsetAsync(B.EL, 0, env_bytes, s));
  CK(cudaMemsetAsync(B.ER, 0, env_bytes, s));
  CK(cudaMemsetAsync(B.ks, 0, sizeof(KrylovState), s));
  cplx* W = B.V + (size_t)DMRG_KRYLOV * vmax;
  GemmDesc* hdescs = B.descs;          // [0, 6) H_eff, [6, 12) environment update, [12] two-site merge
  GemmDesc* edescs = B.descs + 6;
  GemmDesc* mdesc = B.descs + 12;
  auto env = [&](cplx* E, int b) { return E + (size_t)b * 3 * estride; };

  // ER[j] (sites >= j) from ER[j+1] and the right isometry at site j; EL[j+1] (sites <= j) from EL[j] and the left isometry at j
  auto grow_right = [&](int j) {
    launch_env_update(edescs, 1, m->site(j), env(B.ER, j + 1), env(B.ER, j), B.T, B.T2, tmax, estride, m->dim(j), m->dim(j + 1), D,
                      J, U, lay.capb[j], lay.capb[j + 1], s);
    g_ocmps_launches += 4;
  };
  auto grow_left = [&](int j) {
    launch_env_update(edescs, 0, m->site(j), env(B.EL, j), env(B.EL, j + 1), B.T, B.T2, tmax, estride, m->dim(j), m->dim(j + 1), D,
                      J, U, lay.capb[j], lay.capb[j + 1], s);
    g_ocmps_launches += 4;
  };
  // theta of sites b, b+1 -> X, normalised -> V_0 (new Krylov space)
  auto merge_start = [&](int b) {
    const int* dl = m->dim(b);
    const int* dr = m->dim(b + 2);
    const int nmax = lay.capb[b] * D * D * lay.capb[b + 2];
    launch_merge_setup(mdesc, m->site(b), m->site(b + 1), B.X, dl, m->dim(b + 1), dr, D, s);
    launch_zgemm(mdesc, 1, lay.capb[b] * D, D * lay.capb[b + 2], s);
    launch_krylov_dot(B.X, 0, 1, B.X, dl, dr, D, nullptr, B.partial, s);
    launch_krylov_init(B.X, B.V, dl, dr, D, B.ks, B.partial, nmax, s);
    g_ocmps_launches += 4;
  };
  auto heff = [&](int b, const cplx* Vin) {
    launch_heff(hdescs, Vin, W, B.Y, B.Z, vmax, env(B.EL, b), env(B.ER, b + 2), estride, m->dim(b), m->dim(b + 2), m->q(b), m->q(b + 2),
                D, J, U, B.ks, lay.capb[b], lay.capb[b + 2], s);
    g_ocmps_launches += 4;
  };
  // Lanczos solve at bond b (sites b, b+1), gate decomposition, the theta of the next bond left in the MPS
  auto bond_step = [&](int b, bool left, int mm) {
    const int* dl = m->dim(b);
    const int* dr = m->dim(b + 2);
    const int nmax = lay.capb[b] * D * D * lay.capb[b + 2];
    merge_start(b);
    for (int it = 0; it < DMRG_KRYLOV; ++it) {
      const cplx* Vit = B.V + (size_t)it * vmax;
      heff(b, Vit);
      launch_krylov_dot(Vit, 0, 1, W, dl, dr, D, B.ks, B.partial, s);
      launch_krylov_alpha(B.V, vmax, it, W, dl, dr, D, B.ks, B.partial, nmax, s);
      g_ocmps_launches += 2;
      if (it == DMRG_KRYLOV - 1) break;            // the last residual is not needed
      launch_krylov_dot(B.V, vmax, it + 1, W, dl, dr, D, B.ks, B.partial, s);
      launch_krylov_reorth(B.V, vmax, it + 1, W, dl, dr, D, B.ks, B.partial, nmax, s);
      launch_krylov_dot(W, 0, 1, W, dl, dr, D, B.ks, B.partial, s);
      launch_krylov_next(B.V, vmax, it, W, dl, dr, D, B.ks, B.partial, nmax, s);
      g_ocmps_launches += 4;
    }
    launch_krylov_ritz(B.ks, s);
    launch_krylov_combine(B.V, vmax, B.X, dl, dr, D, B.ks, nmax, s);
    launch_krylov_dot(B.X, 0, 1, B.X, dl, dr, D, nullptr, B.partial, s);
    launch_krylov_scale(B.X, dl, dr, D, B.partial, nmax, s);
    g_ocmps_launches += 4;
    const int j1 = b, j2 = b + 1, bm = b + 1;
    DecompArgs a;
    a.kind = left ? DK_GATE_LEFT : DK_GATE_RIGHT;
    a.D = D;
    a.dimL = dl; a.dimR = dr; a.qL = m->q(b); a.qR = m->q(b + 2);
    a.dimNew = m->dim(bm); a.qNew = m->q(bm);
    a.X = B.X;
    a.iso = left ? m->other(j1) : m->other(j2);
    a.partner = left ? m->other(j2) : m->other(j1);
    a.nb_in = nullptr; a.nb_out = nullptr; a.dimNb = nullptr; a.qNb = nullptr;
    const TruncParams tp{cutoff, mm, 1, 0, lay.capb[bm], 1};
    const int capV = left ? lay.capb[b + 2] : lay.capb[b];
    const int capC = left ? lay.capb[b] : lay.capb[b + 2];
    run_decomp(ws, a, tp, capV, capC, lay.capb[bm], s);
    m->cur[j1] ^= 1; m->cur[j2] ^= 1;
  };

  for (int j = L - 1; j >= 2; --j) grow_right(j);
  const int sched[4] = {10, 20, 50, maxm};
  std::vector<double> h_e(nsweeps + 1, 0.0);
  for (int sw = 0; sw < nsweeps && !rc; ++sw) {
    const int mm = std::min(maxm, sched[std::min(sw, 3)]);
    for (int b = 0; b <= L - 2; ++b) {
      bond_step(b, true, mm);
      if (b < L - 2) grow_left(b);
    }
    for (int b = L - 2; b >= 0; --b) {
      bond_step(b, false, mm);
      if (b > 0) grow_right(b + 1);
    }
    CK(cudaMemcpyAsync(B.energies + sw, &B.ks->ritz, sizeof(double), cudaMemcpyDeviceToDevice, s));
    CK(cudaMemcpyAsync(&h_e[sw], B.energies + sw, sizeof(double), cudaMemcpyDeviceToHost, s));
    rc = lease.finish();               // waits for the sweep; reports (and clears) what its kernels flagged
  }
  if (rc) return rc;
  // <psi|H|psi> of the returned state: one H_eff application on the final two-site tensor (bond 0, after truncation)
  merge_start(0);
  heff(0, B.V);
  launch_krylov_dot(B.V, 0, 1, W, m->dim(0), m->dim(2), D, B.ks, B.partial, s);
  launch_partial_total(B.partial, B.energies + nsweeps, s);
  g_ocmps_launches += 2;
  CK(cudaMemcpyAsync(&h_e[nsweeps], B.energies + nsweeps, sizeof(double), cudaMemcpyDeviceToHost, s));
  rc = lease.finish();
  if (rc) return rc;
  m->llim = 0; m->rlim = 2;
  if (energy_out) *energy_out = h_e[nsweeps];
  if (sweep_energies) for (int sw = 0; sw < nsweeps; ++sw) sweep_energies[sw] = h_e[sw];
  return OCMPS_OK;
}

// Entanglement entropy of every bond of the slices first .. first+count-1 (include/correlations.hpp:119-148:
// psi.position(i), SVD of the two-site wavefunction, S = -sum_{p>1e-12} p ln p over the density-matrix eigenvalues).
// The orthogonality centre of a copy of the slice is moved from site 1 to site L with the engine's own gauge moves;
// the spectrum of the move across bond i is the Schmidt spectrum of that bond.  The store is not modified.
int ocmps_store_entanglement_entropy(ocmps_store* store, int first, int count, double* out) {
  if (!store || !out || count < 1 || first < 0 || first + count > store->nslots) return fail(OCMPS_ERR_INVALID, "bad argument");
  ocmps_ctx* ctx = store->ctx;
  const Layout& lay = store->lay;
  const int L = lay.L, D = lay.D;
  if (L < 2) return fail(OCMPS_ERR_INVALID, "entanglement_entropy needs L >= 2");
  CK(cudaSetDevice(ctx->dev));
  WsLease lease;
  int rc = lease.acquire(ctx, L, D, lay.cap, 1);
  if (rc) return rc;
  Workspace* ws = lease[0];
  double* d_out = nullptr;
  CK(cudaMalloc(&d_out, sizeof(double) * (size_t)count * (L - 1)));
  cudaStream_t s = ws->stream;
  ocmps_mps* m = ws->work;
  TruncParams tpo{MIN_CUT, MAX_M, 1, 0, 0, 0};
  for (int z = 0; z < count && !rc; ++z) {
    rc = store_get_async(store, first + z, m, s);
    if (rc) break;
    for (int b = 1; b <= L - 1; ++b) {
      const int j = b - 1, jn = b;
      DecompArgs a;
      a.D = D; a.kind = DK_ORTH_LEFT;
      a.dimNew = m->dim(b); a.qNew = m->q(b); a.partner = ws->cbuf;
      a.dimL = m->dim(b - 1); a.dimR = m->dim(b); a.qL = m->q(b - 1); a.qR = m->q(b);
      a.X = m->site(j); a.iso = m->other(j);
      a.nb_in = m->site(jn); a.nb_out = m->other(jn); a.dimNb = m->dim(b + 1);
      a.qNb = fused_push_enabled() ? m->q(b + 1) : nullptr;
      tpo.cap = lay.capb[b];
      run_decomp(ws, a, tpo, lay.capb[b], lay.capb[b - 1], lay.capb[b], s);
      if (!a.qNb) { launch_zgemm(ws->db.descs + 1, 1, lay.capb[b], D * lay.capb[b + 1], s); g_ocmps_launches += 1; }
      launch_spectrum_entropy(ws->db, d_out + (size_t)z * (L - 1) + (b - 1), s);
      g_ocmps_launches += 1;
      m->cur[j] ^= 1; m->cur[jn] ^= 1;
    }
  }
  if (!rc && (cudaMemcpyAsync(out, d_out, sizeof(double) * (size_t)count * (L - 1), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
              cudaStreamSynchronize(s) != cudaSuccess))
    rc = fail(OCMPS_ERR_CUDA, "entanglement_entropy: copy failed");
  cudaStreamSynchronize(s);
  cudaFree(d_out);
  if (rc) return rc;
  return lease.finish();
}

int ocmps_store_apply_K(ocmps_stepper* st, ocmps_store* in, int Nt, ocmps_store* out) {
  if (!st || !in || !out || Nt < 1 || Nt > in->nslots || Nt > out->nslots) return fail(OCMPS_ERR_INVALID, "bad argument");
  int rc = check_shapes(st, in->lay, "store_apply_K");
  if (rc) return rc;
  rc = check_shapes(st, out->lay, "store_apply_K");
  if (rc) return rc;
  CK(cudaSetDevice(st->ctx->dev));
  const int nch = std::min(Nt, 8);
  WsLease lease;
  rc = lease.acquire(st->ctx, st->L, st->D, st->cap, nch);
  if (rc) return rc;
  const std::vector<Workspace*>& wss = lease.ws;
  for (int c = 0; c < nch; ++c)
    if (!wss[c]->tmpK) {          // kept with the workspace: no allocation per call
      rc = alloc_mps(st->ctx, st->L, st->D, st->cap, &wss[c]->tmpK);
      if (rc) return rc;
    }
  for (int i = 0; i < Nt; ++i) {
    Workspace* ws = wss[i % nch];
    rc = store_get_async(in, i, ws->work, ws->stream);
    if (!rc) rc = apply_K_async(st, ws, ws->work, ws->tmpK, ws->stream);
    if (!rc) rc = store_put_async(out, i, ws->tmpK, ws->stream);
    if (rc) break;
  }
  if (rc) { for (Workspace* w : wss) cudaStreamSynchronize(w->stream); return rc; }
  return lease.finish();
}

// ------------------------------------------------------------------------------------------------
// Hessian (src/OptimalControl.cpp:252-372): prerequisites and rows as ONE stream/event schedule
// ------------------------------------------------------------------------------------------------
// The reference computes psi_t, xi_t, divT, then xiHlist, then the rows (work queue :305-335).  Row r only needs psi_r to
// start and the K.xi slices only at its overlaps, so here everything is enqueued at once and ordered by events:
//   * the psi sweep records an event per stored slice; the chain of row r waits for the event of slice r, i.e. the rows
//     trail the sweep instead of waiting for it (the sweep is the critical path of a sharded Hessian);
//   * the xi sweep records an event per slice as well; K|xi_i> (exactApplyMPO :300-303) follows slice by slice on
//     NK chains;
//   * a row writes its propagated slices -- starting with K|psi_r> itself, whose overlap is the diagonal entry :260-264 --
//     into a per-chain ring of NCH chunks; a finished chunk is overlapped with the matching K.xi slices in one batched
//     transfer-matrix pass on the chain's overlap stream, which also waits for the K.xi store; the row only stalls if
//     it gets NCH chunks ahead of its overlaps;
//   * divT and the fidelity overlaps run at the tail of the two sweep streams.
// With do_psi = do_xi = do_xiH = 0 this is the plain row computation on stores that are already valid.
static int hessian_run(ocmps_stepper* st, ocmps_mps* psi_init, ocmps_mps* psi_target, const double* u, int Nt, ocmps_store* psi_store,
                       ocmps_store* xi_store, ocmps_store* xiH_store, const int* rows, int nrows, int nchains, int do_psi, int do_xi,
                       int do_xiH, double* divT, double* fid, double* ovl, double* norms) {
  if (!st || !psi_store || !xiH_store || !u || (!rows && nrows > 0) || !ovl || !norms || Nt < 3) return fail(OCMPS_ERR_INVALID, "bad argument");
  int rc = check_shapes(st, psi_store->lay, "hessian");
  if (rc) return rc;
  rc = check_shapes(st, xiH_store->lay, "hessian");
  if (rc) return rc;
  if (psi_store->nslots < Nt || xiH_store->nslots < Nt) return fail(OCMPS_ERR_INVALID, "hessian: store has fewer slots than Nt");
  if ((do_xi || do_xiH || divT) && !xi_store) return fail(OCMPS_ERR_INVALID, "hessian: xi store needed");
  if (xi_store) { rc = check_shapes(st, xi_store->lay, "hessian"); if (rc) return rc; if (xi_store->nslots < Nt) return fail(OCMPS_ERR_INVALID, "hessian: store has fewer slots than Nt"); }
  if (do_psi) { rc = sweep_args_ok(st, psi_init, u, Nt, psi_store); if (rc) return rc; }
  if (do_xi) { rc = sweep_args_ok(st, psi_target, u, Nt, xi_store); if (rc) return rc; }
  if (fid && !psi_target) return fail(OCMPS_ERR_INVALID, "hessian: target state needed for the fidelity overlaps");
  for (int i = 0; i < nrows; ++i)
    if (rows[i] < 1 || rows[i] > Nt - 2) return fail(OCMPS_ERR_INVALID, "hessian row out of range [1, Nt-2]");
  if (nchains < 1) nchains = 1;
  nchains = std::min(nchains, std::max(nrows, 1));
  CK(cudaSetDevice(st->ctx->dev));
  // ring of propagated slices per chain: NCH chunks of CH slots
  int CH = 32, NCH = 4;
  if (const char* e = getenv("OCMPS_HESSIAN_CHUNK")) CH = std::max(1, atoi(e));
  if (const char* e = getenv("OCMPS_HESSIAN_RING")) NCH = std::max(2, atoi(e));
  CH = std::min(CH, std::max(1, Nt - 1));
  NCH = std::min(NCH, (Nt - 1 + CH - 1) / CH + 1);
  if (!do_psi && !do_xiH) NCH = 2;                 // nothing to wait for: double buffering is enough
  const int ring = CH * NCH;
  {
    // rows in flight are also bounded by memory: a chain owns two work states, the 2*chi product state of K|psi> with its
    // workspace, and the ring of propagated slices (about 2.3 GB at chi=100 with the default ring)
    Layout l1, l2;
    l1.init(st->L, st->D, st->cap);
    l2.init(st->L, st->D, st->cap, 2);
    const double nD2 = (double)l2.cap * st->D;
    const double per_chain = 16.0 * ((ring + 6.0) * (double)l1.total + 2.0 * (double)l2.total + 2.0 * nD2 * nD2 + 8.0 * nD2 * l2.cap);
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && per_chain > 0.0) {
      int have = 0;                                        // chains of this shape that already own their buffers
      {
        std::lock_guard<std::mutex> lock(st->ctx->mu);
        for (Workspace* w : st->ctx->pool)
          if (!w->busy && w->L == st->L && w->D == st->D && w->cap == st->cap && w->rowstore && w->rowstore->nslots == ring) ++have;
      }
      const int fit = have + (int)std::min<double>(1e6, 0.8 * (double)free_b / per_chain);
      nchains = std::max(1, std::min(nchains, fit));
    }
  }
  const int NK = do_xiH ? std::min(Nt, 8) : 0;
  // workspaces: [0] psi sweep / fidelity overlaps, [1] xi sweep / divT, [2, 2+NK) K.xi chains, then the row chains.
  // Always leased in this order so that every role gets the same workspace (and its buffers and graphs) on every call.
  WsLease lease;
  rc = lease.acquire(st->ctx, st->L, st->D, st->cap, 2 + 8 + nchains);
  if (rc) return rc;
  Workspace* wP = lease[0];
  Workspace* wX = lease[1];
  std::vector<Workspace*> wK(lease.ws.begin() + 2, lease.ws.begin() + 2 + 8);
  std::vector<Workspace*> wss(lease.ws.begin() + 10, lease.ws.end());
  auto sync_all = [&]() { for (Workspace* w : lease.ws) { cudaStreamSynchronize(w->stream); if (w->ovl) cudaStreamSynchronize(w->ovl); } };
  std::vector<ocmps_mps*> psiH(nchains, nullptr);
  for (int c = 0; c < nchains; ++c) {
    Workspace* ws = wss[c];
    if (!ws->psiH) {          // kept with the workspace so that its step graphs stay valid across calls
      rc = alloc_mps(st->ctx, st->L, st->D, st->cap, &ws->psiH);
      if (rc) return rc;
    }
    psiH[c] = ws->psiH;
    if (ws->rowstore && ws->rowstore->nslots != ring) {
      cudaStreamSynchronize(ws->stream);
      cudaFree(ws->rowstore->data); cudaFree(ws->rowstore->dims); cudaFree(ws->rowstore->q); delete ws->rowstore;
      ws->rowstore = nullptr;
    }
    if (!ws->rowstore) {
      rc = ocmps_store_create(st->ctx, st->L, st->D, st->cap, ring, &ws->rowstore);
      if (rc) return rc;
    }
    if (!ws->ovl) CK(cudaStreamCreateWithFlags(&ws->ovl, cudaStreamNonBlocking));
    rc = ensure_overlap_bufs(ws, CH, st->cap, st->cap);      // (may reallocate: before anything is in flight)
    if (rc) return rc;
  }
  for (int k = 0; k < NK; ++k)
    if (!wK[k]->tmpK) { rc = alloc_mps(st->ctx, st->L, st->D, st->cap, &wK[k]->tmpK); if (rc) return rc; }
  const int OB = 64;                                           // slices per batched pass of the divT / fidelity overlaps
  if (divT) { rc = ensure_overlap_bufs(wX, std::min(OB, Nt), st->cap, st->cap); if (rc) return rc; }
  if (fid) { rc = ensure_overlap_bufs(wP, std::min(OB, Nt), st->cap, st->cap); if (rc) return rc; }

  cplx *d_ovl = nullptr, *d_div = nullptr, *d_fid = nullptr;
  double* d_norms = nullptr;
  std::vector<cudaEvent_t> events;
  auto new_event = [&]() { cudaEvent_t e = nullptr; cudaEventCreateWithFlags(&e, cudaEventDisableTiming); events.push_back(e); return e; };
  auto cleanup = [&]() {
    for (cudaEvent_t e : events) if (e) cudaEventDestroy(e);
    cudaFree(d_ovl); cudaFree(d_norms); cudaFree(d_div); cudaFree(d_fid);
  };
  CK(cudaMalloc(&d_ovl, sizeof(cplx) * (size_t)Nt * Nt));
  CK(cudaMalloc(&d_norms, sizeof(double) * Nt));
  CK(cudaMalloc(&d_div, sizeof(cplx) * Nt));
  CK(cudaMalloc(&d_fid, sizeof(cplx) * Nt));
  CK(cudaMemset(d_ovl, 0, sizeof(cplx) * (size_t)Nt * Nt));
  CK(cudaMemset(d_norms, 0, sizeof(double) * Nt));
  CK(cudaStreamSynchronize(cudaStreamLegacy));
  std::vector<cudaEvent_t> ev_psi(Nt, nullptr), ev_xi(Nt, nullptr), ev_xiH;
  if (do_psi) for (int i = 0; i < Nt; ++i) ev_psi[i] = new_event();
  if (do_xi) for (int i = 0; i < Nt; ++i) ev_xi[i] = new_event();
  struct ChainEv { std::vector<cudaEvent_t> ready, freed; };
  std::vector<ChainEv> cev(nchains);
  for (int c = 0; c < nchains; ++c)
    for (int m = 0; m < NCH; ++m) { cev[c].ready.push_back(new_event()); cev[c].freed.push_back(new_event()); }

  // Work queue (the reference's mutex-guarded row counter, src/OptimalControl.cpp:305-335): rows sorted by decreasing
  // length; a chain that has enqueued the last step of its row takes the next row of the queue.  All chains advance one
  // step per pass of the loop below, and so do the two sweeps and the K.xi chains, so no stream is ever given work
  // whose prerequisites have not been enqueued yet.
  std::vector<int> order(rows, rows + nrows);
  std::sort(order.begin(), order.end());
  // A closed chunk waits in `pending` until its overlap pass can be enqueued: the pass has to wait for the events of the
  // K.xi chains, and a stream can only wait for an event that has already been recorded (enqueued) on the host side.
  struct Pending { int row, j0, filled, m; };
  struct ChainState {
    int row = -1; int j = 0; long long chunk = 0; int filled = 0; int j0 = 0; bool xiH_waited = false;
    long long flushed = 0;                     // chunks whose overlap pass has been enqueued
    std::vector<Pending> pending;
  };
  std::vector<ChainState> cs(nchains);
  int next_row = 0;
  int psi_done = do_psi ? -1 : Nt - 1;      // last psi slice whose store has been enqueued
  int xi_next = Nt - 1;                      // next xi slice to be produced (counting down); -1: sweep enqueued
  int kxi_next = Nt - 1;                     // next K.xi slice to enqueue (counting down, the order the xi sweep produces them)
  bool xiH_recorded = !do_xiH;
  auto fail_out = [&](int code) { sync_all(); cleanup(); return code; };
  // development trace (OCMPS_HESSIAN_TRACE=1): when the sweeps, the K.xi store and everything finished, on the device clock
  static const bool trace = [] { const char* e = getenv("OCMPS_HESSIAN_TRACE"); return e && e[0] == '1'; }();
  cudaEvent_t tr[4] = {nullptr, nullptr, nullptr, nullptr};
  const auto host_t0 = std::chrono::steady_clock::now();
  double host_enq_ms = 0.0;
  if (trace) { for (auto& e : tr) cudaEventCreate(&e); cudaEventRecord(tr[0], wP->stream); }

  // enqueues the overlap passes of the closed chunks of chain c (K.xi slices j0 .. j0+filled-1 against the chunk) on the
  // chain's overlap stream -- possible once the events of the K.xi chains exist
  auto flush_pending = [&](int c) -> int {
    ChainState& S = cs[c];
    Workspace* ws = wss[c];
    if (!xiH_recorded) return OCMPS_OK;
    for (const Pending& P : S.pending) {
      cudaStreamWaitEvent(ws->ovl, cev[c].ready[P.m], 0);
      if (!S.xiH_waited) {
        for (cudaEvent_t e : ev_xiH) cudaStreamWaitEvent(ws->ovl, e, 0);
        S.xiH_waited = true;
      }
      const char* skip_env = getenv("OCMPS_HESSIAN_SKIP_OVL");          // timing experiments only: the Hessian is wrong without the overlaps
      const bool skip_ovl = skip_env && skip_env[0] == '1';
      int lrc = skip_ovl ? OCMPS_OK : overlaps_async(ws, side_of_store(xiH_store, P.j0), xiH_store->lay, side_of_store(ws->rowstore, P.m * CH), ws->rowstore->lay,
                               P.filled, 0, ws->ovl);
      if (lrc) return lrc;
      if (cudaMemcpyAsync(d_ovl + (size_t)P.row * Nt + P.j0, ws->d_out, sizeof(cplx) * P.filled, cudaMemcpyDeviceToDevice, ws->ovl) != cudaSuccess)
        return fail(OCMPS_ERR_CUDA, "cudaMemcpyAsync failed");
      cudaEventRecord(cev[c].freed[P.m], ws->ovl);
      ++S.flushed;
    }
    S.pending.clear();
    return OCMPS_OK;
  };
  // closes the open chunk of chain c
  auto close_chunk = [&](int c) -> int {
    ChainState& S = cs[c];
    Workspace* ws = wss[c];
    const int m = (int)(S.chunk % NCH);
    if (cudaEventRecord(cev[c].ready[m], ws->stream) != cudaSuccess) return fail(OCMPS_ERR_CUDA, "cudaEventRecord failed");
    S.pending.push_back({S.row, S.j0, S.filled, m});
    ++S.chunk;
    S.j0 += S.filled;
    S.filled = 0;
    return flush_pending(c);
  };
  // slot of the ring the next slice of chain c goes to, or -1 if the chain has to pause (on the host side only): the first
  // slice of a chunk waits until the overlaps that read the chunk's previous contents are done, which requires that pass
  // to have been enqueued
  auto next_slot = [&](int c) -> int {
    ChainState& S = cs[c];
    const int m = (int)(S.chunk % NCH);
    if (S.filled == 0 && S.chunk >= NCH) {
      if (S.flushed < S.chunk - NCH + 1) return -1;
      cudaStreamWaitEvent(wss[c]->stream, cev[c].freed[m], 0);
    }
    return m * CH + S.filled;
  };

  if (do_psi) {
    rc = sweep_enqueue_init(st, wP, psi_init, psi_store, 0);
    if (rc) return fail_out(rc);
    cudaEventRecord(ev_psi[0], wP->stream);
    psi_done = 0;
  }
  if (do_xi) {
    rc = sweep_enqueue_init(st, wX, psi_target, xi_store, Nt - 1);
    if (rc) return fail_out(rc);
    cudaEventRecord(ev_xi[Nt - 1], wX->stream);
    // the xi sweep (:393-407) has no prerequisites: all of it goes to its stream right away (a graph launch per step)
    for (int i = Nt - 1; i > 0; --i) {
      rc = step_enqueue(st, wX->work, wX, u[i], u[i - 1], false, xi_store, i - 1, wX->stream);
      if (rc) return fail_out(rc);
      cudaEventRecord(ev_xi[i - 1], wX->stream);
    }
  }
  xi_next = -1;
  bool busy = true;
  while (busy) {
    busy = false;
    if (do_psi && psi_done < Nt - 1) {                      // one psi step (:376-390)
      const int i = psi_done;
      rc = step_enqueue(st, wP->work, wP, u[i], u[i + 1], true, psi_store, i + 1, wP->stream);
      if (rc) return fail_out(rc);
      cudaEventRecord(ev_psi[i + 1], wP->stream);
      psi_done = i + 1;
      busy = true;
    }
    for (int rep = 0; rep < 2 && do_xiH && kxi_next >= 0 && kxi_next > xi_next; ++rep) {    // K|xi_i> (:300-303), once the slice has been enqueued
      const int i = kxi_next;
      Workspace* ws = wK[i % NK];
      if (ev_xi[i]) cudaStreamWaitEvent(ws->stream, ev_xi[i], 0);
      rc = store_get_async(xi_store, i, ws->work, ws->stream);
      if (!rc) rc = apply_K_async(st, ws, ws->work, ws->tmpK, ws->stream);
      if (!rc) rc = store_put_async(xiH_store, i, ws->tmpK, ws->stream);
      if (rc) return fail_out(rc);
      --kxi_next;
      busy = true;
      if (kxi_next < 0) {
        for (int k = 0; k < NK; ++k) { cudaEvent_t e = new_event(); cudaEventRecord(e, wK[k]->stream); ev_xiH.push_back(e); }
        xiH_recorded = true;
        for (int c = 0; c < nchains; ++c) { rc = flush_pending(c); if (rc) return fail_out(rc); }
      }
    }
    for (int c = 0; c < nchains; ++c) {
      ChainState& S = cs[c];
      Workspace* ws = wss[c];
      if (S.row < 0) {
        if (next_row >= nrows) continue;
        if (order[next_row] > psi_done) { busy = true; continue; }     // its psi slice has not been enqueued yet
        if (S.chunk >= NCH && S.flushed < S.chunk - NCH + 1) { busy = true; continue; }   // ring full until the K.xi events exist
        S.row = order[next_row++];
        // psiH = K|psi_row> and its norm (src/OptimalControl.cpp:256-257); the state itself is the first slice of the row
        if (ev_psi[S.row]) cudaStreamWaitEvent(ws->stream, ev_psi[S.row], 0);
        rc = store_get_async(psi_store, S.row, ws->work, ws->stream);
        if (!rc) rc = apply_K_async(st, ws, ws->work, psiH[c], ws->stream);
        if (rc) return fail_out(rc);
        launch_norm_only(psiH[c]->site(0), psiH[c]->dim(0), psiH[c]->dim(1), st->D, ws->db.partial, d_norms + S.row, 0, ws->stream);
        g_ocmps_launches += 2;
        S.j = S.row; S.j0 = S.row; S.filled = 0;
        rc = store_put_async(ws->rowstore, next_slot(c), psiH[c], ws->stream);
        if (rc) return fail_out(rc);
        ++S.filled;
        if (S.filled == CH || S.j == Nt - 2) { rc = close_chunk(c); if (rc) return fail_out(rc); }
        if (S.j == Nt - 2) S.row = -1;
        ++S.j;
        busy = true;
      } else {
        // one step forward (:267-277); the slice goes to the chain's ring
        const int slot = next_slot(c);
        if (slot < 0) { busy = true; continue; }
        rc = step_enqueue(st, psiH[c], ws, u[S.j - 1], u[S.j], true, ws->rowstore, slot, ws->stream);
        if (rc) return fail_out(rc);
        ++S.filled;
        if (S.filled == CH || S.j == Nt - 2) { rc = close_chunk(c); if (rc) return fail_out(rc); }
        if (S.j == Nt - 2) S.row = -1;
        ++S.j;
        busy = true;
      }
    }
    if (next_row < nrows) busy = true;
  }
  if (trace) {
    cudaEventRecord(tr[1], wP->stream);
    cudaEventRecord(tr[2], wX->stream);
    if (NK > 0) cudaEventRecord(tr[3], wK[0]->stream);
    host_enq_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - host_t0).count();
  }
  // tails of the sweep streams: fidelity overlaps <target|psi_i> (:242,450) and divT_i = <xi_i|K|psi_i> (:410-419)
  if (fid) {
    for (int z0 = 0; z0 < Nt; z0 += OB) {
      const int nb = std::min(OB, Nt - z0);
      rc = overlaps_async(wP, side_of_mps(psi_target), psi_target->lay, side_of_store(psi_store, z0), psi_store->lay, nb, 0, wP->stream);
      if (rc) return fail_out(rc);
      cudaMemcpyAsync(d_fid + z0, wP->d_out, sizeof(cplx) * nb, cudaMemcpyDeviceToDevice, wP->stream);
    }
  }
  if (divT) {
    if (do_psi) cudaStreamWaitEvent(wX->stream, ev_psi[Nt - 1], 0);
    for (int z0 = 0; z0 < Nt; z0 += OB) {
      const int nb = std::min(OB, Nt - z0);
      rc = overlaps_async(wX, side_of_store(xi_store, z0), xi_store->lay, side_of_store(psi_store, z0), psi_store->lay, nb, 1, wX->stream);
      if (rc) return fail_out(rc);
      cudaMemcpyAsync(d_div + z0, wX->d_out, sizeof(cplx) * nb, cudaMemcpyDeviceToDevice, wX->stream);
    }
  }
  sync_all();
  if (trace) {
    const double host_all_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - host_t0).count();
    float a = 0.f, bq = 0.f, c = 0.f;
    cudaEventElapsedTime(&a, tr[0], tr[1]);
    cudaEventElapsedTime(&bq, tr[0], tr[2]);
    if (NK > 0) cudaEventElapsedTime(&c, tr[0], tr[3]);
    fprintf(stderr, "[ocmps hessian] rows %d chains %d ring %dx%d | host: enqueue %.1f ms, all done %.1f ms | device: psi sweep %.1f ms, xi sweep %.1f ms, "
                    "K.xi chain 0 %.1f ms\n", nrows, nchains, NCH, CH, host_enq_ms, host_all_ms, a, bq, c);
    for (auto& e : tr) cudaEventDestroy(e);
  }
  cudaMemcpy(ovl, d_ovl, sizeof(cplx) * (size_t)Nt * Nt, cudaMemcpyDeviceToHost);
  cudaMemcpy(norms, d_norms, sizeof(double) * Nt, cudaMemcpyDeviceToHost);
  if (divT) cudaMemcpy(divT, d_div, sizeof(cplx) * Nt, cudaMemcpyDeviceToHost);
  if (fid) cudaMemcpy(fid, d_fid, sizeof(cplx) * Nt, cudaMemcpyDeviceToHost);
  cleanup();
  return lease.finish();
}

int ocmps_hessian_rows(ocmps_stepper* st, ocmps_store* psi_store, ocmps_store* xiH_store, const double* u, int Nt, const int* rows,
                       int nrows, int nchains, double* ovl, double* norms) {
  return hessian_run(st, nullptr, nullptr, u, Nt, psi_store, nullptr, xiH_store, rows, nrows, nchains, 0, 0, 0, nullptr, nullptr, ovl, norms);
}

int ocmps_hessian_eval(ocmps_stepper* st, ocmps_mps* psi_init, ocmps_mps* psi_target, const double* u, int Nt, ocmps_store* psi_store,
                       ocmps_store* xi_store, ocmps_store* xiH_store, const int* rows, int nrows, int nchains, int do_psi, int do_xi,
                       double* divT, double* fid, double* ovl, double* norms) {
  if (!psi_target || !divT || !fid) return fail(OCMPS_ERR_INVALID, "null argument");
  return hessian_run(st, psi_init, psi_target, u, Nt, psi_store, xi_store, xiH_store, rows, nrows, nchains, do_psi ? 1 : 0, do_xi ? 1 : 0, 1,
                     divT, fid, ovl, norms);
}

}  // extern "C"
