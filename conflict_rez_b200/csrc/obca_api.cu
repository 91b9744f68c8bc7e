// obca_api.cu -- C ABI (include/obca.h) around the per-instance solver of obca_core.h.
//
// Built by nvcc for sm_100a into libobca_b200.so (the product).  The same file compiles with
// g++ -DOBCA_HOST_EMU into the developer-only single-thread emulation (tools/host_emu), where a
// "device pointer" is a host pointer and a "kernel" is a loop over the instances.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <string>
#include <unordered_set>
#include <vector>

#include "obca_core.h"

using namespace obca;

#ifndef OBCA_HOST_EMU
#include <cuda_runtime.h>
#ifndef CTA_THREADS
#define CTA_THREADS 256
#endif
#ifndef CTAS_PER_SM
#define CTAS_PER_SM 1   // 2 was measured slower (128-register cap, 4 null-space warps, L1 squeezed): 68.9 vs 99.6 solves/s
#endif
#define NWARPS OBCA_NS_WARPS  // warps that own a null-space work area
#else
#define NWARPS 1
#endif

static thread_local std::string g_err;
static int fail(const std::string& msg) {
  g_err = msg;
  return -1;
}

struct ObcaHandle {
  ObcaDims dims;
  Opts opts;
  double dmin, shrink, rho;
  Lay L;
  Stat S;
  Counts cnt;
  int device;
  int slots;
  bool have_static;
  size_t it_stride, wk_stride, rw_stride, ric_stride;  // rw: shared-memory arena, ric: global Riccati arena (0 = the Riccati phase lives in the shared arena)
  // device memory
  Lay* d_L;
  Stat* d_S;
  double* d_tube;
  double *d_xL, *d_xU;
  unsigned char* d_bcls;  // [nx + 16] bound class of every variable (obca_ipm.h BoundCls)
  double blo[8], bhi[8];
  double* d_iter;  // [B][it_stride]
  double* d_work;  // [slots][wk_stride]
  double* d_rw;    // [slots][rw_stride]
  Result* d_res;   // [B]
  int* d_counter;
  int* d_order;    // [B] processing order of the instances (longest expected first), or identity
  bool have_order;
  long long* d_prof;  // [slots][NPROF + 1]
  int64_t launches;
  double* d_hist;       // iteration record [B][hist_cap][OBCA_HIST_FIELDS] (obca_set_history), nullptr: off
  int32_t* d_hist_cnt;  // [B]
  int hist_cap;
};

// Every entry point that touches the device runs on the handle's device and restores the caller's current device
// afterwards (a process may hold handles on several GPUs, and torch keeps its own notion of the current device).
struct DeviceGuard {
#ifndef OBCA_HOST_EMU
  int prev = -1;
  bool switched = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DeviceGuard() {
    if (switched) cudaSetDevice(prev);
  }
#else
  explicit DeviceGuard(int) {}
#endif
};

// ------------------------------------------------------------------------------------------------
// memory helpers
// ------------------------------------------------------------------------------------------------
#ifdef OBCA_HOST_EMU
static int dev_alloc(void** p, size_t bytes) {
  *p = calloc(bytes ? bytes : 1, 1);
  return *p ? 0 : -1;
}
static void dev_free(void* p) { free(p); }
static int h2d(void* d, const void* h, size_t n) {
  memcpy(d, h, n);
  return 0;
}
static int d2h(void* h, const void* d, size_t n) {
  memcpy(h, d, n);
  return 0;
}
static int dev_sync() { return 0; }
#else
#define CUDA_OK(call)                                                             \
  do {                                                                            \
    cudaError_t e_ = (call);                                                      \
    if (e_ != cudaSuccess) return fail(std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)
// Handles come and go (the warm-start pipeline creates one per agent and stage, each with gigabytes of iterates for a 4096 batch), and
// cudaMalloc / cudaFree of such buffers cost ~0.3 s per handle.  The buffers therefore come from the device's stream-ordered memory pool
// with the release threshold lifted: a freed buffer stays in the pool and the next handle reuses it without a driver round trip.
static std::mutex g_pool_mu;
static std::unordered_set<void*> g_pool_ptrs;  // pointers that came from cudaMallocAsync (the others from the cudaMalloc fallback)
static int dev_alloc(void** p, size_t bytes) {
  static bool pool_ready[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    if (dev >= 0 && dev < 64 && !pool_ready[dev]) {
      cudaMemPool_t pool;
      if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        unsigned long long thr = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
      }
      pool_ready[dev] = true;
    }
  }
  const size_t n = bytes ? bytes : 1;
  if (cudaMallocAsync(p, n, 0) == cudaSuccess) {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    g_pool_ptrs.insert(*p);
  } else {
    cudaGetLastError();
    if (cudaMalloc(p, n) != cudaSuccess) return -1;
  }
  if (cudaMemsetAsync(*p, 0, n, 0) != cudaSuccess) return -1;
  return cudaStreamSynchronize(0) == cudaSuccess ? 0 : -1;  // usable from every stream afterwards
}
static void dev_free(void* p) {
  if (!p) return;
  bool pooled;
  {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    pooled = g_pool_ptrs.erase(p) > 0;
  }
  if (pooled) cudaFreeAsync(p, 0);  // free_device synchronises the device before the first free of a handle
  else cudaFree(p);
}
static int h2d(void* d, const void* h, size_t n) { return cudaMemcpy(d, h, n, cudaMemcpyHostToDevice) == cudaSuccess ? 0 : -1; }
static int d2h(void* h, const void* d, size_t n) { return cudaMemcpy(h, d, n, cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : -1; }
static int dev_sync() { return cudaDeviceSynchronize() == cudaSuccess ? 0 : -1; }
#endif

// ------------------------------------------------------------------------------------------------
// kernels (device) / loops (emulation)
// ------------------------------------------------------------------------------------------------
struct PackArgs {
  const double *z, *lam, *mu, *dt, *pl, *pm, *ps;
  double *oz, *olam, *omu, *odt, *opl, *opm, *ops;
};

// node-major user arrays <-> field-major internal x.  One "thread" per (instance, element).
OBCA_HDN void pack_one(const Lay& L, double* iter, size_t it_stride, const PackArgs& A, int b, int e, bool unpack) {
  Scratch W;
  carve_iterate(W, L, iter + (size_t)b * it_stride);
  const int Mv = L.Mv, O = L.O;
  int nz = L.V * Mv * NZ, nl = L.V * Mv * O * 4, npl = L.P * Mv * 4, nps = L.P * Mv * 2;
  if (e < nz) {
    int a = e / (Mv * NZ), n = (e / NZ) % Mv, c = e % NZ;
    size_t src = (size_t)b * nz + e;
    if (unpack) {
      if (A.oz) A.oz[src] = n < L.M[a] ? W.x[L.Z(a, c, n)] : 0.0;
    } else
      W.x[L.Z(a, c, n)] = n < L.M[a] ? A.z[src] : 0.0;
    return;
  }
  e -= nz;
  if (e < nl) {
    int a = e / (Mv * O * 4), n = (e / (O * 4)) % Mv, j = (e / 4) % O, r = e % 4;
    size_t src = (size_t)b * nl + e;
    if (unpack) {
      if (A.olam) A.olam[src] = n < L.M[a] ? W.x[L.LAM(a, j, r, n)] : 0.0;
      if (A.omu) A.omu[src] = n < L.M[a] ? W.x[L.MU(a, j, r, n)] : 0.0;
    } else {
      W.x[L.LAM(a, j, r, n)] = n < L.M[a] ? A.lam[src] : 0.0;
      W.x[L.MU(a, j, r, n)] = n < L.M[a] ? A.mu[src] : 0.0;
    }
    return;
  }
  e -= nl;
  if (e < npl) {
    int p = e / (Mv * 4), n = (e / 4) % Mv, r = e % 4;
    size_t src = (size_t)b * npl + e;
    if (unpack) {
      if (A.opl) A.opl[src] = n < L.Mp[p] ? W.x[L.PL(p, r, n)] : 0.0;
      if (A.opm) A.opm[src] = n < L.Mp[p] ? W.x[L.PM(p, r, n)] : 0.0;
    } else {
      W.x[L.PL(p, r, n)] = (A.pl && n < L.Mp[p]) ? A.pl[src] : 0.0;
      W.x[L.PM(p, r, n)] = (A.pm && n < L.Mp[p]) ? A.pm[src] : 0.0;
    }
    return;
  }
  e -= npl;
  if (e < nps) {
    int p = e / (Mv * 2), n = (e / 2) % Mv, r = e % 2;
    size_t src = (size_t)b * nps + e;
    if (unpack) {
      if (A.ops) A.ops[src] = n < L.Mp[p] ? W.x[L.PS(p, r, n)] : 0.0;
    } else
      W.x[L.PS(p, r, n)] = (A.ps && n < L.Mp[p]) ? A.ps[src] : 0.0;
    return;
  }
  e -= nps;
  if (e == 0) {
    if (unpack) {
      if (A.odt) A.odt[b] = W.x[L.oDT];
    } else
      W.x[L.oDT] = A.dt[b];
  }
}
static inline int pack_elems(const Lay& L) { return L.V * L.Mv * NZ + L.V * L.Mv * L.O * 4 + L.P * L.Mv * 4 + L.P * L.Mv * 2 + 1; }

struct SolveArgs {
  const Lay* L;
  const Stat* S;
  Opts o;
  Counts cnt;
  const double *xL, *xU;
  const unsigned char* bcls;
  double blo[8], bhi[8];
  double *iter, *work, *rw;
  size_t it_stride, wk_stride, rw_stride, ric_stride;
  Result* res;
  int B;
  int* counter;
  const int* order;  // instance processed by the k-th pull of the work counter (nullptr: k itself)
  long long* prof;
  // debug modes: 0 = solve, 1 = eval at stored iterate, 2 = Newton step at stored iterate
  int mode, b_only;
  int rw_in_smem;  // Riccati work arena in dynamic shared memory (else per-slot global memory)
  int hist_cap;
  // The debug modes do not record and the solve has no debug arguments: the two share their slot, so that the iteration record
  // leaves the kernel's parameter block (and the stack frame k_solve copies it to) at its size.
  union {
    struct {
      double dbg_mu, dbg_dw;
    };
    struct {
      double* hist;         // mode 0: iteration record [B][hist_cap][OBCA_HIST_FIELDS], NaN-filled before the launch; nullptr: off
      int32_t* hist_count;  // mode 0: [B] heads evaluated per instance
    };
  };
};

OBCA_HDN void run_instance(const Ctx& ctx, const SolveArgs& A, const Lay& L, const Stat& S, int b, int slot, Shared* sh, double* RW) {
  Scratch W;
  carve_iterate(W, L, A.iter + (size_t)b * A.it_stride);
  carve_work(W, L, A.work + (size_t)slot * A.wk_stride);
  W.ricg = A.rw_in_smem ? nullptr : A.rw + (size_t)slot * A.ric_stride;
  if (A.mode == 0) {
    if (ctx.tid == 0) {  // read by the other threads only after the CTA barrier at the start of ipm_solve
      sh->hist = A.hist ? A.hist + (size_t)b * A.hist_cap * OBCA_HIST_FIELDS : nullptr;
      sh->hist_cap = A.hist_cap, sh->hist_n = 0, sh->hist_attempt = 0;
    }
    if (L.mode == 0) ipm_solve<0>(ctx, L, S, A.o, A.cnt, A.xL, A.xU, A.bcls, W, RW, A.rw_stride, sh, A.res + b);
    else ipm_solve<1>(ctx, L, S, A.o, A.cnt, A.xL, A.xU, A.bcls, W, RW, A.rw_stride, sh, A.res + b);
    if (ctx.tid == 0 && A.hist) A.hist_count[b] = sh->hist_n;
    return;
  }
  double f, gdt;
  for (int q = ctx.tid; q < L.nx; q += ctx.nt) W.gl[q] = 0, W.dx[q] = 0;
  for (int q = ctx.tid; q < L.ny; q += ctx.nt) W.c[q] = 0, W.dy[q] = 0;
  cta_sync(ctx);
  if (A.mode == 3 && L.mode != 0) return;
  if (L.mode == 0) eval_all(ctx, L, S, W, W.x, W.y, W.c, W.gl, &f, &gdt);
  else mpc_eval_all(ctx, L, S, W, W.x, W.y, W.c, W.gl, &f, &gdt);
  if (ctx.tid == 0) A.res[b].obj = f;
  if (A.mode == 2 || A.mode == 3) {
    double mu = A.dbg_mu, dw = A.dbg_dw;
    for (int q = ctx.tid; q < L.nx; q += ctx.nt) {
      double lo = A.xL[q], hi = A.xU[q];
      bool hl = lo > -INFINITY, hu = hi < INFINITY;
      double sg = dw, gp = W.gl[q];
      if (hl) {
        double g = W.x[q] - lo;
        sg += W.zL[q] / g, gp -= mu / g;
        if (!hu) gp += A.o.kappa_d * mu;
      }
      if (hu) {
        double g = hi - W.x[q];
        sg += W.zU[q] / g, gp += mu / g;
        if (!hl) gp -= A.o.kappa_d * mu;
      }
      W.sig[q] = sg, W.gphi[q] = gp;
    }
    cta_sync(ctx);
    if (A.mode == 3) {  // K [dx; dy]: inputs in W.dzU / W.ry, outputs in W.dzL / W.ct
      kkt_apply(ctx, L, S, W, W.dzU, W.ry, W.dzL, W.ct);
      return;
    }
    int ok = L.mode == 0 ? kkt_solve(ctx, L, S, W, RW, &sh->ok) : mpc_kkt_solve(ctx, L, S, W, RW, &sh->ok);
    double rr = 0;
    int nref = 0;
    if (ok && L.mode == 0 && A.o.refine_steps > 0) nref = kkt_refine(ctx, L, S, W, RW, &sh->ok, A.o.refine_steps, A.o.refine_ratio, &rr);
    if (ctx.tid == 0) A.res[b].status = ok, A.res[b].refines = nref, A.res[b].elastic = rr;
  }
}

#ifndef OBCA_HOST_EMU
__global__ void k_pack(const Lay* L, double* iter, size_t it_stride, PackArgs A, int B, int ne, bool unpack) {
  size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= (size_t)B * ne) return;
  pack_one(*L, iter, it_stride, A, (int)(g / ne), (int)(g % ne), unpack);
}
__global__ void k_init_pose(const Lay* L, double* iter, size_t it_stride, const double* pose, int B) {
  int g = blockIdx.x * blockDim.x + threadIdx.x;
  int per = L->V * 3;
  if (g >= B * per) return;
  Scratch W;
  carve_iterate(W, *L, iter + (size_t)(g / per) * it_stride);
  W.init_pose[g % per] = pose[g];
}
__global__ void __launch_bounds__(CTA_THREADS, CTAS_PER_SM) k_solve(SolveArgs A) {
  __shared__ Shared sh;
  __shared__ double red[40];
  __shared__ int cur;
  extern __shared__ __align__(16) double arena[];
  __shared__ Lay sL;
  __shared__ Stat sS;
  {
    const int* srcL = (const int*)A.L;
    int* dstL = (int*)&sL;
    for (int q = threadIdx.x; q < (int)(sizeof(Lay) / sizeof(int)); q += blockDim.x) dstL[q] = srcL[q];
    const double* srcS = (const double*)A.S;
    double* dstS = (double*)&sS;
    for (int q = threadIdx.x; q < (int)(sizeof(Stat) / sizeof(double)); q += blockDim.x) dstS[q] = srcS[q];
  }
  if (threadIdx.x < 8) sh.blo[threadIdx.x] = A.blo[threadIdx.x], sh.bhi[threadIdx.x] = A.bhi[threadIdx.x];
  __syncthreads();
  double* RW = arena;
  __shared__ LdlBuf sldl;
  Ctx ctx{(int)threadIdx.x, (int)blockDim.x, red, &sldl, A.prof ? A.prof + (size_t)blockIdx.x * (NPROF + 1) : nullptr};
  if (ctx.prof && threadIdx.x == 0) ctx.prof[NPROF] = clock64();
  if (A.mode != 0) {
    run_instance(ctx, A, sL, sS, A.b_only, 0, &sh, RW);
    return;
  }
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) cur = atomicAdd(A.counter, 1);
    __syncthreads();
    if (cur >= A.B) break;
    const int b = A.order ? A.order[cur] : cur;
    run_instance(ctx, A, sL, sS, b, blockIdx.x, &sh, RW);
  }
}
__global__ void k_stats(const Result* res, int B, int32_t* status, int32_t* iters, double* obj, double* cviol, double* dual_inf, double* compl_inf, double* elastic) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  if (status) status[b] = res[b].status;
  if (iters) iters[b] = res[b].iters;
  if (obj) obj[b] = res[b].obj;
  if (cviol) cviol[b] = res[b].cviol;
  if (dual_inf) dual_inf[b] = res[b].dual_inf;
  if (compl_inf) compl_inf[b] = res[b].compl_inf;
  if (elastic) elastic[b] = res[b].elastic;
}
#endif

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

const char* obca_version(void) {
#ifdef OBCA_HOST_EMU
  return "obca-b200 0.1.0 (HOST EMULATION - developer tool, not the product)";
#else
#define OBCA_STR2(x) #x
#define OBCA_STR(x) OBCA_STR2(x)
  return "obca-b200 0.1.0 (sm_100a, " OBCA_STR(CTA_THREADS) " threads x " OBCA_STR(CTAS_PER_SM) " CTA/SM)";
#endif
}
const char* obca_last_error(void) { return g_err.c_str(); }

void obca_default_options(ObcaOptions* o) {
  o->tol = 1e-2, o->constr_viol_tol = 1e-2, o->dual_inf_tol = 1.0, o->compl_inf_tol = 1e-4;
  o->mu_init = 0.1, o->dmin = 0.05, o->shrink_tube = 0.5, o->elastic_weight = 1e3, o->max_iter = 3000, o->refine_steps = -1;
}

static void apply_options(ObcaHandle* h, const ObcaOptions* o) {
  h->opts.tol = o->tol, h->opts.constr_viol_tol = o->constr_viol_tol, h->opts.dual_inf_tol = o->dual_inf_tol;
  h->opts.compl_inf_tol = o->compl_inf_tol, h->opts.mu_init = o->mu_init, h->opts.max_iter = o->max_iter;
  h->dmin = o->dmin, h->shrink = o->shrink_tube, h->rho = o->elastic_weight;
  h->opts.refine_steps = o->refine_steps >= 0 ? o->refine_steps : (o->tol > 1e-5 ? 0 : 2);
}

int obca_create(const ObcaDims* dims, const ObcaOptions* opts, int device, ObcaHandle** out) {
  if (!dims || !out) return fail("obca_create: null argument");
  if (dims->K != 5) return fail("obca_create: only K = 5 is supported");
  if (dims->O < 0 || dims->O > OBCA_MAX_O) return fail("obca_create: O out of range");
  if (dims->batch < 1) return fail("obca_create: bad batch");
  if (dims->mode == OBCA_MODE_MPC) {
    if (dims->horizon < 2 || dims->horizon > 4096) return fail("obca_create: MPC horizon out of range");
    if (dims->n_others < 0 || dims->n_others > MAXP) return fail("obca_create: n_others out of range");
  } else if (dims->mode == OBCA_MODE_STATE_WS) {
    if (dims->n_per_set < 1 || dims->n_sets[0] < 2 || dims->n_sets[0] > OBCA_MAX_SETS) return fail("obca_create: state_ws needs n_per_set >= 1 and 2 <= n_sets[0] <= 64");
    if (dims->n_per_set * (dims->n_sets[0] - 1) + 1 > 4096) return fail("obca_create: state_ws horizon out of range");
    if (dims->O != 0) return fail("obca_create: the state warm start has no obstacles (O must be 0)");
  } else if (dims->mode == OBCA_MODE_COLLOCATION) {
    if (dims->V < 1 || dims->V > OBCA_MAX_V) return fail("obca_create: V out of range");
    if (dims->n_per_set < 1) return fail("obca_create: bad n_per_set");
    for (int a = 0; a < dims->V; ++a)
      if (dims->n_sets[a] < 2 || dims->n_sets[a] > OBCA_MAX_SETS) return fail("obca_create: n_sets out of range");
  } else
    return fail("obca_create: unknown mode");
#ifndef OBCA_HOST_EMU
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail("obca_create: no CUDA device (this library has no CPU fallback)");
  if (device < 0 || device >= ndev) return fail("obca_create: bad device index");  // the caller's current device is left alone
#endif
  ObcaHandle* h = new ObcaHandle();
  memset((void*)h, 0, sizeof(*h));
  h->opts = Opts();
  h->dims = *dims;
  h->device = device;
  ObcaOptions o;
  obca_default_options(&o);
  apply_options(h, opts ? opts : &o);
  *out = h;
  return 0;
}

int obca_set_options(ObcaHandle* h, const ObcaOptions* opts) {
  if (!h || !opts) return fail("obca_set_options: null argument");
  bool geom = h->have_static && (opts->dmin != h->dmin || opts->shrink_tube != h->shrink || opts->elastic_weight != h->rho);
  if (geom) return fail("obca_set_options: dmin / shrink_tube / elastic_weight must be set before obca_set_static");
  apply_options(h, opts);
  return 0;
}

static void free_device(ObcaHandle* h) {
#ifndef OBCA_HOST_EMU
  if (h->d_iter || h->d_L) cudaDeviceSynchronize();  // kernels of this handle may still run on another stream: the frees below are stream ordered on stream 0
#endif
  dev_free(h->d_L), dev_free(h->d_S), dev_free(h->d_tube), dev_free(h->d_xL), dev_free(h->d_xU), dev_free(h->d_bcls);
  h->d_bcls = nullptr;
  dev_free(h->d_iter), dev_free(h->d_work), dev_free(h->d_rw), dev_free(h->d_res), dev_free(h->d_counter), dev_free(h->d_order), dev_free(h->d_prof);
  h->d_order = nullptr, h->have_order = false;
  h->d_prof = nullptr;
  h->d_L = nullptr, h->d_S = nullptr, h->d_tube = nullptr, h->d_xL = h->d_xU = nullptr;
  h->d_iter = h->d_work = h->d_rw = nullptr, h->d_res = nullptr, h->d_counter = nullptr;
}

static void free_history(ObcaHandle* h) {
  if (!h->d_hist) return;
  dev_sync();  // a solve on another stream may still write the record: the frees are stream ordered on stream 0
  dev_free(h->d_hist), dev_free(h->d_hist_cnt);
  h->d_hist = nullptr, h->d_hist_cnt = nullptr, h->hist_cap = 0;
}

int obca_destroy(ObcaHandle* h) {
  if (!h) return 0;
  DeviceGuard guard(h->device);
  free_history(h);
  free_device(h);
  delete h;
  return 0;
}

// collocation matrices from their definition (reference: confrez/control/vehicle.py:54-97); the Radau
// points are the roots of P_5 - P_4 mapped to [0,1] (CasADi's collocation_points(5, "radau")).
static void collocation_matrices(double cA[NK][NK], double cB[NK]) {
  const double tau[NK] = {0.0, 0.05710419611451768, 0.27684301363812383, 0.5835904323689168, 0.8602401356562194, 1.0};
  for (int j = 0; j < NK; ++j) {
    // Lagrange basis polynomial j as monomial coefficients p[0] + p[1] t + ...
    double p[NK + 1] = {1, 0, 0, 0, 0, 0, 0};
    int deg = 0;
    for (int k = 0; k < NK; ++k) {
      if (k == j) continue;
      double sc = 1.0 / (tau[j] - tau[k]);
      double q[NK + 1] = {0, 0, 0, 0, 0, 0, 0};
      for (int m = 0; m <= deg; ++m) q[m + 1] += p[m] * sc, q[m] -= p[m] * tau[k] * sc;
      ++deg;
      for (int m = 0; m <= deg; ++m) p[m] = q[m];
    }
    for (int k = 0; k < NK; ++k) {
      double d = 0, tp = 1.0;
      for (int m = 1; m <= deg; ++m) d += m * p[m] * tp, tp *= tau[k];
      cA[j][k] = d;
    }
    double integ = 0;
    for (int m = 0; m <= deg; ++m) integ += p[m] / (m + 1);
    cB[j] = integ;
  }
}

int obca_set_static(ObcaHandle* h, const ObcaStatic* st) {
  if (!h || !st) return fail("obca_set_static: null argument");
  DeviceGuard guard(h->device);
  free_device(h);
  const bool sws = h->dims.mode == OBCA_MODE_STATE_WS;
  const bool mpc = h->dims.mode == OBCA_MODE_MPC || sws;  // the state warm start shares the MPC layout and kernels (obca_mpc.h)
  if (sws) lay_build_state_ws(h->L, h->dims.n_sets[0], h->dims.n_per_set, h->dims.bounded_input != 0, st->final_heading && st->final_heading[0] == st->final_heading[0]);
  else if (mpc) lay_build_mpc(h->L, h->dims.horizon, h->dims.O, h->dims.n_others);
  else lay_build(h->L, h->dims, st->final_heading);
  Lay& L = h->L;
  Stat& S = h->S;
  memset((void*)&S, 0, sizeof(S));
  for (int j = 0; j < L.O; ++j)
    for (int r = 0; r < 4; ++r) {
      S.obsA[j][r][0] = st->obs_A[(j * 4 + r) * 2], S.obsA[j][r][1] = st->obs_A[(j * 4 + r) * 2 + 1];
      S.obsb[j][r] = st->obs_b[j * 4 + r];
    }
  for (int r = 0; r < 4; ++r) S.G[r][0] = st->body_G[2 * r], S.G[r][1] = st->body_G[2 * r + 1], S.g[r] = st->body_g[r];
  S.wb = st->wb, S.dmin = h->dmin, S.rho = h->rho, S.dt_mpc = st->mpc_dt;
  for (int q = 0; q < 4; ++q) S.region[q] = st->region[q];
  for (int q = 0; q < 8; ++q) S.limits[q] = st->limits[q];
  for (int a = 0; a < L.V; ++a) S.heading[a] = (mpc && !sws) ? 0.0 : (L.heading[a] ? st->final_heading[a] : 0.0);
  collocation_matrices(S.cA, S.cB);
  if (st->colloc_A && st->colloc_B && !mpc)  // the caller's constants (the reference builds them with numpy poly1d arithmetic): bit-identical parity
    for (int j = 0; j < NK; ++j) {
      for (int k = 0; k < NK; ++k) S.cA[j][k] = st->colloc_A[j * NK + k];
      S.cB[j] = st->colloc_B[j];
    }
  {
    // inverse of A1[k][j] = cA[j][k] (j, k = 1..K) by Gauss-Jordan with partial pivoting: the interior collocation block
    double M[5][10];
    for (int k = 0; k < 5; ++k)
      for (int j = 0; j < 5; ++j) M[k][j] = S.cA[j + 1][k + 1], M[k][5 + j] = (k == j) ? 1.0 : 0.0;
    for (int c = 0; c < 5; ++c) {
      int pr = c;
      for (int r = c + 1; r < 5; ++r)
        if (fabs(M[r][c]) > fabs(M[pr][c])) pr = r;
      for (int q = 0; q < 10; ++q) std::swap(M[c][q], M[pr][q]);
      const double ip = 1.0 / M[c][c];
      for (int q = 0; q < 10; ++q) M[c][q] *= ip;
      for (int r = 0; r < 5; ++r) {
        if (r == c) continue;
        const double f = M[r][c];
        for (int q = 0; q < 10; ++q) M[r][q] -= f * M[c][q];
      }
    }
    for (int j = 0; j < 5; ++j)
      for (int k = 0; k < 5; ++k) S.cAi[j][k] = M[j][5 + k];  // (A1^-1)[j][k]: x_j = sum_k cAi[j][k] rhs_k
  }
  std::vector<double> tube((size_t)L.V * L.Smax * 2 * 4 * 3);
  for (int a = 0; a < L.V && (!mpc || sws); ++a)
    for (int q = 0; q < L.Smax; ++q)
      for (int body = 0; body < 2; ++body)
        for (int r = 0; r < 4; ++r) {
          size_t src = (((size_t)a * L.Smax + q) * 2 + body) * 4 + r;
          tube[src * 3 + 0] = st->tube_A[src * 2], tube[src * 3 + 1] = st->tube_A[src * 2 + 1];
          tube[src * 3 + 2] = st->tube_b[src] - h->shrink;
        }
  // bounds
  std::vector<double> xL(L.nx, -INFINITY), xU(L.nx, INFINITY);
  const double lo[NZ] = {S.region[0], S.region[2], -INFINITY, S.limits[0], S.limits[2], S.limits[4], S.limits[6]};
  const double hi[NZ] = {S.region[1], S.region[3], INFINITY, S.limits[1], S.limits[3], S.limits[5], S.limits[7]};
  int nb = 0, m_active = 0;
  for (int a = 0; a < L.V; ++a) {
    for (int n = 0; n < L.M[a]; ++n) {
      for (int c = 0; c < NZ; ++c) xL[L.Z(a, c, n)] = lo[c], xU[L.Z(a, c, n)] = hi[c];
      for (int j = 0; j < L.O; ++j) {
        for (int r = 0; r < 4; ++r) xL[L.LAM(a, j, r, n)] = 0, xL[L.MU(a, j, r, n)] = 0;
        xL[L.SD(a, j, n)] = 0, xL[L.EL(a, j, n)] = 0;
      }
    }
    for (int q = 0; q < L.S[a] - 1; ++q)
      for (int r = 0; r < 8; ++r) xL[L.TS(a, q, r)] = 0;
    if (sws) {
      // vehicle.py:140-167: bounds at k < N M only, input bounds only with bounded_input
      for (int c = 0; c < NZ; ++c) xL[L.Z(a, c, L.M[a] - 1)] = -INFINITY, xU[L.Z(a, c, L.M[a] - 1)] = INFINITY;
      if (L.euler != 2)
        for (int n = 0; n < L.M[a]; ++n)
          for (int c = 5; c < NZ; ++c) xL[L.Z(a, c, n)] = -INFINITY, xU[L.Z(a, c, n)] = INFINITY;
      m_active += 7 + 5 * (L.M[a] - 1) + 8 * (L.S[a] - 1) + L.heading[a];
    } else if (mpc) m_active += 5 + 5 * (L.M[a] - 1) + 4 * L.O * L.M[a];
    else m_active += 7 + 5 * L.M[a] + 7 * (L.N[a] - 1) + 4 + L.heading[a] + 4 * L.O * L.M[a] + 8 * (L.S[a] - 1);
  }
  for (int p = 0; p < L.P; ++p) {
    for (int n = 0; n < L.Mp[p]; ++n) {
      for (int r = 0; r < 4; ++r) xL[L.PL(p, r, n)] = 0, xL[L.PM(p, r, n)] = 0;
      xL[L.PSD(p, n)] = 0, xL[L.PSN(p, n)] = 0, xL[L.PEL(p, n)] = 0;
    }
    m_active += 6 * L.Mp[p];
  }
  for (int q = 0; q < L.nx; ++q) nb += (xL[q] > -INFINITY) + (xU[q] < INFINITY);
  // bound classes: 0 free, 1 lower bound 0, 2..7 the two-sided bounds of x, y, v, delta, a, w
  std::vector<unsigned char> bcls(L.nx + 16, 0);
  {
    const int zc[NZ] = {2, 3, 0, 4, 5, 6, 7};
    for (int k = 0; k < 8; ++k) h->blo[k] = -INFINITY, h->bhi[k] = INFINITY;
    h->blo[1] = 0.0;
    for (int c = 0; c < NZ; ++c)
      if (zc[c]) h->blo[zc[c]] = lo[c], h->bhi[zc[c]] = hi[c];
    for (int q = 0; q < L.nx; ++q) {
      int k = -1;
      for (int kk = 0; kk < 8 && k < 0; ++kk)
        if (xL[q] == h->blo[kk] && xU[q] == h->bhi[kk]) k = kk;
      if (k < 0) return fail("obca_set_static: internal error (a variable's bounds match no bound class)");
      bcls[q] = (unsigned char)k;
    }
  }
  h->cnt.m_active = m_active, h->cnt.nb = nb;
  h->it_stride = iterate_doubles(L), h->wk_stride = work_doubles(L);
  h->rw_stride = mpc ? mpc_work_doubles(L) : riccati_work_doubles(L, NWARPS);
  h->ric_stride = 0;
#ifndef OBCA_HOST_EMU
  const size_t smem_cap = (size_t)(CTAS_PER_SM == 1 ? 200 : 100) * 1024;
  if (mpc && h->rw_stride * sizeof(double) > smem_cap) {
    // long horizons (the 271-node state warm start): the stage buffers of the MPC-mode solve live in a per-slot global arena;
    // the shared arena only stages the flat passes
    h->ric_stride = h->rw_stride;
    h->rw_stride = 1024;
  }
  if (!mpc && h->rw_stride * sizeof(double) > smem_cap) {
    // more than 4 vehicles: the stage matrices of the joint Riccati state (7 V + 1) do not fit next to the null-space work areas;
    // the Riccati phase then runs from a per-slot arena in global memory (L2 resident), everything else keeps the shared arena
    h->ric_stride = riccati_only_doubles(L);
    h->rw_stride = (size_t)NWARPS * NSW;
  }
  if (h->rw_stride * sizeof(double) > smem_cap)
    return fail("obca_set_static: the shared-memory work arena of this problem shape exceeds 200 KB");
#endif
#ifdef OBCA_HOST_EMU
  h->slots = 1;
#else
  cudaDeviceProp prop;
  CUDA_OK(cudaGetDeviceProperties(&prop, h->device));
  h->slots = CTAS_PER_SM * prop.multiProcessorCount < h->dims.batch ? CTAS_PER_SM * prop.multiProcessorCount : h->dims.batch;
#endif
  int B = h->dims.batch;
  if (dev_alloc((void**)&h->d_L, sizeof(Lay)) || dev_alloc((void**)&h->d_S, sizeof(Stat)) || dev_alloc((void**)&h->d_tube, tube.size() * 8) ||
      dev_alloc((void**)&h->d_bcls, bcls.size()) || dev_alloc((void**)&h->d_xL, (L.nx + 2) * 8) || dev_alloc((void**)&h->d_xU, (L.nx + 2) * 8) || dev_alloc((void**)&h->d_iter, (size_t)B * h->it_stride * 8) ||
      dev_alloc((void**)&h->d_work, (size_t)h->slots * h->wk_stride * 8) || dev_alloc((void**)&h->d_rw, (size_t)h->slots * (h->ric_stride ? h->ric_stride : h->rw_stride) * 8) ||
      dev_alloc((void**)&h->d_res, (size_t)B * sizeof(Result)) || dev_alloc((void**)&h->d_counter, sizeof(int)) || dev_alloc((void**)&h->d_order, (size_t)B * sizeof(int)) ||
      dev_alloc((void**)&h->d_prof, (size_t)h->slots * (NPROF + 1) * sizeof(long long)))
    return fail("obca_set_static: device allocation failed");
  S.tube = h->d_tube;
  h2d(h->d_tube, tube.data(), tube.size() * 8);
  h2d(h->d_L, &L, sizeof(Lay));
  h2d(h->d_S, &S, sizeof(Stat));
  h2d(h->d_bcls, bcls.data(), bcls.size());
  h2d(h->d_xL, xL.data(), L.nx * 8);
  h2d(h->d_xU, xU.data(), L.nx * 8);
  std::vector<Result> r0(B);
  for (auto& r : r0) memset(&r, 0, sizeof(r)), r.status = OBCA_NOT_SOLVED;
  h2d(h->d_res, r0.data(), B * sizeof(Result));
  h->have_static = true;
  return 0;
}

int obca_set_init_pose(ObcaHandle* h, const double* pose, void* stream) {
  if (!h || !h->have_static) return fail("obca_set_init_pose: call obca_set_static first");
  if (h->L.mode != 0) return fail("obca_set_init_pose: collocation mode only (use obca_set_mpc_params)");
  DeviceGuard guard(h->device);
  int B = h->dims.batch, per = h->L.V * 3;
#ifdef OBCA_HOST_EMU
  (void)stream;
  for (int g = 0; g < B * per; ++g) {
    Scratch W;
    carve_iterate(W, h->L, h->d_iter + (size_t)(g / per) * h->it_stride);
    W.init_pose[g % per] = pose[g];
  }
#else
  k_init_pose<<<(B * per + 255) / 256, 256, 0, (cudaStream_t)stream>>>(h->d_L, h->d_iter, h->it_stride, pose, B);
  h->launches++;
  CUDA_OK(cudaGetLastError());
#endif
  return 0;
}

#ifndef OBCA_HOST_EMU
__global__ void k_mpc_params(const Lay* L, double* iter, size_t it_stride, const double* cur, const double* ref, const double* others, int B) {
  const int N = L->Mv, P = L->P, per = 5 + 3 * N * (1 + P);
  size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= (size_t)B * per) return;
  int b = (int)(g / per), e = (int)(g % per);
  Scratch W;
  carve_iterate(W, *L, iter + (size_t)b * it_stride);
  double v;
  if (e < 5) v = cur[(size_t)b * 5 + e];
  else if (e < 5 + 3 * N) v = ref[(size_t)b * 3 * N + (e - 5)];
  else v = others[(size_t)b * 3 * N * P + (e - 5 - 3 * N)];
  W.init_pose[e] = v;
}
#endif

int obca_set_mpc_params(ObcaHandle* h, const double* cur, const double* ref, const double* others, void* stream) {
  if (!h || !h->have_static) return fail("obca_set_mpc_params: call obca_set_static first");
  if (h->L.mode != 1) return fail("obca_set_mpc_params: the handle was not created in MPC mode");
  if (!cur || !ref || (h->L.P > 0 && !others)) return fail("obca_set_mpc_params: null argument");
  DeviceGuard guard(h->device);
  const int B = h->dims.batch, N = h->L.Mv, P = h->L.P, per = 5 + 3 * N * (1 + P);
#ifdef OBCA_HOST_EMU
  (void)stream;
  for (int b = 0; b < B; ++b) {
    Scratch W;
    carve_iterate(W, h->L, h->d_iter + (size_t)b * h->it_stride);
    for (int e = 0; e < per; ++e)
      W.init_pose[e] = e < 5 ? cur[(size_t)b * 5 + e] : (e < 5 + 3 * N ? ref[(size_t)b * 3 * N + (e - 5)] : others[(size_t)b * 3 * N * P + (e - 5 - 3 * N)]);
  }
#else
  (void)per;
  size_t tot = (size_t)B * per;
  k_mpc_params<<<(unsigned)((tot + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->d_L, h->d_iter, h->it_stride, cur, ref, others, B);
  h->launches++;
  CUDA_OK(cudaGetLastError());
#endif
  return 0;
}

// ------------------------------------------------------------------------------------------------
// DFMA throughput of the device (the FP64 roofline denominator asked for in SURVEY.md 8d)
// ------------------------------------------------------------------------------------------------
#ifndef OBCA_HOST_EMU
__global__ void k_fp64_peak(double* out, int n) {
  double a0 = threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double b = 1.0000001, c = 1e-9;
  for (int i = 0; i < n; ++i) {
    a0 = fma(a0, b, c), a1 = fma(a1, b, c), a2 = fma(a2, b, c), a3 = fma(a3, b, c);
    a4 = fma(a4, b, c), a5 = fma(a5, b, c), a6 = fma(a6, b, c), a7 = fma(a7, b, c);
  }
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}
#endif

int obca_measure_dfma_peak(int device, double* tflops) {
  if (!tflops) return fail("obca_measure_dfma_peak: null argument");
#ifdef OBCA_HOST_EMU
  (void)device;
  *tflops = 0.0;
  return fail("obca_measure_dfma_peak: not available in the host emulation");
#else
  DeviceGuard guard(device);
  cudaDeviceProp prop;
  CUDA_OK(cudaGetDeviceProperties(&prop, device));
  const int blocks = prop.multiProcessorCount * 8, thr = 256, it = 1 << 14;
  double* out = nullptr;
  CUDA_OK(cudaMalloc(&out, (size_t)blocks * thr * sizeof(double)));
  cudaEvent_t e0, e1;
  CUDA_OK(cudaEventCreate(&e0));
  CUDA_OK(cudaEventCreate(&e1));
  float best = 1e30f;
  for (int rep = 0; rep < 4; ++rep) {  // first repetition warms up
    cudaEventRecord(e0);
    k_fp64_peak<<<blocks, thr>>>(out, it);
    cudaEventRecord(e1);
    CUDA_OK(cudaEventSynchronize(e1));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    if (rep > 0 && ms < best) best = ms;
  }
  cudaEventDestroy(e0), cudaEventDestroy(e1), cudaFree(out);
  *tflops = 2.0 * 8 * it * (double)blocks * thr / (best * 1e-3) / 1e12;
  return 0;
#endif
}

// ------------------------------------------------------------------------------------------------
// closed-form dual warm starts (obca_ws.h)
// ------------------------------------------------------------------------------------------------
#ifndef OBCA_HOST_EMU
__global__ void k_dual_ws(const Lay* L, const Stat* S, const double* z, double* lam, double* mu, size_t tot) {
  size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g < tot) ws_obstacle_item(*L, *S, z, lam, mu, g);
}
__global__ void k_joint_dual_ws(const Lay* L, const Stat* S, const double* z, double* pl, double* pm, double* ps, size_t tot) {
  size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g < tot) ws_pair_item(*L, *S, z, pl, pm, ps, g);
}
#endif

int obca_dual_ws(ObcaHandle* h, const double* z, double* lam, double* mu, void* stream) {
  if (!h || !h->have_static) return fail("obca_dual_ws: call obca_set_static first");
  if (!z || !lam || !mu) return fail("obca_dual_ws: null argument");
  DeviceGuard guard(h->device);
  const size_t tot = (size_t)h->dims.batch * h->L.V * h->L.Mv * h->L.O;
#ifdef OBCA_HOST_EMU
  (void)stream;
  for (size_t g = 0; g < tot; ++g) ws_obstacle_item(h->L, h->S, z, lam, mu, g);
#else
  if (tot) {
    k_dual_ws<<<(unsigned)((tot + 127) / 128), 128, 0, (cudaStream_t)stream>>>(h->d_L, h->d_S, z, lam, mu, tot);
    h->launches++;
    CUDA_OK(cudaGetLastError());
  }
#endif
  return 0;
}

int obca_joint_dual_ws(ObcaHandle* h, const double* z, double* pl, double* pm, double* ps, void* stream) {
  if (!h || !h->have_static) return fail("obca_joint_dual_ws: call obca_set_static first");
  if (h->L.mode != 0) return fail("obca_joint_dual_ws: collocation mode only");
  if (h->L.P == 0) return 0;
  if (!z || !pl || !pm || !ps) return fail("obca_joint_dual_ws: null argument");
  DeviceGuard guard(h->device);
  const size_t tot = (size_t)h->dims.batch * h->L.P * h->L.Mv;
#ifdef OBCA_HOST_EMU
  (void)stream;
  for (size_t g = 0; g < tot; ++g) ws_pair_item(h->L, h->S, z, pl, pm, ps, g);
#else
  k_joint_dual_ws<<<(unsigned)((tot + 127) / 128), 128, 0, (cudaStream_t)stream>>>(h->d_L, h->d_S, z, pl, pm, ps, tot);
  h->launches++;
  CUDA_OK(cudaGetLastError());
#endif
  return 0;
}

static int run_pack(ObcaHandle* h, const PackArgs& A, bool unpack, void* stream) {
  int B = h->dims.batch, ne = pack_elems(h->L);
  DeviceGuard guard(h->device);
#ifdef OBCA_HOST_EMU
  (void)stream;
  for (int b = 0; b < B; ++b)
    for (int e = 0; e < ne; ++e) pack_one(h->L, h->d_iter, h->it_stride, A, b, e, unpack);
#else
  size_t tot = (size_t)B * ne;
  k_pack<<<(unsigned)((tot + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->d_L, h->d_iter, h->it_stride, A, B, ne, unpack);
  h->launches++;
  CUDA_OK(cudaGetLastError());
#endif
  return 0;
}

int obca_set_initial(ObcaHandle* h, const double* z, const double* lam, const double* mu, const double* dt, const double* pl,
                     const double* pm, const double* ps, void* stream) {
  if (!h || !h->have_static) return fail("obca_set_initial: call obca_set_static first");
  if (!z || !dt || (h->L.O > 0 && (!lam || !mu))) return fail("obca_set_initial: z, lam, mu, dt are required");
  PackArgs A;
  memset(&A, 0, sizeof(A));
  A.z = z, A.lam = lam, A.mu = mu, A.dt = dt, A.pl = pl, A.pm = pm, A.ps = ps;
  return run_pack(h, A, false, stream);
}

int obca_get_solution(ObcaHandle* h, double* z, double* lam, double* mu, double* dt, double* pl, double* pm, double* ps, void* stream) {
  if (!h || !h->have_static) return fail("obca_get_solution: call obca_set_static first");
  PackArgs A;
  memset(&A, 0, sizeof(A));
  A.oz = z, A.olam = lam, A.omu = mu, A.odt = dt, A.opl = pl, A.opm = pm, A.ops = ps;
  return run_pack(h, A, true, stream);
}

static SolveArgs make_args(ObcaHandle* h, int mode, int b) {
  SolveArgs A;
  A.L = h->d_L, A.S = h->d_S, A.o = h->opts, A.cnt = h->cnt, A.xL = h->d_xL, A.xU = h->d_xU, A.bcls = h->d_bcls;
  for (int k = 0; k < 8; ++k) A.blo[k] = h->blo[k], A.bhi[k] = h->bhi[k];
  A.iter = h->d_iter, A.work = h->d_work, A.rw = h->d_rw;
  A.it_stride = h->it_stride, A.wk_stride = h->wk_stride, A.rw_stride = h->rw_stride, A.ric_stride = h->ric_stride;
  A.res = h->d_res, A.B = h->dims.batch, A.counter = h->d_counter, A.mode = mode, A.b_only = b;
  A.order = h->have_order ? h->d_order : nullptr;
  A.prof = getenv("OBCA_PROFILE") ? h->d_prof : nullptr;
  A.rw_in_smem = h->ric_stride == 0;
  A.hist_cap = h->hist_cap;
  if (mode == 0) A.hist = h->d_hist, A.hist_count = h->d_hist_cnt;
  else A.dbg_mu = 0, A.dbg_dw = 0;  // the debug entry points do not record
  return A;
}

static int launch(ObcaHandle* h, const SolveArgs& A, void* stream) {
  DeviceGuard guard(h->device);
#ifdef OBCA_HOST_EMU
  (void)stream;
  Shared sh;
  for (int k = 0; k < 8; ++k) sh.blo[k] = A.blo[k], sh.bhi[k] = A.bhi[k];
  double red[40];
  Ctx ctx{0, 1, red, nullptr, nullptr};
  if (A.mode == 0 && A.hist) memset(A.hist, 0xFF, (size_t)A.B * A.hist_cap * OBCA_HIST_FIELDS * sizeof(double));  // all-ones bytes: a NaN
  if (A.mode != 0)
    run_instance(ctx, A, *A.L, *A.S, A.b_only, 0, &sh, A.rw);
  else
    for (int b = 0; b < A.B; ++b) run_instance(ctx, A, *A.L, *A.S, b, 0, &sh, A.rw);
#else
  cudaStream_t s = (cudaStream_t)stream;
  if (A.mode == 0) CUDA_OK(cudaMemsetAsync(h->d_counter, 0, sizeof(int), s));
  // rows a solve does not reach read back as NaN (all-ones bytes), not as what the previous solve left there
  if (A.mode == 0 && A.hist) CUDA_OK(cudaMemsetAsync(A.hist, 0xFF, (size_t)A.B * A.hist_cap * OBCA_HIST_FIELDS * sizeof(double), s));
  int grid = A.mode == 0 ? h->slots : 1;
  size_t smem = h->rw_stride * sizeof(double);
  if (smem) CUDA_OK(cudaFuncSetAttribute(k_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_solve<<<grid, CTA_THREADS, smem, s>>>(A);
  h->launches++;
  CUDA_OK(cudaGetLastError());
#endif
  return 0;
}

// ------------------------------------------------------------------------------------------------
// trajectory-side kernels (obca_traj.h)
// ------------------------------------------------------------------------------------------------
#ifndef OBCA_HOST_EMU
struct InterpConst {
  int n_intervals[OBCA_MAX_V];
  double tau[NK];
};
__global__ void k_interpolate(InterpArgs A, InterpConst C, size_t tot) {
  size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= tot) return;
  A.n_intervals = C.n_intervals, A.tau = C.tau;
  interp_item(A, g);
}
__global__ void k_ref_times(const double* grid, const double* clock, int N, double dt_mpc, double* times, size_t tot) {
  size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= tot) return;
  const size_t v = g / N;
  const int k = (int)(g % N);
  times[g] = ref_window_start(grid[v * 3], grid[v * 3 + 1], (int)grid[v * 3 + 2], clock[v]) + k * dt_mpc;
}
__global__ void k_plant_step(const double* state, const double* input, int B, double dt, double wb, int substeps, double* next) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) plant_step(state + (size_t)b * 5, input + (size_t)b * 2, dt, wb, substeps, next + (size_t)b * 5);
}
__global__ void k_shift(const double* in, double* out, int N, int Wd, size_t tot) {
  size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g < tot) shift_item(in, out, N, Wd, g);
}
__global__ void k_ws_interp(const double* in, const double* t, InterpConst C6, int T, int C, int N, double* out, size_t tot) {
  size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g < tot) ws_interp_item(in, t, C6.tau, T, C, N, out, g);
}
static int check_device(int device) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail("no CUDA device (this library has no CPU fallback)");
  if (device < 0 || device >= ndev) return fail("bad device index");
  return 0;
}
#else
static int check_device(int) { return 0; }
#endif

int obca_interpolate(int device, const double* z, const double* dt, const int32_t* n_intervals, const double* tau, int B, int V, int Mmax,
                     const double* times, int T, int per_vehicle_times, int dt_per_vehicle, double* out, void* stream) {
  if (!z || !dt || !n_intervals || !tau || !times || !out) return fail("obca_interpolate: null argument");
  if (B < 1 || V < 1 || V > OBCA_MAX_V || T < 1) return fail("obca_interpolate: bad dimensions");
  for (int a = 0; a < V; ++a)
    if (n_intervals[a] < 1 || n_intervals[a] * NK > Mmax) return fail("obca_interpolate: n_intervals does not fit Mmax");
  if (check_device(device)) return -1;
  DeviceGuard guard(device);
  InterpArgs A;
  A.z = z, A.dt = dt, A.times = times, A.out = out, A.B = B, A.V = V, A.Mmax = Mmax, A.T = T, A.per_vehicle_times = per_vehicle_times, A.dt_per_vehicle = dt_per_vehicle;
  const size_t tot = (size_t)B * V * T;
#ifdef OBCA_HOST_EMU
  (void)stream;
  A.n_intervals = n_intervals, A.tau = tau;
  for (size_t g = 0; g < tot; ++g) interp_item(A, g);
#else
  InterpConst C;
  for (int a = 0; a < V; ++a) C.n_intervals[a] = n_intervals[a];
  for (int k = 0; k < NK; ++k) C.tau[k] = tau[k];
  A.n_intervals = nullptr, A.tau = nullptr;
  k_interpolate<<<(unsigned)((tot + 127) / 128), 128, 0, (cudaStream_t)stream>>>(A, C, tot);
  CUDA_OK(cudaGetLastError());
#endif
  return 0;
}

int obca_interp_ws(int device, const double* in, const double* t, const double* tau, int B, int T, int C, int N, double* out, void* stream) {
  if (!in || !t || !tau || !out) return fail("obca_interp_ws: null argument");
  if (B < 1 || T < 2 || C < 1 || N < 1) return fail("obca_interp_ws: bad dimensions");
  if (check_device(device)) return -1;
  DeviceGuard guard(device);
  const size_t tot = (size_t)B * N * NK * C;
#ifdef OBCA_HOST_EMU
  (void)stream;
  for (size_t g = 0; g < tot; ++g) ws_interp_item(in, t, tau, T, C, N, out, g);
#else
  InterpConst C6;
  for (int a = 0; a < OBCA_MAX_V; ++a) C6.n_intervals[a] = 0;
  for (int k = 0; k < NK; ++k) C6.tau[k] = tau[k];
  k_ws_interp<<<(unsigned)((tot + 127) / 128), 128, 0, (cudaStream_t)stream>>>(in, t, C6, T, C, N, out, tot);
  CUDA_OK(cudaGetLastError());
#endif
  return 0;
}

int obca_mpc_ref_times(int device, const double* grid, const double* clock, int B, int V, int N, double dt_mpc, double* times, void* stream) {
  if (!grid || !clock || !times || B < 1 || V < 1 || N < 1) return fail("obca_mpc_ref_times: bad argument");
  if (check_device(device)) return -1;
  DeviceGuard guard(device);
  const size_t tot = (size_t)B * V * N;
#ifdef OBCA_HOST_EMU
  (void)stream;
  for (size_t g = 0; g < tot; ++g) {
    const size_t v = g / N;
    times[g] = ref_window_start(grid[v * 3], grid[v * 3 + 1], (int)grid[v * 3 + 2], clock[v]) + (int)(g % N) * dt_mpc;
  }
#else
  k_ref_times<<<(unsigned)((tot + 127) / 128), 128, 0, (cudaStream_t)stream>>>(grid, clock, N, dt_mpc, times, tot);
  CUDA_OK(cudaGetLastError());
#endif
  return 0;
}

int obca_plant_step(int device, const double* state, const double* input, int B, double dt, double wb, int substeps, double* next, void* stream) {
  if (!state || !input || !next || B < 1 || substeps < 1) return fail("obca_plant_step: bad argument");
  if (check_device(device)) return -1;
  DeviceGuard guard(device);
#ifdef OBCA_HOST_EMU
  (void)stream;
  for (int b = 0; b < B; ++b) plant_step(state + (size_t)b * 5, input + (size_t)b * 2, dt, wb, substeps, next + (size_t)b * 5);
#else
  k_plant_step<<<(B + 63) / 64, 64, 0, (cudaStream_t)stream>>>(state, input, B, dt, wb, substeps, next);
  CUDA_OK(cudaGetLastError());
#endif
  return 0;
}

int obca_shift_horizon(int device, const double* in, int B, int N, int Wd, double* out, void* stream) {
  if (!in || !out || B < 1 || N < 1 || Wd < 1 || in == out) return fail("obca_shift_horizon: bad argument");
  if (check_device(device)) return -1;
  DeviceGuard guard(device);
  const size_t tot = (size_t)B * N * Wd;
#ifdef OBCA_HOST_EMU
  (void)stream;
  for (size_t g = 0; g < tot; ++g) shift_item(in, out, N, Wd, g);
#else
  k_shift<<<(unsigned)((tot + 127) / 128), 128, 0, (cudaStream_t)stream>>>(in, out, N, Wd, tot);
  CUDA_OK(cudaGetLastError());
#endif
  return 0;
}

int obca_set_order(ObcaHandle* h, const int32_t* order_dev, void* stream) {
  if (!h || !h->have_static) return fail("obca_set_order: call obca_set_static first");
  DeviceGuard guard(h->device);
  if (!order_dev) {
    h->have_order = false;
    return 0;
  }
#ifdef OBCA_HOST_EMU
  (void)stream;
  memcpy(h->d_order, order_dev, (size_t)h->dims.batch * sizeof(int));
#else
  CUDA_OK(cudaMemcpyAsync(h->d_order, order_dev, (size_t)h->dims.batch * sizeof(int), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
#endif
  h->have_order = true;
  return 0;
}

int obca_solve(ObcaHandle* h, void* stream) {
  if (!h || !h->have_static) return fail("obca_solve: call obca_set_static first");
  return launch(h, make_args(h, 0, 0), stream);
}

int obca_set_history(ObcaHandle* h, int32_t capacity) {
  if (!h) return fail("obca_set_history: null handle");
  if (capacity < 0) return fail("obca_set_history: capacity must be >= 0");
  DeviceGuard guard(h->device);
  free_history(h);
  if (capacity == 0) return 0;
  const size_t B = (size_t)h->dims.batch;
  if (dev_alloc((void**)&h->d_hist, B * capacity * OBCA_HIST_FIELDS * sizeof(double)) || dev_alloc((void**)&h->d_hist_cnt, B * sizeof(int32_t))) {
    dev_free(h->d_hist);
    h->d_hist = nullptr, h->d_hist_cnt = nullptr;
    return fail("obca_set_history: device allocation failed");
  }
  h->hist_cap = capacity;
  return 0;
}

int obca_get_history(ObcaHandle* h, double* rows, int32_t* count, void* stream) {
  if (!h || !h->d_hist) return fail("obca_get_history: recording is off (call obca_set_history with a capacity > 0 before obca_solve)");
  DeviceGuard guard(h->device);
  const size_t B = (size_t)h->dims.batch, nrow = B * h->hist_cap * OBCA_HIST_FIELDS * sizeof(double);
#ifdef OBCA_HOST_EMU
  (void)stream;
  if (rows) memcpy(rows, h->d_hist, nrow);
  if (count) memcpy(count, h->d_hist_cnt, B * sizeof(int32_t));
#else
  if (rows) CUDA_OK(cudaMemcpyAsync(rows, h->d_hist, nrow, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  if (count) CUDA_OK(cudaMemcpyAsync(count, h->d_hist_cnt, B * sizeof(int32_t), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
#endif
  return 0;
}

int obca_get_stats(ObcaHandle* h, int32_t* status, int32_t* iters, double* obj, double* cviol, double* dual_inf, double* compl_inf, double* elastic,
                   void* stream) {
  if (!h || !h->have_static) return fail("obca_get_stats: call obca_set_static first");
  DeviceGuard guard(h->device);
  int B = h->dims.batch;
#ifdef OBCA_HOST_EMU
  (void)stream;
  for (int b = 0; b < B; ++b) {
    const Result& r = h->d_res[b];
    if (status) status[b] = r.status;
    if (iters) iters[b] = r.iters;
    if (obj) obj[b] = r.obj;
    if (cviol) cviol[b] = r.cviol;
    if (dual_inf) dual_inf[b] = r.dual_inf;
    if (compl_inf) compl_inf[b] = r.compl_inf;
    if (elastic) elastic[b] = r.elastic;
  }
#else
  k_stats<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->d_res, B, status, iters, obj, cviol, dual_inf, compl_inf, elastic);
  h->launches++;
  CUDA_OK(cudaGetLastError());
#endif
  return 0;
}

int64_t obca_launch_count(const ObcaHandle* h) { return h ? h->launches : 0; }

int obca_debug_profile(ObcaHandle* h, int64_t* out, int n) {
  if (!h || !h->have_static) return fail("obca_debug_profile: call obca_set_static first");
  DeviceGuard guard(h->device);
  if (dev_sync()) return fail("device sync failed");
  std::vector<long long> buf((size_t)h->slots * (NPROF + 1));
  d2h(buf.data(), h->d_prof, buf.size() * sizeof(long long));
  for (int i = 0; i < n && i < NPROF; ++i) {
    out[i] = 0;
    for (int s = 0; s < h->slots; ++s) out[i] += buf[(size_t)s * (NPROF + 1) + i];
  }
  return NPROF;
}

int obca_layout(const ObcaHandle* h, int64_t* out, int n) {
  if (!h || !h->have_static) return fail("obca_layout: call obca_set_static first");
  const Lay& L = h->L;
  const int64_t v[] = {L.V,    L.O,    L.P,    L.Mv,     L.Nmax,  L.Smax,   L.nx,     L.ny,    L.oZ,     L.oLAM,  L.oMU,
                       L.oSD,  L.oEL,  L.oTS,  L.oPL,  L.oPM,    L.oPS,   L.oPSD,   L.oPSN,   L.oPEL,  L.oDT,   L.oYINIT, L.oYCOL, L.oYCONT,
                       L.oYTERM, L.oYOBS, L.oYTUBE, L.oYPAIR, h->cnt.m_active, h->cnt.nb};
  int cntv = (int)(sizeof(v) / sizeof(v[0]));
  for (int i = 0; i < n && i < cntv; ++i) out[i] = v[i];
  return cntv;
}

int obca_debug_get_iterate(ObcaHandle* h, int b, double* x, double* y, double* zL, double* zU) {
  if (!h || !h->have_static || b < 0 || b >= h->dims.batch) return fail("obca_debug_get_iterate: bad argument");
  DeviceGuard guard(h->device);
  if (dev_sync()) return fail("device sync failed");
  Scratch W;
  carve_iterate(W, h->L, h->d_iter + (size_t)b * h->it_stride);
  if (x) d2h(x, W.x, h->L.nx * 8);
  if (y) d2h(y, W.y, h->L.ny * 8);
  if (zL) d2h(zL, W.zL, h->L.nx * 8);
  if (zU) d2h(zU, W.zU, h->L.nx * 8);
  return 0;
}

int obca_debug_set_iterate(ObcaHandle* h, int b, const double* x, const double* y, const double* zL, const double* zU) {
  if (!h || !h->have_static || b < 0 || b >= h->dims.batch) return fail("obca_debug_set_iterate: bad argument");
  DeviceGuard guard(h->device);
  Scratch W;
  carve_iterate(W, h->L, h->d_iter + (size_t)b * h->it_stride);
  if (x) h2d(W.x, x, h->L.nx * 8);
  if (y) h2d(W.y, y, h->L.ny * 8);
  if (zL) h2d(W.zL, zL, h->L.nx * 8);
  if (zU) h2d(W.zU, zU, h->L.nx * 8);
  return 0;
}

int obca_debug_eval(ObcaHandle* h, int b, double* c, double* gl, double* f) {
  if (!h || !h->have_static || b < 0 || b >= h->dims.batch) return fail("obca_debug_eval: bad argument");
  DeviceGuard guard(h->device);
  if (launch(h, make_args(h, 1, b), nullptr)) return -1;
  if (dev_sync()) return fail("obca_debug_eval: kernel failed");
  Scratch W;
  carve_work(W, h->L, h->d_work);
  if (c) d2h(c, W.c, h->L.ny * 8);
  if (gl) d2h(gl, W.gl, h->L.nx * 8);
  Result r;
  d2h(&r, h->d_res + b, sizeof(r));
  if (f) *f = r.obj;
  return 0;
}

int obca_debug_step(ObcaHandle* h, int b, double mu, double delta_w, double* dx, double* dy, int32_t* ok) {
  if (!h || !h->have_static || b < 0 || b >= h->dims.batch) return fail("obca_debug_step: bad argument");
  DeviceGuard guard(h->device);
  SolveArgs A = make_args(h, 2, b);
  A.dbg_mu = mu, A.dbg_dw = delta_w;
  if (launch(h, A, nullptr)) return -1;
  if (dev_sync()) return fail("obca_debug_step: kernel failed");
  Scratch W;
  carve_work(W, h->L, h->d_work);
  if (dx) d2h(dx, W.dx, h->L.nx * 8);
  if (dy) d2h(dy, W.dy, h->L.ny * 8);
  Result r;
  d2h(&r, h->d_res + b, sizeof(r));
  if (ok) *ok = r.status;
  return 0;
}

int obca_debug_kkt_apply(ObcaHandle* h, int b, double delta_w, const double* dx, const double* dy, double* r1, double* r2) {
  if (!h || !h->have_static || b < 0 || b >= h->dims.batch || !dx || !dy) return fail("obca_debug_kkt_apply: bad argument");
  if (h->L.mode != 0) return fail("obca_debug_kkt_apply: collocation mode only");
  DeviceGuard guard(h->device);
  Scratch W;
  carve_work(W, h->L, h->d_work);
  h2d(W.dzU, dx, h->L.nx * 8);
  h2d(W.ry, dy, h->L.ny * 8);
  SolveArgs A = make_args(h, 3, b);
  A.dbg_mu = 0, A.dbg_dw = delta_w;
  if (launch(h, A, nullptr)) return -1;
  if (dev_sync()) return fail("obca_debug_kkt_apply: kernel failed");
  if (r1) d2h(r1, W.dzL, h->L.nx * 8);
  if (r2) d2h(r2, W.ct, h->L.ny * 8);
  return 0;
}

}  // extern "C"
