// obca_ipm.h -- [IPM] per-instance primal-dual interior-point loop (IPM specification in DESIGN.md;
// the CPU restatement used by the parity tests is oracle/ipm.py).
#pragma once

namespace obca {

constexpr int VW = 8;  // elements per thread and batch in the flat passes: enough independent loads in flight to cover DRAM latency


struct Shared {   // lives in shared memory on the device
  int ok;      // kkt_solve: inertia / factorisation flag (must be followed by `again`)
  int again;   // interval_nullspace: another pass needed
  int filt_n;
  double filt_theta[FILTER_MAX], filt_phi[FILTER_MAX];
  unsigned long long bars[8];  // mbarriers of the staged flat passes
  double blo[8], bhi[8];       // bounds of the 8 bound classes (see BoundCls)
  // iteration record (obca_set_history).  `hist` is set per instance before ipm_solve and read by every thread (it decides the
  // extra reduction of d_norm); the rest is thread 0's bookkeeping, kept here rather than in registers of the hot loop
  double* hist;          // rows of the current instance [hist_cap][OBCA_HIST_FIELDS], nullptr: not recording
  int hist_cap, hist_n;  // capacity, heads evaluated so far
  int hist_attempt;      // interior-point run of this instance (ipm_solve restarts)
  int hist_trials, hist_flags;
  double hist_dw, hist_dn;  // delta_w and max |dx| of the current step
  int hist_warm;            // the next head is the first of a warm-started attempt
  int warm;                 // Result::warm of the current instance, set by thread 0 in ipm_solve, cleared after the first attempt
};

// Row of the current head: fields 0..8 and 15, field 14 (flags) so far; the step fields stay NaN until hist_step.  Thread 0.
OBCA_HD void hist_head(Shared* sh, int it, double f, double cviol, double theta, double dual_inf, double compl0, double mu, double E0,
                       bool acceptable, double rho) {
  const int k = sh->hist_n++;
  sh->hist_flags = (acceptable ? OBCA_HIST_F_ACCEPTABLE : 0) | (sh->hist_warm ? OBCA_HIST_F_WARM : 0), sh->hist_trials = 0;
  sh->hist_warm = 0;
  if (k >= sh->hist_cap) return;
  double* r = sh->hist + (size_t)k * OBCA_HIST_FIELDS;
  r[OBCA_HIST_ITER] = it, r[OBCA_HIST_ATTEMPT] = sh->hist_attempt, r[OBCA_HIST_OBJ] = f, r[OBCA_HIST_INF_PR] = cviol, r[OBCA_HIST_THETA] = theta;
  r[OBCA_HIST_INF_DU] = dual_inf, r[OBCA_HIST_COMPL] = compl0, r[OBCA_HIST_MU] = mu, r[OBCA_HIST_ERR] = E0;
  r[OBCA_HIST_FLAGS] = sh->hist_flags, r[OBCA_HIST_RHO] = rho;
}
// Step fields of the current head's row, when its iteration ends (accepted step or barrier reset).  Thread 0.
OBCA_HD void hist_step(Shared* sh, double alpha_pr, double alpha_du, int flags) {
  const int k = sh->hist_n - 1;
  if (k >= sh->hist_cap) return;
  double* r = sh->hist + (size_t)k * OBCA_HIST_FIELDS;
  r[OBCA_HIST_REG] = sh->hist_dw, r[OBCA_HIST_D_NORM] = sh->hist_dn, r[OBCA_HIST_ALPHA_PR] = alpha_pr, r[OBCA_HIST_ALPHA_DU] = alpha_du;
  r[OBCA_HIST_LS_TRIALS] = sh->hist_trials;
  r[OBCA_HIST_FLAGS] = sh->hist_flags | flags | (sh->hist_dw > 0 ? OBCA_HIST_F_INERTIA : 0);
}

// Simple bounds by class instead of two FP64 vectors: one byte per variable.  Class 0: free, 1: lower bound 0 (duals, slacks,
// elastic variables), 2..7: the two-sided bounds of x, y, v, delta, a, w.  The flat passes stage the class bytes next to the
// vectors (1 KB per tile instead of 16 KB for xL and xU): a third less traffic in the passes over the primal vectors.
struct BoundCls {
  const unsigned char* cls;  // [nx], padded to a multiple of 16
  const double *lo, *hi;     // [8] in shared memory
};

struct Counts {
  int m_active;   // number of equality rows
  int nb;         // number of finite bounds
};

OBCA_HD bool finite_d(double v) { return v - v == 0.0; }

// ------------------------------------------------------------------------------------------------
// Flat passes over the primal-dual vectors.  The vectors of one instance (n ~ 9e4 doubles each) live in HBM; a pass
// reads NA of them once.  With 8 warps per SM plain loads cannot keep enough bytes in flight to cover the DRAM latency,
// so on the device the pass is staged: one thread issues 1-D bulk copies (TMA, cp.async.bulk) of the next tiles into the
// shared-memory arena (free outside the KKT solve) while the CTA works on the current tile; completion is tracked by
// mbarriers.  `body(q, v)` receives the NA loaded values of element q and writes its results straight to global memory.
// ------------------------------------------------------------------------------------------------
#ifndef OBCA_ST_TILE
#define OBCA_ST_TILE 1024
#endif
constexpr int ST_TILE = OBCA_ST_TILE;  // elements per tile (4 per thread)
constexpr int ST_STAGES_MAX = 8;

struct Stage {
  double* buf;              // shared-memory arena (nullptr: no staging)
  size_t cap;               // doubles available in it
  unsigned long long* bar;  // ST_STAGES mbarriers in shared memory
};

#if defined(__CUDA_ARCH__)
__device__ __forceinline__ unsigned st_smem(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void st_wait(unsigned long long* bar, unsigned parity) {
  unsigned done = 0;
  const unsigned a = st_smem(bar);
  while (!done)
    asm volatile("{\n\t.reg .pred P1;\n\tmbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\tselp.b32 %0, 1, 0, P1;\n\t}" : "=r"(done) : "r"(a), "r"(parity) : "memory");
}
#endif

// CLS: the class byte of every element is staged too and body(q, v, lo, hi) receives its bounds
template <int NA, bool CLS, class Body>
OBCA_HD void flat_pass_impl(const Ctx& ctx, const Stage& st, const BoundCls* bc, const double* const (&src)[NA], int n, Body&& body) {
#if defined(__CUDA_ARCH__)
  constexpr int TILE_D = NA * ST_TILE + (CLS ? ST_TILE / 8 : 0);  // doubles per stage buffer
  // ring depth 3: measured, a deeper ring (up to 8 tiles in flight) is 8 % slower -- the passes are bound by the FP64 instruction
  // latency of the bodies at 2 warps per scheduler, not by bytes in flight.  Also measured and
  // dropped: a warp-uniform fast path for tiles of plain non-negative variables (constant bounds, the four elements of a thread as one
  // straight-line block): 5.98 vs 5.90 M cycles per iteration, no gain (profiles/r02h_phase_cycles_flat_fast_path_rejected.txt); per-stage
  // "empty" mbarriers instead of the CTA barrier after every tile (warps drifting by a tile): +60 k cycles (profiles/r02n_*)
  const int ST_STAGES = st.cap / TILE_D >= 3 ? 3 : 0;
  if (st.buf && ST_STAGES >= 3 && n >= 4 * ST_TILE && ctx.nt * 4 == ST_TILE) {
    const int ntile = (n + ST_TILE - 1) / ST_TILE;
    if (ctx.tid == 0) {
      for (int k = 0; k < ST_STAGES; ++k) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(st_smem(st.bar + k)) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // earlier generic-proxy accesses of the arena (every thread's own, by the phases before this pass) vs the bulk copies issued
    // below: each thread fences its accesses, the barrier hands them to the issuing thread
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    auto issue = [&](int t) {
      const int stage = t % ST_STAGES, start = t * ST_TILE;
      const int cnt = n - start < ST_TILE ? n - start : ST_TILE;
      const unsigned bytes = (unsigned)(((cnt + 1) & ~1) * 8);
      const unsigned cbytes = CLS ? (unsigned)((cnt + 15) & ~15) : 0u;
      const unsigned bar = st_smem(st.bar + stage);
      double* sb = st.buf + (size_t)stage * TILE_D;
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes * NA + cbytes) : "memory");
#pragma unroll
      for (int a = 0; a < NA; ++a)
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(st_smem(sb + (size_t)a * ST_TILE)),
                     "l"(src[a] + start), "r"(bytes), "r"(bar)
                     : "memory");
      if (CLS)
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(st_smem(sb + (size_t)NA * ST_TILE)),
                     "l"(bc->cls + start), "r"(cbytes), "r"(bar)
                     : "memory");
    };
    if (ctx.tid == 0)
      for (int t = 0; t < ST_STAGES - 1 && t < ntile; ++t) issue(t);
    for (int t = 0; t < ntile; ++t) {
      if (ctx.tid == 0 && t + ST_STAGES - 1 < ntile) issue(t + ST_STAGES - 1);  // its stage was released by the barrier below
      st_wait(st.bar + t % ST_STAGES, (unsigned)((t / ST_STAGES) & 1));
      const double* tb = st.buf + (size_t)(t % ST_STAGES) * TILE_D;
      const unsigned char* cb = (const unsigned char*)(tb + (size_t)NA * ST_TILE);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = ctx.tid + u * ctx.nt, q = t * ST_TILE + e;
        if (q < n) {
          double v[NA];
#pragma unroll
          for (int a = 0; a < NA; ++a) v[a] = tb[a * ST_TILE + e];
          if constexpr (CLS) {
            const int k = cb[e];
            body(q, v, bc->lo[k], bc->hi[k]);
          } else
            body(q, v, 0.0, 0.0);
        }
      }
      __syncthreads();
    }
    if (ctx.tid == 0)
      for (int k = 0; k < ST_STAGES; ++k) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(st_smem(st.bar + k)) : "memory");
    __syncthreads();
    return;
  }
#endif
  (void)st;
  for (int q0 = ctx.tid; q0 < n; q0 += VW * ctx.nt) {
    double v[VW][NA];
    int kc[VW];
#pragma unroll
    for (int u = 0; u < VW; ++u) {
      const int q = q0 + u * ctx.nt;
#pragma unroll
      for (int a = 0; a < NA; ++a) v[u][a] = q < n ? src[a][q] : 0.0;
      kc[u] = (CLS && q < n) ? bc->cls[q] : 0;
    }
#pragma unroll
    for (int u = 0; u < VW; ++u) {
      const int q = q0 + u * ctx.nt;
      if (q < n) {
        if constexpr (CLS) body(q, v[u], bc->lo[kc[u]], bc->hi[kc[u]]);
        else body(q, v[u], 0.0, 0.0);
      }
    }
  }
}

template <int NA, class Body>
OBCA_HD void flat_pass(const Ctx& ctx, const Stage& st, const double* const (&src)[NA], int n, Body&& body) {
  flat_pass_impl<NA, false>(ctx, st, nullptr, src, n, [&](int q, const double* v, double, double) { body(q, v); });
}
template <int NA, class Body>
OBCA_HD void flat_pass_b(const Ctx& ctx, const Stage& st, const BoundCls& bc, const double* const (&src)[NA], int n, Body&& body) {
  flat_pass_impl<NA, true>(ctx, st, &bc, src, n, body);
}

// model dispatch: MODE 0 = collocation OBCA (obca_core.h / obca_kkt.h), MODE 1 = MPC (obca_mpc.h)
template <int MODE>
OBCA_HD void model_eval(const Ctx& ctx, const Lay& L, const Stat& S, const Scratch& W, const double* x, const double* y, double* c, double* gl,
                        double* f, double* gdt) {
  if (MODE == 0) eval_all(ctx, L, S, W, x, y, c, gl, f, gdt);
  else mpc_eval_all(ctx, L, S, W, x, y, c, gl, f, gdt);
}
template <int MODE>
OBCA_HD int model_kkt(const Ctx& ctx, const Lay& L, const Stat& S, const Scratch& W, double* RW, int* ok) {
  if (MODE == 0) return kkt_solve(ctx, L, S, W, RW, ok);
  return mpc_kkt_solve(ctx, L, S, W, RW, ok);
}

// slack <- value of its inequality body, evaluated with slack and elastic variable at zero; on the elastic rows the
// negative part of the body goes to the elastic variable, so that the row starts feasible (oracle/nlp.py:init_slacks)
template <int MODE>
OBCA_HDN void init_slacks(const Ctx& ctx, const Lay& L, const Stat& S, const Scratch& W) {
  for (int it = ctx.tid; it < L.V * L.O * L.Mv; it += ctx.nt) W.x[L.oSD + it] = 0, W.x[L.oEL + it] = 0;
  for (int it = ctx.tid; it < L.V * (L.Smax - 1) * 8; it += ctx.nt) W.x[L.oTS + it] = 0;
  for (int it = ctx.tid; it < L.P * L.Mv; it += ctx.nt) W.x[L.oPSD + it] = 0, W.x[L.oPSN + it] = 0, W.x[L.oPEL + it] = 0;
  cta_sync(ctx);
  double f, gdt;
  model_eval<MODE>(ctx, L, S, W, W.x, nullptr, W.c, nullptr, &f, &gdt);
  for (int it = ctx.tid; it < L.V * L.O * L.Mv; it += ctx.nt) {
    int n = it % L.Mv, aj = it / L.Mv, a = aj / L.O, j = aj % L.O;
    if (n < L.M[a]) {
      double body = W.c[L.YOBS(a, j, 0, n)];
      W.x[L.SD(a, j, n)] = body > 0 ? body : 0.0;
      W.x[L.EL(a, j, n)] = body < 0 ? -body : 0.0;
    }
  }
  for (int it = ctx.tid; it < L.V * (L.Smax - 1) * 8; it += ctx.nt) {
    int a = it / ((L.Smax - 1) * 8), q = (it / 8) % (L.Smax - 1);
    if (q < L.S[a] - 1) W.x[L.oTS + it] = W.c[L.oYTUBE + it];
  }
  for (int it = ctx.tid; it < L.P * L.Mv; it += ctx.nt) {
    int p = it / L.Mv, n = it % L.Mv;
    if (n < L.Mp[p]) {
      double body = W.c[L.YPAIR(p, 0, n)];
      W.x[L.PSD(p, n)] = body > 0 ? body : 0.0;
      W.x[L.PEL(p, n)] = body < 0 ? -body : 0.0;
      W.x[L.PSN(p, n)] = W.c[L.YPAIR(p, 5, n)];
    }
  }
  cta_sync(ctx);
}

OBCA_HDN void push_into_bounds(const Ctx& ctx, const Lay& L, const double* xL, const double* xU, double* x, double k1, double k2) {
  for (int q = ctx.tid; q < L.nx; q += ctx.nt) {
    double lo = xL[q], hi = xU[q], v = x[q];
    bool hl = lo > -INFINITY, hu = hi < INFINITY;
    double pl = hl ? k1 * fmax(1.0, fabs(lo)) : 0.0, pu = hu ? k1 * fmax(1.0, fabs(hi)) : 0.0;
    if (hl && hu) {
      pl = fmin(pl, k2 * (hi - lo));
      pu = fmin(pu, k2 * (hi - lo));
    }
    if (hl) v = fmax(v, lo + pl);
    if (hu) v = fmin(v, hi - pu);
    x[q] = v;
  }
  cta_sync(ctx);
}

// One interior-point run from the point in W.x (slack initialisation, push into the bounds, z = 1, y = 0, mu = mu_init; with
// sh->warm from the stored zL, zU, y and mu0, see obca_warm_start in obca.h).
// `it` and `n_refine` accumulate over the runs of one instance.  Returns the status; *el_out = largest elastic variable.
template <int MODE>
OBCA_HDN int ipm_attempt(const Ctx& ctx, const Lay& L, const Stat& S, const Opts& o, const Counts& cnt, const double* xL,
                         const double* xU, const unsigned char* bcls, const Scratch& W, double* RW, size_t rw_cap, Shared* sh, Result* res, int& it,
                         int& n_refine, double* el_out) {
  const BoundCls bc = {bcls, sh->blo, sh->bhi};
  assume_scratch(W);
  OBCA_ASSUME_STATIC(L, S);
  OBCA_ASSUME_GLOBAL(xL), OBCA_ASSUME_GLOBAL(xU);
  // ---- initial point.  Warm start (IPOPT warm_start_init_point): the stored x, zL, zU, y of the instance instead of z = 1, y = 0
  init_slacks<MODE>(ctx, L, S, W);
  const bool warm = sh->warm;  // after the barrier that ends init_slacks (ipm_solve clears it before a restart)
  push_into_bounds(ctx, L, xL, xU, W.x, warm ? res->ws_bound_push : o.bound_push, warm ? res->ws_bound_push : o.bound_frac);
  for (int q = ctx.tid; q < L.nx; q += ctx.nt) {
    const double zl0 = warm ? fmax(W.zL[q], res->ws_mult_bound_push) : 1.0, zu0 = warm ? fmax(W.zU[q], res->ws_mult_bound_push) : 1.0;
    W.zL[q] = xL[q] > -INFINITY ? zl0 : 0.0;
    W.zU[q] = xU[q] < INFINITY ? zu0 : 0.0;
    W.dx[q] = 0, W.dzL[q] = 0, W.dzU[q] = 0, W.gl[q] = 0;
  }
  for (int q = ctx.tid; q < L.ny; q += ctx.nt) {
    if (!warm) W.y[q] = 0;
    W.dy[q] = 0;
  }
  if (ctx.tid == 0) sh->filt_n = 0, sh->hist_warm = warm;
  cta_sync(ctx);
  const double mu_min = fmin(o.tol, o.compl_inf_tol) / (o.kappa_eps + 1.0);
  double mu = warm ? fmax(mu_min, res->mu0) : o.mu_init;
  double f, gdt;
  model_eval<MODE>(ctx, L, S, W, W.x, W.y, W.c, W.gl, &f, &gdt);
  double th0 = 0;
  for (int q = ctx.tid; q < L.ny; q += ctx.nt) th0 += fabs(W.c[q]);
  th0 = cta_sum(ctx, th0);
  const double theta_max = 1e4 * fmax(1.0, th0), theta_min = 1e-4 * fmax(1.0, th0);
  double dw_last = 0.0;
  bool tiny_last = false, force_mu = false;
  // IPOPT acceptable-point bookkeeping: acceptable_tol 1e-6, acceptable_iter 15
  double best_E = INFINITY, best_f = 0, best_cv = 0, best_du = 0, best_co = 0;
  int n_acceptable = 0;
  int n_rescue = 0;  // line-search failures answered by a barrier reset (see below)
  int status = OBCA_MAXITER_EXCEEDED;
  double dual_inf = 0, cviol = 0, compl0 = 0;
  const Stage st = {RW, rw_cap, sh->bars};
  // barrier terms of the current iterate: carried over from the accepted trial point (bit-identical x), recomputed otherwise
  double bar_cur = 0.0;
  bool bar_valid = false;
  for (;;) {
    // ---- error measures at the current iterate (c, gl, f are up to date)
    double e_du = 0, e_c = 0, e_c1 = 0, s_y = 0, s_z = 0, cmax0 = 0, cmaxmu_lo = INFINITY, cmaxmu_hi = 0;
    double s_log = 0, s_gap = 0;  // barrier pieces: phi = f + mu (-sum log gap + kappa_d sum one-sided gap)
    {
      const double* const src[4] = {W.x, W.zL, W.zU, W.gl};
      flat_pass_b<4>(ctx, st, bc, src, L.nx, [&](int q, const double* v, double lo, double hi) {
        const double xv = v[0], zl = v[1], zu = v[2], gq = v[3];
        e_du = fmax(e_du, fabs(gq - zl + zu));
        const bool hl = lo > -INFINITY, hu = hi < INFINITY;
        // Sigma and the barrier gradient for the CURRENT mu and delta_w = 0 ride along (same inputs): the separate pass is only
        // needed when mu changes below or the inertia correction raises delta_w -- a handful of iterations per solve
        double sg = 0.0, gph = gq;
        if (hl) {
          const double gp = xv - lo, pr = gp * zl, iL = rcp_pos(gp);
          cmax0 = fmax(cmax0, pr), cmaxmu_lo = fmin(cmaxmu_lo, pr), cmaxmu_hi = fmax(cmaxmu_hi, pr);
          s_z += zl;
          sg += zl * iL, gph -= mu * iL;
          if (!hu) gph += o.kappa_d * mu;
          if (!bar_valid) {
            s_log -= log(gp);
            if (!hu) s_gap += gp;
          }
        }
        if (hu) {
          const double gp = hi - xv, pr = gp * zu, iU = rcp_pos(gp);
          cmax0 = fmax(cmax0, pr), cmaxmu_lo = fmin(cmaxmu_lo, pr), cmaxmu_hi = fmax(cmaxmu_hi, pr);
          s_z += zu;
          sg += zu * iU, gph += mu * iU;
          if (!hl) gph -= o.kappa_d * mu;
          if (!bar_valid) {
            s_log -= log(gp);
            if (!hl) s_gap += gp;
          }
        }
        W.sig[q] = sg, W.gphi[q] = gph;
      });
      prof_mark(ctx, 21);
    }
    {
      const double* const src[2] = {W.c, W.y};
      flat_pass<2>(ctx, st, src, L.ny, [&](int, const double* v) {
        e_c = fmax(e_c, fabs(v[0]));
        e_c1 += fabs(v[0]);
        s_y += fabs(v[1]);
      });
    }
    dual_inf = cta_max(ctx, e_du);
    cviol = cta_max(ctx, e_c);
    double theta = cta_sum(ctx, e_c1);
    s_y = cta_sum(ctx, s_y);
    s_z = cta_sum(ctx, s_z);
    if (!bar_valid) {
      s_log = cta_sum(ctx, s_log);
      s_gap = cta_sum(ctx, s_gap);
      bar_cur = s_log + o.kappa_d * s_gap;
      bar_valid = true;
    }
    compl0 = cta_max(ctx, cmax0);
    double pr_lo = cta_min(ctx, cmaxmu_lo), pr_hi = cta_max(ctx, cmaxmu_hi);
    double s_d = fmax(o.s_max, (s_y + s_z) / fmax(1.0, (double)(cnt.m_active + cnt.nb))) / o.s_max;
    double s_c = fmax(o.s_max, s_z / fmax(1.0, (double)cnt.nb)) / o.s_max;
    double E0 = fmax(fmax(dual_inf / s_d, cviol), compl0 / s_c);
    if (ctx.tid == 0 && sh->hist) hist_head(sh, it, f, cviol, theta, dual_inf, compl0, mu, E0, E0 <= 1e-6 && cviol <= 1e-2 && compl0 <= 1e-2, S.rho);
    if (E0 <= o.tol && dual_inf <= o.dual_inf_tol && cviol <= o.constr_viol_tol && compl0 <= o.compl_inf_tol) {
      status = OBCA_SOLVE_SUCCEEDED;
      break;
    }
    if (E0 <= 1e-6 && cviol <= 1e-2 && compl0 <= 1e-2) {
      ++n_acceptable;
      if (E0 < best_E) {
        best_E = E0, best_f = f, best_cv = cviol, best_du = dual_inf, best_co = compl0;
        for (int q = ctx.tid; q < L.nx; q += ctx.nt) W.bx[q] = W.x[q], W.bzL[q] = W.zL[q], W.bzU[q] = W.zU[q];
        for (int q = ctx.tid; q < L.ny; q += ctx.nt) W.by[q] = W.y[q];
      }
      if (n_acceptable >= 15) {
        status = OBCA_SOLVED_TO_ACCEPTABLE_LEVEL;
        break;
      }
    } else
      n_acceptable = 0;
    if (it >= o.max_iter) {
      status = OBCA_MAXITER_EXCEEDED;
      break;
    }
    if (!finite_d(f) || !finite_d(theta) || !finite_d(dual_inf)) {
      status = OBCA_INVALID_NUMBER_DETECTED;
      break;
    }
    // ---- barrier parameter update
    bool sig_ready = true;  // W.sig / W.gphi from the error pass are valid for (mu, delta_w = 0)
    for (;;) {
      double cmu = fmax(fabs(pr_lo - mu), fabs(pr_hi - mu));
      double Emu = fmax(fmax(dual_inf / s_d, cviol), cmu / s_c);
      if ((Emu <= o.kappa_eps * mu || force_mu) && mu > mu_min) {
        mu = fmax(mu_min, fmin(o.kappa_mu * mu, pow(mu, o.theta_mu)));
        if (ctx.tid == 0) sh->filt_n = 0;
        force_mu = false;
        sig_ready = false;
      } else
        break;
    }
    force_mu = false;
    if (ctx.tid == 0 && sh->hist && !sig_ready) sh->hist_flags |= OBCA_HIST_F_MU_LOWERED;  // sig_ready is cleared exactly when mu was lowered
    cta_sync(ctx);
    const double tau = fmax(o.tau_min, 1.0 - mu);
    // ---- gradient of the barrier Lagrangian, barrier objective and grad_phi'dx bookkeeping
    const double phi = f + mu * bar_cur;  // the iterate is strictly inside its bounds
    // ---- search direction with inertia correction
    double dw = 0.0;
    bool first = true, have = false;
    for (;;) {
      if (!sig_ready) {
        const double* const src[4] = {W.x, W.zL, W.zU, W.gl};
        flat_pass_b<4>(ctx, st, bc, src, L.nx, [&](int q, const double* v, double lo, double hi) {
          const double xv = v[0], zl = v[1], zu = v[2];
          const bool hl = lo > -INFINITY, hu = hi < INFINITY;
          double sg = dw, gp = v[3];
          if (hl) {
            const double iL = rcp_pos(xv - lo);
            sg += zl * iL;
            gp -= mu * iL;
            if (!hu) gp += o.kappa_d * mu;
          }
          if (hu) {
            const double iU = rcp_pos(hi - xv);
            sg += zu * iU;
            gp += mu * iU;
            if (!hl) gp -= o.kappa_d * mu;
          }
          W.sig[q] = sg, W.gphi[q] = gp;
        });
      prof_mark(ctx, 22);
      }
      sig_ready = false;  // any further trial of this iteration changes delta_w
      cta_sync(ctx);
      if (model_kkt<MODE>(ctx, L, S, W, RW, &sh->ok)) {
        have = true;
        if (MODE == 0 && o.refine_steps > 0) {
          double rr;
          n_refine += kkt_refine(ctx, L, S, W, RW, &sh->ok, o.refine_steps, o.refine_ratio, &rr);
        }
        break;
      }
      if (first) {
        dw = dw_last == 0.0 ? o.dw_first : fmax(o.dw_min, o.kw_minus * dw_last);
        first = false;
      } else
        dw *= dw_last == 0.0 ? o.kw_plus_first : o.kw_plus;
      if (dw > o.dw_max) break;
    }
    if (!have) {
      status = OBCA_ERROR_IN_STEP_COMPUTATION;
      break;
    }
    if (dw > 0) dw_last = dw;
    if (ctx.tid == 0 && sh->hist) sh->hist_dw = dw;
    // ---- dz, fraction to the boundary, directional derivative of the barrier objective
    double a_pr = 1.0, a_du = 1.0, dphi = 0, rel = 0, r_pr = 0, dn = 0;
    {
      const double* const src[5] = {W.x, W.zL, W.zU, W.gphi, W.dx};
      flat_pass_b<5>(ctx, st, bc, src, L.nx, [&](int, const double* v, double lo, double hi) {
        const double xv = v[0], zl = v[1], zu = v[2], d = v[4];
        rel = fmax(rel, fabs(d) * rcp_pos(1.0 + fabs(xv)));
        dn = fmax(dn, fabs(d));
        if (lo > -INFINITY) {
          const double ig = rcp_pos(xv - lo);
          const double dz = (mu - zl * d) * ig - zl;
          r_pr = fmax(r_pr, -d * ig);            // alpha_pr = tau / max(-d / gap)
          if (dz < 0) a_du = fmin(a_du, -tau * zl / dz);
        }
        if (hi < INFINITY) {
          const double ig = rcp_pos(hi - xv);
          const double dz = (mu + zu * d) * ig - zu;
          r_pr = fmax(r_pr, d * ig);
          if (dz < 0) a_du = fmin(a_du, -tau * zu / dz);
        }
        dphi += v[3] * d;
      });
      prof_mark(ctx, 23);
    }
    // grad_phi'dx = (gphi)'dx - y'J dx ; J dx = -c - (local delta_c terms, negligible) => use the exact product:
    // y'J dx is accumulated from the structure: J dx = -(c) on all rows up to delta_c * dy.
    double yJdx = 0;
    {
      const int o0 = L.oYOBS, o1 = L.oYOBS + L.V * L.O * 4 * L.Mv, p0 = L.oYPAIR, p1 = L.oYPAIR + L.P * 6 * L.Mv;
      const double* const src[3] = {W.y, W.c, W.dy};
      flat_pass<3>(ctx, st, src, L.ny, [&](int q, const double* v) {
        yJdx -= v[0] * v[1];
        if ((q >= o0 && q < o1) || (q >= p0 && q < p1)) yJdx += v[0] * DELTA_C_LOCAL * v[2];
      });
    }
    r_pr = cta_max(ctx, r_pr);
    if (r_pr > tau) a_pr = tau / r_pr;
    a_du = cta_min(ctx, a_du);
    rel = cta_max(ctx, rel);
    if (sh->hist) {  // the only reduction the record adds
      dn = cta_max(ctx, dn);
      if (ctx.tid == 0) sh->hist_dn = dn;
    }
    dphi = cta_sum(ctx, dphi) - cta_sum(ctx, yJdx);
#ifdef OBCA_HOST_EMU
    if (getenv("OBCA_TRACE")) {  // which variable limits the primal step
      int arg = -1, up = 0;
      double best = 2.0;
      for (int q = 0; q < L.nx; ++q) {
        double d = W.dx[q];
        if (xL[q] > -INFINITY && d < 0 && -tau * (W.x[q] - xL[q]) / d < best) best = -tau * (W.x[q] - xL[q]) / d, arg = q, up = 0;
        if (xU[q] < INFINITY && d > 0 && tau * (xU[q] - W.x[q]) / d < best) best = tau * (xU[q] - W.x[q]) / d, arg = q, up = 1;
      }
      const int offs[] = {L.oZ, L.oLAM, L.oMU, L.oSD, L.oEL, L.oTS, L.oPL, L.oPM, L.oPS, L.oPSD, L.oPSN, L.oPEL, L.oDT, L.nx};
      const char* nm[] = {"Z", "LAM", "MU", "SD", "EL", "TS", "PL", "PM", "PS", "PSD", "PSN", "PEL", "DT"};
      for (int k = 0; k < 13 && arg >= 0; ++k)
        if (arg >= offs[k] && arg < offs[k + 1])
          printf("       block %s[%d] (n=%d) %s x=%.3e dx=%.3e\n", nm[k], (arg - offs[k]) / L.Mv, (arg - offs[k]) % L.Mv, up ? "upper" : "lower", W.x[arg], W.dx[arg]);
    }
#endif
    // ---- filter line search
    double a_min;
    if (dphi < 0) {
      a_min = fmin(o.gamma_theta, o.gamma_phi * theta / (-dphi));
      if (theta <= theta_min) a_min = fmin(a_min, o.delta_ls * pow(theta, o.s_theta) / pow(-dphi, o.s_phi));
    } else
      a_min = o.gamma_theta;
    a_min *= o.gamma_alpha;
    double alpha = a_pr;
    bool accepted = false;
    double ft = f, gdt_t;
    // IPOPT compares with a machine-precision slack (Compare_le: lhs - rhs <= 10 eps |base|)
    const double EPS = 2.220446049250313e-16;
    // ... widened to 1e-10 (relative to max(1, |.|)): the structured solve has no iterative refinement, its steps carry ~1e-8
    // relative noise, and near the solution phi / theta changes of that size must not trigger backtracking
    const double slack_phi = 1e-10 * fmax(1.0, fabs(phi)), slack_th = 1e-10 * fmax(1.0, theta);
    // tiny-step rule: a step below 10 eps relative size is accepted without line search and forces a mu update
    if (rel < 10 * EPS) {
      if (tiny_last && mu <= mu_min) {
        // IPOPT: Search_Direction_Becomes_Too_Small (an error for CasADi) unless this iterate passes the acceptable test
        const bool acc_here = E0 <= 1e-6 && cviol <= 1e-2 && compl0 <= 1e-2;
        status = acc_here ? OBCA_SOLVED_TO_ACCEPTABLE_LEVEL : OBCA_SEARCH_DIRECTION_TOO_SMALL;
        break;
      }
      tiny_last = true, force_mu = true;
      for (int q = ctx.tid; q < L.nx; q += ctx.nt) W.xt[q] = W.x[q] + alpha * W.dx[q];
      accepted = true;
      bar_valid = false;  // no trial evaluation: the barrier terms are recomputed in the next error pass
    } else
      tiny_last = false;
    while (alpha >= a_min && !accepted) {
      // trial point and its barrier terms in one pass
      double sbar = 0;
      int bad = 0;
      {
        const double* const src[2] = {W.x, W.dx};
        // sum of log(gap) as log of products: a thread multiplies the gaps of its elements (each within [1e-20, 1e2]) and takes one
        // log whenever the running product approaches the end of the FP64 range (every ~20 elements) and at the end
        double prod = 1.0;
        flat_pass_b<2>(ctx, st, bc, src, L.nx, [&](int q, const double* v, double lo, double hi) {
          const double xn = v[0] + alpha * v[1];
          W.xt[q] = xn;
          const bool hl = lo > -INFINITY, hu = hi < INFINITY;
          if (hl) {
            const double gp = xn - lo;
            if (gp <= 0) bad = 1;
            else prod *= gp;
            if (!hu) sbar += o.kappa_d * gp;
          }
          if (hu) {
            const double gp = hi - xn;
            if (gp <= 0) bad = 1;
            else prod *= gp;
            if (!hl) sbar += o.kappa_d * gp;
          }
          if (prod < 1e-250 || prod > 1e250) sbar -= log(prod), prod = 1.0;  // flush before the running product leaves the FP64 range
        });
        sbar -= log(prod);
      }
      prof_mark(ctx, 24);
      if (ctx.tid == 0 && sh->hist) ++sh->hist_trials;
      cta_sync(ctx);
      model_eval<MODE>(ctx, L, S, W, W.xt, nullptr, W.ct, nullptr, &ft, &gdt_t);
      double tht = 0;
      {
        const double* const src[1] = {W.ct};
        flat_pass<1>(ctx, st, src, L.ny, [&](int, const double* v) { tht += fabs(v[0]); });
      }
      tht = cta_sum(ctx, tht);
      prof_mark(ctx, 25);
      sbar = cta_sum(ctx, sbar);
      const double pht = cta_max(ctx, (double)bad) > 0 ? INFINITY : ft + mu * sbar;
      bool okp = finite_d(pht) && finite_d(tht) && tht <= theta_max;
      if (okp) {
        int nf = sh->filt_n;
        for (int k = 0; k < nf; ++k)
          if (tht - sh->filt_theta[k] > slack_th && pht - sh->filt_phi[k] > slack_phi) okp = false;  // same comparison slack as the acceptance tests
      }
      if (okp) {
        bool switching = theta <= theta_min && dphi < 0 && alpha * pow(-dphi, o.s_phi) > o.delta_ls * pow(theta, o.s_theta);
        if (switching) {
          if (pht - (phi + o.eta_phi * alpha * dphi) <= slack_phi) {
            accepted = true;
            bar_cur = sbar;
            break;
          }
        } else if (tht - (1 - o.gamma_theta) * theta <= slack_th || pht - (phi - o.gamma_phi * theta) <= slack_phi) {
          cta_sync(ctx);
          if (ctx.tid == 0 && sh->filt_n < FILTER_MAX) {
            sh->filt_theta[sh->filt_n] = (1 - o.gamma_theta) * theta;
            sh->filt_phi[sh->filt_n] = phi - o.gamma_phi * theta;
            sh->filt_n++;
          }
          accepted = true;
          bar_cur = sbar;
          break;
        }
      }
      alpha *= 0.5;
    }
    cta_sync(ctx);
    if (!accepted) {
      // IPOPT enters its feasibility-restoration phase here.  This solver has none; what it can do cheaply is leave the corner the
      // iterate is stuck in: raise the barrier parameter again (x10, at most mu_init), forget the filter and iterate on -- a larger mu
      // re-centres the slacks that blocked the step.  Three attempts, then Restoration_Failed as before.
      if (n_rescue < 3 && it < o.max_iter) {
        if (ctx.tid == 0 && sh->hist) hist_step(sh, 0.0, 0.0, OBCA_HIST_F_RESET);  // no step taken
        ++n_rescue;
        mu = fmin(o.mu_init, 10.0 * mu);
        cta_sync(ctx);
        if (ctx.tid == 0) sh->filt_n = 0;
        cta_sync(ctx);
        tiny_last = false, force_mu = false;
        ++it;
        continue;
      }
      status = OBCA_RESTORATION_FAILED;  // becomes Solved_To_Acceptable_Level below when an acceptable point was stored
      break;
    }
    // ---- accept the trial point (dz is recomputed from dx; x + alpha dx reproduces the trial point bit for bit)
    if (ctx.tid == 0 && sh->hist) hist_step(sh, alpha, a_du, tiny_last ? OBCA_HIST_F_TINY_STEP : 0);
    const double iks = 1.0 / o.kappa_sigma;
    {
      const double* const src[4] = {W.x, W.zL, W.zU, W.dx};
      flat_pass_b<4>(ctx, st, bc, src, L.nx, [&](int q, const double* v, double lo, double hi) {
        const double xv = v[0], zl = v[1], zu = v[2], d = v[3];
        const double xn = xv + alpha * d;
        W.x[q] = xn;
        if (lo > -INFINITY) {
          const double i0 = rcp_pos(xv - lo), mg = mu * rcp_pos(xn - lo);
          const double zv = zl + a_du * ((mu - zl * d) * i0 - zl);
          W.zL[q] = fmin(fmax(zv, mg * iks), o.kappa_sigma * mg);
        }
        if (hi < INFINITY) {
          const double i0 = rcp_pos(hi - xv), mg = mu * rcp_pos(hi - xn);
          const double zv = zu + a_du * ((mu + zu * d) * i0 - zu);
          W.zU[q] = fmin(fmax(zv, mg * iks), o.kappa_sigma * mg);
        }
      });
      prof_mark(ctx, 26);
    }
    {
      const double* const src[2] = {W.y, W.dy};
      flat_pass<2>(ctx, st, src, L.ny, [&](int q, const double* v) { W.y[q] = v[0] + alpha * v[1]; });
    }
    cta_sync(ctx);
    model_eval<MODE>(ctx, L, S, W, W.x, W.y, W.c, W.gl, &f, &gdt);
    ++it;
  }
  cta_sync(ctx);
  if (status != OBCA_SOLVE_SUCCEEDED && best_E < INFINITY) {
    // restore the best acceptable point (IPOPT RestoreAcceptablePoint)
    for (int q = ctx.tid; q < L.nx; q += ctx.nt) W.x[q] = W.bx[q], W.zL[q] = W.bzL[q], W.zU[q] = W.bzU[q];
    for (int q = ctx.tid; q < L.ny; q += ctx.nt) W.y[q] = W.by[q];
    status = OBCA_SOLVED_TO_ACCEPTABLE_LEVEL;
    f = best_f, cviol = best_cv, dual_inf = best_du, compl0 = best_co;
    cta_sync(ctx);
  }
  // Elastic variables of the distance rows (exact l1 penalty): at a solution of the reference problem they vanish.  A point
  // that converged with an active elastic variable solves the penalised problem only -- the reference problem is (locally)
  // infeasible there, IPOPT would report Infeasible_Problem_Detected and Opti would raise.
  double el_max = 0;
  for (int q = ctx.tid; q < L.V * L.O * L.Mv; q += ctx.nt) el_max = fmax(el_max, W.x[L.oEL + q]);
  for (int q = ctx.tid; q < L.P * L.Mv; q += ctx.nt) el_max = fmax(el_max, W.x[L.oPEL + q]);
  el_max = cta_max(ctx, el_max);
  *el_out = el_max;
  if (ctx.tid == 0) {
    res->status = status;
    res->iters = it;
    res->obj = f;
    res->cviol = fmax(cviol, el_max);
    res->elastic = el_max;
    res->refines = n_refine;
    res->dual_inf = dual_inf;
    res->compl_inf = compl0;
    res->mu = mu;
    res->dt = W.x[L.oDT];
  }
  cta_sync(ctx);
  return status;
}

// Dual restoration.  The OBCA dual blocks are non-convex (|A'lam|^2 = 1 is an equality): besides the separating direction
// (maximal dual distance) the opposite direction is a stationary point too, and with the elastic variable on the distance row
// the iteration can converge to it -- the elastic variable then carries a "violation" of metres although the shapes are far
// apart (observed from the reference's random first-step duals, vehicle_follower.py:401-402).  IPOPT meets the hard row
// there, fails the line search and enters its restoration phase; the equivalent here is exact and local: every block whose
// elastic variable is active gets the closed-form separating duals of its current poses (obca_ws.h, the same formulas as the
// dual warm start), and the interior-point iteration restarts from that point.
template <int MODE>
OBCA_HDN int dual_restore(const Ctx& ctx, const Lay& L, const Stat& S, const Scratch& W, double thr) {
  assume_scratch(W);
  OBCA_ASSUME_STATIC(L, S);
  double* x = W.x;
  int improved = 0;  // blocks whose distance row gains more than thr from the separating duals: only those justify a restart
  for (int it = ctx.tid; it < L.V * L.O * L.Mv; it += ctx.nt) {
    const int n = it % L.Mv, aj = it / L.Mv, a = aj / L.O, j = aj % L.O;
    if (n >= L.M[a] || !(x[L.EL(a, j, n)] > thr)) continue;
    double lam[4], mu[4];
    const double px = x[L.Z(a, 0, n)], py = x[L.Z(a, 1, n)];
    ws_obstacle_duals(S, j, px, py, x[L.Z(a, 2, n)], lam, mu);
    double d_new = 0, d_old = 0;
    for (int r = 0; r < 4; ++r) {
      const double atb = S.obsA[j][r][0] * px + S.obsA[j][r][1] * py - S.obsb[j][r];
      d_new += atb * lam[r] - S.g[r] * mu[r];
      d_old += atb * x[L.LAM(a, j, r, n)] - S.g[r] * x[L.MU(a, j, r, n)];
    }
    if (d_new > d_old + thr) ++improved;
#ifdef OBCA_HOST_EMU
    if (getenv("OBCA_TRACE_RESTORE")) printf("restore obs j=%d n=%d el=%.4f d_old=%.4f d_new=%.4f pose %.3f %.3f %.3f\n", j, n, x[L.EL(a, j, n)], d_old, d_new, px, py, x[L.Z(a, 2, n)]);
#endif
    for (int r = 0; r < 4; ++r) x[L.LAM(a, j, r, n)] = lam[r], x[L.MU(a, j, r, n)] = mu[r];
  }
  for (int it = ctx.tid; it < L.P * L.Mv; it += ctx.nt) {
    const int p = it / L.Mv, n = it % L.Mv;
    if (n >= L.Mp[p] || !(x[L.PEL(p, n)] > thr)) continue;
    Pose a, b;
    load_pose(L, x, L.pa[p], n, a);
    if (MODE == 1) load_other_pose(L, mpc_par(L, W), p, n, b);
    else load_pose(L, x, L.pb[p], n, b);
    PairBlk B;
    load_pair(L, x, p, n, B);
    pair_residual(S, a, b, B);
    const double d_old = B.c[0] + B.sd - B.el;  // -b_a'lam - b_b'mu - dmin with the current duals
    ws_pair_duals(S, a.x, a.y, a.psi, b.x, b.y, b.psi, B.lam, B.mu, B.s);
    pair_residual(S, a, b, B);
    if (B.c[0] + B.sd - B.el > d_old + thr) ++improved;
    for (int r = 0; r < 4; ++r) x[L.PL(p, r, n)] = B.lam[r], x[L.PM(p, r, n)] = B.mu[r];
    x[L.PS(p, 0, n)] = B.s[0], x[L.PS(p, 1, n)] = B.s[1];
  }
  cta_sync(ctx);
  return (int)cta_sum(ctx, (double)improved);
}

template <int MODE>
OBCA_HDN void ipm_solve(const Ctx& ctx, const Lay& L, const Stat& S, const Opts& o, const Counts& cnt, const double* xL,
                        const double* xU, const unsigned char* bcls, const Scratch& W, double* RW, size_t rw_cap, Shared* sh, Result* res) {
  int it = 0, n_refine = 0, restarts = 0, status;
  double el_max;
  const double thr = fmax(o.constr_viol_tol, 1e-8);
  // S is this CTA's private copy of the static data (shared memory on the device): the penalty weight of the elastic variables
  // may be raised for the instance at hand and is put back before the next one
  double* rho = const_cast<double*>(&S.rho);
  const double rho0 = S.rho;
  // MPC mode: the solves of one handle are consecutive control steps of the same vehicle; a weight that had to be raised stays
  // raised for the next step (the geometry that made the penalty inexact is still there) and is dropped after a failed solve
  const double carry = MODE == 1 ? res->rho_carry : 0.0;
  if (ctx.tid == 0) {  // the arm of obca_warm_start is consumed by this solve
    sh->warm = res->warm;
    res->warm = 0;
  }
  cta_sync(ctx);
  if (carry > rho0) {
    if (ctx.tid == 0) *rho = carry;
    cta_sync(ctx);
  }
  for (;;) {
    status = ipm_attempt<MODE>(ctx, L, S, o, cnt, xL, xU, bcls, W, RW, rw_cap, sh, res, it, n_refine, &el_max);
#ifdef OBCA_HOST_EMU
    if (getenv("OBCA_TRACE_RESTORE")) printf("attempt: status %d it %d el_max %.4f restarts %d rho %.1e\n", status, it, el_max, restarts, S.rho);
#endif
    if (!(status >= 0 && el_max > thr)) break;
    if (restarts >= 5 || it >= o.max_iter) {
      // a converged point of the penalised problem with an active elastic variable: the reference problem (hard distance rows)
      // is locally infeasible there; IPOPT reports Infeasible_Problem_Detected and Opti raises
      status = OBCA_INFEASIBLE_PROBLEM_DETECTED;
      break;
    }
    if (dual_restore<MODE>(ctx, L, S, W, thr) == 0) {
      // The duals already are the separating ones: the minimiser of the PENALISED problem really is closer than dmin -- the
      // l1 penalty was not exact for this instance (the MPC tracking cost, 100 per m^2 and node, can outweigh rho = 1e3).
      // Exact-penalty update: raise the weight and solve again from this point; give up when a 1e4 times larger weight still
      // leaves a violation (then the hard-constrained problem has no solution nearby).
      if (S.rho >= 1e4 * rho0) {
        status = OBCA_INFEASIBLE_PROBLEM_DETECTED;
        break;
      }
      cta_sync(ctx);
      if (ctx.tid == 0) *rho = S.rho * 10.0;
      cta_sync(ctx);
    }
    ++restarts;
    if (ctx.tid == 0) ++sh->hist_attempt, sh->warm = 0;  // restarts start cold (read after the barriers of init_slacks)
  }
  cta_sync(ctx);
  // Which weight the next control step starts with: the l1 penalty is exact when it exceeds the multipliers of the hard distance rows
  // (|y_d| <= rho by the elastic variable's bound multiplier z = rho + y_d >= 0).  Keep the smallest rho0 10^k with a factor 1.25 of
  // margin over the largest |y_d| of this solution -- back to rho0 as soon as the geometry that needed more is gone (a raised weight
  // costs iterations: the elastic bound multipliers start at 1, far from rho).
  double next = 0.0;
  if (MODE == 1 && status >= 0 && S.rho > rho0) {
    double ymax = 0.0;
    for (int q = ctx.tid; q < L.V * L.O * L.Mv; q += ctx.nt) {
      const int n = q % L.Mv, aj = q / L.Mv;
      ymax = fmax(ymax, fabs(W.y[L.YOBS(aj / L.O, aj % L.O, 0, n)]));
    }
    for (int q = ctx.tid; q < L.P * L.Mv; q += ctx.nt) ymax = fmax(ymax, fabs(W.y[L.YPAIR(q / L.Mv, 0, q % L.Mv)]));
    ymax = cta_max(ctx, ymax);
    next = rho0;
    while (next < 1.25 * ymax && next < S.rho) next *= 10.0;
    if (next <= rho0) next = 0.0;
  }
  if (ctx.tid == 0) {
    res->status = status, res->restarts = restarts;
    res->rho_carry = next;
  }
  cta_sync(ctx);  // every warp has evaluated the test on S.rho above before the weight is reset (racecheck: read / write hazard)
  if (ctx.tid == 0) *rho = rho0;
  cta_sync(ctx);
}

}  // namespace obca
