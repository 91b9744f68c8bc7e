// obca_core.h -- per-instance OBCA interior-point solver, written once for the CUDA kernels
// (one CTA per problem instance) and for the single-threaded host emulation that the developer
// tools use to debug the algorithm on machines without a GPU (tools/host_emu; never loaded by
// the package).
//
// Problem (reference: confrez/control/vehicle.py:360-640, multi_vehicle_planner.py:343-480):
//   collocation OBCA NLP of V vehicles sharing one interval length dt.  See DESIGN.md for the
//   mathematics; the section names below match it.
//
//   [LAYOUT]   flat primal/dual vectors, node-minor (coalesced across the threads of a CTA)
//   [EVAL]     residuals c(x), Lagrangian gradient gl = grad f + J'y, objective
//   [LOCAL]    elimination of obstacle / pair / tube blocks onto the vehicle poses
//   [NULLSP]   per (vehicle, interval) Householder QR of the collocation Jacobian -> stage dynamics
//   [RICCATI]  backward / forward recursion over the intervals (state 7V+1, control 5V)
//   [BACKSUB]  multipliers and local variables
//   [IPM]      barrier update, fraction to the boundary, filter line search, convergence tests
#pragma once
#include <math.h>
#include <stdint.h>

#include "obca.h"

#if defined(__CUDACC__)
#define OBCA_HD __host__ __device__ __forceinline__
#define OBCA_HDN __host__ __device__
#else
#define OBCA_HD inline
#define OBCA_HDN inline
#endif

// address-space hints: the work arena is always dynamic shared memory on the device
#if defined(__CUDA_ARCH__)
#define OBCA_ASSUME_SHARED(p) __builtin_assume(__isShared(p))
#define OBCA_ASSUME_GLOBAL(p) __builtin_assume(__isGlobal(p))
#else
#define OBCA_ASSUME_SHARED(p) ((void)0)
#define OBCA_ASSUME_GLOBAL(p) ((void)0)
#endif

// warps per CTA that own a shared-memory work area in the null-space / coupling phases, and whether the Riccati phase
// stages its inputs in shared memory (needs 19 KB more; off when two CTAs share an SM)
#ifndef OBCA_NS_WARPS
#if defined(OBCA_HOST_EMU)
#define OBCA_NS_WARPS 1
#else
#define OBCA_NS_WARPS 8
#endif
#endif
#ifndef OBCA_RIC_PREFETCH
#define OBCA_RIC_PREFETCH 1
#endif

namespace obca {

constexpr int NK = 6;    // nodes per interval (K + 1)
constexpr int NZ = 7;    // x y psi v delta a w
constexpr int NS = 42;   // stage variables of one vehicle interval
constexpr int NW = 35;   // stage variables without node 0
constexpr int NP = 8;    // max free directions per vehicle interval (5 when the collocation Jacobian has full rank)
constexpr int NRED = 7 + NP + 1;  // reduced coordinates: xi(7) p(NP) dt(1)
constexpr int IDT = 7 + NP;       // index of dt in the reduced coordinates
constexpr int NSYM = NRED * (NRED + 1) / 2;
constexpr int NEX = 5;                 // max implied state-constraint rows handed to the previous interval
constexpr int NC = 30 + 5 + NEX;       // max constraint rows of one (vehicle, interval) block
constexpr int NDR = 8;                 // max dropped (dependent) rows recorded per block
constexpr int EXSZ = 1 + NEX * 9;      // emitted rows: count, then (h_xi[7], h_dt, h0) each
// QR record: [35*NC] reflectors / R staircase, [35] tau, [35] pivot column of each staircase row,
// [4] (rank, rows, ndrop, unused), then NDR x (column j, emission slot or -1, staircase length, alpha[35], implied row h[9]), then nu[NEX]
constexpr int QR_TAU = 35 * NC, QR_PIV = QR_TAU + 35, QR_META = QR_PIV + 35, QR_DROP = QR_META + 4, DRSZ = 3 + 35 + 9;
constexpr int QR_NU = QR_DROP + NDR * DRSZ;  // multipliers of the received implied rows
constexpr int QR_BU = QR_NU + NEX;      // coefficients of (a_5, w_5) in the terminal / implied rows before their elimination: [2][NC]
constexpr int QRSZ = QR_BU + 2 * NC;
constexpr int NQ = 25;                  // state variables of the nodes 1..K of a block: the controls are eliminated analytically
constexpr int NU2 = 10;                 // of these (x, y, psi) are eliminated through the constant interior collocation block: the QR sees (v, delta)
constexpr int MAXV = OBCA_MAX_V;
constexpr int MAXP = MAXV * (MAXV - 1) / 2;
constexpr int NXMAX = 7 * MAXV + 1;
constexpr int NUMAX = NP * MAXV;
constexpr int FILTER_MAX = 64;
constexpr double DELTA_C_LOCAL = 1e-8;
#ifndef OBCA_PIVOT_TOL
#define OBCA_PIVOT_TOL 1e-14
#endif
constexpr double PIVOT_TOL = OBCA_PIVOT_TOL;  // relative size below which a Riccati pivot counts as non-positive (wrong inertia -> delta_w is raised)

// ------------------------------------------------------------------------------------------------
// [LAYOUT]
// ------------------------------------------------------------------------------------------------
struct Lay {
  int mode;  // 0 = collocation OBCA (single / joint), 1 = MPC (obca_mpc.h)
  int euler; // mode 1 only: 1 = the Euler-discretised tube-following NLP of Vehicle.state_ws (vehicle.py:99-231) instead of the MPC NLP:
             // forward-Euler dynamics, cost a^2 + w^2, tube sets every npset nodes, a_0 = w_0 = 0, optional final heading; 2 = same
             // with bounded inputs
  int V, O, P, Mv, Nmax, Smax, npset;
  int N[MAXV], M[MAXV], S[MAXV], heading[MAXV];
  int pa[MAXP], pb[MAXP], Mp[MAXP];
  int nPairNodes;  // sum of Mp: the (pair, node) blocks that exist
  // primal fields
  int oZ, oLAM, oMU, oSD, oEL, oTS, oPL, oPM, oPS, oPSD, oPSN, oPEL, oDT, nx;
  // multiplier / residual fields
  int oYINIT, oYCOL, oYCONT, oYTERM, oYOBS, oYTUBE, oYPAIR, ny;
  // Riccati sizes
  int nX, nU;

  OBCA_HD int Z(int a, int c, int n) const { return oZ + (a * NZ + c) * Mv + n; }
  OBCA_HD int LAM(int a, int j, int r, int n) const { return oLAM + ((a * O + j) * 4 + r) * Mv + n; }
  OBCA_HD int MU(int a, int j, int r, int n) const { return oMU + ((a * O + j) * 4 + r) * Mv + n; }
  OBCA_HD int SD(int a, int j, int n) const { return oSD + (a * O + j) * Mv + n; }
  OBCA_HD int EL(int a, int j, int n) const { return oEL + (a * O + j) * Mv + n; }
  OBCA_HD int TS(int a, int q, int r) const { return oTS + (a * (Smax - 1) + q) * 8 + r; }
  OBCA_HD int PL(int p, int r, int n) const { return oPL + (p * 4 + r) * Mv + n; }
  OBCA_HD int PM(int p, int r, int n) const { return oPM + (p * 4 + r) * Mv + n; }
  OBCA_HD int PS(int p, int r, int n) const { return oPS + (p * 2 + r) * Mv + n; }
  OBCA_HD int PSD(int p, int n) const { return oPSD + p * Mv + n; }
  OBCA_HD int PSN(int p, int n) const { return oPSN + p * Mv + n; }
  OBCA_HD int PEL(int p, int n) const { return oPEL + p * Mv + n; }
  OBCA_HD int YINIT(int a, int c) const { return oYINIT + a * NZ + c; }
  OBCA_HD int YCOL(int a, int c, int n) const { return oYCOL + (a * 5 + c) * Mv + n; }
  OBCA_HD int YCONT(int a, int c, int i) const { return oYCONT + (a * NZ + c) * Nmax + i; }
  OBCA_HD int YTERM(int a, int c) const { return oYTERM + a * 5 + c; }
  OBCA_HD int YOBS(int a, int j, int r, int n) const { return oYOBS + ((a * O + j) * 4 + r) * Mv + n; }
  OBCA_HD int YTUBE(int a, int q, int r) const { return oYTUBE + (a * (Smax - 1) + q) * 8 + r; }
  OBCA_HD int YPAIR(int p, int r, int n) const { return oYPAIR + (p * 6 + r) * Mv + n; }
};

inline void lay_offsets(Lay& L);

inline void lay_build(Lay& L, const ObcaDims& d, const double* final_heading) {
  L.mode = 0;
  L.euler = 0;
  L.V = d.V;
  L.O = d.O;
  L.npset = d.n_per_set;
  L.Mv = 0;
  L.Nmax = 0;
  L.Smax = 0;
  for (int a = 0; a < d.V; ++a) {
    L.S[a] = d.n_sets[a];
    L.N[a] = d.n_per_set * (d.n_sets[a] - 1);
    L.M[a] = NK * L.N[a];
    L.heading[a] = final_heading ? (final_heading[a] == final_heading[a]) : 0;
    if (L.M[a] > L.Mv) L.Mv = L.M[a];
    if (L.N[a] > L.Nmax) L.Nmax = L.N[a];
    if (L.S[a] > L.Smax) L.Smax = L.S[a];
  }
  L.P = 0;
  for (int a = 0; a < d.V; ++a)
    for (int b = a + 1; b < d.V; ++b) {
      L.pa[L.P] = a;
      L.pb[L.P] = b;
      L.Mp[L.P] = L.M[a] < L.M[b] ? L.M[a] : L.M[b];
      ++L.P;
    }
  L.nPairNodes = 0;
  for (int p = 0; p < L.P; ++p) L.nPairNodes += L.Mp[p];
  lay_offsets(L);
  L.nX = 7 * L.V + 1;
  L.nU = NP * L.V;
}

inline void lay_offsets(Lay& L) {
  int o = 0;
  L.oZ = o, o += L.V * NZ * L.Mv;
  L.oLAM = o, o += L.V * L.O * 4 * L.Mv;
  L.oMU = o, o += L.V * L.O * 4 * L.Mv;
  L.oSD = o, o += L.V * L.O * L.Mv;
  L.oEL = o, o += L.V * L.O * L.Mv;
  L.oTS = o, o += L.V * (L.Smax - 1) * 8;
  L.oPL = o, o += L.P * 4 * L.Mv;
  L.oPM = o, o += L.P * 4 * L.Mv;
  L.oPS = o, o += L.P * 2 * L.Mv;
  L.oPSD = o, o += L.P * L.Mv;
  L.oPSN = o, o += L.P * L.Mv;
  L.oPEL = o, o += L.P * L.Mv;
  L.oDT = o, o += 1;
  L.nx = o;
  o = 0;
  L.oYINIT = o, o += L.V * NZ;
  L.oYCOL = o, o += L.V * 5 * L.Mv;
  L.oYCONT = o, o += L.V * NZ * L.Nmax;
  L.oYTERM = o, o += L.V * 5;
  L.oYOBS = o, o += L.V * L.O * 4 * L.Mv;
  L.oYTUBE = o, o += L.V * (L.Smax - 1) * 8;
  L.oYPAIR = o, o += L.P * 6 * L.Mv;
  L.ny = o;
}

// MPC problem: one vehicle, N nodes, P other vehicles (parameters); YCOL rows are the dynamics rows
inline void lay_build_mpc(Lay& L, int horizon, int n_obstacles, int n_others) {
  L.mode = 1;
  L.euler = 0;
  L.V = 1, L.O = n_obstacles, L.npset = 1;
  L.Mv = horizon, L.Nmax = 1, L.Smax = 1;
  L.S[0] = 1, L.N[0] = 1, L.M[0] = horizon, L.heading[0] = 0;
  L.P = n_others;
  for (int p = 0; p < n_others; ++p) L.pa[p] = 0, L.pb[p] = 0, L.Mp[p] = horizon;
  L.nPairNodes = n_others * horizon;
  lay_offsets(L);
  L.nX = 5, L.nU = 2;
}


// state warm start (Vehicle.state_ws, vehicle.py:99-231): n_sets strategy sets, nodes_per_set Euler steps per move; nodes
// k = 0 .. nodes_per_set (n_sets - 1), a tube set at every k = nodes_per_set i, i >= 1.  Same flat layout as the MPC problem.
inline void lay_build_state_ws(Lay& L, int n_sets, int nodes_per_set, bool bounded_input, bool has_heading) {
  lay_build_mpc(L, nodes_per_set * (n_sets - 1) + 1, 0, 0);
  L.euler = bounded_input ? 2 : 1;
  L.npset = nodes_per_set;
  L.Smax = n_sets, L.S[0] = n_sets;
  L.heading[0] = has_heading ? 1 : 0;
  lay_offsets(L);
}
// Euler mode: index q >= 1 of the tube set enforced at node n, or -1 (vehicle.py:178-192: k = N i, i = 1 .. M)
OBCA_HD int euler_set_at(const Lay& L, int n) { return (n > 0 && n % L.npset == 0) ? n / L.npset : -1; }

// batch-invariant problem data
struct Stat {
  double obsA[OBCA_MAX_O][4][2], obsb[OBCA_MAX_O][4];
  double G[4][2], g[4];
  double wb, dmin, rho;
  double dt_mpc;  // fixed sample time of the MPC problem (vehicle_follower.py:146)
  double region[4], limits[8];
  double heading[MAXV];
  double cA[NK][NK], cB[NK];  // collocation matrices: cA[j][k] = L_j'(tau_k), cB[k] quadrature weights
  double cAi[5][5];           // inverse of the interior block: sum_j cA[j][k] cAi[j'][k]... i.e. (A1^-1)[j][k], A1[k][j] = cA[j][k], j,k = 1..K
  // tube sets, b already reduced by shrink_tube: [V][Smax][2][4][3] = (ax, ay, b)
  const double* tube;
  OBCA_HD const double* tube_row(const Lay& L, int a, int q, int body, int r) const {
    return tube + ((((a * L.Smax + q) * 2 + body) * 4 + r) * 3);
  }
};

struct Opts {
  double tol, constr_viol_tol, dual_inf_tol, compl_inf_tol, mu_init;
  int max_iter;
  int refine_steps = 0;         // correction solves per Newton system (obca_refine.h)
  double refine_ratio = 1e-10;  // IPOPT residual_ratio_max
  // IPOPT constants (SURVEY.md App. E)
  double kappa_eps = 10.0, kappa_mu = 0.2, theta_mu = 1.5, tau_min = 0.99;
  double bound_push = 1e-2, bound_frac = 1e-2, kappa_sigma = 1e10, kappa_d = 1e-4, s_max = 100.0;
  double gamma_theta = 1e-5, gamma_phi = 1e-8, eta_phi = 1e-8, delta_ls = 1.0, s_theta = 1.1, s_phi = 2.3;
  double gamma_alpha = 0.05;
  double dw_first = 1e-4, dw_min = 1e-20, dw_max = 1e40, kw_minus = 1.0 / 3.0, kw_plus = 8.0, kw_plus_first = 100.0;
};

// per-instance scratch sizes (doubles)
struct Scratch {
  // x-layout vectors
  double *x, *zL, *zU, *dx, *dzL, *dzU, *gl, *gphi, *sig, *xt;
  // y-layout vectors
  double *y, *dy, *c, *ct, *ry;  // ry: correction of dy in the refinement loop (obca_refine.h)
  // best "acceptable" iterate so far (IPOPT StoreAcceptablePoint): x, zL, zU, y
  double *bx, *bzL, *bzU, *by;
  // structured solve
  double* XO;   // [V][O][48][Mv]   obstacle block solves: 12 x (3 coupling cols + 1 rhs), node minor
  double* XP;   // [P][112][Mv]     pair block solves: 16 x (6 + 1), node minor
  double* PH;   // [P][27][Mv]      pair Schur complement on (pose_a, pose_b): 21 sym + 6 grad, node minor
  double* PG;   // [P][6][Mv]       pair contributions to the pose gradient (gl), node minor
  double* HN;   // [V][28][Mv]      node Hessian (sym packed), node minor
  double* GN;   // [V][7][Mv]       node gradient, node minor
  double* HD;   // [V][7][Mv]       node x dt cross Hessian, node minor
  double* TT;   // [V][Nmax][35*13 + 35]   reduced-coordinate map T and particular solution s0
  double* QR;   // [V][Nmax][QRSZ]   Householder factors, tau, pivots, dropped-row records
  double* EM;   // [2][V][Nmax][EXSZ] implied rows emitted to the previous interval (double-buffered by pass)
  double* DF;   // [2][V][Nmax] dirty flags (double-buffered by pass)
  double* MA;   // [V][Nmax][91 + 13]      projected stage Hessian (sym packed 13x13) + gradient
  double* MAB;  // [P][Nmax][169 + 26]     projected cross-vehicle coupling + gradients
  double* RK;   // [Nmax][(nX+1)*nU + nU*nU]   stage records of the Riccati forward pass: Ks' and L
  double* RP;   // [Nmax+1][nX*nX + nX]    cost-to-go
  double* RX;   // [Nmax+1][nX] states, [Nmax][nU] controls
  double* SS;   // [V][Nmax][42] stage solutions
  double* init_pose;  // [V][3]
  double* ricg;       // per-slot global-memory Riccati arena when the stage matrices do not fit shared memory (V > 4), else nullptr
};

// vector lengths are padded to an even number of doubles: every flat vector starts 16-byte aligned, which the bulk
// copies (TMA) of the staged passes need, and may be read one element past its end
OBCA_HD size_t ev(size_t n) { return (n + 1) & ~(size_t)1; }

// per-instance iterate (kept for every instance of the batch): x, zL, zU (x-layout), y (y-layout), init pose
inline size_t iterate_doubles(const Lay& L) {
  size_t par = L.mode == 1 ? 5 + (size_t)3 * L.Mv * (1 + L.P) : (size_t)L.V * 3;  // init poses, or MPC parameters
  return ev(3 * ev(L.nx) + ev(L.ny) + par + 8);
}

// doubles per node of the HN buffer: the packed 7 x 7 node Hessian; in MPC mode the evaluation also uses it as scratch for
// the dynamics / obstacle gradient pieces ([N][5] + [N][O][3], obca_mpc.h), which outgrows 28 per node for O >= 8
OBCA_HD int hn_per_node(const Lay& L) { return (L.mode == 1 && 5 + 3 * L.O > 28) ? 5 + 3 * L.O : 28; }

// per-slot work area (one per resident CTA)
inline size_t work_doubles(const Lay& L) {
  size_t n = 0;
  n += 10 * ev(L.nx) + 5 * ev(L.ny);
  n += (size_t)L.V * L.Mv * L.O * 48;
  n += (size_t)L.P * L.Mv * (112 + 27 + 6);
  n += (size_t)L.V * L.Mv * (hn_per_node(L) + 7 + 7);
  n += (size_t)L.V * L.Nmax * ((NW * NRED + NW) + QRSZ + (NSYM + NRED) + NS + 2 * EXSZ + 2) + EXSZ;
  n += (size_t)L.P * L.Nmax * (NRED * NRED + 2 * NRED);
  n += (size_t)L.Nmax * ((size_t)(L.nX + 1) * L.nU + (size_t)L.nU * L.nU);  // stage records of the Riccati forward pass
  n += (size_t)(L.Nmax + 1) * (L.nX * L.nX + L.nX);
  n += (size_t)(L.Nmax + 1) * L.nX + (size_t)L.Nmax * L.nU;
  return ev(n + 64);
}

OBCA_HD void carve_iterate(Scratch& W, const Lay& L, double* p) {
  const size_t nx = ev(L.nx), ny = ev(L.ny);
  W.x = p, p += nx;
  W.zL = p, p += nx;
  W.zU = p, p += nx;
  W.y = p, p += ny;
  W.init_pose = p;
}

OBCA_HD void carve_work(Scratch& W, const Lay& L, double* p) {
  const size_t nx = ev(L.nx), ny = ev(L.ny);
  W.dx = p, p += nx;
  W.dzL = p, p += nx;
  W.dzU = p, p += nx;
  W.gl = p, p += nx;
  W.gphi = p, p += nx;
  W.sig = p, p += nx;
  W.xt = p, p += nx;
  W.dy = p, p += ny;
  W.c = p, p += ny;
  W.ct = p, p += ny;
  W.bx = p, p += nx;
  W.bzL = p, p += nx;
  W.bzU = p, p += nx;
  W.by = p, p += ny;
  W.ry = p, p += ny;
  W.XO = p, p += (size_t)L.V * L.Mv * L.O * 48;
  W.XP = p, p += (size_t)L.P * L.Mv * 112;
  W.PH = p, p += (size_t)L.P * L.Mv * 27;
  W.PG = p, p += (size_t)L.P * L.Mv * 6;
  W.HN = p, p += (size_t)L.V * L.Mv * hn_per_node(L);
  W.GN = p, p += (size_t)L.V * L.Mv * 7;
  W.HD = p, p += (size_t)L.V * L.Mv * 7;
  W.TT = p, p += (size_t)L.V * L.Nmax * (NW * NRED + NW);
  W.QR = p, p += (size_t)L.V * L.Nmax * QRSZ;
  W.EM = p, p += (size_t)2 * L.V * L.Nmax * EXSZ + EXSZ;
  W.DF = p, p += (size_t)2 * L.V * L.Nmax;
  W.MA = p, p += (size_t)L.V * L.Nmax * (NSYM + NRED);
  W.MAB = p, p += (size_t)L.P * L.Nmax * (NRED * NRED + 2 * NRED);
  W.RK = p, p += (size_t)L.Nmax * ((size_t)(L.nX + 1) * L.nU + (size_t)L.nU * L.nU);
  W.RP = p, p += (size_t)(L.Nmax + 1) * (L.nX * L.nX + L.nX);
  W.RX = p, p += (size_t)(L.Nmax + 1) * L.nX + (size_t)L.Nmax * L.nU;
  W.SS = p;
}

// tells the compiler that every scratch pointer is a global-memory pointer (LDG/STG instead of generic LD/ST)
OBCA_HD void assume_scratch(const Scratch& W) {
  OBCA_ASSUME_GLOBAL(W.x), OBCA_ASSUME_GLOBAL(W.zL), OBCA_ASSUME_GLOBAL(W.zU), OBCA_ASSUME_GLOBAL(W.dx), OBCA_ASSUME_GLOBAL(W.gl);
  OBCA_ASSUME_GLOBAL(W.gphi), OBCA_ASSUME_GLOBAL(W.sig), OBCA_ASSUME_GLOBAL(W.xt), OBCA_ASSUME_GLOBAL(W.y), OBCA_ASSUME_GLOBAL(W.dy);
  OBCA_ASSUME_GLOBAL(W.c), OBCA_ASSUME_GLOBAL(W.ct), OBCA_ASSUME_GLOBAL(W.XO), OBCA_ASSUME_GLOBAL(W.XP), OBCA_ASSUME_GLOBAL(W.PH);
  OBCA_ASSUME_GLOBAL(W.PG), OBCA_ASSUME_GLOBAL(W.HN), OBCA_ASSUME_GLOBAL(W.GN), OBCA_ASSUME_GLOBAL(W.HD), OBCA_ASSUME_GLOBAL(W.TT);
  OBCA_ASSUME_GLOBAL(W.QR), OBCA_ASSUME_GLOBAL(W.EM), OBCA_ASSUME_GLOBAL(W.DF), OBCA_ASSUME_GLOBAL(W.MA), OBCA_ASSUME_GLOBAL(W.MAB);
  OBCA_ASSUME_GLOBAL(W.RK), OBCA_ASSUME_GLOBAL(W.RP), OBCA_ASSUME_GLOBAL(W.RX), OBCA_ASSUME_GLOBAL(W.init_pose);
}

// Lay / Stat live in shared memory inside k_solve (copied once per CTA)
#if defined(__CUDA_ARCH__)
#define OBCA_ASSUME_STATIC(L, S) (__builtin_assume(__isShared(&(L))), __builtin_assume(__isShared(&(S))))
#else
#define OBCA_ASSUME_STATIC(L, S) ((void)0)
#endif

struct Result {
  int status, iters;
  double obj, cviol, dual_inf, compl_inf, mu, dt;
  double elastic;  // largest elastic variable at the returned point
  int refines, restarts;  // correction solves of the refinement loop; dual restorations (obca_ipm.h)
  double rho_carry;       // MPC mode: raised penalty weight kept for the next control step of this vehicle (0: none)
  // obca_warm_start: the next solve starts from the stored iterate (`warm`, cleared by that solve) with barrier parameter mu0 and the
  // pushes of the warm_start_* options in force at the arm.  Here rather than in Opts: k_solve's parameter block keeps its size
  int warm;
  double mu0, ws_bound_push, ws_mult_bound_push;
};

// ------------------------------------------------------------------------------------------------
// execution context: one CTA (device) or one thread (host emulation)
// ------------------------------------------------------------------------------------------------
struct Ctx {
  int tid, nt;
  double* red;  // shared scratch for reductions (>= 40 doubles)
  void* ldl;    // LdlBuf in shared memory: pivot row / column exchange of the Riccati stage factorisation (device only)
  long long* prof;  // optional per-slot phase cycle counters [NPROF + 1] (last = time stamp), or nullptr
};

constexpr int NPROF = 31;  // 16..21: sub-phases of the null-space block (warp 0 only): setup, QR, T columns, store, projection
// phase ids: 0 eval_pairs 1 eval_nodes 2 pair_eliminate 3 node_assemble 4 nullspace 5 cross 6 riccati_bwd 7 riccati_fwd
//            8 expand+node_residual 9 multipliers 10 local_backsub 11 ipm vector ops / line-search bookkeeping
OBCA_HD void prof_mark(const Ctx& ctx, int phase) {
#if defined(__CUDA_ARCH__)
  if (ctx.prof && ctx.tid == 0) {
    long long t = clock64();
    ctx.prof[phase] += t - ctx.prof[NPROF];
    ctx.prof[NPROF] = t;
  }
#else
  (void)ctx;
  (void)phase;
#endif
}

OBCA_HD void cta_sync(const Ctx&) {
#if defined(__CUDA_ARCH__)
  __syncthreads();
#endif
}

// op: 0 sum, 1 max, 2 min.  Deterministic (fixed tree).  All threads get the result.
OBCA_HD double cta_reduce(const Ctx& ctx, double v, int op) {
#if defined(__CUDA_ARCH__)
  for (int o = 16; o > 0; o >>= 1) {
    double w = __shfl_down_sync(0xffffffffu, v, o);
    v = op == 0 ? v + w : (op == 1 ? fmax(v, w) : fmin(v, w));
  }
  int lane = ctx.tid & 31, wid = ctx.tid >> 5, nw = (ctx.nt + 31) >> 5;
  __syncthreads();
  if (lane == 0) ctx.red[wid] = v;
  __syncthreads();
  if (wid == 0) {
    double neutral = op == 0 ? 0.0 : (op == 1 ? -INFINITY : INFINITY);
    v = lane < nw ? ctx.red[lane] : neutral;
    for (int o = 16; o > 0; o >>= 1) {
      double w = __shfl_down_sync(0xffffffffu, v, o);
      v = op == 0 ? v + w : (op == 1 ? fmax(v, w) : fmin(v, w));
    }
    if (lane == 0) ctx.red[32] = v;
  }
  __syncthreads();
  return ctx.red[32];
#else
  (void)ctx;
  (void)op;
  return v;
#endif
}
OBCA_HD double cta_sum(const Ctx& c, double v) { return cta_reduce(c, v, 0); }
OBCA_HD double cta_max(const Ctx& c, double v) { return cta_reduce(c, v, 1); }
OBCA_HD double cta_min(const Ctx& c, double v) { return cta_reduce(c, v, 2); }

// ------------------------------------------------------------------------------------------------
// small dense helpers (thread-local)
// ------------------------------------------------------------------------------------------------
OBCA_HD int sym(int r, int c) { return r >= c ? r * (r + 1) / 2 + c : c * (c + 1) / 2 + r; }

// In-place LDL' without pivoting of the symmetric matrix A (full storage, ld = n, lower part used).
// Returns the number of negative pivots, or -1 when a pivot vanishes.
template <int N>
OBCA_HD int ldl_factor(double* A) {
  int nneg = 0;
  for (int j = 0; j < N; ++j) {
    double d = A[j * N + j];
    for (int k = 0; k < j; ++k) d -= A[j * N + k] * A[j * N + k] * A[k * N + k];
    if (!(fabs(d) > 1e-300)) return -1;
    A[j * N + j] = d;
    if (d < 0) ++nneg;
    double inv = 1.0 / d;
    for (int i = j + 1; i < N; ++i) {
      double v = A[i * N + j];
      for (int k = 0; k < j; ++k) v -= A[i * N + k] * A[j * N + k] * A[k * N + k];
      A[i * N + j] = v * inv;
    }
  }
  return nneg;
}

template <int N>
OBCA_HD void ldl_solve(const double* A, double* b, int stride) {
  for (int i = 0; i < N; ++i) {
    double v = b[i * stride];
    for (int k = 0; k < i; ++k) v -= A[i * N + k] * b[k * stride];
    b[i * stride] = v;
  }
  for (int i = 0; i < N; ++i) b[i * stride] /= A[i * N + i];
  for (int i = N - 1; i >= 0; --i) {
    double v = b[i * stride];
    for (int k = i + 1; k < N; ++k) v -= A[k * N + i] * b[k * stride];
    b[i * stride] = v;
  }
}

// Cholesky of a small SPD matrix in packed lower storage (sym(r, c)); the diagonal holds 1 / L_jj afterwards (the
// solves multiply instead of dividing: FP64 division costs ~30 instructions).  Returns false on a non-positive pivot.
template <int N>
OBCA_HD bool chol_packed(double* A) {
  bool good = true;
#pragma unroll
  for (int j = 0; j < N; ++j) {
    double d = A[sym(j, j)];
#pragma unroll
    for (int k = 0; k < j; ++k) d -= A[sym(j, k)] * A[sym(j, k)];
    if (!(d > 0)) good = false, d = 1.0;
#if defined(__CUDA_ARCH__)
    const double inv = rsqrt(d);  // 1 ulp, a third of the instructions of 1.0 / sqrt(d)
#else
    const double inv = 1.0 / sqrt(d);
#endif
    A[sym(j, j)] = inv;
#pragma unroll
    for (int i = j + 1; i < N; ++i) {
      double v = A[sym(i, j)];
#pragma unroll
      for (int k = 0; k < j; ++k) v -= A[sym(i, k)] * A[sym(j, k)];
      A[sym(i, j)] = v * inv;
    }
  }
  return good;
}

template <int N>
OBCA_HD void chol_solve_packed(const double* A, double* b) {
#pragma unroll
  for (int i = 0; i < N; ++i) {
    double v = b[i];
#pragma unroll
    for (int k = 0; k < i; ++k) v -= A[sym(i, k)] * b[k];
    b[i] = v * A[sym(i, i)];
  }
#pragma unroll
  for (int i = N - 1; i >= 0; --i) {
    double v = b[i];
#pragma unroll
    for (int k = i + 1; k < N; ++k) v -= A[sym(k, i)] * b[k];
    b[i] = v * A[sym(i, i)];
  }
}

// 1 / d for a positive, normal d (gaps to the bounds, pivots).  Device: hardware seed (MUFU.RCP64H, ~20 bits) + two Newton
// steps, within 1 ulp -- a sixth of the instructions of the IEEE division sequence; the flat passes of the interior-point loop
// are bound by exactly that instruction latency.  Host emulation: plain division.
OBCA_HD double rcp_pos(double d) {
#if defined(__CUDA_ARCH__)
  double x;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(d));
  x = fma(x, fma(-d, x, 1.0), x);
  x = fma(x, fma(-d, x, 1.0), x);
  return x;
#else
  return 1.0 / d;
#endif
}

struct Pose {
  double x, y, psi, c, s;
};

// ------------------------------------------------------------------------------------------------
// [EVAL] + [LOCAL] obstacle block at one node
//   c1 = -g'mu + (A t - b)'lam - dmin - sd ; c2 = G'mu + R(psi)'A'lam ; c3 = |A'lam|^2 - 1
// ------------------------------------------------------------------------------------------------
struct ObsBlk {
  double lam[4], mu[4], sd, el;
  double Atb[4];   // A t - b
  double u[2];     // A'lam
  double c[4];
};

OBCA_HD void obs_residual(const Stat& S, int j, const Pose& p, ObsBlk& B) {
  const double(*A)[2] = S.obsA[j];
  B.u[0] = B.u[1] = 0;
  double c1 = -S.dmin - B.sd + B.el;
  double gm0 = 0, gm1 = 0;
  for (int r = 0; r < 4; ++r) {
    B.Atb[r] = A[r][0] * p.x + A[r][1] * p.y - S.obsb[j][r];
    B.u[0] += A[r][0] * B.lam[r];
    B.u[1] += A[r][1] * B.lam[r];
    c1 += B.Atb[r] * B.lam[r] - S.g[r] * B.mu[r];
    gm0 += S.G[r][0] * B.mu[r];
    gm1 += S.G[r][1] * B.mu[r];
  }
  B.c[0] = c1;
  B.c[1] = gm0 + p.c * B.u[0] + p.s * B.u[1];   // (R'u)_0
  B.c[2] = gm1 - p.s * B.u[0] + p.c * B.u[1];   // (R'u)_1
  B.c[3] = B.u[0] * B.u[0] + B.u[1] * B.u[1] - 1.0;
}

// ------------------------------------------------------------------------------------------------
// pair block at one node:  A_i = G R(psi_i)', b_i = A_i t_i + g
//   d = -b_a'lam - b_b'mu - dmin - sd ; e1 = A_a'lam + s ; e2 = A_b'mu - s ; n = 1 - s's - sn
// ------------------------------------------------------------------------------------------------
struct PairBlk {
  double lam[4], mu[4], s[2], sd, sn, el;
  double ua[2], ub[2];     // G'lam, G'mu
  double Rua[2], Rub[2];   // R_a ua, R_b ub
  double ba[4], bb[4];
  double c[6];
};

OBCA_HD void pair_residual(const Stat& S, const Pose& a, const Pose& b, PairBlk& B) {
  B.ua[0] = B.ua[1] = B.ub[0] = B.ub[1] = 0;
  double d = -S.dmin - B.sd + B.el;
  for (int r = 0; r < 4; ++r) {
    B.ua[0] += S.G[r][0] * B.lam[r];
    B.ua[1] += S.G[r][1] * B.lam[r];
    B.ub[0] += S.G[r][0] * B.mu[r];
    B.ub[1] += S.G[r][1] * B.mu[r];
    // A_a row r = G_r R_a' ; R' = [[c, s], [-s, c]]
    double aax = S.G[r][0] * a.c - S.G[r][1] * a.s, aay = S.G[r][0] * a.s + S.G[r][1] * a.c;
    double abx = S.G[r][0] * b.c - S.G[r][1] * b.s, aby = S.G[r][0] * b.s + S.G[r][1] * b.c;
    B.ba[r] = aax * a.x + aay * a.y + S.g[r];
    B.bb[r] = abx * b.x + aby * b.y + S.g[r];
    d -= B.ba[r] * B.lam[r] + B.bb[r] * B.mu[r];
  }
  B.Rua[0] = a.c * B.ua[0] - a.s * B.ua[1];
  B.Rua[1] = a.s * B.ua[0] + a.c * B.ua[1];
  B.Rub[0] = b.c * B.ub[0] - b.s * B.ub[1];
  B.Rub[1] = b.s * B.ub[0] + b.c * B.ub[1];
  B.c[0] = d;
  B.c[1] = B.Rua[0] + B.s[0];
  B.c[2] = B.Rua[1] + B.s[1];
  B.c[3] = B.Rub[0] - B.s[0];
  B.c[4] = B.Rub[1] - B.s[1];
  B.c[5] = 1.0 - B.s[0] * B.s[0] - B.s[1] * B.s[1] - B.sn;
}

OBCA_HD void load_pose(const Lay& L, const double* x, int a, int n, Pose& p) {
  p.x = x[L.Z(a, 0, n)];
  p.y = x[L.Z(a, 1, n)];
  p.psi = x[L.Z(a, 2, n)];
  p.c = cos(p.psi);
  p.s = sin(p.psi);
}

OBCA_HD void load_pair(const Lay& L, const double* x, int p, int n, PairBlk& B) {
  for (int r = 0; r < 4; ++r) B.lam[r] = x[L.PL(p, r, n)], B.mu[r] = x[L.PM(p, r, n)];
  B.s[0] = x[L.PS(p, 0, n)];
  B.s[1] = x[L.PS(p, 1, n)];
  B.sd = x[L.PSD(p, n)];
  B.sn = x[L.PSN(p, n)];
  B.el = x[L.PEL(p, n)];
}

// which tube set (if any) is enforced at node n of vehicle a: returns set index q >= 1 or -1.
// Transition nodes (i = q * n_per_set, k = 0, vehicle.py:570-584) and the end state (last node with the last
// set, vehicle.py:605-617; D = e_K so zF is the last node itself).
OBCA_HD int tube_set_at(const Lay& L, int a, int n) {
  if (n == L.M[a] - 1) return L.S[a] - 1;
  int i = n / NK, k = n % NK;
  if (k == 0 && i > 0 && i % L.npset == 0) return i / L.npset;
  return -1;
}

// ------------------------------------------------------------------------------------------------
// [EVAL] pair phase: residuals, gl of the pair variables, pose-gradient contributions -> PG
// ------------------------------------------------------------------------------------------------
OBCA_HDN void eval_pairs(const Ctx& ctx, const Lay& L, const Stat& S, const double* x, const double* y, double* c,
                         double* gl, double* PG) {
  OBCA_ASSUME_STATIC(L, S);
  OBCA_ASSUME_GLOBAL(x), OBCA_ASSUME_GLOBAL(c), OBCA_ASSUME_GLOBAL(PG);
  if (y) OBCA_ASSUME_GLOBAL(y), OBCA_ASSUME_GLOBAL(gl);
  for (int it = ctx.tid; it < L.nPairNodes; it += ctx.nt) {  // compact index over the existing (pair, node) blocks
    int p = 0, n = it;
    while (n >= L.Mp[p]) n -= L.Mp[p], ++p;
    Pose a, b;
    load_pose(L, x, L.pa[p], n, a);
    load_pose(L, x, L.pb[p], n, b);
    PairBlk B;
    load_pair(L, x, p, n, B);
    pair_residual(S, a, b, B);
    for (int r = 0; r < 6; ++r) c[L.YPAIR(p, r, n)] = B.c[r];
    if (!y) continue;
    double yd = y[L.YPAIR(p, 0, n)], ye1[2] = {y[L.YPAIR(p, 1, n)], y[L.YPAIR(p, 2, n)]};
    double ye2[2] = {y[L.YPAIR(p, 3, n)], y[L.YPAIR(p, 4, n)]}, yn = y[L.YPAIR(p, 5, n)];
    // R_a' ye1, R_b' ye2
    double Rtea[2] = {a.c * ye1[0] + a.s * ye1[1], -a.s * ye1[0] + a.c * ye1[1]};
    double Rteb[2] = {b.c * ye2[0] + b.s * ye2[1], -b.s * ye2[0] + b.c * ye2[1]};
    for (int r = 0; r < 4; ++r) {
      gl[L.PL(p, r, n)] = -yd * B.ba[r] + S.G[r][0] * Rtea[0] + S.G[r][1] * Rtea[1];
      gl[L.PM(p, r, n)] = -yd * B.bb[r] + S.G[r][0] * Rteb[0] + S.G[r][1] * Rteb[1];
    }
    gl[L.PS(p, 0, n)] = ye1[0] - ye2[0] - 2.0 * yn * B.s[0];
    gl[L.PS(p, 1, n)] = ye1[1] - ye2[1] - 2.0 * yn * B.s[1];
    gl[L.PSD(p, n)] = -yd;
    gl[L.PSN(p, n)] = -yn;
    gl[L.PEL(p, n)] = S.rho + yd;
    // pose gradients: d/dt_a = -yd R_a ua ; d/dpsi_a = -yd t_a' R_a' ua + ye1' R_a' ua   (R' = dR/dpsi here)
    double dRua[2] = {-a.s * B.ua[0] - a.c * B.ua[1], a.c * B.ua[0] - a.s * B.ua[1]};
    double dRub[2] = {-b.s * B.ub[0] - b.c * B.ub[1], b.c * B.ub[0] - b.s * B.ub[1]};
    double* g = PG + (size_t)p * 6 * L.Mv + n;  // [P][6][Mv], node minor
    const int gs = L.Mv;
    g[0] = -yd * B.Rua[0];
    g[gs] = -yd * B.Rua[1];
    g[2 * gs] = -yd * (a.x * dRua[0] + a.y * dRua[1]) + ye1[0] * dRua[0] + ye1[1] * dRua[1];
    g[3 * gs] = -yd * B.Rub[0];
    g[4 * gs] = -yd * B.Rub[1];
    g[5 * gs] = -yd * (b.x * dRub[0] + b.y * dRub[1]) + ye2[0] * dRub[0] + ye2[1] * dRub[1];
  }
}

// ------------------------------------------------------------------------------------------------
// [EVAL] node phase.  y == nullptr: residuals and objective only (line-search trial points).
// Returns (through the reductions) the objective f and d(f + y'c)/d dt.
// ------------------------------------------------------------------------------------------------
OBCA_HDN void eval_nodes(const Ctx& ctx, const Lay& L, const Stat& S, const double* init_pose, const double* x,
                         const double* y, double* c, double* gl, const double* PG, double* f_out, double* gdt_out) {
  OBCA_ASSUME_STATIC(L, S);
  OBCA_ASSUME_GLOBAL(x), OBCA_ASSUME_GLOBAL(c), OBCA_ASSUME_GLOBAL(PG), OBCA_ASSUME_GLOBAL(init_pose);
  if (y) OBCA_ASSUME_GLOBAL(y), OBCA_ASSUME_GLOBAL(gl);
  const double dt = x[L.oDT];
  const double idt = 1.0 / dt;
  double f_part = 0, gdt_part = 0;
  for (int it = ctx.tid; it < L.V * L.Mv; it += ctx.nt) {
    int a = it / L.Mv, n = it % L.Mv;
    if (n >= L.M[a]) continue;
    int i = n / NK, k = n % NK, n0 = i * NK;
    double z[NZ];
    for (int q = 0; q < NZ; ++q) z[q] = x[L.Z(a, q, n)];
    Pose p = {z[0], z[1], z[2], cos(z[2]), sin(z[2])};
    double v = z[3], de = z[4], ua = z[5], uw = z[6];
    double tde = tan(de), sec2 = 1.0 + tde * tde;
    // collocation residual: sum_j cA[j][k] z_j / dt - f(z_k, u_k)
    double poly[5];
    for (int q = 0; q < 5; ++q) {
      double s = 0;
      for (int j = 0; j < NK; ++j) s += S.cA[j][k] * x[L.Z(a, q, n0 + j)];
      poly[q] = s * idt;
    }
    double fz[5] = {v * p.c, v * p.s, v * tde / S.wb, ua, uw};
    for (int q = 0; q < 5; ++q) c[L.YCOL(a, q, n)] = poly[q] - fz[q];
    double err = ua * ua + v * v * uw * uw + de * de;
    f_part += S.cB[k] * err * dt;
    // continuity (row i, i >= 1): z_{i-1,K} - z_{i,0}
    if (k == 0 && i >= 1)
      for (int q = 0; q < NZ; ++q) c[L.YCONT(a, q, i)] = x[L.Z(a, q, n - 1)] - z[q];
    if (n == 0) {
      for (int q = 0; q < 3; ++q) c[L.YINIT(a, q)] = z[q] - init_pose[a * 3 + q];
      for (int q = 3; q < NZ; ++q) c[L.YINIT(a, q)] = z[q];
    }
    if (n == L.M[a] - 1) {
      c[L.YTERM(a, 0)] = L.heading[a] ? z[2] - S.heading[a] : 0.0;
      for (int q = 3; q < NZ; ++q) c[L.YTERM(a, q - 2)] = z[q];
    }
    double g[NZ] = {0, 0, 0, 0, 0, 0, 0};
    if (y) {
      double yc[5];
      for (int q = 0; q < 5; ++q) yc[q] = y[L.YCOL(a, q, n)];
      g[3] = S.cB[k] * dt * 2.0 * v * uw * uw;
      g[4] = S.cB[k] * dt * 2.0 * de;
      g[5] = S.cB[k] * dt * 2.0 * ua;
      g[6] = S.cB[k] * dt * 2.0 * v * v * uw;
      for (int q = 0; q < 5; ++q) {
        double s = 0;
        for (int kk = 0; kk < NK; ++kk) s += S.cA[k][kk] * y[L.YCOL(a, q, n0 + kk)];
        g[q] += s * idt;
        gdt_part -= yc[q] * poly[q] * idt;
      }
      gdt_part += S.cB[k] * err;
      g[2] -= yc[0] * (-v * p.s) + yc[1] * (v * p.c);
      g[3] -= yc[0] * p.c + yc[1] * p.s + yc[2] * tde / S.wb;
      g[4] -= yc[2] * v * sec2 / S.wb;
      g[5] -= yc[3];
      g[6] -= yc[4];
      if (k == NK - 1 && i < L.N[a] - 1)
        for (int q = 0; q < NZ; ++q) g[q] += y[L.YCONT(a, q, i + 1)];
      if (k == 0 && i >= 1)
        for (int q = 0; q < NZ; ++q) g[q] -= y[L.YCONT(a, q, i)];
      if (n == 0)
        for (int q = 0; q < NZ; ++q) g[q] += y[L.YINIT(a, q)];
      if (n == L.M[a] - 1) {
        if (L.heading[a]) g[2] += y[L.YTERM(a, 0)];
        for (int q = 3; q < NZ; ++q) g[q] += y[L.YTERM(a, q - 2)];
      }
    }
    // obstacles
    for (int j = 0; j < L.O; ++j) {
      ObsBlk B;
      for (int r = 0; r < 4; ++r) B.lam[r] = x[L.LAM(a, j, r, n)], B.mu[r] = x[L.MU(a, j, r, n)];
      B.sd = x[L.SD(a, j, n)];
      B.el = x[L.EL(a, j, n)];
      f_part += S.rho * B.el;
      obs_residual(S, j, p, B);
      for (int r = 0; r < 4; ++r) c[L.YOBS(a, j, r, n)] = B.c[r];
      if (!y) continue;
      double y1 = y[L.YOBS(a, j, 0, n)], y2[2] = {y[L.YOBS(a, j, 1, n)], y[L.YOBS(a, j, 2, n)]}, y3 = y[L.YOBS(a, j, 3, n)];
      double Ry[2] = {p.c * y2[0] - p.s * y2[1], p.s * y2[0] + p.c * y2[1]};  // R y2
      for (int r = 0; r < 4; ++r) {
        const double* A = S.obsA[j][r];
        gl[L.LAM(a, j, r, n)] = y1 * B.Atb[r] + A[0] * Ry[0] + A[1] * Ry[1] + 2.0 * y3 * (A[0] * B.u[0] + A[1] * B.u[1]);
        gl[L.MU(a, j, r, n)] = -y1 * S.g[r] + S.G[r][0] * y2[0] + S.G[r][1] * y2[1];
      }
      gl[L.SD(a, j, n)] = -y1;
      gl[L.EL(a, j, n)] = S.rho + y1;
      g[0] += y1 * B.u[0];
      g[1] += y1 * B.u[1];
      // d/dpsi of y2' R'u : R' = [[c,s],[-s,c]] -> dR'/dpsi = [[-s,c],[-c,-s]]
      g[2] += y2[0] * (-p.s * B.u[0] + p.c * B.u[1]) + y2[1] * (-p.c * B.u[0] - p.s * B.u[1]);
    }
    // tube set
    int q = tube_set_at(L, a, n);
    if (q >= 1) {
      double fx = p.x + S.wb * p.c, fy = p.y + S.wb * p.s;
      for (int r = 0; r < 4; ++r) {
        const double* tb = S.tube_row(L, a, q, 0, r);
        const double* tf = S.tube_row(L, a, q, 1, r);
        c[L.YTUBE(a, q - 1, r)] = tb[2] - tb[0] * p.x - tb[1] * p.y - x[L.TS(a, q - 1, r)];
        c[L.YTUBE(a, q - 1, 4 + r)] = tf[2] - tf[0] * fx - tf[1] * fy - x[L.TS(a, q - 1, 4 + r)];
        if (y) {
          double yb = y[L.YTUBE(a, q - 1, r)], yf = y[L.YTUBE(a, q - 1, 4 + r)];
          gl[L.TS(a, q - 1, r)] = -yb;
          gl[L.TS(a, q - 1, 4 + r)] = -yf;
          g[0] -= tb[0] * yb + tf[0] * yf;
          g[1] -= tb[1] * yb + tf[1] * yf;
          g[2] -= yf * S.wb * (-tf[0] * p.s + tf[1] * p.c);
        }
      }
    }
    if (y) {
      for (int pp = 0; pp < L.P; ++pp) {
        if (n >= L.Mp[pp]) continue;
        const double* pg = PG + (size_t)pp * 6 * L.Mv + n;
        const int gs = L.Mv;
        if (L.pa[pp] == a) g[0] += pg[0], g[1] += pg[gs], g[2] += pg[2 * gs];
        if (L.pb[pp] == a) g[0] += pg[3 * gs], g[1] += pg[4 * gs], g[2] += pg[5 * gs];
      }
      for (int qq = 0; qq < NZ; ++qq) gl[L.Z(a, qq, n)] = g[qq];
    }
  }
  for (int it = ctx.tid; it < L.P * L.Mv; it += ctx.nt) {
    int pp = it / L.Mv, n = it % L.Mv;
    if (n < L.Mp[pp]) f_part += S.rho * x[L.PEL(pp, n)];
  }
  double f = cta_sum(ctx, f_part);
  for (int a = 0; a < L.V; ++a) f += (L.N[a] * dt) * (L.N[a] * dt);
  *f_out = f;
  if (y) {
    double gdt = cta_sum(ctx, gdt_part);
    for (int a = 0; a < L.V; ++a) gdt += 2.0 * L.N[a] * L.N[a] * dt;
    *gdt_out = gdt;
    if (ctx.tid == 0) gl[L.oDT] = gdt;
  }
}

OBCA_HDN void eval_all(const Ctx& ctx, const Lay& L, const Stat& S, const Scratch& W, const double* x, const double* y,
                       double* c, double* gl, double* f, double* gdt) {
  prof_mark(ctx, 11);
  eval_pairs(ctx, L, S, x, y, c, gl, W.PG);
  cta_sync(ctx);
  prof_mark(ctx, 0);
  eval_nodes(ctx, L, S, W.init_pose, x, y, c, gl, W.PG, f, gdt);
  cta_sync(ctx);
  prof_mark(ctx, 1);
}

}  // namespace obca

#include "obca_kkt.h"
#include "obca_mpc.h"
#include "obca_ws.h"
#include "obca_traj.h"
#include "obca_refine.h"
#include "obca_ipm.h"
