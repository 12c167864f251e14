// Single-thread host build of the device solver source (DG_HOSTSIM).  TEST HARNESS ONLY: lets the
// CPU test-suite exercise the exact kernel source (arithmetic, control flow, memory bounds under
// ASan) on machines without a GPU.  It is not part of the product library and nothing in
// dgsqp_b200/ loads it.  Compiled once per game (-DDG_GAME_MERGE selects the merge game, see csrc/game.cuh).
#define DG_HOSTSIM 1
#include <cstdlib>
#include <cstring>
#include <vector>
#include "../../dgsqp_b200/csrc/sqp_v2.cuh"
#include "../../dgsqp_b200/csrc/host_setup.h"

#ifndef DG_GAME_MERGE
#include "../../dgsqp_b200/csrc/pid_rollout.cuh"
extern "C" int hs_pid_rollout(const dgsqp_racing_game* g, const double* key_pts, int K, const double* s0, const double* xt0,
                              const double* v0, double* q0, double* xy, double* u_ws) {
  RolloutParams P;
  if (ro_fill(g, key_pts, &P) != 0) return -1;
  for (int i = 0; i < K; ++i) ro_agent(P, s0[i], xt0[i], v0[i], q0 + (size_t)i * 6, xy + (size_t)i * (P.N + 1) * 2, u_ws + (size_t)i * P.N * 2);
  return 0;
}
#endif

extern "C" {

struct HsHandle { GameDesc G; SolverParams P; Dims D; std::vector<double> ws, sh; Workspace W; MemPlan plan; std::vector<double*> guards; };
static const double HS_CANARY = -7.25e77;

static void* hs_create_common(const dg_game_struct* g, const dgsqp_params* p, const dgsqp_v2_params* p2) {
  HsHandle* h = new HsHandle();
  if (dg_fill_game(g, &h->G) != 0 || (p2 ? dg_fill_params_v2(p2, &h->P) : dg_fill_params(p, &h->P)) != 0) { delete h; return nullptr; }
  h->D = make_dims(h->G.M, h->G.N);
  Workspace tmp;
  const char* lim = getenv("DG_HOSTSIM_SMEM_DOUBLES");      // tests cover both placements
  size_t budget = lim ? (size_t)atol(lim) : 28000;
  MemPlan pl = plan_memory(h->D, nullptr, nullptr, budget, tmp);
  h->plan = pl;
  h->ws.assign(pl.gmem + 2, 0.0);
  h->sh.assign(pl.smem + 2, 0.0);
#ifdef DG_PLAN_GUARD
  dg_guard_n = 0;
#endif
  plan_memory(h->D, h->ws.data(), h->sh.data(), budget, h->W);
#ifdef DG_PLAN_GUARD
  // guard mode: every buffer of the plan is followed by DG_PLAN_GUARD canary doubles (see plan_memory)
  h->guards.assign(dg_guard_at, dg_guard_at + dg_guard_n);
  for (double* g : h->guards) for (int i = 0; i < DG_PLAN_GUARD; ++i) g[i] = HS_CANARY;
#endif
  game_bind(h->W.E, &h->G);
  { Cta c; game_row_table<false>(c, h->D, h->W.E.rowtab); }
  return h;
}
void* hs_create(const dg_game_struct* g, const dgsqp_params* p) { return hs_create_common(g, p, nullptr); }
void* hs_create_v2(const dg_game_struct* g, const dgsqp_v2_params* p) { return hs_create_common(g, nullptr, p); }
// number of canary doubles behind the buffers of the memory plan that no longer hold the canary (guard build only)
int hs_guard_check(void* hp) {
  HsHandle* h = (HsHandle*)hp;
  int bad = 0;
#ifdef DG_PLAN_GUARD
  for (double* g : h->guards) for (int i = 0; i < DG_PLAN_GUARD; ++i) bad += g[i] != HS_CANARY;
  if (h->guards.empty()) return -1;
#else
  bad = -1;
#endif
  return bad;
}
void hs_set_l0_perturb(void* hp, double v) { ((HsHandle*)hp)->P.dbg_l0_perturb = v; }
void hs_destroy(void* hp) { delete (HsHandle*)hp; }
void hs_dims(void* hp, int* out) { HsHandle* h = (HsHandle*)hp; out[0] = h->D.nq; out[1] = h->D.nu; out[2] = h->D.n; out[3] = h->D.m; }
// memory plan: {hot_in_smem, mats_in_smem, matA_in_smem, sens_in_smem, eig_s set} (as tests/gpu_units/units.cu reports it)
void hs_plan(void* hp, int* out) {
  HsHandle* h = (HsHandle*)hp;
  out[0] = h->plan.hot_in_smem; out[1] = h->plan.mats_in_smem; out[2] = h->plan.matA_in_smem; out[3] = h->plan.sens_in_smem;
  out[4] = h->W.B.eig_s != nullptr;
}

// full evaluation at (u, l): returns Q[n*n], q[n], gtl[n], g[m], x
void hs_evaluate(void* hp, const double* x0, const double* u, const double* l, double* Q, double* q, double* gtl,
                 double* g, double* x) {
  HsHandle* h = (HsHandle*)hp; Cta c;
  SolveCtx X; X.G = &h->G; X.P = &h->P; X.D = h->D; X.W = h->W; X.x0 = x0; X.up_in = nullptr;
  for (int i = 0; i < h->D.nu; ++i) h->W.S.up[i] = 0.0;
  eval_full<false>(c, X, u, l);
  memcpy(Q, h->W.E.Q, sizeof(double) * h->D.n * h->D.n);
  memcpy(q, h->W.E.q, sizeof(double) * h->D.n);
  memcpy(gtl, h->W.E.gtl, sizeof(double) * h->D.n);
  memcpy(g, h->W.E.g, sizeof(double) * h->D.m);
  memcpy(x, h->W.E.x, sizeof(double) * (h->D.N + 1) * h->D.nq);
}
// dense G (m x n) at the last evaluated point, via row extraction; plus G v and G' w products
void hs_G_dense(void* hp, double* Gd) {
  HsHandle* h = (HsHandle*)hp; Cta c;
  for (int r = 0; r < h->D.m; ++r) game_G_row<false>(c, h->D, h->W.E, r, Gd + (size_t)r * h->D.n);
}
void hs_G_times(void* hp, const double* v, double* y) { HsHandle* h = (HsHandle*)hp; Cta c; game_G_times<false>(c, h->D, h->W.E, v, y); }
void hs_GT_times(void* hp, const double* w, double* y) { HsHandle* h = (HsHandle*)hp; Cta c; game_GT_times<false>(c, h->D, h->W.E, w, y); }

int hs_nearest_pd(void* hp, const double* Qin, double* Hout) {
  HsHandle* h = (HsHandle*)hp; Cta c;
  int nn = nearest_pd<false>(c, h->D.n, Qin, h->W.B, h->P.eig_floor, h->P.reg, h->P.conv_approx != 0);
  for (int i = 0; i < h->D.n; ++i) memcpy(Hout + (size_t)i * h->D.n, h->W.B.matA + (size_t)i * h->D.ld, sizeof(double) * h->D.n);
  return nn;
}
// QP at the last evaluated point with the given H (n*n, destroyed) and q; warm != 0 starts from the active set of the
// previous QP of this handle
static int hs_qp_common(HsHandle* h, double* H, const double* q, double* du, double* lam, int* iters, int warm) {
  Cta c;
  int na = 0;
  for (int i = 0; i < h->D.n; ++i) memcpy(h->W.B.matA + (size_t)i * h->D.ld, H + (size_t)i * h->D.n, sizeof(double) * h->D.n);
  std::vector<double> qc(q, q + h->D.n);      // q may alias workspace the solver reuses
  int st = qp_solve_gi<false>(c, h->D, h->W.E, qc.data(), h->W.Q, h->W.B, iters, &na, warm);
  memcpy(du, h->W.Q.xq, sizeof(double) * h->D.n);
  memcpy(lam, h->W.Q.lam, sizeof(double) * h->D.m);
  return st;
}
int hs_qp(void* hp, double* H, const double* q, double* du, double* lam, int* iters) { return hs_qp_common((HsHandle*)hp, H, q, du, lam, iters, 0); }
// H into matA, q into a private copy, the offsets g[m] (if given) in place of the evaluated ones and the warm-start list
// prev[0..k) into Q.act; false if the list is out of range.  The caller restores E.g from gsave.
static bool hs_qp_inputs(HsHandle* h, const double* H, const double* q, const double* g, const int* prev, int k,
                         std::vector<double>& qc, std::vector<double>& gsave) {
  const int n = h->D.n, m = h->D.m;
  if (k < 0 || k > n || (k > 0 && !prev)) return false;
  for (int i = 0; i < k; ++i) if (prev[i] < 0 || prev[i] >= m) return false;
  for (int i = 0; i < n; ++i) memcpy(h->W.B.matA + (size_t)i * h->D.ld, H + (size_t)i * n, sizeof(double) * n);
  qc.assign(q, q + n);
  gsave.assign(h->W.E.g, h->W.E.g + m);
  if (g) memcpy(h->W.E.g, g, sizeof(double) * m);
  for (int i = 0; i < k; ++i) h->W.Q.act[i] = prev[i];
  h->W.Q.act[n] = k;
  return true;
}
// QP at the last evaluated point with H (n*n), q and, if given, the offsets g[m] in place of the evaluated ones; from the
// warm-start list prev[0..k) if k > 0, cold otherwise.  out = {status, main-loop iterations, active rows}
int hs_qp_g(void* hp, const double* H, const double* q, const double* g, const int* prev, int k, double* du, double* lam,
            int* out) {
  HsHandle* h = (HsHandle*)hp; Cta c;
  std::vector<double> qc, gsave;
  if (!hs_qp_inputs(h, H, q, g, prev, k, qc, gsave)) return -1;
  int it = 0, na = 0;
  out[0] = qp_solve_gi<false>(c, h->D, h->W.E, qc.data(), h->W.Q, h->W.B, &it, &na, k > 0);
  out[1] = it; out[2] = na;
  memcpy(du, h->W.Q.xq, sizeof(double) * h->D.n);
  memcpy(lam, h->W.Q.lam, sizeof(double) * h->D.m);
  memcpy(h->W.E.g, gsave.data(), sizeof(double) * h->D.m);
  return 0;
}
// qp_factor and gi_warm_start from prev[0..k) (k >= 1) only: returns iq (-1: H not positive definite, -2: bad list) and
// the S-pair the main loop would start from, act[0..iq), xq[n], lam_act[0..iq)
int hs_warm_start(void* hp, const double* H, const double* q, const double* g, const int* prev, int k, int* act,
                  double* xq, double* lam_act) {
  HsHandle* h = (HsHandle*)hp; Cta c;
  std::vector<double> qc, gsave;
  if (k < 1 || !hs_qp_inputs(h, H, q, g, prev, k, qc, gsave)) return -2;
  int iq = -1;
  if (qp_factor<false>(c, h->D, qc.data(), h->W.Q, h->W.B)) {
    iq = gi_warm_start<false>(c, h->D, h->W.E, qc.data(), h->W.Q, h->W.B, k);
    memcpy(act, h->W.Q.act, sizeof(int) * iq);
    memcpy(xq, h->W.Q.xq, sizeof(double) * h->D.n);
    memcpy(lam_act, h->W.Q.lam_act, sizeof(double) * iq);
  }
  memcpy(h->W.E.g, gsave.data(), sizeof(double) * h->D.m);
  return iq;
}
int hs_qp_warm(void* hp, double* H, const double* q, double* du, double* lam, int* iters) { return hs_qp_common((HsHandle*)hp, H, q, du, lam, iters, 1); }
// qp_factor of H (n*n): returns ok; L (lower triangle, zero above), Y = L^-1 (all n x n entries as stored), xq = -H^-1 q
int hs_factor(void* hp, const double* H, const double* q, double* L, double* Y, double* xq) {
  HsHandle* h = (HsHandle*)hp; Cta c;
  const int n = h->D.n, ld = h->D.ld;
  for (int i = 0; i < n; ++i) memcpy(h->W.B.matA + (size_t)i * ld, H + (size_t)i * n, sizeof(double) * n);
  for (size_t t = 0; t < (size_t)n * ld; ++t) h->W.B.matB[t] = 3.0;    // the factorisation must write Y's zero upper triangle
  std::vector<double> qc(q, q + n);
  const bool ok = qp_factor<false>(c, h->D, qc.data(), h->W.Q, h->W.B);
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) {
      L[(size_t)i * n + j] = j <= i ? h->W.B.matA[(size_t)i * ld + j] : 0.0;
      Y[(size_t)i * n + j] = h->W.B.matB[(size_t)i * ld + j];
    }
  memcpy(xq, h->W.Q.xq, sizeof(double) * n);
  return ok;
}
int hs_lsqr(void* hp, const double* x0, const double* u, double* l_out) {
  HsHandle* h = (HsHandle*)hp; Cta c;
  SolveCtx X; X.G = &h->G; X.P = &h->P; X.D = h->D; X.W = h->W; X.x0 = x0; X.up_in = nullptr;
  for (int i = 0; i < h->D.nu; ++i) h->W.S.up[i] = 0.0;
  std::vector<double> l0(h->D.m, 0.0);
  eval_grad<false>(c, X, u, l0.data(), true);
  return lsqr_dual_init<false>(c, h->D, h->W.E, h->W.L, h->W.E.q, l_out);
}
void hs_solve(void* hp, const double* x0, const double* u_ws, const double* l_ws, const double* u_prev, double* u, double* l, double* x, double* cost, double* cond,
              int* num_iters, int* status, int* qp_solves, int* diag, double* l_init) {
  HsHandle* h = (HsHandle*)hp; Cta c;
  SolveCtx X; X.G = &h->G; X.P = &h->P; X.D = h->D; X.W = h->W; X.x0 = x0; X.up_in = u_prev;
  SolveOut O; O.u = u; O.l = l; O.x = x; O.cost = cost; O.cond = cond; O.num_iters = num_iters; O.status = status;
  O.qp_solves = qp_solves; O.diag = diag; O.l_init = l_init; O.iter_log = nullptr; O.iter_cap = 0;
  if (h->P.policy == 2) sqp_solve_v2<false>(c, X, u_ws, l_ws, O);
  else sqp_solve_v1<false>(c, X, u_ws, l_ws, O);
}
}
