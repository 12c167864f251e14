// Highway-merge dynamic game on device: rollout, derivatives, the lane rows and the costs; the constraint layout and the
// condensed game-KKT data are shared with the racing games (game_layout.cuh, game_kkt.cuh).
//
// Replaces, for the merge scenario of the reference (scripts/DGSQP_merge_monte_carlo.py: three kinematic unicycles under
// RK3, quadratic goal-tracking costs :253-304, lane half-planes with pw_const-switched ramp normals :40-74,316-318,
// pairwise collision rows :306-314, bounds on v / F_x / w_z :130-161), the CasADi functions evaluated by
// DGSQP._evaluate (DGSQP/solvers/DGSQP.py:509-533):
//   evaluate_dynamics (:598-601), evaluate_jacobian_A/B (:607-612), evaluate_hessian_E/F/G (:621-628),
//   f_Du_x (:642-650), f_Cxu (:804-821), f_Du_C (:824-826), f_q (:673-676,898-899), f_Q (:679-727,829-934).
// Differences to the racing games: 4 states per agent (x, y, v, psi), the state cost is present at every stage (costates
// and value-function Hessians of the cost functions pick up a term per stage), no input-rate terms, and the state rows
// the constraints read are (x, y, v): lane rows n(x)'(p - c) at every stage, v bounds for k >= 1.
#pragma once
#include "cta.cuh"
#include "model_unicycle_gen.cuh"

#define DG_MAX_AGENTS 4
#define DG_NQA 4
#define DG_NUA 2
#define DG_MAX_NQ (DG_NQA * DG_MAX_AGENTS)
#define DG_MAX_PAIRS 6
// per-(stage, agent) sizes of the packed second derivatives of the outputs x, y (2 x 10) and their costate
// contraction (10)
#define DG_T2_SZ 20
#define DG_HC_SZ 10
// constraint rows per (stage, agent): 2 lane rows at every stage, bounds on v
#define DG_GAME_ROWS 2
#define DG_GAME_ROWS_N 2
#define DG_BOUND_STATE 2

// lane row  n(x)'(p - (pt - r n(x))) <= 0,  n(x) = na for x < brk, nb otherwise (CasADi pw_const, merge.py:66-74)
struct LaneRow { double brk, na[2], nb[2], pt[2]; };

struct GameDesc {
  int M, N;
  UnicycleParams veh;
  double w_u[2], w_q[4], term_scale;
  double goal[DG_MAX_AGENTS][4];
  double u_ub[2], u_lb[2], v_ub, v_lb;
  double obs_r[DG_MAX_AGENTS];
  double lane_r;
  LaneRow lane[DG_MAX_AGENTS][2];
};

#include "game_layout.cuh"

struct EvalBuf : EvalTables {
  const GameDesc* G;   // lane normals are needed by the matrix-free G products (set by game_bind)
};

// attaches the game record to the workspace table (after plan_memory)
DG_HD void game_bind(EvalBuf& E, const GameDesc* G) { E.G = G; }

// active lane normal at longitudinal position px (pw_const: zero derivative)
DG_DEV void lane_normal(const LaneRow& L, double px, double& n0, double& n1) {
  const bool hi = px >= L.brk;
  n0 = hi ? L.nb[0] : L.na[0];
  n1 = hi ? L.nb[1] : L.na[1];
}

// x_{k+1} = rk3(x_k, u_k)  (dynamics_models.py:202-212,325-333).  v and psi are running sums of the inputs, so the
// serial chain over the horizon only carries additions: (1) thread per agent: v_k, psi_k; (2) thread per (k, agent):
// the RK3 position increments (six sin/cos each) in parallel; (3) thread per agent: x_k, y_k.  Identical arithmetic to a
// stage-by-stage rollout.
template <bool SM>
DG_DEVN void game_rollout(Cta& c, const GameDesc& G, const Dims& D_, const double* u, const double* x0, double* x,
                          double* pre) {
  const Dims D = D_;
  DG_ASSUME_SHARED(x); DG_ASSUME_SHARED(pre);
  const UnicycleParams P = G.veh;
  DG_FOR(a, D.M) {
    double v = x0[a * DG_NQA + 2], psi = x0[a * DG_NQA + 3];
    for (int i = 0; i < DG_NQA; ++i) x[a * DG_NQA + i] = x0[a * DG_NQA + i];
    for (int k = 0; k < D.N; ++k) {
      v += u[uidx(D, a, k, 0)] * P.dt * P.inv_m;
      psi += P.dt * u[uidx(D, a, k, 1)];
      x[(k + 1) * D.nq + a * DG_NQA + 2] = v;
      x[(k + 1) * D.nq + a * DG_NQA + 3] = psi;
    }
  }
  c.sync();
  DG_FOR(t, D.N * D.M) {
    const int k = t / D.M, a = t - k * D.M;
    double inc[DG_NQA];
    unicycle_fd_raw(x + k * D.nq + a * DG_NQA, u + uidx(D, a, k, 0), P, inc);
    pre[t * 2] = inc[0]; pre[t * 2 + 1] = inc[1];
  }
  c.sync();
  DG_FOR(a, D.M) {
    double px = x0[a * DG_NQA], py = x0[a * DG_NQA + 1];
    for (int k = 0; k < D.N; ++k) {
      px += pre[(k * D.M + a) * 2]; py += pre[(k * D.M + a) * 2 + 1];
      x[(k + 1) * D.nq + a * DG_NQA] = px;
      x[(k + 1) * D.nq + a * DG_NQA + 1] = py;
    }
  }
}

template <bool SM>
DG_DEVN void game_linearize(Cta& c, const GameDesc& G, const Dims& D_, const double* u, const EvalBuf& E_, bool second) {
  const EvalBuf E = E_; DG_SH_EVAL(E); const Dims D = D_;
  DG_FOR(t, D.N * D.M) {
    int k = t / D.M, a = t - k * D.M;
    const double* qk = E.x + k * D.nq + a * DG_NQA;
    unicycle_jac(qk, u + uidx(D, a, k, 0), G.veh, E.AB + t * DG_AB_SZ);
    if (second) unicycle_hess(qk, u + uidx(D, a, k, 0), G.veh, E.T2 + t * DG_T2_SZ);
  }
}
// ---- hooks of game_kkt.cuh: lane rows, v bounds ----
// Lane row (k, a, b):  n(x)'(p - (pt - r n(x))) <= 0  for lane b of agent a, n(x) the active normal of lane_normal.  It is
// linear in the position p = (x, y), so its G row is n0 S_x + n1 S_y; RowCoef holds n of the row.
struct RowCoef { double n0, n1; };

DG_DEV double game_state_ub(const GameDesc& G) { return G.v_ub; }
DG_DEV double game_state_lb(const GameDesc& G) { return G.v_lb; }

DG_DEV double game_row_value(const GameDesc& G, const Dims& D, const double*, const double*, const double* x, int k,
                             int a, int b) {
  const LaneRow& L = G.lane[a][b];
  const double px = x[k * D.nq + a * DG_NQA], py = x[k * D.nq + a * DG_NQA + 1];
  double n0, n1;
  lane_normal(L, px, n0, n1);
  return n0 * (px - (L.pt[0] - G.lane_r * n0)) + n1 * (py - (L.pt[1] - G.lane_r * n1));
}

DG_DEV double game_row_Gv(const Dims& D, const EvalBuf& E, const double*, int k, int a, int b) {
  double val = 0.0;
  if (k >= 1) {
    double n0, n1;
    lane_normal(E.G->lane[a][b], E.x[k * D.nq + a * DG_NQA], n0, n1);
    const double* ta = E.tmpS + (a * D.N + (k - 1)) * 3;
    val = n0 * ta[0] + n1 * ta[1];
  }
  return val;
}

DG_DEV void game_row_prep(const Dims& D, const EvalBuf& E, int k, int kind, int a, int b, RowCoef& rc) {
  rc.n0 = 0.0; rc.n1 = 0.0;
  if (kind == K_GAME) lane_normal(E.G->lane[a][b], E.x[k * D.nq + a * DG_NQA], rc.n0, rc.n1);
}

DG_DEV void game_row_G(const Dims& D, const EvalBuf& E, const RowCoef& rc, int k, int a, int, int ta, int j, int kj, int,
                       double& val) {
  if (ta == a && kj < k) {
    const double* Sk = E.S + sens_off(D, ta, k, 0) + j;
    val = rc.n0 * Sk[0] + rc.n1 * Sk[2 * k];
  }
}

// the lane rows read the sensitivities: no sparse row
DG_DEV bool game_row_sparse(const Dims&, int, int, int, int&, int&) { return false; }

DG_DEV void game_row_coefs(const Dims& D, const EvalBuf& E, const double* w, int k, int a, double& cx, double& cy) {
  for (int j = 0; j < 2; ++j) {
    double n0, n1;
    lane_normal(E.G->lane[a][j], E.x[k * D.nq + a * DG_NQA], n0, n1);
    const double wl = w[row_game(D, k, a, j)];
    cx += wl * n0; cy += wl * n1;
  }
}

DG_DEV void game_row_lx(const GameDesc& G, const Dims& D, const double* x, const double* l, int k, int a, int comp,
                        double& v) {
  for (int j = 0; j < 2; ++j) {
    double n0, n1;
    lane_normal(G.lane[a][j], x[k * D.nq + a * DG_NQA], n0, n1);
    v += l[row_game(D, k, a, j)] * (comp == 0 ? n0 : n1);
  }
}

// the lane rows do not read the inputs: only the input-bound rows iub / ilb
DG_DEV double game_row_GT_direct(const Dims&, const double* w, int, int, int, int iub, int ilb) { return w[iub] - w[ilb]; }

// ---- hooks of game_kkt.cuh: costs ----
// stage / terminal state cost of agent f: (k == N ? term_scale : 1) * 1/2 (q^f - goal^f)' diag(w_q) (q^f - goal^f)
DG_DEV double cost_lx(const GameDesc& G, const Dims& D, const double* x, int f, int k, int idx) {
  int blk = idx / DG_NQA, comp = idx - blk * DG_NQA;
  if (blk != f) return 0.0;
  double v = G.w_q[comp] * (x[k * D.nq + idx] - G.goal[f][comp]);
  return k == D.N ? G.term_scale * v : v;
}
DG_DEV double cost_lxx(const GameDesc& G, const Dims& D, int f, int k, int i1, int i2) {
  if (i1 != i2) return 0.0;
  int blk = i1 / DG_NQA, comp = i1 - blk * DG_NQA;
  if (blk != f) return 0.0;
  return k == D.N ? G.term_scale * G.w_q[comp] : G.w_q[comp];
}
DG_DEV double game_term_lx(const GameDesc& G, const Dims& D, const double* x, int f, int idx) { return cost_lx(G, D, x, f, D.N, idx); }
DG_DEV double game_stage_lx(const GameDesc& G, const Dims& D, const double* x, int f, int k, int idx) { return cost_lx(G, D, x, f, k, idx); }
DG_DEV double game_term_lxx(const GameDesc& G, const Dims& D, const double*, int f, int i1, int i2) { return cost_lxx(G, D, f, D.N, i1, i2); }
DG_DEV double game_stage_lxx(const GameDesc& G, const Dims& D, int f, int k, int i1, int i2) { return cost_lxx(G, D, f, k, i1, i2); }

// input cost 1/2 w_u u^2 (t = uidx(a, k, cc)): gradient w_u u, second derivative w_u; no coupling between stages.
// The gradient is read at each sum of game_gradients, so that w_u u + s stays one fused multiply-add per sum.
struct InputGrad { const double* w; const double* u; };
DG_DEV InputGrad game_input_grad(const GameDesc& G, const Dims&, const double* u, const double*, int t, int, int, int cc) {
  return {&G.w_u[cc], &u[t]};
}
DG_DEV double input_grad_plus(const InputGrad& g, double s) { return *g.w * *g.u + s; }
DG_DEV double game_input_hess(const GameDesc& G, const Dims&, int, int cc) { return G.w_u[cc]; }
DG_DEV void game_input_hess_prev(const GameDesc&, int, double&, double&) {}

// Hc entry e: only the outputs x, y have second derivatives
DG_DEV double game_contract_entry(const double* p, const double* T, int e) { return p[0] * T[e] + p[1] * T[DG_HC_SZ + e]; }

DG_DEV int tri4(int r, int cc) { return r * 4 - (r * (r - 1)) / 2 + (cc - r); }

// second-derivative contraction entries:  state indices 2..3 (v, psi) <-> act 0..1, inputs (F, w) <-> act 2..3
DG_DEV double hc_xx(const double* hc, int i, int j) {
  if (i < 2 || j < 2) return 0.0;
  int r = i - 2, cc = j - 2;
  return r <= cc ? hc[tri4(r, cc)] : hc[tri4(cc, r)];
}
DG_DEV double hc_ux(const double* hc, int cu, int j) { return j >= 2 ? hc[tri4(j - 2, 2 + cu)] : 0.0; }
DG_DEV double hc_uu(const double* hc, int c1, int c2) { return c1 <= c2 ? hc[tri4(2 + c1, 2 + c2)] : hc[tri4(2 + c2, 2 + c1)]; }

#include "game_kkt.cuh"

// f_J at the solution (DGSQP.py:476-498, 889-893): thread per agent
template <bool SM>
DG_DEVN void game_costs(Cta& c, const GameDesc& G, const Dims& D_, const double* u, const double* up, const double* x,
                        double* cost) {
  const Dims D = D_;
  DG_FOR(a, D.M) {
    double J = 0.0;
    for (int k = 0; k <= D.N; ++k) {
      double sc = 0.0;
      for (int i = 0; i < DG_NQA; ++i) { double d = x[k * D.nq + a * DG_NQA + i] - G.goal[a][i]; sc += G.w_q[i] * d * d; }
      J += (k == D.N ? G.term_scale : 1.0) * 0.5 * sc;
      if (k < D.N)
        for (int cc = 0; cc < 2; ++cc) { double uk = u[uidx(D, a, k, cc)]; J += 0.5 * G.w_u[cc] * uk * uk; }
    }
    cost[a] = J;
  }
}
