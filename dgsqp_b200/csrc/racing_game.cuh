// Racing dynamic game on device: rollout, derivatives, the input-rate rows and the costs; the constraint layout and the
// condensed game-KKT data are shared with the merge game (game_layout.cuh, game_kkt.cuh).
//
// Replaces, for the racing games of the reference (scripts/DGSQP_ALGAMES_monte_carlo_chicane.py,
// ..._curve.py, DGSQP_monte_carlo_agents.py), the CasADi functions evaluated by
// DGSQP._evaluate (DGSQP/solvers/DGSQP.py:509-533):
//   evaluate_dynamics (:598-601), evaluate_jacobian_A/B (:607-612), evaluate_hessian_E/F/G (:621-628),
//   f_Du_x (:642-650), f_Cxu (:804-821), f_Du_C (:824-826), f_q (:673-676,898-899), f_Q (:679-727,829-934).
// The state cost is terminal only (progress and competition on s), the inputs carry w_u and input-rate costs w_du, and
// the constraints read the states x, y, e_y: track bounds on e_y at k >= 1, input-rate rows at k < N.
#pragma once
#include "cta.cuh"
#include "model_bicycle_gen.cuh"

#define DG_MAX_AGENTS 4
#define DG_MAX_SEGS 8
#define DG_NQA 6
#define DG_NUA 2
#define DG_MAX_NQ (DG_NQA * DG_MAX_AGENTS)
#define DG_MAX_PAIRS 6
// per-(stage, agent) sizes of the packed second derivatives (6 x 15) and their costate contraction (15)
#define DG_T2_SZ 90
#define DG_HC_SZ 15
// constraint rows per (stage, agent): 4 input-rate rows at k < N, track bounds on e_y
#define DG_GAME_ROWS 4
#define DG_GAME_ROWS_N 0
#define DG_BOUND_STATE 5

struct TrackTable {
  int nseg;
  double L;
  double brk[DG_MAX_SEGS];        // nseg-1 interior breakpoints
  double curv[DG_MAX_SEGS];       // curvature per segment
  double cum_len[DG_MAX_SEGS + 1];
  double cum_ang[DG_MAX_SEGS + 1];
  double slope[DG_MAX_SEGS];      // tangent-angle slope per segment
};

struct GameDesc {
  int M, N;
  BicycleParams veh;
  TrackTable trk;
  double w_u[2], w_du[2], c_prog, c_comp;
  double u_ub[2], u_lb[2];
  double rate_ub[2], rate_lb[2];   // per-second rates; constraint uses dt*rate
  double half_width;
  double obs_r[DG_MAX_AGENTS];
};

#include "game_layout.cuh"

struct EvalBuf : EvalTables {};

// attaches the game record to the workspace table (after plan_memory); the racing products need no game data
DG_HD void game_bind(EvalBuf&, const GameDesc*) {}

// ---- track look-ups (radius_arclength_track.py:199-225; CasADi pw_const / pw_lin / fmod) ----
DG_DEV void track_eval(const TrackTable& T, double s, double& kappa, double& psit, double& dpsit) {
  // sb = fmod(fmod(s, L) + L, L).  For 0 <= s < L both fmods are exact subtractions (fmod(s, L) = s and s + L lies in
  // [L, 2L]), so the fast path returns bit-for-bit the same value without the two slow fmod calls.
  double sb;
  if (s >= 0.0 && s < T.L) { const double t = s + T.L; sb = t >= 2.0 * T.L ? t - 2.0 * T.L : t - T.L; }
  else sb = fmod(fmod(s, T.L) + T.L, T.L);
  double kap = T.curv[0];
  double l_prev = T.cum_ang[0] + T.slope[0] * (sb - T.cum_len[0]);
  double ps = l_prev, dp = T.slope[0];
  for (int i = 0; i + 1 < T.nseg; ++i) {
    double ind = sb >= T.brk[i] ? 1.0 : 0.0;
    kap += (T.curv[i + 1] - T.curv[i]) * ind;
    double l_next = T.cum_ang[i + 1] + T.slope[i + 1] * (sb - T.cum_len[i + 1]);
    ps += (l_next - l_prev) * ind;
    dp += (T.slope[i + 1] - T.slope[i]) * ind;
    l_prev = l_next;
  }
  kappa = kap; psit = ps; dpsit = dp;
}

// x_{k+1} = x_k + dt f(x_k,u_k)  (explicit Euler of the Frenet bicycle, dynamics_models.py:1030-1070,90-91).
// Agents are dynamically decoupled and the stage recursion is serial, so only M threads can walk the horizon.  Everything
// that depends on the inputs alone is therefore hoisted into a CTA-wide pre-pass over the N*M stages
//   beta = atan(L_r tan(delta) / L),  c_rot = psidot / v = tan(delta) / (L sqrt(1 + (L_r tan(delta)/L)^2)),
//   c_slip = c_s (tan(delta)/L)^2 / (1 + (L_r tan(delta)/L)^2)
// (pre[(k*M + a)*3 ..]), which leaves two sincos and one division on the serial chain of a stage.
template <bool SM>
DG_DEVN void game_rollout(Cta& c, const GameDesc& G, const Dims& D_, const double* u, const double* x0, double* x,
                          double* pre) {
  // local copies: the tables live in shared memory and would otherwise be re-read after every store
  const Dims D = D_;
  DG_ASSUME_SHARED(x); DG_ASSUME_SHARED(pre);
  const BicycleParams P = G.veh;
  DG_FOR(t, D.N * D.M) {
    const int k = t / D.M, a = t - k * D.M;
    const double t0 = tan(u[uidx(D, a, k, 1)]);
    const double t1 = t0 / P.L;
    const double t5 = t1 * t1;
    const double t6 = (P.Lr * P.Lr) * t5 + 1.0;
    pre[t * 3] = atan(P.Lr * t1);
    pre[t * 3 + 1] = t1 / sqrt(t6);
    pre[t * 3 + 2] = P.c_s * t5 / t6;
  }
  c.sync();
  DG_FOR(a, D.M) {
    double qk[DG_NQA];
    for (int i = 0; i < DG_NQA; ++i) { qk[i] = x0[a * DG_NQA + i]; x[a * DG_NQA + i] = qk[i]; }
    for (int k = 0; k < D.N; ++k) {
      double kap, ps, dp;
      track_eval(G.trk, qk[4], kap, ps, dp);
      const double* pk = pre + (k * D.M + a) * 3;
      const double v = qk[2], sgnv = v > 0 ? 1.0 : -1.0;
      const double t2 = qk[3] + pk[0], t4 = P.dt * v;
      double s2, c2, s3, c3;
      sincos(t2, &s2, &c2);
      sincos(ps + t2, &s3, &c3);
      const double t7 = c2 / (qk[5] * kap - 1.0);
      qk[0] += t4 * c3;
      qk[1] += t4 * s3;
      qk[2] += P.dt * (u[uidx(D, a, k, 0)] - P.inv_m * v * (P.c_da + P.c_dr * sgnv * v + pk[2] * v));
      qk[3] += t4 * (kap * t7 + pk[1]);
      qk[4] += -t4 * t7;
      qk[5] += t4 * s2;
      for (int i = 0; i < DG_NQA; ++i) x[(k + 1) * D.nq + a * DG_NQA + i] = qk[i];
    }
  }
}

template <bool SM>
DG_DEVN void game_linearize(Cta& c, const GameDesc& G, const Dims& D_, const double* u, const EvalBuf& E_, bool second) {
  // local copies: the tables live in shared memory and would otherwise be re-read after every store
  const EvalBuf E = E_; DG_SH_EVAL(E); const Dims D = D_;
  DG_FOR(t, D.N * D.M) {
    int k = t / D.M, a = t - k * D.M;
    const double* qk = E.x + k * D.nq + a * DG_NQA;
    double kap, ps, dp;
    track_eval(G.trk, qk[4], kap, ps, dp);
    double sg = qk[2] > 0 ? 1.0 : -1.0;
    bicycle_jac(qk, u + uidx(D, a, k, 0), G.veh, kap, ps, dp, sg, E.AB + t * DG_AB_SZ);
    if (second) bicycle_hess(qk, u + uidx(D, a, k, 0), G.veh, kap, ps, dp, sg, E.T2 + t * DG_T2_SZ);
  }
}

// ---- hooks of game_kkt.cuh: input-rate rows, track bounds ----
// Rate row (k, a, b), b = 2 cc + (0: upper, 1: lower):  du - dt rate_ub[cc] <= 0  or  dt rate_lb[cc] - du <= 0  with
// du = u^a_k[cc] - u^a_{k-1}[cc]  (u^a_{-1} = up, the previous input).  Its G row has the entries +-1 at u_k, u_{k-1}.
struct RowCoef {};

DG_DEV double game_state_ub(const GameDesc& G) { return G.half_width; }
DG_DEV double game_state_lb(const GameDesc& G) { return -G.half_width; }

DG_DEV double game_row_value(const GameDesc& G, const Dims& D, const double* u, const double* up, const double*, int k,
                             int a, int b) {
  int cc = b >> 1;
  double uk = u[uidx(D, a, k, cc)];
  double um = k == 0 ? up[a * DG_NUA + cc] : u[uidx(D, a, k - 1, cc)];
  double du = uk - um;
  return (b & 1) == 0 ? du - G.veh.dt * G.rate_ub[cc] : G.veh.dt * G.rate_lb[cc] - du;
}

DG_DEV double game_row_Gv(const Dims& D, const EvalBuf&, const double* v, int k, int a, int b) {
  int cc = b >> 1;
  double dv = v[uidx(D, a, k, cc)] - (k > 0 ? v[uidx(D, a, k - 1, cc)] : 0.0);
  return (b & 1) == 0 ? dv : -dv;
}

DG_DEV void game_row_prep(const Dims&, const EvalBuf&, int, int, int, int, RowCoef&) {}

DG_DEV void game_row_G(const Dims&, const EvalBuf&, const RowCoef&, int k, int a, int b, int ta, int, int kj, int cc,
                       double& val) {
  if (ta == a && cc == (b >> 1)) {
    double sg = (b & 1) == 0 ? 1.0 : -1.0;
    if (kj == k) val = sg;
    else if (kj == k - 1) val = -sg;
  }
}

DG_DEV bool game_row_sparse(const Dims& D, int k, int a, int b, int& t1, int& t2) {
  const int neg = (b & 1) == 0 ? 0 : 1;
  t1 = (uidx(D, a, k, b >> 1) << 1) | neg;
  if (k >= 1) t2 = (uidx(D, a, k - 1, b >> 1) << 1) | (neg ^ 1);
  return true;
}

// the rate rows read no state
DG_DEV void game_row_coefs(const Dims&, const EvalBuf&, const double*, int, int, double&, double&) {}
DG_DEV void game_row_lx(const GameDesc&, const Dims&, const double*, const double*, int, int, int, double&) {}

// (G' w)[u^a_k[cc]] of the rate rows of stages k and k+1, then of the input-bound rows iub / ilb
DG_DEV double game_row_GT_direct(const Dims& D, const double* w, int a, int k, int cc, int iub, int ilb) {
  double v = w[row_game(D, k, a, 2 * cc)] - w[row_game(D, k, a, 2 * cc + 1)];
  if (k + 1 < D.N) v -= w[row_game(D, k + 1, a, 2 * cc)] - w[row_game(D, k + 1, a, 2 * cc + 1)];
  v += w[iub] - w[ilb];
  return v;
}

// ---- hooks of game_kkt.cuh: costs ----
// terminal-cost gradient entries of agent f wrt joint x_N:  -c_prog*s_f + sum_b c_comp*atan(s_b - s_f)
DG_DEV double game_term_lx(const GameDesc& G, const Dims& D, const double* x, int f, int idx) {
  const double* xN = x + D.N * D.nq;
  int blk = idx / DG_NQA, comp = idx - blk * DG_NQA;
  if (comp != 4) return 0.0;
  double sf = xN[f * DG_NQA + 4];
  if (blk == f) {
    double v = -G.c_prog;
    for (int b = 0; b < D.M; ++b) if (b != f) { double dd = xN[b * DG_NQA + 4] - sf; v -= G.c_comp / (1.0 + dd * dd); }
    return v;
  }
  double dd = xN[blk * DG_NQA + 4] - sf;
  return G.c_comp / (1.0 + dd * dd);
}

DG_DEV double game_term_lxx(const GameDesc& G, const Dims& D, const double* x, int f, int i1, int i2) {
  const double* xN = x + D.N * D.nq;
  int b1 = i1 / DG_NQA, c1 = i1 - b1 * DG_NQA, b2 = i2 / DG_NQA, c2 = i2 - b2 * DG_NQA;
  if (c1 != 4 || c2 != 4) return 0.0;
  double sf = xN[f * DG_NQA + 4];
  double v = 0.0;
  for (int b = 0; b < D.M; ++b) {
    if (b == f) continue;
    double dd = xN[b * DG_NQA + 4] - sf;
    double d2 = -2.0 * G.c_comp * dd / ((1.0 + dd * dd) * (1.0 + dd * dd));
    // contributes +d2 at (b,b),(f,f), -d2 at (f,b),(b,f)
    if (b1 == b && b2 == b) v += d2;
    if (b1 == f && b2 == f) v += d2;
    if ((b1 == f && b2 == b) || (b1 == b && b2 == f)) v -= d2;
  }
  return v;
}

// no state cost before the terminal stage
DG_DEV double game_stage_lx(const GameDesc&, const Dims&, const double*, int, int, int) { return 0.0; }
DG_DEV double game_stage_lxx(const GameDesc&, const Dims&, int, int, int, int) { return 0.0; }

// d/du^a_k[cc] of the input costs 1/2 w_u u_k^2 + 1/2 w_du (u_k - u_{k-1})^2 of agent a (t = uidx(a, k, cc)), evaluated
// once and added to each sum of game_gradients
struct InputGrad { double v; };
DG_DEV InputGrad game_input_grad(const GameDesc& G, const Dims& D, const double* u, const double* up, int t, int a, int k,
                                 int cc) {
  double uk = u[t];
  double um = k == 0 ? up[a * DG_NUA + cc] : u[t - 2];
  double val = G.w_u[cc] * uk + G.w_du[cc] * (uk - um);
  if (k + 1 < D.N) val -= G.w_du[cc] * (u[t + 2] - uk);
  return {val};
}
DG_DEV double input_grad_plus(const InputGrad& g, double s) { return g.v + s; }

// their second derivatives: d2/du_k[cc]^2, and -w_du between u_k and u_{k-1} (added to v0 / v1 for cr = 0 / 1)
DG_DEV double game_input_hess(const GameDesc& G, const Dims& D, int k, int cc) {
  return G.w_u[cc] + G.w_du[cc] + (k + 1 < D.N ? G.w_du[cc] : 0.0);
}
DG_DEV void game_input_hess_prev(const GameDesc& G, int cr, double& v0, double& v1) {
  if (cr == 0) v0 -= G.w_du[0]; else v1 -= G.w_du[1];
}

// Hc entry e: sum over all six states of p_i * T2[i][e]
DG_DEV double game_contract_entry(const double* p, const double* T, int e) {
  double acc = 0.0;
  for (int i = 0; i < DG_NQA; ++i) acc += p[i] * T[i * DG_HC_SZ + e];
  return acc;
}

DG_DEV int tri5(int r, int cc) { return r * 5 - (r * (r - 1)) / 2 + (cc - r); }

// second-derivative contraction entries:  state indices 2..5 <-> act 0..3, delta <-> act 4
DG_DEV double hc_xx(const double* hc, int i, int j) {
  if (i < 2 || j < 2) return 0.0;
  int r = i - 2, cc = j - 2;
  return r <= cc ? hc[tri5(r, cc)] : hc[tri5(cc, r)];
}
DG_DEV double hc_ux(const double* hc, int cu, int j) { return (cu == 1 && j >= 2) ? hc[tri5(j - 2, 4)] : 0.0; }
DG_DEV double hc_uu(const double* hc, int c1, int c2) { return (c1 == 1 && c2 == 1) ? hc[14] : 0.0; }

#include "game_kkt.cuh"

// f_J at the solution (DGSQP.py:476-498, 889-893): thread per agent
template <bool SM>
DG_DEVN void game_costs(Cta& c, const GameDesc& G, const Dims& D_, const double* u, const double* up, const double* x,
                        double* cost) {
  const Dims D = D_;
  DG_FOR(a, D.M) {
    double J = 0.0;
    for (int k = 0; k < D.N; ++k)
      for (int cc = 0; cc < 2; ++cc) {
        double uk = u[uidx(D, a, k, cc)];
        double um = k == 0 ? up[a * 2 + cc] : u[uidx(D, a, k - 1, cc)];
        J += 0.5 * G.w_u[cc] * uk * uk + 0.5 * G.w_du[cc] * (uk - um) * (uk - um);
      }
    const double* xN = x + D.N * D.nq;
    J += -G.c_prog * xN[a * DG_NQA + 4];
    for (int b = 0; b < D.M; ++b) if (b != a) J += G.c_comp * atan(xN[b * DG_NQA + 4] - xN[a * DG_NQA + 4]);
    cost[a] = J;
  }
}
