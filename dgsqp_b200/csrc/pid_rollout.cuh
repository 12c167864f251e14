// Warm-start generation for the racing games on device (SURVEY 8(f-1)): the PID lane-follower roll-out the reference's
// Monte-Carlo drivers run per sampled agent before every solve
//   scripts/DGSQP_ALGAMES_monte_carlo_chicane.py:411-467, scripts/DGSQP_monte_carlo_agents.py:262-308
//   controllers  DGSQP/solvers/PID.py:74-138 (PID), :187-238 (PIDLaneFollower: steer on 5 (x_tran - ref) + e_psi, speed on v)
//   simulation   CasadiDynamicsModel.step, DGSQP/dynamics/dynamics_models.py:161-186 (one dt of the continuous bicycle
//                :1046-1070, then local_to_global, DGSQP/tracks/radius_arclength_track.py:752-807)
// One thread rolls out one agent: N steps of (PID -> RK4 with 4 sub-steps -> local_to_global), everything in registers.
// Arithmetic follows dgsqp_b200/montecarlo.py: pid_rollout statement by statement (that host version documents the one
// deliberate difference to the reference: classical RK4 instead of SciPy's adaptive RK45).
#pragma once
#include <math.h>

#define RO_MAX_KP 9          // DGSQP_MAX_TRACK_SEGS + 1 key points

struct RolloutParams {
  int N, nkp;                // horizon, number of key points (segments + 1)
  double dt, L_f, L_r, c_da, c_dr, c_s, mass;
  double u_ub[2], u_lb[2], rate_ub[2], rate_lb[2];
  double kp[RO_MAX_KP][6];   // key points: x, y, psi, cumulative s, segment length, curvature (tracks.py: key_pts)
  double L;                  // track length
};

DG_HD double ro_wrap(double th) {
  const double pi = 3.141592653589793;
  return th < -pi ? th + 2 * pi : (th > pi ? th - 2 * pi : th);
}

// montecarlo._track_lookup: curvature (pw_const) and tangent angle (pw_lin) at arclength s
DG_HD void ro_track_lookup(const RolloutParams& P, double s, double& kap, double& psit) {
  const double sb = fmod(fmod(s, P.L) + P.L, P.L);
  int idx = 0;
  double cum = 0.0, cum_idx = 0.0;
  for (int j = 1; j + 1 < P.nkp; ++j) {          // searchsorted(kp[1:-1, 3], sb, side="right")
    cum += P.kp[j][4] * P.kp[j][5];
    if (P.kp[j][3] <= sb) { idx = j; cum_idx = cum; }
  }
  if (idx > P.nkp - 2) idx = P.nkp - 2;
  kap = P.kp[idx + 1][5];
  psit = cum_idx + kap * (sb - P.kp[idx][3]);
}

// tracks.RadiusArclengthTrack.local_to_global: (s, e_y) -> (x, y)
DG_HD void ro_local_to_global(const RolloutParams& P, double s, double ey, double& x, double& y) {
  const double pi = 3.141592653589793;
  if (s < 0) s = s + P.L * ceil(-s / P.L);
  if (s >= P.L) s = s - P.L * floor(s / P.L);
  int is = 0;
  for (int j = 0; j < P.nkp; ++j) if (P.kp[j][3] <= s) is = j;      // searchsorted(kp[:, 3], s, "right") - 1
  if (is > P.nkp - 2) is = P.nkp - 2;
  const double* a = P.kp[is];
  const double* b = P.kp[is + 1];
  const double d = s - a[3], curv = b[5];
  if (curv == 0.0) {
    x = a[0] + (b[0] - a[0]) * d / b[4] + ey * cos(b[2] + pi / 2);
    y = a[1] + (b[1] - a[1]) * d / b[4] + ey * sin(b[2] + pi / 2);
    return;
  }
  const double r = 1.0 / curv, sgn = r >= 0 ? 1.0 : -1.0, ra = fabs(r);
  const double xc = a[0] + ra * cos(a[2] + sgn * pi / 2), yc = a[1] + ra * sin(a[2] + sgn * pi / 2);
  const double span = d / ra;
  const double ang_n = ro_wrap(a[2] + sgn * pi / 2);
  const double ang = -(ang_n >= 0 ? 1.0 : -1.0) * (pi - fabs(ang_n));
  x = xc + (ra - sgn * ey) * cos(ang + sgn * span);
  y = yc + (ra - sgn * ey) * sin(ang + sgn * span);
}

// montecarlo._fc: continuous kinematic bicycle (dynamics_models.py:1046-1070)
DG_HD void ro_fc(const RolloutParams& P, const double* q, double ua, double delta, double* f) {
  const double v = q[2], epsi = q[3], s = q[4], ey = q[5];
  const double beta = atan2(tan(delta) * P.L_r, P.L_f + P.L_r);
  const double psidot = v / P.L_r * sin(beta);
  const double F = -P.c_da * v - P.c_dr * v * fabs(v) - P.c_s * (psidot * psidot);
  double kap, psit;
  ro_track_lookup(P, s, kap, psit);
  const double den = 1.0 - ey * kap, cb = cos(beta + epsi);
  f[0] = v * cos(beta + psit + epsi);
  f[1] = v * sin(beta + psit + epsi);
  f[2] = ua + F / P.mass;
  f[3] = psidot - kap * v * cb / den;
  f[4] = v * cb / den;
  f[5] = v * sin(beta + epsi);
}

struct RoPid { double Kp, Ki, x_ref, u_max, u_min, du_max, du_min, ei, u_prev; };

DG_HD double ro_pid(RoPid& c, double x, double dt) {
  const double e = x - c.x_ref;
  double ei = c.ei + e * dt;
  ei = ei < -100.0 ? -100.0 : (ei > 100.0 ? 100.0 : ei);
  c.ei = ei;
  double u = -(c.Kp * e + c.Ki * ei);
  double du = u - c.u_prev;
  du = du < c.du_min ? c.du_min : (du > c.du_max ? c.du_max : du);
  u = du + c.u_prev;
  u = u < c.u_min ? c.u_min : (u > c.u_max ? c.u_max : u);
  c.u_prev = u;
  return u;
}

// one agent in flight: state, lane and speed references, and the memory of the two controllers ([0] speed, [1] steer);
// the controller constants are re-read from P at every stage so that they need not stay in registers
struct RoAgent { double q[6]; double xt0, v0, ei[2], u_prev[2]; };

DG_HD void ro_start(const RolloutParams& P, double s0, double xt0, double v0, RoAgent& a) {
  ro_local_to_global(P, s0, xt0, a.q[0], a.q[1]);
  a.q[2] = v0; a.q[3] = 0.0; a.q[4] = s0; a.q[5] = xt0;
  a.xt0 = xt0; a.v0 = v0;
  a.ei[0] = a.ei[1] = a.u_prev[0] = a.u_prev[1] = 0.0;
}

// one stage: PID inputs (ua, us), RK4 with 4 sub-steps, then the global position from (s, e_y)
DG_HD void ro_step(const RolloutParams& P, RoAgent& a, double& ua, double& us) {
  double* q = a.q;
  RoPid speed = {1.0, 0.0, a.v0, P.u_ub[0], P.u_lb[0], P.rate_ub[0], P.rate_lb[0], a.ei[0], a.u_prev[0]};
  RoPid steer = {1.0, 0.005, 0.0, P.u_ub[1], P.u_lb[1], P.rate_ub[1], P.rate_lb[1], a.ei[1], a.u_prev[1]};
  ua = ro_pid(speed, q[2], P.dt);
  us = ro_pid(steer, 5.0 * (q[5] - a.xt0) + q[3], P.dt);
  a.ei[0] = speed.ei; a.u_prev[0] = speed.u_prev;
  a.ei[1] = steer.ei; a.u_prev[1] = steer.u_prev;
  const double h = P.dt / 4;
  for (int sub = 0; sub < 4; ++sub) {
    double k1[6], k2[6], k3[6], k4[6], t[6];
    ro_fc(P, q, ua, us, k1);
    for (int i = 0; i < 6; ++i) t[i] = q[i] + 0.5 * h * k1[i];
    ro_fc(P, t, ua, us, k2);
    for (int i = 0; i < 6; ++i) t[i] = q[i] + 0.5 * h * k2[i];
    ro_fc(P, t, ua, us, k3);
    for (int i = 0; i < 6; ++i) t[i] = q[i] + h * k3[i];
    ro_fc(P, t, ua, us, k4);
    for (int i = 0; i < 6; ++i) q[i] = q[i] + h / 6.0 * (k1[i] + 2 * k2[i] + 2 * k3[i] + k4[i]);
  }
  ro_local_to_global(P, q[4], q[5], q[0], q[1]);
}

// one agent: q0[6], xy[(N+1)*2] (may be NULL), u_ws[N*2]
DG_HD void ro_agent(const RolloutParams& P, double s0, double xt0, double v0, double* q0, double* xy, double* u_ws) {
  RoAgent a;
  ro_start(P, s0, xt0, v0, a);
  for (int i = 0; i < 6; ++i) q0[i] = a.q[i];
  if (xy) { xy[0] = a.q[0]; xy[1] = a.q[1]; }
  for (int k = 0; k < P.N; ++k) {
    double ua, us;
    ro_step(P, a, ua, us);
    if (xy) { xy[2 * (k + 1)] = a.q[0]; xy[2 * (k + 1) + 1] = a.q[1]; }
    u_ws[2 * k] = ua; u_ws[2 * k + 1] = us;
  }
}

// host-side fill from the C-ABI game record and the key-point table of the track
static inline int ro_fill(const dgsqp_racing_game* g, const double* key_pts, RolloutParams* P) {
  if (!g || !key_pts || g->N < 1 || g->track_nseg < 1 || g->track_nseg + 1 > RO_MAX_KP) return -1;
  P->N = g->N; P->nkp = g->track_nseg + 1;
  P->dt = g->dt; P->L_f = g->L_f; P->L_r = g->L_r; P->c_da = g->c_da; P->c_dr = g->c_dr; P->c_s = g->c_s; P->mass = g->mass;
  for (int i = 0; i < 2; ++i) { P->u_ub[i] = g->u_ub[i]; P->u_lb[i] = g->u_lb[i]; P->rate_ub[i] = g->rate_ub[i]; P->rate_lb[i] = g->rate_lb[i]; }
  for (int j = 0; j < P->nkp; ++j) for (int i = 0; i < 6; ++i) P->kp[j][i] = key_pts[j * 6 + i];
  P->L = P->kp[P->nkp - 1][3];
  return 0;
}
