// Monte-Carlo instance generation on the device (SURVEY 8(f-1)): NumPy's default generator, the per-trial transforms of
// dgsqp_b200/montecarlo.py and the accept / reject decision of every trial.
//
// Stream: numpy.random.PCG64 (the bit generator of np.random.default_rng) restated -- a 128-bit LCG stepped first, then the
// XSL-RR output of the new state; random() = (next64 >> 11) * 2^-53.  Any draw index is reached from the start state with
// at most 64 affine steps (the LCG-advance algorithm; the powers of the step map come from mc_jump_table on the host).
//
// Layout (trial-major): trial t consumes draws D*t .. D*t+D-1 in the order the scripts draw them within a trial, and output
// instance i is the i-th accepted trial.  So the instances do not depend on how many trials are decided per launch, and
// the first B/2 instances of a B-instance call are those of a B/2-instance call.
//   head-to-head   D = 5:  ego_s, ego_xt, ego_v, d, tar_v           (montecarlo.sample_head_to_head)
//   M agents       D = 3M: (s, x_tran, v) per agent                 (montecarlo.sample_agents, oracle/sampler.sample_agents)
//   merge          D = 12: the order of montecarlo.sample_merge, which this reproduces instance for instance
// The host samplers of the racing games draw batch-sized blocks per quantity instead, so for the same seed they return
// other (identically distributed) instances.
//
// The translation unit that includes this is compiled with -fmad=false: the transforms below are evaluated in NumPy's
// order without contraction.
#pragma once
#include <math.h>
#include <stdint.h>

#ifndef DG_HD
#ifdef __CUDACC__
#define DG_HD __host__ __device__ __forceinline__
#else
#define DG_HD static inline
#endif
#endif

#include "pid_rollout.cuh"

typedef unsigned __int128 mc_u128;

#define MC_PCG_MULT ((((mc_u128)0x2360ED051FC65DA4ULL) << 64) | (mc_u128)0x4385DF649FCCF645ULL)

struct McPcg { mc_u128 state, inc; };

DG_HD double mc_pcg_random(McPcg& g) {
  g.state = g.state * MC_PCG_MULT + g.inc;
  const uint64_t hi = (uint64_t)(g.state >> 64), lo = (uint64_t)g.state;
  const unsigned rot = (unsigned)(g.state >> 122);
  const uint64_t x = hi ^ lo;
  const uint64_t out = (x >> rot) | (x << ((64u - rot) & 63u));
  return (double)(out >> 11) * (1.0 / 9007199254740992.0);
}

// table[2i], table[2i+1] = (A, C) of 2^i steps: state -> A state + C
static inline void mc_jump_table(mc_u128 inc, mc_u128* table) {
  mc_u128 a = MC_PCG_MULT, c = inc;
  for (int i = 0; i < 64; ++i) {
    table[2 * i] = a; table[2 * i + 1] = c;
    c = (a + 1) * c;
    a = a * a;
  }
}

// the generator positioned so that its next random() is draw number d of the stream
DG_HD McPcg mc_pcg_at(const McPcg& g0, const mc_u128* table, uint64_t d) {
  McPcg g = g0;
  for (int i = 0; d; ++i, d >>= 1)
    if (d & 1) g.state = table[2 * i] * g.state + table[2 * i + 1];
  return g;
}

static inline McPcg mc_pcg_from(const dgsqp_pcg64* r) {
  McPcg g;
  g.state = ((mc_u128)r->state_hi << 64) | r->state_lo;
  g.inc = ((mc_u128)r->inc_hi << 64) | r->inc_lo;
  return g;
}

// ----------------------------------------------------------------------------------------------------- racing games
struct McRacing {
  RolloutParams P;
  int M, kind;               // kind: DGSQP_SAMPLE_HEAD_TO_HEAD / DGSQP_SAMPLE_AGENTS
  double first_seg_len, hw, obs_d;
  double rsum[4][4];         // collision distance r_i + r_j
};

static inline int mc_racing_fill(const dgsqp_racing_game* g, const double* key_pts, int kind, McRacing* S) {
  if (!g || g->M < 2 || g->M > DGSQP_MAX_AGENTS || ro_fill(g, key_pts, &S->P) != 0) return -1;
  if (kind != DGSQP_SAMPLE_HEAD_TO_HEAD && kind != DGSQP_SAMPLE_AGENTS) return -1;
  if (kind == DGSQP_SAMPLE_HEAD_TO_HEAD && g->M != 2) return -1;
  S->M = g->M; S->kind = kind;
  S->first_seg_len = g->track_seg_len[0]; S->hw = g->half_width;
  S->obs_d = g->obs_r[0] + g->obs_r[1];
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j)
      // head-to-head: radii [obs_d / 2, obs_d / 2] (montecarlo.sample_head_to_head)
      S->rsum[i][j] = kind == DGSQP_SAMPLE_HEAD_TO_HEAD ? S->obs_d / 2 + S->obs_d / 2 : g->obs_r[i] + g->obs_r[j];
  return 0;
}

DG_HD int mc_racing_draws(const McRacing& S) { return S.kind == DGSQP_SAMPLE_HEAD_TO_HEAD ? 5 : 3 * S.M; }

// start (s, x_tran, v) of every agent of trial t; false when the head-to-head pre-check rejects the trial
template <int M>
DG_HD bool mc_racing_starts(const McRacing& S, const McPcg& g0, const mc_u128* table, int64_t t, double* s, double* xt,
                            double* v) {
  McPcg g = mc_pcg_at(g0, table, (uint64_t)t * (uint64_t)mc_racing_draws(S));
  const double hw = S.hw;
  if (S.kind == DGSQP_SAMPLE_HEAD_TO_HEAD) {
    const double ego_s = fmax(0.1, mc_pcg_random(g) * S.first_seg_len);
    const double ego_xt = mc_pcg_random(g) * hw * 2 - hw;
    const double ego_v = mc_pcg_random(g) + 2;
    const double d = 2 * 3.141592653589793 * mc_pcg_random(g);
    const double tar_v = mc_pcg_random(g) + 2;
    const double tar_s = ego_s + 1.2 * S.obs_d * cos(d);
    const double tar_xt = ego_xt + 1.2 * S.obs_d * sin(d);
    s[0] = ego_s; xt[0] = ego_xt; v[0] = ego_v;
    s[1] = tar_s; xt[1] = tar_xt; v[1] = tar_v;
    return tar_s >= 0 && fabs(tar_xt) <= hw;
  }
#pragma unroll
  for (int a = 0; a < M; ++a) {
    s[a] = fmax(0.1, mc_pcg_random(g) * S.first_seg_len);
    xt[a] = mc_pcg_random(g) * hw * 2 - hw;
    v[a] = mc_pcg_random(g) + 2;
  }
  return true;
}

template <int M>
DG_HD bool mc_racing_collide(const McRacing& S, const RoAgent* ag) {
#pragma unroll
  for (int i = 0; i < M; ++i)
#pragma unroll
    for (int j = i + 1; j < M; ++j) {
      const double dx = ag[i].q[0] - ag[j].q[0], dy = ag[i].q[1] - ag[j].q[1];
      if (sqrt(dx * dx + dy * dy) < S.rsum[i][j]) return true;
    }
  return false;
}

// montecarlo._collision_free over the PID roll-outs of all agents, with the agents advanced in lock-step one stage at a
// time so that a trial stops at its first collision
template <int M>
DG_HD bool mc_racing_accept(const McRacing& S, const double* s, const double* xt, const double* v) {
  RoAgent ag[M];
#pragma unroll
  for (int a = 0; a < M; ++a) ro_start(S.P, s[a], xt[a], v[a], ag[a]);
  if (mc_racing_collide<M>(S, ag)) return false;
#pragma unroll 1
  for (int k = 0; k < S.P.N; ++k) {
#pragma unroll
    for (int a = 0; a < M; ++a) {
      double ua, us;
      ro_step(S.P, ag[a], ua, us);
    }
    if (mc_racing_collide<M>(S, ag)) return false;
  }
  return true;
}

template <int M>
DG_HD bool mc_racing_decide(const McRacing& S, const McPcg& g0, const mc_u128* table, int64_t t) {
  double s[4], xt[4], v[4];
  return mc_racing_starts<M>(S, g0, table, t, s, xt, v) && mc_racing_accept<M>(S, s, xt, v);
}

// agent a of the instance drawn by trial t: its block of x0 (state2q) and of the agent-major warm start
DG_HD void mc_racing_instance(const McRacing& S, const McPcg& g0, const mc_u128* table, int64_t t, int a, double* q0,
                              double* u_ws) {
  double s[4], xt[4], v[4];
  if (S.M == 2) mc_racing_starts<2>(S, g0, table, t, s, xt, v);
  else if (S.M == 3) mc_racing_starts<3>(S, g0, table, t, s, xt, v);
  else mc_racing_starts<4>(S, g0, table, t, s, xt, v);
  ro_agent(S.P, s[a], xt[a], v[a], q0, nullptr, u_ws);
}

// ------------------------------------------------------------------------------------------------------ merge game
// montecarlo.sample_merge: cars 1, 2 on the straight lane, car 3 on the ramp; rejected when the zero-input RK3 roll-outs
// collide, with car 3 rolled out from the zero state (SURVEY App. C #6)
struct McMerge {
  int N;
  double h, th, cth, sth, x_nom3, y_nom3;
  double rsum[3][3];
};

static inline int mc_merge_fill(const dgsqp_merge_game* g, McMerge* S) {
  if (!g || g->M != 3 || g->N < 1) return -1;
  const double pi = 3.141592653589793;
  const double x5_0 = 1.5, x7_0 = g->lane[2][1].brk;
  S->N = g->N; S->h = g->dt;
  S->th = pi / 12; S->cth = cos(S->th); S->sth = sin(S->th);
  S->x_nom3 = 0.25;
  S->y_nom3 = -((x7_0 + x5_0) / 2 - 0.25) * tan(S->th);
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) S->rsum[i][j] = g->obs_r[i] + g->obs_r[j];
  return 0;
}

// x0 of trial t: q = [x, y, v, psi] of the three cars
DG_HD void mc_merge_draw(const McMerge& S, const McPcg& g0, const mc_u128* table, int64_t t, double* q) {
  const double pi = 3.141592653589793;
  McPcg g = mc_pcg_at(g0, table, (uint64_t)t * 12u);
  double r[12];
  for (int i = 0; i < 12; ++i) r[i] = mc_pcg_random(g);
  for (int c = 0; c < 2; ++c) {
    const double x_nom = c == 0 ? 0.0 : 0.5;
    q[4 * c] = x_nom + 0.5 * r[4 * c] - 0.25;
    q[4 * c + 1] = 0.15 + 0.1 * r[4 * c + 1] - 0.05;
    q[4 * c + 2] = 0.3 * (1 + 0.06 * r[4 * c + 2] - 0.03);
    q[4 * c + 3] = 0.0 + (5 * r[4 * c + 3] - 2.5) * pi / 180;
  }
  const double s_ = 0.5 * r[8] - 0.25, ey = 0.1 * r[9] - 0.05;
  q[8] = S.x_nom3 + s_ * S.cth - ey * S.sth;
  q[9] = S.y_nom3 + s_ * S.sth + ey * S.cth;
  q[10] = 0.3 * (1 + 0.06 * r[10] - 0.03);
  q[11] = pi / 12 + (5 * r[11] - 2.5) * pi / 180;
}

DG_HD bool mc_merge_accept(const McMerge& S, const double* q) {
  double p0[3][2], inc[3][2];
  for (int c = 0; c < 3; ++c) {
    const double x = c < 2 ? q[4 * c] : 0.0, y = c < 2 ? q[4 * c + 1] : 0.0;
    const double v = c < 2 ? q[4 * c + 2] : 0.0, psi = c < 2 ? q[4 * c + 3] : 0.0;
    const double ax = S.h * v * cos(psi), ay = S.h * v * sin(psi);
    p0[c][0] = x; p0[c][1] = y;
    inc[c][0] = (ax + 4 * ax + ax) / 6;
    inc[c][1] = (ay + 4 * ay + ay) / 6;
  }
  for (int k = 0; k <= S.N; ++k)
    for (int i = 0; i < 3; ++i)
      for (int j = i + 1; j < 3; ++j) {
        const double dx = (p0[i][0] + (double)k * inc[i][0]) - (p0[j][0] + (double)k * inc[j][0]);
        const double dy = (p0[i][1] + (double)k * inc[i][1]) - (p0[j][1] + (double)k * inc[j][1]);
        if (sqrt(dx * dx + dy * dy) < S.rsum[i][j]) return false;
      }
  return true;
}
