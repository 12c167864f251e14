// Host build of the device sampler source (dgsqp_b200/csrc/mc_sampler.cuh).  TEST HARNESS ONLY: the CPU tests compare the
// stream, the per-trial decisions and the instances with NumPy (tests/test_device_sampler.py); nothing in dgsqp_b200/
// loads it.  Built with -ffp-contract=off, the host counterpart of the sampler unit's -fmad=false.
#include "../../include/dgsqp_b200.h"
#include "../../dgsqp_b200/csrc/mc_sampler.cuh"

extern "C" {

int hs_mc_sizeof_pcg64(void) { return (int)sizeof(dgsqp_pcg64); }

// n doubles of the stream starting at draw number d
void hs_mc_random(const dgsqp_pcg64* rng, uint64_t d, int n, double* out) {
  McPcg g = mc_pcg_from(rng);
  mc_u128 table[128];
  mc_jump_table(g.inc, table);
  g = mc_pcg_at(g, table, d);
  for (int i = 0; i < n; ++i) out[i] = mc_pcg_random(g);
}

// accept flags of trials 0..T-1
int hs_mc_racing_decide(const dgsqp_racing_game* game, const double* key_pts, int kind, const dgsqp_pcg64* rng, int64_t T,
                        uint8_t* flag) {
  McRacing S;
  if (mc_racing_fill(game, key_pts, kind, &S) != 0) return -1;
  const McPcg g0 = mc_pcg_from(rng);
  mc_u128 table[128];
  mc_jump_table(g0.inc, table);
  for (int64_t t = 0; t < T; ++t)
    flag[t] = S.M == 2 ? mc_racing_decide<2>(S, g0, table, t) : S.M == 3 ? mc_racing_decide<3>(S, g0, table, t)
                                                                           : mc_racing_decide<4>(S, g0, table, t);
  return 0;
}

// x0 [n, 6M] and u_ws [n, 2NM] of the instances drawn by the given trials
int hs_mc_racing_instances(const dgsqp_racing_game* game, const double* key_pts, int kind, const dgsqp_pcg64* rng, int n,
                           const int64_t* trial, double* x0, double* u_ws) {
  McRacing S;
  if (mc_racing_fill(game, key_pts, kind, &S) != 0) return -1;
  const McPcg g0 = mc_pcg_from(rng);
  mc_u128 table[128];
  mc_jump_table(g0.inc, table);
  const int nq = 6 * S.M, nu = 2 * S.P.N * S.M;
  for (int b = 0; b < n; ++b)
    for (int a = 0; a < S.M; ++a)
      mc_racing_instance(S, g0, table, trial[b], a, x0 + (size_t)b * nq + 6 * a, u_ws + (size_t)b * nu + (size_t)a * 2 * S.P.N);
  return 0;
}

// accept flags and x0 [T, 12] of trials 0..T-1 of the merge scenario
int hs_mc_merge(const dgsqp_merge_game* game, const dgsqp_pcg64* rng, int64_t T, uint8_t* flag, double* x0) {
  McMerge S;
  if (mc_merge_fill(game, &S) != 0) return -1;
  const McPcg g0 = mc_pcg_from(rng);
  mc_u128 table[128];
  mc_jump_table(g0.inc, table);
  for (int64_t t = 0; t < T; ++t) {
    mc_merge_draw(S, g0, table, t, x0 + t * 12);
    flag[t] = mc_merge_accept(S, x0 + t * 12);
  }
  return 0;
}

}  // extern "C"
