// Constraints, matrix-free constraint Jacobian and condensed game-KKT data shared by the device games (see game.cuh).
//
// Replaces the CasADi functions evaluated by DGSQP._evaluate (DGSQP/solvers/DGSQP.py:509-533):
//   f_Du_x (:642-650), f_Cxu (:804-821), f_Du_C (:824-826), f_q (:673-676,898-899), f_Q (:679-727,829-934).
// The constraint Jacobian G is never materialised: it is kept as the sensitivity rows of the states the constraints
// read (x, y, DG_BOUND_STATE) and applied matrix-free (G v, G' w, single rows on demand).  Collision, input-bound and
// state-bound rows are written here; the game-specific row family (K_GAME) and the cost terms that differ between the
// games come from the hooks of the game header that includes this file (listed in game.cuh).
#pragma once

// f_Cxu: one thread per row
template <bool SM>
DG_DEVN void game_constraints(Cta& c, const GameDesc& G, const Dims& D_, const double* u, const double* up,
                              const double* x, double* g, const int* DG_RESTRICT rowtab) {
  // local copies: the tables live in shared memory and would otherwise be re-read after every store
  const Dims D = D_;
  DG_ASSUME_SHARED(x); DG_ASSUME_SHARED(g); DG_ASSUME_SHARED(up);
  DG_FOR(r, D.m) {
    int k, kind, a, b;
    unpack_row(rowtab[r], k, kind, a, b);
    double val;
    if (kind == K_COLL) {
      double dx = x[k * D.nq + a * DG_NQA] - x[k * D.nq + b * DG_NQA];
      double dy = x[k * D.nq + a * DG_NQA + 1] - x[k * D.nq + b * DG_NQA + 1];
      double rr = G.obs_r[a] + G.obs_r[b];
      val = rr * rr - (dx * dx + dy * dy);
    } else if (kind == K_GAME) val = game_row_value(G, D, u, up, x, k, a, b);
    else if (kind == K_INUB) val = u[uidx(D, a, k, b)] - G.u_ub[b];
    else if (kind == K_INLB) val = G.u_lb[b] - u[uidx(D, a, k, b)];
    else if (kind == K_STUB) val = x[k * D.nq + a * DG_NQA + b] - game_state_ub(G);
    else val = game_state_lb(G) - x[k * D.nq + a * DG_NQA + b];
    g[r] = val;
  }
}

// Sensitivity rows (f_Du_x restricted to x, y, DG_BOUND_STATE): thread per input column (a, j), the agents interleaved
// (t = j * M + a) so that the column length N - kj falls with the thread index: the last threads, which share their
// warps with the costate chains (game_costates), hold the shortest columns.
template <bool SM>
DG_DEVN void game_sens(Cta& c, const Dims& D_, const EvalBuf& E_) {
  // local copies: the tables live in shared memory and would otherwise be re-read after every store
  const EvalBuf E = E_; DG_SH_EVAL(E); const Dims D = D_;
  const int twoN = D.twoN;
  DG_FOR(t, D.M * twoN) {
    int j = t / D.M, a = t - j * D.M, kj = j >> 1, cc = j & 1;
    double s[DG_NQA];
    const double* AB = E.AB + (kj * D.M + a) * DG_AB_SZ;
    for (int i = 0; i < DG_NQA; ++i) s[i] = AB[i * DG_AB_LD + DG_NQA + cc];
    for (int k = kj + 1; k <= D.N; ++k) {
      if (k > kj + 1) {
        const double* Ak = E.AB + ((k - 1) * D.M + a) * DG_AB_SZ;
        double ts[DG_NQA];
        for (int i = 0; i < DG_NQA; ++i) {
          double acc = 0.0;
          for (int jj = 0; jj < DG_NQA; ++jj) acc += Ak[i * DG_AB_LD + jj] * s[jj];
          ts[i] = acc;
        }
        for (int i = 0; i < DG_NQA; ++i) s[i] = ts[i];
      }
      double* Sk = E.S + sens_off(D, a, k, 0) + j;
      Sk[0] = s[0]; Sk[2 * k] = s[1]; Sk[4 * k] = s[DG_BOUND_STATE];
    }
  }
}

template <bool SM>
DG_DEV double sens_dot(const Dims& D, const EvalBuf& E, int a, int k, int row, const double* va) {
  const double* DG_RESTRICT Sk = E.S + sens_off(D, a, k, row);
  double a0 = 0.0, a1 = 0.0;
  for (int j = 0; j < 2 * k; j += 2) { a0 += Sk[j] * va[j]; a1 += Sk[j + 1] * va[j + 1]; }
  return a0 + a1;
}

// y = G v   (v in R^n agent-major, y in R^m).  Two phases with one sync.
template <bool SM>
DG_DEVN void game_G_times(Cta& c, const Dims& D_, const EvalBuf& E_, const double* v, double* y) {
  // local copies: the tables live in shared memory and would otherwise be re-read after every store
  const EvalBuf E = E_; DG_SH_EVAL(E); const Dims D = D_;
  c.sync();
  DG_FOR(t, D.M * D.N * 3) {
    int a = t / (D.N * 3), rem = t - a * D.N * 3, k1 = rem / 3, row = rem - k1 * 3;
    E.tmpS[t] = sens_dot<SM>(D, E, a, k1 + 1, row, v + a * D.twoN);
  }
  c.sync();
  DG_FOR(r, D.m) {
    int k, kind, a, b;
    unpack_row(E.rowtab[r], k, kind, a, b);
    double val;
    if (kind == K_COLL) {
      double dx = E.x[k * D.nq + a * DG_NQA] - E.x[k * D.nq + b * DG_NQA];
      double dy = E.x[k * D.nq + a * DG_NQA + 1] - E.x[k * D.nq + b * DG_NQA + 1];
      const double* ta = E.tmpS + (a * D.N + (k - 1)) * 3;
      const double* tb = E.tmpS + (b * D.N + (k - 1)) * 3;
      val = -2.0 * (dx * (ta[0] - tb[0]) + dy * (ta[1] - tb[1]));
    } else if (kind == K_GAME) val = game_row_Gv(D, E, v, k, a, b);
    else if (kind == K_INUB) val = v[uidx(D, a, k, b)];
    else if (kind == K_INLB) val = -v[uidx(D, a, k, b)];
    else if (kind == K_STUB) val = E.tmpS[(a * D.N + (k - 1)) * 3 + 2];
    else val = -E.tmpS[(a * D.N + (k - 1)) * 3 + 2];
    y[r] = val;
  }
  c.sync();
}

// per (a,k>=1) coefficients of the state rows in  G' w:  cf = [c_x, c_y, c_bound]
template <bool SM>
DG_DEV void game_state_coefs(Cta& c, const Dims& D, const EvalBuf& E, const double* w, double* cf) {
  DG_FOR(t, D.M * D.N) {
    int a = t / D.N, k = t - a * D.N + 1;
    double cx = 0.0, cy = 0.0;
    for (int p = 0; p < D.P; ++p) {
      int i, j;
      pair_ij(D.M, p, i, j);
      if (i != a && j != a) continue;
      double dx = E.x[k * D.nq + i * DG_NQA] - E.x[k * D.nq + j * DG_NQA];
      double dy = E.x[k * D.nq + i * DG_NQA + 1] - E.x[k * D.nq + j * DG_NQA + 1];
      double wl = w[row_coll(D, k, p)] * (i == a ? -2.0 : 2.0);
      cx += wl * dx; cy += wl * dy;
    }
    game_row_coefs(D, E, w, k, a, cx, cy);
    cf[t * 3] = cx; cf[t * 3 + 1] = cy;
    cf[t * 3 + 2] = w[row_stub(D, k, a)] - w[row_stlb(D, k, a)];
  }
}

// input-dependent (sparse) rows of G' w at input (a,k,cc): the game's rows and the input bounds iub / ilb
DG_DEV double game_GT_direct(const Dims& D, const double* w, int a, int k, int cc) {
  return game_row_GT_direct(D, w, a, k, cc, row_inub(D, k, a, cc), row_inlb(D, k, a, cc));
}

// y = G' w  (w in R^m, y in R^n)
template <bool SM>
DG_DEVN void game_GT_times(Cta& c, const Dims& D_, const EvalBuf& E_, const double* w, double* y) {
  // local copies: the tables live in shared memory and would otherwise be re-read after every store
  const EvalBuf E = E_; DG_SH_EVAL(E); const Dims D = D_;
  c.sync();
  game_state_coefs<SM>(c, D, E, w, E.cf);
  c.sync();
  DG_FOR(t, D.n) {
    int a = t / D.twoN, j = t - a * D.twoN, kj = j >> 1, cc = j & 1;
    double acc = game_GT_direct(D, w, a, kj, cc);
    for (int k = kj + 1; k <= D.N; ++k) {
      const double* Sk = E.S + sens_off(D, a, k, 0) + j;
      const double* cf = E.cf + (a * D.N + (k - 1)) * 3;
      acc += cf[0] * Sk[0] + cf[1] * Sk[2 * k] + cf[2] * Sk[4 * k];
    }
    y[t] = acc;
  }
  c.sync();
}

// Entry G[r][t] of the row r = (k, kind, a, b); rc holds what the game's rows precompute per row (game_row_prep).
// game_G_sparse below must list the same +-1 entries.
DG_DEV double game_G_entry(const Dims& D, const EvalBuf& E, const RowCoef& rc, int k, int kind, int a, int b, int t) {
  int ta = t / D.twoN, j = t - ta * D.twoN, kj = j >> 1, cc = j & 1;
  double val = 0.0;
  if (kind == K_COLL) {
    if ((ta == a || ta == b) && kj < k) {
      double dx = E.x[k * D.nq + a * DG_NQA] - E.x[k * D.nq + b * DG_NQA];
      double dy = E.x[k * D.nq + a * DG_NQA + 1] - E.x[k * D.nq + b * DG_NQA + 1];
      const double* Sk = E.S + sens_off(D, ta, k, 0) + j;
      double sg = ta == a ? -2.0 : 2.0;
      val = sg * (dx * Sk[0] + dy * Sk[2 * k]);
    }
  } else if (kind == K_GAME) game_row_G(D, E, rc, k, a, b, ta, j, kj, cc, val);
  else if (kind == K_INUB) { if (ta == a && kj == k && cc == b) val = 1.0; }
  else if (kind == K_INLB) { if (ta == a && kj == k && cc == b) val = -1.0; }
  else {
    if (ta == a && kj < k) {
      double sv = E.S[sens_off(D, ta, k, 2) + j];
      val = kind == K_STUB ? sv : -sv;
    }
  }
  return val;
}

// Rows of G whose only entries are +-1 (input bounds, and the game rows that game_row_sparse accepts): true, and the
// entries as (input index << 1 | negative) in t1 / t2 (-1 = none); false for the rows that read the sensitivities.
DG_DEV bool game_G_sparse(const Dims& D, int r, int& t1, int& t2) {
  int k, kind, a, b;
  decode_row(D, r, k, kind, a, b);
  t1 = t2 = -1;
  if (kind == K_INUB) { t1 = uidx(D, a, k, b) << 1; return true; }
  if (kind == K_INLB) { t1 = (uidx(D, a, k, b) << 1) | 1; return true; }
  if (kind == K_GAME) return game_row_sparse(D, k, a, b, t1, t2);
  return false;
}

// dense row r of G into out[n] (all threads cooperate)
template <bool SM>
DG_DEVN void game_G_row(Cta& c, const Dims& D_, const EvalBuf& E_, int r, double* out) {
  // local copies: the tables live in shared memory and would otherwise be re-read after every store
  const EvalBuf E = E_; DG_SH_EVAL(E); const Dims D = D_;
  int k, kind, a, b;
  decode_row(D, r, k, kind, a, b);
  RowCoef rc;
  game_row_prep(D, E, k, kind, a, b, rc);
  DG_FOR(t, D.n) out[t] = game_G_entry(D, E, rc, k, kind, a, b, t);
  c.sync();
}

// Rows ids[0..cnt) of G, transposed: out[t * ldo + c] = G[ids[c]][t], t < n (one warp per row, lanes along the inputs).
// No barrier: the caller synchronises.  Used by the blocked warm start of the QP (qp_gi.cuh).
template <bool SM>
DG_DEVN void game_G_cols(Cta& c, const Dims& D_, const EvalBuf& E_, const int* ids, int cnt, double* out, int ldo) {
  const EvalBuf E = E_; DG_SH_EVAL(E); const Dims D = D_;
  for (int col = c.warp(); col < cnt; col += c.nwarps()) {
    int k, kind, a, b;
    decode_row(D, ids[col], k, kind, a, b);
    RowCoef rc;
    game_row_prep(D, E, k, kind, a, b, rc);
    for (int t = c.lane(); t < D.n; t += c.wsz) out[t * ldo + col] = game_G_entry(D, E, rc, k, kind, a, b, t);
  }
}

// d(l'C)/dx_k entry idx (state-dependent rows), k>=1
DG_DEV double con_lx(const GameDesc& G, const Dims& D, const double* x, const double* l, int k, int idx) {
  int a = idx / DG_NQA, comp = idx - a * DG_NQA;
  if (comp == DG_BOUND_STATE) return l[row_stub(D, k, a)] - l[row_stlb(D, k, a)];
  if (comp > 1) return 0.0;
  double v = 0.0;
  for (int p = 0; p < D.P; ++p) {
    int i, j;
    pair_ij(D.M, p, i, j);
    if (i != a && j != a) continue;
    double dd = x[k * D.nq + i * DG_NQA + comp] - x[k * D.nq + j * DG_NQA + comp];
    v += l[row_coll(D, k, p)] * (i == a ? -2.0 : 2.0) * dd;
  }
  game_row_lx(G, D, x, l, k, a, comp, v);
  return v;
}

// d2(l'C)/dx_k^2 entry (collision rows only: the game rows are linear in the states), k>=1
DG_DEV double con_lxx(const Dims& D, const double* l, int k, int i1, int i2) {
  int a1 = i1 / DG_NQA, c1 = i1 - a1 * DG_NQA, a2 = i2 / DG_NQA, c2 = i2 - a2 * DG_NQA;
  if (c1 > 1 || c1 != c2) return 0.0;
  double v = 0.0;
  for (int p = 0; p < D.P; ++p) {
    int i, j;
    pair_ij(D.M, p, i, j);
    double lp = l[row_coll(D, k, p)];
    if (a1 == a2) { if (a1 == i || a1 == j) v += -2.0 * lp; }
    else if ((a1 == i && a2 == j) || (a1 == j && a2 == i)) v += 2.0 * lp;
  }
  return v;
}

// Costate chains  p_k = l_x,k + A_k' p_{k+1}:  one chain per (function f, agent block b), one lane per entry of p_k.
// f < M: cost of agent f (terminal and stage state costs); f == M: l'C.
// The chains are packed wsz / DG_NQA to a warp into the last warps of the CTA.  game_sens runs in the same barrier
// interval with its longest columns on the first threads: at chicane, merge and three agents (N = 25) the chain warps
// hold no sensitivity column at 256 threads; otherwise they share their warps with the shortest columns.
template <bool SM>
DG_DEVN void game_costates(Cta& c, const GameDesc& G, const Dims& D_, const EvalBuf& E_, const double* l) {
  // local copies: the tables live in shared memory and would otherwise be re-read after every store
  const EvalBuf E = E_; DG_SH_EVAL(E); const Dims D = D_;
  const int nch = (D.M + 1) * D.M;
  const int cpw = c.wsz >= DG_NQA ? c.wsz / DG_NQA : nch;       // chains per warp (host build: all on its one thread)
  const int ng = (nch + cpw - 1) / cpw, w = c.nwarps() - 1 - c.warp();
  const int nown = ng > w ? (ng - w + c.nwarps() - 1) / c.nwarps() : 0;   // this warp's groups: w, w + nwarps(), ..
  const int per = cpw * DG_NQA;
  for (int it = c.lane(); it < nown * per; it += c.wsz) {
    const int o = it / per, e = it - o * per, t = (w + o * c.nwarps()) * cpw + e / DG_NQA, i = e % DG_NQA;
    if (t >= nch) continue;
    const int f = t / D.M, b = t - f * D.M;
    E.cst[(f * (D.N + 1) + D.N) * D.nq + b * DG_NQA + i] =
        f < D.M ? game_term_lx(G, D, E.x, f, b * DG_NQA + i) : con_lx(G, D, E.x, l, D.N, b * DG_NQA + i);
  }
  c.syncwarp();
  for (int k = D.N - 1; k >= 0; --k) {
    for (int it = c.lane(); it < nown * per; it += c.wsz) {
      const int o = it / per, e = it - o * per, t = (w + o * c.nwarps()) * cpw + e / DG_NQA, j = e % DG_NQA;
      if (t >= nch) continue;
      const int f = t / D.M, b = t - f * D.M;
      const double* Ak = E.AB + (k * D.M + b) * DG_AB_SZ;
      double* out = E.cst + (f * (D.N + 1) + k) * D.nq + b * DG_NQA;
      const double* p = out + D.nq;
      double acc = 0.0;
      if (k >= 1) acc = f < D.M ? game_stage_lx(G, D, E.x, f, k, b * DG_NQA + j) : con_lx(G, D, E.x, l, k, b * DG_NQA + j);
      // explicit fma(A, p, acc): a game whose l_x is a bare product (merge) must not have that product fused instead
      for (int i = 0; i < DG_NQA; ++i) acc = DG_FMA(Ak[i * DG_AB_LD + j], p[i], acc);
      out[j] = acc;
    }
    c.syncwarp();
  }
}

// q (cost gradient, f_q) and G'l from the costates: thread per input (a,k,cc)
template <bool SM>
DG_DEVN void game_gradients(Cta& c, const GameDesc& G, const Dims& D_, const EvalBuf& E_, const double* u,
                            const double* up, const double* l, double* qs) {
  // local copies: the tables live in shared memory and would otherwise be re-read after every store
  const EvalBuf E = E_; DG_SH_EVAL(E); const Dims D = D_;
  DG_FOR(t, D.n) {
    int a = t / D.twoN, j = t - a * D.twoN, k = j >> 1, cc = j & 1;
    const double* Bk = E.AB + (k * D.M + a) * DG_AB_SZ;
    const double* pJ = E.cst + a * (D.N + 1) * D.nq + (k + 1) * D.nq + a * DG_NQA;
    const double* pC = E.cst + D.M * (D.N + 1) * D.nq + (k + 1) * D.nq + a * DG_NQA;
    double bj = 0.0, bc = 0.0;
    for (int i = 0; i < DG_NQA; ++i) { bj += Bk[i * DG_AB_LD + DG_NQA + cc] * pJ[i]; bc += Bk[i * DG_AB_LD + DG_NQA + cc] * pC[i]; }
    const InputGrad ig = game_input_grad(G, D, u, up, t, a, k, cc);
    E.q[t] = input_grad_plus(ig, bj);
    if (qs) {      // grad_u sum_f J^f, only wanted by the v2 merit 'sum_obj_l1' (DGSQP_v2.py:1149-1151)
      // every agent's state costs reach u^a through the states: sum over the cost costates of all functions
      double bs = bj;
      for (int f = 0; f < D.M; ++f) {
        if (f == a) continue;
        const double* pF = E.cst + f * (D.N + 1) * D.nq + (k + 1) * D.nq + a * DG_NQA;
        for (int i = 0; i < DG_NQA; ++i) bs += Bk[i * DG_AB_LD + DG_NQA + cc] * pF[i];
      }
      qs[t] = input_grad_plus(ig, bs);
    }
    E.gtl[t] = game_GT_direct(D, l, a, k, cc) + bc;
  }
}

// Hc[f][k][a][0..DG_HC_SZ) = sum_i p^f_{k+1}[a,i] * T2[k][a][i][:]
template <bool SM>
DG_DEVN void game_contract(Cta& c, const Dims& D_, const EvalBuf& E_) {
  // local copies: the tables live in shared memory and would otherwise be re-read after every store
  const EvalBuf E = E_; DG_SH_EVAL(E); const Dims D = D_;
  DG_FOR(t, (D.M + 1) * D.N * D.M * DG_HC_SZ) {
    int e = t % DG_HC_SZ, r = t / DG_HC_SZ;
    int a = r % D.M; r /= D.M;
    int k = r % D.N, f = r / D.N;
    const double* p = E.cst + f * (D.N + 1) * D.nq + (k + 1) * D.nq + a * DG_NQA;
    const double* T = E.T2 + (k * D.M + a) * DG_T2_SZ;
    E.Hc[t] = game_contract_entry(p, T, e);
  }
}

// Game Hessian Q (f_Q): ONE backward sweep over the stages carrying all M+1 functions (the M costs and
// l'C).   row block a of Q = grad_{u^a} grad_u (J^a + l'C)   (DGSQP.py:920-934)
// Row r (stage-major input index (k_r, a_r, c_r)) of Dxu_Q^f is kept as w^f in E.Wrow[(f*nq + q)*n + r] for every
// function f.  At stage k < k_r the row emits H^f[r, (k,b,cc)] = w^f[b] . B^b_k[:,cc] and
// Q[r][(k,b,cc)] = H^{a_r} + H^M  and, by symmetry of each H^f,  Q[(k,b,cc)][r] = H^b + H^M.
// Every entry of Q is written exactly once, so Q needs no zero-fill and no read-modify-write.
// Per stage, two barrier intervals whose work items are spread over the whole CTA:
//   A: (row r with k_r > k, agent block b): propagate w through A_k^b and emit the two Q entries       [n_later*M items]
//      (function f, new row (a_r,c_r), column j): tv = B_k' V^f  (first half of the same-stage products) [F*nu*nq items]
//      (function f, i1, i2): V_k = lxx_k + A'VA + E.p                                                      [F*nq*nq items]
//   B: (f, new row, b, j): w = tv A_k + (G.p)   and   (new row, b, cc): same-stage block luu + B'VB + F.p
template <bool SM>
DG_DEVN void game_hessian(Cta& c, const GameDesc& G, const Dims& D_, const EvalBuf& E_, const double* DG_RESTRICT l) {
  // local copies: the tables live in shared memory and would otherwise be re-read after every store
  const EvalBuf E = E_; DG_SH_EVAL(E); const Dims D = D_;
  const int n = D.n, nq = D.nq, nu = D.nu, N = D.N, M = D.M, F = D.M + 1;
  double* Vcur = E.Vbuf;
  double* Vnext = E.Vbuf + F * nq * nq;
  double* DG_RESTRICT TV = E.Vbuf + 2 * F * nq * nq;            // [(f*nu + rr)*nq + j]
  DG_FOR(t, F * nq * nq) {
    int f = t / (nq * nq), e = t - f * nq * nq, i1 = e / nq, i2 = e - i1 * nq;
    Vcur[t] = f < M ? game_term_lxx(G, D, E.x, f, i1, i2) : con_lxx(D, l, N, i1, i2);
  }
  c.sync();
  double* DG_RESTRICT Qm = E.Q;
  for (int k = N - 1; k >= 0; --k) {
    const int nlater = n - (k + 1) * nu;                          // rows with k_r > k
    const int nA1 = nlater * M, nA2 = F * nu * nq, nA3 = F * nq * nq;
    for (int t = c.tid(); t < nA1 + nA2 + nA3; t += c.nt()) {
      if (t < nA1) {
        const int b = t / nlater, r = (k + 1) * nu + (t - b * nlater);
        const int kr = r / nu, ar = (r - kr * nu) >> 1, cr = r & 1;
        const int rowQ = uidx(D, ar, kr, cr);
        double* DG_RESTRICT wr = E.Wrow + r;                     // w^f[q] at wr[(f*nq + q)*n]
        const double* DG_RESTRICT ABk = E.AB + (k * M + b) * DG_AB_SZ;
        double hM0 = 0.0, hM1 = 0.0, hA0 = 0.0, hA1 = 0.0, hB0 = 0.0, hB1 = 0.0;
        for (int f = 0; f < F; ++f) {
          double wv[DG_NQA];
#pragma unroll
          for (int i = 0; i < DG_NQA; ++i) wv[i] = wr[(f * nq + b * DG_NQA + i) * n];
          if (f == M || f == ar || f == b) {
            double v0 = 0.0, v1 = 0.0;
#pragma unroll
            for (int i = 0; i < DG_NQA; ++i) { v0 += wv[i] * ABk[i * DG_AB_LD + DG_NQA]; v1 += wv[i] * ABk[i * DG_AB_LD + DG_NQA + 1]; }
            if (f < M && kr == k + 1 && b == ar && f == ar) game_input_hess_prev(G, cr, v0, v1);
            if (f == M) { hM0 = v0; hM1 = v1; }
            if (f == ar) { hA0 = v0; hA1 = v1; }
            if (f == b) { hB0 = v0; hB1 = v1; }
          }
#pragma unroll
          for (int j = 0; j < DG_NQA; ++j) {
            double acc = 0.0;
#pragma unroll
            for (int i = 0; i < DG_NQA; ++i) acc += wv[i] * ABk[i * DG_AB_LD + j];
            wr[(f * nq + b * DG_NQA + j) * n] = acc;
          }
        }
        const int colQ = uidx(D, b, k, 0);
        Qm[rowQ * n + colQ] = hA0 + hM0;  Qm[rowQ * n + colQ + 1] = hA1 + hM1;
        Qm[colQ * n + rowQ] = hB0 + hM0;  Qm[(colQ + 1) * n + rowQ] = hB1 + hM1;
      } else if (t < nA1 + nA2) {
        const int e = t - nA1, f = e / (nu * nq), rem = e - f * nu * nq, rr = rem / nq, j = rem - rr * nq;
        const int ar = rr >> 1, cr = rr & 1;
        const double* DG_RESTRICT ABa = E.AB + (k * M + ar) * DG_AB_SZ;
        const double* DG_RESTRICT Vf = Vcur + f * nq * nq;
        double acc = 0.0;
#pragma unroll
        for (int i = 0; i < DG_NQA; ++i) acc += ABa[i * DG_AB_LD + DG_NQA + cr] * Vf[(ar * DG_NQA + i) * nq + j];
        TV[e] = acc;
      } else {
        // V_k = lxx_k + A'VA + E.p  for every function (into the other buffer)
        const int tt = t - nA1 - nA2;
        const int f = tt / (nq * nq), e = tt - f * nq * nq;
        const int i1 = e / nq, i2 = e - i1 * nq, b1 = i1 / DG_NQA, b2 = i2 / DG_NQA, c1 = i1 - b1 * DG_NQA, c2 = i2 - b2 * DG_NQA;
        const double* DG_RESTRICT A1 = E.AB + (k * M + b1) * DG_AB_SZ;
        const double* DG_RESTRICT A2 = E.AB + (k * M + b2) * DG_AB_SZ;
        const double* DG_RESTRICT Vf = Vcur + f * nq * nq;
        double acc = f < M ? game_stage_lxx(G, D, f, k, i1, i2) : (k >= 1 ? con_lxx(D, l, k, i1, i2) : 0.0);
        if (b1 == b2) acc += hc_xx(E.Hc + ((f * N + k) * M + b1) * DG_HC_SZ, c1, c2);
#pragma unroll
        for (int i = 0; i < DG_NQA; ++i) {
          double rowacc = 0.0;
#pragma unroll
          for (int j = 0; j < DG_NQA; ++j) rowacc += Vf[(b1 * DG_NQA + i) * nq + b2 * DG_NQA + j] * A2[j * DG_AB_LD + c2];
          acc += A1[i * DG_AB_LD + c1] * rowacc;
        }
        Vnext[tt] = acc;
      }
    }
    c.sync();
    const int nB1 = F * nu * nq, nB2 = nu * M * 2;
    for (int t = c.tid(); t < nB1 + nB2; t += c.nt()) {
      if (t < nB1) {
        // w = tv A_k + (G.p)[(ar,cr), ar-block]
        const int f = t / (nu * nq), rem = t - f * nu * nq, rr = rem / nq, q = rem - rr * nq, b = q / DG_NQA, j = q - b * DG_NQA;
        const int ar = rr >> 1, cr = rr & 1;
        const double* DG_RESTRICT ABb = E.AB + (k * M + b) * DG_AB_SZ;
        const double* DG_RESTRICT tv = TV + (f * nu + rr) * nq + b * DG_NQA;
        double acc = b == ar ? hc_ux(E.Hc + ((f * N + k) * M + ar) * DG_HC_SZ, cr, j) : 0.0;
#pragma unroll
        for (int i = 0; i < DG_NQA; ++i) acc += tv[i] * ABb[i * DG_AB_LD + j];
        E.Wrow[(f * nq + q) * n + k * nu + rr] = acc;
      } else {
        // same-stage block luu + B'VB + F.p  of the functions M and a_r
        const int e = t - nB1, rr = e / (M * 2), rem = e - rr * M * 2, b = rem >> 1, cc = rem & 1;
        const int ar = rr >> 1, cr = rr & 1;
        const double* DG_RESTRICT ABb = E.AB + (k * M + b) * DG_AB_SZ;
        double vM = 0.0, vA = 0.0;
        const double* DG_RESTRICT tvM = TV + (M * nu + rr) * nq + b * DG_NQA;
        const double* DG_RESTRICT tvA = TV + (ar * nu + rr) * nq + b * DG_NQA;
#pragma unroll
        for (int i = 0; i < DG_NQA; ++i) { vM += tvM[i] * ABb[i * DG_AB_LD + DG_NQA + cc]; vA += tvA[i] * ABb[i * DG_AB_LD + DG_NQA + cc]; }
        if (b == ar) {
          vM += hc_uu(E.Hc + ((M * N + k) * M + ar) * DG_HC_SZ, cr, cc);
          vA += hc_uu(E.Hc + ((ar * N + k) * M + ar) * DG_HC_SZ, cr, cc);
          if (cc == cr) vA += game_input_hess(G, D, k, cc);
        }
        Qm[uidx(D, ar, k, cr) * n + uidx(D, b, k, cc)] = vA + vM;
      }
    }
    c.sync();
    double* tmp = Vcur; Vcur = Vnext; Vnext = tmp;
  }
}
