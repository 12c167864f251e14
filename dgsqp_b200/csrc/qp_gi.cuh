// QP sub-problem   min 1/2 du'H du + q'du   s.t.  G du <= -g    (DGSQP._solve_qp, DGSQP.py:232-266)
//
// The reference sends this to OSQP (polish=True) through CasADi's conic interface; when polish
// succeeds the result is the exact KKT point of the strictly convex QP.  Here that point is computed
// directly by the Goldfarb-Idnani dual active-set method, one QP per CTA: H = L L' (Cholesky),
// J = L^-T, unconstrained minimiser, then add the most violated constraint / drop blocking ones.
// G is applied matrix-free through the game's sensitivity rows (racing_game.cuh).
// Conventions: slack s_i = -g_i - G_i x >= 0, normal n_i = -G_i', multipliers lam >= 0,
// H x + q + G' lam = 0.
//
// Storage: Y = J' (row-major, leading dimension ld), i.e. J(i,j) = Y[j*ld+i].  Y starts as L^-1 (tri_inverse).
// Every O(n^2) operation of an iteration is spread over the whole CTA: products with J' run warp-per-row, products
// with J and the Householder update of J's trailing columns use the 2D decomposition of cta.cuh (consecutive
// threads = consecutive columns of Y, column groups interleave the rows) with partial sums combined through
// B.part; the triangular solve with R runs on one warp while the others combine the partial sums.
#pragma once
#include "game.cuh"
#include "linalg.cuh"

#define DG_QP_FEAS_TOL 1e-10
#define DG_QP_DEP_TOL 1e-20

struct QpBuf {
  // Y = J' lives in LinBuf::matB, R (upper triangular factor of the active normals in J-coordinates) in
  // LinBuf::matA once the Cholesky factor stored there has been inverted
  double* xq;     // n   primal iterate (du)
  double* dv;     // n   J' n_p
  double* zv;     // n   primal step direction
  double* rv;     // n   dual step direction (active part)
  double* npv;    // n   G row of the entering constraint (normal is -npv); reused for the Householder vector
  double* lam_act;// n
  double* sl;     // m   G x
  double* lam;    // m   output multipliers
  int* act;       // n   active constraint ids
  int* is_act;    // m   flags
};

#define DG_SH_QP(Q) do { DG_ASSUME_SHARED((Q).xq); DG_ASSUME_SHARED((Q).dv); DG_ASSUME_SHARED((Q).zv); DG_ASSUME_SHARED((Q).rv); \
  DG_ASSUME_SHARED((Q).npv); DG_ASSUME_SHARED((Q).lam_act); DG_ASSUME_SHARED((Q).sl); DG_ASSUME_SHARED((Q).act); DG_ASSUME_SHARED((Q).is_act); } while (0)

// out[i] = scale * sum_{j in [j0, n)} Y[j][i] * d[j],  i < n.  All threads; ends with a barrier.
template <bool SM>
DG_DEV void gi_cols_times(Cta& c, int n, int ld, const double* DG_RESTRICT Y, const double* DG_RESTRICT d, int j0,
                          double* DG_RESTRICT part, double* DG_RESTRICT out, double scale) {
  // (inlined: the caller carries the address-space hints)
  const Split2 sp = split2(c, n);
  for (int i = sp.i0; i < n; i += sp.istep) {
    double a0 = 0.0, a1 = 0.0;
    int j = j0 + sp.g;
    for (; j + sp.G < n; j += 2 * sp.G) { a0 += Y[j * ld + i] * d[j]; a1 += Y[(j + sp.G) * ld + i] * d[j + sp.G]; }
    if (j < n) a0 += Y[j * ld + i] * d[j];
    if (sp.G == 1) out[i] = scale * (a0 + a1);
    else part[sp.g * sp.istep + i] = a0 + a1;
  }
  c.sync();
  if (sp.G > 1) {
    if (sp.g == 0) {
      for (int i = sp.i0; i < n; i += sp.istep) {
        double acc = part[i];
        for (int g = 1; g < sp.G; ++g) acc += part[g * sp.istep + i];
        out[i] = scale * acc;
      }
    }
    c.sync();
  }
}

// ---- warm start of the dual active-set method from the active set of the previous QP of this instance ------------------
// (SolverParams::qp_warm; BASELINE north_star: "per-instance warm start").  Successive QPs of one instance -- the next SQP
// iteration, the relaxed steps of the watchdog -- share most of their active set, and the cold method spends one
// O(n^2) iteration per constraint it adds.  Starting from Y = L^-1 and c = Y q (left in Q.dv by qp_factor):
//   (1) D = J' N_W = -Y G_W' for all k previous constraints at once: the rows of G are written side by side into matA
//       (game_G_cols) and multiplied IN PLACE by the lower-triangular Y, eight columns per thread (row j of the product
//       only reads rows <= j, so one barrier between the products and the stores suffices);
//   (2) blocked Householder QR of D (n x k): one warp factors a panel of DG_WS_PW columns (lanes along the rows; a
//       column that is linearly dependent on the accepted ones -- same test as the main loop -- ends the panel and is
//       skipped) and leaves the panel's Gram entries v_a'v_b, i.e. the inverse of the compact-WY factor T; then every
//       thread applies the block reflector  y <- y - V T'(V'y)  to one target column -- the n columns of Y, the
//       remaining columns of D and c -- in two passes over the rows, with no barrier and no reduction in between.
//       R is the factor the main loop continues with;
//   (3) the equality-constrained minimiser on that set in the cancellation-free form of gi_polish:
//       t = R^-T g_W,  lam = R^-1 (t + c1),  x = J1 t - J2 c2;
//   (4) while a multiplier is negative: drop the most negative one (Givens re-triangularisation, c rotated alike) and
//       redo (3).
// (x, lam >= 0, W) is then an S-pair, from which the method continues unchanged.  The QP is strictly convex, so the
// solution is the one the cold start reaches (up to rounding); only the path differs.
// Scratch: previous ids / source columns in Q.rv (as ints), reflector scalars v0 / 2/(v'v) in the two spare vectors of the
// 8n region behind Q.lam_act, g_W in Q.npv, the Gram block and the panel control words in B.part.
// Returns the number of active constraints; Q.act / Q.is_act / Q.lam_act / Q.xq are set accordingly.
#define DG_WS_PW 8      // panel width of the blocked QR
#define DG_WS_CW 8      // columns of D per thread in the in-place product

// v[0..8) = p[0..8): 128-bit loads when p allows (every thread of the warp reads the same address in the callers below,
// so the alignment branch is uniform)
DG_DEV void ws_load8(const double* DG_RESTRICT p, double (&v)[8]) {
#ifndef DG_HOSTSIM
  if ((reinterpret_cast<uintptr_t>(p) & 15) == 0) {
    const double2 a = reinterpret_cast<const double2*>(p)[0], b = reinterpret_cast<const double2*>(p)[1];
    const double2 d = reinterpret_cast<const double2*>(p)[2], e = reinterpret_cast<const double2*>(p)[3];
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = d.x; v[5] = d.y; v[6] = e.x; v[7] = e.y;
  } else {
    const double a0 = p[0], a7 = p[7];
    const double2 a = reinterpret_cast<const double2*>(p + 1)[0], b = reinterpret_cast<const double2*>(p + 1)[1];
    const double2 d = reinterpret_cast<const double2*>(p + 1)[2];
    v[0] = a0; v[1] = a.x; v[2] = a.y; v[3] = b.x; v[4] = b.y; v[5] = d.x; v[6] = d.y; v[7] = a7;
  }
#else
  for (int q = 0; q < 8; ++q) v[q] = p[q];
#endif
}

// Block reflector of one panel of the warm start's QR on ONE target column y (stride st): reflector q (q < pa) starts at
// row p0 + q with leading entry v0s[q]; its tail is column q of the panel V (row j at V + j*ld).  Two passes over the
// rows, RB rows per step with all loads of y issued first (RB = 2 for shared memory, 8 when y is streamed from L2).
// PAD8: the panel is processed as DG_WS_PW columns wide whatever pa is -- the coefficients w_q of the missing reflectors
// are zero, what is read in their place (finite entries of the same rows) never reaches the result.  The caller
// guarantees that those reads stay inside the rows (kk + PW <= ld) and that p0 + PW <= n; otherwise the masked path runs.
template <bool PAD8, int RB>
DG_DEV void ws_apply_panel(double* DG_RESTRICT y, int st, const double* DG_RESTRICT V, int ld, int p0, int pa, int n,
                           const double* DG_RESTRICT v0s, const double* DG_RESTRICT scs, const double* DG_RESTRICT gram) {
  constexpr int PW = DG_WS_PW;
  const int ph = PAD8 ? PW : pa;                   // rows of the panel's triangle handled apart
  double z[PW], w[PW];
#pragma unroll
  for (int q = 0; q < PW; ++q) z[q] = 0.0;
#pragma unroll
  for (int r = 0; r < PW; ++r) {
    if (PAD8 || r < pa) {
      const double yv = y[(p0 + r) * st];
      const double* DG_RESTRICT vr = V + (p0 + r) * ld;
#pragma unroll
      for (int q = 0; q < PW; ++q) if (q <= r) z[q] = fma(q == r ? v0s[q] : vr[q], yv, z[q]);
    }
  }
  {
    int j = p0 + ph;
    if (PAD8) {
      for (; j + RB <= n; j += RB) {
        double yv[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) yv[r] = y[(j + r) * st];
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          double a[PW];
          ws_load8(V + (j + r) * ld, a);
#pragma unroll
          for (int q = 0; q < PW; ++q) z[q] = fma(a[q], yv[r], z[q]);
        }
      }
    }
    for (; j < n; ++j) {
      const double y0 = y[j * st];
      double a[PW];
#pragma unroll
      for (int q = 0; q < PW; ++q) a[q] = (PAD8 || q < pa) ? V[j * ld + q] : 0.0;
#pragma unroll
      for (int q = 0; q < PW; ++q) z[q] = fma(a[q], y0, z[q]);
    }
  }
  // w = T' z: forward substitution with the Gram block (T^-1 = triu(V'V) with 1/sc on the diagonal)
#pragma unroll
  for (int q = 0; q < PW; ++q) {
    double a = z[q];
#pragma unroll
    for (int a2 = 0; a2 < PW; ++a2) if (a2 < q) a -= (q < pa ? gram[a2 * PW + q] : 0.0) * w[a2];
    w[q] = q < pa ? scs[q] * a : 0.0;
  }
#pragma unroll
  for (int r = 0; r < PW; ++r) {
    if (PAD8 || r < pa) {
      const double* DG_RESTRICT vr = V + (p0 + r) * ld;
      double yv = y[(p0 + r) * st];
#pragma unroll
      for (int q = 0; q < PW; ++q) if (q <= r) yv = fma(-(q == r ? v0s[q] : vr[q]), w[q], yv);
      y[(p0 + r) * st] = yv;
    }
  }
  {
    int j = p0 + ph;
    if (PAD8) {
      for (; j + RB <= n; j += RB) {
        double yv[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) yv[r] = y[(j + r) * st];
#pragma unroll
        for (int r = 0; r < RB; ++r) {
          double a[PW];
          ws_load8(V + (j + r) * ld, a);
          double s0 = 0.0, s1 = 0.0;               // two partial sums per row: shorter dependent chains
#pragma unroll
          for (int q = 0; q < PW; q += 2) { s0 = fma(a[q], w[q], s0); s1 = fma(a[q + 1], w[q + 1], s1); }
          yv[r] -= s0 + s1;
        }
#pragma unroll
        for (int r = 0; r < RB; ++r) y[(j + r) * st] = yv[r];
      }
    }
    for (; j < n; ++j) {
      double y0 = y[j * st];
      double a[PW];
#pragma unroll
      for (int q = 0; q < PW; ++q) a[q] = (PAD8 || q < pa) ? V[j * ld + q] : 0.0;
#pragma unroll
      for (int q = 0; q < PW; ++q) y0 = fma(-a[q], w[q], y0);
      y[j * st] = y0;
    }
  }
}

template <bool SM>
DG_DEVN int gi_warm_start(Cta& c, const Dims& D_, const EvalBuf& E_, const double* DG_RESTRICT qv, const QpBuf& Q_, const LinBuf& B_, int nprev) {
  const EvalBuf E = E_; DG_SH_EVAL(E); const QpBuf Q = Q_; DG_SH_QP(Q); const LinBuf B = B_; DG_SH_LIN(B); const Dims D = D_;
  const int n = D.n, ld = B.ld;
  constexpr int PW = DG_WS_PW, CW = DG_WS_CW;
  double* DG_RESTRICT Y = B.matB;
  double* DG_RESTRICT Rm = B.matA;
  int* DG_RESTRICT ids = (int*)Q.rv;               // [0, n): previous active ids, [n, 2n): source column of accepted column a
  int* DG_RESTRICT src = ids + n;
  int* DG_RESTRICT spr = (int*)Q.xq;               // [0, 2n): the <= 2 entries (input index << 1 | negative) of a sparse row, -1 = none; -2 = dense row
  double* DG_RESTRICT v0s = Q.lam_act + n;         // the two vectors of the 8n region that the QP does not use (plan_memory)
  double* DG_RESTRICT scs = Q.lam_act + 2 * n;
  double* DG_RESTRICT rt = Q.npv;
  double* DG_RESTRICT cv = Q.dv;                   // c = J'q: qp_factor left Y q here
  double* DG_RESTRICT gram = B.part;               // PW x PW
  int* DG_RESTRICT ctl = (int*)(B.part + PW * PW); // {accepted columns of the panel, panel ended at a dependent column}
  (void)qv;
  c.sync();
  DG_FOR(k, nprev) {
    const int p = Q.act[k];
    ids[k] = p; rt[k] = E.g[p];
    int t1, t2;
    if (!game_G_sparse(D, p, t1, t2)) t1 = t2 = -2;
    spr[2 * k] = t1; spr[2 * k + 1] = t2;
  }
  c.sync();
  // (1) rows of G side by side, then D = -Y G_W' in place.  Input-bound and rate rows have one or two entries +-1: a
  // chunk of columns that holds only such rows is gathered from the columns of Y instead.
  game_G_cols<SM>(c, D, E, ids, nprev, Rm, ld);
  c.sync();
  {
    const Split2 sp = split2(c, n);
    for (int c0 = 0; c0 < nprev; c0 += sp.G * CW) {
      const int cbase = c0 + sp.g * CW;
      const int cw = nprev - cbase < CW ? nprev - cbase : CW;
      bool dense = false;
      for (int q = 0; q < cw; ++q) dense = dense || spr[2 * (cbase + q)] == -2;
      for (int jb = ((n - 1) / sp.istep) * sp.istep; jb >= 0; jb -= sp.istep) {
        const int j = jb + sp.i0;
        const bool live = j < n && cw > 0 && sp.i0 < sp.istep;
        double acc[CW];
#pragma unroll
        for (int q = 0; q < CW; ++q) acc[q] = 0.0;
        if (live) {
          const double* DG_RESTRICT Yj = Y + j * ld;
          if (!dense) {
#pragma unroll
            for (int q = 0; q < CW; ++q) {
              if (q < cw) {
                const int t1 = spr[2 * (cbase + q)], t2 = spr[2 * (cbase + q) + 1];
                double a = 0.0;
                if (t1 >= 0 && (t1 >> 1) <= j) a = (t1 & 1) ? -Yj[t1 >> 1] : Yj[t1 >> 1];
                if (t2 >= 0 && (t2 >> 1) <= j) a += (t2 & 1) ? -Yj[t2 >> 1] : Yj[t2 >> 1];
                acc[q] = a;
              }
            }
          } else if (cw == CW) {
            int i = 0;
            for (; i + 1 <= j; i += 2) {
              const double y0 = Yj[i], y1 = Yj[i + 1];
              const double* DG_RESTRICT g0 = Rm + i * ld + cbase;
              const double* DG_RESTRICT g1 = g0 + ld;
              double a[CW], b[CW];
#pragma unroll
              for (int q = 0; q < CW; ++q) { a[q] = g0[q]; b[q] = g1[q]; }
#pragma unroll
              for (int q = 0; q < CW; ++q) acc[q] = fma(y0, a[q], acc[q]);
#pragma unroll
              for (int q = 0; q < CW; ++q) acc[q] = fma(y1, b[q], acc[q]);
            }
            if (i <= j) {
              const double y0 = Yj[i];
              const double* DG_RESTRICT g0 = Rm + i * ld + cbase;
#pragma unroll
              for (int q = 0; q < CW; ++q) acc[q] = fma(y0, g0[q], acc[q]);
            }
          } else {
            for (int i = 0; i <= j; ++i) {
              const double y0 = Yj[i];
              const double* DG_RESTRICT g0 = Rm + i * ld + cbase;
              double a[CW];
#pragma unroll
              for (int q = 0; q < CW; ++q) a[q] = q < cw ? g0[q] : 0.0;
#pragma unroll
              for (int q = 0; q < CW; ++q) acc[q] = fma(y0, a[q], acc[q]);
            }
          }
        }
        c.sync();                                  // every row <= j of these columns has been read
        if (live) {
#pragma unroll
          for (int q = 0; q < CW; ++q) if (q < cw) Rm[j * ld + cbase + q] = -acc[q];
        }
      }
    }
  }
  c.sync();
  c.lapf(PH_WS_D);
  // (2) blocked Householder QR; accepted column a (pivot row a) <- source column src[a].  Panel factorisation: warp t
  // owns column t of the panel (lanes along the rows); per reflector the scalars are formed by every thread, each warp
  // takes the product of the reflector with its column -- an update for the later columns, a Gram entry for the earlier
  // ones -- and the owner of the next column leaves its pivot-row norm: one barrier per reflector.
  double* DG_RESTRICT znb = B.part + PW * PW + 4;  // pivot-row norm of the panel column that is factored next
  double* DG_RESTRICT dallb = znb + PW;            // |column|^2 of the panel columns (orthogonal transformations keep it)
  int iq = 0, kk = 0;
  bool gaps = false;
  while (kk < nprev && iq < n) {
    const int pw = nprev - kk < PW ? nprev - kk : PW;
    for (int t = c.warp(); t < pw; t += c.nwarps()) {
      double da = 0.0, zn = 0.0;
      for (int j = c.lane(); j < n; j += c.wsz) { const double d = Rm[j * ld + kk + t]; da = fma(d, d, da); if (j >= iq) zn = fma(d, d, zn); }
      da = c.warp_sum(da);
      if (t == 0) zn = c.warp_sum(zn);
      if (c.lane() == 0) { dallb[t] = da; if (t == 0) znb[0] = zn; }
    }
    c.sync();
    int pa = 0, dep = 0;
    for (int q = 0; q < pw; ++q) {
      const int s = kk + q, p = iq + q;
      if (p >= n) { dep = 1; break; }
      const double zn = znb[q], dq = dallb[q];
      if (!(zn > DG_QP_DEP_TOL * dq && zn > 0.0)) { dep = 1; break; }     // linearly dependent on the accepted ones
      const double d0 = Rm[p * ld + s];
      double alpha = sqrt(zn);
      if (d0 > 0.0) alpha = -alpha;
      const double v0 = d0 - alpha;
      const double vv = 2.0 * (zn - alpha * d0);
      const double sc = vv > 0.0 ? 2.0 / vv : 0.0;
      for (int t = c.warp(); t < pw; t += c.nwarps()) {
        if (t == q) continue;
        double dot = 0.0;
        for (int j = p + c.lane(); j < n; j += c.wsz) {
          const double vj = j == p ? v0 : Rm[j * ld + s];
          dot = fma(vj, Rm[j * ld + kk + t], dot);
        }
        dot = c.warp_sum(dot);
        if (t < q) { if (c.lane() == 0) gram[t * PW + q] = dot; }
        else {
          const double wsc = dot * sc;
          double zn_next = 0.0;
          for (int j = p + c.lane(); j < n; j += c.wsz) {
            const double vj = j == p ? v0 : Rm[j * ld + s];
            const double nv = fma(-vj, wsc, Rm[j * ld + kk + t]);
            Rm[j * ld + kk + t] = nv;
            if (j > p) zn_next = fma(nv, nv, zn_next);
          }
          if (t == q + 1) { zn_next = c.warp_sum(zn_next); if (c.lane() == 0) znb[t] = zn_next; }
        }
      }
      c.sync();                                    // d0 and column s have been read; the updates and znb are visible
      if (c.tid() == 0) {
        Rm[p * ld + s] = alpha; v0s[p] = v0; scs[p] = sc;
        src[p] = s; Q.act[p] = ids[s]; Q.is_act[ids[s]] = 1;
      }
      ++pa;
    }
    c.sync();
    c.lapf(PH_WS_QR);
    const int knext = kk + pa + dep;
    if (pa > 0) {
      // block reflector on the columns of Y, the source columns behind the panel and c: thread per target column, the
      // three kinds of target on different warps.  The panel's own columns after a dependent one (knext .. kk + pw)
      // already carry the panel's reflectors (the in-panel updates above); a second application would undo them.
      const int kend = nprev - kk < PW ? nprev : kk + PW, p0 = iq, nrem = nprev - kend;      // kk + pw
      const int sD = (n + c.wsz - 1) / c.wsz * c.wsz, sC = sD + (nrem + c.wsz - 1) / c.wsz * c.wsz;
      const double* DG_RESTRICT V = Rm + kk;
      const bool pad8 = kk + PW <= ld && p0 + PW <= n;
      constexpr int RBY = SM ? 2 : 8;              // Y is streamed from L2 in the SM = false instantiation
      for (int slot = c.tid(); slot <= sC; slot += c.nt()) {
        if (pad8) {
          if (slot < n) ws_apply_panel<true, RBY>(Y + slot, ld, V, ld, p0, pa, n, v0s + p0, scs + p0, gram);
          else if (slot >= sD && slot - sD < nrem) ws_apply_panel<true, 2>(Rm + kend + (slot - sD), ld, V, ld, p0, pa, n, v0s + p0, scs + p0, gram);
          else if (slot == sC) ws_apply_panel<true, 2>(cv, 1, V, ld, p0, pa, n, v0s + p0, scs + p0, gram);
        } else {
          double* DG_RESTRICT tp = nullptr; int st = ld;
          if (slot < n) tp = Y + slot;
          else if (slot >= sD && slot - sD < nrem) tp = Rm + kend + (slot - sD);
          else if (slot == sC) { tp = cv; st = 1; }
          if (tp) ws_apply_panel<false, 2>(tp, st, V, ld, p0, pa, n, v0s + p0, scs + p0, gram);
        }
      }
      c.sync();
      c.lapf(PH_WS_APPLY);
    }
    if (dep) gaps = true;
    iq += pa; kk = knext;
  }
  if (iq == 0) return 0;
  if (gaps) {
    // close the gaps skipped columns left: accepted column a sits in source column src[a] >= a (ascending: a target
    // column is never the source of a later one)
    for (int a = 0; a < iq; ++a) {
      const int s = src[a];
      if (s != a) {
        DG_FOR(j, a + 1) Rm[j * ld + a] = Rm[j * ld + s];
        if (c.tid() == 0) rt[a] = rt[s];
        c.sync();
      }
    }
  }
#ifdef DG_WARM_STATS
  int ws_drops = 0;
#endif
  // (3)/(4) multipliers on the accepted set; drop negative ones.  Everything that touches R -- the two substitutions, the
  // search for the most negative multiplier, the Givens re-triangularisation of a drop (c and t = R^-T g_W rotate with
  // the rows of R, so the forward substitution runs once) -- stays on warp 0 without CTA barriers; the rotations are
  // recorded (Q.lam, free until the main loop) and every thread then applies the whole sequence to its own column of Y.
  double* DG_RESTRICT tv = Q.zv;                   // t = R^-T g_W
  double* DG_RESTRICT wk = Q.xq;                   // back-substitution work vector (the sparse-row table is dead)
  double* DG_RESTRICT rinv = B.part + 256;         // 1 / R_kk
  double* DG_RESTRICT rot = Q.lam;
  int* DG_RESTRICT drec = src;                     // (position, active count before the drop) per recorded drop
  const int rot_cap = D.m / 2, drop_cap = n / 2;
  bool first = true;
  while (true) {
    if (c.warp() == 0) {
      if (first) {
        for (int k = c.lane(); k < iq; k += c.wsz) { tv[k] = rt[k]; rinv[k] = 1.0 / Rm[k * ld + k]; }
        c.syncwarp();
        // forward substitution with R' (right-looking: row k of R is contiguous)
        for (int k = 0; k < iq; ++k) {
          const double tk = tv[k] * rinv[k];
          c.syncwarp();
          if (c.lane() == 0) tv[k] = tk;
          for (int j = k + 1 + c.lane(); j < iq; j += c.wsz) tv[j] -= Rm[k * ld + j] * tk;
          c.syncwarp();
        }
      }
      int nd = 0, nr = 0, more = 0;
      while (true) {
        // back substitution lam = R^-1 (t + c1) (column-oriented, like the main loop); lane k % wsz keeps lam_k
        for (int k = c.lane(); k < iq; k += c.wsz) wk[k] = tv[k] + cv[k];
        c.syncwarp();
        for (int k = iq - 1; k >= 0; --k) {
          const double lk = wk[k] * rinv[k];
          if (c.lane() == k % c.wsz) Q.lam_act[k] = lk;
          for (int j = c.lane(); j < k; j += c.wsz) wk[j] -= Rm[j * ld + k] * lk;
          c.syncwarp();
        }
        double bv = 0.0; int bk = 0x7fffffff;
        for (int k = c.lane(); k < iq; k += c.wsz) { const double lk = Q.lam_act[k]; if (lk < bv) { bv = lk; bk = k; } }
        c.warp_argmin(bv, bk);
        if (!(bv < 0.0)) break;
        const int ldrop = bk, len = iq - 1 - ldrop;
        if (nd >= drop_cap || nr + len > rot_cap) { more = 1; break; }   // record buffers full: apply to Y first
#ifdef DG_WARM_STATS
        ++ws_drops;
#endif
        // drop ldrop: shift the ids and the columns of R, re-triangularise with Givens rotations
        if (c.lane() == 0) { drec[2 * nd] = ldrop; drec[2 * nd + 1] = iq; Q.is_act[Q.act[ldrop]] = 0; }
        for (int k0 = ldrop; k0 < iq - 1; k0 += c.wsz) {
          const int k = k0 + c.lane();
          const int v = k < iq - 1 ? Q.act[k + 1] : 0;
          c.syncwarp();
          if (k < iq - 1) Q.act[k] = v;
        }
        for (int i = c.lane(); i < iq; i += c.wsz) {
          for (int j = ldrop; j < iq - 1; ++j) Rm[i * ld + j] = Rm[i * ld + j + 1];
          Rm[i * ld + iq - 1] = 0.0;
        }
        c.syncwarp();
        for (int j = ldrop; j < iq - 1; ++j) {
          const double a = Rm[j * ld + j], b = Rm[(j + 1) * ld + j];
          const double h = hypot(a, b);
          double cs = 1.0, sn = 0.0;
          if (h != 0.0) { cs = a / h; sn = b / h; }
          c.syncwarp();                         // a, b read by every lane before the rows change
          if (h != 0.0) {
            for (int col = j + c.lane(); col < iq - 1; col += c.wsz) {
              const double r0 = Rm[j * ld + col], r1 = Rm[(j + 1) * ld + col];
              Rm[j * ld + col] = cs * r0 + sn * r1;
              Rm[(j + 1) * ld + col] = -sn * r0 + cs * r1;
            }
          }
          if (c.lane() == 0) {
            rot[2 * (nr + j - ldrop)] = cs; rot[2 * (nr + j - ldrop) + 1] = sn;
            const double c0 = cv[j], c1 = cv[j + 1];
            cv[j] = cs * c0 + sn * c1; cv[j + 1] = -sn * c0 + cs * c1;
            const double t0 = tv[j], t1 = tv[j + 1];
            tv[j] = cs * t0 + sn * t1; tv[j + 1] = -sn * t0 + cs * t1;
          }
          c.syncwarp();
        }
        for (int k = ldrop + c.lane(); k < iq - 1; k += c.wsz) rinv[k] = 1.0 / Rm[k * ld + k];
        c.syncwarp();
        nr += len; ++nd; --iq;
        if (iq == 0) break;
      }
      if (c.lane() == 0) { ctl[0] = iq; ctl[1] = nd; ctl[2] = more; }
    }
    c.sync();
    iq = ctl[0];
    const int nd = ctl[1], more = ctl[2];
    if (nd > 0) {
      // the recorded rotations on the rows of Y: thread per column, the loads of a step ahead of its dependent chain
      DG_FOR(i, n) {
        int rb = 0;
        for (int d = 0; d < nd; ++d) {
          const int ldrop = drec[2 * d], last = drec[2 * d + 1] - 1;
          const double* DG_RESTRICT rr = rot + 2 * (rb - ldrop);
          double t = Y[ldrop * ld + i];
          int j = ldrop;
          for (; j + 3 < last; j += 4) {
            const double u0 = Y[(j + 1) * ld + i], u1 = Y[(j + 2) * ld + i], u2 = Y[(j + 3) * ld + i], u3 = Y[(j + 4) * ld + i];
            const double c0 = rr[2 * j], s0 = rr[2 * j + 1], c1 = rr[2 * j + 2], s1 = rr[2 * j + 3];
            const double c2 = rr[2 * j + 4], s2 = rr[2 * j + 5], c3 = rr[2 * j + 6], s3 = rr[2 * j + 7];
            Y[j * ld + i] = c0 * t + s0 * u0; t = -s0 * t + c0 * u0;
            Y[(j + 1) * ld + i] = c1 * t + s1 * u1; t = -s1 * t + c1 * u1;
            Y[(j + 2) * ld + i] = c2 * t + s2 * u2; t = -s2 * t + c2 * u2;
            Y[(j + 3) * ld + i] = c3 * t + s3 * u3; t = -s3 * t + c3 * u3;
          }
          for (; j < last; ++j) {
            const double cs = rr[2 * j], sn = rr[2 * j + 1];
            const double u1 = Y[(j + 1) * ld + i];
            Y[j * ld + i] = cs * t + sn * u1; t = -sn * t + cs * u1;
          }
          Y[last * ld + i] = t;
          rb += last - ldrop;
        }
      }
      c.sync();
    }
    if (!more) break;
    first = false;
  }
  // x = J1 t - J2 c2 = Y' [t; -c2]
  c.sync();
  c.lapf(PH_WS_MULT);
  for (int j = iq + c.tid(); j < n; j += c.nt()) tv[j] = -cv[j];
  c.sync();
  gi_cols_times<SM>(c, n, ld, Y, tv, 0, B.part, Q.xq, 1.0);
#ifdef DG_WARM_STATS
  fprintf(stderr, "WS nprev %d iq_end %d drops %d\n", nprev, iq, ws_drops);
#endif
  return iq;
}

// Cholesky of H (in B.matA, destroyed), Y = L^-1 into B.matB, unconstrained minimiser into Q.xq, empty active set.
// Returns false (uniformly) when H is not positive definite.
template <bool SM>
DG_DEVN bool qp_factor(Cta& c, const Dims& D_, const double* DG_RESTRICT qv, const QpBuf& Q_, const LinBuf& B_) {
  // local copies: the tables live in shared memory and would otherwise be re-read after every store
  const QpBuf Q = Q_; DG_SH_QP(Q); const LinBuf B = B_; DG_SH_LIN(B); const Dims D = D_;
  const int n = D.n, m = D.m, ld = B.ld;
  double* DG_RESTRICT Y = B.matB;
  {
    bool ok = false;
#ifndef DG_HOSTSIM
    if (c.nt() == 256 && n > 128 && n <= 256) {
      // larger games (3-4 agents): the blocked panels until at most 128 columns remain, then the register tiles on the
      // trailing block (its lower triangle is what the panels leave updated)
      const int base = (n - 128 + DG_CHOL_NB - 1) / DG_CHOL_NB * DG_CHOL_NB;
      ok = cholesky_lower<SM>(c, n, ld, B.matA, B.sp, B.part, base);
      if (ok) {
        c.sync();
        LinBuf Bt = B;
        Bt.matA = B.matA + (size_t)base * ld + base;
        ok = cholesky_tiles<8, SM>(c, n - base, Bt, true);
      }
    } else if (!cholesky_tiles_dispatch<SM>(c, n, B, ok))
#endif
    ok = cholesky_lower<SM>(c, n, ld, B.matA, B.sp, B.part, n);
    if (!ok) return false;
  }
  c.lap(PH_CHOL);
#ifndef DG_HOSTSIM
  if (!tri_inverse_tiles_dispatch<SM>(c, n, B))
#endif
  tri_inverse<SM>(c, n, ld, B.matA, Y, B.sp, B.part);
  c.sync();
  c.lapf(PH_TRINV);
  // x = -J J' q = -Y' (Y q):   t = Y q (warp per row), x_i = -sum_j Y[j][i] t_j
  for (int j = c.warp(); j < n; j += c.nwarps()) {
    const double* DG_RESTRICT Yj = Y + j * ld;
    double p = 0.0;
    for (int i = c.lane(); i <= j; i += c.wsz) p += Yj[i] * qv[i];
    p = c.warp_sum(p);
    if (c.lane() == 0) Q.dv[j] = p;
  }
  DG_FOR(r, m) Q.is_act[r] = 0;
  c.sync();
  gi_cols_times<SM>(c, n, ld, Y, Q.dv, 0, B.part, Q.xq, -1.0);
  c.lap2(PH_TRINV, PH_QP_X0);
  return true;
}

// The dual active-set iteration from the S-pair (Q.xq, Q.act[0..iq0), Q.lam_act) with factors Y = J' (B.matB) and R (B.matA).
// returns 0 ok, 2 infeasible, 3 iteration limit.  Output: Q.xq (du), Q.lam (l_hat).
template <bool SM>
DG_DEVN int qp_gi_loop(Cta& c, const Dims& D_, const EvalBuf& E_, const QpBuf& Q_, const LinBuf& B_, int iq0,
                       int* n_iter_out, int* n_active_out) {
  // local copies: the tables live in shared memory and would otherwise be re-read after every store
  const EvalBuf E = E_; DG_SH_EVAL(E); const QpBuf Q = Q_; DG_SH_QP(Q); const LinBuf B = B_; DG_SH_LIN(B); const Dims D = D_;
  const int n = D.n, m = D.m, ld = B.ld;
  double* DG_RESTRICT Y = B.matB;
  double* DG_RESTRICT Rm = B.matA;
  DG_FOR(r, m) Q.lam[r] = 0.0;
  int iq = iq0, it = 0;
  const int max_iter = 10 * (n + m);
  const Split2 sp = split2(c, n);                 // one decomposition for every n-wide sweep of the loop (integer divisions)
  int status = 0;
  while (true) {
    // slacks of all constraints, most violated one
    game_G_times<SM>(c, D, E, Q.xq, Q.sl);
    double best; int bi;
    {
      double bv = 1e300; int bidx = 0x7fffffff;
      DG_FOR(r, m) {
        double sv = Q.is_act[r] ? 0.0 : -E.g[r] - Q.sl[r];
        if (sv < bv) { bv = sv; bidx = r; }
      }
      c.argmin(bv, bidx, best, bi);
    }
    if (!(best < -DG_QP_FEAS_TOL)) break;
    const int p = bi;
    game_G_row<SM>(c, D, E, p, Q.npv);                 // npv = G[p,:]  (normal is -npv)
    c.lapf(PH_GI_SLACK);
    double lam_p = 0.0;
    bool added = false;
    while (!added) {
      if (++it > max_iter) { status = 3; break; }
      // d = J' n_p = -Y npv   (2D over the CTA: thread = row of Y, column groups interleave the columns);  also npv . x
      double dd_tail = 0.0, dd_all = 0.0, gx = 0.0;
      if constexpr (!SM) {
        // Y in the L2-resident workspace: the sweep is bound by L2 latency, so every lane keeps 16 loads in flight --
        // a warp takes four rows at a time, lanes along the rows (coalesced), 128 columns per pass, all loads issued
        // before the first use
        for (int j0 = 4 * c.warp(); j0 < n; j0 += 4 * c.nwarps()) {
          double acc[4] = {0.0, 0.0, 0.0, 0.0};
          for (int i0 = 0; i0 < n; i0 += 4 * c.wsz) {
            double y[4][4], v[4];
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const int i = i0 + c.lane() + u * c.wsz;
                y[r][u] = (i < n && j0 + r < n) ? Y[(j0 + r) * ld + i] : 0.0;
              }
#pragma unroll
            for (int u = 0; u < 4; ++u) { const int i = i0 + c.lane() + u * c.wsz; v[u] = i < n ? Q.npv[i] : 0.0; }
#pragma unroll
            for (int r = 0; r < 4; ++r) acc[r] += (y[r][0] * v[0] + y[r][1] * v[1]) + (y[r][2] * v[2] + y[r][3] * v[3]);
          }
#pragma unroll
          for (int r = 0; r < 4; ++r) {
            double a = c.warp_sum(acc[r]);
            if (c.lane() == 0 && j0 + r < n) {
              a = -a;
              Q.dv[j0 + r] = a;
              dd_all += a * a;
              if (j0 + r >= iq) dd_tail += a * a;
            }
          }
        }
      } else {
        for (int j = sp.i0; j < n; j += sp.istep) {
          const double* DG_RESTRICT Yj = Y + j * ld;
          double a0 = 0.0, a1 = 0.0;
          int i = sp.g;
          for (; i + sp.G < n; i += 2 * sp.G) { a0 += Yj[i] * Q.npv[i]; a1 += Yj[i + sp.G] * Q.npv[i + sp.G]; }
          if (i < n) a0 += Yj[i] * Q.npv[i];
          B.part[sp.g * sp.istep + j] = a0 + a1;
        }
        c.sync();
        if (sp.g == 0) {
          for (int j = sp.i0; j < n; j += sp.istep) {
            double acc = B.part[j];
            for (int g = 1; g < sp.G; ++g) acc += B.part[g * sp.istep + j];
            acc = -acc;
            Q.dv[j] = acc;
            dd_all += acc * acc;
            if (j >= iq) dd_tail += acc * acc;
          }
        }
      }
      DG_FOR(i, n) gx += Q.npv[i] * Q.xq[i];
      c.sum3(dd_tail, dd_all, gx);
      const double zn = dd_tail, dall = dd_all;
      // z = J[:, iq:] d[iq:]  (2D over the CTA);  r = R^-1 d[:iq]  (column-oriented back substitution on the last warp,
      // while the first column group combines the partial sums of z)
      {
        for (int i = sp.i0; i < n; i += sp.istep) {
          double a0 = 0.0, a1 = 0.0;
          int j = iq + sp.g;
          if constexpr (!SM) {
            // L2-resident Y: eight loads in flight per thread
            double a2 = 0.0, a3 = 0.0;
            for (; j + 7 * sp.G < n; j += 8 * sp.G) {
              double y[8];
#pragma unroll
              for (int u = 0; u < 8; ++u) y[u] = Y[(j + u * sp.G) * ld + i];
              a0 += y[0] * Q.dv[j] + y[4] * Q.dv[j + 4 * sp.G]; a1 += y[1] * Q.dv[j + sp.G] + y[5] * Q.dv[j + 5 * sp.G];
              a2 += y[2] * Q.dv[j + 2 * sp.G] + y[6] * Q.dv[j + 6 * sp.G]; a3 += y[3] * Q.dv[j + 3 * sp.G] + y[7] * Q.dv[j + 7 * sp.G];
            }
            for (; j + 3 * sp.G < n; j += 4 * sp.G) {
              const double y0 = Y[j * ld + i], y1 = Y[(j + sp.G) * ld + i], y2 = Y[(j + 2 * sp.G) * ld + i], y3 = Y[(j + 3 * sp.G) * ld + i];
              a0 += y0 * Q.dv[j]; a1 += y1 * Q.dv[j + sp.G]; a2 += y2 * Q.dv[j + 2 * sp.G]; a3 += y3 * Q.dv[j + 3 * sp.G];
            }
            a0 += a2; a1 += a3;
          }
          for (; j + sp.G < n; j += 2 * sp.G) { a0 += Y[j * ld + i] * Q.dv[j]; a1 += Y[(j + sp.G) * ld + i] * Q.dv[j + sp.G]; }
          if (j < n) a0 += Y[j * ld + i] * Q.dv[j];
          if (sp.G == 1) Q.zv[i] = a0 + a1;
          else B.part[sp.g * sp.istep + i] = a0 + a1;
        }
        if (sp.G > 1) {
          c.sync();
          if (sp.g == 0) {
            for (int i = sp.i0; i < n; i += sp.istep) {
              double acc = B.part[i];
              for (int g = 1; g < sp.G; ++g) acc += B.part[g * sp.istep + i];
              Q.zv[i] = acc;
            }
          }
        }
        if (c.warp() == c.nwarps() - 1) {
          // reciprocal pivots first (independent divisions), so that the serial chain below only multiplies;
          // they are parked in the tail of zv's partial-sum scratch (part[256..], beyond the G*cw <= 256 partial sums)
          double* DG_RESTRICT rinv = B.part + 256;
          for (int i = c.lane(); i < iq; i += c.wsz) { Q.rv[i] = Q.dv[i]; rinv[i] = 1.0 / Rm[i * ld + i]; }
          c.syncwarp();
          for (int i = iq - 1; i >= 0; --i) {
            const double ri = Q.rv[i] * rinv[i];
            c.syncwarp();
            if (c.lane() == 0) Q.rv[i] = ri;
            for (int j = c.lane(); j < i; j += c.wsz) Q.rv[j] -= Rm[j * ld + i] * ri;
            c.syncwarp();
          }
        }
      }
      c.sync();
      c.lapf(PH_GI_DZ);
      // dual step bound t1, primal step length t2
      double t1 = 1e300; int ldrop = -1;
      {
        double bv = 1e300; int bk = 0x7fffffff;
        DG_FOR(k, iq) {
          const double rk = Q.rv[k];
          if (rk > 0.0) { const double tk = Q.lam_act[k] / rk; if (tk < bv) { bv = tk; bk = k; } }
        }
        if (iq > 0) { c.argmin(bv, bk, t1, ldrop); if (!(t1 < 1e300)) ldrop = -1; }
      }
      double t2 = 1e300;
      if (zn > DG_QP_DEP_TOL * dall && zn > 0.0) t2 = (E.g[p] + gx) / zn;      // -s_p / |d2|^2
      const double t = t1 < t2 ? t1 : t2;
      if (t >= 1e300) { status = 2; break; }
      c.sync();                                   // rv / lam_act read by everyone before they change
      if (t2 < 1e300) { DG_FOR(i, n) Q.xq[i] += t * Q.zv[i]; }
      DG_FOR(k, iq) Q.lam_act[k] -= t * Q.rv[k];
      lam_p += t;
      c.lapf(PH_GI_STEP);
      if (t2 <= t1) {
        // full step: add p.  Householder P on d[iq:] -> (alpha, 0, ..); J[:, iq:] <- J[:, iq:] P, and
        // J2 v = z - alpha J[:, iq] needs no extra product.
        const int len = n - iq;
        const double d0 = Q.dv[iq];
        double alpha = sqrt(zn);
        if (d0 > 0.0) alpha = -alpha;
        const double vv = 2.0 * (zn - alpha * d0);
        if (vv > 0.0) {
          const double sc = 2.0 / vv;
          // w = (J2 v) * 2/(v'v) into npv (the entering row is not needed any more)
          DG_FOR(i, n) Q.npv[i] = (Q.zv[i] - alpha * Y[iq * ld + i]) * sc;
          c.sync();
          for (int i = sp.i0; i < n; i += sp.istep) {
            const double wi = Q.npv[i];
            double* DG_RESTRICT col = Y + iq * ld + i;
            int j = sp.g;
            if constexpr (!SM) {
              // L2-resident Y: eight independent read-modify-writes per step
              for (; j + 7 * sp.G < len; j += 8 * sp.G) {
                double y[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) y[u] = col[(j + u * sp.G) * ld];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                  const int jj = j + u * sp.G;
                  col[jj * ld] = y[u] - (jj == 0 ? d0 - alpha : Q.dv[iq + jj]) * wi;
                }
              }
            }
            for (; j < len; j += sp.G) col[j * ld] -= (j == 0 ? d0 - alpha : Q.dv[iq + j]) * wi;
          }
        }
        DG_FOR(i, iq) Rm[i * ld + iq] = Q.dv[i];
        if (c.tid() == 0) {
          Rm[iq * ld + iq] = alpha;
          Q.act[iq] = p; Q.is_act[p] = 1; Q.lam_act[iq] = lam_p;
        }
        ++iq;
        added = true;
        c.sync();
        c.lapf(PH_GI_ADD);
      } else {
        c.sync();
        // partial step: drop active constraint ldrop (Givens re-triangularisation), keep p
        if (c.tid() == 0) {
          Q.is_act[Q.act[ldrop]] = 0;
          for (int k = ldrop; k < iq - 1; ++k) { Q.act[k] = Q.act[k + 1]; Q.lam_act[k] = Q.lam_act[k + 1]; }
        }
        DG_FOR(i, iq) {
          for (int j = ldrop; j < iq - 1; ++j) Rm[i * ld + j] = Rm[i * ld + j + 1];
          Rm[i * ld + iq - 1] = 0.0;
        }
        c.sync();
        if (ldrop < iq - 1) {
          // Givens re-triangularisation.  The rotations form a serial chain only through R: one warp computes them and
          // rotates R (lanes along the columns), parking (cs, sn) in the partial-sum scratch; then every thread applies
          // the whole sequence to its own column of J (= column of the rows ldrop..iq-1 of Y) in registers -- two
          // barriers per drop instead of two per rotation.  Same arithmetic, same order as rotating row pairs one by one.
          double* DG_RESTRICT rot = B.part;
          if (c.warp() == 0) {
            for (int j = ldrop; j < iq - 1; ++j) {
              const double a = Rm[j * ld + j], b = Rm[(j + 1) * ld + j];
              const double h = hypot(a, b);
              double cs = 1.0, sn = 0.0;
              if (h != 0.0) { cs = a / h; sn = b / h; }
              c.syncwarp();                         // a, b read by every lane before the rows change
              if (h != 0.0) {
                for (int col = j + c.lane(); col < iq - 1; col += c.wsz) {
                  double r0 = Rm[j * ld + col], r1 = Rm[(j + 1) * ld + col];
                  Rm[j * ld + col] = cs * r0 + sn * r1;
                  Rm[(j + 1) * ld + col] = -sn * r0 + cs * r1;
                }
              }
              if (c.lane() == 0) { rot[2 * (j - ldrop)] = cs; rot[2 * (j - ldrop) + 1] = sn; }
              c.syncwarp();
            }
          }
          c.sync();
          DG_FOR(i, n) {
            double t = Y[ldrop * ld + i];
            for (int j = ldrop; j < iq - 1; ++j) {
              const double cs = rot[2 * (j - ldrop)], sn = rot[2 * (j - ldrop) + 1];
              const double u1 = Y[(j + 1) * ld + i];
              if (cs == 1.0 && sn == 0.0) { Y[j * ld + i] = t; t = u1; }      // h == 0: no rotation
              else { Y[j * ld + i] = cs * t + sn * u1; t = -sn * t + cs * u1; }
            }
            Y[(iq - 1) * ld + i] = t;
          }
          c.sync();
        }
        --iq;
        c.lapf(PH_GI_DROP);
      }
    }
    if (status != 0) break;
  }
  if (status == 0) {
    c.sync();
    DG_FOR(k, iq) Q.lam[Q.act[k]] = Q.lam_act[k];
    c.sync();
  }
  if (c.tid() == 0) Q.act[n] = status == 0 ? iq : 0;               // remembered for a warm start of the next QP
  if (n_iter_out) *n_iter_out = it;
  if (n_active_out) *n_active_out = iq;
  c.lap(PH_GI);
  return status;
}

// Polish: the KKT point of the final active set W re-evaluated from the final factors without the cancellation the
// iteration carries.  The method starts at the unconstrained minimiser x0 = -H^-1 q and moves by x += t z; when H is
// ill-conditioned (reg = 0 games: eigenvalues at the 1e-10 floor, condition 1e11) x0 is ~1e10 |q| along the near-null
// directions and the steps cancel it, which leaves errors of 1e-5..1e-3 in x and 1e-2 in lam.  With J = [J1 J2], J'N = [R; 0]
// (N = -G_W') and c = J'q the same point is
//     x = J1 R^-T g_W - J2 c2,        lam_W = R^-1 (R^-T g_W + c1)
// in which the large components c1 never meet (measured against an extended-precision KKT solve on the merge game: 1e-10
// in x, 1e-8 in lam).  This is the role OSQP's polish step has in the reference (DGSQP.py:186, polish=True: reduced KKT
// system of the active set + iterative refinement); the oracle applies the same formula (oracle/qp.py).
template <bool SM>
DG_DEVN void gi_polish(Cta& c, const Dims& D_, const EvalBuf& E_, const double* DG_RESTRICT qv, const QpBuf& Q_, const LinBuf& B_, int iq) {
  const EvalBuf E = E_; DG_SH_EVAL(E); const QpBuf Q = Q_; DG_SH_QP(Q); const LinBuf B = B_; DG_SH_LIN(B); const Dims D = D_;
  const int n = D.n, ld = B.ld;
  double* DG_RESTRICT Y = B.matB;
  double* DG_RESTRICT Rm = B.matA;
  c.sync();
  // c = J' q = Y q into Q.dv
  if constexpr (!SM) {
    for (int j = c.warp(); j < n; j += c.nwarps()) {
      double acc = 0.0;
      for (int i = c.lane(); i < n; i += c.wsz) acc += Y[j * ld + i] * qv[i];
      acc = c.warp_sum(acc);
      if (c.lane() == 0) Q.dv[j] = acc;
    }
    c.sync();
  } else {
    const Split2 sp = split2(c, n);
    for (int j = sp.i0; j < n; j += sp.istep) {
      const double* DG_RESTRICT Yj = Y + j * ld;
      double a0 = 0.0, a1 = 0.0;
      int i = sp.g;
      for (; i + sp.G < n; i += 2 * sp.G) { a0 += Yj[i] * qv[i]; a1 += Yj[i + sp.G] * qv[i + sp.G]; }
      if (i < n) a0 += Yj[i] * qv[i];
      B.part[sp.g * sp.istep + j] = a0 + a1;
    }
    c.sync();
    if (sp.g == 0) {
      for (int j = sp.i0; j < n; j += sp.istep) {
        double acc = B.part[j];
        for (int g = 1; g < sp.G; ++g) acc += B.part[g * sp.istep + j];
        Q.dv[j] = acc;
      }
    }
    c.sync();
  }
  // w = [R^-T g_W ; -c2] into Q.zv,  lam_W = R^-1 (w1 + c1) into Q.lam_act
  if (c.warp() == 0) {
    double* DG_RESTRICT tv = Q.zv;
    double* DG_RESTRICT rinv = B.part + 256;
    for (int k = c.lane(); k < iq; k += c.wsz) { tv[k] = E.g[Q.act[k]]; rinv[k] = 1.0 / Rm[k * ld + k]; }
    c.syncwarp();
    for (int k = 0; k < iq; ++k) {
      const double tk = tv[k] * rinv[k];
      c.syncwarp();
      if (c.lane() == 0) tv[k] = tk;
      for (int j = k + 1 + c.lane(); j < iq; j += c.wsz) tv[j] -= Rm[k * ld + j] * tk;
      c.syncwarp();
    }
    for (int k = c.lane(); k < iq; k += c.wsz) Q.lam_act[k] = tv[k] + Q.dv[k];
    c.syncwarp();
    for (int k = iq - 1; k >= 0; --k) {
      const double lk = Q.lam_act[k] * rinv[k];
      c.syncwarp();
      if (c.lane() == 0) Q.lam_act[k] = lk;
      for (int j = c.lane(); j < k; j += c.wsz) Q.lam_act[j] -= Rm[j * ld + k] * lk;
      c.syncwarp();
    }
  } else {
    for (int j = iq + c.tid() - c.wsz; j < n; j += c.nt() - c.wsz) Q.zv[j] = -Q.dv[j];
  }
  if (c.nt() <= c.wsz) { for (int j = iq; j < n; ++j) Q.zv[j] = -Q.dv[j]; }     // one-warp (and host) builds: warp 0 does both
  c.sync();
  gi_cols_times<SM>(c, n, ld, Y, Q.zv, 0, B.part, Q.xq, 1.0);
  DG_FOR(k, iq) Q.lam[Q.act[k]] = Q.lam_act[k];
  c.sync();
}

// _solve_qp's solver call.  H (symmetric positive definite) is expected in B.matA and is destroyed.
// warm != 0: start from the active set of the previous QP of this instance (ids in Q.act[0..), count parked in Q.act[n];
// the SQP drivers reset the count at the start of an instance).
// returns 0 ok, 1 not PD, 2 infeasible, 3 iteration limit.  Output: Q.xq (du), Q.lam (l_hat).
template <bool SM>
DG_DEV int qp_solve_gi(Cta& c, const Dims& D, const EvalBuf& E, const double* qv, const QpBuf& Q, const LinBuf& B,
                       int* n_iter_out, int* n_active_out, int warm) {
  if (!qp_factor<SM>(c, D, qv, Q, B)) return 1;
  int iq = 0;
  if (warm) {
    const int nprev = Q.act[D.n];
    if (nprev > 0 && nprev <= D.n) { iq = gi_warm_start<SM>(c, D, E, qv, Q, B, nprev); c.lapf(PH_QP_WARM); }
  }
  int na = 0;
  const int st = qp_gi_loop<SM>(c, D, E, Q, B, iq, n_iter_out, &na);
  if (n_active_out) *n_active_out = na;
#ifdef DG_WARM_STATS
  fprintf(stderr, "GI iq0 %d iters %d na %d st %d\n", iq, n_iter_out ? *n_iter_out : -1, na, st);
#endif
  if (st == 0) { gi_polish<SM>(c, D, E, qv, Q, B, na); c.lap(PH_GI); }
  return st;
}
