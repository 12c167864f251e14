// CTA-cooperative dense FP64 kernels for one n x n problem (n ~ 100-200), row-major storage.
//
// nearest_pd() replaces DGSQP._nearestPD (DGSQP/solvers/DGSQP.py:1290-1296: B=(A+A')/2; eigh;
// negative eigenvalues -> floor; U diag(s) U'; re-symmetrise).  Only the negative part of the
// spectrum changes, so   nearestPD(A) = B + sum_{s_i<0} (floor - s_i) u_i u_i'   and only the
// negative eigenpairs are needed: Householder tridiagonalisation, Sturm-count multisection for the
// negative eigenvalues, inverse iteration on the tridiagonal matrix, back-transformation.  When the
// Sturm count at 0 is zero the projection is the identity and the whole eigen-solve is skipped.
//
// Performance notes (B200): these routines are latency bound (n ~ 100 wide, ~n dependent steps), so
// they are written to (1) keep every global access coalesced across the CTA (thread = column),
// (2) expose instruction-level parallelism in the per-thread loops (explicit 4-way unrolling on
// __restrict__ pointers: read-modify-write loops otherwise serialise on possible aliasing), and
// (3) spend as few CTA barriers as possible (fused reductions, blocked Cholesky with the panel in
// shared memory, warp-private back-transformation).
#pragma once
#include "cta.cuh"

#define DG_EIG_CHUNK 16     // eigenvectors computed concurrently by inverse iteration
#ifndef DG_EIG_INVIT
#define DG_EIG_INVIT 2      // inverse-iteration sweeps per eigenvector (shifts are accurate to ~1 ulp of |T|: H agrees with
                            // eigh to 3e-15 relative with 2 as with 3 sweeps, 1.4e-14 with one; tests/test_kernel_source_host.py)
#endif
#define DG_EIG_SMALL 2       // eigenvectors whose inverse-iteration scratch fits the small shared-memory block LinBuf::eig_s
                            // (merge game: 11.5 KB beside the 212 KB of the split placement)
#define DG_CHOL_NB 8        // Cholesky panel width
#ifndef DG_MAX_THREADS
#define DG_MAX_THREADS 256
#endif
#define DG_PART_SZ 512      // doubles in LinBuf::part

struct LinBuf {
  int ld;         // leading dimension of matA / matB
  double* matA;   // n*ld  tridiagonalisation workspace W (reflectors) -> H = nearestPD + reg I -> Cholesky factor L
  double* matB;   // n*ld  inverse-iteration scratch + eigenvectors (during nearest_pd) -> J' of the QP (qp_gi.cuh)
  double* Zg;     // n*n   global spill for the eigenvectors when they do not fit beside the scratch in matB
  // phase-aliased small vectors (one region of 8n doubles, see plan_memory)
  double* dg;     // n     tridiagonal diagonal
  double* od;     // n     off-diagonal (od[k] couples k, k+1)
  double* od2;    // n     od^2
  double* tau;    // n
  double* lam;    // n     negative eigenvalues (ascending)
  double* pv;     // n
  double* wv;     // n
  double* sp;     // n*DG_CHOL_NB  Cholesky panel (aliases the seven vectors above)
  double* part;   // max(DG_PART_SZ, 2n)  partial sums of the 2D-decomposed products, scratch vectors
  double* eig_s;  // 6*n*DG_EIG_SMALL or null: shared-memory scratch of the inverse iteration when matB lives in the L2 workspace
};

#ifdef DG_NO_SH_LIN
#define DG_SH_LIN(B) do { } while (0)
#else
#define DG_SH_LIN(B) do { DG_ASSUME_SHARED((B).matA); DG_ASSUME_SHARED((B).matB); DG_ASSUME_SHARED((B).dg); DG_ASSUME_SHARED((B).od); \
  DG_ASSUME_SHARED((B).od2); DG_ASSUME_SHARED((B).tau); DG_ASSUME_SHARED((B).lam); DG_ASSUME_SHARED((B).pv); DG_ASSUME_SHARED((B).wv); \
  DG_ASSUME_SHARED((B).sp); DG_ASSUME_SHARED((B).part); } while (0)
#endif

#ifdef DG_NO_SH_T
#define DG_SH_LIN_T(B) do { } while (0)
#else
#define DG_SH_LIN_T(B) DG_SH_LIN(B)
#endif
#define DG_SH_LIN_P(B) DG_SH_LIN(B)

// Householder reduction of the symmetric matrix W = B.matA (full storage, both triangles kept consistent)
// to tridiagonal form; reflector k is stored in W[k+2.., k] (v[0] = 1 implicit) with tau[k].
// Both O(len^2) parts of a step -- p = tau A22 v and A22 -= v w' + w v' -- are spread over the whole CTA with the 2D
// decomposition (thread = column, column groups interleave the rows).  Four barriers per step.
// kstop < n - 1: only the steps k < kstop are taken (dg, od, tau, reflectors of those columns; the trailing matrix is left
// updated in W for a register-resident continuation, see nearest_pd).
template <bool SM>
DG_DEVN void sym_tridiag(Cta& c, int n, const LinBuf& B_, int kstop) {
  // local copies: the tables live in shared memory and would otherwise be re-read after every store
  const LinBuf B = B_; DG_SH_LIN_T(B);
  double* DG_RESTRICT W = B.matA;
  const int ld = B.ld;
  double* DG_RESTRICT pv = B.pv;
  double* DG_RESTRICT wv = B.wv;
  double* DG_RESTRICT part = B.part;
  // norm of the first column below the sub-diagonal
  double nrm = 0.0;
  for (int i = c.tid() + 2; i < n; i += c.nt()) { double xv = W[i * ld]; nrm += xv * xv; }
  double xn2 = c.sum(nrm);
  for (int k = 0; k + 1 < n && k < kstop; ++k) {
    const int len = n - k - 1;            // x = W[k+1.., k]
    const int off = k + 1;
    const double alpha = W[off * ld + k];
    double tauk = 0.0, beta = alpha, scale = 0.0;
    if (xn2 > 0.0) {
      beta = -copysign(sqrt(alpha * alpha + xn2), alpha);
      tauk = (beta - alpha) / beta;
      scale = 1.0 / (alpha - beta);
    }
    if (c.tid() == 0) { B.dg[k] = W[k * ld + k]; B.od[k] = beta; B.od2[k] = beta * beta; B.tau[k] = tauk; }
    if (tauk == 0.0) {
      // nothing to annihilate: next column norm straight from memory
      nrm = 0.0;
      for (int i = c.tid() + 2; i < len; i += c.nt()) { double xv = W[(off + i) * ld + off]; nrm += xv * xv; }
      xn2 = c.sum(nrm);
      continue;
    }
    const Split2 sp = split2(c, len);
    const double* DG_RESTRICT vc = W + off * ld + k;            // x_j = vc[j*ld]
    if constexpr (!SM) {
      // W may live in the L2-resident workspace: the column goes through shared memory once (pv is free until v is formed)
      DG_FOR(i, len) pv[i] = vc[i * ld];
      c.sync();
    }
    // partial products  sum_{j>=1, j = g (mod G)} A22[j][i] x_j   (the j = 0 term has v_0 = 1 and no scale)
    for (int i = sp.i0; i < len; i += sp.istep) {
      const double* DG_RESTRICT col = W + off * ld + off + i;
      double a0 = 0.0, a1 = 0.0;
      int j = sp.g == 0 ? sp.G : sp.g;
      if constexpr (!SM) {
        // L2 latency bound: eight loads in flight per thread
        double a2 = 0.0, a3 = 0.0;
        for (; j + 7 * sp.G < len; j += 8 * sp.G) {
          double y[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) y[u] = col[(j + u * sp.G) * ld];
          a0 += y[0] * pv[j] + y[4] * pv[j + 4 * sp.G]; a1 += y[1] * pv[j + sp.G] + y[5] * pv[j + 5 * sp.G];
          a2 += y[2] * pv[j + 2 * sp.G] + y[6] * pv[j + 6 * sp.G]; a3 += y[3] * pv[j + 3 * sp.G] + y[7] * pv[j + 7 * sp.G];
        }
        for (; j < len; j += sp.G) a0 += col[j * ld] * pv[j];
        a0 += a2; a1 += a3;
      } else {
        for (; j + sp.G < len; j += 2 * sp.G) { a0 += col[j * ld] * vc[j * ld]; a1 += col[(j + sp.G) * ld] * vc[(j + sp.G) * ld]; }
        if (j < len) a0 += col[j * ld] * vc[j * ld];
      }
      part[sp.g * sp.istep + i] = a0 + a1;
    }
    c.sync();
    double pdot = 0.0;
    if (sp.g == 0) {
      for (int i = sp.i0; i < len; i += sp.istep) {
        double acc = part[i];
        for (int g = 1; g < sp.G; ++g) acc += part[g * sp.istep + i];
        const double pi = (W[off * ld + off + i] + scale * acc) * tauk;
        const double xi = SM ? vc[i * ld] : pv[i];
        const double vi = i == 0 ? 1.0 : xi * scale;
        pv[i] = vi; wv[i] = pi;
        pdot += pi * vi;
      }
    }
    const double hk = 0.5 * tauk * c.sum(pdot);
    if (sp.g == 0) {
      for (int i = sp.i0; i < len; i += sp.istep) {
        wv[i] -= hk * pv[i];
        if (i > 0) W[(off + i) * ld + k] = pv[i];                  // keep the reflector
      }
    }
    c.sync();
    // A22 -= v w' + w v'; the next column norm (row 0 of the updated block, columns >= 2) on the fly.  Both products are
    // rounded on their own (DG_MUL): entries (i, j) and (j, i) then add the same two numbers and A22 stays exactly symmetric.
    // A contracted form rounds the two entries differently; the steps below take the reflector from a column but A22 v
    // from rows, and the asymmetry cost a degenerate cluster of eigenvalues up to 1e-4 of H (tests/test_gpu_units.py).
    nrm = 0.0;
    for (int j = sp.i0; j < len; j += sp.istep) {
      const double vj = pv[j], wj = wv[j];
      double* DG_RESTRICT col = W + off * ld + off + j;
      int i = sp.g;
      if constexpr (!SM) {
        // eight independent read-modify-writes per step
        for (; i + 7 * sp.G < len; i += 8 * sp.G) {
          double y[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) y[u] = col[(i + u * sp.G) * ld];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int iu = i + u * sp.G;
            const double cv = y[u] - (DG_MUL(pv[iu], wj) + DG_MUL(wv[iu], vj));
            col[iu * ld] = cv;
            if (iu == 0 && j >= 2) nrm += cv * cv;
          }
        }
      }
      for (; i < len; i += sp.G) {
        const double cv = col[i * ld] - (DG_MUL(pv[i], wj) + DG_MUL(wv[i], vj));
        col[i * ld] = cv;
        if (i == 0 && j >= 2) nrm += cv * cv;
      }
    }
    xn2 = c.sum(nrm);
  }
  if (c.tid() == 0 && kstop >= n - 1) { B.dg[n - 1] = W[(n - 1) * ld + (n - 1)]; B.od[n - 1] = 0.0; B.od2[n - 1] = 0.0; }
  c.sync();
}

#ifndef DG_HOSTSIM
// ---- register-resident tridiagonalisation on 2D tiles (256-thread CTAs, n <= 16*T <= 128) ----------------------------
// The column-per-thread form above pulls every entry of the Householder vectors through shared memory once per THREAD
// (three broadcasts of ~n/2 doubles per thread and step: ~2500 shared-memory wavefronts per step at n = 100 -- the
// shared-memory pipe, not the FP64 pipe, bounds it; ncu: 58 % LSU utilisation inside the phase).  Here the threads form a
// 16 x 16 grid and thread (ti, tj) keeps the cyclic tile  A[ti + 16 ra][tj + 16 cb], ra, cb < T,  of the full symmetric
// matrix in registers, so a step needs only the 2T entries of each vector that belong to the thread's rows and columns.
// Step k (off = k + 1), two barriers:
//   scalars (beta, tau, scale) from the 16 partial norms the holders of column off left, by every thread
//   v for the thread's rows and columns from the raw column x (zero on dead indices: no masks)
//   partial products sum_cb a[ra][cb] v_cb, reduced over the 16 lanes of the thread row with a reduce-scatter butterfly
//   (8 double shuffles), p = tau A v into shared memory; v'Av per warp                               -> barrier
//   A -= v c' + p v'  with  c = p - 2 hk v  (= v w' + w v', w = p - hk v, without a second vector exchange)
//   the holders of column off + 1 publish it (raw) with their partial norms                           -> barrier
// Dead tile rows / columns (all indices <= k) are skipped by a CTA-uniform switch on off >> 4; what remains of the dead
// entries only collects values that are multiplied by zeros of v.  Same outputs as sym_tridiag.
// Scratch: 424 doubles of B.part.
DG_DEV void tile_reduce_scatter(double (&q)[8], int l16) {
  // sum over the 16 lanes of a half warp; lane l16 ends with the total of entry (l16 >> 1) & 7 in q[0]
  {
    const bool b = (l16 >> 3) & 1;
    double snd[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) snd[i] = b ? q[i] : q[i + 4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { const double r = __shfl_xor_sync(0xffffffffu, snd[i], 8); q[i] = (b ? q[i + 4] : q[i]) + r; }
  }
  {
    const bool b = (l16 >> 2) & 1;
    double snd[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) snd[i] = b ? q[i] : q[i + 2];
#pragma unroll
    for (int i = 0; i < 2; ++i) { const double r = __shfl_xor_sync(0xffffffffu, snd[i], 4); q[i] = (b ? q[i + 2] : q[i]) + r; }
  }
  {
    const bool b = (l16 >> 1) & 1;
    const double snd = b ? q[0] : q[1];
    const double r = __shfl_xor_sync(0xffffffffu, snd, 2);
    q[0] = (b ? q[1] : q[0]) + r;
  }
  q[0] += __shfl_xor_sync(0xffffffffu, q[0], 1);
}

// Householder scalars of the column published in xs / pn (alpha = xs[off], |x[off+1:]|^2 from the 16 partial norms):
// beta = -sign(alpha) |x|, tau = (beta - alpha) / beta, scale = 1 / (alpha - beta), formed from one reciprocal square root
// and one reciprocal instead of a square root and two divisions (the chain sits between two barriers of every step).
struct TileHh { double beta, tau, scale; };
DG_DEV TileHh tile_householder(const double* DG_RESTRICT xs, const double* DG_RESTRICT pn, int off) {
  const double2* DG_RESTRICT p2 = reinterpret_cast<const double2*>(pn);
  const double2 p0 = p2[0], p1 = p2[1], p2_ = p2[2], p3 = p2[3], p4 = p2[4], p5 = p2[5], p6 = p2[6], p7 = p2[7];
  const double xn2 = (((p0.x + p0.y) + (p1.x + p1.y)) + ((p2_.x + p2_.y) + (p3.x + p3.y))) + (((p4.x + p4.y) + (p5.x + p5.y)) + ((p6.x + p6.y) + (p7.x + p7.y)));
  const double alpha = xs[off];
  TileHh h; h.beta = alpha; h.tau = 0.0; h.scale = 0.0;
  if (xn2 > 0.0) {
    const double s2 = fma(alpha, alpha, xn2);
    const double rn = rsqrt(s2);                                   // 1 / |x|
    const double nrm = s2 * rn;
    h.beta = -copysign(nrm, alpha);
    h.tau = (alpha - h.beta) * copysign(rn, alpha);                // (beta - alpha) / beta,  1 / beta = -sign(alpha) / |x|
    h.scale = __drcp_rn(alpha - h.beta);
  }
  return h;
}

template <int T, int S, bool SM>
DG_DEV void tridiag_tile_step(Cta& c, int n, int k, int ld, double (&a)[T][T], double* DG_RESTRICT W, const LinBuf& B,
                              double* DG_RESTRICT xs, double* DG_RESTRICT pn, double* DG_RESTRICT pb, double* DG_RESTRICT hp,
                              TileHh& hh) {
  const int tj = c.tid() & 15, ti = c.tid() >> 4, off = k + 1;
  const double tauk = hh.tau, scale = hh.scale;
  double vr[T], vc[T];
#pragma unroll
  for (int r = S; r < T; ++r) { const int j = ti + 16 * r; vr[r] = j == off ? 1.0 : xs[j] * scale; }
#pragma unroll
  for (int r = S; r < T; ++r) { const int i = tj + 16 * r; vc[r] = i == off ? 1.0 : xs[i] * scale; }
  if (tj == (k & 15)) {
#pragma unroll
    for (int r = S; r < T; ++r) { const int j = ti + 16 * r; if (j > off && j < n) W[j * ld + k] = vr[r]; }   // keep the reflector
  }
  // partial products and v'Av
  double q[8];
#pragma unroll
  for (int r = 0; r < 8; ++r) q[r] = 0.0;
  double vav = 0.0;
#pragma unroll
  for (int r = S; r < T; ++r) {
    double acc = 0.0;
#pragma unroll
    for (int cb = S; cb < T; ++cb) acc = fma(a[r][cb], vc[cb], acc);
    q[r] = acc;
    vav = fma(vr[r], acc, vav);
  }
  tile_reduce_scatter(q, tj);
  vav = c.warp_sum(vav);
  {
    const int idx = (tj >> 1) & 7;
    if ((tj & 1) == 0 && idx < T) pb[ti + 16 * idx] = tauk * q[0];
    if (c.lane() == 0) hp[c.warp()] = vav;
  }
  c.sync();
  double hk;
  {
    const double2* DG_RESTRICT h2 = reinterpret_cast<const double2*>(hp);
    const double2 h0 = h2[0], h1 = h2[1], h2_ = h2[2], h3 = h2[3];
    hk = 0.5 * tauk * tauk * (((h0.x + h0.y) + (h1.x + h1.y)) + ((h2_.x + h2_.y) + (h3.x + h3.y)));
  }
  // A -= v c' + p v': first the tile column that contains column off, whose holders publish it (raw, with their partial
  // norms) for the next step
  double pr[T], cc[T];
#pragma unroll
  for (int r = S; r < T; ++r) pr[r] = pb[ti + 16 * r];
#pragma unroll
  for (int cb = S; cb < T; ++cb) cc[cb] = fma(-2.0 * hk, vc[cb], pb[tj + 16 * cb]);
#pragma unroll
  for (int r = S; r < T; ++r) a[r][S] = fma(-vr[r], cc[S], fma(-pr[r], vc[S], a[r][S]));
  if (tj == (off & 15)) {
    double nrm = 0.0;
#pragma unroll
    for (int r = 0; r < T; ++r) {
      const int j = ti + 16 * r;
      double val = 0.0;
      if (r >= S) {
        const double av = a[r][S];
        if (j == off) B.dg[off] = av;
        if (j > off && j < n) val = av;
      }
      xs[j] = val;
      if (j >= off + 2) nrm = fma(val, val, nrm);
    }
    pn[ti] = nrm;
  }
  c.sync();
  // the scalars of the next step (a chain of dependent special-function and FP64 operations) beside the rest of the update
  if (off + 1 < n) {
    hh = tile_householder(xs, pn, off + 1);
    if (c.tid() == 0) { B.od[off] = hh.beta; B.od2[off] = hh.beta * hh.beta; B.tau[off] = hh.tau; }
  }
#pragma unroll
  for (int r = S; r < T; ++r)
#pragma unroll
    for (int cb = S + 1; cb < T; ++cb) a[r][cb] = fma(-vr[r], cc[cb], fma(-pr[r], vc[cb], a[r][cb]));
}

#define DG_TILE_CASE(m) case m: if constexpr (m < T) tridiag_tile_step<T, m, SM>(c, n, k, ld, a, W, B, xs, pn, pb, hp, hh); break;
// Qraw != null: the tiles are loaded as sym(Qraw) = (Qraw + Qraw')/2 straight from the row-major n x n matrix (no pass through W).
template <int T, bool SM>
DG_DEVN void sym_tridiag_tiles(Cta& c, int n, const LinBuf& B_, const double* DG_RESTRICT Qraw) {
  static_assert(T >= 1 && T <= 8, "tiles of at most 8 x 8 entries per thread");
  const LinBuf B = B_; DG_SH_LIN_T(B);
  double* DG_RESTRICT W = B.matA;
  const int ld = B.ld;
  const int tj = c.tid() & 15, ti = c.tid() >> 4;
  double* DG_RESTRICT xs = B.part;                                // [128] raw column of the step
  double* DG_RESTRICT pn = B.part + 128;                          // [16]  partial norms of its holders
  double* DG_RESTRICT pb = B.part + 144;                          // [128] p = tau A v
  double* DG_RESTRICT hp = B.part + 272;                          // [8]   v'Av per warp
  double a[T][T];
#pragma unroll
  for (int r = 0; r < T; ++r)
#pragma unroll
    for (int cb = 0; cb < T; ++cb) {
      const int j = ti + 16 * r, i = tj + 16 * cb;
      a[r][cb] = (j < n && i < n) ? (Qraw ? 0.5 * (Qraw[j * n + i] + Qraw[i * n + j]) : W[j * ld + i]) : 0.0;
    }
  DG_FOR(t, 128) { xs[t] = 0.0; pb[t] = 0.0; }
  c.sync();
  if (tj == 0) {
    double nrm = 0.0;
#pragma unroll
    for (int r = 0; r < T; ++r) {
      const int j = ti + 16 * r;
      if (j < n) {
        const double av = a[r][0];
        if (j == 0) B.dg[0] = av;
        else { xs[j] = av; if (j >= 2) nrm = fma(av, av, nrm); }
      }
    }
    pn[ti] = nrm;
  }
  c.sync();
  TileHh hh = tile_householder(xs, pn, 1);
  if (c.tid() == 0) { B.od[0] = hh.beta; B.od2[0] = hh.beta * hh.beta; B.tau[0] = hh.tau; }
  for (int k = 0; k + 1 < n; ++k) {
    switch ((k + 1) >> 4) { DG_TILE_CASE(0) DG_TILE_CASE(1) DG_TILE_CASE(2) DG_TILE_CASE(3) DG_TILE_CASE(4) DG_TILE_CASE(5) DG_TILE_CASE(6) DG_TILE_CASE(7) default: break; }
  }
  if (c.tid() == 0) { B.od[n - 1] = 0.0; B.od2[n - 1] = 0.0; }
  c.sync();
}
#undef DG_TILE_CASE

DG_DEV bool sym_tridiag_tiles_applies(const Cta& c, int n) { return c.nt() == 256 && n >= 33 && n <= 128; }
template <bool SM>
DG_DEV bool sym_tridiag_tiles_dispatch(Cta& c, int n, const LinBuf& B, const double* DG_RESTRICT Qraw) {
  if (!sym_tridiag_tiles_applies(c, n)) return false;
  const int T = (n + 15) >> 4;
  switch (T) {
    case 3: sym_tridiag_tiles<3, SM>(c, n, B, Qraw); break;
    case 4: sym_tridiag_tiles<4, SM>(c, n, B, Qraw); break;
    case 5: sym_tridiag_tiles<5, SM>(c, n, B, Qraw); break;
    case 6: sym_tridiag_tiles<6, SM>(c, n, B, Qraw); break;
    case 7: sym_tridiag_tiles<7, SM>(c, n, B, Qraw); break;
    default: sym_tridiag_tiles<8, SM>(c, n, B, Qraw); break;
  }
  return true;
}

#endif

// number of eigenvalues of tridiag(dg, od) that are < x   (od2 = od^2).
// Sturm sequence in product form  p_i = (d_i - x) p_{i-1} - e_{i-1}^2 p_{i-2}  (sign changes = negative pivots of
// the ratio form q_i = p_i / p_{i-1} that LAPACK's dstebz counts): one dependent FMA per row instead of a
// division.  The pair (p_{i-1}, p_i) is rescaled by powers of two, which leaves the signs untouched; an exact zero
// is replaced like dstebz's pivmin rule (q = -pivmin).
// Every thread of the CTA walks its own chain (one probe each), so what matters is the length of the dependent chain
// per row: the product e^2 p_{i-2} is formed off the chain, the pivmin rule is a select, and the range check runs once
// per four rows behind a rarely taken branch.  (With M = max(1, 2|T|) the pair grows by at most 2M per row, so between
// two checks it stays below 2^512 (2M)^4 < 2^1023 as long as |T| < 2^60; larger matrices check every row.)
DG_DEV int sturm_count(int n, const double* DG_RESTRICT dg, const double* DG_RESTRICT od2, double x, double pivmin) {
  const double BIG = 1.3407807929942597e154 /* 2^512 */, SMALL = 7.458340731200207e-155 /* 2^-512 */;
  int cnt = 0;
  double pm = 1.0, pc = dg[0] - x;
  if (fabs(pc) < pivmin) pc = -pivmin;
  cnt += pc < 0.0;
  const bool wide = !(pivmin < 2.2250738585072014e-308 * 1.3e36);     // pivmin = tiny * max(1, |T|^2): |T| >= 2^60
#define DG_STURM_ROW(i) { \
    const double t = od2[(i) - 1] * pm, lim = pivmin * fabs(pc); \
    double pn = fma(dg[(i)] - x, pc, -t); \
    pn = fabs(pn) < lim ? -pivmin * pc : pn; \
    cnt += (pn < 0.0) != (pc < 0.0); \
    pm = pc; pc = pn; }
#define DG_STURM_RANGE() { \
    const double ap = fabs(pc); \
    if (ap > BIG) { pc *= SMALL; pm *= SMALL; } else if (ap < SMALL) { pc *= BIG; pm *= BIG; } }
  int i = 1;
  if (!wide) {
    for (; i + 3 < n; i += 4) {
      DG_STURM_ROW(i) DG_STURM_ROW(i + 1) DG_STURM_ROW(i + 2) DG_STURM_ROW(i + 3)
      DG_STURM_RANGE()
    }
  }
  for (; i < n; ++i) { DG_STURM_ROW(i) DG_STURM_RANGE() }
#undef DG_STURM_ROW
#undef DG_STURM_RANGE
  return cnt;
}

// Solve (T - lam I) y = b in place (y overwrites b) by Gaussian elimination with partial pivoting; returns |y|^2.
// fw: 5 arrays of n (reciprocal pivot, sup1, sup2, mult, swapped) and y are INTERLEAVED over the vectors of a chunk:
// element i of this thread's vector sits at [i * st] (st = chunk width), so that the threads of a warp
// touch consecutive words.
// One thread walks the whole chain, so the recurrences are arranged to keep as little as possible on it: pivots are
// stored as reciprocals (the back substitution multiplies), the running entries of y stay in registers (no
// store -> load round trip through shared memory per row) and |y|^2 is accumulated beside the chain.
DG_DEV double tridiag_shift_solve(int n, const double* DG_RESTRICT dg, const double* DG_RESTRICT od, double lam, double tiny,
                                  double* DG_RESTRICT fw, double* DG_RESTRICT y, int st, bool refactor) {
  // (fw and y are disjoint: the loads of the factors can run ahead of the stores into y)
  double* ra = fw; double* b1 = fw + n * st; double* b2 = fw + 2 * n * st; double* ml = fw + 3 * n * st; double* sw = fw + 4 * n * st;
  const double rtiny = 1.0 / tiny;
  if (refactor) {
    // work row "cur" = (p, q, r) starting at column i
    double p = dg[0] - lam, q = n > 1 ? od[0] : 0.0, r = 0.0;
    for (int i = 0; i + 1 < n; ++i) {
      const double sub = od[i], nd = dg[i + 1] - lam, ns = i + 2 < n ? od[i + 1] : 0.0;
      if (fabs(sub) > fabs(p)) {
        const double rs = 1.0 / sub;                // pivot row is the next row (sub, nd, ns); sub is off the chain
        const double m = p * rs;
        ra[i * st] = fabs(sub) < tiny ? (sub < 0.0 ? -rtiny : rtiny) : rs;
        b1[i * st] = nd; b2[i * st] = ns; ml[i * st] = m; sw[i * st] = 1.0;
        p = q - m * nd; q = r - m * ns; r = 0.0;
      } else {
        if (p == 0.0) p = tiny;
        const double rp = 1.0 / p;
        const double m = sub * rp;
        ra[i * st] = fabs(p) < tiny ? (p < 0.0 ? -rtiny : rtiny) : rp;
        b1[i * st] = q; b2[i * st] = r; ml[i * st] = m; sw[i * st] = 0.0;
        p = nd - m * q; q = ns - m * r; r = 0.0;
      }
    }
    if (fabs(p) < tiny) p = p < 0.0 ? -tiny : tiny;
    ra[(n - 1) * st] = 1.0 / p; b1[(n - 1) * st] = 0.0; b2[(n - 1) * st] = 0.0;
  }
  // forward elimination of the right-hand side: one fused multiply-add per row on the chain
  double yc = y[0];
  for (int i = 0; i + 1 < n; ++i) {
    const double yn = y[(i + 1) * st], m = ml[i * st];
    if (sw[i * st] != 0.0) { y[i * st] = yn; yc = yc - m * yn; }
    else { y[i * st] = yc; yc = yn - m * yc; }
  }
  // back substitution
  double y1 = yc * ra[(n - 1) * st], y2 = 0.0, nr = y1 * y1;
  y[(n - 1) * st] = y1;
  for (int i = n - 2; i >= 0; --i) {
    const double t = (y[i * st] - b2[i * st] * y2 - b1[i * st] * y1) * ra[i * st];
    y[i * st] = t;
    nr += t * t;
    y2 = y1; y1 = t;
  }
  return nr;
}

// One inverse-iteration sweep of one eigenvector (thread-serial): start vector on the first sweep, solve, normalise.
DG_DEV void invit_sweep(int n, const double* DG_RESTRICT dg, const double* DG_RESTRICT od, double lam, double tiny,
                        double* DG_RESTRICT fw, double* DG_RESTRICT z, int st, bool first, int seed) {
  if (first)
    for (int i = 0; i < n; ++i) z[i * st] = 1.0 + 0.37 * (double)(((i + 1) * 7919 + seed * 104729) % 97) / 97.0;
  double nr = tridiag_shift_solve(n, dg, od, lam, tiny, fw, z, st, first);
  nr = DG_RSQRT(nr);
  for (int i = 0; i < n; ++i) z[i * st] *= nr;
}

#ifndef DG_HOSTSIM
// The same count by the 16 lanes of a half warp together (every lane returns it).  The recurrence is linear,
// (p_i, p_{i-1})' = M_i (p_{i-1}, p_{i-2})' with M_i = [[d_i - x, -e_{i-1}^2], [1, 0]], so lane l multiplies the matrices of its
// ceil(n/16) rows, a Hillis-Steele scan over the 16 lanes (4 steps of 2x2 products through shuffles, every product
// renormalised by a power of two: signs are all that matters) gives each lane the pair entering its rows, and the lane
// re-walks its rows from there with the zero rule of sturm_count, counting sign changes.  A probe costs ~0.7 kcycles instead
// of the ~9 kcycles of the n-row dependent chain, at 16 instead of 256 probes per round.
DG_DEV void sturm_norm4(double& a, double& b, double& c2, double& d) {
  const double m = fmax(fmax(fabs(a), fabs(b)), fmax(fabs(c2), fabs(d)));
  const int eb = (__double2hiint(m) >> 20) & 0x7ff;
  if (eb > 0 && eb < 0x7fe) {
    const double sc = __hiloint2double((2046 - eb) << 20, 0);      // 2^-(eb - 1023)
    a *= sc; b *= sc; c2 *= sc; d *= sc;
  }
}
DG_DEV int sturm_count_group16(int n, const double* DG_RESTRICT dg, const double* DG_RESTRICT od2, double x, double pivmin, int l16) {
  const int RL = (n + 15) >> 4, i0 = l16 * RL, i1 = i0 + RL < n ? i0 + RL : n;
  // product of this lane's rows (identity for lanes beyond the matrix)
  double p11 = 1.0, p12 = 0.0, p21 = 0.0, p22 = 1.0;
  for (int i = i0; i < i1; ++i) {
    const double a = dg[i] - x, b = i > 0 ? od2[i - 1] : 0.0;
    const double n11 = fma(a, p11, -b * p21), n12 = fma(a, p12, -b * p22);
    p21 = p11; p22 = p12; p11 = n11; p12 = n12;
  }
  sturm_norm4(p11, p12, p21, p22);
  // inclusive scan: later rows on the left
#pragma unroll
  for (int o = 1; o < 16; o <<= 1) {
    const double t11 = __shfl_up_sync(0xffffffffu, p11, o, 16), t12 = __shfl_up_sync(0xffffffffu, p12, o, 16);
    const double t21 = __shfl_up_sync(0xffffffffu, p21, o, 16), t22 = __shfl_up_sync(0xffffffffu, p22, o, 16);
    if (l16 >= o) {
      const double n11 = fma(p11, t11, p12 * t21), n12 = fma(p11, t12, p12 * t22);
      const double n21 = fma(p21, t11, p22 * t21), n22 = fma(p21, t12, p22 * t22);
      p11 = n11; p12 = n12; p21 = n21; p22 = n22;
      sturm_norm4(p11, p12, p21, p22);
    }
  }
  // pair entering this lane's rows: first column of the product of all earlier lanes, (1, 0)' for lane 0
  double pc = __shfl_up_sync(0xffffffffu, p11, 1, 16), pm = __shfl_up_sync(0xffffffffu, p21, 1, 16);
  if (l16 == 0) { pc = 1.0; pm = 0.0; }
  int cnt = 0;
  for (int i = i0; i < i1; ++i) {
    const double t = (i > 0 ? od2[i - 1] : 0.0) * pm, lim = pivmin * fabs(pc);
    double pn = fma(dg[i] - x, pc, -t);
    pn = fabs(pn) < lim ? -pivmin * pc : pn;
    cnt += (pn < 0.0) != (pc < 0.0);
    pm = pc; pc = pn;
  }
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o, 16);
  return cnt;
}
#endif

// Negative eigenvalues of the tridiagonal matrix into B.lam[0..nneg): Sturm-count multisection.  All
// eigenvalues are refined together: each round spends the CTA's nt probes evenly over the brackets.
// lo/hi: nneg doubles each; first: nneg ints of scratch.
template <bool SM>
DG_DEV void negative_eigenvalues(Cta& c, int n, const LinBuf& B, int nneg, double tnorm, double pivmin,
                                 double* lo, double* hi, int* first) {
  // (inlined into nearest_pd, which carries the address-space hints: repeating a hint on the same pointer inside an
  //  inlined callee makes nvcc 12.9 drop the guarded code)
  DG_FOR(j, nneg) { lo[j] = -tnorm * 1.0000001 - pivmin; hi[j] = 0.0; first[j] = 0x7fffffff; }
  c.sync();
  int per = c.nt() / nneg;                       // probes per eigenvalue per round
  if (per < 1) per = 1;
  const int groups = c.nt() / per;               // eigenvalues refined concurrently
  int rounds = (int)ceil(54.0 * 0.6931471805599453 / log((double)per + 1.0));
  if (rounds < 1) rounds = 1;
  for (int j0 = 0; j0 < nneg; j0 += groups) {
    const int g = c.tid() / per, t = c.tid() - g * per, j = j0 + g;
    const bool act = g < groups && j < nneg;
    for (int rd = 0; rd < rounds; ++rd) {
      double a = 0.0, h = 0.0;
      if (act) {
        a = lo[j];
        h = (hi[j] - a) / (double)(per + 1);
        // first[j] = smallest probe index whose count reaches j+1.  (In floating point the counts of the product-form
        // Sturm sequence need not be monotone in the shift, so "count reached here but not at the previous probe"
        // can hold for several probes: the minimum makes the choice unique.)
        if (sturm_count(n, B.dg, B.od2, a + h * (double)(t + 1), pivmin) >= j + 1) DG_ATOMIC_MIN(&first[j], t);
      }
      c.sync();
      if (act && t == 0) {
        const int f = first[j];
        first[j] = 0x7fffffff;
        if (f == 0x7fffffff) lo[j] = a + h * (double)per;
        else { if (f > 0) lo[j] = a + h * (double)f; hi[j] = a + h * (double)(f + 1); }
      }
      c.sync();
    }
  }
  DG_FOR(j, nneg) B.lam[j] = 0.5 * (lo[j] + hi[j]);
  c.sync();
}

#ifndef DG_HOSTSIM
// ---- eigenvector of the tridiagonal matrix by one warp: twisted factorisation (Fernando / Parlett-Dhillon) ---------------
// With D+_i = p_i / p_{i-1} (leading minors of T - lam I) and D-_i = r_i / r_{i+1} (trailing minors),
//   gamma_k = D+_k + D-_k - (d_k - lam),   twist index r = argmin |gamma_k|,
//   z_r = 1,   z_i = -(e_i / D+_i) z_{i+1} (i < r),   z_i = -(e_{i-1} / D-_i) z_{i-1} (i > r)
// solves (T - lam I) z = gamma_r e_r: one factorisation from each end instead of the LU + 2 x 2 substitutions of inverse
// iteration, and every recurrence is a scan -- the minors through the 2x2 products of sturm_count_group16 (32 lanes), the
// entries of z as running products kept as (mantissa, exponent) pairs so that no range is lost.  Lane l owns the rows
// [l R, (l+1) R), R = ceil(n/32) <= 4.  The caller accepts the vector only if its residual |gamma_r| |z_r| / |z| is at
// rounding level (returned) and falls back to inverse iteration otherwise; clusters always take the inverse iteration.
struct MantExp { double f; int e; };                   // value = f * 2^e, f = 0 or |f| in [1, 2)
DG_DEV MantExp me_norm(double v, int e) {
  MantExp r; r.f = v; r.e = e;
  const int eb = (__double2hiint(v) >> 20) & 0x7ff;
  if (eb > 0 && eb < 0x7ff) { r.f = __hiloint2double((__double2hiint(v) & 0x800fffff) | 0x3ff00000, __double2loint(v)); r.e = e + eb - 1023; }
  else if (eb == 0) { r.f = 0.0; r.e = -(1 << 28); }
  return r;
}
DG_DEV MantExp me_mul(MantExp a, MantExp b) { return me_norm(a.f * b.f, a.e + b.e); }
template <int R>
DG_DEV double twisted_eigvec(Cta& c, int n, const double* DG_RESTRICT dg, const double* DG_RESTRICT od, const double* DG_RESTRICT od2,
                             double lam, double pivmin, double* DG_RESTRICT z, double& rq_shift) {
  const int l = c.lane(), i0 = l * R;
  double dp[R], dm[R], a[R], e[R];                      // D+, D-, d_i - lam, e_i (couples i, i+1)
#pragma unroll
  for (int r = 0; r < R; ++r) { const int i = i0 + r; a[r] = i < n ? dg[i] - lam : 1.0; e[r] = i + 1 < n ? od[i] : 0.0; }
  // forward minors
  {
    double p11 = 1.0, p12 = 0.0, p21 = 0.0, p22 = 1.0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int i = i0 + r;
      if (i < n) {
        const double b = i > 0 ? od2[i - 1] : 0.0;
        const double n11 = fma(a[r], p11, -b * p21), n12 = fma(a[r], p12, -b * p22);
        p21 = p11; p22 = p12; p11 = n11; p12 = n12;
      }
    }
    sturm_norm4(p11, p12, p21, p22);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double t11 = __shfl_up_sync(0xffffffffu, p11, o), t12 = __shfl_up_sync(0xffffffffu, p12, o);
      const double t21 = __shfl_up_sync(0xffffffffu, p21, o), t22 = __shfl_up_sync(0xffffffffu, p22, o);
      if (l >= o) {
        const double n11 = fma(p11, t11, p12 * t21), n12 = fma(p11, t12, p12 * t22);
        const double n21 = fma(p21, t11, p22 * t21), n22 = fma(p21, t12, p22 * t22);
        p11 = n11; p12 = n12; p21 = n21; p22 = n22;
        sturm_norm4(p11, p12, p21, p22);
      }
    }
    double pc = __shfl_up_sync(0xffffffffu, p11, 1), pm = __shfl_up_sync(0xffffffffu, p21, 1);
    if (l == 0) { pc = 1.0; pm = 0.0; }
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int i = i0 + r;
      dp[r] = 1.0;
      if (i < n) {
        const double t = (i > 0 ? od2[i - 1] : 0.0) * pm, lim = pivmin * fabs(pc);
        double pn = fma(a[r], pc, -t);
        pn = fabs(pn) < lim ? -pivmin * pc : pn;
        dp[r] = pn / pc;
        pm = pc; pc = pn;
      }
    }
  }
  // backward minors: (r_i, r_{i+1})' = [[d_i - lam, -e_i^2], [1, 0]] (r_{i+1}, r_{i+2})'
  {
    double p11 = 1.0, p12 = 0.0, p21 = 0.0, p22 = 1.0;
#pragma unroll
    for (int r = R - 1; r >= 0; --r) {
      const int i = i0 + r;
      if (i < n) {
        const double b = e[r] * e[r];
        const double n11 = fma(a[r], p11, -b * p21), n12 = fma(a[r], p12, -b * p22);
        p21 = p11; p22 = p12; p11 = n11; p12 = n12;
      }
    }
    sturm_norm4(p11, p12, p21, p22);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double t11 = __shfl_down_sync(0xffffffffu, p11, o), t12 = __shfl_down_sync(0xffffffffu, p12, o);
      const double t21 = __shfl_down_sync(0xffffffffu, p21, o), t22 = __shfl_down_sync(0xffffffffu, p22, o);
      if (l + o < 32) {
        const double n11 = fma(p11, t11, p12 * t21), n12 = fma(p11, t12, p12 * t22);
        const double n21 = fma(p21, t11, p22 * t21), n22 = fma(p21, t12, p22 * t22);
        p11 = n11; p12 = n12; p21 = n21; p22 = n22;
        sturm_norm4(p11, p12, p21, p22);
      }
    }
    double rc = __shfl_down_sync(0xffffffffu, p11, 1), rm = __shfl_down_sync(0xffffffffu, p21, 1);
    if (l == 31) { rc = 1.0; rm = 0.0; }
#pragma unroll
    for (int r = R - 1; r >= 0; --r) {
      const int i = i0 + r;
      dm[r] = 1.0;
      if (i < n) {
        const double t = e[r] * e[r] * rm, lim = pivmin * fabs(rc);
        double rn = fma(a[r], rc, -t);
        rn = fabs(rn) < lim ? -pivmin * rc : rn;
        dm[r] = rn / rc;
        rm = rc; rc = rn;
      }
    }
  }
  // twist index
  double gbest = 1e300; int kbest = 0x7fffffff;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int i = i0 + r;
    if (i < n) { const double g = fabs(dp[r] + dm[r] - a[r]); if (g < gbest) { gbest = g; kbest = i; } }
  }
  double gmin = gbest; int kr = kbest;
  c.warp_argmin(gmin, kr);
  double gsig = 0.0;                                      // gamma_r with its sign
#pragma unroll
  for (int r = 0; r < R; ++r) if (i0 + r == kr) gsig = dp[r] + dm[r] - a[r];
  gsig = c.warp_sum(gsig);
  // multipliers: rows above the twist use D+ (z_i = mu_i z_{i+1}), rows below use D- (z_i = mu_i z_{i-1}); scans of running
  // products in (mantissa, exponent) form.  up[r] = prod_{j=i}^{kr-1} mu_j for i < kr; dn[r] = prod_{j=kr+1}^{i} mu_j for i > kr
  MantExp zr[R];
  {
    // upward part: suffix products of mu_j = -e_j / D+_j over j in [i, kr)
    MantExp loc = {1.0, 0};
    MantExp part[R];
#pragma unroll
    for (int r = R - 1; r >= 0; --r) {
      const int i = i0 + r;
      if (i < kr && i < n) loc = me_mul(loc, me_norm(-e[r] / dp[r], 0));
      part[r] = loc;
    }
    MantExp tot = loc;                                     // product of this lane's rows that lie above the twist
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double tf = __shfl_down_sync(0xffffffffu, tot.f, o); const int te = __shfl_down_sync(0xffffffffu, tot.e, o);
      if (l + o < 32) { MantExp t2 = {tf, te}; tot = me_mul(tot, t2); }
    }
    double cf = __shfl_down_sync(0xffffffffu, tot.f, 1); int ce = __shfl_down_sync(0xffffffffu, tot.e, 1);
    if (l == 31) { cf = 1.0; ce = 0; }
    MantExp carry = {cf, ce};                              // product over all later lanes
#pragma unroll
    for (int r = 0; r < R; ++r) zr[r] = me_mul(part[r], carry);
  }
  {
    // downward part: prefix products of mu_j = -e_{j-1} / D-_j over j in (kr, i]
    MantExp loc = {1.0, 0};
    MantExp part[R];
    const double eprev = __shfl_up_sync(0xffffffffu, e[R - 1], 1);      // e_{i0-1}: couples the previous lane's last row with this lane's first
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int i = i0 + r;
      if (i > kr && i < n) {
        const double em1 = r > 0 ? e[r - 1] : eprev;
        loc = me_mul(loc, me_norm(-em1 / dm[r], 0));
      }
      part[r] = loc;
    }
    MantExp tot = loc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double tf = __shfl_up_sync(0xffffffffu, tot.f, o); const int te = __shfl_up_sync(0xffffffffu, tot.e, o);
      if (l >= o) { MantExp t2 = {tf, te}; tot = me_mul(tot, t2); }
    }
    double cf = __shfl_up_sync(0xffffffffu, tot.f, 1); int ce = __shfl_up_sync(0xffffffffu, tot.e, 1);
    if (l == 0) { cf = 1.0; ce = 0; }
    MantExp carry = {cf, ce};
#pragma unroll
    for (int r = 0; r < R; ++r) { const int i = i0 + r; if (i > kr) zr[r] = me_mul(part[r], carry); }
  }
  // common scale, 2-norm, store
  int emax = -(1 << 28);
#pragma unroll
  for (int r = 0; r < R; ++r) { const int i = i0 + r; if (i < n && zr[r].f != 0.0 && zr[r].e > emax) emax = zr[r].e; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { const int t = __shfl_xor_sync(0xffffffffu, emax, o); emax = t > emax ? t : emax; }
  double zv[R], nr = 0.0;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int i = i0 + r;
    const int de = zr[r].e - emax;
    zv[r] = (i < n && zr[r].f != 0.0 && de > -1000) ? ldexp(zr[r].f, de) : 0.0;
    nr = fma(zv[r], zv[r], nr);
  }
  nr = c.warp_sum(nr);
  const double sc = DG_RSQRT(nr);
#pragma unroll
  for (int r = 0; r < R; ++r) { const int i = i0 + r; if (i < n) z[i] = zv[r] * sc; }
  // residual of the unit vector: |gamma_r| |z_r|
  double zk = 0.0;
#pragma unroll
  for (int r = 0; r < R; ++r) if (i0 + r == kr) zk = fabs(zv[r]) * sc;
  zk = c.warp_sum(zk);
  rq_shift = gsig * zk * zk;                              // Rayleigh quotient of z minus lam ((T - lam I) z = gamma_r z_r e_r)
  // TRUE residual |(T - lam I) z| of the stored unit vector: gamma_r z_r only bounds it when the pivots carry no growth
  const double zprev = __shfl_up_sync(0xffffffffu, zv[R - 1], 1), znext = __shfl_down_sync(0xffffffffu, zv[0], 1);
  const double eprev2 = __shfl_up_sync(0xffffffffu, e[R - 1], 1);
  double rs = 0.0;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int i = i0 + r;
    if (i < n) {
      const double zm = r > 0 ? zv[r - 1] : (l > 0 ? zprev : 0.0), zp = r + 1 < R ? zv[r + 1] : (l < 31 ? znext : 0.0);
      const double em = r > 0 ? e[r - 1] : (l > 0 ? eprev2 : 0.0);
      const double ri = (a[r] * zv[r] + em * zm + e[r] * zp) * sc;
      rs = fma(ri, ri, rs);
    }
  }
  rs = c.warp_sum(rs);
  return sqrt(rs);
}
#endif

#ifndef DG_HOSTSIM
// The same multisection for up to 16 negative eigenvalues with half-warp probes (sturm_count_group16): 16 probes per round
// instead of 256, each ~10x cheaper than a thread's chain; the brackets live in the registers of the half warps that refine
// them (every probe group of an eigenvalue applies the same update), the winners go through three rotating arrays of
// `first`, so a round has ONE barrier.  first: 3 * 16 ints.
template <bool SM>
DG_DEV void negative_eigenvalues_grp(Cta& c, int n, const LinBuf& B, int nneg, double tnorm, double pivmin, int* first) {
  const int slots = c.nt() >> 4, slot = c.tid() >> 4, l16 = c.tid() & 15;
  DG_FOR(j, 48) first[j] = 0x7fffffff;
  c.sync();
  int per = slots / nneg;
  if (per < 1) per = 1;
  const int g = slot / per, t = slot - g * per;
  const bool act = g < nneg && g * per + t < slots && slot < nneg * per;
  const double rper = 1.0 / (double)(per + 1);
  int rounds = (int)ceil(54.0 * 0.6931471805599453 / log((double)per + 1.0));
  if (rounds < 1) rounds = 1;
  double lo = -tnorm * 1.0000001 - pivmin, hi = 0.0;
  for (int rd = 0; rd < rounds; ++rd) {
    int* DG_RESTRICT fb = first + 16 * (rd % 3);
    const double h = (hi - lo) * rper;
    const int cnt = sturm_count_group16(n, B.dg, B.od2, lo + h * (double)(t + 1), pivmin, l16);
    if (act && l16 == 0 && cnt >= g + 1) DG_ATOMIC_MIN(&fb[g], t);
    c.sync();
    if (act) {
      const int f = fb[g];
      if (f == 0x7fffffff) lo = lo + h * (double)per;
      else { const double a = lo; if (f > 0) lo = a + h * (double)f; hi = a + h * (double)(f + 1); }
    }
    // the array of the previous round has been read by everyone (before this round's barrier): clear it for round rd + 2
    if (c.tid() < 16) first[16 * ((rd + 2) % 3) + c.tid()] = 0x7fffffff;
  }
  if (act && t == 0 && l16 == 0) B.lam[g] = 0.5 * (lo + hi);
  c.sync();
}
#endif

#ifndef DG_HOSTSIM
// Back-transformation of the eigenvectors of the tridiagonal matrix, y = H_0 H_1 ... H_{n-3} z: one warp per vector, the
// vector in REGISTERS (lane l holds the entries l, l+32, ..), the reflector tails (column k of W below row k+1) fetched
// one step ahead of the dependent chain  dot -> warp sum -> update.  Z: vector-major, n entries per vector.
template <int RPL>
DG_DEV void backtransform_regs(Cta& c, int n, int ld, const double* DG_RESTRICT W, const double* DG_RESTRICT tau,
                               double* DG_RESTRICT Z, int nvec) {
  // reflector k as a register vector: v_j = 0 (j <= k), 1 (j == k+1), W[j][k] (j > k+1)
  auto load = [&](double (&v)[RPL], int k) {
#pragma unroll
    for (int r = 0; r < RPL; ++r) { const int j = c.lane() + 32 * r; v[r] = (j > k + 1 && j < n) ? W[j * ld + k] : (j == k + 1 ? 1.0 : 0.0); }
  };
  for (int jv = c.warp(); jv < nvec; jv += c.nwarps()) {
    double* DG_RESTRICT z = Z + (size_t)jv * n;
    double zr[RPL], va[RPL], vb[RPL], na[RPL], nb[RPL];
#pragma unroll
    for (int r = 0; r < RPL; ++r) { const int j = c.lane() + 32 * r; zr[r] = j < n ? z[j] : 0.0; }
    // two reflectors per pass: H_{k-1} H_k z = z - v_k a - v_{k-1} b with a = tau_k v_k'z, b = tau_{k-1} (v_{k-1}'z - (v_{k-1}'v_k) a):
    // the three dot products of a pass share one shuffle-sum latency (half as many dependent chains as one reflector at a time)
    int k = n - 3;
    if (k >= 1) { load(na, k); load(nb, k - 1); }
    for (; k >= 1; k -= 2) {
      const double ta = tau[k], tb = tau[k - 1];
#pragma unroll
      for (int r = 0; r < RPL; ++r) { va[r] = na[r]; vb[r] = nb[r]; }
      if (k - 2 >= 1) { load(na, k - 2); load(nb, k - 3); }
      double d[3] = {0.0, 0.0, 0.0};
#pragma unroll
      for (int r = 0; r < RPL; ++r) { d[0] = fma(va[r], zr[r], d[0]); d[1] = fma(vb[r], zr[r], d[1]); d[2] = fma(va[r], vb[r], d[2]); }
      c.warp_sum_n(d);
      const double a = ta * d[0], b = tb * (d[1] - d[2] * a);
#pragma unroll
      for (int r = 0; r < RPL; ++r) zr[r] = fma(-b, vb[r], fma(-a, va[r], zr[r]));
    }
    if (k == 0) {                                             // odd number of reflectors: the last one alone
      load(va, 0);
      double pp = 0.0;
#pragma unroll
      for (int r = 0; r < RPL; ++r) pp = fma(va[r], zr[r], pp);
      pp = c.warp_sum(pp) * tau[0];
#pragma unroll
      for (int r = 0; r < RPL; ++r) zr[r] = fma(-pp, va[r], zr[r]);
    }
#pragma unroll
    for (int r = 0; r < RPL; ++r) { const int j = c.lane() + 32 * r; if (j < n) z[j] = zr[r]; }
  }
}
#endif

// matA <- nearestPD(Qraw) + reg*I  (n x n, leading dimension B.ld).  Qraw is row-major n x n (global memory, read
// twice).  matB is scratch.  Returns the number of negative eigenvalues (uniform across threads).
template <bool SM>
DG_DEVN int nearest_pd(Cta& c, int n, const double* DG_RESTRICT Qraw, const LinBuf& B_,
                       double floor_val, double reg, bool conv_approx) {
  // local copies: the tables live in shared memory and would otherwise be re-read after every store
  const LinBuf B = B_; DG_SH_LIN_P(B);
  const int ld = B.ld;
  double* DG_RESTRICT Hm = B.matA;
  c.lap(PH_OTHER);
  int nneg = 0;
  const double* Zall = nullptr;
  if (conv_approx) {
    // symmetric part into W (the register-tile tridiagonalisation loads it from Qraw itself)
#ifndef DG_HOSTSIM
    if (!sym_tridiag_tiles_applies(c, n))
#endif
    {
      DG_FOR(t, n * n) {
        int i = t / n, j = t - i * n;
        Hm[i * ld + j] = 0.5 * (Qraw[i * n + j] + Qraw[j * n + i]);
      }
      c.sync();
    }
    c.lapf(PH_PD_SYM);
#ifndef DG_HOSTSIM
    if (c.nt() == 256 && n > 128 && n <= 256) {
      // larger games (3-4 agents): the generic steps until the trailing matrix fits the register tiles, then the tile form
      // on the trailing 128 x 128 block (same algorithm continued: shifted views of W, dg, od, tau)
      const int base = n - 128;
      sym_tridiag<SM>(c, n, B, base);
      LinBuf Bt = B;
      Bt.matA = B.matA + (size_t)base * ld + base; Bt.dg = B.dg + base; Bt.od = B.od + base; Bt.od2 = B.od2 + base; Bt.tau = B.tau + base;
      sym_tridiag_tiles<8, SM>(c, 128, Bt, nullptr);
    } else if (!sym_tridiag_tiles_dispatch<SM>(c, n, B, Qraw))
#endif
    sym_tridiag<SM>(c, n, B, n);
    c.lap(PH_PD_TRIDIAG);
    double tn = 0.0;
    DG_FOR(i, n) {
      double r = fabs(B.dg[i]) + fabs(B.od[i]) + (i > 0 ? fabs(B.od[i - 1]) : 0.0);
      tn = fmax(tn, r);
    }
    const double tnorm = c.max(tn);
    const double pivmin = 2.2250738585072014e-308 * fmax(1.0, tnorm * tnorm);
#ifndef DG_HOSTSIM
    if ((c.nt() & 31) == 0 && pivmin < 2.2250738585072014e-308 * 1.3e36)
      nneg = sturm_count_group16(n, B.dg, B.od2, 0.0, pivmin, c.tid() & 15);   // every half warp computes the same count
    else
#endif
    nneg = sturm_count(n, B.dg, B.od2, 0.0, pivmin);      // every thread computes the same count
    if (nneg > 0) {
      // scratch carved from matB: [first (n ints) | itw (5 n CH, interleaved) | Zt (n CH, interleaved) | Z (nneg n, vector major)]
      const int CH = DG_EIG_CHUNK;
      double* scr = B.matB;
      int* cnts = (int*)scr;
      double* itw = scr + ((n + 1) / 2 + 1);
      double* Zt = itw + 5 * n * CH;
      double* Zs = Zt + n * CH;
      const long cap = ((long)n * ld - (Zs - scr)) / n;    // eigenvectors that fit behind the scratch
      double* Z = nneg <= cap ? Zs : B.Zg;
      // matB in the L2 workspace (split / global placement): the serial chains of the inverse iteration would walk L2; the
      // usual one to three vectors run in a small shared-memory block instead, interleaved with stride nneg
      int st = CH;
      if constexpr (!SM) {                 // (SM = true: matB is shared memory already, and the pointers keep their address space)
        if (B.eig_s && nneg <= DG_EIG_SMALL) { st = nneg; itw = B.eig_s; Zt = itw + 5 * n * st; }
      }
#ifndef DG_HOSTSIM
      if (nneg <= 16 && (c.nt() & 31) == 0 && c.nt() >= 16 * nneg && pivmin < 2.2250738585072014e-308 * 1.3e36)
        negative_eigenvalues_grp<SM>(c, n, B, nneg, tnorm, pivmin, cnts);
      else
#endif
      negative_eigenvalues<SM>(c, n, B, nneg, tnorm, pivmin, B.pv, B.wv, cnts);
      c.lapf(PH_PD_EIGVAL);
      // --- eigenvectors: without clusters one warp per vector by twisted factorisation (accepted when every residual is at
      // rounding level); otherwise in chunks by inverse iteration (thread per vector) with Gram-Schmidt inside clusters
      const double tiny = fmax(tnorm, 1.0) * 1.1e-16;
      bool fast_ok = false;
#ifndef DG_HOSTSIM
      if (n >= 33 && n <= 128 && (c.nt() & 31) == 0 && pivmin < 2.2250738585072014e-308 * 1.3e36) {
        bool sep = true;
        for (int jj = 1; jj < nneg; ++jj) if (fabs(B.lam[jj] - B.lam[jj - 1]) <= 1e-3 * tnorm) sep = false;
        if (sep) {
          if (c.tid() == 0) cnts[0] = 0;
          c.sync();
          const double tol = 8e-15 * fmax(tnorm, 1.0);     // true residual of the unit vector: what inverse iteration reaches
          for (int jv = c.warp(); jv < nneg; jv += c.nwarps()) {
            double shift = 0.0;
            const double res = n <= 64 ? twisted_eigvec<2>(c, n, B.dg, B.od, B.od2, B.lam[jv], pivmin, Z + (size_t)jv * n, shift)
                                       : twisted_eigvec<4>(c, n, B.dg, B.od, B.od2, B.lam[jv], pivmin, Z + (size_t)jv * n, shift);
            if (c.lane() == 0 && !(res <= tol)) cnts[0] = 1;
          }
          c.sync();
          fast_ok = cnts[0] == 0;
          c.sync();                              // (the flag word is scratch of the inverse iteration below)
        }
      }
#endif
      for (int j0 = 0; j0 < nneg && !fast_ok; j0 += CH) {
        const int kc = nneg - j0 < CH ? nneg - j0 : CH;
        bool cluster = false;
        for (int jj = 1; jj < kc; ++jj)
          if (fabs(B.lam[j0 + jj] - B.lam[j0 + jj - 1]) <= 1e-3 * tnorm) cluster = true;
        // a cluster may straddle the chunk boundary: the vectors the previous chunks finished (vector-major in Z) take part
        // in the Gram-Schmidt of this chunk
        const bool cross = j0 > 0 && fabs(B.lam[j0] - B.lam[j0 - 1]) <= 1e-3 * tnorm;
        cluster = cluster || cross;
        for (int itn = 0; itn < DG_EIG_INVIT; ++itn) {
          DG_FOR(jj, kc) {
            // (the stride is a compile-time constant on the common path: the serial chains index six arrays with it)
            if (SM || st == CH) invit_sweep(n, B.dg, B.od, B.lam[j0 + jj], tiny, itw + jj, Zt + jj, CH, itn == 0, j0 + jj);
            else invit_sweep(n, B.dg, B.od, B.lam[j0 + jj], tiny, itw + jj, Zt + jj, st, itn == 0, j0 + jj);
          }
          c.sync();
          if (cluster) {
            if (c.warp() == 0) {                   // modified Gram-Schmidt inside clusters, lanes along the vectors
              for (int jj = cross ? 0 : 1; jj < kc; ++jj) {
                double* z = Zt + jj;
                bool changed = false;
                for (int ip = j0 - 1; cross && ip >= 0; --ip) {      // finished vectors of earlier chunks (eigenvalues ascend)
                  if (fabs(B.lam[j0 + jj] - B.lam[ip]) > 1e-3 * tnorm) break;
                  const double* zp = Z + (size_t)ip * n;
                  double dt = 0.0;
                  for (int i = c.lane(); i < n; i += c.wsz) dt += zp[i] * z[i * st];
                  dt = c.warp_sum(dt);
                  for (int i = c.lane(); i < n; i += c.wsz) z[i * st] -= dt * zp[i];
                  c.syncwarp();
                  changed = true;
                }
                for (int ii = 0; ii < jj; ++ii) {
                  if (fabs(B.lam[j0 + jj] - B.lam[j0 + ii]) > 1e-3 * tnorm) continue;
                  const double* zi = Zt + ii;
                  double dt = 0.0;
                  for (int i = c.lane(); i < n; i += c.wsz) dt += zi[i * st] * z[i * st];
                  dt = c.warp_sum(dt);
                  for (int i = c.lane(); i < n; i += c.wsz) z[i * st] -= dt * zi[i * st];
                  c.syncwarp();
                  changed = true;
                }
                if (changed) {
                  double nr = 0.0;
                  for (int i = c.lane(); i < n; i += c.wsz) nr += z[i * st] * z[i * st];
                  nr = 1.0 / sqrt(c.warp_sum(nr));
                  for (int i = c.lane(); i < n; i += c.wsz) z[i * st] *= nr;
                  c.syncwarp();
                }
              }
            }
            c.sync();
          }
        }
        // de-interleave the chunk into the vector-major store
        for (int e = c.tid(); e < kc * n; e += c.nt()) { int jj = e / n, i = e - jj * n; Z[(size_t)(j0 + jj) * n + i] = Zt[i * st + jj]; }
        c.sync();
      }
      c.lapf(PH_PD_INVIT);
      // back-transform y = H_0 H_1 ... H_{n-2} z (last reflector first): one warp per eigenvector, no CTA barrier inside
#ifndef DG_HOSTSIM
      if (n <= 64) backtransform_regs<2>(c, n, ld, Hm, B.tau, Z, nneg);
      else if (n <= 128) backtransform_regs<4>(c, n, ld, Hm, B.tau, Z, nneg);
      else if (n <= 256) backtransform_regs<8>(c, n, ld, Hm, B.tau, Z, nneg);
      else
#endif
      for (int jv = c.warp(); jv < nneg; jv += c.nwarps()) {
        double* DG_RESTRICT z = Z + (size_t)jv * n;
        for (int k = n - 3; k >= 0; --k) {
          const double tk = B.tau[k];
          if (tk == 0.0) continue;
          const int len = n - k - 1;
          const double* DG_RESTRICT vcol = Hm + (k + 1) * ld + k;
          double pp = 0.0;
          for (int i = c.lane(); i < len; i += c.wsz) pp += (i == 0 ? 1.0 : vcol[i * ld]) * z[k + 1 + i];
          pp = c.warp_sum(pp) * tk;
          for (int i = c.lane(); i < len; i += c.wsz) z[k + 1 + i] -= pp * (i == 0 ? 1.0 : vcol[i * ld]);
          c.syncwarp();
        }
      }
      c.sync();
      c.lapf(PH_PD_BACK);
      Zall = Z;
    }
  }
  // H = sym(Q) + sum_j (floor - lam_j) y_j y_j' + reg I   (the reflectors in matA are dead now)
  // (Qraw is streamed from L2: the loads of four entries are issued before the first is used)
  for (int t0 = c.tid(); t0 < n * n; t0 += 4 * c.nt()) {
    double q1[4], q2[4];
    int ii[4], jj[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int t = t0 + u * c.nt();
      ii[u] = t / n; jj[u] = t - ii[u] * n;
      const bool in = t < n * n;
      q1[u] = in ? Qraw[ii[u] * n + jj[u]] : 0.0; q2[u] = in ? Qraw[jj[u] * n + ii[u]] : 0.0;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (t0 + u * c.nt() < n * n) {
        const int i = ii[u], j = jj[u];
        double acc = 0.5 * (q1[u] + q2[u]);
        for (int jv = 0; jv < nneg; ++jv) acc += (floor_val - B.lam[jv]) * Zall[(size_t)jv * n + i] * Zall[(size_t)jv * n + j];
        if (i == j) acc += reg;
        Hm[i * ld + j] = acc;
      }
    }
  }
  c.sync();
  c.lap(PH_PD_EIG);
  return nneg;
}

// In-place lower Cholesky of the symmetric matrix Hm (row-major, leading dimension ld), blocked right-looking with
// the panel (n x NB) staged in `sp`.  Per panel: warp 0 factors the NB x NB diagonal block (warp-level
// synchronisation only), then thread r solves its own panel row against it, then the trailing lower triangle is
// updated by the whole CTA.  Four barriers per panel.  scr: NB + 1 doubles of scratch.
// Returns false (uniformly) on a non-positive pivot.
// kstop (a multiple of the panel width) < n: only the panels below kstop are factored; the lower triangle of the trailing
// matrix is left updated for a register-tile continuation (qp_factor).
template <bool SM>
DG_DEVN bool cholesky_lower(Cta& c, int n, int ld, double* DG_RESTRICT Hm, double* DG_RESTRICT sp, double* DG_RESTRICT scr, int kstop) {
  DG_ASSUME_SHARED(Hm); DG_ASSUME_SHARED(sp); DG_ASSUME_SHARED(scr);
  constexpr int NB = DG_CHOL_NB;
  for (int k0 = 0; k0 < n && k0 < kstop; k0 += NB) {
    const int nb = n - k0 < NB ? n - k0 : NB;
    const int rows = n - k0;
    // stage panel rows k0.. : sp[(i-k0)*NB + t] = Hm[i][k0+t]
    for (int e = c.tid(); e < rows * NB; e += c.nt()) {
      int r = e / NB, t = e - r * NB;
      sp[e] = t < nb ? Hm[(k0 + r) * ld + k0 + t] : 0.0;
    }
    c.sync();
    if (c.warp() == 0) {
      bool ok = true;
      for (int kk = 0; kk < nb; ++kk) {
        double piv = sp[kk * NB + kk];
        for (int t = 0; t < kk; ++t) piv -= sp[kk * NB + t] * sp[kk * NB + t];
        if (!(piv > 0.0)) ok = false;
        const double inv = DG_RSQRT(piv);
        c.syncwarp();                               // pivot read by every lane before it is overwritten
        for (int r = kk + c.lane(); r < nb; r += c.wsz) {
          double v;
          if (r == kk) { v = piv * inv; scr[kk] = inv; }          // sqrt(piv)
          else {
            v = sp[r * NB + kk];
            for (int t = 0; t < kk; ++t) v -= sp[r * NB + t] * sp[kk * NB + t];
            v *= inv;
          }
          sp[r * NB + kk] = v;
        }
        c.syncwarp();
      }
      if (c.lane() == 0) scr[NB] = ok ? 1.0 : 0.0;
    }
    c.sync();
    if (scr[NB] == 0.0) return false;
    // panel rows below the diagonal block: x Ld' = a, row by row (thread = row)
    for (int r = nb + c.tid(); r < rows; r += c.nt()) {
      double x[NB];
#pragma unroll
      for (int kk = 0; kk < NB; ++kk) {
        double v = sp[r * NB + kk];
#pragma unroll
        for (int t = 0; t < kk; ++t) v -= x[t] * sp[kk * NB + t];
        x[kk] = kk < nb ? v * scr[kk] : 0.0;
      }
#pragma unroll
      for (int t = 0; t < NB; ++t) sp[r * NB + t] = x[t];
    }
    c.sync();
    // write the finished panel back (upper part of the diagonal block is left untouched: never read)
    for (int e = c.tid(); e < rows * NB; e += c.nt()) {
      int r = e / NB, t = e - r * NB;
      if (t < nb && t <= r) Hm[(k0 + r) * ld + k0 + t] = sp[e];
    }
    // trailing update of the lower triangle, spread over all threads: work item (gi, jl) owns column
    // j = j0 + jl and the rows i = j + gi, j + gi + groups, ...  (a warp shares i: the panel row is a broadcast)
    const int j0 = k0 + nb;
    const int ncol = n - j0;
    if (ncol > 0) {
      int groups = c.nt() / ncol;
      if (groups < 1) groups = 1;
      for (int e = c.tid(); e < ncol * groups; e += c.nt()) {
        const int gi = e / ncol, j = j0 + (e - gi * ncol);
        double lj[NB];
#pragma unroll
        for (int t = 0; t < NB; ++t) lj[t] = sp[(j - k0) * NB + t];
        double* DG_RESTRICT col = Hm + j;
        for (int i = j + gi; i < n; i += groups) {
          const double* DG_RESTRICT r0 = sp + (i - k0) * NB;
          double s0 = 0.0, s1 = 0.0;                   // two chains instead of one 8-deep dependent one
#pragma unroll
          for (int t = 0; t < NB; t += 2) { s0 += r0[t] * lj[t]; s1 += r0[t + 1] * lj[t + 1]; }
          col[i * ld] -= s0 + s1;
        }
      }
    }
    c.sync();
  }
  return true;
}

#ifndef DG_HOSTSIM
// ---- Cholesky and triangular inverse on 2D register tiles (256-thread CTAs, n <= 16*T <= 128) -------------------------
// Same 16 x 16 thread grid and cyclic tiles as sym_tridiag_tiles: the column-per-thread forms above move ~n/2 doubles
// per THREAD and step through shared memory (the LSU, not the FP64 pipe, bounds them); a tile needs the T entries of the
// step's column that belong to its rows and the T that belong to its columns.
// Cholesky, iteration k (one barrier): the raw column k (published by its holders in the previous iteration) gives
// 1/sqrt(d) and l = x/sqrt(d) for the thread's rows and columns; beside that dependent chain the rank-1 update of step
// k - 1 is finished (all tile columns but the one done early); then the tile column that contains column k + 1 is updated,
// its holders publish column k + 1, barrier.  L is written column by column into W (lower triangle).
template <int T, int S, bool SM>
DG_DEV bool chol_tile_iter(Cta& c, int n, int k, int ld, double (&a)[T][T], double* DG_RESTRICT W, double* DG_RESTRICT xs2,
                           double (&lrp)[T], double (&lcp)[T]) {
  const int tj = c.tid() & 15, ti = c.tid() >> 4;
  const double* DG_RESTRICT xs = xs2 + (k & 1) * 128;
  double* DG_RESTRICT xn = xs2 + ((k & 1) ^ 1) * 128;
  const double d = xs[k];
  double xr[T], xc[T];
#pragma unroll
  for (int r = S; r < T; ++r) { xr[r] = xs[ti + 16 * r]; xc[r] = xs[tj + 16 * r]; }
  // finish step k - 1 beside the reciprocal square root
#pragma unroll
  for (int r = S; r < T; ++r)
#pragma unroll
    for (int cb = S + 1; cb < T; ++cb) a[r][cb] = fma(-lrp[r], lcp[cb], a[r][cb]);
  if (!(d > 0.0)) return false;
  const double inv = DG_RSQRT(d);
#pragma unroll
  for (int r = S; r < T; ++r) { lrp[r] = xr[r] * inv; lcp[r] = xc[r] * inv; }
  if (tj == (k & 15)) {
#pragma unroll
    for (int r = S; r < T; ++r) { const int j = ti + 16 * r; if (j >= k && j < n) W[j * ld + k] = lrp[r]; }
  }
  if (k + 1 < n) {
    const bool same = ((k + 1) >> 4) == S;
    if (same) {
#pragma unroll
      for (int r = S; r < T; ++r) a[r][S] = fma(-lrp[r], lcp[S], a[r][S]);
    } else if constexpr (S + 1 < T) {
#pragma unroll
      for (int r = S; r < T; ++r) a[r][S + 1] = fma(-lrp[r], lcp[S + 1], a[r][S + 1]);
    }
    if (tj == ((k + 1) & 15)) {
#pragma unroll
      for (int r = 0; r < T; ++r) {
        const int j = ti + 16 * r;
        double val = 0.0;
        if (r >= S && j > k && j < n) {
          if constexpr (S + 1 < T) val = same ? a[r][S] : a[r][S + 1];
          else val = a[r][S];
        }
        xn[j] = val;
      }
    }
  }
  c.sync();
  return true;
}
#define DG_CHT_CASE(m) case m: if constexpr (m < T) ok = chol_tile_iter<T, m, SM>(c, n, k, ld, a, W, xs2, lrp, lcp); break;
// lower_only: the matrix is valid in its lower triangle only (continuation of cholesky_lower): the tiles mirror it.
template <int T, bool SM>
DG_DEVN bool cholesky_tiles(Cta& c, int n, const LinBuf& B_, bool lower_only) {
  const LinBuf B = B_; DG_SH_LIN_T(B);
  double* DG_RESTRICT W = B.matA;
  const int ld = B.ld;
  const int tj = c.tid() & 15, ti = c.tid() >> 4;
  double* DG_RESTRICT xs2 = B.part;                               // two buffers of 128: raw column of the iteration
  double a[T][T], lrp[T], lcp[T];
#pragma unroll
  for (int r = 0; r < T; ++r) {
    lrp[r] = 0.0; lcp[r] = 0.0;
#pragma unroll
    for (int cb = 0; cb < T; ++cb) {
      const int j = ti + 16 * r, i = tj + 16 * cb;
      a[r][cb] = (j < n && i < n) ? ((lower_only && i > j) ? W[i * ld + j] : W[j * ld + i]) : 0.0;
    }
  }
  DG_FOR(t, 256) xs2[t] = 0.0;
  c.sync();
  if (tj == 0) {
#pragma unroll
    for (int r = 0; r < T; ++r) { const int j = ti + 16 * r; if (j < n) xs2[j] = a[r][0]; }
  }
  c.sync();
  bool ok = true;
  for (int k = 0; k < n && ok; ++k) {
    switch (k >> 4) { DG_CHT_CASE(0) DG_CHT_CASE(1) DG_CHT_CASE(2) DG_CHT_CASE(3) DG_CHT_CASE(4) DG_CHT_CASE(5) DG_CHT_CASE(6) DG_CHT_CASE(7) default: break; }
  }
  c.sync();
  return ok;
}
#undef DG_CHT_CASE

// Triangular inverse Y = L^-1 on tiles: the tiles start as the identity and carry  e_i - sum_{j<k} L[i][j] Y[j][:] ; iteration
// k reads the final row k of Y (published by its holders in the previous iteration) and column k of L (straight from W,
// broadcast inside a thread row), finishes the update of step k - 1 beside those loads, updates the tile row that contains
// row k + 1, whose holders scale it by 1/L[k+1][k+1], publish it and store it as row k + 1 of Y.  One barrier per iteration.
template <int T, int S, bool SM>
DG_DEV void trinv_tile_iter(Cta& c, int n, int k, int ld, double (&a)[T][T], const double* DG_RESTRICT W, double* DG_RESTRICT Y,
                            double* DG_RESTRICT xr2, const double* DG_RESTRICT rdiag, double (&mp)[T], double (&yp)[T]) {
  const int tj = c.tid() & 15, ti = c.tid() >> 4;
  const double* DG_RESTRICT xrow = xr2 + (k & 1) * 128;
  double* DG_RESTRICT xnext = xr2 + ((k & 1) ^ 1) * 128;
  double m[T], yk[T];
#pragma unroll
  for (int r = S; r < T; ++r) { const int i = ti + 16 * r; m[r] = (i > k && i < n) ? W[i * ld + k] : 0.0; }
#pragma unroll
  for (int cb = 0; cb <= S; ++cb) yk[cb] = xrow[tj + 16 * cb];
  // finish step k - 1: tile rows above the one done early
#pragma unroll
  for (int r = S + 1; r < T; ++r)
#pragma unroll
    for (int cb = 0; cb <= S; ++cb) a[r][cb] = fma(-mp[r], yp[cb], a[r][cb]);
  if (k + 1 < n) {
    const bool same = ((k + 1) >> 4) == S;
    const double rd = rdiag[k + 1];
    if (same) {
#pragma unroll
      for (int cb = 0; cb <= S; ++cb) a[S][cb] = fma(-m[S], yk[cb], a[S][cb]);
    } else if constexpr (S + 1 < T) {
#pragma unroll
      for (int cb = 0; cb <= S; ++cb) a[S + 1][cb] = fma(-m[S + 1], yk[cb], a[S + 1][cb]);
    }
    if (ti == ((k + 1) & 15)) {
#pragma unroll
      for (int cb = 0; cb < T; ++cb) {
        const int i = tj + 16 * cb;
        double val = 0.0;
        if (cb <= S + 1 && i <= k + 1) {
          if constexpr (S + 1 < T) val = (same ? a[S][cb] : a[S + 1][cb]) * rd;
          else val = a[S][cb] * rd;
        }
        xnext[i] = val;
        if (i < n) Y[(k + 1) * ld + i] = val;
      }
    }
  }
#pragma unroll
  for (int r = S; r < T; ++r) mp[r] = m[r];
#pragma unroll
  for (int cb = 0; cb <= S; ++cb) yp[cb] = yk[cb];
  c.sync();
}
#define DG_TIT_CASE(m) case m: if constexpr (m < T) trinv_tile_iter<T, m, SM>(c, n, k, ld, a, W, Y, xr2, rdiag, mp, yp); break;
template <int T, bool SM>
DG_DEVN void tri_inverse_tiles(Cta& c, int n, const LinBuf& B_) {
  const LinBuf B = B_; DG_SH_LIN_T(B);
  const double* DG_RESTRICT W = B.matA;
  double* DG_RESTRICT Y = B.matB;
  const int ld = B.ld;
  const int tj = c.tid() & 15, ti = c.tid() >> 4;
  double* DG_RESTRICT xr2 = B.part;                               // two buffers of 128: final row k of Y
  double* DG_RESTRICT rdiag = B.part + 256;                       // 1 / L[k][k]
  double a[T][T], mp[T], yp[T];
#pragma unroll
  for (int r = 0; r < T; ++r) {
    mp[r] = 0.0; yp[r] = 0.0;
#pragma unroll
    for (int cb = 0; cb < T; ++cb) a[r][cb] = (ti + 16 * r == tj + 16 * cb) ? 1.0 : 0.0;
  }
  DG_FOR(t, 256) xr2[t] = 0.0;
  DG_FOR(t, n) rdiag[t] = 1.0 / W[t * ld + t];
  c.sync();
  if (ti == 0) {
    // row 0 of Y: (1 / L00, 0, ..)
#pragma unroll
    for (int cb = 0; cb < T; ++cb) { const int i = tj + 16 * cb; const double val = i == 0 ? rdiag[0] : 0.0; if (i < 128) xr2[i] = val; if (i < n) Y[i] = val; }
  }
  c.sync();
  for (int k = 0; k < n; ++k) {
    switch (k >> 4) { DG_TIT_CASE(0) DG_TIT_CASE(1) DG_TIT_CASE(2) DG_TIT_CASE(3) DG_TIT_CASE(4) DG_TIT_CASE(5) DG_TIT_CASE(6) DG_TIT_CASE(7) default: break; }
  }
}
#undef DG_TIT_CASE

template <bool SM>
DG_DEV bool cholesky_tiles_dispatch(Cta& c, int n, const LinBuf& B, bool& ok) {
  if (c.nt() != 256 || n < 33 || n > 128) return false;
  switch ((n + 15) >> 4) {
    case 3: ok = cholesky_tiles<3, SM>(c, n, B, false); break;
    case 4: ok = cholesky_tiles<4, SM>(c, n, B, false); break;
    case 5: ok = cholesky_tiles<5, SM>(c, n, B, false); break;
    case 6: ok = cholesky_tiles<6, SM>(c, n, B, false); break;
    case 7: ok = cholesky_tiles<7, SM>(c, n, B, false); break;
    default: ok = cholesky_tiles<8, SM>(c, n, B, false); break;
  }
  return true;
}
template <bool SM>
DG_DEV bool tri_inverse_tiles_dispatch(Cta& c, int n, const LinBuf& B) {
  if (c.nt() != 256 || n < 33 || n > 128) return false;
  switch ((n + 15) >> 4) {
    case 3: tri_inverse_tiles<3, SM>(c, n, B); break;
    case 4: tri_inverse_tiles<4, SM>(c, n, B); break;
    case 5: tri_inverse_tiles<5, SM>(c, n, B); break;
    case 6: tri_inverse_tiles<6, SM>(c, n, B); break;
    case 7: tri_inverse_tiles<7, SM>(c, n, B); break;
    default: tri_inverse_tiles<8, SM>(c, n, B); break;
  }
  return true;
}

#endif


// Y = L^{-1} (lower triangular; L and Y row-major with leading dimension ld: Y[i][c]; the strict upper triangle of Y
// is zero-filled because the active-set solver treats Y as dense).  Blocked by NB = 8 rows:
//   diagonal blocks   Y_bb = L_bb^{-1}                       thread per column, 8-step chains, reciprocals hoisted
//   block row i >= 1  M = Y_ii L_i,0:i   (8 x 8i)            item per entry, <= 8 FMAs
//                     Y_i,0:i = -M Y_0:i,0:i                 item per entry: dot product over the rows c..8i of column c
// Two barriers per block row; every O(n^3) product is spread over the whole CTA (the column-recursive form it
// replaces kept one lane pair per column busy for n dependent dot products).
// Mi: 8*n doubles of scratch, rdiag: n doubles.  The GI solver uses J = L^{-T} = Y' through J(i,j) = Y[j*ld+i].
template <bool SM>
DG_DEVN void tri_inverse(Cta& c, int n, int ld, const double* DG_RESTRICT Lm, double* DG_RESTRICT Y,
                         double* DG_RESTRICT Mi, double* DG_RESTRICT rdiag) {
  DG_ASSUME_SHARED(Lm); DG_ASSUME_SHARED(Y); DG_ASSUME_SHARED(Mi); DG_ASSUME_SHARED(rdiag);
  constexpr int NB = 8;
  const int nblk = (n + NB - 1) / NB;
  DG_FOR(i, n) rdiag[i] = 1.0 / Lm[i * ld + i];
  DG_FOR(t, n * n) { const int i = t / n, j = t - i * n; if (j > i) Y[i * ld + j] = 0.0; }
  c.sync();
  DG_FOR(cc, n) {
    const int b = cc / NB, end = (b + 1) * NB < n ? (b + 1) * NB : n;
    Y[cc * ld + cc] = rdiag[cc];
    for (int i = cc + 1; i < end; ++i) {
      double acc = 0.0;
      for (int j = cc; j < i; ++j) acc += Lm[i * ld + j] * Y[j * ld + cc];
      Y[i * ld + cc] = -acc * rdiag[i];
    }
  }
  c.sync();
  for (int ib = 1; ib < nblk; ++ib) {
    const int r0 = ib * NB, nb = n - r0 < NB ? n - r0 : NB, w = r0;
    for (int e = c.tid(); e < nb * w; e += c.nt()) {
      const int r = e / w, t = e - r * w;
      const double* DG_RESTRICT Yr = Y + (r0 + r) * ld + r0;
      double acc = 0.0;
      for (int s2 = 0; s2 <= r; ++s2) acc += Yr[s2] * Lm[(r0 + s2) * ld + t];
      Mi[e] = acc;
    }
    c.sync();
    for (int e = c.tid(); e < nb * w; e += c.nt()) {
      const int r = e / w, cc = e - r * w;
      const double* DG_RESTRICT Mr = Mi + r * w;
      double a0 = 0.0, a1 = 0.0;
      int t = w - 1;
      for (; t - 1 >= cc; t -= 2) { a0 += Mr[t] * Y[t * ld + cc]; a1 += Mr[t - 1] * Y[(t - 1) * ld + cc]; }
      if (t >= cc) a0 += Mr[t] * Y[t * ld + cc];
      Y[(r0 + r) * ld + cc] = -(a0 + a1);
    }
    c.sync();
  }
}
