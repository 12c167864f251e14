// Stage-level test kernel: runs single stages of the solver -- evaluate -> nearestPD -> QP and the LSQR dual
// initialisation, nearestPD of an arbitrary matrix, the QP factorisation, a cold and a warm QP with an arbitrary
// Hessian (and optionally arbitrary constraint offsets and warm-start list), the warm start alone, the matrix-free G
// products -- for a batch of instances (one CTA each) and returns every intermediate together with the memory plan it
// ran with.  TEST ONLY (tests/test_gpu_units.py, tests/test_gpu_qp.py, tests/test_gpu_parity.py).
// Compiled once per game: -DDG_GAME_MERGE selects the merge game (csrc/game.cuh).
#include <cuda_runtime.h>
#include <cstdio>
#include <vector>
#include "../../dgsqp_b200/csrc/sqp_v1.cuh"
#include "../../dgsqp_b200/csrc/host_setup.h"

enum { U_STAGES = 0, U_NEAREST_PD = 1, U_FACTOR = 2, U_QP = 3, U_G = 4, U_WARM = 5 };

struct UnitArgs {
  int B, mode, nrows;
  const double *x0, *u, *l;              // evaluation point (U_STAGES, U_QP, U_G)
  const double *Hin, *qin, *q2in;        // nearestPD input (U_NEAREST_PD); QP Hessian and gradients (U_FACTOR, U_QP)
  const double *v, *w; const int* rows;  // U_G: G v, G' w, rows / columns of G
  const double* gin;                     // U_QP, U_WARM: constraint offsets [B, m] in place of the evaluated g (or null)
  const int *prev, *kprev; int kmax;     // U_QP, U_WARM: warm-start list prev[B, kmax], kprev[b] ids of it (or null)
  double *Q, *q, *gtl, *g, *H, *du, *lam, *l0, *du2, *lam2, *L, *Y, *Gv, *GTw, *Grow, *Gcol, *lam_act;
  int *nneg, *qpst, *qpit, *lsqr_it, *qpst2, *qpit2, *qpna, *qpna2, *ok, *eig_s, *act, *iq;
  double* ws; size_t ws_stride; size_t smem_doubles;
};

template <bool SM>
__global__ void __launch_bounds__(256, 1) units_kernel(const GameDesc* Gp, const SolverParams* Pp, UnitArgs A) {
  extern __shared__ double s_dyn[];
  Cta c;
  c.flip = 0;
  __shared__ SolveCtx sX;
  if (threadIdx.x == 0) {
    sX.G = Gp; sX.P = Pp; sX.D = make_dims(Gp->M, Gp->N);
    plan_memory(sX.D, A.ws + (size_t)blockIdx.x * A.ws_stride, s_dyn, A.smem_doubles, sX.W);
    game_bind(sX.W.E, Gp);
    if (blockIdx.x == 0) *A.eig_s = sX.W.B.eig_s != nullptr;
  }
  __syncthreads();
  SolveCtx& X = sX;
  const Dims& D = X.D; const int n = D.n, m = D.m, ld = D.ld;
  double* matA = X.W.B.matA; double* matB = X.W.B.matB;
  game_row_table<SM>(c, D, X.W.E.rowtab);
  for (int inst = blockIdx.x; inst < A.B; inst += gridDim.x) {
    c.sync();
    const double* u = A.u ? A.u + (size_t)inst * n : nullptr;
    const double* l = A.l ? A.l + (size_t)inst * m : nullptr;
    if (A.mode == U_STAGES || A.mode == U_QP || A.mode == U_G || A.mode == U_WARM) {
      if (threadIdx.x == 0) X.x0 = A.x0 + (size_t)inst * D.nq;
      DG_FOR(j, D.nu) X.W.S.up[j] = 0.0;
      c.sync();
      eval_full<SM>(c, X, u, l);
      c.sync();
      DG_FOR(t, n * n) A.Q[(size_t)inst * n * n + t] = X.W.E.Q[t];
      DG_FOR(t, n) { A.q[(size_t)inst * n + t] = X.W.E.q[t]; A.gtl[(size_t)inst * n + t] = X.W.E.gtl[t]; }
      DG_FOR(t, m) A.g[(size_t)inst * m + t] = X.W.E.g[t];
      c.sync();
      if (A.gin) { DG_FOR(t, m) X.W.E.g[t] = A.gin[(size_t)inst * m + t]; }
      const int kp = A.prev ? A.kprev[inst] : 0;
      DG_FOR(t, kp) X.W.Q.act[t] = A.prev[(size_t)inst * A.kmax + t];
      if (c.tid() == 0) X.W.Q.act[n] = kp;
      c.sync();
    }
    if (A.mode == U_STAGES) {
      int nneg = nearest_pd<SM>(c, n, X.W.E.Q, X.W.B, Pp->eig_floor, Pp->reg, Pp->conv_approx != 0);
      DG_FOR(t, n * n) A.H[(size_t)inst * n * n + t] = matA[(t / n) * ld + (t % n)];
      c.sync();
      int it = 0, na = 0;
      int st = qp_solve_gi<SM>(c, D, X.W.E, X.W.E.q, X.W.Q, X.W.B, &it, &na, 0);
      DG_FOR(t, n) A.du[(size_t)inst * n + t] = X.W.Q.xq[t];
      DG_FOR(t, m) A.lam[(size_t)inst * m + t] = X.W.Q.lam[t];
      c.sync();
      DG_FOR(t, m) X.W.S.l[t] = 0.0;
      c.sync();
      eval_grad<SM>(c, X, u, X.W.S.l, true);
      int li = lsqr_dual_init<SM>(c, D, X.W.E, X.W.L, X.W.E.q, X.W.S.l);
      DG_FOR(t, m) A.l0[(size_t)inst * m + t] = X.W.S.l[t];
      if (c.tid() == 0) { A.nneg[inst] = nneg; A.qpst[inst] = st; A.qpit[inst] = it; A.lsqr_it[inst] = li; }
    } else if (A.mode == U_NEAREST_PD) {
      // the raw matrix goes where the evaluation leaves it (global workspace)
      DG_FOR(t, n * n) X.W.E.Q[t] = A.Hin[(size_t)inst * n * n + t];
      c.sync();
      int nneg = nearest_pd<SM>(c, n, X.W.E.Q, X.W.B, Pp->eig_floor, Pp->reg, Pp->conv_approx != 0);
      DG_FOR(t, n * n) A.H[(size_t)inst * n * n + t] = matA[(t / n) * ld + (t % n)];
      if (c.tid() == 0) A.nneg[inst] = nneg;
    } else if (A.mode == U_FACTOR) {
      DG_FOR(t, n * n) matA[(t / n) * ld + (t % n)] = A.Hin[(size_t)inst * n * n + t];
      // a finite non-zero fill: the factorisation has to write the zero strict upper triangle of Y itself (the solver
      // treats Y as dense, and matB holds the eigenvector scratch of nearest_pd before)
      DG_FOR(t, n * ld) matB[t] = 3.0;
      DG_FOR(t, n) X.W.E.q[t] = A.qin[(size_t)inst * n + t];
      c.sync();
      const bool ok = qp_factor<SM>(c, D, X.W.E.q, X.W.Q, X.W.B);
      c.sync();
      DG_FOR(t, n * n) {
        const int i = t / n, j = t - i * n;
        A.L[(size_t)inst * n * n + t] = j <= i ? matA[i * ld + j] : 0.0;
        A.Y[(size_t)inst * n * n + t] = matB[i * ld + j];
      }
      DG_FOR(t, n) A.du[(size_t)inst * n + t] = X.W.Q.xq[t];
      if (c.tid() == 0) A.ok[inst] = ok;
    } else if (A.mode == U_QP) {
      // QP at (H, q) on the evaluated constraints (or on gin), cold or from the list prev; then, with q2, a warm QP
      // from the first QP's active set
      for (int pass = 0; pass < (A.q2in ? 2 : 1); ++pass) {
        const double* qi = (pass == 0 ? A.qin : A.q2in) + (size_t)inst * n;
        DG_FOR(t, n * n) matA[(t / n) * ld + (t % n)] = A.Hin[(size_t)inst * n * n + t];
        DG_FOR(t, n) X.W.E.q[t] = qi[t];
        c.sync();
        int it = 0, na = 0;
        const int st = qp_solve_gi<SM>(c, D, X.W.E, X.W.E.q, X.W.Q, X.W.B, &it, &na, pass > 0 || A.prev);
        c.sync();
        DG_FOR(t, n) (pass == 0 ? A.du : A.du2)[(size_t)inst * n + t] = X.W.Q.xq[t];
        DG_FOR(t, m) (pass == 0 ? A.lam : A.lam2)[(size_t)inst * m + t] = X.W.Q.lam[t];
        if (c.tid() == 0) {
          (pass == 0 ? A.qpst : A.qpst2)[inst] = st; (pass == 0 ? A.qpit : A.qpit2)[inst] = it;
          (pass == 0 ? A.qpna : A.qpna2)[inst] = na;
        }
        c.sync();
      }
    } else if (A.mode == U_WARM) {
      // qp_factor and gi_warm_start from prev only: the S-pair (act[0..iq), xq, lam_act[0..iq)) the main loop starts from
      DG_FOR(t, n * n) matA[(t / n) * ld + (t % n)] = A.Hin[(size_t)inst * n * n + t];
      DG_FOR(t, n) X.W.E.q[t] = A.qin[(size_t)inst * n + t];
      c.sync();
      int iq = -1;
      if (qp_factor<SM>(c, D, X.W.E.q, X.W.Q, X.W.B)) {
        const int kp = X.W.Q.act[n];
        iq = kp > 0 ? gi_warm_start<SM>(c, D, X.W.E, X.W.E.q, X.W.Q, X.W.B, kp) : 0;
      }
      c.sync();
      DG_FOR(t, n) A.du[(size_t)inst * n + t] = X.W.Q.xq[t];
      DG_FOR(t, n) {
        A.act[(size_t)inst * n + t] = t < iq ? X.W.Q.act[t] : -1;
        A.lam_act[(size_t)inst * n + t] = t < iq ? X.W.Q.lam_act[t] : 0.0;
      }
      if (c.tid() == 0) A.iq[inst] = iq;
    } else if (A.mode == U_G) {
      // the operands go where the solver keeps them (SQP iterate vectors, QP scratch, matA)
      DG_FOR(t, n) X.W.S.du[t] = A.v[(size_t)inst * n + t];
      DG_FOR(t, m) X.W.S.dl[t] = A.w[(size_t)inst * m + t];
      c.sync();
      game_G_times<SM>(c, D, X.W.E, X.W.S.du, X.W.S.Gdu);
      c.sync();
      game_GT_times<SM>(c, D, X.W.E, X.W.S.dl, X.W.S.tn);
      c.sync();
      DG_FOR(t, m) A.Gv[(size_t)inst * m + t] = X.W.S.Gdu[t];
      DG_FOR(t, n) A.GTw[(size_t)inst * n + t] = X.W.S.tn[t];
      const int* rows = A.rows + (size_t)inst * A.nrows;
      for (int k = 0; k < A.nrows; ++k) {
        c.sync();
        game_G_row<SM>(c, D, X.W.E, rows[k], X.W.Q.npv);
        DG_FOR(t, n) A.Grow[((size_t)inst * A.nrows + k) * n + t] = X.W.Q.npv[t];
      }
      int* ids = (int*)X.W.Q.rv;
      DG_FOR(k, A.nrows) ids[k] = rows[k];
      c.sync();
      game_G_cols<SM>(c, D, X.W.E, ids, A.nrows, matA, ld);
      c.sync();
      DG_FOR(t, A.nrows * n) { const int k = t / n, j = t - k * n; A.Gcol[((size_t)inst * A.nrows + k) * n + j] = matA[j * ld + k]; }
    }
    c.sync();
  }
}

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e)); return -2; } } while (0)

// device copies of the host arrays of one call; outputs are copied back by fetch(), everything is freed on exit
struct DevArrays {
  struct Out { void* h; void* d; size_t bytes; };
  std::vector<void*> all; std::vector<Out> outs; cudaError_t err = cudaSuccess;
  template <class T> T* in(const T* h, size_t cnt) {
    if (!h || err != cudaSuccess) return nullptr;
    void* d = nullptr;
    if ((err = cudaMalloc(&d, sizeof(T) * cnt)) != cudaSuccess) return nullptr;
    all.push_back(d);
    err = cudaMemcpy(d, h, sizeof(T) * cnt, cudaMemcpyHostToDevice);
    return (T*)d;
  }
  template <class T> T* zeros(size_t cnt) {
    if (err != cudaSuccess) return nullptr;
    void* d = nullptr;
    if ((err = cudaMalloc(&d, sizeof(T) * cnt)) != cudaSuccess) return nullptr;
    all.push_back(d);
    err = cudaMemset(d, 0, sizeof(T) * cnt);
    return (T*)d;
  }
  template <class T> T* out(T* h, size_t cnt) {
    if (!h) return nullptr;
    T* d = zeros<T>(cnt);
    if (d) outs.push_back({h, d, sizeof(T) * cnt});
    return d;
  }
  cudaError_t fetch() {
    for (const Out& o : outs) if (err == cudaSuccess) err = cudaMemcpy(o.h, o.d, o.bytes, cudaMemcpyDeviceToHost);
    return err;
  }
  ~DevArrays() { for (void* d : all) cudaFree(d); }
};

// smem_limit_doubles < 0: the device maximum; otherwise that many doubles of shared memory (at most the maximum).
// plan[5] = {hot_in_smem (the SM = true instantiation ran), mats_in_smem, matA_in_smem, sens_in_smem, eig_s set}
static int units_launch(const dg_game_struct* game, const dgsqp_params* params, int threads, long smem_limit_doubles,
                        UnitArgs& A, DevArrays& da, int* plan) {
  GameDesc G; SolverParams P;
  if (dg_fill_game(game, &G) || dg_fill_params(params, &P)) return -1;
  if (threads < 32 || threads > 256 || threads % 32) return -1;
  if (da.err != cudaSuccess) { fprintf(stderr, "units: %s\n", cudaGetErrorString(da.err)); return -2; }
  Dims D = make_dims(G.M, G.N);
  int optin = 0; CK(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, 0));
  cudaFuncAttributes fa; CK(cudaFuncGetAttributes(&fa, units_kernel<true>));
  size_t budget = ((size_t)optin - fa.sharedSizeBytes - 64) / sizeof(double);
  if (smem_limit_doubles >= 0 && (size_t)smem_limit_doubles < budget) budget = (size_t)smem_limit_doubles;
  Workspace tmp; MemPlan pl = plan_memory(D, nullptr, nullptr, budget, tmp);
  const int grid = A.B < 64 ? A.B : 64;
  GameDesc* dG = da.in(&G, 1); SolverParams* dP = da.in(&P, 1);
  A.ws = da.zeros<double>(pl.gmem * grid); A.ws_stride = pl.gmem; A.smem_doubles = budget;
  int eig_s = 0; A.eig_s = da.out(&eig_s, 1);
  if (da.err != cudaSuccess) { fprintf(stderr, "units: %s\n", cudaGetErrorString(da.err)); return -2; }
  cudaDeviceSetLimit(cudaLimitStackSize, 8192);
  size_t smem = sizeof(double) * pl.smem;
  if (pl.hot_in_smem) {
    CK(cudaFuncSetAttribute(units_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    units_kernel<true><<<grid, threads, smem>>>(dG, dP, A);
  } else {
    CK(cudaFuncSetAttribute(units_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    units_kernel<false><<<grid, threads, smem>>>(dG, dP, A);
  }
  CK(cudaGetLastError()); CK(cudaDeviceSynchronize());
  CK(da.fetch());
  plan[0] = pl.hot_in_smem; plan[1] = pl.mats_in_smem; plan[2] = pl.matA_in_smem; plan[3] = pl.sens_in_smem; plan[4] = eig_s;
  return 0;
}

static UnitArgs units_args(int B, int mode) { UnitArgs A = {}; A.B = B; A.mode = mode; return A; }

static Dims units_dims(const dg_game_struct* game) {
  GameDesc G;
  if (dg_fill_game(game, &G)) return make_dims(2, 2);
  return make_dims(G.M, G.N);
}

extern "C" {

// evaluate -> nearestPD -> QP at (u, l), and the LSQR dual initialisation at u
int units_run(const dg_game_struct* game, const dgsqp_params* params, int B, int threads, long smem_limit_doubles, const double* x0,
              const double* u, const double* l, double* Q, double* q, double* gtl, double* g, double* H,
              double* du, double* lam, double* l0, int* nneg, int* qpst, int* qpit, int* lsqr_it, int* plan) {
  const Dims D = units_dims(game); const size_t n = D.n, m = D.m;
  DevArrays da; UnitArgs A = units_args(B, U_STAGES);
  A.x0 = da.in(x0, B * D.nq); A.u = da.in(u, B * n); A.l = da.in(l, B * m);
  A.Q = da.out(Q, B * n * n); A.q = da.out(q, B * n); A.gtl = da.out(gtl, B * n); A.g = da.out(g, B * m); A.H = da.out(H, B * n * n);
  A.du = da.out(du, B * n); A.lam = da.out(lam, B * m); A.l0 = da.out(l0, B * m);
  A.nneg = da.out(nneg, B); A.qpst = da.out(qpst, B); A.qpit = da.out(qpit, B); A.lsqr_it = da.out(lsqr_it, B);
  return units_launch(game, params, threads, smem_limit_doubles, A, da, plan);
}

// H = nearestPD(Qin) + reg I of every Qin[B, n, n]
int units_nearest_pd(const dg_game_struct* game, const dgsqp_params* params, int B, int threads, long smem_limit_doubles,
                     const double* Qin, double* H, int* nneg, int* plan) {
  const Dims D = units_dims(game); const size_t n = D.n;
  DevArrays da; UnitArgs A = units_args(B, U_NEAREST_PD);
  A.Hin = da.in(Qin, B * n * n); A.H = da.out(H, B * n * n); A.nneg = da.out(nneg, B);
  return units_launch(game, params, threads, smem_limit_doubles, A, da, plan);
}

// qp_factor: ok, L (lower triangle, zero above), Y = L^-1 (all n x n entries as stored), xq = -H^-1 q
int units_factor(const dg_game_struct* game, const dgsqp_params* params, int B, int threads, long smem_limit_doubles,
                 const double* H, const double* q, int* ok, double* L, double* Y, double* xq, int* plan) {
  const Dims D = units_dims(game); const size_t n = D.n;
  DevArrays da; UnitArgs A = units_args(B, U_FACTOR);
  A.Hin = da.in(H, B * n * n); A.qin = da.in(q, B * n);
  A.ok = da.out(ok, B); A.L = da.out(L, B * n * n); A.Y = da.out(Y, B * n * n); A.du = da.out(xq, B * n);
  return units_launch(game, params, threads, smem_limit_doubles, A, da, plan);
}

// the optional constraint offsets gin[B, m] and warm-start lists prev[B, kmax] (kprev[b] ids each) of U_QP / U_WARM
static int units_qp_inputs(const Dims& D, int B, const double* gin, const int* prev, const int* kprev, int kmax,
                           UnitArgs& A, DevArrays& da) {
  if (prev) {
    if (!kprev || kmax < 1 || kmax > D.n) return -1;
    for (int b = 0; b < B; ++b) {
      if (kprev[b] < 0 || kprev[b] > kmax) return -1;
      for (int k = 0; k < kprev[b]; ++k) if (prev[(size_t)b * kmax + k] < 0 || prev[(size_t)b * kmax + k] >= D.m) return -1;
    }
    A.prev = da.in(prev, (size_t)B * kmax); A.kprev = da.in(kprev, B); A.kmax = kmax;
  }
  A.gin = da.in(gin, (size_t)B * D.m);
  return 0;
}

// evaluation at (x0, u, l) (constraints of the QP, offsets replaced by gin if given), a QP at (H, q) -- cold, or from
// the warm-start list prev if given -- and, if q2 is given, a warm QP at (H, q2) from the first QP's active set.
// it / na: main-loop iterations and active rows at the end
int units_qp(const dg_game_struct* game, const dgsqp_params* params, int B, int threads, long smem_limit_doubles,
             const double* x0, const double* u, const double* l, const double* H, const double* q, const double* q2,
             const double* gin, const int* prev, const int* kprev, int kmax,
             double* Q, double* qe, double* gtl, double* g, int* st, int* it, int* na, double* du, double* lam,
             int* st2, int* it2, int* na2, double* du2, double* lam2, int* plan) {
  const Dims D = units_dims(game); const size_t n = D.n, m = D.m;
  DevArrays da; UnitArgs A = units_args(B, U_QP);
  if (units_qp_inputs(D, B, gin, prev, kprev, kmax, A, da)) return -1;
  A.x0 = da.in(x0, B * D.nq); A.u = da.in(u, B * n); A.l = da.in(l, B * m);
  A.Hin = da.in(H, B * n * n); A.qin = da.in(q, B * n); A.q2in = da.in(q2, B * n);
  A.Q = da.out(Q, B * n * n); A.q = da.out(qe, B * n); A.gtl = da.out(gtl, B * n); A.g = da.out(g, B * m);
  A.qpst = da.out(st, B); A.qpit = da.out(it, B); A.qpna = da.out(na, B); A.du = da.out(du, B * n); A.lam = da.out(lam, B * m);
  if (q2) {
    A.qpst2 = da.out(st2, B); A.qpit2 = da.out(it2, B); A.qpna2 = da.out(na2, B);
    A.du2 = da.out(du2, B * n); A.lam2 = da.out(lam2, B * m);
  }
  return units_launch(game, params, threads, smem_limit_doubles, A, da, plan);
}

// evaluation at (x0, u, l) (offsets replaced by gin if given), qp_factor of H and gi_warm_start from prev: iq (-1: H
// not positive definite), act[B, n] (-1 from iq on), xq[B, n], lam_act[B, n] (0 from iq on)
int units_warm(const dg_game_struct* game, const dgsqp_params* params, int B, int threads, long smem_limit_doubles,
               const double* x0, const double* u, const double* l, const double* H, const double* q,
               const double* gin, const int* prev, const int* kprev, int kmax,
               int* iq, int* act, double* xq, double* lam_act, int* plan) {
  const Dims D = units_dims(game); const size_t n = D.n, m = D.m;
  DevArrays da; UnitArgs A = units_args(B, U_WARM);
  if (!prev || units_qp_inputs(D, B, gin, prev, kprev, kmax, A, da)) return -1;
  A.x0 = da.in(x0, B * D.nq); A.u = da.in(u, B * n); A.l = da.in(l, B * m);
  A.Hin = da.in(H, B * n * n); A.qin = da.in(q, B * n);
  A.iq = da.out(iq, B); A.act = da.out(act, B * n); A.du = da.out(xq, B * n); A.lam_act = da.out(lam_act, B * n);
  // the evaluation outputs of U_WARM go to scratch
  A.Q = da.zeros<double>(B * n * n); A.q = da.zeros<double>(B * n); A.gtl = da.zeros<double>(B * n); A.g = da.zeros<double>(B * m);
  return units_launch(game, params, threads, smem_limit_doubles, A, da, plan);
}

// evaluation at (x0, u, l), then G v (game_G_times), G' w (game_GT_times), rows[B, nrows] of G by game_G_row and the
// same rows by game_G_cols (nrows <= n)
int units_G(const dg_game_struct* game, const dgsqp_params* params, int B, int threads, long smem_limit_doubles,
            const double* x0, const double* u, const double* l, const double* v, const double* w, const int* rows, int nrows,
            double* Q, double* qe, double* gtl, double* g, double* Gv, double* GTw, double* Grow, double* Gcol, int* plan) {
  const Dims D = units_dims(game); const size_t n = D.n, m = D.m;
  if (nrows < 1 || nrows > D.n) return -1;
  for (int i = 0; i < B * nrows; ++i) if (rows[i] < 0 || rows[i] >= D.m) return -1;
  DevArrays da; UnitArgs A = units_args(B, U_G);
  A.x0 = da.in(x0, B * D.nq); A.u = da.in(u, B * n); A.l = da.in(l, B * m);
  A.v = da.in(v, B * n); A.w = da.in(w, B * m); A.rows = da.in(rows, (size_t)B * nrows); A.nrows = nrows;
  A.Q = da.out(Q, B * n * n); A.q = da.out(qe, B * n); A.gtl = da.out(gtl, B * n); A.g = da.out(g, B * m);
  A.Gv = da.out(Gv, B * m); A.GTw = da.out(GTw, B * n);
  A.Grow = da.out(Grow, (size_t)B * nrows * n); A.Gcol = da.out(Gcol, (size_t)B * nrows * n);
  return units_launch(game, params, threads, smem_limit_doubles, A, da, plan);
}

}
