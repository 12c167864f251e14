// Constraint-row layout and workspace table shared by the device games (see game.cuh).
//
// Included by a game header after it has defined
//   DG_NQA, DG_NUA        states and inputs per agent
//   DG_GAME_ROWS          game-specific rows per agent at the stages k < N (racing: 4 input-rate rows, merge: 2 lane rows)
//   DG_GAME_ROWS_N        game-specific rows per agent at the terminal stage (racing: 0, merge: 2)
//   DG_BOUND_STATE        the state the state-bound rows read (racing: e_y = 5, merge: v = 2)
//   GameDesc
// Per (stage k, agent) the rows are [game rows, input upper bounds (k < N), input lower bounds (k < N), state upper
// and lower bound (k >= 1)], preceded at k >= 1 by the P pairwise collision rows of the stage (DGSQP.py:730-821).
#pragma once
#include "cta.cuh"

// d fd / d [q;u] per (stage, agent): DG_NQA rows of DG_AB_LD entries, the input columns start at DG_NQA
#define DG_AB_LD (DG_NQA + DG_NUA)
#define DG_AB_SZ (DG_NQA * DG_AB_LD)
// rows per agent at k == 0, 0 < k < N and k == N
#define DG_ROWS_0 (DG_GAME_ROWS + 2 * DG_NUA)
#define DG_ROWS_K (DG_GAME_ROWS + 2 * DG_NUA + 2)
#define DG_ROWS_N (DG_GAME_ROWS_N + 2)

struct Dims {
  int M, N, nq, nu, n, m, P, nc0, nck, ncN, twoN;
  int ld;        // leading dimension of the n x n work matrices (odd: conflict-free row AND column walks in shared memory)
  int sens_sz;   // doubles of packed sensitivity rows per agent
};

DG_HD Dims make_dims(int M, int N) {
  Dims d;
  d.M = M; d.N = N; d.nq = DG_NQA * M; d.nu = DG_NUA * M; d.n = d.nu * N;
  d.P = M * (M - 1) / 2;
  d.nc0 = DG_ROWS_0 * M; d.nck = d.P + DG_ROWS_K * M; d.ncN = d.P + DG_ROWS_N * M;
  d.m = d.nc0 + (N - 1) * d.nck + d.ncN;
  d.twoN = 2 * N;
  d.ld = d.n | 1;
  d.sens_sz = 3 * N * (N + 1);
  return d;
}

// row kinds; K_GAME is the game-specific family (racing: rate rows, b = 2 * input + (0: upper, 1: lower); merge: lane
// rows, b = lane), b of the bound rows is the input or DG_BOUND_STATE
enum { K_COLL = 0, K_GAME = 1, K_INUB = 2, K_INLB = 3, K_STUB = 4, K_STLB = 5 };

DG_DEV int row_off(const Dims& D, int k) { return k == 0 ? 0 : D.nc0 + (k - 1) * D.nck; }
DG_DEV int row_coll(const Dims& D, int k, int p) { return row_off(D, k) + p; }                        // k>=1
DG_DEV int row_agent(const Dims& D, int k, int a) {
  return k == 0 ? DG_ROWS_0 * a : (k < D.N ? row_off(D, k) + D.P + DG_ROWS_K * a : row_off(D, k) + D.P + DG_ROWS_N * a);
}
DG_DEV int row_game(const Dims& D, int k, int a, int r) { return row_agent(D, k, a) + r; }
DG_DEV int row_inub(const Dims& D, int k, int a, int c) { return row_agent(D, k, a) + DG_GAME_ROWS + c; }            // k<N
DG_DEV int row_inlb(const Dims& D, int k, int a, int c) { return row_agent(D, k, a) + DG_GAME_ROWS + DG_NUA + c; }   // k<N
DG_DEV int row_stub(const Dims& D, int k, int a) { return row_agent(D, k, a) + (k < D.N ? DG_ROWS_0 : DG_GAME_ROWS_N); }  // k>=1
DG_DEV int row_stlb(const Dims& D, int k, int a) { return row_agent(D, k, a) + (k < D.N ? DG_ROWS_0 + 1 : DG_GAME_ROWS_N + 1); }  // k>=1

DG_DEV void pair_ij(int M, int p, int& i, int& j) {
  i = 0;
  int rem = p;
  while (rem >= M - 1 - i) { rem -= M - 1 - i; ++i; }
  j = i + 1 + rem;
}

DG_DEV void decode_row(const Dims& D, int r, int& k, int& kind, int& a, int& b) {
  int w;
  if (r < D.nc0) { k = 0; w = r; }
  else { k = 1 + (r - D.nc0) / D.nck; if (k > D.N) k = D.N; w = r - row_off(D, k); }
  if (k >= 1) {
    if (w < D.P) { kind = K_COLL; pair_ij(D.M, w, a, b); return; }
    w -= D.P;
  }
  if (k < D.N) {
    int per = k == 0 ? DG_ROWS_0 : DG_ROWS_K;
    a = w / per; w -= a * per;
    if (w < DG_GAME_ROWS) { kind = K_GAME; b = w; }
    else if (w < DG_GAME_ROWS + DG_NUA) { kind = K_INUB; b = w - DG_GAME_ROWS; }
    else if (w < DG_ROWS_0) { kind = K_INLB; b = w - (DG_GAME_ROWS + DG_NUA); }
    else if (w == DG_ROWS_0) { kind = K_STUB; b = DG_BOUND_STATE; }
    else { kind = K_STLB; b = DG_BOUND_STATE; }
  } else {
    a = w / DG_ROWS_N; w -= a * DG_ROWS_N;
    if (DG_GAME_ROWS_N > 0 && w < DG_GAME_ROWS_N) { kind = K_GAME; b = w; }
    else { kind = w == DG_GAME_ROWS_N ? K_STUB : K_STLB; b = DG_BOUND_STATE; }
  }
}

// The row layout only depends on (M, N): the decode (three integer divisions) is tabulated once per instance
// (EvalBuf::rowtab, packed k | kind << 6 | a << 9 | b << 11) for the loops that walk all m rows.
DG_DEV int pack_row(const Dims& D, int r) {
  int k, kind, a, b;
  decode_row(D, r, k, kind, a, b);
  return k | (kind << 6) | (a << 9) | (b << 11);
}
DG_DEV void unpack_row(int p, int& k, int& kind, int& a, int& b) { k = p & 63; kind = (p >> 6) & 7; a = (p >> 9) & 3; b = (p >> 11) & 7; }

DG_DEV int uidx(const Dims& D, int a, int k, int c) { return a * D.twoN + 2 * k + c; }

template <bool SM>
DG_DEVN void game_row_table(Cta& c, const Dims& D_, int* rowtab) {
  const Dims D = D_;
  DG_FOR(r, D.m) rowtab[r] = pack_row(D, r);
  c.sync();
}

// Per-CTA workspace views (global memory unless noted); a game's EvalBuf derives from this table
struct EvalTables {
  double* x;     // (N+1)*nq
  double* AB;    // N*M*DG_AB_SZ   d fd / d [q;u]  per (k,a)
  double* T2;    // N*M*DG_T2_SZ   second derivatives per (k,a)
  double* S;     // M*3N(N+1)   sensitivity rows (x, y, DG_BOUND_STATE) of stages 1..N wrt own inputs, packed: row (a,k,r)
                 //             holds the 2k columns of inputs u^a_0..u^a_{k-1} at  a*sens_sz + 3k(k-1) + r*2k
  double* g;     // m
  double* q;     // n   [grad_{u^a} J^a]_a
  double* gtl;   // n   G' l
  double* cst;   // (M+1)*(N+1)*nq  costates: f<M of J^f, f==M of l'C
  double* Hc;    // (M+1)*N*M*DG_HC_SZ   sum_i p_i * T2[i]
  double* Vbuf;  // 2*(M+1)*nq*nq  DP value-function Hessians of all functions (double buffered)
  double* Q;     // n*n raw game Hessian (row major)
  double* Wrow;  // (M+1)*nq*n  running rows of Dxu_Q^f in the Hessian DP, [(f*nq+q)*n + r]
  double* tmpS;  // M*N*3   state-row products for G v (and the merge rollout's position increments)
  double* cf;    // M*N*3   per (a,k) coefficients for G' w
  double* lbuf;  // m       staged copy of the multipliers the evaluation runs with
  int* rowtab;   // m       packed row decode (global memory, read-only after game_row_table)
};

// shared-memory residency hints for the buffer tables (SM instantiation only)
#define DG_SH_EVAL(E) do { DG_ASSUME_SHARED((E).x); DG_ASSUME_SHARED((E).g); DG_ASSUME_SHARED((E).q); DG_ASSUME_SHARED((E).gtl); \
  DG_ASSUME_SHARED((E).tmpS); DG_ASSUME_SHARED((E).cf); DG_ASSUME_SHARED((E).AB); DG_ASSUME_SHARED((E).cst); DG_ASSUME_SHARED((E).Hc); \
  DG_ASSUME_SHARED((E).Vbuf); DG_ASSUME_SHARED((E).Wrow); DG_ASSUME_SHARED((E).T2); DG_ASSUME_SHARED((E).S); DG_ASSUME_SHARED((E).lbuf); } while (0)

// start of packed sensitivity row (a, k, r): k in 1..N, r in {0:x, 1:y, 2:DG_BOUND_STATE}; 2k entries
DG_DEV int sens_off(const Dims& D, int a, int k, int r) { return a * D.sens_sz + 3 * k * (k - 1) + r * 2 * k; }
