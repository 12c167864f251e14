// CTA-cooperative execution context.
//
// Every solver routine in this directory is written as a function executed by ALL threads of
// one thread block (one game instance per CTA): strided loops over `c.tid`, `c.sync()` between
// dependent phases, block-wide reductions through `c.sum/max/argmin`.  Control flow is uniform:
// every branch is decided from values all threads read identically (shared memory or reduction
// results).
//
// The same source also compiles with a plain C++ compiler (DG_HOSTSIM) as a one-thread "CTA";
// that build exists only for tests/hostsim (algorithm debugging under ASan on machines without a
// GPU).  It is never linked into the product library.
#pragma once
#include <math.h>
#include <stdint.h>

// phases of the per-instance profile (cycles, dgsqp_last_phase_cycles)
enum { PH_LIN_FULL = 0, PH_ADJ_FULL, PH_HESS, PH_PD_TRIDIAG, PH_PD_EIG, PH_CHOL, PH_TRINV, PH_GI, PH_LSQR,
       PH_LIN_GRAD, PH_ADJ_GRAD, PH_MERIT, PH_OTHER,
       // sub-phases, only counted by the profiling build (-DDG_FINE_PHASES: c.lapf); in the product build their time
       // stays in the coarse phase around them (pd_eig / active_set / tri_inverse)
       PH_PD_SYM, PH_PD_EIGVAL, PH_PD_INVIT, PH_PD_BACK, PH_GI_SLACK, PH_GI_DZ, PH_GI_STEP, PH_GI_ADD, PH_GI_DROP, PH_QP_X0, PH_QP_WARM,
       PH_WS_D, PH_WS_QR, PH_WS_APPLY, PH_WS_MULT,       // stages of the warm start (the rest of it stays in qp_warm)
       DG_NPHASE };

#ifdef DG_HOSTSIM
#define DG_RSQRT(x) (1.0 / sqrt(x))
#define DG_FMA(a, b, c) ((a) * (b) + (c))
// a * b rounded on its own, also when the host build contracts products into FMAs (tests/hostsim_lib.py, fma=True)
static inline double dg_mul_rn(double a, double b) { volatile double r = a * b; return r; }
#define DG_MUL(a, b) dg_mul_rn((a), (b))
#define DG_ATOMIC_MIN(p, v) do { if ((v) < *(p)) *(p) = (v); } while (0)
#define DG_DEV static inline
#define DG_HD static inline
#define DG_DEVN static
#define DG_CONST static const
#define DG_RESTRICT
struct Cta {
  inline int tid() const { return 0; }
  inline int nt() const { return 1; }
  inline int lane() const { return 0; }
  inline int warp() const { return 0; }
  inline int nwarps() const { return 1; }
  static constexpr int wsz = 1;   // lanes per warp
  double* red = nullptr;
  inline void sync() {}
  inline double sum(double v) { return v; }
  inline double max(double v) { return v; }
  inline void max3(double& a, double& b, double& d) {}
  inline double min(double v) { return v; }
  inline int imin(int v) { return v; }
  inline int isum(int v) { return v; }
  // smallest value, ties -> smallest index; every thread gets the winner
  inline void argmin(double v, int idx, double& ov, int& oi) { ov = v; oi = idx; }
  inline double warp_sum(double v) { return v; }
  template <int N> inline void warp_sum_n(double (&)[N]) {}
  inline void warp_argmin(double&, int&) {}
  inline void syncwarp() {}
  inline void sum2(double& a, double& b) {}
  inline void sum3(double& a, double& b, double& d) {}
  inline void sum4(double& a, double& b, double& d, double& e) {}
  inline int bcast0(int v) { return v; }
  inline void lap(int) {}
  inline void lapf(int) {}
  inline void lap2(int, int) {}
};
#else
#define DG_RSQRT(x) rsqrt(x)
// a * b + c as one rounding, pinned: the compiler may not choose which product of a sum it contracts
#define DG_FMA(a, b, c) __fma_rn((a), (b), (c))
// a * b rounded on its own: never contracted into a neighbouring addition
#define DG_MUL(a, b) __dmul_rn((a), (b))
#define DG_ATOMIC_MIN(p, v) atomicMin((p), (v))
#define DG_DEV __device__ __forceinline__
#define DG_HD __host__ __device__ __forceinline__
#define DG_DEVN __device__ __noinline__
#define DG_CONST __device__ const
#ifdef DG_NO_RESTRICT
#define DG_RESTRICT
#else
#define DG_RESTRICT __restrict__
#endif
// CTA-wide scratch of the reductions (2 buffers x 160 doubles) and the phase counters: file-scope shared
// variables, so no pointer has to be fetched from the (local-memory resident) Cta object
__shared__ __align__(16) double dg_s_red[320];
__shared__ long long dg_s_ph[DG_NPHASE + 1];

struct Cta {
  // thread coordinates come straight from the special registers: a Cta is passed by reference through
  // non-inlined functions, so data members would be re-read from local memory all over the hot loops
  __device__ __forceinline__ int tid() const { return (int)threadIdx.x; }
  __device__ __forceinline__ int nt() const { return (int)blockDim.x; }
  __device__ __forceinline__ int lane() const { return (int)(threadIdx.x & 31u); }
  __device__ __forceinline__ int warp() const { return (int)(threadIdx.x >> 5); }
  __device__ __forceinline__ int nwarps() const { return (int)((blockDim.x + 31u) >> 5); }
  static constexpr int wsz = 32;  // lanes per warp
  // phase profile: cycles between consecutive lap() calls are charged to the phase named by the later call
  // (thread 0 only; counters live in shared memory: ph[0..DG_NPHASE) cycles, ph[DG_NPHASE] = time of the last lap)
  __device__ __forceinline__ void lap(int id) {
    if (tid() == 0) { long long t = clock64(); dg_s_ph[id] += t - dg_s_ph[DG_NPHASE]; dg_s_ph[DG_NPHASE] = t; }
  }
#ifdef DG_FINE_PHASES
  __device__ __forceinline__ void lapf(int id) { lap(id); }
  __device__ __forceinline__ void lap2(int, int fine) { lap(fine); }      // the profiling build charges the sub-phase
#else
  __device__ __forceinline__ void lapf(int) {}
  __device__ __forceinline__ void lap2(int coarse, int) { lap(coarse); }
#endif
  __device__ __forceinline__ void sync() { __syncthreads(); }
  __device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
  }
  // N independent warp sums, butterfly stage by stage (the N shuffles of a stage are in flight together)
  template <int N>
  __device__ __forceinline__ void warp_sum_n(double (&v)[N]) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int t = 0; t < N; ++t) v[t] += __shfl_xor_sync(0xffffffffu, v[t], o);
    }
  }
  // smallest value over the warp, ties -> smallest index; every lane gets the winner
  __device__ __forceinline__ void warp_argmin(double& v, int& idx) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double v2 = __shfl_xor_sync(0xffffffffu, v, o);
      const int i2 = __shfl_xor_sync(0xffffffffu, idx, o);
      if (v2 < v || (v2 == v && i2 < idx)) { v = v2; idx = i2; }
    }
  }
  // Block reductions use two alternating scratch buffers, so one barrier per reduction suffices: a thread
  // can only reach the next reduction that reuses a buffer after passing the barrier of the one in between.
  int flip = 0;
  __device__ __forceinline__ double* next_buf() { flip ^= 1; return dg_s_red + flip * 160; }
  __device__ __forceinline__ void syncwarp() { __syncwarp(); }
  // sum of the nwarps (<= 16) per-warp partials at b[0..]: fixed pairwise tree, identical in every thread
  __device__ __forceinline__ double tree16(const double* b) const {
    if (nwarps() == 8) {
      // the default CTA width: four 128-bit loads and a fixed pairwise tree
      const double2 p0 = reinterpret_cast<const double2*>(b)[0], p1 = reinterpret_cast<const double2*>(b)[1];
      const double2 p2 = reinterpret_cast<const double2*>(b)[2], p3 = reinterpret_cast<const double2*>(b)[3];
      return ((p0.x + p0.y) + (p1.x + p1.y)) + ((p2.x + p2.y) + (p3.x + p3.y));
    }
    double t[16];
#pragma unroll
    for (int w = 0; w < 16; ++w) t[w] = w < nwarps() ? b[w] : 0.0;
#pragma unroll
    for (int s = 8; s > 0; s >>= 1)
#pragma unroll
      for (int w = 0; w < s; ++w) t[w] += t[w + s];
    return t[0];
  }
  __device__ __forceinline__ double sum(double v) {
    v = warp_sum(v);
    double* b = next_buf();
    if (lane() == 0) b[warp()] = v;
    __syncthreads();
    return tree16(b);
  }
  __device__ __forceinline__ void sum2(double& a0, double& a1) {
    a0 = warp_sum(a0); a1 = warp_sum(a1);
    double* b = next_buf();
    if (lane() == 0) { b[warp()] = a0; b[32 + warp()] = a1; }
    __syncthreads();
    a0 = tree16(b); a1 = tree16(b + 32);
  }
  __device__ __forceinline__ void sum3(double& a0, double& a1, double& a2) {
    a0 = warp_sum(a0); a1 = warp_sum(a1); a2 = warp_sum(a2);
    double* b = next_buf();
    if (lane() == 0) { b[warp()] = a0; b[32 + warp()] = a1; b[64 + warp()] = a2; }
    __syncthreads();
    a0 = tree16(b); a1 = tree16(b + 32); a2 = tree16(b + 64);
  }
  __device__ __forceinline__ void sum4(double& a0, double& a1, double& a2, double& a3) {
    a0 = warp_sum(a0); a1 = warp_sum(a1); a2 = warp_sum(a2); a3 = warp_sum(a3);
    double* b = next_buf();
    if (lane() == 0) { b[warp()] = a0; b[32 + warp()] = a1; b[64 + warp()] = a2; b[96 + warp()] = a3; }
    __syncthreads();
    a0 = tree16(b); a1 = tree16(b + 32); a2 = tree16(b + 64); a3 = tree16(b + 96);
  }
  __device__ __forceinline__ double max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    double* b = next_buf();
    if (lane() == 0) b[warp()] = v;
    __syncthreads();
    double r = b[0];
    for (int w = 1; w < nwarps(); ++w) r = fmax(r, b[w]);
    return r;
  }
  __device__ __forceinline__ void max3(double& a0, double& a1, double& a2) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      a0 = fmax(a0, __shfl_xor_sync(0xffffffffu, a0, o));
      a1 = fmax(a1, __shfl_xor_sync(0xffffffffu, a1, o));
      a2 = fmax(a2, __shfl_xor_sync(0xffffffffu, a2, o));
    }
    double* b = next_buf();
    if (lane() == 0) { b[warp()] = a0; b[32 + warp()] = a1; b[64 + warp()] = a2; }
    __syncthreads();
    double r0 = b[0], r1 = b[32], r2 = b[64];
    for (int w = 1; w < nwarps(); ++w) { r0 = fmax(r0, b[w]); r1 = fmax(r1, b[32 + w]); r2 = fmax(r2, b[64 + w]); }
    a0 = r0; a1 = r1; a2 = r2;
  }
  __device__ __forceinline__ double min(double v) { return -max(-v); }
  // value of thread 0 to every thread (CTA-uniform decisions taken from something only one thread reads, e.g. a clock)
  __device__ __forceinline__ int bcast0(int v) {
    int* b = (int*)next_buf();
    if (tid() == 0) b[0] = v;
    __syncthreads();
    return b[0];
  }
  __device__ __forceinline__ int imin(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { int t = __shfl_xor_sync(0xffffffffu, v, o); v = t < v ? t : v; }
    int* b = (int*)next_buf();
    if (lane() == 0) b[warp()] = v;
    __syncthreads();
    int r = b[0];
    for (int w = 1; w < nwarps(); ++w) { int t = b[w]; r = t < r ? t : r; }
    return r;
  }
  __device__ __forceinline__ int isum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    int* b = (int*)next_buf();
    if (lane() == 0) b[warp()] = v;
    __syncthreads();
    int r = 0;
    for (int w = 0; w < nwarps(); ++w) r += b[w];
    return r;
  }
  __device__ __forceinline__ void argmin(double v, int idx, double& ov, int& oi) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      double v2 = __shfl_xor_sync(0xffffffffu, v, o);
      int i2 = __shfl_xor_sync(0xffffffffu, idx, o);
      if (v2 < v || (v2 == v && i2 < idx)) { v = v2; idx = i2; }
    }
    double* b = next_buf();
    if (lane() == 0) { b[warp()] = v; ((int*)(b + 32))[warp()] = idx; }
    __syncthreads();
    ov = b[0]; oi = ((int*)(b + 32))[0];
    for (int w = 1; w < nwarps(); ++w) {
      double v2 = b[w]; int i2 = ((int*)(b + 32))[w];
      if (v2 < ov || (v2 == ov && i2 < oi)) { ov = v2; oi = i2; }
    }
  }
};
#endif

// Address-space hint: in the SM = true instantiation of the solver every hot buffer is known to be shared-memory
// resident (plan_memory), which lets the compiler emit LDS/STS with 32-bit addressing instead of generic accesses.
// RULE: state a hint once per pointer and only at the top of a non-inlined (DG_DEVN) function.  nvcc 12.9 silently
// drops code when the same pointer value is hinted twice inside one function body (e.g. caller + inlined callee).
#ifdef DG_HOSTSIM
#define DG_ASSUME_SHARED(p) do { } while (0)
#else
#define DG_ASSUME_SHARED(p) do { if (SM) __builtin_assume(__isShared((const void*)(p))); } while (0)
#endif

// nanoseconds of a monotonic clock (device: %globaltimer; host build: steady_clock) for DGSQPParams.time_limit
#ifdef DG_HOSTSIM
#include <chrono>
static inline double dg_now_ns() { return (double)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
#else
__device__ __forceinline__ double dg_now_ns() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return (double)t; }
#endif

#define DG_FOR(i, n) for (int i = c.tid(); i < (n); i += c.nt())
// same loop with the thread numbering rotated by `off`: lets independent phases inside one barrier interval run on
// different warps instead of piling up on the low thread ids
#define DG_FOR_OFF(i, n, off) for (int i = (c.tid() + c.nt() - ((off) % c.nt())) % c.nt(); i < (n); i += c.nt())

// 2D decomposition of a (len columns) x (depth) iteration space over the CTA: consecutive threads own consecutive
// columns (conflict-free / coalesced), the G column groups interleave the depth index.
//   for (int i = s.i0; i < len; i += s.istep) for (int j = j_begin + s.g; j < j_end; j += s.G) ...
struct Split2 { int i0, istep, g, G; };
DG_DEV Split2 split2(const Cta& c, int len) {
  int cw = (len + Cta::wsz - 1) / Cta::wsz * Cta::wsz;
  if (cw > c.nt()) cw = c.nt();
  if (cw < 1) cw = 1;
  Split2 s;
  s.G = c.nt() / cw; s.g = c.tid() / cw; s.i0 = c.tid() - s.g * cw; s.istep = cw;
  if (s.g >= s.G) s.i0 = len;                  // leftover threads idle
  return s;
}
