// Monte-Carlo instance generation on the device: dgsqp_sample_racing / dgsqp_sample_merge (include/dgsqp_b200.h).
// Stream, trial layout and decisions: mc_sampler.cuh.  Per block of trials the host loop below runs
//   1. the decision kernel  (one thread per trial: its draws, the pre-check, the roll-outs up to the first collision),
//   2. a stable compaction of the accepted trials (cub::DeviceSelect::Flagged, trial order),
//   3. the output kernel    (one thread per accepted instance and agent: x0 and the warm start, recomputed),
// and reads back one count, until B instances are accepted or max_trials trials are spent.  The block size only sets how
// much is decided per launch; the instances do not depend on it.
// Compiled with -fmad=false (see __graft_entry__.py): the draw transforms follow NumPy's evaluation order.
#include <cuda_runtime.h>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <math.h>
#include <stdint.h>
#include <string>

#include "abi_common.h"
#include "mc_sampler.cuh"

namespace {

const int MC_THREADS = 128;
const int64_t MC_MIN_BLOCK = 1 << 16, MC_MAX_BLOCK = 1 << 24;   // trials decided per launch

template <int M>
__global__ void __launch_bounds__(MC_THREADS, 1) mc_racing_decide_kernel(const McRacing* __restrict__ S, McPcg g0, const mc_u128* __restrict__ table,
                                                                      int64_t t0, int T, uint8_t* __restrict__ flag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= T) return;
  flag[i] = mc_racing_decide<M>(*S, g0, table, t0 + i) ? 1 : 0;
}

// instance b = offset + i of the output <- trial t0 + sel[i]; one thread per (instance, agent)
__global__ void __launch_bounds__(MC_THREADS, 1) mc_racing_output_kernel(const McRacing* __restrict__ Sp, McPcg g0, const mc_u128* __restrict__ table,
                                                                      int64_t t0, const int* __restrict__ sel, int count,
                                                                      int offset, double* __restrict__ x0,
                                                                      double* __restrict__ u_ws, int64_t* __restrict__ trial) {
  const McRacing& S = *Sp;
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= (int64_t)count * S.M) return;
  const int i = (int)(j / S.M), a = (int)(j - (int64_t)i * S.M);
  const int64_t t = t0 + sel[i], b = offset + i;
  const int nq = 6 * S.M, n = 2 * S.P.N * S.M;
  mc_racing_instance(S, g0, table, t, a, x0 + b * nq + 6 * a, u_ws + b * n + (int64_t)a * 2 * S.P.N);
  if (trial && a == 0) trial[b] = t;
}

__global__ void __launch_bounds__(MC_THREADS, 1) mc_merge_decide_kernel(const McMerge* __restrict__ S, McPcg g0, const mc_u128* __restrict__ table,
                                                                     int64_t t0, int T, uint8_t* __restrict__ flag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= T) return;
  double q[12];
  mc_merge_draw(*S, g0, table, t0 + i, q);
  flag[i] = mc_merge_accept(*S, q) ? 1 : 0;
}

__global__ void __launch_bounds__(MC_THREADS, 1) mc_merge_output_kernel(const McMerge* __restrict__ S, McPcg g0, const mc_u128* __restrict__ table,
                                                                     int64_t t0, const int* __restrict__ sel, int count,
                                                                     int offset, double* __restrict__ x0,
                                                                     int64_t* __restrict__ trial) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const int64_t t = t0 + sel[i], b = offset + i;
  double q[12];
  mc_merge_draw(*S, g0, table, t, q);
  for (int k = 0; k < 12; ++k) x0[b * 12 + k] = q[k];
  if (trial) trial[b] = t;
}

// Device buffers of one call: the game record (read from global memory: as a kernel argument, the dynamically indexed
// key-point table would be copied to every thread's stack), the jump table, the flags and ids of one block, the selected count, cub's scratch.
struct McBuffers {
  void* game = nullptr;
  mc_u128* table = nullptr;
  uint8_t* flag = nullptr;
  int* sel = nullptr;
  int* nsel = nullptr;
  void* tmp = nullptr;
  size_t tmp_bytes = 0;
  ~McBuffers() { cudaFree(game); cudaFree(table); cudaFree(flag); cudaFree(sel); cudaFree(nsel); cudaFree(tmp); }
};

// The host loop shared by both games.  decide(t0, T) and output(t0, count, offset) enqueue the two kernels on st.
template <class Decide, class Output>
int mc_run(const char* who, const void* game, size_t game_bytes, const dgsqp_pcg64* rng, int32_t B, int64_t max_trials, int32_t* accepted, int64_t* trials_used,
           cudaStream_t st, McBuffers& buf, Decide decide, Output output) {
  const std::string tag = std::string(who) + ": ";
  *accepted = 0; *trials_used = 0;
  const McPcg g0 = mc_pcg_from(rng);
  mc_u128 table[128];
  mc_jump_table(g0.inc, table);
  const int64_t cap = max_trials < MC_MAX_BLOCK ? max_trials : MC_MAX_BLOCK;
  CUDA_TRY(cudaMalloc(&buf.game, game_bytes));
  CUDA_TRY(cudaMalloc(&buf.table, sizeof(table)));
  CUDA_TRY(cudaMalloc(&buf.flag, cap));
  CUDA_TRY(cudaMalloc(&buf.sel, sizeof(int) * cap));
  CUDA_TRY(cudaMalloc(&buf.nsel, sizeof(int)));
  thrust::counting_iterator<int> ids(0);
  CUDA_TRY(cub::DeviceSelect::Flagged(nullptr, buf.tmp_bytes, ids, buf.flag, buf.sel, buf.nsel, (int)cap, st));
  CUDA_TRY(cudaMalloc(&buf.tmp, buf.tmp_bytes));
  CUDA_TRY(cudaMemcpyAsync(buf.game, game, game_bytes, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(buf.table, table, sizeof(table), cudaMemcpyHostToDevice, st));
  int64_t t0 = 0;
  int32_t have = 0;
  while (have < B && t0 < max_trials) {
    // size the block from the acceptance rate seen so far (20 % margin); the result does not depend on it
    int64_t T = MC_MIN_BLOCK;
    if (have > 0) T = (int64_t)((double)(B - have) * (double)t0 / (double)have * 1.2) + 1;
    else if (t0 > 0) T = 8 * t0;
    T = T < MC_MIN_BLOCK ? MC_MIN_BLOCK : (T > cap ? cap : T);
    if (T > max_trials - t0) T = max_trials - t0;
    decide(t0, (int)T);
    CUDA_TRY(cudaGetLastError());
    size_t tb = buf.tmp_bytes;
    CUDA_TRY(cub::DeviceSelect::Flagged(buf.tmp, tb, ids, buf.flag, buf.sel, buf.nsel, (int)T, st));
    int nsel = 0;
    CUDA_TRY(cudaMemcpyAsync(&nsel, buf.nsel, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    const int take = nsel < B - have ? nsel : B - have;
    if (take > 0) {
      output(t0, take, have);
      CUDA_TRY(cudaGetLastError());
    }
    if (take == B - have && take > 0) {
      int last = 0;       // trials used = id of the B-th accepted trial + 1
      CUDA_TRY(cudaMemcpyAsync(&last, buf.sel + take - 1, sizeof(int), cudaMemcpyDeviceToHost, st));
      CUDA_TRY(cudaStreamSynchronize(st));
      *trials_used = t0 + last + 1;
    } else {
      *trials_used = t0 + T;
    }
    have += take;
    *accepted = have;
    t0 += T;
  }
  CUDA_TRY(cudaStreamSynchronize(st));
  if (have < B)
    return dg_set_err(DGSQP_EINVAL, tag + "max_trials = " + std::to_string(max_trials) + " trials accepted " +
                                        std::to_string(have) + " of " + std::to_string(B) + " instances");
  return DGSQP_OK;
}

int mc_check_common(const dgsqp_pcg64* rng, int32_t B, int64_t max_trials, const double* x0, int32_t* accepted,
                    int64_t* trials_used) {
  if (!rng || !accepted || !trials_used) return dg_set_err(DGSQP_EINVAL, "NULL argument");
  if (B < 0 || max_trials <= 0) return dg_set_err(DGSQP_EINVAL, "invalid B / max_trials");
  if (B > 0 && !x0) return dg_set_err(DGSQP_EINVAL, "NULL buffer");
  return DGSQP_OK;
}

}  // namespace

extern "C" {

int dgsqp_sample_racing(const dgsqp_racing_game* game, const double* key_pts, int32_t kind, const dgsqp_pcg64* rng, int device,
                        int32_t B, int64_t max_trials, double* x0, double* u_ws, int64_t* trial, int32_t* accepted,
                        int64_t* trials_used, void* stream) {
  McRacing S;
  if (mc_racing_fill(game, key_pts, kind, &S) != 0) return dg_set_err(DGSQP_EINVAL, "dgsqp_sample_racing: invalid game / key points / kind");
  if (int rc = mc_check_common(rng, B, max_trials, x0, accepted, trials_used)) return rc;
  if (B > 0 && !u_ws) return dg_set_err(DGSQP_EINVAL, "NULL buffer");
  *accepted = 0; *trials_used = 0;
  if (cudaSetDevice(device) != cudaSuccess || cudaFree(nullptr) != cudaSuccess)
    return dg_set_err(DGSQP_ECUDA, "dgsqp_sample_racing: no usable CUDA device (there is no CPU fallback)");
  if (B == 0) return DGSQP_OK;
  cudaStream_t st = (cudaStream_t)stream;
  McBuffers buf;
  auto decide = [&](int64_t t0, int T) {
    const int grid = (T + MC_THREADS - 1) / MC_THREADS;
    if (S.M == 2) mc_racing_decide_kernel<2><<<grid, MC_THREADS, 0, st>>>((const McRacing*)buf.game, mc_pcg_from(rng), buf.table, t0, T, buf.flag);
    else if (S.M == 3) mc_racing_decide_kernel<3><<<grid, MC_THREADS, 0, st>>>((const McRacing*)buf.game, mc_pcg_from(rng), buf.table, t0, T, buf.flag);
    else mc_racing_decide_kernel<4><<<grid, MC_THREADS, 0, st>>>((const McRacing*)buf.game, mc_pcg_from(rng), buf.table, t0, T, buf.flag);
    dg_launches.fetch_add(1);
  };
  auto output = [&](int64_t t0, int count, int offset) {
    const int grid = (int)(((int64_t)count * S.M + MC_THREADS - 1) / MC_THREADS);
    mc_racing_output_kernel<<<grid, MC_THREADS, 0, st>>>((const McRacing*)buf.game, mc_pcg_from(rng), buf.table, t0, buf.sel, count, offset, x0, u_ws, trial);
    dg_launches.fetch_add(1);
  };
  return mc_run("dgsqp_sample_racing", &S, sizeof(S), rng, B, max_trials, accepted, trials_used, st, buf, decide, output);
}

int dgsqp_sample_merge(const dgsqp_merge_game* game, const dgsqp_pcg64* rng, int device, int32_t B, int64_t max_trials,
                       double* x0, int64_t* trial, int32_t* accepted, int64_t* trials_used, void* stream) {
  McMerge S;
  if (mc_merge_fill(game, &S) != 0) return dg_set_err(DGSQP_EINVAL, "dgsqp_sample_merge: invalid game (the merge scenario has 3 cars, N >= 1)");
  if (int rc = mc_check_common(rng, B, max_trials, x0, accepted, trials_used)) return rc;
  *accepted = 0; *trials_used = 0;
  if (cudaSetDevice(device) != cudaSuccess || cudaFree(nullptr) != cudaSuccess)
    return dg_set_err(DGSQP_ECUDA, "dgsqp_sample_merge: no usable CUDA device (there is no CPU fallback)");
  if (B == 0) return DGSQP_OK;
  cudaStream_t st = (cudaStream_t)stream;
  McBuffers buf;
  auto decide = [&](int64_t t0, int T) {
    mc_merge_decide_kernel<<<(T + MC_THREADS - 1) / MC_THREADS, MC_THREADS, 0, st>>>((const McMerge*)buf.game, mc_pcg_from(rng), buf.table, t0, T, buf.flag);
    dg_launches.fetch_add(1);
  };
  auto output = [&](int64_t t0, int count, int offset) {
    mc_merge_output_kernel<<<(count + MC_THREADS - 1) / MC_THREADS, MC_THREADS, 0, st>>>((const McMerge*)buf.game, mc_pcg_from(rng), buf.table, t0, buf.sel,
                                                                                       count, offset, x0, trial);
    dg_launches.fetch_add(1);
  };
  return mc_run("dgsqp_sample_merge", &S, sizeof(S), rng, B, max_trials, accepted, trials_used, st, buf, decide, output);
}

}  // extern "C"
