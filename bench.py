#!/usr/bin/env python3
"""Headline benchmark: converged 2-agent chicane game solves / s (BASELINE.json configs[1]) and the other BASELINE games.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload chicane|curve|agents3|agents4|merge] [--batch B] [--total T] [--dump-outputs DIR]

A step = one pass of the solver over B synthetic instances per GPU (randomised initial conditions + warm start,
dgsqp_b200.montecarlo; B = 10 000 for the headline workload).  `value` is measured with the inputs resident in HBM (CUDA
events on the launching stream), `e2e` through the host-buffer C-ABI call with the H2D / D2H copies inside the timed region.
N > 1: one process per GPU under torchrun, instances sharded with no collective on the solve path (weak scaling: B per
GPU; `--total T` shards T instances over the ranks instead = strong scaling, BASELINE configs[4] "1 M merge instances"),
statistics gathered at the end, time = max over ranks.

Workloads (BASELINE.json configs): chicane = configs[1] (10 k instances, the headline); curve = configs[2] (the script's
theta x N sweep, B instances spread over its 12 cells, reported per cell like scripts/process_data_curve.py:98-110);
agents3 / agents4 = configs[3]; merge = configs[4].  configs[0] (one instance on the CPU) is reported inside every line as
`single_instance`: latency of one `solve()` on the GPU next to one CPU solve of the same instance.

`--impl reference` times the CPU oracle (NumPy restatement of the reference solver; the reference itself needs CasADi +
OSQP which are not installable offline) on all host cores: one persistent pool, one instance per task, BLAS pinned to one
thread per process.
"""
import os

# BLAS/OpenMP must be single-threaded in every process of the CPU arms (one oracle process per core): set before ANY import
# of numpy / torch, and overriding whatever the launcher exported
for _k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS", "VECLIB_MAXIMUM_THREADS"):
    os.environ[_k] = "1"

import argparse  # noqa: E402
import json  # noqa: E402
import math  # noqa: E402
import pathlib  # noqa: E402
import sys  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True             # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "converged_game_solves_per_sec"
UNIT = "solves/s"
CURVE_THETAS = (45.0, 75.0, 90.0)          # scripts/DGSQP_ALGAMES_monte_carlo_curve.py:134-146
CURVE_NS = (10, 15, 20, 25)
DEFAULT_BATCH = dict(chicane=10000, curve=12000, agents3=4000, agents4=2000, merge=10000)
MU_VIO = 1e-10                             # deterministic penalty-weight switch (DESIGN.md D2): the setting of the oracle and
                                           # of every parity fixture; the class default 0 is the literal DGSQP.py:560 rule
CPU_ARM_BUDGET_S = 200.0                   # wall budget of the whole `--impl reference` run
CPU_BASELINE_BUDGET_S = 20.0               # wall budget of the cpu_baseline leg inside the GPU arm
OUTPUT_FIELDS = ("u", "l", "x", "cost", "cond", "num_iters", "status", "qp_solves")   # BatchResult arrays
DUMP_BUDGET_BYTES = 60 * 10 ** 6           # array data of --dump-outputs: with the .npy headers below 64 MB


# ----------------------------------------------------------------------------- workloads
def make_cells(workload, batch):
    """A workload is a list of cells; a cell = (key, game, params, sampler(game, B, seed), instances).  `key` is what a CPU
    worker needs to rebuild the oracle of the cell."""
    import dgsqp_b200 as dg
    from dgsqp_b200.montecarlo import sample_head_to_head, sample_agents, sample_merge
    if workload == "chicane":
        return [dict(key=("chicane", 45.0, 25), game=dg.chicane_game(), params=dg.chicane_params(), B=batch,
                     sampler=lambda g, B, seed: sample_head_to_head(g, B, seed=seed), label="chicane_45_N25")]
    if workload == "curve":
        cells = []
        per = max(1, batch // (len(CURVE_THETAS) * len(CURVE_NS)))
        for th in CURVE_THETAS:
            for N in CURVE_NS:
                cells.append(dict(key=("curve", th, N), game=dg.curve_game(th, N), params=dg.curve_params(N), B=per,
                                  sampler=lambda g, B, seed: sample_head_to_head(g, B, seed=1 + seed),   # script seed 1
                                  label=f"curve_{th:g}_N{N}"))
        return cells
    if workload in ("agents3", "agents4"):
        M = int(workload[-1])
        return [dict(key=("agents", M, 25), game=dg.agents_game(M=M), params=dg.agents_params(), B=batch,
                     sampler=lambda g, B, seed: sample_agents(g, B, seed=seed), label=f"agents_M{M}_90_N25")]
    if workload == "merge":
        return [dict(key=("merge", 3, 20), game=dg.merge_game(), params=dg.merge_params(), B=batch,
                     sampler=lambda g, B, seed: sample_merge(g, B, seed=1 + seed), label="merge_N20")]   # script seed 1
    raise SystemExit(f"unknown workload {workload}")


def workload_config(workload, cells, batch, total):
    names = dict(chicane="chicane_2agent_N25_mc", curve="curve_2agent_theta45-75-90_N10-25_mc",
                 agents3="agents3_curve90_N25_mc", agents4="agents4_curve90_N25_mc", merge="merge_3agent_N20_mc")
    g, p = cells[0]["game"], cells[0]["params"]
    cfg = dict(workload=names[workload], instances_per_gpu=batch, agents=g.M,
               horizon=(g.N if len(cells) == 1 else [int(n) for n in CURVE_NS]),
               n=(g.n if len(cells) == 1 else [c["game"].n for c in cells[:len(CURVE_NS)]]),
               m=(g.m if len(cells) == 1 else [c["game"].m for c in cells[:len(CURVE_NS)]]),
               solver=f"DGSQP v1 (DGSQPParams: reg={p.reg:g}, nonmono_ls, {p.sqp_iters} SQP iters, tol {p.p_tol:g}; "
                      f"mu_vio_thresh={MU_VIO:g}, exact polished QP)",
               l2_policy="256 MiB buffer written between timed steps (L2 flush)",
               sampler_seed=(1 if workload in ("curve", "merge") else 0))
    if len(cells) > 1:
        cfg["cells"] = [c["label"] for c in cells]
        cfg["instances_per_cell"] = cells[0]["B"]
    if total:
        cfg["total_instances"] = total
    return cfg


# ----------------------------------------------------------------------------- CPU arms
_ORACLES, _NATIVES = {}, {}


def _oracle_for(key):
    if key not in _ORACLES:
        from oracle.dgsqp_v1 import OracleDGSQP
        kind = key[0]
        if kind == "merge":
            from oracle.merge_game import MergeGame
            _ORACLES[key] = OracleDGSQP(MergeGame(N=key[2]), reg=0.0)
        else:
            from oracle.racing_game import RacingGame
            from oracle.track import chicane_track, curve_track
            if kind == "chicane":
                _ORACLES[key] = OracleDGSQP(RacingGame(chicane_track(), M=2, N=key[2]), reg=1e-3)
            elif kind == "curve":
                g = RacingGame(curve_track(curve_angle=key[1] * math.pi / 180), M=2, N=key[2], rate_ub=(10.0, 4.5),
                               rate_lb=(-10.0, -4.5), obs_r=0.2)
                _ORACLES[key] = OracleDGSQP(g, reg=0.0)
            else:
                g = RacingGame(curve_track(curve_angle=math.pi / 2), M=key[1], N=key[2], obs_r=0.4)
                _ORACLES[key] = OracleDGSQP(g, reg=1e-3)
    return _ORACLES[key]


def _oracle_worker(args):
    key, x0, u_ws = args
    t0 = time.perf_counter()
    r = _oracle_for(key).solve(x0, u_ws)
    return bool(r["status"]), int(r["num_iters"]), r["msg"], r["u"], time.perf_counter() - t0


def _native_worker(args):
    key, x0, u_ws = args
    if key not in _NATIVES:
        sys.path.insert(0, str(ROOT / "tests"))
        import dgsqp_b200 as dg
        from hostsim_lib import HostSim
        kind = key[0]
        if kind == "merge":
            _NATIVES[key] = HostSim(dg.merge_game(key[2]), dg.merge_params(key[2]))
        elif kind == "chicane":
            _NATIVES[key] = HostSim(dg.chicane_game(key[1], key[2]), dg.chicane_params(key[2]))
        elif kind == "curve":
            _NATIVES[key] = HostSim(dg.curve_game(key[1], key[2]), dg.curve_params(key[2]))
        else:
            _NATIVES[key] = HostSim(dg.agents_game(M=key[1], N=key[2]), dg.agents_params(key[2]))
    t0 = time.perf_counter()
    r = _NATIVES[key].solve(x0, u_ws)
    return int(r["status"]) <= 1, int(r["num_iters"]), time.perf_counter() - t0


class CpuPool:
    """One persistent pool for a whole arm: workers keep their solver objects; tasks are single instances handed out
    dynamically (imap_unordered, chunksize 1), so a step's wall time is not the slowest statically assigned chunk."""

    def __init__(self, cores):
        import multiprocessing as mp
        self.cores = cores
        self.pool = mp.get_context("fork").Pool(cores)

    def run(self, worker, tasks):
        t0 = time.perf_counter()
        out = [None] * len(tasks)
        for i, r in self.pool.imap_unordered(_indexed, [(worker, i, t) for i, t in enumerate(tasks)], chunksize=1):
            out[i] = r
        return out, time.perf_counter() - t0

    def close(self):
        self.pool.close()
        self.pool.join()


def _indexed(a):
    worker, i, t = a
    return i, worker(t)


def cell_tasks(cells, samples, count):
    """`count` tasks taken round-robin over the cells (instance j of cell c), largest problems first inside a round."""
    tasks, j = [], 0
    while len(tasks) < count:
        for c, (x0, u_ws) in zip(cells, samples):
            if j < len(x0) and len(tasks) < count:
                tasks.append((c["key"], x0[j], u_ws[j]))
        j += 1
        if j > max(len(s[0]) for s in samples):
            break
    return tasks


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        import statistics
        return dict(sm_mhz=(statistics.median(self.samples) if self.samples else None), sm_max_mhz=self.max_mhz,
                    reasons=sorted(self.reasons), samples=len(self.samples))


# ----------------------------------------------------------------------------- algorithmic work model
def algorithmic_flops(game, diag, num_qp, lsqr_iters=20):
    """FP64 flops of the path by the counts the kernel reports (DESIGN.md, 'Measurement'; conventions of
    SURVEY 8(d): multiply-add = 2 flops, dense formulas without credit for agent block sparsity)."""
    import numpy as np
    n, m, N, nq, nu, M = game.n, game.m, game.N, game.n_q, game.n_u, game.M
    F_jac = N * N * nq * nq * nu + m * nq * n
    F_hess = (M + 1) * N * N * nu * nq * (nq + nu)
    F_pd = 4.0 / 3.0 * n ** 3                   # Householder tridiagonalisation (negative eigenpairs are O(n^2) each)
    F_chol = 2.0 / 3.0 * n ** 3                 # Cholesky + triangular inverse
    F_gi = 5.0 * n * n + 2.0 * 3 * M * N * N    # J'n, z, Householder update, slack evaluation
    F_lsqr = lsqr_iters * (8.0 * 3 * M * N * N + 8.0 * lsqr_iters * m)
    full, grad, gi = (diag[:, k].astype(np.float64) for k in range(3))
    return float((full * (F_jac + F_hess) + grad * F_jac + num_qp * (F_pd + F_chol) + gi * F_gi + F_lsqr).sum())


def algorithmic_bytes(game, B):
    """HBM bytes the path has to move: inputs + outputs per instance (SURVEY 8(d): ~8.5 KB at chicane size)."""
    per = 8 * (game.n_q + game.n + (game.n + game.m + (game.N + 1) * game.n_q + game.M + 3)) + 3 * 4
    return per * B


# ----------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="chicane", choices=["chicane", "curve", "agents3", "agents4", "merge"])
    ap.add_argument("--batch", type=int, default=0, help="instances per GPU per step (default: per workload)")
    ap.add_argument("--total", type=int, default=0, help="total instances per step sharded over the ranks (strong scaling)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="instances per step of the CPU arms (0 = from the time budget)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write the last step's result arrays (rank 0) to DIR/<cell>_<field>.npy, "
                         "float64; above 60 MB a fixed seeded sample of the instances")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the GPU arm (--impl ours)")
    # stdout carries exactly one JSON line: NCCL's own prints (version banner, NCCL_DEBUG output) go to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    if args.impl == "reference" and rank != 0:
        return                                              # rank 0 alone runs the CPU arm

    import numpy as np

    batch = args.batch or DEFAULT_BATCH[args.workload]
    if args.total:
        batch = (args.total + world - 1) // world
    cells = make_cells(args.workload, batch)
    config = workload_config(args.workload, cells, batch, args.total)
    scaling = "strong" if args.total else "weak"

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        pool = CpuPool(cores)
        n_steps = args.steps + args.warmup
        # calibration (untimed): one instance per core -> mean seconds per instance, workers import and build their oracles
        cal_samples = [c["sampler"](c["game"], max(2, (2 * cores) // len(cells) + 1), 1000) for c in cells]
        cal, _ = pool.run(_oracle_worker, cell_tasks(cells, cal_samples, cores))
        t_inst = float(np.mean([r[4] for r in cal]))
        n_s = args.cpu_sample or int(min(16 * cores, max(cores, CPU_ARM_BUDGET_S * cores / (n_steps * t_inst))))
        per_cell = (n_s * n_steps + len(cells) - 1) // len(cells) + 1
        samples = [c["sampler"](c["game"], per_cell, 0) for c in cells]
        tasks = cell_tasks(cells, samples, n_s * n_steps)
        vals, its, secs, busy = [], [], [], []
        for s in range(n_steps):
            out, dt = pool.run(_oracle_worker, tasks[s * n_s:(s + 1) * n_s])
            if s >= args.warmup:
                vals.append(sum(o[0] for o in out) / dt)
                its.append(sum(o[1] for o in out) / dt)
                secs.append(dt)
                busy.append(sum(o[0] for o in out) / (sum(o[4] for o in out) / cores))
        pool.close()
        value = float(np.mean(vals))
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                    ms_per_step=1e3 * float(np.mean(secs)), higher_is_better=True, scaling=scaling, vs_baseline=None,
                    dtype="f64", data="synthetic", config=config, impl="reference",
                    sqp_iters_per_sec=float(np.mean(its)),
                    cpu_baseline=dict(value=value, unit=UNIT, cores=cores, kind="port",
                                      sample=f"{n_s} {args.workload} instances per step (one persistent pool of {cores} oracle "
                                             f"processes, dynamic scheduling, BLAS single-threaded; {t_inst:.2f} s per instance "
                                             f"per core)", busy_time_value=float(np.mean(busy))),
                    e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ our arm (GPU)
    import torch
    import dgsqp_b200 as dg
    from dgsqp_b200 import _abi
    from dgsqp_b200.sharding import shard_stats, gather_stats
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: dgsqp_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    lib = _abi.load()
    stream = torch.cuda.current_stream(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    pin = lambda a: torch.from_numpy(a).pin_memory().numpy()
    for c in cells:
        x0, u_ws = c["sampler"](c["game"], c["B"], rank)         # each rank owns its shard of the global batch
        c["x0"], c["u_ws"] = x0, u_ws
        c["solver"] = dg.DGSQP(c["game"], c["params"], print_method=None, device=local_rank, mu_vio_thresh=MU_VIO)
        c["x0_d"], c["u_d"] = torch.from_numpy(x0).to(dev), torch.from_numpy(u_ws).to(dev)
        c["out"] = c["solver"].alloc_outputs(c["B"], dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def device_step():
        flush.fill_(1)
        evs = []
        for c in cells:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            c["res"] = c["solver"]._solve_batch_device(c["x0_d"], c["u_d"], None, stream.cuda_stream, c["out"], sync=False)
            e1.record(stream)
            evs.append((e0, e1))
        return evs

    for _ in range(args.warmup):
        device_step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = lib.dgsqp_kernel_launches()
    barrier()
    evs = [device_step() for _ in range(args.steps)]
    barrier()
    launches = lib.dgsqp_kernel_launches() - launches0
    cell_ms = np.array([[e0.elapsed_time(e1) for e0, e1 in step] for step in evs])      # [steps, cells]
    sampler.stop_flag = True
    sampler.join(timeout=2)
    t_dev = float(cell_ms.sum()) / 1e3
    for c in cells:
        r = c["res"]
        c["status"], c["iters"], c["qps"] = r.status.cpu().numpy(), r.num_iters.cpu().numpy(), r.qp_solves.cpu().numpy()
        c["cond"] = r.cond.cpu().numpy()
        c["diag"] = c["solver"].last_diag(c["B"])
    if args.dump_outputs and rank == 0:
        dump_outputs(pathlib.Path(args.dump_outputs), cells)

    # end-to-end through the host-buffer C-ABI call (pinned host memory, copies inside the timed region)
    for c in cells:
        c["x0_p"], c["u_p"] = pin(c["x0"]), pin(c["u_ws"])
        c["solver"].solve_batch(c["x0_p"][:64], c["u_p"][:64])
    barrier()
    e2e_secs, h2d, d2h = [], 0, 0
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for c in cells:
            c["r_h"] = c["solver"].solve_batch(c["x0_p"], c["u_p"])
        e2e_secs.append(time.perf_counter() - t0)
    barrier()
    t_e2e = sum(e2e_secs)
    for c in cells:
        r_h = c["r_h"]
        assert np.array_equal(r_h.status, c["status"]), "host path and device path disagree"
        h2d += c["x0_p"].nbytes + c["u_p"].nbytes
        d2h += sum(a.nbytes for a in (r_h.u, r_h.l, r_h.x, r_h.cost, r_h.cond, r_h.num_iters, r_h.status, r_h.qp_solves))

    # max over ranks, totals over ranks
    conv_local = int(sum((c["status"] <= 1).sum() for c in cells))
    iters_local = int(sum(c["iters"].sum() for c in cells))
    t_dev_max, t_e2e_max, conv_tot, iters_tot = t_dev, t_e2e, conv_local, iters_local
    if dist is not None:
        tt = torch.tensor([t_dev, t_e2e], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_dev_max, t_e2e_max = float(tt[0]), float(tt[1])
        cc = torch.tensor([conv_local, iters_local], dtype=torch.float64, device=dev)
        dist.all_reduce(cc, op=dist.ReduceOp.SUM)
        conv_tot, iters_tot = int(cc[0]), int(cc[1])
    cell_vecs = [shard_stats(c["status"], c["iters"], c["qps"], c["cond"]) for c in cells]
    vec = np.sum(cell_vecs, axis=0)
    vec[13], vec[14] = max(v[13] for v in cell_vecs), max(v[14] for v in cell_vecs)
    stats = gather_stats(vec)

    if rank == 0:
        K = args.steps
        value = conv_tot * K / t_dev_max
        peak_tf = C_double_peak(lib, local_rank)
        fl = sum(algorithmic_flops(c["game"], c["diag"], c["qps"].astype(np.float64)) for c in cells)
        ach_tf = fl * K / t_dev / 1e12
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except Exception:
            pass
        # DRAM traffic of the dominant kernel from the committed `ncu --set full` capture (per instance, scaled to the
        # launch): profiles/ncu_traffic.json, written from the raw page of the same kernel on one wave of instances
        traffic, traffic_src = None, None
        try:
            tj = json.loads((ROOT / "profiles" / "ncu_traffic.json").read_text()).get(config["workload"])
            if tj:
                traffic, traffic_src = tj["dram_bytes_per_instance"] * cells[0]["B"], tj["source"]
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        hbm_bytes = sum(algorithmic_bytes(c["game"], c["B"]) for c in cells)
        hbm_ach = hbm_bytes * K / t_dev / 1e9
        B_all = sum(c["B"] for c in cells)
        diag_all = np.vstack([c["diag"] for c in cells])
        line = dict(
            metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=K, warmup=args.warmup,
            ms_per_step=1e3 * t_dev_max / K, higher_is_better=True, scaling=scaling, vs_baseline=None, dtype="f64",
            data="synthetic", config=config, sqp_iters_per_sec=iters_tot * K / t_dev_max,
            solves_per_sec_all=stats["count"] * K / t_dev_max,
            e2e=dict(value=conv_tot * K / t_e2e_max, unit=UNIT, h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h),
            gpu_launches=int(launches),
            roofline=dict(bound="fp64", achieved=ach_tf, peak=peak_tf, unit="TFLOP/s",
                          frac=(ach_tf / peak_tf if peak_tf else None), traffic=traffic, traffic_source=traffic_src,
                          note="peak = FP64 FMA probe kernel measured in this run (MEASURED_PEAKS.json has no FP64 "
                               "figure); achieved = algorithmic flops from per-instance work counters / "
                               "CUDA-event time of dgsqp_solve_kernel (the only kernel of a step)"),
            roofline_hbm=dict(bound="hbm", achieved=hbm_ach, peak=hbm_peak, unit="GB/s", frac=hbm_ach / hbm_peak,
                              traffic=None, peak_source="measured" if "hbm_gbs" in peaks else "fallback"),
            clocks=sampler.summary(),
            stats={k: stats[k] for k in ("count", "converged", "conv_abs_tol", "conv_rel_tol", "max_it", "diverged",
                                         "qp_fail", "mean_iters", "std_iters", "sum_qp")},
            work=dict(full_evals=float(diag_all[:, 0].mean()), grad_evals=float(diag_all[:, 1].mean()),
                      qp_active_set_iters=float(diag_all[:, 2].mean()), algorithmic_mflop_per_instance=fl / B_all / 1e6))
        if len(cells) > 1:
            # per (theta, N) cell like scripts/process_data_curve.py:98-110
            per = []
            for j, c in enumerate(cells):
                conv = c["status"] <= 1
                per.append(dict(cell=c["label"], instances=c["B"], converged=int(conv.sum()),
                                max_it=int((c["status"] == 2).sum()), failed=int((c["status"] >= 3).sum()),
                                avg_iters=float(c["iters"][conv].mean()) if conv.any() else None,
                                avg_qp_solves=float(c["qps"][conv].mean()) if conv.any() else None,
                                ms_per_step=float(cell_ms[:, j].mean()),
                                solves_per_sec_all=c["B"] / float(cell_ms[:, j].mean()) * 1e3))
            line["cells"] = per
        if not args.no_cpu_baseline and world == 1:
            line.update(cpu_legs(args, cells, cores, np))
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def dump_outputs(out_dir, cells):
    """The arrays the timed device path returned in its last step, one file per cell and BatchResult field, in float64
    (integer fields convert exactly).  When all instances exceed DUMP_BUDGET_BYTES, every cell keeps the same fraction of
    its instances, drawn by default_rng(0) and kept in batch order: the sample depends on the batch size alone, so two
    builds run with the same arguments dump the same instances."""
    import numpy as np
    out_dir.mkdir(parents=True, exist_ok=True)
    res = [c["res"] for c in cells]
    row_bytes = [8 * sum(int(np.prod(getattr(r, f).shape[1:])) for f in OUTPUT_FIELDS) for r in res]
    frac = min(1.0, DUMP_BUDGET_BYTES / sum(rb * c["B"] for rb, c in zip(row_bytes, cells)))
    for c, r in zip(cells, res):
        keep = int(frac * c["B"])
        idx = np.sort(np.random.default_rng(0).choice(c["B"], keep, replace=False)) if keep < c["B"] else slice(None)
        for f in OUTPUT_FIELDS:
            np.save(out_dir / f"{c['label']}_{f}.npy", getattr(r, f).cpu().numpy().astype(np.float64)[idx])


def cpu_legs(args, cells, cores, np):
    """cpu_baseline (oracle port), cpu_native (kernel source compiled for the host), parity of the GPU results with the oracle
    on the same sample, and BASELINE configs[0]: single-instance latency GPU vs CPU."""
    from dgsqp_b200 import _abi
    out = {}
    pool = CpuPool(cores)
    samples = [(c["x0"], c["u_ws"]) for c in cells]
    cal, _ = pool.run(_oracle_worker, cell_tasks(cells, samples, cores))     # untimed: imports + one instance per core
    t_inst = float(np.mean([r[4] for r in cal]))
    n_s = args.cpu_sample or int(min(16 * cores, max(cores, CPU_BASELINE_BUDGET_S * cores / t_inst)))
    tasks = cell_tasks(cells, samples, n_s)
    res, dt = pool.run(_oracle_worker, tasks)
    conv = sum(o[0] for o in res)
    out["cpu_baseline"] = dict(value=conv / dt, unit=UNIT, cores=cores, kind="port",
                               sample=f"first {len(tasks)} instances of the same batch (round-robin over the cells), one "
                                      f"persistent pool of {cores} oracle processes, dynamic scheduling, {dt:.1f} s wall",
                               sqp_iters_per_sec=sum(o[1] for o in res) / dt,
                               busy_time_value=conv / (sum(o[4] for o in res) / cores))
    # parity of the GPU results with the oracle on that sample (status, iteration count; u on KKT-converged ones)
    msgs = _abi.STATUS_MSG
    same, worst, n_u_cmp = 0, 0.0, 0
    pos = {c["key"]: 0 for c in cells}
    by_key = {c["key"]: c for c in cells}
    for (key, _, _), (st_o, it_o, msg_o, u_o, _) in zip(tasks, res):
        c, i = by_key[key], pos[key]
        pos[key] += 1
        if msgs[int(c["status"][i])] == msg_o and int(c["iters"][i]) == it_o:
            same += 1
            if msg_o == "conv_abs_tol":
                u_gpu = c["res"].u[i].cpu().numpy()
                worst = max(worst, float(np.abs(u_gpu - u_o).max() / max(1.0, np.abs(u_o).max())))
                n_u_cmp += 1
    out["parity"] = dict(sample=len(tasks), identical_status_and_iters=same, max_rel_err_u_conv_abs_tol=worst,
                         compared_u=n_u_cmp, against="oracle port (product mode: exact QP, re-orthogonalised LSQR)")
    try:
        n_n = min(16 * cores, min(len(s[0]) for s in samples) * len(cells))
        ntasks = cell_tasks(cells, samples, n_n)
        pool.run(_native_worker, ntasks[:cores])                             # build / load per worker
        nres, ndt = pool.run(_native_worker, ntasks)
        out["cpu_native"] = dict(value=sum(o[0] for o in nres) / ndt, unit=UNIT, solves_per_sec_all=len(nres) / ndt,
                                 sqp_iters_per_sec=sum(o[1] for o in nres) / ndt, cores=cores,
                                 kind="kernel source compiled for the host (tests/hostsim, single-thread C++ build of the same "
                                      "solver), one instance per core",
                                 sample=f"first {len(ntasks)} instances of the same batch, {ndt:.1f} s wall")
        native_lat = [o[2] for o in nres[:8]]
    except Exception as e:                      # the yardstick is optional (needs g++ artefacts of the tests)
        out["cpu_native"] = dict(unavailable=str(e)[:200])
        native_lat = []
    pool.close()
    # BASELINE configs[0]: one instance at a time through solve_batch(B = 1) on the GPU vs the CPU solves of the same instances
    c0 = cells[-1]
    k = min(8, c0["B"])
    gpu_lat = []
    for i in range(k):
        t0 = time.perf_counter()
        c0["solver"].solve_batch(c0["x0"][i:i + 1], c0["u_ws"][i:i + 1])
        gpu_lat.append(time.perf_counter() - t0)
    own = [o[4] for (key, _, _), o in zip(tasks, res) if key == c0["key"]][:k]
    out["single_instance"] = dict(cell=c0["label"], instances=k, gpu_ms_median=1e3 * float(np.median(gpu_lat)),
                                  cpu_port_ms_median=1e3 * float(np.median(own)) if own else None,
                                  cpu_native_ms_median=1e3 * float(np.median(native_lat)) if native_lat else None,
                                  note="BASELINE configs[0]: latency of one solve (B = 1, one CTA of the persistent kernel, host "
                                       "buffers) vs one CPU solve of the same instances")
    return out


def C_double_peak(lib, device):
    import ctypes
    v = ctypes.c_double(0.0)
    rc = lib.dgsqp_measure_fp64_peak(int(device), ctypes.byref(v))
    return float(v.value) if rc == 0 else None


if __name__ == "__main__":
    main()
