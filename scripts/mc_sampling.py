#!/usr/bin/env python3
"""Cost of drawing the Monte-Carlo instances, device against host, next to the solve of the same batch.

    python scripts/mc_sampling.py [--repeats 5] [--out profiles/mc_sampling.json] [--skip-host]

For every bench.py workload at its default batch (chicane 10 000, curve 12 cells x 1 000, agents3 4 000, agents4 2 000,
merge 10 000) and for merge at 1 000 000 instances:
  device_ms      dgsqp_b200.montecarlo.sample_*_cuda, CUDA events around warmed-up calls (median, min, max of --repeats)
  trials         trials the device sampler consumed (last accepted trial id + 1)
  host_s         the NumPy sampler of bench.py at the same size (agents4: at host_instances = 100, not extrapolated)
  solve_ms       DGSQP.solve_batch on the device path for the sampled batch (CUDA events)
  e2e            sample + solve_batch + last_stats, host clock, instances / s
The card name and power limit are read with a read-only nvidia-smi query and written beside the numbers.
"""
import argparse
import json
import pathlib
import subprocess
import sys
import time

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402


def cells():
    import dgsqp_b200 as dg
    from dgsqp_b200 import montecarlo as mc
    h2h = (mc.sample_head_to_head, mc.sample_head_to_head_cuda)
    ag = (mc.sample_agents, mc.sample_agents_cuda)
    mg = (mc.sample_merge, mc.sample_merge_cuda)
    out = [("chicane", [(dg.chicane_game(), dg.chicane_params(), 10000, 0)], h2h, None)]
    out.append(("curve", [(dg.curve_game(th, N), dg.curve_params(N), 1000, 1) for th in (45.0, 75.0, 90.0)
                          for N in (10, 15, 20, 25)], h2h, None))
    out.append(("agents3", [(dg.agents_game(3), dg.agents_params(), 4000, 0)], ag, None))
    out.append(("agents4", [(dg.agents_game(4), dg.agents_params(), 2000, 0)], ag, 100))
    out.append(("merge", [(dg.merge_game(), dg.merge_params(), 10000, 1)], mg, None))
    out.append(("merge_1M", [(dg.merge_game(), dg.merge_params(), 1000000, 1)], mg, None))
    return out


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "mc_sampling.json"))
    ap.add_argument("--skip-host", action="store_true", help="do not time the host samplers")
    a = ap.parse_args()
    import torch
    import dgsqp_b200 as dg
    if not torch.cuda.is_available():
        raise SystemExit("mc_sampling.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    results = dict(gpu=gpu_info(), torch=torch.__version__, repeats=a.repeats, workloads={})
    print("[mc_sampling]", results["gpu"], flush=True)
    for name, cs, (host_fn, dev_fn), host_B in cells():
        rec = dict(instances=0, trials=0, device_ms=[], solve_ms=0.0, e2e_s=0.0, host_s=None, host_instances=None)
        solvers = [dg.DGSQP(g, p, print_method=None, mu_vio_thresh=1e-10) for g, p, _, _ in cs]
        for (g, p, B, seed), solver in zip(cs, solvers):       # warm-up: module load, allocator, every shape
            x0, u = dev_fn(g, min(B, 64), seed=seed)
            solver.solve_batch(x0, u)
        torch.cuda.synchronize()
        for r in range(a.repeats):                               # sampling alone, every cell of the workload per repeat
            e0, e1 = ev(), ev()
            e0.record()
            for g, p, B, seed in cs:
                dev_fn(g, B, seed=seed)
            e1.record()
            e1.synchronize()
            rec["device_ms"].append(e0.elapsed_time(e1))
        for (g, p, B, seed), solver in zip(cs, solvers):        # sample + solve + statistics, once
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e0, e1, e2 = ev(), ev(), ev()
            e0.record()
            x0, u, trial = dev_fn(g, B, seed=seed, return_trials=True)
            e1.record()
            solver.solve_batch(x0, u)
            e2.record()
            stats = solver.last_stats()
            rec["e2e_s"] += time.perf_counter() - t0
            e2.synchronize()
            rec["solve_ms"] += e1.elapsed_time(e2)
            rec["instances"] += B
            rec["trials"] += int(trial[-1].item()) + 1
            rec.setdefault("converged", 0)
            rec["converged"] += int(stats[1] + stats[2])
            del x0, u, trial
        if not a.skip_host:
            t0 = time.perf_counter()
            n = 0
            for g, p, B, seed in cs:
                Bh = host_B or B
                host_fn(g, Bh, seed=seed)
                n += Bh
            rec["host_s"], rec["host_instances"] = time.perf_counter() - t0, n
        d = np.array(rec["device_ms"])
        rec["device_ms"] = dict(median=float(np.median(d)), min=float(d.min()), max=float(d.max()), all=d.tolist())
        rec["device_share_of_solve"] = rec["device_ms"]["median"] / rec["solve_ms"]
        rec["e2e_instances_per_s"] = rec["instances"] / rec["e2e_s"]
        if rec["host_s"] is not None:
            per_host = rec["host_s"] / rec["host_instances"]
            per_dev = rec["device_ms"]["median"] * 1e-3 / rec["instances"]
            rec["host_over_device_per_instance"] = per_host / per_dev
        results["workloads"][name] = rec
        print(f"[mc_sampling] {name}: {rec['instances']} instances / {rec['trials']} trials, device "
              f"{rec['device_ms']['median']:.2f} ms [{rec['device_ms']['min']:.2f}, {rec['device_ms']['max']:.2f}], solve "
              f"{rec['solve_ms']:.1f} ms ({100 * rec['device_share_of_solve']:.2f} %), e2e {rec['e2e_instances_per_s']:.0f}/s, "
              f"host {rec['host_s']} s for {rec['host_instances']}", flush=True)
    out = pathlib.Path(a.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(json.dumps(results, indent=1))
    print("[mc_sampling] wrote", out)


if __name__ == "__main__":
    main()
