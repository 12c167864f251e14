#!/usr/bin/env python3
"""Large-sample parity fixture: (status, iterations, QP solves, costs, solutions u) of the CPU oracle on the first COUNT
instances of the product sampler's 10 k chicane batch (dgsqp_b200.montecarlo.sample_head_to_head, seed 0 -- the batch
bench.py runs).  Inputs are stored with the results so that the fixture does not depend on the sampler's floating-point
environment.  u is stored for the converged instances only (NaN rows elsewhere: nothing compares them), which with the
default COUNT keeps the file under 1 MB.

    python tests/golden/make_golden_stats.py [COUNT] [PROCS]
"""
import json
import multiprocessing as mp
import os
import pathlib
import sys
import time

for _k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ[_k] = "1"       # before numpy is imported: one BLAS thread per worker process
import numpy as np  # noqa: E402

ROOT = pathlib.Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
OUT = pathlib.Path(__file__).resolve().parent


def work(args):
    i, x0, u_ws = args
    from oracle.dgsqp_v1 import OracleDGSQP
    from oracle.racing_game import RacingGame
    from oracle.track import chicane_track
    global ORC
    try:
        ORC
    except NameError:
        ORC = OracleDGSQP(RacingGame(chicane_track(), M=2, N=25))
    r = ORC.solve(x0, u_ws)
    return i, r["msg"], int(r["num_iters"]), int(r["qp_solves"]), np.asarray(r["cost"], float), np.asarray(r["u"], float)


if __name__ == "__main__":
    count = int(sys.argv[1]) if len(sys.argv) > 1 else 750
    procs = int(sys.argv[2]) if len(sys.argv) > 2 else (os.cpu_count() or 1)
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"
    import dgsqp_b200 as dg
    from dgsqp_b200.montecarlo import sample_head_to_head
    x0, u_ws = sample_head_to_head(dg.chicane_game(), 10000, seed=0)
    x0, u_ws = x0[:count], u_ws[:count]
    t0 = time.time()
    with mp.get_context("fork").Pool(procs) as pool:
        out = pool.map(work, [(i, x0[i], u_ws[i]) for i in range(count)], chunksize=4)
    out.sort(key=lambda o: o[0])
    msgs = ["conv_abs_tol", "conv_rel_tol", "max_it", "diverged", "qp_fail", "time_limit"]
    status = np.array([msgs.index(o[1]) for o in out], dtype=np.int32)
    u = np.stack([o[5] for o in out]).astype(np.float64)
    u[status > 1] = np.nan
    np.savez_compressed(OUT / "chicane_N25_seed0_stats.npz", x0=x0, u_ws=u_ws, status=status,
                        num_iters=np.array([o[2] for o in out], dtype=np.int32),
                        qp_solves=np.array([o[3] for o in out], dtype=np.int32),
                        cost=np.stack([o[4] for o in out]), u=u)
    (OUT / "chicane_N25_seed0_stats.json").write_text(json.dumps(dict(
        name="chicane_N25_seed0_stats", count=count, seed=0, generator="tests/golden/make_golden_stats.py (CPU oracle)",
        seconds=time.time() - t0, hist={m: sum(o[1] == m for o in out) for m in msgs}), indent=1))
    print("done", count, "instances in", time.time() - t0, "s")
