#!/usr/bin/env python3
"""How far is the PRODUCT mode of the oracle (what the CUDA path implements) from the LITERAL reference rules?

The reference cannot run offline (CasADi / OSQP), so the deviations D1-D3 of DESIGN.md are quantified by running the
oracle itself in literal mode on the large-sample chicane fixture (tests/golden/chicane_N25_seed0_stats.npz, whose stored
results are the product mode) and counting the instances whose ``(msg, num_iters)`` change:

  D1  QP: OSQP restated at its defaults + polish (oracle/osqp_admm.py) instead of the exact KKT point
  D2  ``_get_mu`` threshold 0 (DGSQP.py:560) instead of 1e-10
  D3  SciPy's plain ``lsqr(GG', Gq)`` (DGSQP.py:323-324) instead of the re-orthogonalised recurrences

    python scripts/literal_mode_study.py [--count 1000] [--procs 6] [--variants all,d1,d2,d3,all_rho25,all_rho100]

Writes profiles/r2_literal_mode_study.json and prints the agreement table.  CPU only.
"""
import argparse
import json
import multiprocessing as mp
import os
import pathlib
import sys
import time

for _k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ[_k] = "1"
ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import numpy as np  # noqa: E402

VARIANTS = {
    "all": dict(qp_method="osqp", mu_vio_thresh=0.0, dual_init_method="scipy"),
    "d1": dict(qp_method="osqp"),
    "d2": dict(mu_vio_thresh=0.0),
    "d3": dict(dual_init_method="scipy"),
    # chaos floor: the PRODUCT mode against itself with the dual initialisation perturbed by one ulp / by 1e-12 relative
    "ulp": dict(l0_perturb=2.2e-16),
    "eps1e-12": dict(l0_perturb=1e-12),
    "all_rho25": dict(qp_method="osqp", mu_vio_thresh=0.0, dual_init_method="scipy", osqp_kw=dict(adaptive_rho_interval=25)),
    "all_rho100": dict(qp_method="osqp", mu_vio_thresh=0.0, dual_init_method="scipy", osqp_kw=dict(adaptive_rho_interval=100)),
}
_SOLVERS = {}


def _work(args):
    variant, i, x0, u_ws = args
    from oracle.dgsqp_v1 import OracleDGSQP
    from oracle.racing_game import RacingGame
    from oracle.track import chicane_track
    if variant not in _SOLVERS:
        _SOLVERS[variant] = OracleDGSQP(RacingGame(chicane_track(), M=2, N=25), reg=1e-3, **VARIANTS[variant])
    s = _SOLVERS[variant]
    t0 = time.perf_counter()
    r = s.solve(x0, u_ws)
    qs = s.qp_stats
    osqp = [q for q in qs if "osqp_status" in q]
    return dict(i=i, msg=r["msg"], num_iters=int(r["num_iters"]), qp_solves=int(r["qp_solves"]), u=r["u"],
                secs=time.perf_counter() - t0, n_qp=len(qs), n_osqp_unsolved=sum(q["osqp_status"] != "solved" for q in osqp),
                n_osqp_unpolished=sum(not q["polished"] for q in osqp), osqp_iters=sum(q["iters"] for q in osqp))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--count", type=int, default=1000)
    ap.add_argument("--procs", type=int, default=max(1, (os.cpu_count() or 2) - 2))
    ap.add_argument("--variants", default="all,d1,d2,d3")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r2_literal_mode_study.json"))
    args = ap.parse_args()
    d = np.load(ROOT / "tests/golden/chicane_N25_seed0_stats.npz")
    msgs = ["conv_abs_tol", "conv_rel_tol", "max_it", "diverged", "qp_fail", "time_limit"]
    n = min(args.count, len(d["status"]))
    report = {}
    out_path = pathlib.Path(args.out)
    if out_path.exists():
        report = json.loads(out_path.read_text())
    with mp.get_context("fork").Pool(args.procs) as pool:
        for variant in args.variants.split(","):
            t0 = time.time()
            rs = pool.map(_work, [(variant, i, d["x0"][i], d["u_ws"][i]) for i in range(n)], chunksize=1)
            same = same_status = 0
            errs, changed = [], []
            for r in rs:
                i = r["i"]
                pm, pi = msgs[int(d["status"][i])], int(d["num_iters"][i])
                same_status += r["msg"] == pm
                if r["msg"] == pm and r["num_iters"] == pi:
                    same += 1
                    if pm == "conv_abs_tol":
                        errs.append(float(np.abs(r["u"] - d["u"][i]).max() / max(1.0, np.abs(d["u"][i]).max())))
                else:
                    changed.append((i, pm, pi, r["msg"], r["num_iters"]))
            conv_lit = sum(r["msg"].startswith("conv") for r in rs)
            conv_prod = int((d["status"][:n] <= 1).sum())
            errs = np.array(errs) if errs else np.zeros(1)
            rep = dict(settings={k: (v if not isinstance(v, dict) else v) for k, v in VARIANTS[variant].items()}, instances=n,
                       identical_msg_and_iters=same, identical_msg=int(same_status), converged_literal=conv_lit,
                       converged_product=conv_prod, mean_iters_literal=float(np.mean([r["num_iters"] for r in rs])),
                       mean_iters_product=float(d["num_iters"][:n].mean()),
                       u_rel_err_on_identical_conv_abs=dict(median=float(np.median(errs)), p99=float(np.quantile(errs, 0.99)),
                                                            max=float(errs.max()), above_1e6=int((errs > 1e-6).sum()), count=len(errs)),
                       qp_total=sum(r["n_qp"] for r in rs), osqp_not_solved=sum(r["n_osqp_unsolved"] for r in rs),
                       osqp_not_polished=sum(r["n_osqp_unpolished"] for r in rs), osqp_admm_iters=sum(r["osqp_iters"] for r in rs),
                       cpu_seconds=float(sum(r["secs"] for r in rs)), wall_seconds=time.time() - t0,
                       changed_first20=changed[:20])
            report[variant] = rep
            print(f"{variant:10s} identical (msg, iters) {same}/{n}  identical msg {same_status}/{n}  converged literal {conv_lit} / "
                  f"product {conv_prod}  u err (identical conv_abs) max {errs.max():.1e}  QPs {rep['qp_total']} "
                  f"(osqp unsolved {rep['osqp_not_solved']}, unpolished {rep['osqp_not_polished']})  {time.time() - t0:.0f} s", flush=True)
            out_path.write_text(json.dumps(report, indent=1))


if __name__ == "__main__":
    main()
