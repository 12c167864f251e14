#!/usr/bin/env python3
"""Monte-Carlo sweep on the GPU in place of the reference's per-instance loops:

    python scripts/monte_carlo.py chicane --num 10000            # scripts/DGSQP_ALGAMES_monte_carlo_chicane.py
    python scripts/monte_carlo.py curve --theta 45 75 90 --N 10 15 20 25 --num 1000    # ..._curve.py (seed 1, reg 0)
    python scripts/monte_carlo.py agents --M 3 --num 1000        # scripts/DGSQP_monte_carlo_agents.py
    python scripts/monte_carlo.py merge --num 1000 [--out merge.pkl]   # scripts/DGSQP_merge_monte_carlo.py (seed 1)

--sample-on-device draws the instances on the GPU (dgsqp_b200.montecarlo.sample_*_cuda: same distributions, trial-major
stream; for merge the same instances) and keeps them there for the solve.

Prints the summary table of scripts/process_data_curve.py per cell and optionally pickles the records
(``results['dgsqp']`` of the reference's data files)."""
import argparse
import pathlib
import pickle
import sys

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parents[1]))
import dgsqp_b200 as dg
from dgsqp_b200.drivers import default_sampler, run_monte_carlo, summary_table


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("game", choices=["chicane", "curve", "agents", "merge"])
    ap.add_argument("--num", type=int, default=1000)
    ap.add_argument("--theta", type=float, nargs="+", default=[45.0])
    ap.add_argument("--N", type=int, nargs="+", default=None)
    ap.add_argument("--M", type=int, default=3)
    ap.add_argument("--seed", type=int, default=None)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    ap.add_argument("--sample-on-device", action="store_true", help="draw the instances on the GPU")
    a = ap.parse_args()
    cells = []
    if a.game == "chicane":
        for N in a.N or [25]:
            cells.append((f"chicane N: {N}", dg.chicane_game(N=N), dg.chicane_params(N), 0))
    elif a.game == "curve":
        for th in a.theta:
            for N in a.N or [25]:
                cells.append((f"Track parameter: {th:g}, N: {N}", dg.curve_game(th, N), dg.curve_params(N), 1))
    elif a.game == "agents":
        for N in a.N or [25]:
            cells.append((f"agents M: {a.M}, N: {N}", dg.agents_game(a.M, 90.0, N), dg.agents_params(N), 0))
    else:
        for N in a.N or [20]:
            cells.append((f"merge N: {N}", dg.merge_game(N), dg.merge_params(N), 1))
    out = {}
    for title, game, params, seed in cells:
        solver = dg.DGSQP(game, params, print_method=None, device=a.device)
        sampler = default_sampler(game, device=a.device) if a.sample_on_device else None
        records, stats = run_monte_carlo(solver, a.num, sampler=sampler, seed=seed if a.seed is None else a.seed)
        summary_table(records, title)
        out[title] = dict(dgsqp=records, stats=stats)
    if a.out:
        with open(a.out, "wb") as f:
            pickle.dump(out, f)


if __name__ == "__main__":
    main()
