"""Batched Monte-Carlo driver: the loop of the reference's scripts with the per-instance solve replaced by one
``solve_batch`` per chunk.

Mirrors ``scripts/DGSQP_ALGAMES_monte_carlo_chicane.py:381-511`` / ``..._curve.py`` / ``DGSQP_monte_carlo_agents.py:232-330``
/ ``DGSQP_merge_monte_carlo.py:424-510``: sample instances (initial conditions + warm start), solve, collect one record per
sample with the keys the post-processing scripts read (``scripts/process_data_curve.py:44-110``,
``process_data_merge.py:30-67``: ``solve_info['status' | 'msg' | 'num_iters' | 'qp_solves' | 'cond' | 'time' | 'cost']``),
and print the same summary table.  The solver is any object with the ``solve_batch(x0, u_ws)`` of :class:`dgsqp_b200.DGSQP`.
"""
import time

import numpy as np

from . import _abi
from .sharding import shard_stats, combine_stats


def default_sampler(game, device=None):
    """The sampler of the script a game record was taken from; with a CUDA ``device`` ordinal its GPU version, which
    returns CUDA tensors (``montecarlo.sample_*_cuda``)."""
    from .games import MergeGame
    from .montecarlo import sample_head_to_head, sample_agents, sample_merge
    if device is not None:
        from . import montecarlo as mc
        fn = mc.sample_merge_cuda if isinstance(game, MergeGame) else \
            mc.sample_head_to_head_cuda if game.M == 2 else mc.sample_agents_cuda
        return lambda B, seed: fn(game, B, seed=seed, device=device)
    if isinstance(game, MergeGame):
        return lambda B, seed: sample_merge(game, B, seed=seed)
    if game.M == 2:
        return lambda B, seed: sample_head_to_head(game, B, seed=seed)
    return lambda B, seed: sample_agents(game, B, seed=seed)


def run_monte_carlo(solver, num, sampler=None, seed=0, chunk=10000, keep_trajectories=False):
    """Solve ``num`` sampled instances in chunks of ``chunk``.  Returns ``(records, stats)``: ``records`` is the list the
    reference pickles as ``results['dgsqp']`` (one dict with ``solve_info`` and ``init`` per sample), ``stats`` the merged
    statistics (``sharding.combine_stats``).  A sampler that returns CUDA tensors keeps the instances on the device: each
    chunk is solved on the device path and its results are copied to the host once to build the records."""
    game = solver.game
    sampler = default_sampler(game) if sampler is None else sampler
    x0, u_ws = sampler(num, seed)
    on_device = hasattr(x0, "is_cuda")
    records, vectors = [], []
    for lo in range(0, num, chunk):
        hi = min(num, lo + chunk)
        t0 = time.perf_counter()
        res = solver.solve_batch(x0[lo:hi], u_ws[lo:hi])
        dt = (time.perf_counter() - t0) / max(hi - lo, 1)          # amortised wall time per instance
        init_x0, init_u = x0[lo:hi], u_ws[lo:hi]
        if on_device:
            fields = ("status", "num_iters", "qp_solves", "cost", "cond") + (("u", "l", "x") if keep_trajectories else ())
            for f in fields:
                setattr(res, f, getattr(res, f).cpu().numpy())
            init_x0, init_u = init_x0.cpu().numpy(), init_u.cpu().numpy()
        vectors.append(shard_stats(res.status, res.num_iters, res.qp_solves, res.cond))
        for i in range(hi - lo):
            info = dict(time=dt, num_iters=int(res.num_iters[i]), status=bool(res.status[i] <= 1),
                        msg=_abi.STATUS_MSG[int(res.status[i])], qp_solves=int(res.qp_solves[i]), cost=res.cost[i].copy(),
                        cond=dict(p_feas=float(res.cond[i, 0]), comp=float(res.cond[i, 1]), stat=float(res.cond[i, 2])))
            rec = dict(solve_info=info, init=dict(x0=init_x0[i].copy(), u_ws=init_u[i].copy()))
            if keep_trajectories:
                rec["u"], rec["l"] = res.u[i].copy(), res.l[i].copy()
                rec["q"] = res.x[i].reshape(game.N + 1, game.n_q).copy()
            records.append(rec)
    return records, combine_stats(vectors)


def summary_table(records, title="", print_method=print):
    """The per-cell table of ``scripts/process_data_curve.py:98-110`` (DG-SQP column) from a list of records."""
    msgs = [r["solve_info"]["msg"] for r in records]
    conv = [r["solve_info"] for r in records if r["solve_info"]["status"]]
    n_conv = len(conv)
    n_max = sum(m in ("max_it", "max_iters") for m in msgs)
    n_div = sum(m in ("diverged", "qp_fail") for m in msgs)
    it = np.array([c["num_iters"] for c in conv], dtype=float)
    qp = np.array([c["qp_solves"] for c in conv], dtype=float)
    tm = np.array([c["time"] for c in conv], dtype=float)
    f = lambda a, fn: (fn(a) if len(a) else float("nan"))
    w = 9
    rows = [("Converged", f"{n_conv:d}"), ("Failed", f"{n_div:d}"), ("Max", f"{n_max:d}"),
            ("Avg iters", f"{f(it, np.mean):4.2f}"), ("Std iters", f"{f(it, np.std):4.2f}"),
            ("Avg solves", f"{f(qp, np.mean):4.2f}"), ("Std solves", f"{f(qp, np.std):4.2f}"),
            ("Avg time", f"{f(tm, np.mean):.2e}"), ("Std time", f"{f(tm, np.std):.2e}")]
    print_method("========================================")
    if title:
        print_method(title)
    print_method("           |   SQP   ")
    for name, val in rows:
        print_method("%s|%s" % (name.ljust(11), val.rjust(w)))
    return dict(converged=n_conv, failed=n_div, max_it=n_max, avg_iters=f(it, np.mean), avg_solves=f(qp, np.mean))
