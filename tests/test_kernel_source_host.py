"""The CUDA kernel source, compiled for the host as a one-thread CTA (tests/hostsim), against the oracle.
Catches arithmetic / control-flow / indexing errors on machines without a GPU; the multi-thread behaviour
(synchronisation, reductions) is covered by the -m gpu tests."""
import json
import pathlib

import numpy as np
import pytest

import dgsqp_b200 as dg
from hostsim_lib import HostSim
from oracle.dgsqp_v1 import OracleDGSQP, nearest_pd
from oracle.qp import solve_qp_gi, kkt_residuals
from oracle.racing_game import RacingGame
from oracle.track import chicane_track, curve_track

GOLDEN = pathlib.Path(__file__).parent / "golden"
MSG = {0: "conv_abs_tol", 1: "conv_rel_tol", 2: "max_it", 3: "diverged", 4: "qp_fail"}


def _instance(og, seed=0):
    rng = np.random.default_rng(seed)
    M = og.M
    x0 = np.concatenate([[0, 0, 2.2 + 0.3 * a, 0.0, 0.4 + 0.9 * a, 0.5 - 0.5 * a] for a in range(M)])
    for a in range(M):
        x0[6 * a], x0[6 * a + 1], _ = og.track.local_to_global((x0[6 * a + 4], x0[6 * a + 5], 0.0))
    u = rng.normal(size=og.n) * 0.15
    l = np.abs(rng.normal(size=og.m)) * 0.3 * (rng.random(og.m) < 0.3)
    return x0, u, l


@pytest.mark.parametrize("M,N", [(2, 25), (3, 10), (4, 6)])
def test_evaluate_and_G_products(M, N, asan=False):
    tr_o = curve_track(curve_angle=np.pi / 2) if M > 2 else chicane_track()
    og = RacingGame(tr_o, M=M, N=N, obs_r=0.4)
    game = dg.agents_game(M=M, N=N) if M > 2 else dg.chicane_game(N=N)
    hs = HostSim(game, dg.DGSQPParams(N=N, nonmono_ls=True), asan=asan)
    x0, u, l = _instance(og, seed=M)
    Q, q, G, g, x = og.evaluate(u, l, x0, np.zeros(og.n_u), True)
    Q2, q2, gtl2, g2, x2 = hs.evaluate(x0, u, l)
    sc = max(1.0, np.abs(Q).max())
    assert np.abs(x - x2).max() < 1e-12 and np.abs(g - g2).max() < 1e-12 and np.abs(q - q2).max() < 1e-11
    assert np.abs(G.T @ l - gtl2).max() < 1e-11 and np.abs(Q - Q2).max() < 1e-11 * sc
    assert np.abs(G - hs.G_dense()).max() < 1e-12
    rng = np.random.default_rng(0)
    v, w = rng.normal(size=og.n), rng.normal(size=og.m)
    assert np.abs(G @ v - hs.G_times(v)).max() < 1e-11 and np.abs(G.T @ w - hs.GT_times(w)).max() < 1e-11


def test_nearest_pd_and_qp(chicane_full):
    og, game, params = chicane_full
    hs = HostSim(game, params)
    for seed in range(3):
        x0, u, l = _instance(og, seed)
        Q, q, G, g, _ = og.evaluate(u, l, x0, np.zeros(4), True)
        hs.evaluate(x0, u, l)
        H = nearest_pd(Q) + 1e-3 * np.eye(og.n)
        H2, nneg = hs.nearest_pd(Q)
        assert nneg == int((np.linalg.eigvalsh((Q + Q.T) / 2) < 0).sum()) and nneg > 0
        assert np.abs(H - H2).max() < 1e-10 * max(1.0, np.abs(H).max())
        du, lam = solve_qp_gi(H, q, G, g)
        st, du2, lam2, it = hs.qp(H, q)
        assert st == 0 and np.abs(du - du2).max() < 1e-8 and np.abs(lam - lam2).max() < 1e-7
        r = kkt_residuals(H, q, G, g, du2, lam2)
        assert r["stat"] < 1e-8 and r["feas"] < 1e-9 and r["dual"] == 0.0 and r["comp"] < 1e-8


def test_nearest_pd_many_negative_eigenvalues_and_clusters(chicane_full):
    """More negative eigenvalues than one inverse-iteration chunk, with a degenerate cluster."""
    og, game, params = chicane_full
    hs = HostSim(game, params)
    rng = np.random.default_rng(3)
    n = og.n
    U, _ = np.linalg.qr(rng.normal(size=(n, n)))
    s = np.concatenate([-np.linspace(0.5, 3.0, 20), [-1.0, -1.0, -1.0 - 1e-9], rng.uniform(0.1, 5, n - 23)])
    Q = (U * s) @ U.T
    H2, nneg = hs.nearest_pd(Q)
    assert nneg == 23
    assert np.abs(H2 - (nearest_pd(Q) + 1e-3 * np.eye(n))).max() < 1e-9
    Hp, nn0 = hs.nearest_pd((U * np.abs(s)) @ U.T)
    assert nn0 == 0


def test_nearest_pd_cluster_across_inverse_iteration_chunks(chicane_full):
    """A degenerate cluster of negative eigenvalues that straddles the boundary between two inverse-iteration chunks
    (16 vectors each): its vectors must be orthogonalised against the ones the previous chunk finished (ADVICE r1)."""
    og, game, params = chicane_full
    hs = HostSim(game, params)
    rng = np.random.default_rng(11)
    n = og.n
    U, _ = np.linalg.qr(rng.normal(size=(n, n)))
    s = np.concatenate([-np.linspace(10.0, 4.0, 14), [-2.0, -2.0, -2.0 - 1e-12, -2.0 + 1e-12, -2.0], [-1.0, -0.5],
                        rng.uniform(0.1, 5, n - 21)])
    Q = (U * s) @ U.T
    H2, nneg = hs.nearest_pd(Q)
    assert nneg == 21
    assert np.abs(H2 - (nearest_pd(Q) + 1e-3 * np.eye(n))).max() < 1e-9
    assert np.linalg.eigvalsh(H2).min() > 0.9e-3


def test_lsqr_dual_init(chicane_full):
    """Dual initialisation: same recurrences / stopping rules as scipy.sparse.linalg.lsqr with reorthogonalised
    Golub-Kahan vectors.  Kernel source == oracle to rounding, iteration for iteration; the literal SciPy call
    (what the reference runs) lies within its own reproducibility band of that result."""
    import scipy.sparse as sp
    import scipy.sparse.linalg as spla
    og, game, params = chicane_full
    hs = HostSim(game, params)
    sol = OracleDGSQP(og)
    for seed in range(3):
        x0, u, _ = _instance(og, seed)
        q, G, _, _ = og.evaluate(u, np.zeros(og.m), x0, np.zeros(4), False)
        l0 = sol.dual_init(q, G)
        l0h, itn = hs.lsqr(x0, u)
        assert itn == sol.lsqr_iters
        assert np.abs(l0 - l0h).max() < 1e-10 * max(1.0, np.abs(l0).max())
        # SciPy itself: dense vs sparse operator already disagree at the 1e-5..1e-2 level
        dense = np.maximum(0, -spla.lsqr(G @ G.T, G @ q)[0])
        Gs = sp.csc_matrix(G)
        sparse = np.maximum(0, -spla.lsqr(Gs @ Gs.T, G @ q)[0])
        spread = np.abs(dense - sparse).max()
        assert np.abs(l0 - dense).max() < max(50 * spread, 5e-2 * np.abs(l0).max())


def test_solve_matches_golden(chicane_full):
    """Full solves of the kernel source vs. the oracle's committed results.  With the oracle's dual
    initialisation handed in (so the LSQR chaos is out of the picture) the iteration path must agree."""
    _, game, params = chicane_full
    hs = HostSim(game, params)
    data = np.load(GOLDEN / "chicane_N25_seed0.npz")
    meta = json.loads((GOLDEN / "chicane_N25_seed0.json").read_text())
    B = data["x0"].shape[0]
    same = 0
    for i in range(B):
        r = hs.solve(data["x0"][i], data["u_ws"][i], data["l_init"][i])
        ok = MSG[r["status"]] == meta["msg"][i] and r["num_iters"] == meta["num_iters"][i]
        same += ok
        if ok and meta["msg"][i] == "conv_abs_tol":
            assert np.abs(r["u"] - data["u"][i]).max() < 1e-6 * max(1.0, np.abs(data["u"][i]).max())
            assert np.abs(r["l"] - data["l"][i]).max() < 1e-6 * max(1.0, np.abs(data["l"][i]).max())
            assert np.abs(r["x"].ravel() - data["x"][i]).max() < 1e-6 * max(1.0, np.abs(data["x"][i]).max())
    assert same >= 0.95 * B, f"identical (status, iters) on {same}/{B}"


# tolerance: the curve configuration runs with reg = 0 (DGSQP_ALGAMES_monte_carlo_curve.py:161), so the projected
# Hessian keeps eigenvalues of 1e-10 (cond ~1e11) and the QP step amplifies the 1e-13 differences between
# LAPACK's eigh and the device eigen-solver; 1e-6 is kept for the regularised games.
@pytest.mark.parametrize("name,mk,tol,limit", [
    ("curve45_N15_seed1", lambda: (dg.curve_game(45.0, 15), dg.curve_params(15)), 1e-4, None),
    ("agents3_N15_seed0", lambda: (dg.agents_game(3, 90.0, 15), dg.agents_params(15)), 1e-6, None),
    # round-2 fixtures (tests/golden/make_golden_r2.py): the N = 25 curves and four agents at N = 25 (n = 200)
    ("curve75_N25_seed1", lambda: (dg.curve_game(75.0, 25), dg.curve_params(25)), 1e-6, None),
    ("curve90_N25_seed1", lambda: (dg.curve_game(90.0, 25), dg.curve_params(25)), 1e-6, None),
    ("agents4_N25_seed0", lambda: (dg.agents_game(4, 90.0, 25), dg.agents_params(25)), 1e-6, 4)])
def test_solve_other_games_match_golden(name, mk, tol, limit):
    game, params = mk()
    hs = HostSim(game, params)
    data = np.load(GOLDEN / f"{name}.npz")
    meta = json.loads((GOLDEN / f"{name}.json").read_text())
    B = data["x0"].shape[0] if limit is None else limit
    same = 0
    for i in range(B):
        r = hs.solve(data["x0"][i], data["u_ws"][i], data["l_init"][i])
        ok = MSG[r["status"]] == meta["msg"][i] and r["num_iters"] == meta["num_iters"][i]
        same += ok
        if ok and meta["msg"][i] == "conv_abs_tol":
            assert np.abs(r["u"] - data["u"][i]).max() < tol * max(1.0, np.abs(data["u"][i]).max())
    # reg = 0 at N = 25: the oracle itself keeps 9-10 of the 12 paths under a one-ulp perturbation (profiles/r2_chaos_floor_curve_N25.json)
    need = 8 if name.startswith(("curve75_N25", "curve90_N25")) else 0.9 * B
    assert same >= need, f"identical (status, iters) on {same}/{B}"


def test_v2_policy_matches_oracle_and_golden():
    """Kernel source of the v2 step policy (sqp_v2.cuh) against the v2 oracle: live on a Newton-like and a 'max'
    decrease setting, and on the committed golden instances."""
    from oracle.dgsqp_v2 import OracleDGSQPV2
    from oracle.sampler import sample_head_to_head
    N = 15
    game, og = dg.chicane_game(N=N), RacingGame(chicane_track(), M=2, N=N)
    for kw in (dict(reg=1e-3, p_tol=1e-3, d_tol=1e-3, sqp_iters=50),
               dict(reg=1.0, reg_decay=0.8, sqp_iters=60, merit_decrease_condition="max")):
        hs, sol = HostSim(game, dg.DGSQPV2Params(N=N, **kw)), OracleDGSQPV2(og, **kw)
        rng = np.random.default_rng(0)
        for i in range(3):
            x0, u_ws = sample_head_to_head(og, rng)
            r, h = sol.solve(x0, u_ws), hs.solve(x0, u_ws)
            assert MSG[h["status"]] == r["msg"] and h["num_iters"] == r["num_iters"] and h["qp_solves"] == r["qp_solves"]
            assert h["diag"][6] == r["m_steps"]
            assert np.abs(h["u"] - r["u"]).max() < 1e-9 and np.abs(h["l"] - r["l"]).max() < 1e-8
    data = np.load(GOLDEN / "chicane_v2_N15_seed0.npz")
    meta = json.loads((GOLDEN / "chicane_v2_N15_seed0.json").read_text())
    hs = HostSim(game, dg.DGSQPV2Params(N=N, **meta["solver_kw"]))
    for i in range(4):
        h = hs.solve(data["x0"][i], data["u_ws"][i], data["l_init"][i])
        assert MSG[h["status"]] == meta["msg"][i] and h["num_iters"] == meta["num_iters"][i]
        assert np.abs(h["u"] - data["u"][i]).max() < 1e-8


def test_v2_sum_obj_merit_matches_oracle():
    """v2 merit 'sum_obj_l1' (DGSQP_v2.py:1149-1151,1161-1164) in the kernel source against the oracle: with the
    non-monotone policy (m-steps against the merit memory) and with nms = False, where every iteration runs the
    Armijo line search on phi = sum_a J^a + mu sum(s)."""
    from oracle.dgsqp_v2 import OracleDGSQPV2
    from oracle.sampler import sample_head_to_head
    N = 10
    game, og = dg.chicane_game(N=N), RacingGame(chicane_track(), M=2, N=N)
    ls_total = 0
    for kw in (dict(reg=1e-3, reg_decay=0.9, nms=False, sqp_iters=30, merit_decrease=0.3, merit_function="sum_obj_l1"),
               dict(reg=1e-1, reg_decay=0.8, nms_frequency=2, sqp_iters=40, merit_function="sum_obj_l1",
                    merit_decrease_condition="max")):
        hs, sol = HostSim(game, dg.DGSQPV2Params(N=N, **kw)), OracleDGSQPV2(og, **kw)
        rng = np.random.default_rng(1)
        for i in range(3):
            x0, u_ws = sample_head_to_head(og, rng)
            r, h = sol.solve(x0, u_ws), hs.solve(x0, u_ws)
            assert MSG[h["status"]] == r["msg"] and h["num_iters"] == r["num_iters"] and h["qp_solves"] == r["qp_solves"]
            assert h["diag"][7] == sol.n_ls_evals
            ls_total += sol.n_ls_evals
            assert np.abs(h["u"] - r["u"]).max() < 1e-9 and np.abs(h["l"] - r["l"]).max() < 1e-8
    assert ls_total > 0            # the line search on the summed costs was exercised


def test_kernel_source_under_asan_ubsan():
    """One evaluate + nearestPD + QP + short solve of the kernel source under AddressSanitizer / UBSan
    (separate process: the sanitizer runtime has to be preloaded)."""
    import os
    import subprocess
    import sys
    import hostsim_lib
    hostsim_lib.build(asan=True)
    libasan = subprocess.check_output(["gcc", "-print-file-name=libasan.so"], text=True).strip()
    env = dict(os.environ, LD_PRELOAD=libasan, ASAN_OPTIONS="detect_leaks=0:abort_on_error=1",
               UBSAN_OPTIONS="halt_on_error=1")
    code = (
        "import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import numpy as np, dgsqp_b200 as dg\n"
        "from hostsim_lib import HostSim\n"
        "from dgsqp_b200.montecarlo import sample_head_to_head\n"
        "for N, M in ((6, 2), (5, 3)):\n"
        "    game = dg.chicane_game(N=N) if M == 2 else dg.agents_game(M=M, N=N)\n"
        "    hs = HostSim(game, dg.DGSQPParams(N=N, nonmono_ls=True, sqp_iters=6, line_search_iters=8), asan=True)\n"
        "    rng = np.random.default_rng(0)\n"
        "    x0 = np.concatenate([[0.3*a, 0.2*a, 2.5, 0.0, 0.3 + 0.9*a, 0.4 - 0.4*a] for a in range(M)])\n"
        "    u = rng.normal(size=game.n) * 0.1\n"
        "    Q, q, gtl, g, x = hs.evaluate(x0, u, np.abs(rng.normal(size=game.m)) * 0.1)\n"
        "    H, nneg = hs.nearest_pd(Q)\n"
        "    st, du, lam, it = hs.qp(H, q)\n"
        "    r = hs.solve(x0, u)\n"
        "    assert np.all(np.isfinite(r['u'])), r\n"
        "print('ASAN-OK')\n") % (str(pathlib.Path(__file__).resolve().parents[1]), str(pathlib.Path(__file__).resolve().parent))
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ASAN-OK" in out.stdout, out.stdout[-2000:] + out.stderr[-4000:]


def test_large_sample_fixture_subset():
    """Kernel source against the large-sample oracle fixture (tests/golden/chicane_N25_seed0_stats.npz, the first 750
    instances of the batch bench.py runs): a 96-instance slice here, all of them on the GPU (test_gpu_parity.py).
    Measured over all 1000 with this host build: identical (status, iterations) on 989, identical status on 992; on the
    541 identical KKT-converged instances u agrees to 2.6e-7 and the QP counts are equal; the instances that differ
    are long non-converging paths (max_it / conv_rel_tol flips), where the iteration is chaotic in the last bits."""
    d = dict(np.load(GOLDEN / "chicane_N25_seed0_stats.npz").items())
    hs = HostSim(dg.chicane_game(), dg.chicane_params())
    same = 0
    for i in range(300, 396):
        h = hs.solve(d["x0"][i], d["u_ws"][i])
        if h["status"] == d["status"][i] and h["num_iters"] == d["num_iters"][i]:
            same += 1
            if d["status"][i] == 0:
                assert h["qp_solves"] == d["qp_solves"][i]
                assert np.abs(h["u"] - d["u"][i]).max() < 1e-6 * max(1.0, np.abs(d["u"][i]).max())
                assert np.abs(h["cost"] - d["cost"][i]).max() < 1e-6 * max(1.0, np.abs(d["cost"][i]).max())
    assert same >= 93


@pytest.mark.parametrize("budget", ["28000", "0"])
def test_no_buffer_overruns_guard_build(budget, monkeypatch):
    """Guard build of the kernel source: every buffer of the memory plan is followed by 16 canary doubles.  Full solves
    of short- and full-horizon games (n = 40 .. 150, both placements, v1 and v2, racing and merge) must leave all of them
    intact.  (This is the check that would have caught the eigenvector-scratch overrun of nearest_pd for n < 97.)"""
    from dgsqp_b200.montecarlo import sample_head_to_head, sample_agents, sample_merge
    monkeypatch.setenv("DG_HOSTSIM_SMEM_DOUBLES", budget)
    cases = [(dg.chicane_game(N=10), dg.chicane_params(10), lambda g: sample_head_to_head(g, 3, seed=2)),
             (dg.chicane_game(), dg.chicane_params(), lambda g: sample_head_to_head(g, 3, seed=0)),
             (dg.curve_game(45.0, 15), dg.curve_params(15), lambda g: sample_head_to_head(g, 3, seed=1)),
             (dg.agents_game(3, 90.0, 15), dg.agents_params(15), lambda g: sample_agents(g, 2, seed=0)),
             (dg.agents_game(3, 90.0, 25), dg.agents_params(25), lambda g: sample_agents(g, 1, seed=0)),
             (dg.merge_game(N=10), dg.merge_params(10), lambda g: sample_merge(g, 3, seed=1)),
             (dg.merge_game(), dg.merge_params(), lambda g: sample_merge(g, 2, seed=1)),
             (dg.chicane_game(N=10), dg.DGSQPV2Params(N=10, reg=1e-1, reg_decay=0.8, nms_frequency=2, sqp_iters=30),
              lambda g: sample_head_to_head(g, 2, seed=3)),
             (dg.merge_game(N=10), dg.DGSQPV2Params(N=10, reg=1e-3, nms=False, sqp_iters=20, merit_function="sum_obj_l1"),
              lambda g: sample_merge(g, 2, seed=1))]
    for game, params, sampler in cases:
        hs = HostSim(game, params, guard=True)
        assert hs.guard_check() == 0
        x0, u_ws = sampler(game)
        for i in range(x0.shape[0]):
            r = hs.solve(x0[i], u_ws[i])
            assert r["status"] in (0, 1, 2, 3, 4)
            assert hs.guard_check() == 0, f"buffer overrun in {game.name} (n = {game.n})"


def test_v2_u_prev_matches_oracle():
    """Receding-horizon input of the v2 policy: u_prev (DGSQP_v2.py:311,328) enters the stage-0 rate cost and rate
    constraints; kernel source == oracle, and the v1 policy ignores it (DGSQP.py:305 zeroes u_prev)."""
    from oracle.dgsqp_v2 import OracleDGSQPV2
    from oracle.sampler import sample_head_to_head
    N = 10
    kw = dict(reg=1e-2, reg_decay=0.8, nms_frequency=2, sqp_iters=40, p_tol=1e-4, d_tol=1e-4)
    game, og = dg.chicane_game(N=N), RacingGame(chicane_track(), M=2, N=N)
    hs, sol = HostSim(game, dg.DGSQPV2Params(N=N, **kw)), OracleDGSQPV2(og, **kw)
    hs1 = HostSim(game, dg.chicane_params(N))
    rng = np.random.default_rng(0)
    up = np.array([1.5, 0.3, -1.0, -0.2])
    for i in range(3):
        x0, u_ws = sample_head_to_head(og, rng)
        r0, r = sol.solve(x0, u_ws), sol.solve(x0, u_ws, u_prev=up)
        h = hs.solve(x0, u_ws, u_prev=up)
        assert MSG[h["status"]] == r["msg"] and h["num_iters"] == r["num_iters"]
        assert np.abs(h["u"] - r["u"]).max() < 1e-9 and np.abs(h["cost"] - r["cost"]).max() < 1e-9
        assert np.abs(r["u"] - r0["u"]).max() > 1e-2                      # the previous input matters
        a, b = hs1.solve(x0, u_ws), hs1.solve(x0, u_ws, u_prev=up)
        assert np.array_equal(a["u"], b["u"])                              # v1: ignored


def test_qp_warm_start_same_equilibria_fewer_iterations():
    """The active-set QP starts from the previous QP's active set (qp_gi.cuh: gi_warm_start, dgsqp_params.qp_warm_start,
    on by default).  The strictly convex QP has one solution, so full solves reach the same equilibria as the cold start
    (``qp_warm_start = 0``, the reference's behaviour, DGSQP.py:240-241) with far fewer active-set iterations."""
    from dgsqp_b200.montecarlo import sample_head_to_head, sample_merge
    for game, params, (x0, u_ws) in ((dg.chicane_game(N=15), dg.chicane_params(15), sample_head_to_head(dg.chicane_game(N=15), 6, seed=2)),
                                      (dg.merge_game(N=10), dg.merge_params(10), sample_merge(dg.merge_game(N=10), 4, seed=1))):
        cold, warm = HostSim(game, params, qp_warm=False), HostSim(game, params, qp_warm=True)
        it_c = it_w = agree = 0
        for i in range(x0.shape[0]):
            a, b = cold.solve(x0[i], u_ws[i]), warm.solve(x0[i], u_ws[i])
            it_c, it_w = it_c + a["diag"][2], it_w + b["diag"][2]
            if a["status"] == b["status"] and a["num_iters"] == b["num_iters"]:
                agree += 1
                if a["status"] == 0:
                    assert a["qp_solves"] == b["qp_solves"]
                    assert np.abs(a["x"] - b["x"]).max() < 1e-6 * max(1.0, np.abs(a["x"]).max())
        assert agree >= x0.shape[0] - 1 and it_w < 0.6 * it_c


@pytest.mark.parametrize("nonmono,merit", [(True, "stat_l1"), (False, "stat_l1"), (True, "stat"), (False, "stat")])
def test_ablation_variants_match_oracle(nonmono, merit):
    """The four solver variants of scripts/DGSQP_monte_carlo_ablation.py:166-225 (watchdog on / off x merit with / without
    the l1 penalty): kernel source == oracle."""
    from oracle.sampler import sample_head_to_head
    N = 15
    game, og = dg.chicane_game(N=N), RacingGame(chicane_track(), M=2, N=N)
    params = dg.DGSQPParams(dt=0.1, N=N, reg=1e-3, nonmono_ls=nonmono, merit_function=merit, line_search_iters=50,
                            sqp_iters=50, p_tol=1e-3, d_tol=1e-3, beta=0.01, tau=0.5)
    hs, sol = HostSim(game, params), OracleDGSQP(og, reg=1e-3, nonmono_ls=nonmono, merit_function=merit)
    rng = np.random.default_rng(7)
    same = 0
    for i in range(5):
        x0, u_ws = sample_head_to_head(og, rng)
        r, h = sol.solve(x0, u_ws), hs.solve(x0, u_ws)
        if MSG[h["status"]] == r["msg"] and h["num_iters"] == r["num_iters"]:
            same += 1
            assert h["qp_solves"] == r["qp_solves"]
            if r["msg"] == "conv_abs_tol":
                assert np.abs(h["u"] - r["u"]).max() < 1e-6 * max(1.0, np.abs(r["u"]).max())
    assert same >= 4


@pytest.mark.parametrize("theta,N", [(45.0, 10), (75.0, 15), (90.0, 20)])
def test_curve_sweep_cells_match_oracle(theta, N):
    """Cells of the curve sweep (scripts/DGSQP_ALGAMES_monte_carlo_curve.py:134-146: theta x N, seed 1, reg = 0) with
    short horizons (n = 40, 60, 80): kernel source vs oracle.  With reg = 0 the QP Hessian keeps the clipped eigenvalues
    at the 1e-10 floor; along those directions the curvature is known to +-1e-13 only (rounding of the eigen-solver), so
    the polished QP solution -- and with it the iteration count -- is implementation dependent at the 1e-3 level whenever
    such a direction is not pinned by active constraints (DESIGN.md, 'reg = 0 games').  Asserted: every instance reaches
    the same convergence class (converged / not converged) on both sides, KKT-converged equilibria satisfy the
    tolerances, and where the whole path agrees the trajectories agree."""
    from oracle.sampler import sample_head_to_head
    og = RacingGame(curve_track(curve_angle=theta * np.pi / 180), M=2, N=N, rate_ub=(10.0, 4.5), rate_lb=(-10.0, -4.5), obs_r=0.2)
    hs, sol = HostSim(dg.curve_game(theta, N), dg.curve_params(N)), OracleDGSQP(og, reg=0.0)
    rng = np.random.default_rng(1)
    same = same_class = 0
    for i in range(4):
        x0, u_ws = sample_head_to_head(og, rng)
        r, h = sol.solve(x0, u_ws), hs.solve(x0, u_ws)
        same_class += (h["status"] <= 1) == bool(r["status"])
        if h["status"] == 0:
            assert h["cond"][0] < 1e-3 and h["cond"][1] < 1e-3 and h["cond"][2] < 1e-3
        if MSG[h["status"]] == r["msg"] and h["num_iters"] == r["num_iters"]:
            same += 1
            if r["msg"] == "conv_abs_tol":
                assert np.abs(h["x"] - r["x"]).max() < 1e-5 * max(1.0, np.abs(r["x"]).max())
    assert same_class >= 3 and same >= (2 if theta < 90.0 else 1)
