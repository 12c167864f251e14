"""Parity tests proper: the CUDA path, called through the C ABI, against the CPU oracle.
Run on the B200 box:  python -m pytest tests -m gpu
"""
import json
import pathlib

import numpy as np
import pytest

import dgsqp_b200 as dg
from dgsqp_b200.montecarlo import sample_head_to_head, sample_agents

pytestmark = pytest.mark.gpu
GOLDEN = pathlib.Path(__file__).parent / "golden"
MSG = {0: "conv_abs_tol", 1: "conv_rel_tol", 2: "max_it", 3: "diverged", 4: "qp_fail"}


def _rel(a, b):
    return np.abs(a - b).max() / max(1.0, np.abs(b).max())


# ------------------------------------------------------------------ stage level (K1..K3, K0)
@pytest.mark.parametrize("threads", [64, 128, 256])
def test_stages_vs_oracle(threads):
    """Rollout+derivatives, KKT assembly, eigen-projection, QP and LSQR of the CUDA path, each against the
    oracle on the same inputs (chicane, N = 25)."""
    from gpu_units_lib import run_stages
    from oracle.dgsqp_v1 import OracleDGSQP, nearest_pd
    from oracle.qp import solve_qp_gi, kkt_residuals
    from oracle.racing_game import RacingGame
    from oracle.track import chicane_track
    game, params = dg.chicane_game(), dg.chicane_params()
    og = RacingGame(chicane_track(), M=2, N=25)
    B = 6
    x0, u = sample_head_to_head(game, B, seed=11)
    rng = np.random.default_rng(5)
    l = np.abs(rng.normal(size=(B, game.m))) * 0.3 * (rng.random((B, game.m)) < 0.2)
    out = run_stages(game, params, x0, u, l, threads=threads)
    sol = OracleDGSQP(og)
    for i in range(B):
        Q, q, G, g, _ = og.evaluate(u[i], l[i], x0[i], np.zeros(4), True)
        assert _rel(out["Q"][i], Q) < 1e-12 and _rel(out["q"][i], q) < 1e-12
        assert _rel(out["gtl"][i], G.T @ l[i]) < 1e-12 and _rel(out["g"][i], g) < 1e-13
        H = nearest_pd(Q) + params.reg * np.eye(game.n)
        assert out["nneg"][i] == int((np.linalg.eigvalsh((Q + Q.T) / 2) < 0).sum())
        assert _rel(out["H"][i], H) < 1e-11
        du, lam = solve_qp_gi(H, q, G, g)
        assert out["qpst"][i] == 0
        assert _rel(out["du"][i], du) < 1e-8 and _rel(out["lam"][i], lam) < 1e-7
        r = kkt_residuals(H, q, G, g, out["du"][i], out["lam"][i])
        assert r["stat"] < 1e-8 and r["feas"] < 1e-9 and r["dual"] == 0.0 and r["comp"] < 1e-8
        q0, G0, _, _ = og.evaluate(u[i], np.zeros(game.m), x0[i], np.zeros(4), False)
        l0 = sol.dual_init(q0, G0)
        assert int(out["lsqr_it"][i]) == sol.lsqr_iters
        assert np.abs(out["l0"][i] - l0).max() < 1e-9 * max(1.0, np.abs(l0).max())


# ------------------------------------------------------------------ full solves vs golden (oracle) results
def _golden(name):
    return np.load(GOLDEN / f"{name}.npz"), json.loads((GOLDEN / f"{name}.json").read_text())


@pytest.mark.parametrize("name,mk,tol,max_diff", [
    ("chicane_N25_seed0", lambda: (dg.chicane_game(), dg.chicane_params()), 1e-6, 1),
    ("curve45_N15_seed1", lambda: (dg.curve_game(45.0, 15), dg.curve_params(15)), 1e-6, 1),
    ("agents3_N15_seed0", lambda: (dg.agents_game(3, 90.0, 15), dg.agents_params(15)), 1e-6, 0)])
def test_solve_vs_golden_shared_dual_init(name, mk, tol, max_diff):
    """Same instances, same dual initialisation as the oracle run: identical status and iteration count (at most
    `max_diff` instances of the fixture may differ: 47/48, 24/24, 16/16 with the host build of the kernel source), and
    equilibria -- inputs, states, MULTIPLIERS, costs -- within 1e-6 relative on the instances that converge by the KKT test
    (measured 1e-11 or better: both sides polish the QP's KKT point, qp_gi.cuh gi_polish / oracle/qp.py)."""
    game, params = mk()
    data, meta = _golden(name)
    solver = dg.DGSQP(game, params, print_method=None, mu_vio_thresh=1e-10)
    res = solver.solve_batch(data["x0"], data["u_ws"], data["l_init"])
    B = data["x0"].shape[0]
    same = np.array([res.msg[i] == meta["msg"][i] and int(res.num_iters[i]) == meta["num_iters"][i] for i in range(B)])
    assert same.sum() >= B - max_diff, f"identical (status, iters): {same.sum()}/{B}"
    checked = 0
    for i in np.where(same)[0]:
        if meta["msg"][i] != "conv_abs_tol":
            continue
        checked += 1
        assert _rel(res.u[i], data["u"][i]) < tol and _rel(res.x[i], data["x"][i]) < tol
        assert _rel(res.l[i], data["l"][i]) < tol
        assert _rel(res.cost[i], data["cost"][i]) < tol
        assert int(res.qp_solves[i]) == meta["qp_solves"][i]
    assert checked >= 3


def test_solve_vs_golden_own_lsqr():
    """End to end with the on-device (reorthogonalised) LSQR dual initialisation."""
    game, params = dg.chicane_game(), dg.chicane_params()
    data, meta = _golden("chicane_N25_seed0")
    res = dg.DGSQP(game, params, print_method=None, mu_vio_thresh=1e-10).solve_batch(data["x0"], data["u_ws"])
    B = data["x0"].shape[0]
    same = np.array([res.msg[i] == meta["msg"][i] and int(res.num_iters[i]) == meta["num_iters"][i] for i in range(B)])
    assert same.sum() >= B - 2, f"identical (status, iters): {same.sum()}/{B}"
    for i in np.where(same)[0]:
        if meta["msg"][i] == "conv_abs_tol":
            assert _rel(res.u[i], data["u"][i]) < 1e-6 and _rel(res.x[i], data["x"][i]) < 1e-6
            assert _rel(res.l[i], data["l"][i]) < 1e-6


def test_live_oracle_small():
    """A few short-horizon instances against the oracle run live (no fixtures involved)."""
    from oracle.dgsqp_v1 import OracleDGSQP
    from oracle.racing_game import RacingGame
    from oracle.track import chicane_track
    N = 10
    game, params = dg.chicane_game(N=N), dg.chicane_params(N=N)
    x0, u_ws = sample_head_to_head(game, 6, seed=3)
    oracle = OracleDGSQP(RacingGame(chicane_track(), M=2, N=N))
    refs = [oracle.solve(x0[i], u_ws[i]) for i in range(6)]
    l0 = np.stack([r["init"]["l"] for r in refs])
    res = dg.DGSQP(game, params, print_method=None, mu_vio_thresh=1e-10).solve_batch(x0, u_ws, l0)
    ok = 0
    for i, r in enumerate(refs):
        if res.msg[i] == r["msg"] and int(res.num_iters[i]) == r["num_iters"]:
            ok += 1
            if r["msg"] == "conv_abs_tol":
                assert _rel(res.u[i], r["u"]) < 1e-6 and _rel(res.l[i], r["l"]) < 1e-6
    assert ok >= 5


# ------------------------------------------------------------------ full-size properties (10k chicane games)
@pytest.fixture(scope="module")
def big_batch():
    game, params = dg.chicane_game(), dg.chicane_params()
    x0, u_ws = sample_head_to_head(game, 10000, seed=0)
    solver = dg.DGSQP(game, params, print_method=None, mu_vio_thresh=1e-10)
    return game, params, solver, x0, u_ws, solver.solve_batch(x0, u_ws)


def test_full_size_status_and_kkt(big_batch):
    game, params, solver, x0, u_ws, res = big_batch
    assert set(np.unique(res.status)) <= {0, 1, 2, 3, 4}
    conv = res.status == 0
    assert conv.mean() > 0.3
    # converged by the KKT test => the reported conditions satisfy the tolerances (DGSQP.py:391)
    assert np.all(res.cond[conv, 0] < params.p_tol) and np.all(res.cond[conv, 1] < params.d_tol)
    assert np.all(res.cond[conv, 2] < params.d_tol)
    assert np.all(res.num_iters[res.status == 2] == params.sqp_iters)
    assert np.all(res.num_iters <= params.sqp_iters) and np.all(res.qp_solves >= res.num_iters * (res.status != 0))
    assert np.all(np.isfinite(res.u[conv])) and np.all(np.isfinite(res.l[conv])) and np.all(res.l[conv] >= 0)
    # x_out is the rollout of u_out from x0 (DGSQP.py:476): check a sample against the oracle's dynamics
    from oracle.racing_game import RacingGame
    from oracle.track import chicane_track
    og = RacingGame(chicane_track(), M=2, N=25)
    for i in np.where(conv)[0][:5]:
        x = og.rollout(res.u[i], x0[i])
        assert np.abs(x.ravel() - res.x[i]).max() < 1e-10
        g = og.constraints(x, res.u[i], np.zeros(4))
        assert g.max() < params.p_tol
        assert np.allclose(og.costs(x, res.u[i], np.zeros(4)), res.cost[i], atol=1e-9)


def test_full_size_deterministic_and_batch_independent(big_batch):
    game, params, solver, x0, u_ws, res = big_batch
    again = solver.solve_batch(x0, u_ws)
    assert np.array_equal(again.status, res.status) and np.array_equal(again.num_iters, res.num_iters)
    # bit patterns: an instance that ends in 'qp_fail' / 'diverged' may legitimately carry NaNs (NaN != NaN)
    bits = lambda a: np.ascontiguousarray(a).view(np.int64)
    assert np.array_equal(bits(again.u), bits(res.u)) and np.array_equal(bits(again.l), bits(res.l))
    # an instance's result does not depend on its position or on its batch mates
    idx = np.array([7, 4242, 9999, 123, 5000])
    sub = solver.solve_batch(x0[idx], u_ws[idx])
    assert np.array_equal(sub.status, res.status[idx]) and np.array_equal(sub.num_iters, res.num_iters[idx])
    assert np.array_equal(bits(sub.u), bits(res.u[idx]))
    perm = np.random.default_rng(0).permutation(2000)
    p = solver.solve_batch(x0[perm], u_ws[perm])
    assert np.array_equal(bits(p.u), bits(res.u[perm])) and np.array_equal(p.status, res.status[perm])


def test_device_path_equals_host_path(big_batch):
    import torch
    game, params, solver, x0, u_ws, res = big_batch
    dev = torch.device("cuda:0")
    r = solver.solve_batch(torch.from_numpy(x0[:512]).to(dev), torch.from_numpy(u_ws[:512]).to(dev))
    assert r.u.is_cuda
    assert np.array_equal(r.u.cpu().numpy(), res.u[:512]) and np.array_equal(r.status.cpu().numpy(), res.status[:512])


# ------------------------------------------------------------------ reference surface and edge cases
def test_solver_class_surface():
    game, params = dg.chicane_game(N=10), dg.chicane_params(N=10)
    solver = dg.DGSQP(game, params, print_method=None, mu_vio_thresh=1e-10)
    assert (solver.N, solver.M, solver.n_u, solver.n_q) == (10, 2, 4, 12) and sum(solver.n_c) == game.m
    x0, u_ws = sample_head_to_head(game, 1, seed=5)
    states = []
    for a in range(2):
        s = dg.VehicleState(t=0.0)
        s.x.x, s.x.y, s.v.v_long, s.p.e_psi, s.p.s, s.p.x_tran = x0[0, 6 * a:6 * a + 6]
        states.append(s)
    with pytest.raises(RuntimeError, match="incompatible with required shape"):
        solver.set_warm_start(np.zeros((9, 4)))
    solver.set_warm_start(solver.agent_to_stage_major(u_ws)[0])
    assert np.array_equal(solver.u_ws, u_ws[0])
    info = solver.solve(states)
    assert set(info) >= {"time", "num_iters", "status", "cost", "cond", "iter_data", "msg", "init"}
    assert info["msg"] in MSG.values() and set(info["cond"]) == {"p_feas", "comp", "stat"}
    assert solver.q_pred.shape == (11, 12) and solver.u_pred.shape == (10, 4) and solver.l_pred.shape == (game.m,)
    assert np.allclose(solver.q_pred[0], x0[0])
    ref = solver.solve_batch(x0, u_ws)
    assert np.array_equal(solver.agent_to_stage_major(ref.u)[0], solver.u_pred)
    # step(): applies u_0 to the states and shifts the warm start (DGSQP.py:283-297)
    u_pred = solver.u_pred.copy()
    info2 = solver.step(states)
    assert states[0].u.u_a == solver.u_pred[0, 0] and states[1].u.u_steer == solver.u_pred[0, 3]
    if info2["msg"] not in ("diverged", "qp_fail"):
        shifted = np.vstack((solver.u_pred[1:], solver.u_pred[-1]))
        assert np.array_equal(solver.u_ws, solver.stage_to_agent_major(shifted[None])[0])
    preds = solver.get_prediction()
    assert len(preds) == 2 and len(preds[0].x) == 11 and len(preds[0].u_a) == 10
    assert np.allclose(u_pred, solver.u_pred)


def test_reference_constructor_form():
    """DGSQP(joint_dynamics, costs, agent_constraints, shared_constraints, bounds, params) -- the reference's own argument
    list (DGSQP.py:25-33) with plain callables -- builds the same solver as the game record (the identified numbers agree with the literals to
    1e-12, e.g. the steering-rate limit pi comes back as (dt pi) / dt): same status and iterations, results to 1e-8."""
    from test_frontend import _script_args
    N = 10
    args = _script_args(N=N)
    params = dg.chicane_params(N=N)
    a = dg.DGSQP(*args, params, print_method=None, mu_vio_thresh=1e-10)
    b = dg.DGSQP(dg.chicane_game(N=N), params, print_method=None, mu_vio_thresh=1e-10)
    x0, u_ws = sample_head_to_head(dg.chicane_game(N=N), 8, seed=4)
    ra, rb = a.solve_batch(x0, u_ws), b.solve_batch(x0, u_ws)
    assert np.array_equal(ra.status, rb.status) and np.array_equal(ra.num_iters, rb.num_iters)
    conv = ra.status == 0
    assert conv.sum() >= 3 and _rel(ra.u[conv], rb.u[conv]) < 1e-8 and _rel(ra.l[conv], rb.l[conv]) < 1e-8


def test_edge_batches():
    game, params = dg.chicane_game(N=10), dg.chicane_params(N=10)
    solver = dg.DGSQP(game, params, print_method=None, mu_vio_thresh=1e-10)
    empty = solver.solve_batch(np.zeros((0, 12)), np.zeros((0, game.n)))
    assert empty.u.shape == (0, game.n) and empty.status.shape == (0,)
    x0, u_ws = sample_head_to_head(game, 3, seed=1)
    one = solver.solve_batch(x0[:1], u_ws[:1])
    three = solver.solve_batch(x0, u_ws)
    assert np.array_equal(one.u[0], three.u[0])
    zero_ws = solver.solve_batch(x0, np.zeros_like(u_ws))          # cold start still terminates with a status
    assert set(np.unique(zero_ws.status)) <= {0, 1, 2, 3, 4}
    with pytest.raises(RuntimeError):
        solver.solve_batch(x0, u_ws[:, :-1])
    # non-finite input must not hang or crash: it ends as a failure status
    bad = x0.copy()
    bad[0, 2] = np.nan
    r = solver.solve_batch(bad, u_ws)
    assert r.status[0] in (2, 3, 4) and np.array_equal(r.u[1:], three.u[1:])


@pytest.mark.parametrize("M", [3, 4])
def test_multi_agent_games_run_and_satisfy_kkt(M):
    N = 25
    game, params = dg.agents_game(M=M, N=N), dg.agents_params(N)
    x0, u_ws = sample_agents(game, 64, seed=0)
    res = dg.DGSQP(game, params, print_method=None, mu_vio_thresh=1e-10).solve_batch(x0, u_ws)
    conv = res.status == 0
    assert conv.sum() >= 8
    assert np.all(res.cond[conv] < 1e-3)
    from oracle.racing_game import RacingGame
    from oracle.track import curve_track
    og = RacingGame(curve_track(curve_angle=np.pi / 2), M=M, N=N, obs_r=0.4)
    i = int(np.where(conv)[0][0])
    # independent KKT check of the returned point with the oracle's derivatives
    Q, q, G, g, x = og.evaluate(res.u[i], res.l[i], x0[i], np.zeros(2 * M), True)
    assert np.abs(q + G.T @ res.l[i]).max() < 1e-3 and g.max() < 1e-3 and np.abs(g * res.l[i]).max() < 1e-3
    assert np.abs(x.ravel() - res.x[i]).max() < 1e-10


# ------------------------------------------------------------------ v2 step policy (DGSQPV2Params)
def test_v2_solve_vs_golden():
    """The v2 policy on device against the v2 oracle's golden results: identical status / iteration count / QP count
    and equilibria within 1e-6 relative."""
    data, meta = _golden("chicane_v2_N15_seed0")
    game = dg.chicane_game(N=15)
    solver = dg.DGSQP(game, dg.DGSQPV2Params(N=15, **meta["solver_kw"]), print_method=None, mu_vio_thresh=1e-10)
    B = data["x0"].shape[0]
    for l0 in (data["l_init"], None):
        res = solver.solve_batch(data["x0"], data["u_ws"], l0)
        same = np.array([res.msg[i] == meta["msg"][i] and int(res.num_iters[i]) == meta["num_iters"][i] for i in range(B)])
        assert same.sum() >= B - 1, f"identical (status, iters): {same.sum()}/{B}"
        for i in np.where(same)[0]:
            assert _rel(res.u[i], data["u"][i]) < 1e-6 and _rel(res.x[i], data["x"][i]) < 1e-6
            assert _rel(res.l[i], data["l"][i]) < 1e-6
            assert int(res.qp_solves[i]) == meta["qp_solves"][i]
    again = solver.solve_batch(data["x0"], data["u_ws"])
    bits = lambda a: np.ascontiguousarray(a).view(np.int64)
    assert np.array_equal(bits(again.u), bits(res.u)) and np.array_equal(again.num_iters, res.num_iters)


def test_v2_batch_kkt_and_limits():
    """A 512-instance v2 batch with a Newton-like setting: KKT tolerances at converged points; 'max_it' means the
    m-step budget was spent; unsupported options are rejected."""
    N = 25
    game = dg.chicane_game(N=N)
    params = dg.DGSQPV2Params(N=N, reg=1e-3, p_tol=1e-3, d_tol=1e-3, sqp_iters=40)
    x0, u_ws = sample_head_to_head(game, 512, seed=2)
    solver = dg.DGSQP(game, params, print_method=None, mu_vio_thresh=1e-10)
    res = solver.solve_batch(x0, u_ws)
    conv = res.status == 0
    assert conv.mean() > 0.3 and set(np.unique(res.status)) <= {0, 1, 2, 3, 4}
    assert np.all(res.cond[conv, 0] < params.p_tol) and np.all(res.cond[conv, 1] < params.d_tol)
    assert np.all(res.cond[conv, 2] < params.d_tol)
    d = solver.last_diag(512)
    assert np.all(d[res.status == 2, 6] == params.sqp_iters) and np.all(d[:, 6] <= params.sqp_iters)
    with pytest.raises(ValueError):
        dg.DGSQP(game, dg.DGSQPV2Params(N=N, merit_function="sum_obj"), print_method=None, mu_vio_thresh=1e-10)
    with pytest.raises(ValueError):
        dg.DGSQP(game, dg.DGSQPV2Params(N=N, merit_decrease_condition="wolfe"), print_method=None, mu_vio_thresh=1e-10)


# ------------------------------------------------------------------ merge scenario (BASELINE config 5)
def test_merge_vs_golden():
    """Merge game (three unicycles, RK3, lane half-planes) on device against the oracle's golden results
    (scripts/DGSQP_merge_monte_carlo.py: seed 1, zero warm start, reg = 0): identical status / iterations / QP counts
    on every instance; trajectories, costs, inputs and multipliers within 1e-6 (measured 3e-8 / 5e-8: reg = 0 leaves
    eigenvalues of the QP Hessian at the 1e-10 floor, condition ~1e11, and only the polished KKT point -- gi_polish -- is
    reproducible there; the un-polished active-set iterate agreed to 1e-5 in u and 1e-4 in l)."""
    from dgsqp_b200.montecarlo import sample_merge
    data, meta = _golden("merge_N20_seed1")
    game, params = dg.merge_game(), dg.merge_params()
    x0, u_ws = sample_merge(game, 32, seed=1)
    assert np.array_equal(x0, data["x0"]) and not u_ws.any()
    solver = dg.DGSQP(game, params, print_method=None, mu_vio_thresh=1e-10)
    B = x0.shape[0]
    for l0 in (data["l_init"], None):
        res = solver.solve_batch(x0, u_ws, l0)
        same = np.array([res.msg[i] == meta["msg"][i] and int(res.num_iters[i]) == meta["num_iters"][i] for i in range(B)])
        # reg = 0: a rare instance meets the 1e-3 KKT test an iteration earlier / later depending on summation order
        # (159 of 160 instances identical between the kernel source and the oracle); allow one such instance here
        assert same.sum() >= B - 1, f"identical (status, iters): {same.sum()}/{B}"
        assert all(res.msg[i] == meta["msg"][i] for i in range(B))
        for i in np.where(same)[0]:
            assert int(res.qp_solves[i]) == meta["qp_solves"][i]
            assert _rel(res.x[i], data["x"][i]) < 1e-6 and _rel(res.cost[i], data["cost"][i]) < 1e-6
            assert _rel(res.u[i], data["u"][i]) < 1e-6 and _rel(res.l[i], data["l"][i]) < 1e-6
    # n = 120: the two n x n work matrices (232 KB) do not fit in shared memory, the pool and the sensitivities do;
    # with a small cap everything moves to the global workspace -- same answer
    plan = solver.memory_plan()
    assert not plan["mats_in_smem"] and plan["sens_in_smem"]
    solver.set_smem_limit(16 * 1024)
    assert not solver.memory_plan()["sens_in_smem"]
    low = solver.solve_batch(x0, u_ws)
    assert np.array_equal(low.status, res.status) and np.array_equal(low.num_iters, res.num_iters)
    assert _rel(low.x, res.x) < 1e-6


@pytest.mark.parametrize("name,mk,max_diff,min_checked,ltol", [
    ("curve75_N25_seed1", lambda: (dg.curve_game(75.0, 25), dg.curve_params(25)), 4, 4, 1e-4),
    ("curve90_N25_seed1", lambda: (dg.curve_game(90.0, 25), dg.curve_params(25)), 4, 3, 1e-4),
    ("agents4_N25_seed0", lambda: (dg.agents_game(4, 90.0, 25), dg.agents_params(25)), 1, 5, 1e-6)])
def test_round2_configs_vs_golden(name, mk, max_diff, min_checked, ltol):
    """The BASELINE configurations VERDICT r1 found without a GPU parity test -- the 75 and 90 degree curves at N = 25
    (configs[2]) and FOUR agents at N = 25 (configs[3]: n = 200, m = 1150, both work matrices in the L2 workspace, hybrid
    generic + register-tile tridiagonalisation) -- against the oracle's golden results (tests/golden/make_golden_r2.py):
    identical status and iteration count, and u, x, l, costs within 1e-6 relative on the instances that converge by the
    KKT test on the same path, with the oracle's and with the device's own dual initialisation.  Four agents (reg = 1e-3):
    one chaotic instance allowed.  The curve script runs with reg = 0 (DGSQP_ALGAMES_monte_carlo_curve.py:161): the
    projected Hessian keeps eigenvalues at the 1e-10 floor (condition ~1e11) and at N = 25 the iteration path is not
    reproducible in the last bits by ANYONE -- the oracle rerun with its own dual initialisation perturbed by one ulp
    keeps 9-10 of these 12 instances (profiles/r2_chaos_floor_curve_N25.json), the host build of the kernel source 9 --
    so 8 of 12 identical paths are required there, and the multipliers of the reg = 0 games are compared to 1e-4 (measured
    3.6e-6 on one curve-75 and 1.4e-5 on one curve-90 instance: u and x agree to 1e-6, the multipliers solve a system with
    the 1e11 condition)."""
    game, params = mk()
    data, meta = _golden(name)
    solver = dg.DGSQP(game, params, print_method=None, mu_vio_thresh=1e-10)
    B = data["x0"].shape[0]
    for l0 in (data["l_init"], None):
        res = solver.solve_batch(data["x0"], data["u_ws"], l0)
        same = np.array([res.msg[i] == meta["msg"][i] and int(res.num_iters[i]) == meta["num_iters"][i] for i in range(B)])
        assert same.sum() >= B - max_diff, f"identical (status, iters): {same.sum()}/{B}"
        checked = 0
        for i in np.where(same)[0]:
            if meta["msg"][i] != "conv_abs_tol":
                continue
            checked += 1
            assert _rel(res.u[i], data["u"][i]) < 1e-6 and _rel(res.x[i], data["x"][i]) < 1e-6
            assert _rel(res.l[i], data["l"][i]) < ltol and _rel(res.cost[i], data["cost"][i]) < 1e-6
            assert int(res.qp_solves[i]) == meta["qp_solves"][i]
        assert checked >= min_checked


def test_merge_vs_golden_128_more():
    """Merge scenario beyond the first 32 samples: accepted samples 32..159 of the script's seeded sampler against the
    oracle (tests/golden/merge_N20_seed1_b.*): identical (status, iterations) on at least 126 of 128 (reg = 0: a rare
    instance meets the KKT test one iteration earlier or later); states, inputs and costs within 1e-6, multipliers within
    1e-5 (reg = 0, condition ~1e11: measured 2.6e-6 on the worst of the 128 instances, 1e-7 typical)."""
    from dgsqp_b200.montecarlo import sample_merge
    data, meta = _golden("merge_N20_seed1_b")
    game, params = dg.merge_game(), dg.merge_params()
    x0, u_ws = sample_merge(game, 160, seed=1)
    x0, u_ws = x0[32:], u_ws[32:]
    assert np.array_equal(x0, data["x0"])
    res = dg.DGSQP(game, params, print_method=None, mu_vio_thresh=1e-10).solve_batch(x0, u_ws)
    B = x0.shape[0]
    same = np.array([res.msg[i] == meta["msg"][i] and int(res.num_iters[i]) == meta["num_iters"][i] for i in range(B)])
    assert same.sum() >= B - 2, f"identical (status, iters): {same.sum()}/{B}"
    for i in np.where(same)[0]:
        assert _rel(res.x[i], data["x"][i]) < 1e-6 and _rel(res.cost[i], data["cost"][i]) < 1e-6
        assert _rel(res.u[i], data["u"][i]) < 1e-6 and _rel(res.l[i], data["l"][i]) < 1e-5


def test_merge_batch_properties():
    """4096 merge instances: KKT tolerances at converged points (checked independently with the oracle's derivatives on
    a sample), x_out is the RK3 rollout of u_out, bitwise run-to-run determinism, batch-position independence, solver
    class surface for the unicycle states."""
    from dgsqp_b200.montecarlo import sample_merge
    from oracle.merge_game import MergeGame
    game, params = dg.merge_game(), dg.merge_params()
    B = 4096
    x0, u_ws = sample_merge(game, B, seed=1)
    solver = dg.DGSQP(game, params, print_method=None, mu_vio_thresh=1e-10)
    res = solver.solve_batch(x0, u_ws)
    assert set(np.unique(res.status)) <= {0, 1, 2, 3, 4}
    conv = res.status == 0
    assert conv.mean() > 0.9
    assert np.all(res.cond[conv] < 1e-3) and np.all(res.l[conv] >= 0)
    og = MergeGame(N=20)
    for i in np.where(conv)[0][:4]:
        Q, q, G, g, x = og.evaluate(res.u[i], res.l[i], x0[i], np.zeros(6), True)
        assert np.abs(x.ravel() - res.x[i]).max() < 1e-11
        assert np.abs(q + G.T @ res.l[i]).max() < 1e-3 and g.max() < 1e-3 and np.abs(g * res.l[i]).max() < 1e-3
        assert np.allclose(og.costs(x, res.u[i], np.zeros(6)), res.cost[i], rtol=1e-12)
    again = solver.solve_batch(x0, u_ws)
    bits = lambda a: np.ascontiguousarray(a).view(np.int64)
    assert np.array_equal(again.status, res.status) and np.array_equal(bits(again.u), bits(res.u))
    idx = np.array([5, 4000, 77, 2048])
    sub = solver.solve_batch(x0[idx], u_ws[idx])
    assert np.array_equal(bits(sub.u), bits(res.u[idx])) and np.array_equal(sub.num_iters, res.num_iters[idx])
    # reference surface: solve(states) with the unicycle state2q order
    states = [dg.VehicleState(t=0.0, x=dg.Position(x=x0[0, 4 * a], y=x0[0, 4 * a + 1]),
                              v=dg.BodyLinearVelocity(v_long=x0[0, 4 * a + 2]),
                              e=dg.OrientationEuler(psi=x0[0, 4 * a + 3])) for a in range(3)]
    info = solver.solve(states)
    assert info["msg"] == res.msg[0] and info["num_iters"] == int(res.num_iters[0])
    assert solver.q_pred.shape == (21, 12) and solver.u_pred.shape == (20, 6)
    assert np.array_equal(solver.u_pred, solver.agent_to_stage_major(res.u[:1])[0])


def test_small_horizon_games_eigen_scratch():
    """Games with n < 97 (the eigenvector scratch of nearest_pd is larger than one n x n matrix there): full solves of
    short-horizon chicane and merge games against the oracle run live."""
    from dgsqp_b200.montecarlo import sample_merge
    from oracle.dgsqp_v1 import OracleDGSQP
    from oracle.merge_game import MergeGame
    N = 10
    game, params = dg.merge_game(N=N), dg.merge_params(N)
    x0, u_ws = sample_merge(game, 6, seed=1)
    res = dg.DGSQP(game, params, print_method=None, mu_vio_thresh=1e-10).solve_batch(x0, u_ws)
    orc = OracleDGSQP(MergeGame(N=N), reg=0.0)
    for i in range(6):
        r = orc.solve(x0[i], u_ws[i])
        assert res.msg[i] == r["msg"] and int(res.num_iters[i]) == r["num_iters"]
        assert _rel(res.x[i], r["x"].ravel()) < 1e-6


def test_v2_sum_obj_merit_live_oracle():
    """v2 merit 'sum_obj_l1' on device against the oracle run live (nms = False: every iteration line-searches the
    summed costs; and the default non-monotone policy), short-horizon chicane and merge games."""
    from dgsqp_b200.montecarlo import sample_merge
    from oracle.dgsqp_v2 import OracleDGSQPV2
    from oracle.merge_game import MergeGame
    from oracle.racing_game import RacingGame
    from oracle.track import chicane_track
    N = 10
    cases = [(dg.chicane_game(N=N), RacingGame(chicane_track(), M=2, N=N), sample_head_to_head(dg.chicane_game(N=N), 4, seed=2)),
             (dg.merge_game(N=N), MergeGame(N=N), sample_merge(dg.merge_game(N=N), 4, seed=1))]
    for kw in (dict(reg=1e-3, reg_decay=0.9, nms=False, sqp_iters=30, merit_decrease=0.3, merit_function="sum_obj_l1"),
               dict(reg=1e-1, reg_decay=0.8, nms_frequency=2, sqp_iters=40, merit_function="sum_obj_l1")):
        for game, og, (x0, u_ws) in cases:
            res = dg.DGSQP(game, dg.DGSQPV2Params(N=N, **kw), print_method=None, mu_vio_thresh=1e-10).solve_batch(x0, u_ws)
            sol = OracleDGSQPV2(og, **kw)
            for i in range(x0.shape[0]):
                r = sol.solve(x0[i], u_ws[i])
                assert res.msg[i] == r["msg"] and int(res.num_iters[i]) == r["num_iters"]
                assert int(res.qp_solves[i]) == r["qp_solves"]
                if r["status"]:
                    assert _rel(res.u[i], r["u"]) < 1e-6 and _rel(res.x[i], r["x"].ravel()) < 1e-6


def test_device_statistics_match_host_statistics(big_batch):
    """dgsqp_batch_stats (statistics reduced on the device) == the host-side shard statistics of the same results."""
    import torch
    from dgsqp_b200.sharding import shard_stats, combine_stats
    game, params, solver, x0, u_ws, res = big_batch
    dev = torch.device("cuda:0")
    r = solver.solve_batch(torch.from_numpy(x0[:3000]).to(dev), torch.from_numpy(u_ws[:3000]).to(dev))
    dv = solver.batch_stats(r)
    hv = shard_stats(res.status[:3000], res.num_iters[:3000], res.qp_solves[:3000], res.cond[:3000])
    assert np.array_equal(dv[:13], hv[:13])                    # counts and integer sums are exact in double
    assert dv[13] == hv[13] and dv[14] == hv[14]
    s = combine_stats([dv])
    assert s["count"] == 3000 and s["converged"] == int((res.status[:3000] <= 1).sum())
    assert np.array_equal(solver.batch_stats(res)[:13], shard_stats(res.status, res.num_iters, res.qp_solves, res.cond)[:13])


def test_fused_statistics_equal_host_statistics(big_batch):
    """SURVEY 8(f-2): the statistics the solve kernel accumulates in its epilogue (dgsqp_last_stats) equal the host
    reduction of the returned arrays entry for entry (counts and iteration sums are exact; the maxima bitwise)."""
    from dgsqp_b200.sharding import shard_stats
    game, params, solver, x0, u_ws, res = big_batch
    again = solver.solve_batch(x0[:3000], u_ws[:3000])
    fused = solver.last_stats()
    host = shard_stats(again.status, again.num_iters, again.qp_solves, again.cond)
    assert fused[0] == 3000 and np.array_equal(fused[:15], host[:15])


def test_large_sample_parity():
    """The CUDA path on the first 750 instances of the bench batch against the oracle's stored results
    (tests/golden/chicane_N25_seed0_stats.npz): identical (status, iterations) on at least 99 % -- the bar BASELINE.json
    states (host build of the kernel source on the first 1000: 995 cold start / 997 warm start) -- and KKT-converged
    equilibria within 1e-6 relative (measured on the first 1000: max 2e-7, median 1e-15)."""
    d = dict(np.load(GOLDEN / "chicane_N25_seed0_stats.npz").items())
    B = len(d["status"])
    res = dg.DGSQP(dg.chicane_game(), dg.chicane_params(), print_method=None, mu_vio_thresh=1e-10).solve_batch(d["x0"], d["u_ws"])
    same = (res.status == d["status"]) & (res.num_iters == d["num_iters"])
    print(f"identical (status, iters): {int(same.sum())}/{B}; identical status: {int((res.status == d['status']).sum())}")
    assert same.mean() >= 0.99 and (res.status == d["status"]).mean() >= 0.99
    # every instance that converged by the KKT test on the same path: inputs and costs to 1e-6, same QP count
    kkt0 = same & (d["status"] == 0)
    assert kkt0.sum() > B // 2 and (res.qp_solves[kkt0] == d["qp_solves"][kkt0]).sum() >= kkt0.sum() - 1
    err0 = np.abs(res.u[kkt0] - d["u"][kkt0]).max(axis=1) / np.maximum(1.0, np.abs(d["u"][kkt0]).max(axis=1))
    assert err0.max() < 1e-6
    cerr = np.abs(res.cost[kkt0] - d["cost"][kkt0]).max(axis=1) / np.maximum(1.0, np.abs(d["cost"][kkt0]).max(axis=1))
    assert cerr.max() < 1e-6
    # conv_rel_tol is a stagnation test, not a KKT test (DGSQP.py:454-462): such instances stop at non-stationary points
    # where the iteration is not contractive; they are counted in `same` above and reported, not compared point-wise
    rel = same & (d["status"] == 1)
    err1 = np.abs(res.u[rel] - d["u"][rel]).max(axis=1) / np.maximum(1.0, np.abs(d["u"][rel]).max(axis=1))
    print(f"conv_rel_tol: {int(rel.sum())} identical, u within 1e-6 on {int((err1 < 1e-6).sum())}, max {err1.max():.1e}")
    assert (err1 < 1e-6).mean() >= 0.95
