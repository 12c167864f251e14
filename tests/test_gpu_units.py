"""Single solver stages on arbitrary inputs, at every size branch, CTA width and memory placement.

One case table, two backends.  Every case runs on the host build of the kernel source (tests/hostsim: one-thread CTA,
SM = false, none of the GPU-only code) on CPU, which validates the inputs, the references and the tolerances; the same
cases run on the CUDA kernels (tests/gpu_units/units.cu) in the tests marked ``gpu``, parametrised by CTA width and
shared-memory budget.  The GPU tolerances are about ten times the host build's error on the same input (clustered
spectra: the cluster bar), and never looser than the bars of the existing stage tests.

Stages and references (float64 LAPACK where it is accurate enough, np.longdouble where it is not):
  nearestPD  H = sym(Q) + sum_{s_i < 0} (floor - s_i) u_i u_i' + reg I  (eigh of sym(Q)), nneg exactly
  qp_factor  Cholesky L and Y = L^-1 by a plain long-double loop, xq = -H^-1 q
  QP         oracle.qp.solve_qp_gi and the KKT residuals, cold and warm (gi_warm_start)
  evaluate   Q, q, G'l, g and the matrix-free G products against the oracle games

The branch a case reaches follows from n, the CTA width, the spectrum and the memory plan (``branches``); the plan each
run reports is asserted, and ``test_case_table_reaches_every_branch`` checks that the table covers all of them."""
import functools
import os

import numpy as np
import pytest

import dgsqp_b200 as dg
from dgsqp_b200.games import MergeGame

EPS = np.finfo(np.float64).eps
SMEM_DEFAULT = 28000            # doubles: the shared-memory budget of the "smem" placement (B200: at most ~28600 available)
BUDGETS = ("smem", "split", "global")

# ------------------------------------------------------------------ games: n = 2 M N (merge: 2 M N with M = 3)
SIZES = {     # n: (label, game factory)
    32: ("M2N8", lambda: dg.chicane_game(N=8)),
    36: ("M3N6", lambda: dg.agents_game(3, 90.0, 6)),
    48: ("M2N12", lambda: dg.chicane_game(N=12)),
    64: ("M2N16", lambda: dg.chicane_game(N=16)),
    68: ("M2N17", lambda: dg.chicane_game(N=17)),
    96: ("M2N24", lambda: dg.chicane_game(N=24)),
    100: ("chicane", lambda: dg.chicane_game()),
    120: ("merge", lambda: dg.merge_game()),
    128: ("M4N16", lambda: dg.agents_game(4, 90.0, 16)),
    132: ("M2N33", lambda: dg.chicane_game(N=33)),
    150: ("M3N25", lambda: dg.agents_game(3, 90.0, 25)),
    200: ("M4N25", lambda: dg.agents_game(4, 90.0, 25)),
    256: ("M4N32", lambda: dg.agents_game(4, 90.0, 32)),
    258: ("M3N43", lambda: dg.agents_game(3, 90.0, 43)),
}
NARROW = {32: (32, 64, 96, 128), 36: (32, 96), 64: (32, 64), 68: (32, 96, 128), 100: (32, 64, 96, 128),
          120: (64, 96), 132: (32, 128), 200: (96,), 256: (64,), 258: (32, 96, 128)}


@functools.lru_cache(maxsize=None)
def game_of(n):
    return SIZES[n][1]()


def params_of(game):
    if isinstance(game, MergeGame):
        return dg.merge_params(game.N)
    return dg.chicane_params(game.N) if game.M == 2 else dg.agents_params(game.N)


def oracle_of(game):
    from oracle.merge_game import MergeGame as OMerge
    from oracle.racing_game import RacingGame
    from oracle.track import chicane_track, curve_track
    if isinstance(game, MergeGame):
        return OMerge(N=game.N)
    if game.M == 2:
        return RacingGame(chicane_track(), M=2, N=game.N)
    return RacingGame(curve_track(curve_angle=np.pi / 2), M=game.M, N=game.N, obs_r=0.4)


def hostsim(game, budget_doubles):
    from hostsim_lib import HostSim
    old = os.environ.get("DG_HOSTSIM_SMEM_DOUBLES")
    os.environ["DG_HOSTSIM_SMEM_DOUBLES"] = str(budget_doubles)
    try:
        return HostSim(game, params_of(game))
    finally:
        if old is None:
            del os.environ["DG_HOSTSIM_SMEM_DOUBLES"]
        else:
            os.environ["DG_HOSTSIM_SMEM_DOUBLES"] = old


@functools.lru_cache(maxsize=None)
def budget_doubles(n, budget):
    """Shared-memory budget of a placement: "smem" the default, "global" none, "split" the largest budget that puts matA
    but not matB in shared memory (so that the inverse-iteration block eig_s fits too); None where no split exists."""
    if budget == "smem":
        return SMEM_DEFAULT
    if budget == "global":
        return 0
    game = game_of(n)
    plan = lambda b: hostsim(game, b).plan()
    if not plan(SMEM_DEFAULT)[2]:
        return None
    if not plan(SMEM_DEFAULT)[1]:
        return SMEM_DEFAULT
    lo, hi = 0, SMEM_DEFAULT           # plan(lo) keeps matB out of shared memory, plan(hi) does not
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (lo, mid) if plan(mid)[1] else (mid, hi)
    return lo if plan(lo)[2] else None


def placement(plan):
    """'smem' (SM = true: every hot buffer in shared memory), 'split' (matA in shared memory, matB in L2) or 'global'."""
    if plan["hot_in_smem"]:
        return "smem"
    return "split" if plan["matA_in_smem"] and not plan["mats_in_smem"] else "global"


def plan_dict(t):
    return dict(zip(("hot_in_smem", "mats_in_smem", "matA_in_smem", "sens_in_smem", "eig_s"), t))


# ------------------------------------------------------------------ nearestPD inputs: Q = U diag(s) U'
def eig_cap(n):
    """Eigenvectors that fit behind the inverse-iteration scratch in matB (linalg.cuh, nearest_pd); more go to Zg."""
    ld = n | 1
    return (n * ld - ((n + 1) // 2 + 1 + 6 * n * 16)) // n


def spectra(n):
    """name -> (negative eigenvalues, scale, clustered).  Negatives stay >= 1e-6 |Q| away from zero (nneg is exact)."""
    sep = lambda k: -np.linspace(6.0, 0.5, k) if k > 1 else np.array([-1.5])
    out = {"pos": (np.array([]), 1.0, False), "sep1": (sep(1), 1.0, False), "sep2": (sep(2), 1.0, False),
           "sep3": (sep(3), 1.0, False), "neg16": (sep(16), 1.0, False), "neg17": (sep(17), 1.0, False),
           "clus3": (np.array([-5.0, -2.0, -2.0 * (1 + 1e-12), -2.0 * (1 - 1e-12)]), 1.0, True),
           # a 5-fold cluster at ascending positions 14..18: it straddles the boundary of the 16-vector chunks
           "straddle": (np.concatenate([-np.linspace(10.0, 4.0, 14), [-2.0, -2.0, -2.0 - 1e-12, -2.0 + 1e-12, -2.0],
                                        [-1.0, -0.5]]), 1.0, True),
           "huge": (sep(2), 1e19, False)}     # |Q| ~ 1e19: pivmin >= 1.3e36 DBL_MIN, the scalar Sturm count
    cap = eig_cap(n)
    if cap >= 4:                              # below n ~ 97 every eigenvector lives in Zg anyway
        out["spill"] = (sep(cap + 3), 1.0, False)
    return out


@functools.lru_cache(maxsize=None)
def npd_inputs(n, seed=0):
    rng = np.random.default_rng(seed + n)
    names, Qs = [], []
    for name, (neg, scale, _) in spectra(n).items():
        U, _ = np.linalg.qr(rng.normal(size=(n, n)))
        s = np.concatenate([neg, rng.uniform(0.1, 5.0, n - len(neg))]) * scale
        rng.shuffle(s)
        Q = (U * s) @ U.T
        Q = Q + 1e-14 * scale * rng.normal(size=(n, n))           # not exactly symmetric: the kernel symmetrises
        names.append(name)
        Qs.append(Q)
    return names, np.array(Qs)


@functools.lru_cache(maxsize=None)
def npd_reference(n):
    game = game_of(n)
    p = params_of(game)
    names, Qs = npd_inputs(n)
    refs = []
    for Q in Qs:
        S = 0.5 * (Q + Q.T)
        s, U = np.linalg.eigh(S)
        neg = s < 0
        H = S + (U[:, neg] * (1e-10 - s[neg])) @ U[:, neg].T + p.reg * np.eye(n)
        refs.append((H, int(neg.sum()), float(np.sum(1e-10 - s[neg]))))
    return refs


@functools.lru_cache(maxsize=None)
def npd_host(n, budget):
    hs = hostsim(game_of(n), budget_doubles(n, budget))
    _, Qs = npd_inputs(n)
    res = [hs.nearest_pd(Q) for Q in Qs]
    return np.array([r[0] for r in res]), np.array([r[1] for r in res]), plan_dict(hs.plan())


def npd_errors(n, H, nneg):
    """Per instance: max|H - H_ref| and its bar (1e-11 |Q|, clusters 1e-9 |Q|), nneg and the reference count, the
    asymmetry |H - H'| (rounding of (floor - lambda) z_i z_j, formed left to right) and its bound, lambda_min(H)."""
    names, Qs = npd_inputs(n)
    reg = params_of(game_of(n)).reg
    out = []
    for i, name in enumerate(names):
        Href, nref, wsum = npd_reference(n)[i]
        clustered = spectra(n)[name][2]
        scale = max(1.0, np.abs(Qs[i]).max())
        bar = (1e-9 if clustered else 1e-11) * scale
        asym = np.abs(H[i] - H[i].T).max()
        out.append(dict(name=name, err=np.abs(H[i] - Href).max(), bar=bar, scale=scale, nneg=int(nneg[i]), nref=nref,
                        asym=asym, asym_bound=8 * EPS * (wsum + reg + scale),
                        lmin=np.linalg.eigvalsh(0.5 * (H[i] + H[i].T)).min() if reg > 0 and scale < 1e3 else None,
                        reg=reg))
    return out


def check_npd(errs, tols=None):
    for k, e in enumerate(errs):
        tol = e["bar"] if tols is None else tols[k]
        assert e["nneg"] == e["nref"], f"{e['name']}: nneg {e['nneg']} != {e['nref']}"
        assert e["err"] <= tol, f"{e['name']}: max|H - H_ref| = {e['err']:.3g} > {tol:.3g}"
        assert e["asym"] <= e["asym_bound"], f"{e['name']}: asymmetry {e['asym']:.3g}"
        if e["lmin"] is not None:
            assert e["lmin"] >= 0.9 * e["reg"], f"{e['name']}: lambda_min(H) = {e['lmin']:.3g}"


def gpu_tol(host_err, bar, scale):
    """About ten times the host build's error on the same input, never looser than the existing bar."""
    return min(bar, max(10.0 * host_err, 1e-14 * scale))


# ------------------------------------------------------------------ qp_factor inputs and the long-double reference
FACTOR_CONDS = (1e2, 1e6, 1e10)


@functools.lru_cache(maxsize=None)
def factor_inputs(n, seed=0):
    rng = np.random.default_rng(seed + 7 * n)
    Hs, qs = [], []
    for cond in FACTOR_CONDS + (None,):
        U, _ = np.linalg.qr(rng.normal(size=(n, n)))
        s = 4.0 * np.geomspace(1.0 / cond, 1.0, n) if cond else np.concatenate([[-1.0], rng.uniform(0.5, 4.0, n - 1)])
        rng.shuffle(s)
        H = (U * s) @ U.T
        Hs.append(0.5 * (H + H.T))
        qs.append(rng.normal(size=n))
    return np.array(Hs), np.array(qs)


def chol_inv_longdouble(H):
    """Lower Cholesky factor and its inverse in extended precision, row by row."""
    n = H.shape[0]
    A = H.astype(np.longdouble)
    L = np.zeros((n, n), dtype=np.longdouble)
    for j in range(n):
        d = A[j, j] - np.dot(L[j, :j], L[j, :j])
        L[j, j] = np.sqrt(d)
        L[j + 1:, j] = (A[j + 1:, j] - L[j + 1:, :j] @ L[j, :j]) / L[j, j]
    Y = np.zeros((n, n), dtype=np.longdouble)
    for i in range(n):
        row = -(L[i, :i] @ Y[:i, :]) if i else np.zeros(n, dtype=np.longdouble)
        row[i] += 1
        Y[i] = row / L[i, i]
    return L, Y


@functools.lru_cache(maxsize=None)
def factor_reference(n):
    Hs, qs = factor_inputs(n)
    out = []
    for k in range(len(FACTOR_CONDS)):
        L, Y = chol_inv_longdouble(Hs[k])
        xq = -(Y.T @ (Y @ qs[k].astype(np.longdouble)))
        out.append((L, Y, xq))
    return out


@functools.lru_cache(maxsize=None)
def factor_host(n, budget):
    hs = hostsim(game_of(n), budget_doubles(n, budget))
    Hs, qs = factor_inputs(n)
    res = [hs.factor(H, q) for H, q in zip(Hs, qs)]
    return (np.array([r[0] for r in res]), np.array([r[1] for r in res]), np.array([r[2] for r in res]),
            np.array([r[3] for r in res]), plan_dict(hs.plan()))


def factor_errors(n, ok, L, Y, xq):
    """Per SPD instance: relative errors of L, Y L - I, xq, and the strict upper triangle of Y; ok of every instance."""
    refs = factor_reference(n)
    out = []
    for k, cond in enumerate(FACTOR_CONDS):
        Lr, Yr, xr = refs[k]
        Lr, xr = Lr.astype(np.float64), xr.astype(np.float64)
        out.append(dict(cond=cond, ok=bool(ok[k]),
                        L=np.abs(L[k] - Lr).max() / np.abs(Lr).max(),
                        YL=np.abs(Y[k].astype(np.longdouble) @ L[k].astype(np.longdouble) - np.eye(n)).max().astype(np.float64),
                        xq=np.abs(xq[k] - xr).max() / max(1.0, np.abs(xr).max()),
                        upper=np.abs(np.triu(Y[k], 1)).max()))
    return out, [bool(v) for v in ok[len(FACTOR_CONDS):]]


def factor_bars(n, cond):
    """Bars from the conditioning alone (the GPU is held to min(bar, 10 x host error))."""
    return dict(L=50 * n * EPS * cond, YL=50 * n * EPS * np.sqrt(cond), xq=50 * n * EPS * cond)


def check_factor(n, errs, indef_ok, tols=None):
    for k, e in enumerate(errs):
        bars = factor_bars(n, e["cond"]) if tols is None else tols[k]
        assert e["ok"], f"cond {e['cond']:g}: factorisation refused an SPD matrix"
        assert e["upper"] == 0.0, f"cond {e['cond']:g}: strict upper triangle of Y not zero ({e['upper']:.3g})"
        for key in ("L", "YL", "xq"):
            assert e[key] <= bars[key], f"cond {e['cond']:g}: {key} error {e[key]:.3g} > {bars[key]:.3g}"
    assert not any(indef_ok), "an indefinite H was factored"


# ------------------------------------------------------------------ QP / G inputs: evaluated games
QP_GAMES = (100, 120, 132, 150, 200, 258)       # chicane N25, merge N20, M2 N33, agents 3 and 4 at N25, M3 N43
QP_WIDTHS = {100: (64, 128, 256), 120: (64, 96, 256), 132: (256,), 150: (96, 256), 200: (64, 256), 258: (128, 256)}
QP_REG = 1e-3


@functools.lru_cache(maxsize=None)
def game_inputs(n, B=2, seed=0):
    """B evaluation points (x0, u, l) of the game of size n."""
    game, og = game_of(n), oracle_of(game_of(n))
    rng = np.random.default_rng(seed + n)
    if isinstance(game, MergeGame):
        from dgsqp_b200.montecarlo import sample_merge
        x0, _ = sample_merge(game, B, seed=1)
    else:
        M = game.M
        x0 = []
        for b in range(B):
            x = np.concatenate([[0, 0, 2.2 + 0.3 * a + 0.1 * b, 0.0, 0.4 + 0.9 * a + 0.2 * b, 0.45 - 0.3 * a] for a in range(M)])
            for a in range(M):
                x[6 * a], x[6 * a + 1], _ = og.track.local_to_global((x[6 * a + 4], x[6 * a + 5], 0.0))
            x0.append(x)
        x0 = np.array(x0)
    u = rng.normal(size=(B, game.n)) * 0.15
    l = np.abs(rng.normal(size=(B, game.m))) * 0.3 * (rng.random((B, game.m)) < 0.3)
    return x0, u, l


@functools.lru_cache(maxsize=None)
def game_reference(n):
    """Oracle evaluation (Q, q, G, g) per instance, H = nearestPD(Q) + 1e-3 I, q2 (perturbed q), the cold and warm
    reference QP solutions, and the seeded G-product operands."""
    from oracle.dgsqp_v1 import nearest_pd
    from oracle.qp import solve_qp_gi
    game, og = game_of(n), oracle_of(game_of(n))
    x0, u, l = game_inputs(n)
    rng = np.random.default_rng(100 + n)
    out = []
    for i in range(x0.shape[0]):
        Q, q, G, g, _ = og.evaluate(u[i], l[i], x0[i], np.zeros(og.n_u), True)
        H = nearest_pd(Q) + QP_REG * np.eye(n)
        q2 = q + 0.05 * max(1.0, np.abs(q).max()) * rng.normal(size=n)
        du, lam = solve_qp_gi(H, q, G, g)
        du2, lam2 = solve_qp_gi(H, q2, G, g)
        rows = np.sort(np.concatenate([[0, game.m - 1], rng.choice(np.arange(1, game.m - 1), size=min(30, n) - 2, replace=False)]))
        out.append(dict(Q=Q, q=q, G=G, g=g, H=H, q2=q2, du=du, lam=lam, du2=du2, lam2=lam2, v=rng.normal(size=n),
                        w=rng.normal(size=game.m), rows=rows))
    return out


def rel(a, b):
    return np.abs(a - b).max() / max(1.0, np.abs(b).max())


def check_eval(ref, Q, q, gtl, g, l):
    assert rel(Q, ref["Q"]) < 1e-12 and rel(q, ref["q"]) < 1e-12
    assert rel(gtl, ref["G"].T @ l) < 1e-12 and rel(g, ref["g"]) < 1e-13


def check_qp(ref, st, du, lam, q, key=""):
    """At the bars of the stage test.  Where the active rows of the reference solution are linearly dependent the
    multipliers are not unique (G' lam is, through the KKT residuals)."""
    from oracle.qp import kkt_residuals
    assert st == 0, f"QP{key} status {st}"
    assert rel(du, ref["du" + key]) < 1e-8
    act = np.where(np.abs(ref["g"] + ref["G"] @ ref["du" + key]) < 1e-9)[0]
    if len(act) == 0 or np.linalg.matrix_rank(ref["G"][act]) == len(act):
        assert rel(lam, ref["lam" + key]) < 1e-7
    r = kkt_residuals(ref["H"], q, ref["G"], ref["g"], du, lam)
    assert r["stat"] < 1e-8 and r["feas"] < 1e-9 and r["dual"] == 0.0 and r["comp"] < 1e-8, r


def check_G(ref, Gv, GTw, rows):
    G = ref["G"]
    assert np.abs(G @ ref["v"] - Gv).max() < 1e-11 * max(1.0, np.abs(G).max())
    assert np.abs(G.T @ ref["w"] - GTw).max() < 1e-11 * max(1.0, np.abs(G).max())
    assert np.abs(G[ref["rows"]] - rows).max() < 1e-12 * max(1.0, np.abs(G).max())


# ------------------------------------------------------------------ branches a run takes (linalg.cuh / qp_gi.cuh / game_kkt.cuh)
def npd_branches(n, threads, plan, name):
    neg, scale, clustered = spectra(n)[name]
    nneg = len(neg)
    wide_sturm = scale < 1e18                      # pivmin < 1.3e36 DBL_MIN: the half-warp Sturm counts
    b = {f"width{threads}", "placement_" + placement(plan)}
    if threads == 256 and 33 <= n <= 128:
        b.add(f"tridiag_tiles_T{(n + 15) // 16}")
    elif threads == 256 and 128 < n <= 256:
        b.add("tridiag_hybrid")
    else:
        b.add("tridiag_generic_gt256" if n > 256 else "tridiag_generic")
    b.add("sturm_grp16" if wide_sturm else "sturm_scalar")
    if nneg == 0:
        return b | {"identity_path"}
    b.add("multisect_grp" if nneg <= 16 and threads >= 16 * nneg and wide_sturm else "multisect_cta")
    if 33 <= n <= 128 and wide_sturm and not clustered:
        b.add(f"twisted_R{2 if n <= 64 else 4}")
    else:
        b.add("invit_cluster" if clustered else "invit")
        if name == "straddle":
            b.add("invit_cross_chunk")
        if plan["eig_s"] and not plan["hot_in_smem"] and nneg <= 2:
            b.add("eig_s")
    if nneg > eig_cap(n):
        b.add("Zg")
    b.add({2: "backtransform_RPL2", 4: "backtransform_RPL4", 8: "backtransform_RPL8"}.get(
        1 if n > 256 else (2 if n <= 64 else 4 if n <= 128 else 8), "backtransform_scalar"))
    return b


def factor_branches(n, threads, plan):
    b = {f"width{threads}", "placement_" + placement(plan)}
    if threads == 256 and 33 <= n <= 128:
        b |= {f"chol_tiles_T{(n + 15) // 16}", f"trinv_tiles_T{(n + 15) // 16}"}
    elif threads == 256 and 128 < n <= 256:
        b |= {"chol_hybrid", "trinv_generic"}
    else:
        b |= {"chol_generic", "trinv_generic"}
    return b


def costate_groups_wrap(game, threads):
    nqa = 4 if isinstance(game, MergeGame) else 6
    nch = (game.M + 1) * game.M
    cpw = 32 // nqa
    return (nch + cpw - 1) // cpw > threads // 32


def game_branches(n, threads, plan):
    game = game_of(n)
    b = {f"width{threads}", "placement_" + placement(plan), "qp_warm_start"}
    b.add("game_merge" if isinstance(game, MergeGame) else f"game_racing_M{game.M}")
    if costate_groups_wrap(game, threads):
        b.add("costate_groups_wrap")
    return b


REQUIRED = ({f"tridiag_tiles_T{t}" for t in range(3, 9)} | {f"chol_tiles_T{t}" for t in range(3, 9)}
            | {f"trinv_tiles_T{t}" for t in range(3, 9)}
            | {"tridiag_hybrid", "tridiag_generic", "tridiag_generic_gt256", "chol_hybrid", "chol_generic",
               "twisted_R2", "twisted_R4", "invit", "invit_cluster", "invit_cross_chunk", "identity_path",
               "backtransform_RPL2", "backtransform_RPL4", "backtransform_RPL8", "backtransform_scalar",
               "multisect_grp", "multisect_cta", "sturm_grp16", "sturm_scalar", "Zg", "eig_s",
               "placement_smem", "placement_split", "placement_global", "width32", "width96", "width256",
               "qp_warm_start", "game_merge", "game_racing_M3", "game_racing_M4", "costate_groups_wrap"})


def npd_cells():
    for n in SIZES:
        for threads in (256,) + NARROW.get(n, ()):
            for budget in BUDGETS:
                if budget == "split" and budget_doubles(n, budget) is None:
                    continue
                if threads != 256 and budget == "split" and n not in (68, 100):
                    continue
                yield n, threads, budget


def qp_cells():
    for n in QP_GAMES:
        for threads in QP_WIDTHS[n]:
            for budget in BUDGETS:
                if budget == "split" and budget_doubles(n, budget) is None:
                    continue
                yield n, threads, budget


def cell_id(c):
    return f"n{c[0]}-{SIZES[c[0]][0]}-t{c[1]}-{c[2]}"


@functools.lru_cache(maxsize=None)
def host_plan(n, budget):
    """The memory plan of a budget: plan_memory is the same function of the budget on both backends."""
    return plan_dict(hostsim(game_of(n), budget_doubles(n, budget)).plan())


def expected_plan(n, budget):
    return placement(host_plan(n, budget))


# ================================================================== host build (CPU)
def test_case_table_reaches_every_branch():
    """Every branch of the GPU-only code is the target of at least one case of the table."""
    reached = set()
    for n, threads, budget in npd_cells():
        plan = host_plan(n, budget)
        for name in spectra(n):
            reached |= npd_branches(n, threads, plan, name)
        reached |= factor_branches(n, threads, plan)
    for n, threads, budget in qp_cells():
        reached |= game_branches(n, threads, host_plan(n, budget))
    assert not REQUIRED - reached, f"not reached: {sorted(REQUIRED - reached)}"
    # the placements the budgets are meant to give
    assert expected_plan(100, "smem") == "smem" and expected_plan(100, "split") == "split"
    assert expected_plan(128, "split") == "split" and expected_plan(258, "global") == "global"
    assert all(expected_plan(n, "global") == "global" for n in SIZES)
    # nneg = 16 vs 17 straddles the half-warp multisection at 256 threads; the spill case exceeds the Zg cap
    assert len(spectra(100)["neg16"][0]) == 16 and len(spectra(100)["neg17"][0]) == 17
    assert eig_cap(100) == 4 and eig_cap(256) == 160 and len(spectra(256)["spill"][0]) > 160


@pytest.mark.parametrize("n,budget", [(n, b) for n in SIZES for b in BUDGETS if budget_doubles(n, b) is not None],
                         ids=lambda v: str(v))
def test_host_nearest_pd(n, budget):
    H, nneg, plan = npd_host(n, budget)
    check_npd(npd_errors(n, H, nneg))


def _cpu_has_fma():
    try:
        return any(ln.startswith("flags") and " fma " in ln + " " for ln in open("/proc/cpuinfo"))
    except OSError:
        return False


@pytest.mark.skipif(not _cpu_has_fma(), reason="needs a CPU with FMA instructions")
@pytest.mark.parametrize("n", [32, 36, 64, 68, 100, 150])
def test_host_nearest_pd_contracted_products(n):
    """The kernel source compiled with its products contracted into FMAs wherever the compiler likes (as nvcc compiles it)
    must keep the nearestPD accuracy: a contracted rank-2 update A22 -= v w' + w v' in sym_tridiag left A22 asymmetric
    and cost the straddling and the 3-fold cluster up to 1e-4 of H."""
    from hostsim_lib import HostSim
    old = os.environ.get("DG_HOSTSIM_SMEM_DOUBLES")
    os.environ["DG_HOSTSIM_SMEM_DOUBLES"] = "0"
    try:
        hs = HostSim(game_of(n), params_of(game_of(n)), fma=True)
    finally:
        if old is None:
            del os.environ["DG_HOSTSIM_SMEM_DOUBLES"]
        else:
            os.environ["DG_HOSTSIM_SMEM_DOUBLES"] = old
    _, Qs = npd_inputs(n)
    res = [hs.nearest_pd(Q) for Q in Qs]
    check_npd(npd_errors(n, np.array([r[0] for r in res]), np.array([r[1] for r in res])))


@pytest.mark.parametrize("n", list(SIZES))
def test_host_factor(n):
    ok, L, Y, xq, _ = factor_host(n, "smem")
    errs, indef = factor_errors(n, ok, L, Y, xq)
    check_factor(n, errs, indef)


@pytest.mark.parametrize("n", QP_GAMES)
def test_host_evaluate_qp_and_G(n):
    game = game_of(n)
    hs = hostsim(game, SMEM_DEFAULT)
    x0, u, l = game_inputs(n)
    for i, ref in enumerate(game_reference(n)):
        Q, q, gtl, g, _ = hs.evaluate(x0[i], u[i], l[i])
        check_eval(ref, Q, q, gtl, g, l[i])
        check_G(ref, hs.G_times(ref["v"]), hs.GT_times(ref["w"]), hs.G_dense()[ref["rows"]])
        st, du, lam, _ = hs.qp(ref["H"], q)
        check_qp(ref, st, du, lam, q)
        st, du, lam, _ = hs.qp_warm(ref["H"], ref["q2"])
        check_qp(ref, st, du, lam, ref["q2"], "2")


# ================================================================== CUDA kernels (B200)
@pytest.mark.gpu
@pytest.mark.parametrize("cell", list(npd_cells()), ids=cell_id)
def test_gpu_nearest_pd(cell):
    import gpu_units_lib as U
    n, threads, budget = cell
    game = game_of(n)
    names, Qs = npd_inputs(n)
    out = U.nearest_pd(game, params_of(game), Qs, threads=threads, smem_limit_doubles=budget_doubles(n, budget))
    assert out["plan"] == host_plan(n, budget)
    Hh, nh, _ = npd_host(n, budget)
    host = npd_errors(n, Hh, nh)
    errs = npd_errors(n, out["H"], out["nneg"])
    # separated spectra: ten times the host build's error; clusters: the cluster bar (the register-tile tridiagonalisation
    # contracts its rank-2 update, which leaves 3-fold clusters at 1e-10; the host build has no contracted products)
    check_npd(errs, [h["bar"] if spectra(n)[h["name"]][2] else gpu_tol(h["err"], h["bar"], h["scale"]) for h in host])


@pytest.mark.gpu
@pytest.mark.parametrize("cell", [c for c in npd_cells() if c[2] != "split" or c[1] == 256], ids=cell_id)
def test_gpu_factor(cell):
    import gpu_units_lib as U
    n, threads, budget = cell
    game = game_of(n)
    Hs, qs = factor_inputs(n)
    out = U.factor(game, params_of(game), Hs, qs, threads=threads, smem_limit_doubles=budget_doubles(n, budget))
    assert out["plan"] == host_plan(n, budget)
    host, _ = factor_errors(n, *factor_host(n, "smem")[:4])
    tols = []
    for h in host:
        bars = factor_bars(n, h["cond"])
        tols.append({k: min(bars[k], max(10 * h[k], n * EPS)) for k in ("L", "YL", "xq")})
    errs, indef = factor_errors(n, out["ok"], out["L"], out["Y"], out["xq"])
    check_factor(n, errs, indef, tols)


@pytest.mark.gpu
@pytest.mark.parametrize("cell", list(qp_cells()), ids=cell_id)
def test_gpu_evaluate_qp_and_G(cell):
    import gpu_units_lib as U
    n, threads, budget = cell
    game = game_of(n)
    params, refs = params_of(game), game_reference(n)
    x0, u, l = game_inputs(n)
    lim = budget_doubles(n, budget)
    H = np.array([r["H"] for r in refs])
    q = np.array([r["q"] for r in refs])
    q2 = np.array([r["q2"] for r in refs])
    out = U.qp(game, params, x0, u, l, H, q, q2, threads=threads, smem_limit_doubles=lim)
    gp = U.G_products(game, params, x0, u, l, np.array([r["v"] for r in refs]), np.array([r["w"] for r in refs]),
                      np.array([r["rows"] for r in refs]), threads=threads, smem_limit_doubles=lim)
    assert out["plan"] == gp["plan"] == host_plan(n, budget)
    for i, ref in enumerate(refs):
        check_eval(ref, out["Q"][i], out["q"][i], out["gtl"][i], out["g"][i], l[i])
        check_eval(ref, gp["Q"][i], gp["q"][i], gp["gtl"][i], gp["g"][i], l[i])
        check_qp(ref, out["st"][i], out["du"][i], out["lam"][i], q[i])
        check_qp(ref, out["st2"][i], out["du2"][i], out["lam2"][i], q2[i], "2")
        check_G(ref, gp["Gv"][i], gp["GTw"][i], gp["rows"][i])
        assert np.array_equal(gp["cols"][i], gp["rows"][i])       # game_G_cols == game_G_row, entry for entry
