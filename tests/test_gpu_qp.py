"""The dual active-set QP (qp_gi.cuh: qp_factor, gi_warm_start, qp_gi_loop, gi_polish) on QPs with a known answer,
on infeasible QPs and from given warm-start lists.

The constraint matrix is the matrix-free G of an evaluated game; the offsets g, the gradient q and the Hessian H are
chosen by the test.  One case table, two backends: every case runs on the host build of the kernel source on CPU and, in
the tests marked ``gpu``, on the CUDA kernels at several CTA widths and memory placements.

References, in np.longdouble:
  known answer  pick x*, an independent set W of rows of G, lam_W >= 1e-3 and slacks >= 1e-3 on the other rows; then
                q = -H x* - G_W' lam_W, g_W = -G_W x*, g_i = -G_i x* - s_i.  The reference is the equality-constrained
                minimiser on W of the rounded (q, g).
  infeasible    an upper and a lower bound of one input with contradicting offsets: status 2, and the oracle raises
  warm start    steps (1)-(4) of gi_warm_start restated: walk the ids in order and accept a column when |d2|^2 > 1e-20 |d|^2
                (d = J'n); the equality-constrained minimiser on the accepted set; drop the most negative multiplier
                until none is negative.  Only exact dependences (duplicates, bound / bound / rate triples, the two bounds
                of one input) and clearly independent columns are used, so the 1e-20 test is never near its threshold.

The host build is held to the bars of the stage test (du 1e-8, lam 1e-7, stationarity 1e-8, feasibility 1e-9,
complementarity 1e-8; du at least 10 eps cond(H)); the GPU to ten times the host build's error where that is tighter (see
tol), with the host build's status and accepted ids, and where the path is determined (same_path) its active-row count
and main-loop iteration count."""
import functools
import sys

import numpy as np
import pytest

from test_gpu_units import (BUDGETS, SIZES, budget_doubles, chol_inv_longdouble, game_inputs, game_of, host_plan,
                            hostsim, oracle_of, params_of, placement, rel)

LD = np.longdouble
PW = 8                      # DG_WS_PW: panel width of the warm start's blocked QR
DEP_TOL = 1e-20             # DG_QP_DEP_TOL
QP_SIZES = (32, 36, 100, 120, 150, 258)
WIDTHS = {32: (32, 256), 36: (96, 256), 100: (32, 128, 256), 120: (96, 256), 150: (96, 256), 258: (128, 256)}
H_KINDS = ("game", "spd1e2", "spd1e8")
BARS = dict(du=1e-8, lam=1e-7, stat=1e-8, feas=1e-9, comp=1e-8)
EPS = np.finfo(np.float64).eps


def du_bar(P, hk):
    """The du bar, or 10 eps cond(H) where that is larger: the forward error of x cannot fall below eps cond(H) (cond
    1e8: 2.2e-7).  The residual bars do not depend on the conditioning."""
    return max(BARS["du"], 10 * EPS * np.linalg.cond(P["H"][hk]))


def w_sizes(n):
    return (0, 1, 7, 8, 9, 16, 17) + tuple(range(n - 9, n + 1))


# ------------------------------------------------------------------ the evaluated game and its rows
@functools.lru_cache(maxsize=None)
def problem(n):
    """G of the game at the first point of game_inputs, the Hessians, their long-double inverse Cholesky factors and
    the rows by kind: input upper / lower bounds per input, rate rows (+1 at j1, -1 at j2), the other non-zero rows."""
    from oracle.dgsqp_v1 import nearest_pd
    game, og = game_of(n), oracle_of(game_of(n))
    x0, u, l = game_inputs(n)
    Q, _, G, _, _ = og.evaluate(u[0], l[0], x0[0], np.zeros(og.n_u), True)
    rng = np.random.default_rng(300 + n)
    Hs = {"game": nearest_pd(Q) + 1e-3 * np.eye(n)}
    for name, cond in (("spd1e2", 1e2), ("spd1e8", 1e8)):
        U, _ = np.linalg.qr(rng.normal(size=(n, n)))
        s = 4.0 * np.geomspace(1.0 / cond, 1.0, n)
        rng.shuffle(s)
        H = (U * s) @ U.T
        Hs[name] = 0.5 * (H + H.T)
    kinds = sys.modules[type(og).__module__]
    ub, lb, rate, dense = {}, {}, [], []
    for r, (k, kind, a, b) in enumerate(og.rows):
        nz = np.flatnonzero(G[r])
        if kind == kinds.IN_UB:
            ub[og.uidx(a, k, b)] = r
        elif kind == kinds.IN_LB:
            lb[og.uidx(a, k, b)] = r
        elif len(nz) == 2 and sorted(G[r, nz]) == [-1.0, 1.0] and kind == getattr(kinds, "RATE", -1):
            rate.append((r, int(nz[G[r, nz] > 0][0]), int(nz[G[r, nz] < 0][0])))
        elif len(nz):
            dense.append(r)
    assert len(ub) == len(lb) == n
    Y = {h: chol_inv_longdouble(H)[1] for h, H in Hs.items()}
    return dict(n=n, m=G.shape[0], G=G, H=Hs, Y=Y, ub=ub, lb=lb, rate=rate, dense=dense, x0=x0[0], u=u[0], l=l[0])


def eq_solve(P, hk, A, q, g, dtype=LD):
    """Minimiser of 1/2 x'Hx + q'x on G_A x = -g_A (A independent) and its multipliers (H x + q + G_A' lam = 0).  With
    Y = L^-1 and Z = Y G_A' the system H x + G_A' lam = a, G_A x = b is solved by  lam = (Z'Z)^-1 (Z'Y a - b),
    x = Y'(Y a - Z lam);  in long double with two steps of iterative refinement (Z'Z squares the conditioning)."""
    Y = P["Y"][hk].astype(dtype)
    A = list(A)
    a = -np.asarray(q, dtype=dtype)
    if not A:
        return Y.T @ (Y @ a), np.zeros(0, dtype=dtype)
    GA = P["G"][A].astype(dtype)
    b = -np.asarray(g, dtype=dtype)[A]
    Z = Y @ GA.T
    if dtype == LD:
        Ys = chol_inv_longdouble(Z.T @ Z)[1]
        Sinv = lambda r: Ys.T @ (Ys @ r)
    else:
        Sinv = lambda r, S=Z.T @ Z: np.linalg.solve(S, r)

    def solve(ra, rb):
        ya = Y @ ra
        lam = Sinv(Z.T @ ya - rb)
        return Y.T @ (ya - Z @ lam), lam
    x, lam = solve(a, b)
    if dtype == LD:
        H = P["H"][hk].astype(LD)
        for _ in range(2):
            dx, dl = solve(a - H @ x - GA.T @ lam, b - GA @ x)
            x, lam = x + dx, lam + dl
    return x, lam


def pick_rows(P, k, rng, avoid=(), dense_max=6):
    """k linearly independent rows: up to dense_max (at most k // 3) rows that read the sensitivities, and bounds of
    distinct inputs, none on the inputs in avoid nor on the pivot inputs of the dense rows (pivoted QR), so that even
    k = n rows stay well conditioned."""
    import scipy.linalg as sla
    n, G = P["n"], P["G"]
    free = np.array([j for j in range(n) if j not in avoid])
    for _ in range(50):
        nd = min(k // 3, dense_max)
        rows = [int(r) for r in rng.choice(P["dense"], size=nd, replace=False)] if nd else []
        piv = free[sla.qr(G[rows][:, free], pivoting=True)[2][:nd]] if nd else []
        js = rng.choice(np.setdiff1d(free, piv), size=k - nd, replace=False)
        rows += [P["ub"][j] if rng.random() < 0.5 else P["lb"][j] for j in js]
        rows = [int(r) for r in rng.permutation(rows)]
        Gn = G[rows] / np.linalg.norm(G[rows], axis=1, keepdims=True) if k else None
        if k == 0 or np.linalg.cond(Gn) < 1e6:
            return rows
    raise AssertionError("no independent row set found")


def known_answer(P, hk, W, rng, weak=(), dependent=False):
    """(q, g) whose QP has the solution x* with the active set W (lam_W >= 1e-3), the rows weak tight with lam = 0 and
    slacks >= 1e-3 elsewhere; the reference (x, lam) of the rounded (q, g) in long double.  dependent: W holds one
    dependent row (its last), so lam is not unique and only x is compared."""
    n, m, G = P["n"], P["m"], P["G"].astype(LD)
    xs = LD(0.5) * rng.normal(size=n).astype(LD)
    lamW = 10.0 ** rng.uniform(-3, 0, len(W))
    s = 10.0 ** rng.uniform(-3, 0, m)
    s[list(W) + list(weak)] = 0.0
    H = P["H"][hk].astype(LD)
    q = -(H @ xs + G[list(W)].T @ lamW.astype(LD)) if len(W) else -(H @ xs)
    g = -(G @ xs) - s.astype(LD)
    q, g = q.astype(np.float64), g.astype(np.float64)
    Wi = list(W[:-1]) if dependent else list(W)
    x, lamWi = eq_solve(P, hk, Wi, q, g)
    lam = np.zeros(m, dtype=LD)
    lam[Wi] = lamWi
    slack = -g.astype(LD) - P["G"].astype(LD) @ x
    others = np.setdiff1d(np.arange(m), list(W) + list(weak))
    tight = list(W) + list(weak)
    assert slack[others].min() > 5e-4 and (not tight or np.abs(slack[tight]).max() < 1e-10)
    assert dependent or not Wi or lamWi.min() > 5e-4
    return q, g, x.astype(np.float64), lam.astype(np.float64)


# ------------------------------------------------------------------ warm-start reference (gi_warm_start steps (1)-(4))
def ws_reference(P, hk, q, g, ids):
    """The S-pair gi_warm_start leaves from the list ids, and the branches it takes: the panel walk of the blocked QR
    (kk, pa, dep, pad8), the drops and the re-entries of the drop loop when its rotation record is full."""
    n, m, ld = P["n"], P["m"], P["n"] | 1
    Y = P["Y"][hk]
    Zall = -(Y @ P["G"][list(ids)].T.astype(LD))            # d = J'n = -Y G_i' of every listed row
    basis, acc, br, deps = [], [], set(), []
    kk = iq = 0
    while kk < len(ids) and iq < n:
        pw = min(PW, len(ids) - kk)
        pa = dep = 0
        for t in range(pw):
            if iq + t >= n:
                dep = 1
                break
            d = Zall[:, kk + t].copy()
            dd = d @ d
            for _ in range(2):
                for b in basis:
                    d -= (b @ d) * b
            ratio = float((d @ d) / dd)
            assert ratio > 1e-12 or ratio < 1e-26, f"column {kk + t} too close to the dependence threshold ({ratio:.3g})"
            if not ratio > DEP_TOL:
                dep = 1
                break
            basis.append(d / np.sqrt(d @ d))
            acc.append(ids[kk + t])
            pa += 1
        if dep:
            br.add("ws_dep_mid_panel" if 1 <= pa <= pw - 2 else "ws_dep_panel_edge")
            deps.append(("first" if kk == 0 else "last" if kk + pw == len(ids) else "middle", pa))
        if pa and not (kk + PW <= ld and iq + PW <= n):
            br.add("ws_masked_panel")
        iq += pa
        kk += pa + dep
    # (3)/(4): float64 decides the drops (the margins are asserted), long double gives the final S-pair
    A = list(acc)
    nd = nr = ndrops = 0
    while A:
        _, lam = eq_solve(P, hk, A, q, g, np.float64)
        k = int(np.argmin(lam))
        if not lam[k] < 0.0:
            break
        scale = max(1.0, np.abs(lam).max())
        srt = np.sort(lam)
        assert np.abs(lam).min() > 1e-9 * scale, "a multiplier of the warm start too close to zero"
        assert len(lam) == 1 or srt[1] - srt[0] > 1e-8 * scale, "two drop candidates too close"
        ln = len(A) - 1 - k
        if nd >= n // 2 or nr + ln > m // 2:                 # record full: rotations applied, loop re-entered
            br.add("ws_drop_more")
            nd = nr = 0
        nd += 1
        nr += ln
        ndrops += 1
        del A[k]
    if ndrops:
        br.add("ws_drop")
        if not A:
            br.add("ws_all_dropped")
    x, lam = eq_solve(P, hk, A, q, g)
    return dict(act=[int(a) for a in A], x=x.astype(np.float64), lam=lam.astype(np.float64), branches=br, deps=deps)


# ------------------------------------------------------------------ the case table
@functools.lru_cache(maxsize=None)
def cases(n):
    """Every case of size n: kind "known" (reference x, lam; "unique": lam is unique), "infeasible", with an optional
    warm-start list "prev" and, for warm starts, the reference S-pair "ws"."""
    P = problem(n)
    rng = np.random.default_rng(500 + n)
    out = []

    def known(name, hk, W, weak=(), dependent=False, lists=()):
        q, g, x, lam = known_answer(P, hk, W, rng, weak, dependent)
        base = dict(kind="known", hk=hk, q=q, g=g, x=x, lam=lam, W=list(W), unique=not dependent)
        out.append(dict(base, name=name, prev=None))
        for lname, ids in lists:
            out.append(dict(base, name=f"{name}-{lname}", prev=[int(i) for i in ids],
                            ws=ws_reference(P, hk, q, g, ids)))

    for hk in H_KINDS:
        for k in w_sizes(n):
            W = pick_rows(P, k, rng)
            lists = [("final", W)] if k == n else []
            known(f"{hk}-W{k}", hk, W, lists=lists)
    # weakly active rows: tight with lam = 0
    W = pick_rows(P, 12, rng)
    known("weak", "game", W[:9], weak=W[9:])
    # a tight dependent set: bound / bound / rate triple (racing games) or both bounds of one input (merge game)
    if P["rate"]:
        r, j1, j2 = P["rate"][len(P["rate"]) // 2]
        dep = [P["ub"][j1], P["ub"][j2], r]
    else:
        j1 = j2 = n // 2
        dep = [P["ub"][j1], P["lb"][j1]]
    W = pick_rows(P, 7, rng, avoid=(j1, j2))
    known("dependent", "game", W + dep, dependent=True)
    # warm-start lists on one known-answer QP: the final set, permuted, and with one dependent column at every panel
    # column of the first, a middle and the last panel
    kw = PW * ((n - 9 - PW + 1) // PW) + PW - 1              # |W| + 1 fills the last panel
    W = pick_rows(P, kw - len(dep) + 1, rng, avoid=(j1, j2))
    W = dep[:-1] + W                                       # the rows the dependent one depends on come first
    lists = [("final", W), ("perm", list(rng.permutation(W)))]
    mid = (kw + 1) // PW // 2
    for pos in list(range(1, PW)) + list(range(PW * mid, PW * mid + PW)) + list(range(kw + 1 - PW, kw + 1)):
        lists.append((f"dup{pos}", W[:pos] + [W[0]] + W[pos:]))
    for pos in range(PW * mid, PW * mid + PW):
        lists.append((f"dep{pos}", W[:pos] + [dep[-1]] + W[pos:]))
    known("warm", "game", W, lists=lists)
    # a superset whose extra rows must be dropped, a list of n rows of which more than n / 2 drop (the rotation record
    # fills), a list of which every row drops, and the vertex of an SPD Hessian from its n rows
    W = pick_rows(P, n // 4, rng)
    extra = pick_rows(P, n - len(W), rng, avoid=[j for j in range(n) if P["ub"][j] in W or P["lb"][j] in W],
                      dense_max=0)
    sup = list(W) + extra[:len(W)]
    known("drops", "spd1e2", W, lists=[("superset", rng.permutation(sup)), ("full", rng.permutation(list(W) + extra))])
    W0 = pick_rows(P, 3, rng)
    known("empty", "game", [], lists=[("all_drop", [W0[0], W0[0], W0[1]])])
    Wv = pick_rows(P, n, rng)
    known("vertex", "spd1e8", Wv, lists=[("final", Wv), ("perm", rng.permutation(Wv))])
    # infeasible: u_j <= a and u_j >= a + 1
    q, g, _, _ = known_answer(P, "game", [], rng)
    j = n // 3
    g = g.copy()
    g[P["ub"][j]], g[P["lb"][j]] = -0.2, 1.2
    for name, prev in (("infeasible", None), ("infeasible-warm2", [P["ub"][j], P["lb"][j]]),
                       ("infeasible-warm1", [P["lb"][j]])):
        out.append(dict(kind="infeasible", name=name, hk="game", q=q, g=g, prev=prev))
    return out


def warm_cases(n):
    return [c for c in cases(n) if c["prev"] is not None and c["kind"] == "known"]


def arrays(n, cs):
    P = problem(n)
    return (np.array([P["H"][c["hk"]] for c in cs]), np.array([c["q"] for c in cs]), np.array([c["g"] for c in cs]),
            [c["prev"] if c["prev"] is not None else [] for c in cs])


# ------------------------------------------------------------------ errors and checks
def qp_bars(P, c):
    return dict(BARS, du=du_bar(P, c["hk"]))


def qp_errors(P, c, du, lam):
    from oracle.qp import kkt_residuals
    r = kkt_residuals(P["H"][c["hk"]], c["q"], P["G"], c["g"], du, lam)
    return dict(du=rel(du, c["x"]), lam=rel(lam, c["lam"]) if c["unique"] else 0.0, stat=r["stat"], feas=r["feas"],
                comp=r["comp"], dual=r["dual"])


def ws_errors(c, act, xq, lam_act):
    ref = c["ws"]
    same = list(act) == ref["act"]
    return dict(same=same, x=rel(xq, ref["x"]), lam=rel(np.asarray(lam_act), ref["lam"]) if same and len(act) else 0.0)


def tol(host_err, bar, hk):
    """Ten times the host build's error, but not below a hundredth of the bar (a quarter at condition 1e8, where the
    rounding of nvcc's contracted products is amplified): the host build's error on one input can be zero by chance."""
    return min(bar, max(10.0 * host_err, bar / (4.0 if hk == "spd1e8" else 100.0)))


def dual_bar(c):
    """No negative multiplier; a weakly active row (exact multiplier 0) may come out at -1e-12 after the polish."""
    return 1e-12 if c["name"] == "weak" else 0.0


def same_path(c):
    """Cases whose add / drop path is the host build's step for step: margins of at least 1e-3 (no weakly active rows)
    and a Hessian far from singular (at condition 1e8 rounding differences reorder the adds and drops)."""
    return c["name"] != "weak" and c["hk"] != "spd1e8"


@functools.lru_cache(maxsize=None)
def host_run(n, budget):
    """Every case on the host build: (status, du, lam, iterations, active rows) and, for warm-start lists, the S-pair."""
    P = problem(n)
    hs = hostsim(game_of(n), budget_doubles(n, budget))
    hs.evaluate(P["x0"], P["u"], P["l"])
    qp, ws = [], []
    for c in cases(n):
        H = P["H"][c["hk"]]
        qp.append(hs.qp_g(H, c["q"], c["g"], c["prev"]))
        if c["prev"] is not None and c["kind"] == "known":
            ws.append(hs.warm_start(H, c["q"], c["g"], c["prev"]))
    return qp, ws


def check_host(n, budget):
    P = problem(n)
    qp, ws = host_run(n, budget)
    bad = []
    for c, (st, du, lam, it, na) in zip(cases(n), qp):
        if c["kind"] == "infeasible":
            if st != 2:
                bad.append(f"{c['name']}: status {st}")
            continue
        if st != 0:
            bad.append(f"{c['name']}: status {st}")
            continue
        e, bars = qp_errors(P, c, du, lam), qp_bars(P, c)
        bad += [f"{c['name']}: {k} {e[k]:.3g}" for k in BARS if e[k] > bars[k]]
        if e["dual"] > dual_bar(c):
            bad.append(f"{c['name']}: negative multiplier {-e['dual']:.3g}")
        if c["prev"] is not None and sorted(c["ws"]["act"]) == sorted(c["W"]) and it != 0:
            bad.append(f"{c['name']}: {it} main-loop iterations from the final active set")
    for c, (act, xq, lam_act) in zip(warm_cases(n), ws):
        e = ws_errors(c, act, xq, lam_act)
        if not e["same"]:
            bad.append(f"{c['name']}: warm start kept {len(act)} rows, the reference {len(c['ws']['act'])}")
        elif e["x"] > du_bar(P, c["hk"]) or e["lam"] > BARS["lam"]:
            bad.append(f"{c['name']}: warm start x {e['x']:.3g} lam {e['lam']:.3g}")
    assert not bad, f"{len(bad)} failures: " + "; ".join(bad[:20])


# ------------------------------------------------------------------ branches
def qp_cells():
    for n in QP_SIZES:
        for threads in WIDTHS[n]:
            for budget in BUDGETS:
                if budget_doubles(n, budget) is not None:
                    yield n, threads, budget


def cell_id(c):
    return f"n{c[0]}-{SIZES[c[0]][0]}-t{c[1]}-{c[2]}"


REQUIRED = {"ws_dep_mid_panel", "ws_dep_panel_edge", "ws_masked_panel", "ws_drop", "ws_drop_more", "ws_all_dropped",
            "gi_partial_step", "gi_dependent_drop_step", "gi_infeasible", "vertex",
            "width32", "width96", "width128", "width256", "placement_smem", "placement_split", "placement_global"}


def test_case_table_reaches_every_branch():
    """The table reaches every branch of the warm start and the main loop listed in REQUIRED, at every width and
    placement; a dependent column sits at every panel column of a first (after column 0), a middle and a last panel.
    The main-loop branches are read from the oracle's cold solve, which takes the kernel's path step for step."""
    from oracle.qp import QPFailure, solve_qp_gi
    reached, deps = set(), set()
    for n in QP_SIZES:
        P = problem(n)
        for c in cases(n):
            if c["kind"] == "infeasible":
                reached.add("gi_infeasible")
                continue
            if c["prev"] is not None:
                reached |= c["ws"]["branches"]
                deps |= {(kind, pa) for kind, pa in c["ws"]["deps"]}
                continue
            if len(c["W"]) == n:
                reached.add("vertex")
            stats = {}
            solve_qp_gi(P["H"][c["hk"]], c["q"], P["G"], c["g"], stats=stats)
            if stats["n_drop"] > stats["n_drop_dep"]:
                reached.add("gi_partial_step")
            if stats["n_drop_dep"]:
                reached.add("gi_dependent_drop_step")
    for n, threads, budget in qp_cells():
        reached |= {f"width{threads}", "placement_" + placement(host_plan(n, budget))}
    assert not REQUIRED - reached, f"not reached: {sorted(REQUIRED - reached)}"
    want = {("first", pa) for pa in range(1, PW)} | {(k, pa) for k in ("middle", "last") for pa in range(PW)}
    assert not want - deps, f"dependent columns not placed: {sorted(want - deps)}"
    with pytest.raises(QPFailure, match="infeasible"):
        c = [c for c in cases(QP_SIZES[0]) if c["kind"] == "infeasible"][0]
        P = problem(QP_SIZES[0])
        solve_qp_gi(P["H"][c["hk"]], c["q"], P["G"], c["g"])


# ================================================================== host build (CPU)
@pytest.mark.parametrize("n", QP_SIZES)
def test_oracle_infeasible(n):
    """The oracle refuses the infeasible cases as the kernel does (status 2)."""
    from oracle.qp import QPFailure, solve_qp_gi
    P = problem(n)
    for c in cases(n):
        if c["kind"] == "infeasible" and c["prev"] is None:
            with pytest.raises(QPFailure, match="infeasible"):
                solve_qp_gi(P["H"][c["hk"]], c["q"], P["G"], c["g"])


@pytest.mark.parametrize("n,budget", [(n, b) for n in QP_SIZES for b in ("smem", "global")], ids=str)
def test_host_qp(n, budget):
    check_host(n, budget)


# ================================================================== CUDA kernels (B200)
@pytest.mark.gpu
@pytest.mark.parametrize("cell", list(qp_cells()), ids=cell_id)
def test_gpu_qp(cell):
    import gpu_units_lib as U
    n, threads, budget = cell
    game, P = game_of(n), problem(n)
    lim = budget_doubles(n, budget)
    cs, wcs = cases(n), warm_cases(n)
    hqp, hws = host_run(n, "smem")
    rep = lambda v, B: np.repeat(v[None], B, axis=0)
    H, q, g, prev = arrays(n, cs)
    B = len(cs)
    out = U.qp(game, params_of(game), rep(P["x0"], B), rep(P["u"], B), rep(P["l"], B), H, q, g=g, prev=prev,
               threads=threads, smem_limit_doubles=lim)
    H, q, g, prev = arrays(n, wcs)
    Bw = len(wcs)
    ws = U.warm_start(game, params_of(game), rep(P["x0"], Bw), rep(P["u"], Bw), rep(P["l"], Bw), H, q, g, prev,
                      threads=threads, smem_limit_doubles=lim)
    assert out["plan"] == ws["plan"] == host_plan(n, budget)
    bad = []
    for i, (c, (hst, hdu, hlam, hit, hna)) in enumerate(zip(cs, hqp)):
        st, it, na = int(out["st"][i]), int(out["it"][i]), int(out["na"][i])
        if st != hst:
            bad.append(f"{c['name']}: status {st}, host {hst}")
            continue
        if c["kind"] == "infeasible":
            continue
        if same_path(c) and (na != hna or it != hit):
            bad.append(f"{c['name']}: {na} active rows in {it} iterations, host {hna} in {hit}")
        e, eh, bars = qp_errors(P, c, out["du"][i], out["lam"][i]), qp_errors(P, c, hdu, hlam), qp_bars(P, c)
        bad += [f"{c['name']}: {k} {e[k]:.3g} (host {eh[k]:.3g})" for k in BARS if e[k] > tol(eh[k], bars[k], c["hk"])]
        if e["dual"] > dual_bar(c):
            bad.append(f"{c['name']}: negative multiplier {-e['dual']:.3g}")
    for i, (c, h) in enumerate(zip(wcs, hws)):
        if list(ws["act"][i]) != list(h[0]):
            bad.append(f"{c['name']}: warm start kept {list(ws['act'][i])}, host {list(h[0])}")
            continue
        e, eh = ws_errors(c, ws["act"][i], ws["xq"][i], ws["lam_act"][i]), ws_errors(c, *h)
        if e["x"] > tol(eh["x"], du_bar(P, c["hk"]), c["hk"]) or e["lam"] > tol(eh["lam"], BARS["lam"], c["hk"]):
            bad.append(f"{c['name']}: warm start x {e['x']:.3g} lam {e['lam']:.3g} (host {eh['x']:.3g} {eh['lam']:.3g})")
    assert not bad, f"{len(bad)} failures: " + "; ".join(bad[:20])
