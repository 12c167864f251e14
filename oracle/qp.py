"""Exact dense QP solver for the SQP sub-problem.  Oracle-only.

The reference hands  min 1/2 du'H du + q'du  s.t.  G du <= -g  to OSQP through
CasADi's ``conic`` (``DGSQP/solvers/DGSQP.py:246-249``, ``polish=True``).  When
OSQP's polish succeeds the answer is the exact KKT point of a strictly convex
QP and therefore solver independent; this module computes that point with the
Goldfarb-Idnani dual active-set method (Math. Prog. 27, 1983) restated from the
paper: start at the unconstrained minimiser, add the most violated constraint,
take partial (drop a blocking active constraint) or full (add it) steps.

Conventions: s_i(x) = -g_i - G_i x >= 0, normal n_i = -G_i^T, multipliers lam >= 0 with
H x + q + G^T lam = 0.
"""
import numpy as np
import scipy.linalg as sla

FEAS_TOL = 1e-10
DEP_TOL = 1e-20        # |d2|^2 <= DEP_TOL*|d|^2  ->  normal linearly dependent on the active set


class QPFailure(Exception):
    pass


def solve_qp_gi(H, q, G, g, max_iter=None, feas_tol=FEAS_TOL, stats=None, polish=True):
    n, m = H.shape[0], G.shape[0]
    if max_iter is None:
        max_iter = 10 * (n + m)
    try:
        L = np.linalg.cholesky(H)
    except np.linalg.LinAlgError as e:
        raise QPFailure("H not positive definite") from e
    J = sla.solve_triangular(L, np.eye(n), lower=True).T        # J J^T = H^-1
    x = -sla.cho_solve((L, True), q)
    R = np.zeros((n, n))
    act = []                                                    # active constraint ids
    lam_act = np.zeros(0)
    iq = 0
    it = 0
    n_add = n_drop = n_drop_dep = 0
    while True:
        s = -g - G @ x
        if iq:
            s[act] = 0.0                                        # active rows sit on their boundary
        p = int(np.argmin(s))
        if s[p] >= -feas_tol:
            break
        npv = -G[p]
        lam_p = 0.0
        while True:
            it += 1
            if it > max_iter:
                raise QPFailure("iteration limit")
            d = J.T @ npv
            z = J[:, iq:] @ d[iq:]
            r = sla.solve_triangular(R[:iq, :iq], d[:iq], lower=False) if iq else np.zeros(0)
            # largest dual step keeping lam_act >= 0
            t1, ldrop = np.inf, -1
            for k in range(iq):
                if r[k] > 0.0:
                    tk = lam_act[k] / r[k]
                    if tk < t1:
                        t1, ldrop = tk, k
            # z'n = |d2|^2 (J2'n = d2): the normal is independent of the active ones iff d2 != 0
            zn = d[iq:] @ d[iq:]
            if zn > DEP_TOL * (d @ d) and zn > 0.0:
                sp = -g[p] - G[p] @ x
                t2 = -sp / zn
            else:
                t2 = np.inf
            t = min(t1, t2)
            if not np.isfinite(t):
                raise QPFailure("infeasible")
            if np.isfinite(t2):
                x = x + t * z
            lam_act = lam_act - t * r
            lam_p += t
            if t2 <= t1:
                # full step: constraint p becomes active.  Householder on d[iq:] keeps J's
                # trailing columns an H-orthonormal basis of the active-normal null space.
                dd = d[iq:].copy()
                alpha = np.linalg.norm(dd)
                if dd[0] > 0:
                    alpha = -alpha
                v = dd
                v[0] -= alpha
                vv = v @ v
                if vv > 0.0:
                    w = J[:, iq:] @ v
                    J[:, iq:] -= np.outer(w, (2.0 / vv) * v)
                R[:iq, iq] = d[:iq]
                R[iq, iq] = alpha
                act.append(p)
                lam_act = np.append(lam_act, lam_p)
                iq += 1
                n_add += 1
                break
            # partial step: drop blocking constraint ldrop, keep working on p
            for j in range(ldrop, iq - 1):
                R[:, j] = R[:, j + 1]
            R[:, iq - 1] = 0.0
            for j in range(ldrop, iq - 1):
                a, b = R[j, j], R[j + 1, j]
                h = np.hypot(a, b)
                if h == 0.0:
                    continue
                c, sn = a / h, b / h
                Rj, Rj1 = R[j, j:iq].copy(), R[j + 1, j:iq].copy()
                R[j, j:iq] = c * Rj + sn * Rj1
                R[j + 1, j:iq] = -sn * Rj + c * Rj1
                Jj, Jj1 = J[:, j].copy(), J[:, j + 1].copy()
                J[:, j] = c * Jj + sn * Jj1
                J[:, j + 1] = -sn * Jj + c * Jj1
            del act[ldrop]
            lam_act = np.delete(lam_act, ldrop)
            iq -= 1
            n_drop += 1
            n_drop_dep += not np.isfinite(t2)           # p dependent on the active set: a pure dual step
    # Polish.  The iteration starts at the unconstrained minimiser x0 = -H^-1 q and moves by x += t z; for an
    # ill-conditioned H (reg = 0 games: eigenvalues at the 1e-10 floor) x0 is ~1e10 |q| along the near-null directions and
    # the steps cancel it, leaving errors of 1e-5..1e-3 in x and 1e-2 in lam.  The KKT point of the final active set W is
    # therefore re-evaluated from the final factors in a form where the large terms never meet: with J = [J1 J2],
    # J'N_W = [R; 0] and c = J'q,   x = J1 R^-T g_W - J2 c2,   lam_W = R^-1 (R^-T g_W + c1)   (1e-10 / 1e-8 against an
    # extended-precision KKT solve).  It is the role OSQP's polish (reduced KKT system of the active set + iterative
    # refinement) plays in the reference (DGSQP.py:186, polish=True); the CUDA path applies the same formula (gi_polish).
    if polish:
        c = J.T @ q
        if iq:
            tp = sla.solve_triangular(R[:iq, :iq], g[act], trans="T", lower=False)
            x = J[:, :iq] @ tp - J[:, iq:] @ c[iq:]
            lam_act = sla.solve_triangular(R[:iq, :iq], tp + c[:iq], lower=False)
        else:
            x = -J @ c
    lam = np.zeros(m)
    if iq:
        lam[act] = lam_act
    if stats is not None:
        stats.update(iters=it, n_add=n_add, n_drop=n_drop, n_drop_dep=n_drop_dep, n_active=iq)
    return x, lam


def kkt_residuals(H, q, G, g, x, lam):
    """Necessary and sufficient optimality conditions of the strictly convex QP."""
    r_stat = np.abs(H @ x + q + G.T @ lam).max()
    c = G @ x + g
    return dict(stat=r_stat, feas=max(0.0, c.max()), dual=max(0.0, -lam.min()),
                comp=np.abs(lam * c).max())
