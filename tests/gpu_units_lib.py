"""ctypes loader of the stage-level test kernel (tests/gpu_units/units.cu), built once per game: racing games and the
merge game (-DDG_GAME_MERGE).  TEST ONLY.

Every entry point runs a batch with one CTA per instance at the given CTA width and shared-memory budget
(``smem_limit_doubles``: None = the device maximum, otherwise that many doubles) and returns the memory plan it ran with
as ``out["plan"]`` (see PLAN_KEYS)."""
import ctypes as C
import os
import pathlib
import subprocess

import numpy as np

from dgsqp_b200.games import params_to_struct, MergeGame

HERE = pathlib.Path(__file__).resolve().parent / "gpu_units"
NVCC = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-shared",
        "-Xcompiler", "-fPIC"]
PLAN_KEYS = ("hot_in_smem", "mats_in_smem", "matA_in_smem", "sens_in_smem", "eig_s")
_libs = {}


def _out(merge):
    return HERE / ("libdgsqp_units_merge.so" if merge else "libdgsqp_units.so")


def build():
    """Builds the racing and the merge library side by side (each is one nvcc run of about a minute)."""
    srcs = [HERE / "units.cu"] + sorted((HERE.parents[1] / "dgsqp_b200" / "csrc").glob("*.cuh")) \
        + sorted((HERE.parents[1] / "dgsqp_b200" / "csrc").glob("*.h"))
    procs = []
    for merge in (False, True):
        out = _out(merge)
        if out.exists() and all(out.stat().st_mtime >= s.stat().st_mtime for s in srcs):
            continue
        cmd = [*NVCC, *(["-DDG_GAME_MERGE=1"] if merge else []), "-o", str(out), str(HERE / "units.cu")]
        procs.append((cmd, subprocess.Popen(cmd)))
    for cmd, p in procs:
        if p.wait() != 0:
            raise subprocess.CalledProcessError(p.returncode, cmd)
    return _out(False), _out(True)


def _lib(merge):
    if merge not in _libs:
        env = os.environ.get("DG_UNITS_MERGE_LIB" if merge else "DG_UNITS_LIB")
        if not env:
            build()
        _libs[merge] = C.CDLL(env or str(_out(merge)))
    return _libs[merge]


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f64(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


def _call(name, game, params, threads, smem_limit_doubles, *args):
    lib = _lib(isinstance(game, MergeGame))
    gs, ps = game.to_struct(), params_to_struct(params)
    plan = np.zeros(len(PLAN_KEYS), np.int32)
    lim = -1 if smem_limit_doubles is None else int(smem_limit_doubles)
    rc = getattr(lib, name)(C.byref(gs), C.byref(ps), *args[:1], C.c_int(threads), C.c_long(lim), *args[1:], _p(plan))
    assert rc == 0, f"{name} failed: {rc}"
    return dict(zip(PLAN_KEYS, (int(v) for v in plan)))


def run_stages(game, params, x0, u, l, threads=128, smem_limit_doubles=None):
    """evaluate -> nearestPD -> QP at (u, l), and the LSQR dual initialisation at u, for a batch."""
    B, n, m = x0.shape[0], game.n, game.m
    x0, u, l = (_f64(a) for a in (x0, u, l))
    out = dict(Q=np.zeros((B, n, n)), H=np.zeros((B, n, n)), q=np.zeros((B, n)), gtl=np.zeros((B, n)),
               du=np.zeros((B, n)), g=np.zeros((B, m)), lam=np.zeros((B, m)), l0=np.zeros((B, m)),
               nneg=np.zeros(B, np.int32), qpst=np.zeros(B, np.int32), qpit=np.zeros(B, np.int32),
               lsqr_it=np.zeros(B, np.int32))
    out["plan"] = _call("units_run", game, params, threads, smem_limit_doubles, C.c_int(B), _p(x0), _p(u), _p(l),
                        *(_p(out[k]) for k in ("Q", "q", "gtl", "g", "H", "du", "lam", "l0", "nneg", "qpst", "qpit",
                                               "lsqr_it")))
    return out


def nearest_pd(game, params, Q, threads=256, smem_limit_doubles=None):
    """H = nearestPD(Q) + reg I and the number of negative eigenvalues, for Q[B, n, n]."""
    Q = _f64(Q)
    B = Q.shape[0]
    out = dict(H=np.zeros_like(Q), nneg=np.zeros(B, np.int32))
    out["plan"] = _call("units_nearest_pd", game, params, threads, smem_limit_doubles, C.c_int(B), _p(Q), _p(out["H"]),
                        _p(out["nneg"]))
    return out


def factor(game, params, H, q, threads=256, smem_limit_doubles=None):
    """qp_factor: ok, L (lower), Y = L^-1 (every stored entry), xq = -H^-1 q."""
    H, q = _f64(H), _f64(q)
    B, n = q.shape
    out = dict(ok=np.zeros(B, np.int32), L=np.zeros((B, n, n)), Y=np.zeros((B, n, n)), xq=np.zeros((B, n)))
    out["plan"] = _call("units_factor", game, params, threads, smem_limit_doubles, C.c_int(B), _p(H), _p(q),
                        *(_p(out[k]) for k in ("ok", "L", "Y", "xq")))
    return out


def _warm_lists(prev, B):
    """A list of B warm-start lists (id sequences) as the padded array prev[B, kmax] and the counts kprev[B]."""
    if prev is None:
        return None, None, 0
    assert len(prev) == B
    kmax = max(1, max(len(p) for p in prev))
    arr, cnt = np.zeros((B, kmax), np.int32), np.array([len(p) for p in prev], np.int32)
    for b, p in enumerate(prev):
        arr[b, :len(p)] = p
    return arr, cnt, kmax


def qp(game, params, x0, u, l, H, q, q2=None, g=None, prev=None, threads=256, smem_limit_doubles=None):
    """Evaluation at (x0, u, l), a QP at (H, q) on its constraints -- with the offsets g[B, m] in place of the evaluated
    ones if given; cold, or from the warm-start lists prev (B id sequences) if given -- and, with q2, a warm QP at
    (H, q2) from the first QP's active set.  it / na: main-loop iterations and active rows at the end."""
    x0, u, l, H, q, q2, g = (_f64(a) for a in (x0, u, l, H, q, q2, g))
    B, n, m = x0.shape[0], game.n, game.m
    pv, kp, kmax = _warm_lists(prev, B)
    out = dict(Q=np.zeros((B, n, n)), q=np.zeros((B, n)), gtl=np.zeros((B, n)), g=np.zeros((B, m)),
               st=np.zeros(B, np.int32), it=np.zeros(B, np.int32), na=np.zeros(B, np.int32), du=np.zeros((B, n)),
               lam=np.zeros((B, m)), st2=np.zeros(B, np.int32), it2=np.zeros(B, np.int32), na2=np.zeros(B, np.int32),
               du2=np.zeros((B, n)), lam2=np.zeros((B, m)))
    out["plan"] = _call("units_qp", game, params, threads, smem_limit_doubles, C.c_int(B), _p(x0), _p(u), _p(l), _p(H),
                        _p(q), _p(q2), _p(g), _p(pv), _p(kp), C.c_int(kmax),
                        *(_p(out[k]) for k in ("Q", "q", "gtl", "g", "st", "it", "na", "du", "lam", "st2", "it2", "na2",
                                               "du2", "lam2")))
    return out


def warm_start(game, params, x0, u, l, H, q, g, prev, threads=256, smem_limit_doubles=None):
    """Evaluation at (x0, u, l) (offsets g[B, m] in place of the evaluated ones if given), qp_factor of H and
    gi_warm_start from the lists prev: per instance the S-pair the main loop would start from, as "act" (list of ids),
    "xq" and "lam_act" (array of len(act))."""
    x0, u, l, H, q, g = (_f64(a) for a in (x0, u, l, H, q, g))
    B, n = x0.shape[0], game.n
    pv, kp, kmax = _warm_lists(prev, B)
    iq, act, xq, lam = np.zeros(B, np.int32), np.zeros((B, n), np.int32), np.zeros((B, n)), np.zeros((B, n))
    plan = _call("units_warm", game, params, threads, smem_limit_doubles, C.c_int(B), _p(x0), _p(u), _p(l), _p(H), _p(q),
                 _p(g), _p(pv), _p(kp), C.c_int(kmax), _p(iq), _p(act), _p(xq), _p(lam))
    assert (iq >= 0).all(), "units_warm: H not positive definite"
    return dict(act=[act[b, :iq[b]].copy() for b in range(B)], xq=xq,
                lam_act=[lam[b, :iq[b]].copy() for b in range(B)], plan=plan)


def G_products(game, params, x0, u, l, v, w, rows, threads=256, smem_limit_doubles=None):
    """Evaluation at (x0, u, l); G v, G' w, and rows[B, k] of G by game_G_row ("rows") and by game_G_cols ("cols")."""
    x0, u, l, v, w = (_f64(a) for a in (x0, u, l, v, w))
    rows = np.ascontiguousarray(rows, dtype=np.int32)
    B, n, m = x0.shape[0], game.n, game.m
    k = rows.shape[1]
    out = dict(Q=np.zeros((B, n, n)), q=np.zeros((B, n)), gtl=np.zeros((B, n)), g=np.zeros((B, m)),
               Gv=np.zeros((B, m)), GTw=np.zeros((B, n)), rows=np.zeros((B, k, n)), cols=np.zeros((B, k, n)))
    out["plan"] = _call("units_G", game, params, threads, smem_limit_doubles, C.c_int(B), _p(x0), _p(u), _p(l), _p(v),
                        _p(w), _p(rows), C.c_int(k), *(_p(out[k2]) for k2 in ("Q", "q", "gtl", "g", "Gv", "GTw", "rows",
                                                                             "cols")))
    return out
