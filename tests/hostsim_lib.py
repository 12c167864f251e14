"""Builds and loads the single-thread host build of the kernel source (tests/hostsim/hostsim.cpp).
TEST HARNESS ONLY -- the product never loads this."""
import ctypes as C
import pathlib
import subprocess

import numpy as np

from dgsqp_b200._abi import RacingGameStruct, MergeGameStruct, ParamsStruct, ParamsV2Struct
from dgsqp_b200.games import params_to_struct, params_v2_to_struct, MergeGame
from dgsqp_b200.solver_types import DGSQPV2Params

HERE = pathlib.Path(__file__).resolve().parent / "hostsim"
_libs = {}


def build(asan=False, merge=False, guard=False, fma=False):
    out = HERE / ("libhostsim" + ("_merge" if merge else "") + ("_asan" if asan else "") + ("_guard" if guard else "")
                  + ("_fma" if fma else "") + ".so")
    srcs = [HERE / "hostsim.cpp"] + sorted((HERE.parents[1] / "dgsqp_b200" / "csrc").glob("*.cuh")) \
        + sorted((HERE.parents[1] / "dgsqp_b200" / "csrc").glob("*.h"))
    if out.exists() and all(out.stat().st_mtime >= s.stat().st_mtime for s in srcs):
        return out
    flags = ["-O1", "-g", "-fsanitize=address,undefined", "-fno-omit-frame-pointer"] if asan else ["-O2"]
    if merge:
        flags = flags + ["-DDG_GAME_MERGE=1"]
    if guard:
        flags = flags + ["-DDG_PLAN_GUARD=16"]      # canary gaps behind every buffer of the memory plan (hs_guard_check)
    if fma:
        flags = flags + ["-mfma", "-ffp-contract=fast"]   # products contracted into FMAs wherever the compiler likes, as nvcc does
    subprocess.check_call(["g++", *flags, "-shared", "-fPIC", "-std=c++17", "-o", str(out), str(HERE / "hostsim.cpp")])
    return out


def load(asan=False, merge=False, guard=False, fma=False):
    if (asan, merge, guard, fma) in _libs:
        return _libs[(asan, merge, guard, fma)]
    lib = C.CDLL(str(build(asan, merge, guard, fma)))
    gs = MergeGameStruct if merge else RacingGameStruct
    lib.hs_create.restype = C.c_void_p
    lib.hs_create.argtypes = [C.POINTER(gs), C.POINTER(ParamsStruct)]
    lib.hs_create_v2.restype = C.c_void_p
    lib.hs_create_v2.argtypes = [C.POINTER(gs), C.POINTER(ParamsV2Struct)]
    for name in ["hs_destroy", "hs_dims", "hs_evaluate", "hs_G_dense", "hs_G_times", "hs_GT_times", "hs_nearest_pd",
                 "hs_qp", "hs_qp_warm", "hs_qp_g", "hs_warm_start", "hs_factor", "hs_plan", "hs_lsqr", "hs_solve"]:
        getattr(lib, name).argtypes = None
    lib.hs_nearest_pd.restype = C.c_int
    lib.hs_qp.restype = C.c_int
    lib.hs_qp_warm.restype = C.c_int
    lib.hs_qp_g.restype = C.c_int
    lib.hs_warm_start.restype = C.c_int
    lib.hs_factor.restype = C.c_int
    lib.hs_lsqr.restype = C.c_int
    lib.hs_guard_check.restype = C.c_int
    lib.hs_guard_check.argtypes = [C.c_void_p]
    _libs[(asan, merge, guard, fma)] = lib
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class HostSim:
    def __init__(self, game, params, asan=False, guard=False, qp_warm=True, mu_vio_thresh=1e-10, fma=False):
        self.lib = load(asan, merge=isinstance(game, MergeGame), guard=guard, fma=fma)
        self.game = game
        gs = game.to_struct()
        if isinstance(params, DGSQPV2Params):
            ps = params_v2_to_struct(params, mu_vio_thresh=mu_vio_thresh, qp_warm_start=qp_warm)
            self.h = C.c_void_p(self.lib.hs_create_v2(C.byref(gs), C.byref(ps)))
        else:
            ps = params_to_struct(params, mu_vio_thresh=mu_vio_thresh, qp_warm_start=qp_warm)
            self.h = C.c_void_p(self.lib.hs_create(C.byref(gs), C.byref(ps)))
        assert self.h.value, "hs_create failed"
        dims = np.zeros(4, dtype=np.int32)
        self.lib.hs_dims(self.h, _p(dims))
        self.nq, self.nu, self.n, self.m = (int(v) for v in dims)

    def __del__(self):
        if getattr(self, "h", None) is not None and self.h.value:
            self.lib.hs_destroy(self.h)
            self.h = None

    def guard_check(self):
        """Guard build only: number of damaged canary doubles behind the buffers of the memory plan (0 = no overrun)."""
        return int(self.lib.hs_guard_check(self.h))

    def evaluate(self, x0, u, l):
        n, m = self.n, self.m
        Q, q, gtl, g = np.zeros((n, n)), np.zeros(n), np.zeros(n), np.zeros(m)
        x = np.zeros((self.game.N + 1, self.nq))
        x0, u, l = (np.ascontiguousarray(v, dtype=np.float64) for v in (x0, u, l))
        self.lib.hs_evaluate(self.h, _p(x0), _p(u), _p(l), _p(Q), _p(q), _p(gtl), _p(g), _p(x))
        return Q, q, gtl, g, x

    def G_dense(self):
        G = np.zeros((self.m, self.n))
        self.lib.hs_G_dense(self.h, _p(G))
        return G

    def G_times(self, v):
        y = np.zeros(self.m)
        v = np.ascontiguousarray(v, dtype=np.float64)
        self.lib.hs_G_times(self.h, _p(v), _p(y))
        return y

    def GT_times(self, w):
        y = np.zeros(self.n)
        w = np.ascontiguousarray(w, dtype=np.float64)
        self.lib.hs_GT_times(self.h, _p(w), _p(y))
        return y

    def nearest_pd(self, Q):
        H = np.zeros_like(Q)
        Q = np.ascontiguousarray(Q, dtype=np.float64)
        nneg = self.lib.hs_nearest_pd(self.h, _p(Q), _p(H))
        return H, nneg

    def qp(self, H, q):
        H = np.ascontiguousarray(H, dtype=np.float64).copy()
        q = np.ascontiguousarray(q, dtype=np.float64)
        du, lam = np.zeros(self.n), np.zeros(self.m)
        it = C.c_int(0)
        st = self.lib.hs_qp(self.h, _p(H), _p(q), _p(du), _p(lam), C.byref(it))
        return st, du, lam, it.value

    def qp_warm(self, H, q):
        """QP at (H, q) started from the active set of the previous QP of this handle (gi_warm_start)."""
        H = np.ascontiguousarray(H, dtype=np.float64).copy()
        q = np.ascontiguousarray(q, dtype=np.float64)
        du, lam = np.zeros(self.n), np.zeros(self.m)
        it = C.c_int(0)
        st = self.lib.hs_qp_warm(self.h, _p(H), _p(q), _p(du), _p(lam), C.byref(it))
        return st, du, lam, it.value

    def qp_g(self, H, q, g=None, prev=None):
        """QP at (H, q) on the evaluated constraints with the offsets g in their place (if given), from the warm-start
        list prev (gi_warm_start) if given, cold otherwise: (status, du, lam, main-loop iterations, active rows)."""
        H, q, g = (None if a is None else np.ascontiguousarray(a, dtype=np.float64) for a in (H, q, g))
        prev = np.ascontiguousarray([] if prev is None else prev, dtype=np.int32)
        du, lam, out = np.zeros(self.n), np.zeros(self.m), np.zeros(3, dtype=np.int32)
        rc = self.lib.hs_qp_g(self.h, _p(H), _p(q), None if g is None else _p(g), _p(prev), C.c_int(len(prev)), _p(du),
                              _p(lam), _p(out))
        assert rc == 0, "hs_qp_g: bad warm-start list"
        return int(out[0]), du, lam, int(out[1]), int(out[2])

    def warm_start(self, H, q, g, prev):
        """qp_factor and gi_warm_start only: the S-pair (act, xq, lam_act) the main loop would start from."""
        H, q, g = (None if a is None else np.ascontiguousarray(a, dtype=np.float64) for a in (H, q, g))
        prev = np.ascontiguousarray(prev, dtype=np.int32)
        act, xq, lam_act = np.zeros(self.n, dtype=np.int32), np.zeros(self.n), np.zeros(self.n)
        iq = self.lib.hs_warm_start(self.h, _p(H), _p(q), None if g is None else _p(g), _p(prev), C.c_int(len(prev)),
                                    _p(act), _p(xq), _p(lam_act))
        assert iq >= 0, f"hs_warm_start failed: {iq}"
        return act[:iq].copy(), xq, lam_act[:iq].copy()

    def factor(self, H, q):
        """qp_factor: (ok, L, Y = L^-1 as stored, xq = -H^-1 q)."""
        H = np.ascontiguousarray(H, dtype=np.float64)
        q = np.ascontiguousarray(q, dtype=np.float64)
        L, Y, xq = np.zeros((self.n, self.n)), np.zeros((self.n, self.n)), np.zeros(self.n)
        ok = self.lib.hs_factor(self.h, _p(H), _p(q), _p(L), _p(Y), _p(xq))
        return bool(ok), L, Y, xq

    def plan(self):
        """Memory plan: (hot_in_smem, mats_in_smem, matA_in_smem, sens_in_smem, eig_s set)."""
        out = np.zeros(5, dtype=np.int32)
        self.lib.hs_plan(self.h, _p(out))
        return tuple(int(v) for v in out)

    def lsqr(self, x0, u):
        l = np.zeros(self.m)
        x0, u = (np.ascontiguousarray(v, dtype=np.float64) for v in (x0, u))
        itn = self.lib.hs_lsqr(self.h, _p(x0), _p(u), _p(l))
        return l, itn

    def solve(self, x0, u_ws, l_ws=None, u_prev=None):
        n, m = self.n, self.m
        x0, u_ws = (np.ascontiguousarray(v, dtype=np.float64) for v in (x0, u_ws))
        u, l, x = np.zeros(n), np.zeros(m), np.zeros((self.game.N + 1, self.nq))
        cost, cond = np.zeros(self.game.M), np.zeros(3)
        it, st, qp = C.c_int(0), C.c_int(0), C.c_int(0)
        diag = np.zeros(8, dtype=np.int32)
        l_init = np.zeros(m)
        if l_ws is not None:
            l_ws = np.ascontiguousarray(l_ws, dtype=np.float64)
        if u_prev is not None:
            u_prev = np.ascontiguousarray(u_prev, dtype=np.float64)
        self.lib.hs_solve(self.h, _p(x0), _p(u_ws), _p(l_ws) if l_ws is not None else None,
                          _p(u_prev) if u_prev is not None else None, _p(u), _p(l), _p(x), _p(cost), _p(cond), C.byref(it),
                          C.byref(st), C.byref(qp), _p(diag), _p(l_init))
        return dict(u=u, l=l, x=x, cost=cost, cond=cond, num_iters=it.value, status=st.value, qp_solves=qp.value,
                    diag=diag, l_init=l_init)
