"""Batched Monte-Carlo instance generation (host side, vectorised over instances).

Instance distributions and the PID warm start follow the reference drivers
(``scripts/DGSQP_ALGAMES_monte_carlo_chicane.py:384-467`` for the 2-agent head-to-head games,
``scripts/DGSQP_monte_carlo_agents.py:257-308`` for M independent agents; controllers
``DGSQP/solvers/PID.py:74-138,187-238``).  Differences, both irrelevant to the solve path:

* the one-step simulation inside the PID roll-out uses classical RK4 with 4 sub-steps instead of
  SciPy's adaptive RK45 (``dynamics_models.py:161-186``) so that it vectorises;
* rejection sampling is done on whole batches, so the random stream is consumed in a different
  order than the sequential script (the reference scripts for these games are unseeded anyway).

``sample_merge`` follows ``scripts/DGSQP_merge_monte_carlo.py:424-495`` (seeded, ``default_rng(1)``) and consumes
the random stream in exactly the script's order (12 draws per trial, rejected trials included).

``sample_head_to_head_cuda``, ``sample_agents_cuda`` and ``sample_merge_cuda`` draw the same distributions on the GPU
(``dgsqp_sample_racing`` / ``dgsqp_sample_merge``, csrc/mc_sampler.cuh) and return CUDA tensors that
``DGSQP.solve_batch`` takes on its device path.  They read ``default_rng(seed)``'s stream trial-major: trial t consumes a
fixed block of draws (head-to-head 5, M agents 3M, merge 12) and instance i is the i-th accepted trial, so the result
does not depend on B beyond its length.  For merge that is the order of ``sample_merge``, which the device sampler
reproduces instance for instance; the host racing samplers above draw batch-sized blocks per quantity, so for the same
seed they return other instances of the same distribution.
"""
import numpy as np

from .games import RacingGame, MergeGame, NQA, NUA


def _track_lookup(track, s):
    L = track.track_length
    sb = np.fmod(np.fmod(s, L) + L, L)
    kp = track.key_pts
    idx = np.clip(np.searchsorted(kp[1:-1, 3], sb, side="right"), 0, kp.shape[0] - 2)
    curv = kp[1:, 5][idx]
    cum_ang = np.concatenate([[0.0], np.cumsum(kp[1:, 4] * kp[1:, 5])])
    psit = cum_ang[idx] + curv * (sb - kp[idx, 3])
    return curv, psit


def _fc(game: RacingGame, q, u):
    """Continuous kinematic-bicycle dynamics, q [B,6], u [B,2] (dynamics_models.py:1046-1070)."""
    v, epsi, s, ey = q[:, 2], q[:, 3], q[:, 4], q[:, 5]
    a, delta = u[:, 0], u[:, 1]
    beta = np.arctan2(np.tan(delta) * game.L_r, game.L_f + game.L_r)
    psidot = v / game.L_r * np.sin(beta)
    F = -game.c_da * v - game.c_dr * v * np.abs(v) - game.c_s * psidot ** 2
    kap, psit = _track_lookup(game.track, s)
    den = 1.0 - ey * kap
    cb = np.cos(beta + epsi)
    return np.stack([v * np.cos(beta + psit + epsi), v * np.sin(beta + psit + epsi), a + F / game.mass,
                     psidot - kap * v * cb / den, v * cb / den, v * np.sin(beta + epsi)], axis=1)


def _rk4(game, q, u, dt, substeps=4):
    h = dt / substeps
    for _ in range(substeps):
        k1 = _fc(game, q, u)
        k2 = _fc(game, q + 0.5 * h * k1, u)
        k3 = _fc(game, q + 0.5 * h * k2, u)
        k4 = _fc(game, q + h * k3, u)
        q = q + h / 6.0 * (k1 + 2 * k2 + 2 * k3 + k4)
    return q


class _BatchPID:
    def __init__(self, B, dt, Kp, Ki, x_ref, u_max, u_min, du_max, du_min):
        self.dt, self.Kp, self.Ki = dt, Kp, Ki
        self.x_ref = x_ref
        self.u_max, self.u_min, self.du_max, self.du_min = u_max, u_min, du_max, du_min
        self.ei = np.zeros(B)
        self.u_prev = np.zeros(B)

    def solve(self, x):
        e = x - self.x_ref
        self.ei = np.clip(self.ei + e * self.dt, -100, 100)
        u = -(self.Kp * e + self.Ki * self.ei)
        du = np.clip(u - self.u_prev, self.du_min, self.du_max)
        u = np.clip(du + self.u_prev, self.u_min, self.u_max)
        self.u_prev = u
        return u


def pid_rollout(game: RacingGame, s0, xt0, v0):
    """PID lane-follower roll-out for a batch of single agents; returns q0 [B,6], xy [B,N+1,2], u_ws [B,N,2]."""
    B, N, dt, track = len(s0), game.N, game.dt, game.track
    steer = _BatchPID(B, dt, 1.0, 0.005, 0.0, game.u_ub[1], game.u_lb[1], game.rate_ub[1], game.rate_lb[1])
    speed = _BatchPID(B, dt, 1.0, 0.0, v0, game.u_ub[0], game.u_lb[0], game.rate_ub[0], game.rate_lb[0])
    x, y, _ = track.local_to_global((s0, xt0, np.zeros(B)))
    q = np.stack([x, y, v0, np.zeros(B), s0, xt0], axis=1)
    q0 = q.copy()
    xy = np.zeros((B, N + 1, 2))
    xy[:, 0] = q[:, :2]
    u_ws = np.zeros((B, N, NUA))
    for k in range(N):
        u_a = speed.solve(q[:, 2])
        u_s = steer.solve(5.0 * (q[:, 5] - xt0) + q[:, 3])
        u = np.stack([u_a, u_s], axis=1)
        q = _rk4(game, q, u, dt)
        gx, gy, _ = track.local_to_global((q[:, 4], q[:, 5], q[:, 3]))
        q[:, 0], q[:, 1] = gx, gy
        xy[:, k + 1] = q[:, :2]
        u_ws[:, k] = u
    return q0, xy, u_ws


def pid_rollout_device(game: RacingGame, s0, xt0, v0, device=0):
    """Same roll-out on the GPU (``dgsqp_pid_rollout``, one thread per agent): NumPy in, NumPy out.  Agrees with
    :func:`pid_rollout` to rounding (CUDA and NumPy transcendental functions differ in the last ulp)."""
    import ctypes as C
    from . import _abi
    lib = _abi.load()
    s0, xt0, v0 = (np.ascontiguousarray(a, dtype=np.float64) for a in (s0, xt0, v0))
    K, N = len(s0), game.N
    q0, xy, u_ws = np.empty((K, 6)), np.empty((K, N + 1, 2)), np.empty((K, N, NUA))
    kp = np.ascontiguousarray(game.track.key_pts, dtype=np.float64)
    gs = game.to_struct()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    _abi.check(lib.dgsqp_pid_rollout(C.byref(gs), p(kp), int(device), K, p(s0), p(xt0), p(v0), p(q0), p(xy), p(u_ws), 0, None))
    return q0, xy, u_ws


def _collision_free(xys, radii):
    M = len(xys)
    ok = np.ones(xys[0].shape[0], dtype=bool)
    for i in range(M):
        for j in range(i + 1, M):
            d = np.linalg.norm(xys[i] - xys[j], axis=2)
            ok &= ~np.any(d < radii[i] + radii[j], axis=1)
    return ok


def sample_head_to_head(game: RacingGame, B, seed=0, device=None):
    """B accepted 2-agent instances: x0 [B,12], u_ws [B,n] agent-major.  ``device``: CUDA ordinal to run the PID
    roll-outs on the GPU (``pid_rollout_device``) instead of NumPy."""
    assert game.M == 2
    pid_rollout = globals()["pid_rollout"] if device is None else (lambda g, s, xt, v: pid_rollout_device(g, s, xt, v, device))
    rng = np.random.default_rng(seed)
    first_seg_len = game.track.cl_segs[0, 0]
    hw = game.half_width
    obs_d = game.obs_r[0] + game.obs_r[1]
    x0s, uws = [], []
    have = 0
    while have < B:
        K = max(256, int(1.6 * (B - have)))
        ego_s = np.maximum(0.1, rng.random(K) * first_seg_len)
        ego_xt = rng.random(K) * hw * 2 - hw
        ego_v = rng.random(K) + 2
        d = 2 * np.pi * rng.random(K)
        tar_v = rng.random(K) + 2
        tar_s = ego_s + 1.2 * obs_d * np.cos(d)
        tar_xt = ego_xt + 1.2 * obs_d * np.sin(d)
        keep = (tar_s >= 0) & (np.abs(tar_xt) <= hw)
        ego_s, ego_xt, ego_v, tar_s, tar_xt, tar_v = (a[keep] for a in (ego_s, ego_xt, ego_v, tar_s, tar_xt, tar_v))
        e0, exy, eu = pid_rollout(game, ego_s, ego_xt, ego_v)
        t0, txy, tu = pid_rollout(game, tar_s, tar_xt, tar_v)
        ok = _collision_free([exy, txy], [obs_d / 2, obs_d / 2])
        x0s.append(np.hstack([e0, t0])[ok])
        uws.append(np.hstack([eu.reshape(len(eu), -1), tu.reshape(len(tu), -1)])[ok])
        have += int(ok.sum())
    return np.ascontiguousarray(np.vstack(x0s)[:B]), np.ascontiguousarray(np.vstack(uws)[:B])


def sample_agents(game: RacingGame, B, seed=0, device=None):
    """B accepted M-agent instances: x0 [B,6M], u_ws [B,n] agent-major (``device`` as in sample_head_to_head)."""
    pid_rollout = globals()["pid_rollout"] if device is None else (lambda g, s, xt, v: pid_rollout_device(g, s, xt, v, device))
    rng = np.random.default_rng(seed)
    first_seg_len = game.track.cl_segs[0, 0]
    hw = game.half_width
    x0s, uws = [], []
    have = 0
    while have < B:
        K = max(256, int(2.0 * (B - have)))
        q0s, xys, us = [], [], []
        for _ in range(game.M):
            s = np.maximum(0.1, rng.random(K) * first_seg_len)
            xt = rng.random(K) * hw * 2 - hw
            v = rng.random(K) + 2
            q0, xy, u = pid_rollout(game, s, xt, v)
            q0s.append(q0)
            xys.append(xy)
            us.append(u.reshape(K, -1))
        ok = _collision_free(xys, game.obs_r)
        x0s.append(np.hstack(q0s)[ok])
        uws.append(np.hstack(us)[ok])
        have += int(ok.sum())
    return np.ascontiguousarray(np.vstack(x0s)[:B]), np.ascontiguousarray(np.vstack(uws)[:B])


def sample_merge(game: MergeGame, B, seed=1):
    """B accepted merge instances: x0 [B, 4M] (q = [x, y, v, psi] per car), u_ws [B, n] = 0 (the script never calls
    set_warm_start, DGSQP.py:179).  Trial t of the script uses draws 12t..12t+11 of ``default_rng(seed)``; a trial is
    rejected when the zero-input RK3 roll-outs collide -- with car 3 rolled out from the ZERO state, because the script
    never initialises ``car3_q_ws[0]`` (:486-488; SURVEY App. C #6)."""
    assert game.M == 3
    rng = np.random.default_rng(seed)
    th = np.pi / 12
    x5_0, x7_0 = 1.5, game.lanes[2][1][0]
    h, N = game.dt, game.N
    out, have = [], 0
    while have < B:
        K = max(64, int(1.5 * (B - have)))
        r = rng.random((K, 12))
        cars = []
        for c, x_nom in enumerate((0.0, 0.5)):
            x = x_nom + 0.5 * r[:, 4 * c] - 0.25
            y = 0.15 + 0.1 * r[:, 4 * c + 1] - 0.05
            v = 0.3 * (1 + 0.06 * r[:, 4 * c + 2] - 0.03)
            p = 0.0 + (5 * r[:, 4 * c + 3] - 2.5) * np.pi / 180
            cars.append(np.stack([x, y, v, p], axis=1))
        x_nom, y_nom = 0.25, -((x7_0 + x5_0) / 2 - 0.25) * np.tan(th)
        s_, ey = 0.5 * r[:, 8] - 0.25, 0.1 * r[:, 9] - 0.05
        x = x_nom + s_ * np.cos(th) - ey * np.sin(th)
        y = y_nom + s_ * np.sin(th) + ey * np.cos(th)
        v = 0.3 * (1 + 0.06 * r[:, 10] - 0.03)
        p = np.pi / 12 + (5 * r[:, 11] - 2.5) * np.pi / 180
        cars.append(np.stack([x, y, v, p], axis=1))
        # zero-input roll-outs: v and psi stay constant, rk3 advances the position by (a1 + 4 a2 + a3)/6 per step
        xys = []
        for q0 in (cars[0], cars[1], np.zeros_like(cars[2])):
            a = np.stack([h * q0[:, 2] * np.cos(q0[:, 3]), h * q0[:, 2] * np.sin(q0[:, 3])], axis=1)
            inc = (a + 4 * a + a) / 6
            xys.append(q0[:, None, :2] + np.arange(N + 1)[None, :, None] * inc[:, None, :])
        ok = _collision_free(xys, list(game.obs_r))
        acc = np.hstack(cars)[ok]
        out.append(acc)
        have += len(acc)
    x0 = np.ascontiguousarray(np.vstack(out)[:B])
    return x0, np.zeros((B, game.n))


def _pcg64_state(seed):
    from . import _abi
    st = np.random.default_rng(seed).bit_generator.state["state"]
    m = (1 << 64) - 1
    return _abi.Pcg64Struct(st["state"] >> 64, st["state"] & m, st["inc"] >> 64, st["inc"] & m)


def _sample_cuda(game, B, seed, device, stream, max_trials, return_trials, kind):
    import ctypes as C
    import torch
    from . import _abi
    lib = _abi.load()
    dev = torch.device("cuda", device)
    if max_trials is None:          # four agents accept about 1 trial in 2 000
        max_trials = max(1 << 20, 20000 * B)
    x0 = torch.empty((B, game.n_q), dtype=torch.float64, device=dev)
    u_ws = (torch.empty if kind is not None else torch.zeros)((B, game.n), dtype=torch.float64, device=dev)
    trial = torch.empty(B, dtype=torch.int64, device=dev) if return_trials else None
    if stream is None:
        stream = torch.cuda.current_stream(dev).cuda_stream
    acc, used = C.c_int32(0), C.c_int64(0)
    rng = _pcg64_state(seed)
    v = lambda t: C.c_void_p(t.data_ptr()) if t is not None and t.numel() else None
    if kind is None:
        rc = lib.dgsqp_sample_merge(C.byref(game.to_struct()), C.byref(rng), int(device), int(B), int(max_trials), v(x0),
                                    v(trial), C.byref(acc), C.byref(used), C.c_void_p(stream))
    else:
        kp = np.ascontiguousarray(game.track.key_pts, dtype=np.float64)
        rc = lib.dgsqp_sample_racing(C.byref(game.to_struct()), kp.ctypes.data_as(C.c_void_p), kind, C.byref(rng), int(device),
                                     int(B), int(max_trials), v(x0), v(u_ws), v(trial), C.byref(acc), C.byref(used),
                                     C.c_void_p(stream))
    _abi.check(rc)
    return (x0, u_ws, trial) if return_trials else (x0, u_ws)


def sample_head_to_head_cuda(game: RacingGame, B, seed=0, device=0, stream=None, max_trials=None, return_trials=False):
    """B accepted 2-agent instances drawn on the GPU: float64 CUDA tensors x0 [B,12], u_ws [B,n] agent-major (and with
    ``return_trials`` the int64 trial id of every instance).  Same distribution and warm start as
    :func:`sample_head_to_head`, trial-major stream (module docstring).  ``stream``: a ``cudaStream_t`` as int (default:
    torch's current stream); ``max_trials``: give up with an error after that many trials (default
    ``max(2^20, 20 000 B)``)."""
    from . import _abi
    assert game.M == 2
    return _sample_cuda(game, B, seed, device, stream, max_trials, return_trials, _abi.SAMPLE_HEAD_TO_HEAD)


def sample_agents_cuda(game: RacingGame, B, seed=0, device=0, stream=None, max_trials=None, return_trials=False):
    """B accepted M-agent instances drawn on the GPU, as :func:`sample_agents` (arguments as in
    :func:`sample_head_to_head_cuda`)."""
    from . import _abi
    return _sample_cuda(game, B, seed, device, stream, max_trials, return_trials, _abi.SAMPLE_AGENTS)


def sample_merge_cuda(game: MergeGame, B, seed=1, device=0, stream=None, max_trials=None, return_trials=False):
    """The instances of ``sample_merge(game, B, seed)`` drawn on the GPU: x0 [B, 12] (bit for bit the same) and a zero
    warm start [B, n] as CUDA tensors (arguments as in :func:`sample_head_to_head_cuda`)."""
    assert game.M == 3
    return _sample_cuda(game, B, seed, device, stream, max_trials, return_trials, None)
