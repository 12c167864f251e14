"""Monte-Carlo instance generation on the device (csrc/mc_sampler.cuh, dgsqp_sampler.cu) against NumPy.

The reference for the racing games is a NumPy twin of the trial-major stream below: ``rng.random((K, D))`` with the
transforms of ``montecarlo.sample_head_to_head`` / ``sample_agents``, the roll-outs of ``montecarlo.pid_rollout`` and the
test of ``montecarlo._collision_free``.  For merge the reference is ``montecarlo.sample_merge`` itself, which reads the
stream in the same order.  CPU: the sampler source compiled for the host; GPU: the library through the C ABI."""
import ctypes as C
import pathlib
import subprocess

import numpy as np
import pytest

import dgsqp_b200 as dg
from dgsqp_b200 import _abi
from dgsqp_b200.montecarlo import _collision_free, _pcg64_state, pid_rollout, sample_merge

HERE = pathlib.Path(__file__).resolve().parent
H2H, AGENTS = _abi.SAMPLE_HEAD_TO_HEAD, _abi.SAMPLE_AGENTS
RACING = {"chicane": (lambda: dg.chicane_game(), H2H), "curve90_N10": (lambda: dg.curve_game(90.0, 10), H2H),
          "curve90_N25": (lambda: dg.curve_game(90.0, 25), H2H), "agents3": (lambda: dg.agents_game(3), AGENTS),
          "agents4": (lambda: dg.agents_game(4), AGENTS)}


def twin_racing(game, kind, seed, K, chunk=1 << 20):
    """Accepted trial ids among trials 0..K-1, their x0 and warm starts."""
    rng, first, hw, M = np.random.default_rng(seed), game.track.cl_segs[0, 0], game.half_width, game.M
    ids_all, x0s, uws = [], [], []
    for lo in range(0, K, chunk):
        r = rng.random((min(chunk, K - lo), 5 if kind == H2H else 3 * M))
        if kind == H2H:
            obs_d = game.obs_r[0] + game.obs_r[1]
            ego_s, ego_xt, ego_v = np.maximum(0.1, r[:, 0] * first), r[:, 1] * hw * 2 - hw, r[:, 2] + 2
            d, tar_v = 2 * np.pi * r[:, 3], r[:, 4] + 2
            tar_s, tar_xt = ego_s + 1.2 * obs_d * np.cos(d), ego_xt + 1.2 * obs_d * np.sin(d)
            starts, radii = [(ego_s, ego_xt, ego_v), (tar_s, tar_xt, tar_v)], [obs_d / 2, obs_d / 2]
            ids = np.flatnonzero((tar_s >= 0) & (np.abs(tar_xt) <= hw))
        else:
            starts = [(np.maximum(0.1, r[:, 3 * a] * first), r[:, 3 * a + 1] * hw * 2 - hw, r[:, 3 * a + 2] + 2) for a in range(M)]
            radii, ids = list(game.obs_r), np.arange(len(r))
        # stage 0 first: only trials that pass it are rolled out (the positions are the roll-out's first row)
        xy0 = [np.stack(game.track.local_to_global((s[ids], xt[ids], np.zeros(len(ids))))[:2], axis=1)[:, None] for s, xt, _ in starts]
        ids = ids[_collision_free(xy0, radii)]
        outs = [pid_rollout(game, s[ids], xt[ids], v[ids]) for s, xt, v in starts]
        ok = _collision_free([o[1] for o in outs], radii)
        ids_all.append(lo + ids[ok])
        x0s.append(np.hstack([o[0] for o in outs])[ok])
        uws.append(np.hstack([o[2].reshape(len(ids), -1) for o in outs])[ok])
    return np.concatenate(ids_all), np.vstack(x0s), np.vstack(uws)


# ----------------------------------------------------------------------------------------------- host build of the source
@pytest.fixture(scope="module")
def hlib(tmp_path_factory):
    out = tmp_path_factory.mktemp("mc") / "libmc_sampler_host.so"
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-std=c++17", "-o", str(out),
                           str(HERE / "hostsim" / "mc_sampler_host.cpp")])
    lib = C.CDLL(str(out))
    lib.hs_mc_random.argtypes = [C.POINTER(_abi.Pcg64Struct), C.c_uint64, C.c_int, C.c_void_p]
    lib.hs_mc_racing_decide.argtypes = [C.POINTER(_abi.RacingGameStruct), C.c_void_p, C.c_int, C.POINTER(_abi.Pcg64Struct),
                                        C.c_int64, C.c_void_p]
    lib.hs_mc_racing_instances.argtypes = [C.POINTER(_abi.RacingGameStruct), C.c_void_p, C.c_int, C.POINTER(_abi.Pcg64Struct),
                                           C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.hs_mc_merge.argtypes = [C.POINTER(_abi.MergeGameStruct), C.POINTER(_abi.Pcg64Struct), C.c_int64, C.c_void_p, C.c_void_p]
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.mark.parametrize("seed", [0, 1, 12345, 2 ** 63 + 7])
def test_pcg64_stream_and_jump_ahead_match_numpy(hlib, seed):
    n = 100000
    out = np.empty(n)
    hlib.hs_mc_random(C.byref(_pcg64_state(seed)), 0, n, _p(out))
    assert np.array_equal(out, np.random.default_rng(seed).random(n))
    for d in (1, 12, 2 ** 32 + 3, 10 ** 12):
        rng = np.random.default_rng(seed)
        rng.bit_generator.advance(d)
        one = np.empty(1)
        hlib.hs_mc_random(C.byref(_pcg64_state(seed)), d, 1, _p(one))
        assert one[0] == rng.random(), d


def test_pcg64_struct_matches_header(hlib):
    assert hlib.hs_mc_sizeof_pcg64() == C.sizeof(_abi.Pcg64Struct) == 32


@pytest.mark.parametrize("seed", [0, 1])
@pytest.mark.parametrize("name", ["chicane", "curve90_N10", "agents3", "agents4"])
def test_racing_decisions_and_instances_on_host(hlib, name, seed):
    mk, kind = RACING[name]
    game, K = mk(), 20000
    gs, kp = game.to_struct(), np.ascontiguousarray(game.track.key_pts)
    flag = np.empty(K, dtype=np.uint8)
    assert hlib.hs_mc_racing_decide(C.byref(gs), _p(kp), kind, C.byref(_pcg64_state(seed)), K, _p(flag)) == 0
    ids, x0, u = twin_racing(game, kind, seed, K)
    assert len(ids) > 0 and np.array_equal(np.flatnonzero(flag), ids)
    trial = ids.astype(np.int64)
    x0h, uh = np.empty_like(x0), np.empty_like(u)
    assert hlib.hs_mc_racing_instances(C.byref(gs), _p(kp), kind, C.byref(_pcg64_state(seed)), len(trial), _p(trial),
                                       _p(x0h), _p(uh)) == 0
    assert np.abs(x0h - x0).max() < 1e-13 and np.abs(uh - u).max() < 1e-12


@pytest.mark.parametrize("seed", [0, 1])
def test_merge_decisions_and_x0_on_host(hlib, seed):
    game, K = dg.merge_game(), 20000
    flag, x0 = np.empty(K, dtype=np.uint8), np.empty((K, 12))
    assert hlib.hs_mc_merge(C.byref(game.to_struct()), C.byref(_pcg64_state(seed)), K, _p(flag), _p(x0)) == 0
    ids = np.flatnonzero(flag)
    ref, u = sample_merge(game, len(ids), seed=seed)
    assert np.array_equal(x0[ids], ref) and not u.any()


def test_sampler_rejects_invalid_records():
    lib = _abi.load()
    acc, used, rng = C.c_int32(), C.c_int64(), _pcg64_state(0)
    kp = np.zeros((16, 6))
    buf = np.zeros(64)

    def racing(g, kind, B=4, max_trials=1000):
        return lib.dgsqp_sample_racing(C.byref(g), _p(kp), kind, C.byref(rng), 0, B, max_trials, _p(buf), _p(buf), None,
                                       C.byref(acc), C.byref(used), None)
    g = dg.agents_game(4).to_struct(); g.M = 5
    assert racing(g, AGENTS) == -1
    g = dg.chicane_game().to_struct(); g.track_nseg = 9
    assert racing(g, H2H) == -1
    assert racing(dg.agents_game(3).to_struct(), H2H) == -1
    assert racing(dg.chicane_game().to_struct(), 7) == -1
    assert racing(dg.chicane_game().to_struct(), H2H, B=-1) == -1
    assert racing(dg.chicane_game().to_struct(), H2H, max_trials=0) == -1
    mg = dg.merge_game().to_struct(); mg.M = 2
    assert lib.dgsqp_sample_merge(C.byref(mg), C.byref(rng), 0, 4, 1000, _p(buf), None, C.byref(acc), C.byref(used), None) == -1


def test_sampler_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = _abi.load()
    acc, used, rng = C.c_int32(), C.c_int64(), _pcg64_state(0)
    game = dg.chicane_game()
    kp, buf = np.ascontiguousarray(game.track.key_pts), np.zeros(8 * game.n)
    assert lib.dgsqp_sample_racing(C.byref(game.to_struct()), _p(kp), H2H, C.byref(rng), 0, 8, 1000, _p(buf), _p(buf), None,
                                   C.byref(acc), C.byref(used), None) == -2
    assert b"no CPU fallback" in lib.dgsqp_last_error()
    assert lib.dgsqp_sample_merge(C.byref(dg.merge_game().to_struct()), C.byref(rng), 0, 8, 1000, _p(buf), None, C.byref(acc),
                                  C.byref(used), None) == -2


# ------------------------------------------------------------------------------------------------------------ on the GPU
def _cuda_sampler(kind):
    from dgsqp_b200.montecarlo import sample_head_to_head_cuda, sample_agents_cuda
    return sample_head_to_head_cuda if kind == H2H else sample_agents_cuda


@pytest.mark.gpu
@pytest.mark.parametrize("name,B", [("chicane", 10000), ("curve90_N10", 2000), ("curve90_N25", 2000), ("agents3", 4000),
                                    ("agents4", 2000)])
def test_racing_on_device_against_the_twin(name, B):
    mk, kind = RACING[name]
    game, seed = mk(), 3
    x0, u, trial = (t.cpu().numpy() for t in _cuda_sampler(kind)(game, B, seed=seed, return_trials=True))
    assert x0.shape == (B, game.n_q) and u.shape == (B, game.n) and np.all(np.diff(trial) > 0)
    K = int(trial[-1]) + 1
    ids, tx0, tu = twin_racing(game, kind, seed, K)
    flips = len(np.setxor1d(ids, trial))
    print(f"{name}: {B} instances from {K} trials, {flips} flipped decisions")
    assert flips <= max(1, -(-K // 10000))
    _, di, ti = np.intersect1d(trial, ids, return_indices=True)
    assert len(di) >= B - flips
    assert np.abs(x0[di] - tx0[ti]).max() < 1e-12 and np.abs(u[di] - tu[ti]).max() < 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2])
def test_merge_on_device_is_sample_merge(seed):
    from dgsqp_b200.montecarlo import sample_merge_cuda
    game, B = dg.merge_game(), 100000
    x0, u, trial = (t.cpu().numpy() for t in sample_merge_cuda(game, B, seed=seed, return_trials=True))
    ref, _ = sample_merge(game, B, seed=seed)
    assert np.array_equal(x0, ref) and u.shape == (B, game.n) and not u.any()
    assert np.all(np.diff(trial) > 0)
    r = np.random.default_rng(seed).random((int(trial[-1]) + 1, 12))
    assert np.array_equal(0.0 + 0.5 * r[trial, 0] - 0.25, x0[:, 0])     # each instance comes from its trial's draws


@pytest.mark.gpu
def test_prefix_property_and_repeatability():
    from dgsqp_b200.montecarlo import sample_merge_cuda
    cases = [(dg.chicane_game(), _cuda_sampler(H2H), 2000), (dg.agents_game(4), _cuda_sampler(AGENTS), 200),
             (dg.merge_game(), sample_merge_cuda, 20000)]
    for game, fn, B in cases:
        full = [t.cpu().numpy() for t in fn(game, B, seed=5, return_trials=True)]
        half = [t.cpu().numpy() for t in fn(game, B // 2, seed=5, return_trials=True)]
        again = [t.cpu().numpy() for t in fn(game, B, seed=5, return_trials=True)]
        for a, h, b in zip(full, half, again):
            assert np.array_equal(a[:B // 2], h) and np.array_equal(a, b)


@pytest.mark.gpu
def test_edge_cases_and_stream():
    import torch
    from dgsqp_b200.montecarlo import sample_head_to_head_cuda, sample_merge_cuda
    game = dg.chicane_game()
    x0, u = sample_head_to_head_cuda(game, 0)
    assert x0.shape == (0, 12) and u.shape == (0, game.n)
    x1, u1, t1 = sample_head_to_head_cuda(game, 1, seed=4, return_trials=True)
    x8, u8, t8 = sample_head_to_head_cuda(game, 8, seed=4, return_trials=True)
    assert torch.equal(x1, x8[:1]) and torch.equal(u1, u8[:1]) and torch.equal(t1, t8[:1])
    assert sample_merge_cuda(dg.merge_game(), 0)[0].shape == (0, 12)
    # a budget of trials that runs out: an error, no hang, and the rows written so far are the first instances
    lib = _abi.load()
    acc, used = C.c_int32(), C.c_int64()
    xb, ub = torch.full((8, 12), np.nan, dtype=torch.float64, device="cuda"), torch.zeros((8, game.n), dtype=torch.float64, device="cuda")
    rc = lib.dgsqp_sample_racing(C.byref(game.to_struct()), _p(np.ascontiguousarray(game.track.key_pts)), H2H,
                                 C.byref(_pcg64_state(4)), 0, 8, int(t8[2]) + 1, C.c_void_p(xb.data_ptr()),
                                 C.c_void_p(ub.data_ptr()), None, C.byref(acc), C.byref(used), None)
    assert rc == -1 and acc.value == 3 and used.value == int(t8[2]) + 1
    assert b"max_trials" in lib.dgsqp_last_error()
    assert torch.equal(xb[:3], x8[:3]) and torch.isnan(xb[3:]).all()
    with pytest.raises(_abi.DgsqpLibraryError):
        sample_head_to_head_cuda(game, 8, seed=4, max_trials=int(t8[2]) + 1)
    # a side stream
    s = torch.cuda.Stream()
    xs, us, ts = sample_head_to_head_cuda(game, 8, seed=4, stream=s.cuda_stream, return_trials=True)
    s.synchronize()
    assert torch.equal(xs, x8) and torch.equal(us, u8) and torch.equal(ts, t8)


@pytest.mark.gpu
def test_device_samples_feed_the_device_solve():
    from dgsqp_b200.montecarlo import sample_head_to_head_cuda, sample_merge_cuda
    for game, params, fn, B in [(dg.chicane_game(), dg.chicane_params(), sample_head_to_head_cuda, 500),
                                (dg.merge_game(), dg.merge_params(), sample_merge_cuda, 2000)]:
        solver = dg.DGSQP(game, params, print_method=None, mu_vio_thresh=1e-10)
        x0, u = fn(game, B, seed=1)
        res = solver.solve_batch(x0, u)
        st = res.status.cpu().numpy()
        assert set(np.unique(st)) <= set(_abi.STATUS_MSG) and (st <= 1).mean() > 0.5
        stats = solver.last_stats()
        assert stats[0] == B and stats[1:7].sum() == B
