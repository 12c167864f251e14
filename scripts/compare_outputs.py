"""Byte-for-byte comparison of two builds of the solver.

  python scripts/compare_outputs.py host --parent REV_OR_DIR
      Builds the host simulation of the kernel source (tests/hostsim) for this tree and for the parent (a source tree,
      or a git revision exported to a temporary directory) and compares HostSim.evaluate (Q, q, G'l, g, x) and full
      solves on chicane N = 25, agents (3, 10) and (4, 6), curve and merge instances, under the v1 and v2 policies, in
      the default build and in the guard build at both memory placements.  The host build runs each CTA as one thread
      and does not contract multiply-adds, so it checks the arithmetic and its order but neither the lane / warp
      mapping of the device code nor the compiler's choice of fused multiply-adds; the `npy` comparison covers those.
      Building writes libhostsim*.so next to tests/hostsim of each tree (build products that git ignores).
  python scripts/compare_outputs.py npy DIR_A DIR_B
      Compares the arrays two runs of `bench.py --dump-outputs` wrote (same workload and arguments, one B200 run each).

Exit status 0 when every array is identical byte for byte.  Meant for changes that must not alter a single result,
such as a different thread mapping of the same arithmetic.
"""
import argparse
import os
import pathlib
import subprocess
import sys
import tempfile

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]


def _cases(dg):
    v2 = lambda N: dg.DGSQPV2Params(N=N, reg=1e-2, reg_decay=0.8, nms_frequency=2, sqp_iters=40)
    from dgsqp_b200.montecarlo import sample_head_to_head, sample_agents, sample_merge
    return [
        ("chicane25_v1", dg.chicane_game(), dg.chicane_params(), lambda g: sample_head_to_head(g, 3, seed=0)),
        ("chicane25_v2", dg.chicane_game(), v2(25), lambda g: sample_head_to_head(g, 2, seed=4)),
        ("agents3_10_v1", dg.agents_game(3, 90.0, 10), dg.agents_params(10), lambda g: sample_agents(g, 2, seed=0)),
        ("agents4_6_v1", dg.agents_game(4, 90.0, 6), dg.agents_params(6), lambda g: sample_agents(g, 2, seed=1)),
        ("agents4_6_v2", dg.agents_game(4, 90.0, 6), v2(6), lambda g: sample_agents(g, 1, seed=2)),
        ("curve45_15_v1", dg.curve_game(45.0, 15), dg.curve_params(15), lambda g: sample_head_to_head(g, 2, seed=1)),
        ("merge20_v1", dg.merge_game(), dg.merge_params(), lambda g: sample_merge(g, 2, seed=1)),
        ("merge10_v2", dg.merge_game(N=10), v2(10), lambda g: sample_merge(g, 2, seed=3)),
    ]


def dump(root, out):
    """Runs in a process of its own: imports the package and the host simulation of `root`."""
    sys.path[:0] = [str(root), str(root / "tests")]
    import dgsqp_b200 as dg
    from hostsim_lib import HostSim
    res = {}
    for guard, budgets in ((False, ("28000",)), (True, ("28000", "0"))):
        for budget in budgets:
            os.environ["DG_HOSTSIM_SMEM_DOUBLES"] = budget
            for name, game, params, sampler in _cases(dg):
                tag = f"{name}_{'guard' if guard else 'plain'}_{budget}"
                hs = HostSim(game, params, guard=guard)
                x0, u_ws = sampler(game)
                rng = np.random.default_rng(7)
                for i in range(x0.shape[0]):
                    u = u_ws[i] + 0.05 * rng.normal(size=game.n)
                    l = np.abs(rng.normal(size=game.m)) * 0.3 * (rng.random(game.m) < 0.3)
                    for f, v in zip(("Q", "q", "gtl", "g", "x"), hs.evaluate(x0[i], u, l)):
                        res[f"{tag}_eval{i}_{f}"] = v.copy()
                    r = hs.solve(x0[i], u_ws[i])
                    for f in ("u", "l", "x", "cost", "cond", "num_iters", "status", "qp_solves", "diag", "l_init"):
                        res[f"{tag}_solve{i}_{f}"] = np.asarray(r[f])
                    if guard:
                        res[f"{tag}_solve{i}_guard"] = np.asarray(hs.guard_check())
    np.savez(out, **res)


def _same(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def _report(pairs):
    bad = [k for k, a, b in pairs if not _same(a, b)]
    for k in bad:
        print("DIFFERENT:", k)
    print(f"{len(pairs) - len(bad)}/{len(pairs)} arrays identical")
    return 0 if not bad and pairs else 1


def host(parent):
    with tempfile.TemporaryDirectory() as tmp:
        tmp = pathlib.Path(tmp)
        proot = pathlib.Path(parent)
        if not proot.is_dir():
            proot = tmp / "parent"
            proot.mkdir()
            arc = subprocess.run(["git", "-C", str(ROOT), "archive", parent], check=True, capture_output=True).stdout
            subprocess.run(["tar", "-x", "-C", str(proot)], input=arc, check=True)
        outs = {}
        for tag, root in (("parent", proot.resolve()), ("child", ROOT)):
            outs[tag] = tmp / f"{tag}.npz"
            subprocess.run([sys.executable, "-B", __file__, "_dump", str(root), str(outs[tag])], check=True)
        a, b = np.load(outs["parent"]), np.load(outs["child"])
        keys = sorted(set(a.files) | set(b.files))
        missing = [k for k in keys if k not in a.files or k not in b.files]
        for k in missing:
            print("MISSING:", k)
        return _report([(k, a[k], b[k]) for k in keys if k not in missing]) or (1 if missing else 0)


def npy(da, db):
    da, db = pathlib.Path(da), pathlib.Path(db)
    fa = sorted(p.name for p in da.glob("*.npy"))
    fb = sorted(p.name for p in db.glob("*.npy"))
    if fa != fb:
        print("file sets differ:", sorted(set(fa) ^ set(fb)))
        return 1
    return _report([(f, np.load(da / f), np.load(db / f)) for f in fa])


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    sub = ap.add_subparsers(dest="cmd", required=True)
    h = sub.add_parser("host")
    h.add_argument("--parent", required=True, help="source tree or git revision of the parent build")
    n = sub.add_parser("npy")
    n.add_argument("a")
    n.add_argument("b")
    d = sub.add_parser("_dump")
    d.add_argument("root")
    d.add_argument("out")
    a = ap.parse_args()
    if a.cmd == "_dump":
        dump(pathlib.Path(a.root), a.out)
        return 0
    return host(a.parent) if a.cmd == "host" else npy(a.a, a.b)


if __name__ == "__main__":
    sys.exit(main())
