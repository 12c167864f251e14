"""Stage-level comparison GPU vs host build: evaluate, nearestPD, QP, LSQR dual init."""
import sys, pathlib
ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
import numpy as np
import dgsqp_b200 as dg
from dgsqp_b200.montecarlo import sample_head_to_head
from hostsim_lib import HostSim
from gpu_units_lib import run_stages

B = int(sys.argv[1]) if len(sys.argv) > 1 else 16
threads = int(sys.argv[2]) if len(sys.argv) > 2 else 128
game, params = dg.chicane_game(), dg.chicane_params()
x0, u = sample_head_to_head(game, B, seed=0)
rng = np.random.default_rng(5)
n, m = game.n, game.m
l = np.abs(rng.normal(size=(B, m))) * 0.3 * (rng.random((B, m)) < 0.2)
o = run_stages(game, params, x0, u, l, threads=threads)
Q, q, gtl, g, H, du, lam, l0 = (o[k] for k in ("Q", "q", "gtl", "g", "H", "du", "lam", "l0"))
nneg, qpst, qpit, lit = o["nneg"], o["qpst"], o["qpit"], o["lsqr_it"]
hs = HostSim(game, params)
for i in range(B):
    Qh, qh, gtlh, gh, xh = hs.evaluate(x0[i], u[i], l[i])
    Hh, nnh = hs.nearest_pd(Qh)
    sth, duh, lamh, ith = hs.qp(Hh, qh)
    l0h, lih = hs.lsqr(x0[i], u[i])
    print(f"{i:3d} dQ {np.abs(Q[i]-Qh).max():.1e} dq {np.abs(q[i]-qh).max():.1e} dgtl {np.abs(gtl[i]-gtlh).max():.1e} dg {np.abs(g[i]-gh).max():.1e} | "
          f"nneg {nneg[i]}/{nnh} dH {np.abs(H[i]-Hh).max():.1e} | qp st {qpst[i]}/{sth} it {qpit[i]}/{ith} ddu {np.abs(du[i]-duh).max():.1e} dlam {np.abs(lam[i]-lamh).max():.1e} | "
          f"lsqr it {lit[i]}/{lih} dl0 {np.abs(l0[i]-l0h).max():.1e}")
