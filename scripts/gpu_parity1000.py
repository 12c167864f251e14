"""CUDA path vs the large-sample oracle fixture: the numbers behind tests/test_gpu_parity.py::test_large_sample_parity."""
import sys, pathlib
ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import numpy as np
import dgsqp_b200 as dg
d = dict(np.load(ROOT / "tests/golden/chicane_N25_seed0_stats.npz").items())
res = dg.DGSQP(dg.chicane_game(), dg.chicane_params(), print_method=None, mu_vio_thresh=1e-10).solve_batch(d["x0"], d["u_ws"])
same = (res.status == d["status"]) & (res.num_iters == d["num_iters"])
print(f"identical (status, iters): {int(same.sum())}/{len(same)}; identical status: {int((res.status == d['status']).sum())}")
for code, name in ((0, "conv_abs_tol"), (1, "conv_rel_tol")):
    m = same & (d["status"] == code)
    err = np.abs(res.u[m] - d["u"][m]).max(axis=1) / np.maximum(1.0, np.abs(d["u"][m]).max(axis=1))
    qpeq = int((res.qp_solves[m] == d["qp_solves"][m]).sum())
    print(f"{name}: {int(m.sum())} identical; rel err of u: median {np.median(err):.1e} 90% {np.quantile(err, .9):.1e} 99% {np.quantile(err, .99):.1e} "
          f"max {err.max():.1e}; > 1e-6: {int((err > 1e-6).sum())}; qp counts equal {qpeq}")
    idx = np.where(m)[0][np.argsort(-err)[:5]]
    print("   worst:", [(int(i), int(d["num_iters"][i]), int(res.qp_solves[i]), int(d["qp_solves"][i]), float(f"{e:.1e}")) for i, e in zip(idx, np.sort(err)[::-1][:5])])
bad = np.where(~same)[0]
print("mismatches (idx, oracle status/iters, gpu status/iters):", [(int(i), int(d["status"][i]), int(d["num_iters"][i]), int(res.status[i]), int(res.num_iters[i])) for i in bad])
