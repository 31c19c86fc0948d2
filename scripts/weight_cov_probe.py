"""Full against diagonal Laplace covariance of the weight-space posterior (run_iteration(weight_covariance=...)).

1. Accuracy: median ratio of the variance of the sampled function phi(x)' omega to the GP's Laplace predictive variance on every 32nd
   point of each direction's grid, and the same for Var(f(x_p) - f(x_q)) of point pairs on one line (the quantity that decides the
   per-sample arg-max).  The full covariance comes from the DEVICE factor (ppbo_rff_hessian_factor) at the device optimum; the GP
   side is the oracle's (Sigma^-1 + W)^-1 by a general inverse (W is indefinite).
2. Time at the bench shape (Ackley-20D, N = 5200, F = 1000, S = 32768, 20 grids of 1024 points), one GPU, CUDA events: the pieces
   of the full mode (Hessian product + potrf, the Phi~ transform and slicing, the biased contraction against the plain one) and the
   whole run_iteration, cold and appended, diagonal against full.

    python scripts/weight_cov_probe.py [--no-table] [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ppbo_oracle as O  # noqa: E402


def variance_table(ops, torch, names=("camel2d", "levy10d", "ackley20d")):
    import scipy.linalg
    from ppbo_b200 import synthetic
    rows = []
    for name in names:
        p = synthetic.make_problem(name)
        X, Q, m, th = p["X"], p["Q"], p["m"], p["theta"]
        Sig = O.regularize_covariance(O.se_kernel(X, X, th), svd_roundtrip=False)
        f = O.fmap_tight(Sig, Q, m, th[0], np.zeros(X.shape[0]))
        Sinv = np.linalg.inv(Sig)
        post = np.linalg.inv(Sinv - O.create_Lambda(f, Q, m, th[0]))
        npl = p["grids"][:, ::32].shape[1]
        G = p["grids"][:, ::32].reshape(-1, X.shape[1])
        _, Sp = O.mu_Sigma_pred(X, G, th, O.se_kernel, Sinv, f, post, svd_roundtrip=False)
        PhiX = O.rff_features(p["W"], p["b"], X, th[2])
        Pd = ops.to_dev(PhiX)
        w, hd, _ = ops.rff_fit(Pd, Q, m, th[0])
        F = PhiX.shape[0]
        buf = ops.rff_hessian_factor_buffer(F, Pd.device)
        info = ops.rff_hessian_factor(Pd, Q, m, th[0], w, buf)
        L = np.tril(ops.hessian_factor_views(buf, F)[0].cpu().numpy())
        Pg = O.rff_features(p["W"], p["b"], G, th[2])
        V = scipy.linalg.solve_triangular(L, Pg, lower=True)
        Cf = V.T @ V
        Cd = Pg.T @ (Pg / (-hd.cpu().numpy())[:, None])
        ii, jj = [], []
        for b in range(p["grids"].shape[0]):
            for a in range(0, npl, 3):
                ii.append(b * npl + a)
                jj.append(b * npl + (a + npl // 2) % npl)
        ii, jj = np.array(ii), np.array(jj)

        def dv(C):
            return C[ii, ii] + C[jj, jj] - 2 * C[ii, jj]
        vg, dg = np.diag(Sp), dv(Sp)
        rows.append(dict(problem=name, N=int(X.shape[0]), info=int(info),
                         var_full=float(np.median(np.diag(Cf) / vg)), var_diag=float(np.median(np.diag(Cd) / vg)),
                         dvar_full=float(np.median(dv(Cf) / dg)), dvar_diag=float(np.median(dv(Cd) / dg))))
        print("%-10s N=%5d  variance full %.3g diag %.3g   line difference full %.3g diag %.3g" % (
            name, X.shape[0], rows[-1]["var_full"], rows[-1]["var_diag"], rows[-1]["dvar_full"], rows[-1]["dvar_diag"]), flush=True)
    return rows


def timings(ops, torch, reps=20):
    from ppbo_b200 import iteration as it
    from ppbo_b200 import synthetic
    dev = torch.device("cuda", 0)
    p = synthetic.make_problem("ackley20d", Q=201)
    Q0, m, th, S = 200, p["m"], p["theta"], p["S"]
    X = torch.from_numpy(p["X"]).to(dev)
    W, b, grids = (torch.from_numpy(np.ascontiguousarray(p[k])).to(dev) for k in ("W", "b", "grids"))
    B, P, D = p["grids"].shape
    F = p["F"]
    ev = lambda: torch.cuda.Event(enable_timing=True)     # noqa: E731

    def timed(fn, n=reps):
        fn()
        torch.cuda.synchronize()
        t = []
        for _ in range(n):
            a, z = ev(), ev()
            a.record()
            fn()
            z.record()
            torch.cuda.synchronize()
            t.append(a.elapsed_time(z))
        return float(np.median(t))

    out = {}
    # pieces, at the bench problem's optimum
    N = Q0 * (m + 1)
    Pd = ops.rff_features(W, b, X[:N].contiguous(), th[2], feature_major=True)
    w, hd, _ = ops.rff_fit(Pd, Q0, m, th[0])
    buf = ops.rff_hessian_factor_buffer(F, dev)
    out["hessian_factor_ms"] = timed(lambda: ops.rff_hessian_factor(Pd, Q0, m, th[0], w, buf, sync=False))
    H = torch.empty((F, F), dtype=torch.float64, device=dev)
    Lview = ops.hessian_factor_views(buf, F)[0]

    def potrf_only():
        H.copy_(Lview)
        ops.potrf_lower(H)
    out["potrf_1000_ms_incl_copy_and_sync"] = timed(potrf_only)
    r = it.RFFFit()
    r.omega_map, r.L = w, buf
    PhiT = it.rff_grid_features(W, b, th[2], grids)
    out["grid_transform_and_slice_ms"] = timed(lambda: it.rff_transform_grids(r, PhiT, slices=it.SAMPLING_SLICES))
    out["grid_slice_only_ms"] = timed(lambda: it.SlicedGrids(PhiT))
    mu, Gt = it.rff_transform_grids(r, PhiT, slices=it.SAMPLING_SLICES)
    zp = it.rff_prepare_normals(F, 0, S, P, dev, seed=0)
    dp = it.rff_prepare_samples(_diag_fit(w, hd), 0, S, P, seed=0)
    Gd = it.SlicedGrids(PhiT)
    out["normal_slice_ms"] = timed(lambda: it.rff_prepare_normals(F, 0, S, P, dev, seed=0))
    out["diag_sample_slice_ms"] = timed(lambda: it.rff_prepare_samples(_diag_fit(w, hd), 0, S, P, seed=0))
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    out["contraction_biased_ms"] = timed(lambda: ops.ozaki_rowmax(zp.planes, zp.scale, S, Gt.planes, Gt.scale, P, B, F, zp.slices,
                                                                  err=err, bias=mu), n=10)
    out["contraction_plain_ms"] = timed(lambda: ops.ozaki_rowmax(dp.planes, dp.scale, S, Gd.planes, Gd.scale, P, B, F, dp.slices,
                                                                 err=err), n=10)

    # whole iterations: cold (Q0) and appended (Q0 + 1), alternating the two modes
    def iteration(cov, appended):
        state = it.IterationState(p["kernel"], th, D, m, Q0 + 1, dev, W, b)
        d = {"X": X[:N].contiguous(), "W": W, "b": b, "grids": grids}
        timers = []
        it.run_iteration(d, p["kernel"], th, Q0, m, S, seed=0, state=state, weight_covariance=cov,
                         timers=None if appended else timers)
        if appended:
            d = {"block": X[N:N + m + 1].contiguous(), "W": W, "b": b, "grids": grids}
            it.run_iteration(d, p["kernel"], th, Q0 + 1, m, S, seed=0, state=state, weight_covariance=cov, timers=timers)
        torch.cuda.synchronize()
        t0 = timers[0][1]
        return {name: t0.elapsed_time(e) for name, e in timers}
    res = {k: [] for k in ("diag_cold", "full_cold", "diag_appended", "full_appended")}
    for _ in range(2):
        iteration("diag", False), iteration("full", False)
    for _ in range(8):
        for cov in ("diag", "full"):
            for appended in (False, True):
                res["%s_%s" % (cov, "appended" if appended else "cold")].append(iteration(cov, appended))
    for k, v in res.items():
        out["iteration_" + k] = {name: float(np.median([x[name] for x in v])) for name in v[0]}
    return out


def _diag_fit(w, hd):
    from ppbo_b200 import iteration as it
    r = it.RFFFit()
    r.omega_map, r.hess_diag = w, hd
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--no-table", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from ppbo_b200 import ops
    torch.cuda.set_device(0)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("GPU:", gpu, flush=True)
    res = {"gpu": gpu}
    if not args.no_table:
        res["variance_table"] = variance_table(ops, torch)
    res["timings"] = timings(ops, torch)
    print(json.dumps(res["timings"], indent=1))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "weight_cov_probe.json"), "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
