"""The camphor/Cu(111) kernel on the scaled pipeline (camphor6d at Q = 200, S = 32768, P = 1024, F = 1000: N = 5200, 6 lines).

1. Posterior mean of the 6 x 1024 candidates at N = 5200: the lifted SE form in mat-vec mode against the materialising path
   (tuning key 11: the 6144 x 5200 cross-covariance of the difference-form kernel, then a GEMV); CUDA events, the two alternated,
   medians over the rounds, and the largest difference between them.
2. The one-GPU iteration through run_iteration, cold and appended, with its stage marks (ms from "start"); gp_tail - sampling is
   how long the reduction waited for the GP chain after the contraction had finished.
3. The camphor Sigma Gram (difference form, fused shrinkage) at N = 5200.
4. Median ratio of the sampled functions' variance to the GP's Laplace predictive variance on every 32nd point of the six lines,
   both weight covariances (as scripts/weight_cov_probe.py does for the SE problems).

    python scripts/camphor_probe.py [--rounds 30] [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys
from ctypes import POINTER, c_double

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ppbo_oracle as O  # noqa: E402


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), [s.strip() for s in r.stdout.splitlines()[0].split(",")])) if r.returncode == 0 else {}


def problem():
    from ppbo_b200 import synthetic
    return synthetic.make_problem("camphor6d", Q=200, S=32768, P=1024, F=1000)


def mean_paths(ops, torch, p, rounds):
    from ppbo_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    X = torch.from_numpy(p["X"]).to(dev)
    Y = torch.from_numpy(p["grids"].reshape(-1, 6).copy()).to(dev)
    N, PT = X.shape[0], Y.shape[0]
    alpha = torch.from_numpy(np.random.RandomState(0).randn(N)).to(dev)
    ls, sf = p["theta"][1], p["theta"][2]
    lsh = np.full(6, float(ls))
    lsp = lsh.ctypes.data_as(POINTER(c_double))
    mu_m = torch.empty(PT, dtype=torch.float64, device=dev)
    ws = torch.empty(PT * N + 64, dtype=torch.float64, device=dev)

    def lifted():
        return ops.posterior_mean(p["kernel"], X, ls, sf, alpha, Y)

    def materialised():
        lib.ppbo_set_tuning(11, 1)
        try:
            rc = lib.ppbo_predict(2, X.data_ptr(), N, 6, lsp, float(sf), 0.0, N, 0, alpha.data_ptr(), None, None, 0, None, 0,
                                  Y.data_ptr(), PT, 1, mu_m.data_ptr(), None, ws.data_ptr(), ws.numel() * 8,
                                  torch.cuda.current_stream().cuda_stream)
        finally:
            lib.ppbo_set_tuning(11, 0)
        assert rc == 0, lib.ppbo_last_error()
        return mu_m
    ev = lambda: torch.cuda.Event(enable_timing=True)     # noqa: E731
    t = {"lifted": [], "materialised": []}
    for fn in (lifted, materialised):
        fn()
    torch.cuda.synchronize()
    for _ in range(rounds):
        for name, fn in (("lifted", lifted), ("materialised", materialised)):
            a, z = ev(), ev()
            a.record()
            fn()
            z.record()
            torch.cuda.synchronize()
            t[name].append(a.elapsed_time(z))
    diff = float((lifted() - materialised()).abs().max())
    out = {k + "_ms_median": float(np.median(v)) for k, v in t.items()}
    out.update({k + "_ms_min": float(np.min(v)) for k, v in t.items()})
    out.update(max_abs_diff=diff, bound_1e12_sf2_sum_abs_alpha=1e-12 * sf * sf * float(alpha.abs().sum()), rounds=rounds, N=N, PT=PT)
    return out


def iterations(ops, torch, p, reps):
    from ppbo_b200 import iteration as it
    dev = torch.device("cuda", 0)
    Q0, m, th, S = p["Q"] - 1, p["m"], p["theta"], p["S"]
    N = Q0 * (m + 1)
    X = torch.from_numpy(p["X"]).to(dev)
    W, b, grids = (torch.from_numpy(np.ascontiguousarray(p[k])).to(dev) for k in ("W", "b", "grids"))

    def one(cov, appended):
        state = it.IterationState(p["kernel"], th, 6, m, Q0 + 1, dev, W, b)
        d = {"X": X[:N].contiguous(), "W": W, "b": b, "grids": grids}
        timers = []
        it.run_iteration(d, p["kernel"], th, Q0, m, S, seed=0, state=state, weight_covariance=cov, timers=None if appended else timers)
        if appended:
            d = {"block": X[N:N + m + 1].contiguous(), "W": W, "b": b, "grids": grids}
            it.run_iteration(d, p["kernel"], th, Q0 + 1, m, S, seed=0, state=state, weight_covariance=cov, timers=timers)
        torch.cuda.synchronize()
        t0 = timers[0][1]
        return {name: t0.elapsed_time(e) for name, e in timers}
    keys = [(c, a) for c in ("diag", "full") for a in (False, True)]
    for k in keys:
        one(*k)
    res = {k: [] for k in keys}
    for _ in range(reps):
        for k in keys:
            res[k].append(one(*k))
    out = {}
    for (cov, app), runs in res.items():
        names = runs[0].keys()
        med = {n: float(np.median([r[n] for r in runs])) for n in names}
        med["gp_tail_minus_sampling"] = float(np.median([r["gp_tail"] - r["sampling"] for r in runs])) if "gp_tail" in med else None
        out["%s_%s" % (cov, "appended" if app else "cold")] = med
    out["reserved_sms"] = dict(appended=it.OVERLAP_RESERVED_SMS, cold=it.OVERLAP_RESERVED_SMS_COLD)
    return out


def gram(ops, torch, p, rounds):
    dev = torch.device("cuda", 0)
    X = torch.from_numpy(p["X"]).to(dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)     # noqa: E731
    ops.gram_regularized(p["kernel"], X, p["theta"][1], p["theta"][2], 1e-6)
    t = []
    for _ in range(rounds):
        a, z = ev(), ev()
        a.record()
        ops.gram_regularized(p["kernel"], X, p["theta"][1], p["theta"][2], 1e-6)
        z.record()
        torch.cuda.synchronize()
        t.append(a.elapsed_time(z))
    return dict(N=int(X.shape[0]), ms_median=float(np.median(t)))


def variance(ops, torch, p):
    import scipy.linalg
    X, Q, m, th = p["X"], p["Q"], p["m"], p["theta"]
    Sig = O.regularize_covariance(O.camphor_copper_kernel(X, X, th), svd_roundtrip=False)
    f = O.fmap_tight(Sig, Q, m, th[0], np.zeros(X.shape[0]))
    Sinv = np.linalg.inv(Sig)
    post = np.linalg.inv(Sinv - O.create_Lambda(f, Q, m, th[0]))
    G = p["grids"][:, ::32].reshape(-1, 6)
    _, Sp = O.mu_Sigma_pred(X, G, th, O.camphor_copper_kernel, Sinv, f, post, svd_roundtrip=False)
    PhiX = O.rff_features(p["W"], p["b"], X, th[2])
    Pd = ops.to_dev(PhiX)
    w, hd, _ = ops.rff_fit(Pd, Q, m, th[0])
    F = PhiX.shape[0]
    buf = ops.rff_hessian_factor_buffer(F, Pd.device)
    info = ops.rff_hessian_factor(Pd, Q, m, th[0], w, buf)
    L = np.tril(ops.hessian_factor_views(buf, F)[0].cpu().numpy())
    Pg = O.rff_features(p["W"], p["b"], G, th[2])
    V = scipy.linalg.solve_triangular(L, Pg, lower=True)
    vg = np.diag(Sp)
    return dict(info=int(info), var_full=float(np.median((V * V).sum(axis=0) / vg)),
                var_diag=float(np.median((Pg * Pg / (-hd.cpu().numpy())[:, None]).sum(axis=0) / vg)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from ppbo_b200 import ops
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    p = problem()
    res = dict(card=card())
    res["mean_6x1024_N5200"] = mean_paths(ops, torch, p, a.rounds)
    print(json.dumps(res["mean_6x1024_N5200"]), flush=True)
    res["iteration_one_gpu"] = iterations(ops, torch, p, max(5, a.rounds // 3))
    print(json.dumps(res["iteration_one_gpu"]), flush=True)
    res["sigma_gram"] = gram(ops, torch, p, a.rounds)
    res["variance_ratio"] = variance(ops, torch, p)
    res["card_after"] = card()
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "camphor_probe.json"), "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
