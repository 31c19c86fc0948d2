"""Cost and result of the continuous mu* search (iteration.mustar_ascent, ppbo_mu_maximize) on one GPU:
  * the search alone (CUDA events, median of --reps) on the GP fits of the Ackley-20D and Levy-10D bench problems and a camphor
    problem grown to N = 5200, for K in {32, 128, 296} design-row starts (+ the best candidate of the iteration's lines), with the
    distribution of the steps each start took and mu*(ascent) - mu*(discrete stand-in mustar_over_candidates);
  * run_iteration at the bench shape (Ackley-20D, S = 32768), cold and appended, with and without an incumbent, alternating: wall
    time and the stage marks;
  * on the camel2d_full / hartmann6d_full fixtures (the reference's own posterior mean, alpha = Sigma^-1 fMAP): mu* and |x* - x*_ref|
    against the stored differential-evolution result.
Prints the card and its power limit with the numbers; --out DIR writes r04_mustar_ascent_probe.{json,txt} there."""
import argparse
import io
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from ppbo_b200 import iteration, ops, synthetic  # noqa: E402
from ppbo_b200.spectral import periodic_mask  # noqa: E402

OUT = io.StringIO()


def say(*a):
    s = " ".join(str(x) for x in a)
    print(s)
    OUT.write(s + "\n")


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else torch.cuda.get_device_name()


def events_ms(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times)), float(np.min(times))


def search_alone(dev, reps):
    res = {}
    for name, kw in (("ackley20d", {}), ("levy10d", {"Q": 200}), ("camphor6d", {"Q": 200})):
        p = synthetic.make_problem(name, **kw)
        X = ops.to_dev(p["X"], dev)
        g = iteration.gp_fit(X, p["kernel"], p["theta"], p["Q"], p["m"], tol=1e-9)
        cand = ops.to_dev(p["grids"], dev).reshape(-1, p["D"])
        disc = float(iteration.mustar_over_candidates(g, cand))
        for K in (32, 128, 296):
            med, mn = events_ms(lambda: iteration.mustar_ascent(g, cand, K), reps)
            cmu = iteration.posterior_mean(g, cand)
            X0 = iteration.mustar_starts(g.f_map, g.X, cmu, cand, K)
            xb, fb, _, _, _, its = ops.mu_maximize(g.kernel, g.X, g.lengthscales, g.theta[2], g.alpha, X0,
                                                   periodic_mask=periodic_mask(g.kernel))
            its = its.cpu().numpy()
            r = dict(N=int(X.shape[0]), D=p["D"], K=K, starts=int(X0.shape[0]), median_ms=med, min_ms=mn,
                     iters_min=int(its.min()), iters_median=float(np.median(its)), iters_p90=float(np.percentile(its, 90)),
                     iters_max=int(its.max()), at_cap=int((its == ops.MU_MAXIMIZE_MAX_ITER).sum()), mustar=float(fb),
                     mustar_minus_discrete=float(fb) - disc)
            res["%s_K%d" % (name, K)] = r
            say("search alone  %-10s N=%5d D=%2d K=%3d (%3d starts): median %.3f ms (min %.3f)  steps min/median/p90/max %d/%g/%g/%d"
                "  at cap %d  mu* %.12g  mu* - discrete %.3e" % (name, r["N"], r["D"], K, r["starts"], med, mn, r["iters_min"],
                                                                 r["iters_median"], r["iters_p90"], r["iters_max"], r["at_cap"],
                                                                 r["mustar"], r["mustar_minus_discrete"]))
        del g
        torch.cuda.empty_cache()
    return res


def stages(timers):
    out, prev = {}, None
    for name, ev in timers:
        if prev is not None:
            out[name] = out.get(name, 0.0) + prev.elapsed_time(ev)
        prev = ev
    return out


def pipeline(dev, reps):
    p = synthetic.make_problem("ackley20d", Q=200 + reps + 1)
    m, theta, kernel, S, D = p["m"], p["theta"], p["kernel"], p["S"], p["D"]
    n0 = 200 * (m + 1)
    X = torch.from_numpy(p["X"]).to(dev)
    W, b, grids = (torch.from_numpy(p[k]).to(dev) for k in ("W", "b", "grids"))
    inc = torch.empty(D + 1, dtype=torch.float64, device=dev)
    res = {}

    def timed(d, Q, state, incumbent, seed):
        timers = []
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sums = iteration.run_iteration(d, kernel, theta, Q, m, S, seed=seed, state=state, timers=timers, incumbent=incumbent)[0]
        sums.cpu()
        if incumbent is not None:
            incumbent.cpu()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3, stages(timers)
    d0 = {"X": X[:n0], "W": W, "b": b, "grids": grids}
    for tag in ("none", "incumbent"):                                   # warm-up of both
        timed(d0, 200, None, inc if tag == "incumbent" else None, 1)
    cold = {"none": [], "incumbent": []}
    for k in range(2 * reps):
        tag = ("none", "incumbent")[k % 2]
        cold[tag].append(timed(d0, 200, None, inc if tag == "incumbent" else None, 1))
    states = {t: iteration.IterationState(kernel, theta, D, m, p["Q"], dev, W, b) for t in ("none", "incumbent")}
    for t, st in states.items():
        timed(d0, 200, st, inc if t == "incumbent" else None, 1)
    app = {"none": [], "incumbent": []}
    for k in range(reps):
        blk = X[(200 + k) * (m + 1):(201 + k) * (m + 1)].contiguous()
        d = {"block": blk, "W": W, "b": b, "grids": grids}
        for t in (("none", "incumbent") if k % 2 == 0 else ("incumbent", "none")):
            app[t].append(timed(d, 201 + k, states[t], inc if t == "incumbent" else None, 2 + k))
    for mode, runs in (("cold", cold), ("appended", app)):
        for t, lst in runs.items():
            wall = float(np.median([w for w, _ in lst]))
            st = {s: float(np.median([x[s] for _, x in lst if s in x])) for s in lst[0][1]}
            res["%s_%s" % (mode, t)] = dict(wall_ms=wall, stages_ms=st)
            say("run_iteration %-8s %-9s wall median %.2f ms  stages %s" % (mode, t, wall,
                                                                             " ".join("%s=%.2f" % kv for kv in st.items())))
    return res


def against_reference(dev):
    import scipy.linalg
    from conftest import load_golden
    from oracle import ppbo_oracle as O
    res = {}
    for name in ("camel2d_full", "hartmann6d_full", "camphor6d_full"):
        gd = load_golden(name)
        X, theta = gd["X"], gd["theta"]
        Sigma = O.regularize_covariance(O.KERNELS[gd["kernel"]](X, X, theta), svd_roundtrip=False)
        alpha = scipy.linalg.cho_solve(scipy.linalg.cho_factor(Sigma, lower=True), gd["fMAP"])
        Xd, ad, fd = ops.to_dev(X, dev), ops.to_dev(alpha, dev), ops.to_dev(gd["fMAP"], dev)
        X0 = iteration.mustar_starts(fd, Xd, n_starts=iteration.MUSTAR_STARTS)
        call = lambda: ops.mu_maximize(gd["kernel"], Xd, theta[1], theta[2], ad, X0, periodic_mask=periodic_mask(gd["kernel"]))
        med, _ = events_ms(call, 20)
        xb, fb = call()[:2]
        dx = xb.cpu().numpy() - gd["xstar"]
        if gd["kernel"] == "camphor_copper_kernel":
            per = [0, 1, 3, 4, 5]
            dx[per] -= np.round(dx[per])
        r = dict(mustar=float(fb), mustar_ref=float(gd["mustar"]), dx_max=float(np.abs(dx).max()), search_ms=med)
        res[name] = r
        say("vs reference  %-16s mu* %.15g  reference %.15g  (diff %.2e)  |x* - x*_ref| %.2e  search %.3f ms" % (
            name, r["mustar"], r["mustar_ref"], r["mustar"] - r["mustar_ref"], r["dx_max"], med))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"card": card()}
    say("card, power limit:", res["card"])
    res["search_alone"] = search_alone(dev, a.reps)
    res["against_reference"] = against_reference(dev)
    res["run_iteration"] = pipeline(dev, max(4, a.reps // 2))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "r04_mustar_ascent_probe.json"), "w") as fh:
            json.dump(res, fh, indent=1)
        with open(os.path.join(a.out, "r04_mustar_ascent_probe.txt"), "w") as fh:
            fh.write(OUT.getvalue())


if __name__ == "__main__":
    main()
