"""Covariance-kernel cost of the Matern kernels against SE on one GPU (CUDA events, warm-up, kernels alternated round by round):

  * the symmetric Sigma build with fused shrinkage at N = 5200, D = 20;
  * a 26-row append (ppbo_gram_append) to that Sigma;
  * the mat-vec posterior mean on 20480 candidates;
  * a 32-point ppbo_mu_pred_points window (one differential-evolution window);

and one cold plus five appended one-GPU iterations at the bench shape (Ackley-20D, Q = 200, S = 32768) for SE and Matern-5/2,
host clock around each synchronised iteration.  Prints one JSON object (medians in ms) with the card's name and power limit, and
writes it to --out if given.

  python scripts/matern_probe.py --rounds 20 --out /tmp/matern_probe.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KERNELS = ("SE_kernel", "Matern32_kernel", "Matern52_kernel")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=20)
    ap.add_argument("--iterations", type=int, default=1, help="repeats of the cold + 5 appended iterations per kernel")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("matern_probe needs a CUDA device")
    from ppbo_b200 import iteration as it
    from ppbo_b200 import ops, synthetic
    dev = torch.device("cuda", torch.cuda.current_device())
    rng = np.random.RandomState(0)
    N, D, add, C, W_pts = 5200, 20, 26, 20480, 32
    ls, sf, s = 0.3, 0.5, it.SHRINKAGE
    X = ops.to_dev(rng.rand(N + add, D))
    Y = ops.to_dev(rng.rand(C, D))
    alpha = ops.to_dev(rng.randn(N))
    pts = rng.rand(W_pts, D)
    cap = N + add
    S = torch.empty((cap, cap), dtype=torch.float64, device=dev)

    def sym(k):
        ops.gram_regularized(k, X[:N], ls, sf, s, out=S[:N, :N])

    def app(k):
        ops.gram_append(k, X, N, ls, sf, s, S)

    def mean(k):
        ops.posterior_mean(k, X[:N], ls, sf, alpha, Y)

    def window(k):
        ops.mu_pred_points(k, X[:N], ls, sf, alpha, pts)
    cases = {"sigma_sym_5200": sym, "append_26": app, "posterior_mean_20480": mean, "mu_pred_points_32": window}
    times = {c: {k: [] for k in KERNELS} for c in cases}
    for k in KERNELS:                                   # warm-up: module load, attributes, scratch pools
        for fn in cases.values():
            fn(k)
    torch.cuda.synchronize()
    for _ in range(a.rounds):
        for c, fn in cases.items():
            for k in KERNELS:
                if c == "append_26":
                    sym(k)                               # the append grows the matrix of its own kernel
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn(k)
                e1.record()
                e1.synchronize()
                times[c][k].append(e0.elapsed_time(e1))
    res = {"card": card(), "rounds": a.rounds,
           "kernel_ms": {c: {k: float(np.median(v)) for k, v in d.items()} for c, d in times.items()}}

    # one cold and five appended one-GPU iterations at the bench shape
    it_ms = {}
    for k in ("SE_kernel", "Matern52_kernel"):
        prob = synthetic.make_problem("ackley20d", Q=205, kernel=k)
        theta, m = prob["theta"], prob["m"]
        Xb = ops.to_dev(prob["X"])
        W, b, grids = ops.to_dev(prob["W"]), ops.to_dev(prob["b"]), ops.to_dev(prob["grids"])
        runs = []
        for rep in range(a.iterations + 1):              # the first repetition warms up
            state = it.IterationState(k, theta, D, m, 205, dev, W, b)
            step = []
            for j in range(6):
                Q = 200 + j
                d = ({"X": Xb[:200 * (m + 1)].contiguous(), "W": W, "b": b, "grids": grids} if j == 0 else
                     {"block": Xb[(Q - 1) * (m + 1):Q * (m + 1)].contiguous(), "W": W, "b": b, "grids": grids})
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                it.run_iteration(d, k, theta, Q, m, prob["S"], seed=0, state=state)
                torch.cuda.synchronize()
                step.append(1e3 * (time.perf_counter() - t0))
            if rep:
                runs.append(step)
        runs = np.array(runs)
        it_ms[k] = {"cold": float(np.median(runs[:, 0])), "appended": [float(x) for x in np.median(runs[:, 1:], axis=0)]}
    res["iteration_ms"] = it_ms
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
