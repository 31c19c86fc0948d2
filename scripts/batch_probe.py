"""Cost of batch queries on one GPU: iteration.select_batch (greedy joint EI, two launches per pick, one D2H copy at the end) for
q in {1, 2, 4, 8, 16} at B = 20 and B = 256 lines with S = 32768 samples, and a steady-state run_iteration (one appended comparison
set per call, ackley20d bench shape) with batch=8 against the same call without it, alternating.  Prints the card and its power
limit with the numbers; --out writes them as JSON."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ppbo_b200 import iteration, synthetic  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else torch.cuda.get_device_name()


def time_select(B, S, q, dev, reps):
    fmax = torch.from_numpy(np.random.RandomState(B).randn(B, S)).to(dev)
    mustar = torch.tensor([1.5], dtype=torch.float64, device=dev)
    for _ in range(3):
        iteration.select_batch(fmax, mustar, q, B)[0].cpu()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        idx, qei = iteration.select_batch(fmax, mustar, q, B)
        idx.cpu(), qei.cpu()                      # the one copy of the result a caller makes
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b) * 1e3)
    return float(np.median(times)), float(np.min(times))


def steady(dev, pairs, Q0=200):
    prob = synthetic.make_problem("ackley20d", Q=Q0 + 2 * pairs + 2)
    m, theta, kernel, S = prob["m"], prob["theta"], prob["kernel"], prob["S"]
    n0 = Q0 * (m + 1)
    inp = iteration.IterationInputs(prob["X"][:n0], None, prob["W"], prob["b"], None, prob["grids"]).to_device(dev)
    st = iteration.IterationState(kernel, theta, prob["D"], m, prob["Q"], dev, inp["W"], inp["b"])
    iteration.run_iteration(inp, kernel, theta, Q0, m, S, seed=1, state=st)
    X = torch.from_numpy(prob["X"]).to(dev)
    out = {"none": [], "batch8": []}
    Q = Q0
    for k in range(2 * pairs + 2):
        blk = X[Q * (m + 1):(Q + 1) * (m + 1)].contiguous()
        d = {"block": blk, "W": inp["W"], "b": inp["b"], "grids": inp["grids"]}
        tag = "batch8" if k % 2 else "none"
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = iteration.run_iteration(d, kernel, theta, Q + 1, m, S, seed=1 + k, state=st, batch=8 if k % 2 else None)
        res[0].cpu()
        if len(res) == 4:
            res[3][0].cpu()
        torch.cuda.synchronize()
        if k >= 2:                                # the first pair warms the appended path of both variants
            out[tag].append((time.perf_counter() - t0) * 1e3)
        Q += 1
    return {t: {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "n": len(v)} for t, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--pairs", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("batch_probe needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"card": card(), "select_batch_us": {}}
    print("card, power limit:", res["card"])
    for B in (20, 256):
        for q in (1, 2, 4, 8, 16):
            med, mn = time_select(B, 32768, q, dev, a.reps)
            res["select_batch_us"]["B=%d q=%d" % (B, q)] = {"median": med, "min": mn}
            print("select_batch B=%3d S=32768 q=%2d: median %8.1f us  min %8.1f us  (%.1f us per pick)" % (B, q, med, mn, med / q))
    res["steady_run_iteration"] = steady(dev, a.pairs)
    for t, v in res["steady_run_iteration"].items():
        print("steady run_iteration %-6s: median %.2f ms  min %.2f ms  (n=%d)" % (t, v["median_ms"], v["min_ms"], v["n"]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
