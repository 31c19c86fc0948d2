"""Laplace fit at the Ackley-20D shape; PPBO_TRACE in the environment prints the iteration trace."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from ppbo_b200 import ops, synthetic
name = sys.argv[1] if len(sys.argv) > 1 else "ackley20d"
tol = float(sys.argv[2]) if len(sys.argv) > 2 else 1e-8
prob = synthetic.make_problem(name)
X = ops.to_dev(prob["X"]); th = prob["theta"]; Q, m = prob["Q"], prob["m"]
Sigma = ops.gram_regularized(prob["kernel"], X, th[1], th[2], 1e-6)
for _ in range(2):
    fit = ops.laplace_fit(Sigma, Q, m, th[0], tol=tol)
torch.cuda.synchronize()
ts = []
for _ in range(5):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); fit = ops.laplace_fit(Sigma, Q, m, th[0], tol=tol); b.record(); torch.cuda.synchronize()
    ts.append(a.elapsed_time(b))
print("%s laplace_fit tol=%g: %.2f ms %s" % (name, tol, float(np.median(ts)), fit.stats))
W = ops.to_dev(prob["W"]); b = ops.to_dev(prob["b"])
Phi = ops.rff_features(W, b, X, th[2], feature_major=True)
for _ in range(2):
    r = ops.rff_fit(Phi, Q, m, th[0], tol=tol)
torch.cuda.synchronize()
ts = []
for _ in range(5):
    a, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); r = ops.rff_fit(Phi, Q, m, th[0], tol=tol); b2.record(); torch.cuda.synchronize()
    ts.append(a.elapsed_time(b2))
print("%s rff_fit tol=%g: %.2f ms %s" % (name, tol, float(np.median(ts)), r[2]))
