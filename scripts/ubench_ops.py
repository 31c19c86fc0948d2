"""GPU micro-timings of the building blocks at the Ackley-20D sizes (run under gpurun; prints a table)."""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from ppbo_b200 import _lib, ops, synthetic, iteration

dev = torch.device("cuda", 0)


def timeit(fn, reps=5, warm=2, setup=None):
    for _ in range(warm):
        if setup: setup()
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        if setup: setup()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def main():
    rng = np.random.RandomState(0)
    for n in (1000, 5000):
        A0 = torch.randn(n, n, dtype=torch.float64, device=dev)
        A = A0 @ A0.T + n * torch.eye(n, dtype=torch.float64, device=dev)
        W = A.clone()
        if n >= 2000:
            _lib.load().ppbo_set_tuning(8, 1)
            t1 = timeit(lambda: ops.potrf_lower(W), setup=lambda: W.copy_(A))
            _lib.load().ppbo_set_tuning(8, 0)
            print("potrf n=%d, general GEMM kernel for panel and look-ahead: %.3f ms" % (n, t1))
        if n >= 2000:
            _lib.load().ppbo_set_tuning(9, 1)
            t1 = timeit(lambda: ops.potrf_lower(W), setup=lambda: W.copy_(A))
            _lib.load().ppbo_set_tuning(9, 0)
            print("potrf n=%d, general GEMM kernel for the trailing update: %.3f ms" % (n, t1))
        t = timeit(lambda: ops.potrf_lower(W), setup=lambda: W.copy_(A))
        W.copy_(A)
        info, ws = ops.potrf_lower(W)
        L = torch.tril(W)
        err = float((L @ L.T - A).abs().max() / A.abs().max())
        print("potrf n=%d: %.3f ms  (%.2f TFLOP/s)  info=%d relerr=%.2e" % (n, t, n ** 3 / 3 / t / 1e9, info, err))
        if "--potrf-only" in sys.argv:
            continue
        b = torch.randn(n, dtype=torch.float64, device=dev)
        t = timeit(lambda: ops.potrs_vec(W, ws, b))
        x = ops.potrs_vec(W, ws, b)
        print("potrs_vec n=%d: %.3f ms  resid=%.2e" % (n, t, float((A @ x - b).abs().max() / b.abs().max())))
        Wb = ops.blockinv_build(W, ws)
        t = timeit(lambda: ops.potrs_vec_blockinv(W, Wb, b))
        x = ops.potrs_vec_blockinv(W, Wb, b)
        print("potrs_vec_blockinv n=%d: %.3f ms  resid=%.2e" % (n, t, float((A @ x - b).abs().max() / b.abs().max())))
        X = torch.randn(2048, n, dtype=torch.float64, device=dev)
        t = timeit(lambda: ops.trsm_right_lower(W, ws, X))
        print("trsm nrhs=2048 n=%d: %.3f ms (%.2f TFLOP/s)" % (n, t, 2048 * n * n / t / 1e9))
        t = timeit(lambda: ops.gemv(A, b))
        print("gemv n=%d: %.3f ms (%.0f GB/s)" % (n, t, 8 * n * n / t / 1e6))
    if "--potrf-only" in sys.argv:
        return
    for (M, N, K) in ((5000, 5000, 128), (5000, 5000, 5000), (1000, 1000, 5000), (4096, 4096, 4096)):
        A = torch.randn(M, K, dtype=torch.float64, device=dev); B = torch.randn(N, K, dtype=torch.float64, device=dev)
        C = torch.zeros(M, N, dtype=torch.float64, device=dev)
        t = timeit(lambda: ops.gemm_nt(A, B, C, 1.0, 1.0))
        print("gemm_nt %dx%dx%d: %.3f ms (%.2f TFLOP/s)" % (M, N, K, t, 2.0 * M * N * K / t / 1e9))
    shapes = ((5000, 5000, 128), (5000, 5000, 256), (2500, 2500, 128), (2500, 2500, 256), (5000, 128, 128), (5000, 128, 256))
    if "--all-gemm" in sys.argv:
        shapes += ((5000, 128, 5000), (4096, 4096, 4096), (1000, 1000, 5000))
    for (M, N, K) in shapes:
        A = torch.randn(M, K, dtype=torch.float64, device=dev); B = torch.randn(N, K, dtype=torch.float64, device=dev)
        C = torch.zeros(M, N, dtype=torch.float64, device=dev)
        ref = A @ B.T
        for cfg in range(6):
            C.zero_()
            ops.gemm_nt_cfg(cfg, A, B, C, 1.0, 0.0)
            err = float((C - ref).abs().max() / ref.abs().max())
            t = timeit(lambda: ops.gemm_nt_cfg(cfg, A, B, C, 1.0, 1.0))
            print("  cfg %d %dx%dx%d: %.3f ms (%.2f TFLOP/s) err=%.1e" % (cfg, M, N, K, t, 2.0 * M * N * K / t / 1e9, err))
    Om = torch.randn(32768, 1000, dtype=torch.float64, device=dev)
    PhiT = torch.randn(20, 1024, 1000, dtype=torch.float64, device=dev)
    if "--no-rowmax" not in sys.argv:
        t = timeit(lambda: ops.rff_eval_argmax(Om, PhiT), reps=3, warm=1)
        print("rowmax S=32768 F=1000 P=1024 B=20: %.2f ms (%.2f TFLOP/s)" % (t, 2.0 * 32768 * 1000 * 1024 * 20 / t / 1e9))
    if "--gemm-only" in sys.argv:
        return
    prob = synthetic.make_problem("ackley20d")
    X = ops.to_dev(prob["X"]); th = prob["theta"]; Q, m = prob["Q"], prob["m"]
    t = timeit(lambda: ops.gram_regularized("SE_kernel", X, th[1], th[2], 1e-6))
    N = X.shape[0]
    print("gram N=%d D=20: %.3f ms (%.0f GB/s write)" % (N, t, 8 * N * N / t / 1e6))
    Sigma = ops.gram_regularized("SE_kernel", X, th[1], th[2], 1e-6)
    t = timeit(lambda: ops.diffspace_gram(Sigma, Q, m))
    print("diffspace_gram: %.3f ms" % t)
    for it in (1, 2, 3, 100):
        t = timeit(lambda: ops.laplace_fit(Sigma, Q, m, th[0], max_iter=it), reps=3, warm=1)
        fit = ops.laplace_fit(Sigma, Q, m, th[0], max_iter=it)
        print("laplace_fit max_iter=%d: %.2f ms  stats=%s n_neg=%d" % (it, t, fit.stats, fit.n_neg))
    W = ops.to_dev(prob["W"]); b = ops.to_dev(prob["b"])
    Phi = ops.rff_features(W, b, X, th[2], feature_major=True)
    for it in (1, 2, 100):
        t = timeit(lambda: ops.rff_fit(Phi, Q, m, th[0], max_iter=it), reps=3, warm=1)
        print("rff_fit max_iter=%d: %.2f ms %s" % (it, t, ops.rff_fit(Phi, Q, m, th[0], max_iter=it)[2]))


if __name__ == "__main__":
    main()
