"""GPU probe of the tcgen05 INT8 path: timing of slicing and of the fused GEMM + row max at the Ackley-20D shape."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ppbo_b200 import _lib, ops  # noqa: E402


def timeit(fn, reps=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def ubench(dev):
    lib = _lib.load()
    blocks = 148
    out = torch.zeros(blocks, dtype=torch.int64, device=dev)
    for N in (32, 64, 128, 256):
        for mode in (0, 1):
            for nacc in (1, 2, 3, 4, 6, 7):
                if nacc * N > 448:
                    continue
                iters = 4096
                ops.check(lib.ppbo_ozaki_mma_rate(N, mode, nacc, iters, blocks, ops._p(out), ops._stream()), "mma_rate")
                torch.cuda.synchronize()
                c = out.double().mean().item() / iters
                print("N=%3d mode=%d nacc=%d: %.1f clk/MMA (floor %d) -> %.0f int8 TOP/s chip at 1.9 GHz" % (
                    N, mode, nacc, c, N // 2, 2.0 * 128 * N * 32 / c * 148 * 1.9e9 / 1e12), flush=True)


def main():
    dev = torch.device("cuda", 0)
    if "--ubench" in sys.argv:
        return ubench(dev)
    S, F, P, B = 32768, 1000, 1024, 20
    if len(sys.argv) > 1:
        S = int(sys.argv[1])
    torch.manual_seed(0)
    Om = torch.randn(S, F, dtype=torch.float64, device=dev)
    PhiT = 0.02 * torch.cos(3 * torch.randn(B, P, F, dtype=torch.float64, device=dev))
    lib = _lib.load()
    ref = ops.rff_eval_argmax(Om, PhiT)
    for ks, ng in ((6, 1), (6, 2), (6, 4), (6, 8), (6, 16), (5, 4), (7, 4)):
        lib.ppbo_set_tuning(4, ng)
        ta = timeit(lambda: ops.ozaki_slice(Om, 0, ks))
        tb = timeit(lambda: ops.ozaki_slice(PhiT, 1, ks))
        ap, asc = ops.ozaki_slice(Om, 0, ks)
        bp, bsc = ops.ozaki_slice(PhiT, 1, ks)
        fmax = torch.empty((B, S), dtype=torch.float64, device=dev)
        arg = torch.empty((B, S), dtype=torch.int32, device=dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)

        def run():
            ops.ozaki_rowmax(ap, asc, S, bp, bsc, P, B, F, ks, fmax=fmax, arg=arg, err=err)
        t = timeit(run, reps=3, warm=1)
        flop = 2.0 * S * F * P * B
        iops = flop * ks * (ks + 1) / 2
        d = (fmax - ref[0]).abs().max().item() / ref[0].abs().max().item()
        same = (arg == ref[1]).double().mean().item()
        print("slices=%d groups=%d: slice A %.3f ms, slice B %.3f ms, gemm+rowmax %.3f ms = %.1f TFLOP/s FP64-equivalent, %.0f TOP/s int8; "
              "max rel diff vs DMMA %.2e, same argmax %.6f" % (ks, ng, ta, tb, t, flop / t / 1e9, iops / t / 1e9, d, same), flush=True)
    lib.ppbo_set_tuning(4, 0)


if __name__ == "__main__":
    main()
