"""The timer marks of the one-GPU schedules of run_iteration.  bench.py takes its stage times between consecutive marks and plans
the sample shares from the gp_fit, mustar, rff_fit and sampling stages, so every schedule records the same names in the same order
in each covariance mode, with and without a persistent model, cold and appended."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

OVERLAPPED = ["start", "grid_features", "rff_fit", "sampling", "gp_tail", "acquisition"]
OVERLAPPED_FULL = ["start", "grid_features", "rff_fit", "grid_transform", "sampling", "gp_tail", "acquisition"]
SEQUENTIAL = ["start", "grid_features", "gp_fit", "mustar", "rff_fit", "acquisition"]


@pytest.mark.parametrize("overlap,cov,S,marks", [
    pytest.param(True, "diag", 4096, OVERLAPPED, id="overlapped-diag"),
    pytest.param(True, "full", 4096, OVERLAPPED_FULL, id="overlapped-full"),
    pytest.param(False, "diag", 4096, SEQUENTIAL, id="sequential-diag"),
    pytest.param(False, "full", 4096, SEQUENTIAL, id="sequential-full"),
    # below the INT8 threshold there is nothing to overlap: the FP64 engine runs the sequential schedule
    pytest.param(True, "diag", 64, SEQUENTIAL, id="fp64-diag"),
    pytest.param(True, "full", 64, SEQUENTIAL, id="fp64-full"),
])
def test_one_gpu_schedule_marks(overlap, cov, S, marks):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from ppbo_b200 import iteration as it
    from ppbo_b200 import synthetic
    prob = synthetic.make_problem("levy10d", Q=41, P=256, F=500, S=S)
    theta, m, kernel = prob["theta"], prob["m"], prob["kernel"]
    B, P, D = prob["grids"].shape
    assert it.sampling_engine(S, P, prob["F"]) == ("i8" if S == 4096 else "f64")
    dev = torch.device("cuda", torch.cuda.current_device())
    X = torch.from_numpy(prob["X"]).to(dev)
    W, b, grids = (torch.from_numpy(np.ascontiguousarray(prob[k])).to(dev) for k in ("W", "b", "grids"))
    Q0 = prob["Q"] - 1
    n0 = Q0 * (m + 1)
    cold = {"X": X[:n0].contiguous(), "W": W, "b": b, "grids": grids}
    appended = {"block": X[n0:].contiguous(), "W": W, "b": b, "grids": grids}
    saved = it.OVERLAP_SAMPLING
    try:
        it.OVERLAP_SAMPLING = overlap
        state = it.IterationState(kernel, theta, D, m, Q0 + 1, dev, W, b)
        for what, d, Q, st in (("no state", cold, Q0, None), ("cold", cold, Q0, state), ("appended", appended, Q0 + 1, state)):
            timers = []
            it.run_iteration(d, kernel, theta, Q, m, S, seed=3, timers=timers, state=st, weight_covariance=cov)
            torch.cuda.synchronize()
            assert [name for name, _ in timers] == marks, what
    finally:
        it.OVERLAP_SAMPLING = saved
