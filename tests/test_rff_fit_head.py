"""The head of the cold weight-space fit.  From a null omega0 (a known zero start) the first Newton step is taken with the identity
Hessian without factorising it: the same bits as the full step from an explicit zero vector, one factorisation fewer."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from ppbo_b200 import ops as _ops
    return _ops


def _problem(ops, name):
    """(Phi_X feature-major, Q, m, sigma) at the bench shape (Ackley-20D, F = 1000) or of a golden case"""
    if name == "bench":
        from ppbo_b200 import synthetic
        p = synthetic.make_problem("ackley20d")
        X, W, b, theta, Q, m = p["X"], p["W"], p["b"], p["theta"], p["Q"], p["m"]
    else:
        g = np.load(os.path.join(GOLDEN, name + ".npz"))
        X, W, b, theta, Q, m = g["X"], g["rff_W"], g["rff_b"], g["theta"], int(g["Q"]), int(g["m"])
    Phi = ops.rff_features(ops.to_dev(W), ops.to_dev(b), ops.to_dev(X), float(theta[2]), feature_major=True)
    return Phi, Q, m, float(theta[0])


@pytest.mark.parametrize("name", ["bench", "hartmann6d"])
def test_identity_first_step_is_bit_identical(ops, name):
    """the null start and the explicit zero vector walk the same path; only the first factorisation is saved"""
    Phi, Q, m, sigma = _problem(ops, name)
    zero = torch.zeros(Phi.shape[0], dtype=torch.float64, device=Phi.device)
    w0, hd0, st0 = ops.rff_fit(Phi, Q, m, sigma, omega0=None, tol=1e-8)
    wz, hdz, stz = ops.rff_fit(Phi, Q, m, sigma, omega0=zero, tol=1e-8)
    torch.cuda.synchronize()
    assert st0["info"] == 0 and stz["info"] == 0
    assert torch.equal(w0, wz)
    assert torch.equal(hd0, hdz)
    assert stz["factorizations"] - st0["factorizations"] == 1, (st0, stz)
    assert st0["iterations"] == stz["iterations"] and st0["chord_steps"] == stz["chord_steps"]
