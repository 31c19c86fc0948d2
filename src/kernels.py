"""Covariance functions with the reference's names and call signature (src/kernels.py:3-53): k(X1, X2, theta) on host
numpy arrays, theta = (sigma, l, sigma_f), returning a host float64 matrix.  The arithmetic runs on the GPU
(ppbo_kernel_matrix, ppbo_b200/csrc/gram.cu); there is no CPU implementation behind these names.

`theta[1]` may also be a length-D sequence of per-dimension length-scales (ARD) -- a strict generalisation of the
reference, whose SE kernel is isotropic.  The Matern kernels (nu = 3/2, 5/2, GPy's parametrisation) are additions beyond the
reference, with the same theta and the same ARD rule."""
import os
import sys

import numpy as np

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if _ROOT not in sys.path:
    sys.path.insert(0, _ROOT)

from ppbo_b200 import ops  # noqa: E402


def _check(theta):
    l, sigma_f = theta[1], theta[2]
    if np.any(np.asarray(l, dtype=float) <= 0) or sigma_f <= 0:
        print("Check hyperparameter values!")          # reference behaviour: warn, do not raise (src/kernels.py:22-23)


def _evaluate(name, X1, X2, theta):
    _check(theta)
    X1 = np.atleast_2d(np.asarray(X1, dtype=np.float64))
    X2 = np.atleast_2d(np.asarray(X2, dtype=np.float64))
    return ops.kernel_matrix(name, ops.to_dev(X1), ops.to_dev(X2), theta[1], theta[2]).cpu().numpy()


def dist(X1, X2):
    """squared Euclidean distances between the rows of X1 and X2 (src/kernels.py:3-11), on the GPU (ppbo_sqdist)"""
    X1 = np.atleast_2d(np.asarray(X1, dtype=np.float64))
    X2 = np.atleast_2d(np.asarray(X2, dtype=np.float64))
    return ops.sqdist(ops.to_dev(X1), ops.to_dev(X2)).cpu().numpy()


def d(x1, x2):
    """|x1_i - x2_j| (src/kernels.py:14-16); index helper used by callers on tiny vectors, host only."""
    return np.abs(np.subtract.outer(x1, x2))


def SE_kernel(X1, X2, theta):
    """sigma_f^2 exp(-|x - y|^2 / (2 l^2))   (src/kernels.py:19-25)"""
    return _evaluate("SE_kernel", X1, X2, theta)


def RQ_kernel(X1, X2, theta):
    """sigma_f^2 (1 + |x - y|^2 / (4 l^2))^-2   (src/kernels.py:27-34, alpha = 2)"""
    return _evaluate("RQ_kernel", X1, X2, theta)


def camphor_copper_kernel(X1, X2, theta):
    """period-1 periodic kernel on coordinates 0,1,3,4,5 times an SE kernel with l + 0.05 on coordinate 2 (src/kernels.py:36-53)"""
    return _evaluate("camphor_copper_kernel", X1, X2, theta)


def Matern32_kernel(X1, X2, theta):
    """sigma_f^2 (1 + sqrt(3) r) exp(-sqrt(3) r),  r = |(x - y) / l|   (Matern nu = 3/2; not in the reference)"""
    return _evaluate("Matern32_kernel", X1, X2, theta)


def Matern52_kernel(X1, X2, theta):
    """sigma_f^2 (1 + sqrt(5) r + 5 r^2 / 3) exp(-sqrt(5) r),  r = |(x - y) / l|   (Matern nu = 5/2; not in the reference)"""
    return _evaluate("Matern52_kernel", X1, X2, theta)
