"""Random Fourier basis of a stationary kernel: W drawn from the kernel's spectral density, b uniform on [0, 2 pi).

phi(x) = sqrt(2 sf^2 / F) cos(W x + b) then has E[phi(x)' phi(y)] = k(x, y) (Rahimi & Recht).  One function serves
Hsampler.generate_basis (global numpy stream, reference order) and synthetic.make_problem (a private RandomState).
"""
import numpy as np

MATERN_NU = {"Matern32_kernel": 1.5, "Matern52_kernel": 2.5}


def draw_rff_basis(kernel, F, D, lengthscales, rng=np.random):
    """(W [F x D] or None, b [F]) for `kernel` from `rng` (the np.random module or a RandomState).

    SE:        W = randn(F, D) / l, then b  (the reference's draws, src/random_fourier_sampler.py:42-43).
    Matern-nu: z = randn(F, D), u = chisquare(2 nu, F), W = z / l * sqrt(2 nu / u), then b.  Each row of W is a multivariate
               Student-t with 2 nu degrees of freedom: ONE u per feature row, shared by all dimensions (a u per entry would give
               a product of one-dimensional Matern kernels, which is another kernel).
    RQ, camphor: no basis (W is None); b is still drawn, as the reference does.
    `lengthscales` is a scalar or a length-D sequence (ARD)."""
    if kernel == "SE_kernel":
        W = rng.randn(F, D) / lengthscales
    elif kernel in MATERN_NU:
        two_nu = 2.0 * MATERN_NU[kernel]
        z = rng.randn(F, D)
        u = rng.chisquare(two_nu, F)
        W = z / np.asarray(lengthscales, dtype=float) * np.sqrt(two_nu / u)[:, None]
    else:
        W = None
    b = rng.uniform(low=0, high=2 * np.pi, size=F)
    return W, b
