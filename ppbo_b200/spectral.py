"""Random Fourier basis of a stationary kernel: W drawn from the kernel's spectral density, b uniform on [0, 2 pi).

phi(x) = sqrt(2 sf^2 / F) cos(W x + b) then has E[phi(x)' phi(y)] = k(x, y) (Rahimi & Recht).  One function serves
Hsampler.generate_basis (global numpy stream, reference order) and synthetic.make_problem (a private RandomState).
"""
import numpy as np
import scipy.special

MATERN_NU = {"Matern32_kernel": 1.5, "Matern52_kernel": 2.5}

# camphor_copper_kernel (src/kernels.py:36-53): period-1 factor on coordinates 0, 1, 3, 4, 5, SE factor on coordinate 2
CAMPHOR_PERIODIC = (0, 1, 3, 4, 5)
CAMPHOR_SE_DIM, CAMPHOR_SE_SHIFT = 2, 0.05
PERIODIC_PMF_TAIL = 1e-17


def periodic_mask(kernel):
    """bit d set <=> coordinate d of `kernel` has period 1 (camphor: 0b111011; every other kernel: 0).  The one place that knows it:
    the batched maximiser wraps these coordinates instead of projecting them."""
    if kernel == "camphor_copper_kernel":
        return sum(1 << d for d in CAMPHOR_PERIODIC)
    return 0


def periodic_pmf(l):
    """(ks, p): the spectrum of the period-1 kernel exp(-2 sin^2(pi t) / l^2) = sum_k p_k cos(2 pi k t).  With kappa = 1 / l^2,
    p_k = exp(-kappa) I_|k|(kappa) = ive(|k|, kappa) and sum_k p_k = 1.  ks = -K..K for the first K whose two-sided tail
    2 sum_{k > K} p_k is below PERIODIC_PMF_TAIL; p is renormalised over them."""
    kappa = 1.0 / float(l) ** 2
    kmax = 64
    while True:
        pk = scipy.special.ive(np.arange(kmax + 1), kappa)
        if pk[-1] < 1e-30 * pk.max():
            break
        kmax *= 2
    tail = 2.0 * np.cumsum(pk[::-1])[::-1]             # tail[K] = 2 sum_{k >= K} p_k
    tail = np.append(tail[1:], 0.0)                    # tail[K] = 2 sum_{k > K} p_k
    K = int(np.argmax(tail < PERIODIC_PMF_TAIL))
    ks = np.arange(-K, K + 1)
    p = pk[np.abs(ks)]
    return ks, p / p.sum()


def periodic_frequencies(u, l):
    """integer frequencies k ~ p (periodic_pmf(l)) by inverse CDF of the uniforms u: the smallest k whose cumulative pmf exceeds u"""
    ks, p = periodic_pmf(l)
    idx = np.searchsorted(np.cumsum(p), u, side="right")
    return ks[np.minimum(idx, len(ks) - 1)]


def draw_rff_basis(kernel, F, D, lengthscales, rng=np.random):
    """(W [F x D] or None, b [F]) for `kernel` from `rng` (the np.random module or a RandomState).

    SE:        W = randn(F, D) / l, then b  (the reference's draws, src/random_fourier_sampler.py:42-43).
    Matern-nu: z = randn(F, D), u = chisquare(2 nu, F), W = z / l * sqrt(2 nu / u), then b.  Each row of W is a multivariate
               Student-t with 2 nu degrees of freedom: ONE u per feature row, shared by all dimensions (a u per entry would give
               a product of one-dimensional Matern kernels, which is another kernel).
    camphor:   the product of the period-1 factor on coordinates 0, 1, 3, 4, 5 and the SE factor on coordinate 2 has the product
               spectral measure, so every ENTRY of the periodic columns is its own draw: u = uniform(0, 1, (F, 5)) for the five
               periodic columns in column order, k = periodic_frequencies(u, l_0), W[:, d] = 2 pi k; then z = randn(F),
               W[:, 2] = z / (l_2 + 0.05); then b.  The length-scales are those of the device kernel (l_0 for every periodic
               coordinate, l_2 + 0.05 for coordinate 2), and every sampled function is exactly periodic in the five coordinates.
    RQ:        no basis (W is None); b is still drawn, as the reference does.
    `lengthscales` is a scalar or a length-D sequence (ARD)."""
    if kernel == "SE_kernel":
        W = rng.randn(F, D) / lengthscales
    elif kernel in MATERN_NU:
        two_nu = 2.0 * MATERN_NU[kernel]
        z = rng.randn(F, D)
        u = rng.chisquare(two_nu, F)
        W = z / np.asarray(lengthscales, dtype=float) * np.sqrt(two_nu / u)[:, None]
    elif kernel == "camphor_copper_kernel":
        if D != 6:
            raise ValueError("camphor_copper_kernel is defined for D = 6 only")
        ls = np.broadcast_to(np.asarray(lengthscales, dtype=float), (D,))
        u = rng.uniform(0, 1, (F, len(CAMPHOR_PERIODIC)))
        z = rng.randn(F)
        W = np.empty((F, D))
        W[:, CAMPHOR_PERIODIC] = 2 * np.pi * periodic_frequencies(u, ls[0])
        W[:, CAMPHOR_SE_DIM] = z / (ls[CAMPHOR_SE_DIM] + CAMPHOR_SE_SHIFT)
    else:
        W = None
    b = rng.uniform(low=0, high=2 * np.pi, size=F)
    return W, b
