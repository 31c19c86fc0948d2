"""Continuous mu* and x* on the scaled pipeline: the multi-start ascent of the posterior mean (ppbo_mu_maximize,
iteration.mustar_ascent, run_iteration(incumbent=...)).

mu_grad_ref below is the FP64 numpy reference of mu(x) = sum_i alpha_i k(x, X_i) and its gradient for every kernel kind; the CPU
tests check it against central differences and check the start rule, the GPU tests check the kernel against it."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from conftest import load_golden

torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = ("SE_kernel", "RQ_kernel", "Matern32_kernel", "Matern52_kernel")
CAMPHOR = "camphor_copper_kernel"
CAMPHOR_PERIODIC = (0, 1, 3, 4, 5)


def mu_grad_ref(kernel, X, ls, sf, alpha, x, magnitudes=False):
    """mu [P], grad [P, D] at the points x [P, D]; magnitudes=True also returns sum_i |alpha_i k_i| [P] and the sums of the
    magnitudes of the gradient terms [P, D] (the scale of the rounding of any summation order)"""
    X, x, alpha = np.asarray(X, float), np.atleast_2d(np.asarray(x, float)), np.asarray(alpha, float)
    D = X.shape[1]
    ls = np.broadcast_to(np.asarray(ls, float), (D,))
    sf2 = sf * sf
    dl = x[:, None, :] - X[None, :, :]                                    # [P, N, D]
    if kernel == CAMPHOR:
        per = list(CAMPHOR_PERIODIC)
        l0, lz = ls[0], ls[2] + 0.05
        E = (2.0 * np.sin(np.pi * dl[..., per]) ** 2).sum(-1) / l0 ** 2 + 0.5 * dl[..., 2] ** 2 / lz ** 2
        k = sf2 * np.exp(-E)
        dE = np.empty_like(dl)
        dE[..., per] = 2.0 * np.pi / l0 ** 2 * np.sin(2.0 * np.pi * dl[..., per])
        dE[..., 2] = dl[..., 2] / lz ** 2
        terms = -(k * alpha)[..., None] * dE
    else:
        r2 = ((dl / ls) ** 2).sum(-1)
        if kernel == "SE_kernel":
            k = sf2 * np.exp(-0.5 * r2)
            dk2 = -k
        elif kernel == "RQ_kernel":
            t = 1.0 + 0.25 * r2
            k, dk2 = sf2 / t ** 2, -sf2 / t ** 3
        elif kernel == "Matern32_kernel":
            a = np.sqrt(3.0 * r2)
            k, dk2 = sf2 * (1.0 + a) * np.exp(-a), -3.0 * sf2 * np.exp(-a)
        else:
            a = np.sqrt(5.0 * r2)
            k, dk2 = sf2 * (1.0 + a + a * a / 3.0) * np.exp(-a), -(5.0 / 3.0) * sf2 * (1.0 + a) * np.exp(-a)
        terms = (alpha * dk2)[..., None] * dl / ls ** 2
    mu, g = k @ alpha, terms.sum(1)
    if magnitudes:
        return mu, g, np.abs(k * alpha).sum(1), np.abs(terms).sum(1)
    return mu, g


def _mask(kernel):
    return sum(1 << d for d in CAMPHOR_PERIODIC) if kernel == CAMPHOR else 0


def _pg(x, g, mask):
    """projected-gradient stationarity measure of the ascent (|clip(x + g) - x| on the box coordinates, |g| on the periodic ones)"""
    per = np.array([(mask >> d) & 1 for d in range(x.shape[-1])], bool)
    box = np.abs(np.clip(x + g, 0.0, 1.0) - x)
    return np.where(per, np.abs(g), box).max(-1)


def _random_model(kernel, N, D, seed):
    rng = np.random.RandomState(seed)
    X = rng.uniform(0, 1, (N, D))
    ls = rng.uniform(0.2, 0.6, D) if kernel != CAMPHOR else np.full(D, 0.3)
    return X, ls, 0.7, rng.randn(N)


# ------------------------------------------------------------------------------------------------ CPU: the reference itself
@pytest.mark.parametrize("kernel,D,ard", [("SE_kernel", 3, False), ("SE_kernel", 4, True), ("RQ_kernel", 3, True),
                                          ("Matern32_kernel", 3, True), ("Matern52_kernel", 5, True), (CAMPHOR, 6, False)])
def test_reference_gradient_central_differences(kernel, D, ard):
    X, ls, sf, alpha = _random_model(kernel, 23, D, 1)
    if not ard:
        ls = np.full(D, ls[0])
    rng = np.random.RandomState(2)
    pts = [rng.uniform(0, 1, D), X[4] + 0.0, X[7] + 1e-3]                # a design row and a point next to one
    if kernel == CAMPHOR:
        X[0, 0], X[1, 3] = 0.002, 0.998
        near = X[0].copy()
        near[0] = 0.9995                                                  # across camphor's seam from row 0
        pts += [near, np.r_[0.0005, X[1, 1:3], 0.9999, X[1, 4:]]]
    h = 1e-6
    for x in pts:
        _, g = mu_grad_ref(kernel, X, ls, sf, alpha, x)
        fd = np.empty(D)
        for d in range(D):
            e = np.zeros(D)
            e[d] = h
            fd[d] = (mu_grad_ref(kernel, X, ls, sf, alpha, x + e)[0][0] - mu_grad_ref(kernel, X, ls, sf, alpha, x - e)[0][0]) / (2 * h)
        scale = sf * sf * np.abs(alpha).sum()
        assert np.abs(g[0] - fd).max() <= 1e-6 * scale, (kernel, x, g[0], fd)


def test_start_rule_cpu():
    from ppbo_b200 import iteration
    X = torch.tensor([[0.1, 0.1], [0.2, 0.2], [0.3, 0.3], [0.4, 0.4], [0.5, 0.5]], dtype=torch.float64)
    f = torch.tensor([1.0, 3.0, 2.0, 3.0, 3.0], dtype=torch.float64)     # a three-way tie at the top
    cand = torch.tensor([[0.9, 0.9], [0.3, 0.3], [0.7, 0.7], [0.3, 0.3]], dtype=torch.float64)
    cmu = torch.tensor([0.0, 5.0, 1.0, 5.0], dtype=torch.float64)          # the best candidate equals design row 2, and is tied
    prev = torch.tensor([0.65, 0.35], dtype=torch.float64)
    S = iteration.mustar_starts(f, X, cmu, cand, n_starts=4, prev=prev)
    assert torch.equal(S, torch.tensor([[0.2, 0.2], [0.4, 0.4], [0.5, 0.5], [0.3, 0.3], [0.3, 0.3], [0.65, 0.35]], dtype=torch.float64))
    assert torch.equal(iteration.mustar_starts(f, X, n_starts=2), X[[1, 3]])
    assert iteration.mustar_starts(f, X, n_starts=99).shape == (5, 2)      # at most every design row
    assert torch.equal(iteration.mustar_starts(f, X, cmu, cand, n_starts=1), torch.tensor([[0.2, 0.2], [0.3, 0.3]], dtype=torch.float64))


# ------------------------------------------------------------------------------------------------ GPU: the kernel
def _dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


def _maximize(kernel, X, ls, sf, alpha, X0, **kw):
    from ppbo_b200 import ops
    dev = _dev()
    kw.setdefault("periodic_mask", _mask(kernel))
    out = ops.mu_maximize(kernel, ops.to_dev(X, dev), ls, sf, ops.to_dev(alpha, dev), ops.to_dev(X0, dev), **kw)
    return [t.cpu().numpy() for t in out]


_VG_CASES = [(k, D, N) for k in KINDS for D in (1, 2, 6, 20, 32) for N in (1, 37, 1025, 5200)] + [(CAMPHOR, 6, N) for N in (1, 37, 1025, 5200)]


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,D,N", _VG_CASES)
def test_value_and_gradient(kernel, D, N):
    """max_iter = 0: mu and grad mu at the starts.  Value: 1e-12 of sigma_f^2 sum|alpha|.  Gradient, per coordinate: 1e-12 of the sum
    of the magnitudes of its N terms.  Each term carries a few roundings (the kernel's exp / sqrt / sincospi and three products:
    < 10 eps relative) and any summation order of N terms adds at most (N/128 + 7 + 2) eps of the magnitude sum (a sequential run
    of N/128 terms per thread, the 5-level shuffle tree, two warp levels); at N = 5200 that is < 60 eps = 7e-15 of the magnitude
    sum, so 1e-12 leaves two orders of margin for the reference's own rounding."""
    X, ls, sf, alpha = _random_model(kernel, N, D, 10 + D + N)
    rng = np.random.RandomState(N)
    X0 = np.vstack([rng.uniform(0, 1, (5, D)), X[:1]])
    xb, fb, xo, fo, go, it = _maximize(kernel, X, ls, sf, alpha, X0, max_iter=0)
    mu, g, _, gmag = mu_grad_ref(kernel, X, ls, sf, alpha, X0, magnitudes=True)
    scale = sf * sf * np.abs(alpha).sum()
    assert np.array_equal(xo, X0) and np.all(it == 0)
    assert np.abs(fo - mu).max() <= 1e-12 * scale
    assert np.all(np.abs(go - g) <= 1e-12 * gmag + 1e-300), np.abs(go - g).max()
    r = int(np.argmax(fo))
    assert fb[0] == fo[r] and np.array_equal(xb, xo[r])


@pytest.mark.gpu
def test_argument_errors():
    from ppbo_b200 import ops
    from ppbo_b200._lib import PPBOError
    dev = _dev()
    X = torch.rand((7, 3), dtype=torch.float64, device=dev)
    a = torch.ones(7, dtype=torch.float64, device=dev)
    X0 = torch.rand((2, 3), dtype=torch.float64, device=dev)
    ok = ops.mu_maximize("SE_kernel", X, 0.3, 1.0, a, X0)
    torch.cuda.synchronize()
    assert ok[0].shape == (3,)
    bad = [dict(X0=X0[:0]), dict(max_iter=-1), dict(gtol=-1.0), dict(gtol=float("inf")), dict(gtol=float("nan")), dict(kernel=3),
           dict(kernel=9), dict(periodic_mask=8)]
    for b in bad:
        kw = dict(kernel="SE_kernel", X0=X0, max_iter=10, gtol=1e-10, periodic_mask=0)
        kw.update(b)
        with pytest.raises(PPBOError):
            ops.mu_maximize(kw["kernel"], X, 0.3, 1.0, a, kw["X0"], max_iter=kw["max_iter"], gtol=kw["gtol"], periodic_mask=kw["periodic_mask"])
    X33 = torch.rand((7, 33), dtype=torch.float64, device=dev)
    with pytest.raises(PPBOError):
        ops.mu_maximize("SE_kernel", X33, 0.3, 1.0, a, torch.rand((2, 33), dtype=torch.float64, device=dev))
    with pytest.raises(PPBOError):                                        # camphor is defined for D = 6 only
        ops.mu_maximize(CAMPHOR, X, 0.3, 1.0, a, X0)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", KINDS)
def test_planted_interior_maximum(kernel):
    """one design row with alpha > 0: mu = alpha k(x, c) has its only maximum at c; starts in its basin reach it"""
    c = np.array([0.37, 0.61, 0.52])
    rng = np.random.RandomState(3)
    X0 = c + rng.uniform(-0.1, 0.1, (8, 3))
    xb, fb, xo, fo, go, it = _maximize(kernel, c[None], [0.3, 0.4, 0.5], 0.8, np.array([2.0]), X0)
    assert np.abs(xo - c).max() <= 1e-6, np.abs(xo - c).max()
    assert np.all(np.abs(fo - 2.0 * 0.64) <= 1e-12 * 2.0 * 0.64)


@pytest.mark.gpu
def test_planted_maximum_outside_the_box():
    """a peak at (1.3, 0.5): the ascent ends on the face x_0 = 1 with the KKT conditions (g_0 >= 0 pointing out of the box, g_1 = 0
    to the tolerance) holding in the FP64 reference"""
    from ppbo_b200 import ops
    X, ls, sf, alpha = np.array([[1.3, 0.5]]), [0.3, 0.3], 1.0, np.array([1.0])
    X0 = np.array([[0.8, 0.4], [0.2, 0.9], [0.99, 0.51]])
    xb, fb, xo, fo, go, it = _maximize("SE_kernel", X, ls, sf, alpha, X0)
    assert np.all(xo[:, 0] == 1.0)
    _, g = mu_grad_ref("SE_kernel", X, ls, sf, alpha, xo)
    assert np.all(g[:, 0] > 0)
    assert np.all(np.abs(g[:, 1]) <= 10 * ops.MU_MAXIMIZE_GTOL * sf * sf) and np.abs(xo[:, 1] - 0.5).max() <= 1e-8


@pytest.mark.gpu
def test_camphor_seam():
    """a peak at 0.995 on the periodic coordinate 0, started from 0.01: reached across the seam with the mask, stuck at the face
    x_0 = 0 without it"""
    c = np.array([0.995, 0.5, 0.5, 0.5, 0.5, 0.5])
    X0 = c.copy()[None]
    X0[0, 0] = 0.01
    xb, fb, xo, fo, go, it = _maximize(CAMPHOR, c[None], 0.3, 0.5, np.array([1.0]), X0)
    assert abs(xo[0, 0] - 0.995) <= 1e-6 and np.abs(xo[0, 1:] - 0.5).max() <= 1e-6
    xb, fb, xo, fo, go, it = _maximize(CAMPHOR, c[None], 0.3, 0.5, np.array([1.0]), X0, periodic_mask=0)
    assert xo[0, 0] == 0.0 and go[0, 0] < 0


# ------------------------------------------------------------------------------------------------ GPU: full-size models
def _golden_model(name):
    from ppbo_b200 import iteration, ops
    g = load_golden(name)
    return iteration.gp_fit(ops.to_dev(g["X"], _dev()), g["kernel"], g["theta"], g["Q"], g["m"], tol=1e-9)


def _bench_model(name):
    from ppbo_b200 import iteration, ops, synthetic
    p = synthetic.make_problem(name)
    return iteration.gp_fit(ops.to_dev(p["X"], _dev()), p["kernel"], p["theta"], p["Q"], p["m"], tol=1e-9)


_MODELS = {}


def _model(name):
    if name not in _MODELS:
        _MODELS[name] = _golden_model(name) if name.endswith("_full") else _bench_model(name)
    return _MODELS[name]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["camel2d_full", "hartmann6d_full", "camphor6d_full", "ackley20d", "levy10d"])
def test_properties_full_size(name):
    """every start ends at or above its start value; every end point is stationary in the FP64 reference (projected gradient
    within 1e-8 of sigma_f^2 sum|alpha|: the kernel stops at 1e-10 or when no step of its line search raises its own rounded mu)
    or reports the iteration cap; two calls give the same bits"""
    from ppbo_b200 import iteration, ops
    g = _model(name)
    dev = _dev()
    X0 = iteration.mustar_starts(g.f_map, g.X, n_starts=iteration.MUSTAR_STARTS)
    args = (g.kernel, g.X, g.lengthscales, g.theta[2], g.alpha)
    mask = _mask(g.kernel)
    f0 = ops.mu_maximize(*args, X0, max_iter=0, periodic_mask=mask)[3]
    r1 = ops.mu_maximize(*args, X0, periodic_mask=mask)
    r2 = ops.mu_maximize(*args, X0, periodic_mask=mask)
    for a, b in zip(r1, r2):
        assert torch.equal(a, b)
    xo, fo, it = r1[2].cpu().numpy(), r1[3].cpu().numpy(), r1[5].cpu().numpy()
    assert np.all(fo >= f0.cpu().numpy())
    X, alpha = g.X.cpu().numpy(), g.alpha.cpu().numpy()
    sf = g.theta[2]
    _, gr = mu_grad_ref(g.kernel, X, g.lengthscales, sf, alpha, xo)
    pg = _pg(xo, gr, mask)
    scale = sf * sf * np.abs(alpha).sum()
    stationary = pg <= 1e-8 * scale
    assert np.all(stationary | (it == ops.MU_MAXIMIZE_MAX_ITER)), (pg / scale, it)
    print("\n[mustar ascent] %s: iterations min/median/max %d/%d/%d, max pg %.2e of the scale" % (
        name, it.min(), np.median(it), it.max(), (pg / scale).max()))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["camel2d_full", "hartmann6d_full", "camphor6d_full"])
def test_against_reference_search(name):
    """On the reference's own posterior mean (alpha = Sigma^-1 fMAP of the stored reference fit, which reproduces the stored mu* at
    the stored x* to 1e-8) the ascent's mu* is at least the reference's differential-evolution mu* less 1e-9 relative.  Where both
    searches end in the same basin (camel2d, hartmann6d) x* is the reference's within 5e-3: the reference's L-BFGS-B polish stops
    early on a flat top (its mu* is 2.5e-7 .. 7e-7 relative below the ascent's), and 5e-3 is 2 % of the length-scale.  On
    camphor6d the reference's search ends in a lower local maximum (mu* 0.011516, one of its three local results) than the ascent
    (0.011841): there x* is compared with nothing, and the ascent's mu* must exceed the reference's by more than the 1e-6 that
    separates one basin's polishes."""
    import scipy.linalg
    from oracle import ppbo_oracle as O
    from ppbo_b200 import iteration, ops
    gd = load_golden(name)
    dev = _dev()
    X, theta = gd["X"], gd["theta"]
    kern = O.KERNELS[gd["kernel"]]
    Sigma = O.regularize_covariance(kern(X, X, theta), svd_roundtrip=False)
    alpha = scipy.linalg.cho_solve(scipy.linalg.cho_factor(Sigma, lower=True), gd["fMAP"])
    Xd, ad, fd = ops.to_dev(X, dev), ops.to_dev(alpha, dev), ops.to_dev(gd["fMAP"], dev)
    ref_mu, ref_x = float(gd["mustar"]), gd["xstar"]
    at_ref = ops.mu_maximize(gd["kernel"], Xd, theta[1], theta[2], ad, ops.to_dev(ref_x[None], dev), max_iter=0)[1]
    assert abs(float(at_ref) - ref_mu) <= 1e-8 * abs(ref_mu)      # the same function (alpha by a solve at cond(Sigma) ~ 1e7)
    X0 = iteration.mustar_starts(fd, Xd, n_starts=iteration.MUSTAR_STARTS)
    xb, fb = ops.mu_maximize(gd["kernel"], Xd, theta[1], theta[2], ad, X0, periodic_mask=_mask(gd["kernel"]))[:2]
    mustar, xstar = float(fb), xb.cpu().numpy()
    dx = xstar - ref_x
    if gd["kernel"] == CAMPHOR:
        per = list(CAMPHOR_PERIODIC)
        dx[per] -= np.round(dx[per])
    print("\n[mustar vs reference] %s: mu* %.15g (reference %.15g), |x* - x*_ref| %.2e" % (name, mustar, ref_mu, np.abs(dx).max()))
    assert mustar >= ref_mu - 1e-9 * abs(ref_mu)
    if name == "camphor6d_full":
        assert mustar >= ref_mu * (1 + 1e-6)
    else:
        assert np.abs(dx).max() <= 5e-3


# ------------------------------------------------------------------------------------------------ GPU: run_iteration
def _problem(dev, S):
    from ppbo_b200 import synthetic
    prob = synthetic.make_problem("levy10d", Q=41, P=256, F=500, S=S)
    t = {k: torch.from_numpy(np.ascontiguousarray(prob[k])).to(dev) for k in ("X", "W", "b", "grids")}
    return prob, t


def _check_incumbent(g, t, prob, sums, sums0, rff, inc, S, cov, grids):
    from ppbo_b200 import iteration, ops
    assert torch.equal(sums[:, 1:], sums0[:, 1:])
    PhiT = iteration.rff_grid_features(t["W"], t["b"], prob["theta"][2], grids)
    fmax, _ = iteration.rff_sampled_maxima(rff, PhiT, 0, S, seed=5, covariance=cov)
    assert torch.equal(ops.acq_reduce_dev(fmax, inc[:1])[:, 0], sums[:, 0])
    B, P, D = grids.shape
    mu = float(inc[0])
    scale = prob["theta"][2] ** 2 * float(g.alpha.abs().sum())
    assert mu >= float(iteration.posterior_mean(g, grids.reshape(B * P, D)).max()) - 1e-12 * scale
    assert mu >= float(iteration.posterior_mean(g, g.X).max()) - 1e-12 * scale
    _, gr = mu_grad_ref(prob["kernel"], g.X.cpu().numpy(), prob["theta"][1], prob["theta"][2], g.alpha.cpu().numpy(), inc[1:].cpu().numpy())
    x = inc[1:].cpu().numpy()
    assert np.all((x >= 0) & (x <= 1))
    mu_ref, _ = mu_grad_ref(prob["kernel"], g.X.cpu().numpy(), prob["theta"][1], prob["theta"][2], g.alpha.cpu().numpy(), x)
    assert abs(mu_ref[0] - mu) <= 1e-12 * scale


@pytest.mark.gpu
@pytest.mark.parametrize("cov", ["diag", "full"])
@pytest.mark.parametrize("S", [4096, 64], ids=["i8", "f64"])
def test_run_iteration_incumbent(S, cov):
    """one GPU, both engines (INT8 overlapped / FP64 sequential), both weight covariances, cold and appended"""
    from ppbo_b200 import iteration
    dev = _dev()
    prob, t = _problem(dev, S)
    Qc, m, D = 30, prob["m"], prob["D"]
    assert iteration.sampling_engine(S, t["grids"].shape[1], prob["F"]) == ("i8" if S == 4096 else "f64")
    Xc, blk = t["X"][:Qc * (m + 1)], t["X"][Qc * (m + 1):]

    def run(state, d, Q, inc=None, batch=None):
        return iteration.run_iteration(d, prob["kernel"], prob["theta"], Q, m, S, seed=5, weight_covariance=cov, state=state,
                                       incumbent=inc, batch=batch)

    def new_state():
        return iteration.IterationState(prob["kernel"], prob["theta"], D, m, prob["Q"], dev, t["W"], t["b"])
    d0 = {"X": Xc, "W": t["W"], "b": t["b"], "grids": t["grids"]}
    d1 = {"block": blk, "W": t["W"], "b": t["b"], "grids": t["grids"]}
    st0, st1 = new_state(), new_state()
    inc = torch.empty(D + 1, dtype=torch.float64, device=dev)
    for d, Q in ((d0, Qc), (d1, prob["Q"])):
        sums0, _, _ = run(st0, d, Q)
        sums, g, rff = run(st1, d, Q, inc)
        _check_incumbent(g, t, prob, sums, sums0, rff, inc, S, cov, t["grids"])
        assert st1.xstar is not None and torch.equal(st1.xstar, inc[1:])
    sums_b, _, _, (idx, qei) = iteration.run_iteration({"X": t["X"], "W": t["W"], "b": t["b"], "grids": t["grids"]}, prob["kernel"],
                                                       prob["theta"], prob["Q"], m, S, seed=5, weight_covariance=cov, incumbent=inc,
                                                       batch=3)
    assert np.array_equal(qei.cpu().numpy()[:1], sums_b.cpu().numpy()[idx.cpu().numpy()[:1], 0] / S)


@pytest.mark.gpu
def test_run_iteration_incumbent_errors():
    from ppbo_b200 import iteration
    from ppbo_b200._lib import PPBOError
    dev = _dev()
    prob, t = _problem(dev, 64)
    d = {"X": t["X"], "W": t["W"], "b": t["b"], "grids": t["grids"]}
    args = (d, prob["kernel"], prob["theta"], prob["Q"], prob["m"], 64)
    with pytest.raises(PPBOError):
        iteration.run_iteration(*args, incumbent=torch.empty(prob["D"], dtype=torch.float64, device=dev))
    with pytest.raises(PPBOError):
        iteration.run_iteration(*args, incumbent=torch.empty(prob["D"] + 1, dtype=torch.float64))
    with pytest.raises(PPBOError):
        iteration.run_iteration(*args, incumbent=torch.empty(prob["D"] + 1, dtype=torch.float64, device=dev), shard_mustar=True)


@pytest.mark.gpu
def test_loop_through_xstar():
    """three appended iterations: the lines of iteration k + 1 go through iteration k's x* (e_d with coordinate d freed); mu* is
    finite, x* in the box, and the previous x* is among the starts"""
    from ppbo_b200 import iteration, ops, synthetic
    dev = _dev()
    S = 4096
    prob = synthetic.make_problem("levy10d", Q=40, P=128, F=500, S=S)
    m, D = prob["m"], prob["D"]
    X = torch.from_numpy(prob["X"]).to(dev)
    W, b = (torch.from_numpy(prob[k]).to(dev) for k in ("W", "b"))
    state = iteration.IterationState(prob["kernel"], prob["theta"], D, m, 43, dev, W, b)
    inc = torch.empty(D + 1, dtype=torch.float64, device=dev)
    grids = torch.from_numpy(prob["grids"]).to(dev)
    Q, d = 40, {"X": X, "W": W, "b": b, "grids": grids}
    rng = np.random.RandomState(8)
    seen = []
    for k in range(3):
        if k > 0:
            xstar = inc[1:].cpu().numpy()
            xs = np.tile(xstar, (D, 1))
            xs[np.arange(D), np.arange(D)] = 0.0
            alphas = np.sort(rng.uniform(0, 1, (D, 128)), axis=1)
            grids = ops.to_dev(iteration.line_grids(np.eye(D), xs, alphas), dev)
            on_line = grids.cpu().numpy()[np.arange(D), :, :]
            for dd in range(D):                                           # every line goes through x*
                rest = np.delete(on_line[dd], dd, axis=1)
                assert np.allclose(rest, np.delete(xstar, dd)[None, :], atol=0, rtol=0)
            block = torch.from_numpy(synthetic.make_design(D, 1, m, seed=100 + k)[0]).to(dev)
            Q += 1
            d = {"block": block, "W": W, "b": b, "grids": grids}
        prev = state.xstar.clone() if state.xstar is not None else None
        _, g, _ = iteration.run_iteration(d, prob["kernel"], prob["theta"], Q, m, S, seed=3 + k, state=state, incumbent=inc)
        mu = float(inc[0])
        x = inc[1:].cpu().numpy()
        assert np.isfinite(mu) and np.all((x >= 0) & (x <= 1))
        if prev is not None:
            B, P, _ = grids.shape
            cmu = iteration.posterior_mean(g, grids.reshape(B * P, D))
            starts = iteration.mustar_starts(g.f_map, g.X, cmu, grids.reshape(B * P, D), prev=prev)
            assert torch.equal(starts[-1], prev)
            # the search from these starts is the one run_iteration ran
            xb, fb = ops.mu_maximize(g.kernel, g.X, g.lengthscales, g.theta[2], g.alpha, starts)[:2]
            assert torch.equal(fb, inc[:1]) and torch.equal(xb, inc[1:])
        seen.append(mu)
    assert len(seen) == 3


# ------------------------------------------------------------------------------------------------ GPU: several ranks
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_n_rank_incumbent_equals_single_rank(world):
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "mgpu_mustar_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "MGPU_MUSTAR_OK world=%d" % world in r.stdout
