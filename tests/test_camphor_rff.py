"""camphor_copper_kernel on the scaled pipeline: its exact random Fourier basis, its posterior mean as an SE kernel on lifted
coordinates (mat-vec mode of the stream kernel), and the batched maximiser with its periodic coordinates wrapped at the seam.

The FP64 references live here (the shared oracle is used unchanged): the difference-form camphor kernel with the device's
length-scale rule (l_0 for the periodic coordinates 0, 1, 3, 4, 5, l_2 + 0.05 for coordinate 2) and the random Fourier features."""
import os
from ctypes import POINTER, c_double

import numpy as np
import pytest
import scipy.special

from ppbo_b200 import spectral

torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu
PERIODIC = (0, 1, 3, 4, 5)
MASK = 0b111011


# ----------------------------------------------------------------------------------------------- FP64 references
def camphor_ref(X1, X2, ls, sf):
    """sf^2 prod_{d periodic} exp(-2 sin^2(pi |x_d - y_d|) / l_0^2) exp(-(x_2 - y_2)^2 / (2 (l_2 + 0.05)^2)), difference form,
    torch float64 on the device of X1 (numpy arrays go to the CPU)"""
    X1, X2 = (torch.as_tensor(np.asarray(X), dtype=torch.float64) if not torch.is_tensor(X) else X for X in (X1, X2))
    ls = np.broadcast_to(np.asarray(ls, dtype=float), (6,))
    e = torch.zeros((X1.shape[0], X2.shape[0]), dtype=torch.float64, device=X1.device)
    for d in range(6):
        r = (X1[:, d][:, None] - X2[:, d][None, :]).abs()
        if d == 2:
            e += 0.5 * r * r / (ls[2] + 0.05) ** 2
        else:
            e += 2.0 * torch.sin(np.pi * r) ** 2 / ls[0] ** 2
    return sf * sf * torch.exp(-e)


def features(W, b, X, sf):
    """phi(X) [F x n] = sqrt(2 sf^2 / F) cos(W X' + b)"""
    return np.sqrt(2.0 * sf * sf / W.shape[0]) * np.cos(W @ X.T + b[:, None])


def _hsampler(D, F, theta):
    from types import SimpleNamespace
    from random_fourier_sampler import Hsampler

    def camphor_copper_kernel():
        pass
    gp = SimpleNamespace(D=D, m=3, X=np.zeros((4, D)), xstar=None, xstars_local=None, n_gausshermite_sample_points=200,
                         obs_indices=[0], kernel=camphor_copper_kernel, theta=theta)
    return Hsampler(gp, nFeatures=F)


LS_ARD = [0.21, 0.5, 0.33, 0.7, 0.9, 0.4]        # the device reads l_0 (periodic) and l_2 (SE) of these


def _pairs(rng, n):
    """random pairs, pairs across the seam of one periodic coordinate, pairs differing in coordinate 2 only, pairs differing in two
    periodic coordinates only"""
    X, Y = rng.rand(n, 6), rng.rand(n, 6)
    k = n // 4
    Y[:k] = X[:k]
    for i in range(k):
        d = PERIODIC[i % 5]
        X[i, d], Y[i, d] = rng.uniform(0, 0.06), rng.uniform(0.94, 1.0)
    Y[k:2 * k] = X[k:2 * k]
    Y[k:2 * k, 2] = rng.rand(k)
    Y[2 * k:3 * k] = X[2 * k:3 * k]
    Y[2 * k:3 * k, [0, 3]] = rng.rand(k, 2)
    return X, Y


# ----------------------------------------------------------------------------------------------- host
@pytest.mark.parametrize("l", [0.05, 0.26, 1.0, 4.0])
def test_pmf_normalised_and_reproduces_the_periodic_factor(l):
    ks, p = spectral.periodic_pmf(l)
    assert abs(p.sum() - 1.0) <= 1e-15
    assert np.array_equal(ks, -ks[::-1]) and np.all(p >= 0) and np.array_equal(p, p[::-1])
    K = ks[-1]
    assert 2 * scipy.special.ive(np.arange(K + 1, K + 400), 1.0 / l ** 2).sum() < spectral.PERIODIC_PMF_TAIL
    t = np.linspace(-1.5, 1.5, 4001)
    series = (p[:, None] * np.cos(2 * np.pi * ks[:, None] * t[None, :])).sum(axis=0)
    assert np.abs(series - np.exp(-2.0 * np.sin(np.pi * t) ** 2 / l ** 2)).max() <= 1e-14


def test_inverse_cdf_equals_independent_searchsorted():
    u = np.random.RandomState(3).uniform(0, 1, (500, 5))
    u[0, :3] = [0.0, 0.5, np.nextafter(1.0, 0.0)]
    for l in (0.05, 0.26, 1.0):
        ks, p = spectral.periodic_pmf(l)
        cdf = np.cumsum(p)
        ref = np.array([ks[min(int(np.argmax(cdf > v)) if (cdf > v).any() else len(ks) - 1, len(ks) - 1)] for v in u.ravel()])
        assert np.array_equal(spectral.periodic_frequencies(u, l).ravel(), ref)


def test_generate_basis_consumes_global_stream_in_order():
    """Hsampler.generate_basis for camphor: uniforms (F, 5) for the periodic columns, normals (F) for coordinate 2, then b"""
    F = 300
    h = _hsampler(6, F, [0.01, LS_ARD, 0.7])
    np.random.seed(11)
    h.generate_basis()
    after = np.random.get_state()
    np.random.seed(11)
    u = np.random.uniform(0, 1, (F, 5))
    z = np.random.randn(F)
    b = np.random.uniform(low=0, high=2 * np.pi, size=F)[:, None]
    ref = np.random.get_state()
    assert after[0] == ref[0] and np.array_equal(after[1], ref[1]) and after[2:] == ref[2:]
    assert np.array_equal(h.b, b)
    W = np.empty((F, 6))
    W[:, PERIODIC] = 2 * np.pi * spectral.periodic_frequencies(u, LS_ARD[0])
    W[:, 2] = z / (LS_ARD[2] + 0.05)
    assert np.array_equal(h.W, W)
    assert spectral.periodic_mask("camphor_copper_kernel") == MASK
    for other in ("SE_kernel", "RQ_kernel", "Matern32_kernel", "Matern52_kernel"):
        assert spectral.periodic_mask(other) == 0


@pytest.mark.parametrize("ls", [0.26, LS_ARD], ids=["iso", "ard"])
def test_feature_gram_matches_kernel(ls):
    """E[phi(x)' phi(y)] = k(x, y): on 400 pairs (across the seam, along coordinate 2, along two periodic coordinates, random) the
    feature product of F = 2e5 features is within 4 / sqrt(F) sf^2 of the kernel"""
    F, sf = 200000, 0.7
    W, b = spectral.draw_rff_basis("camphor_copper_kernel", F, 6, ls, np.random.RandomState(1))
    X, Y = _pairs(np.random.RandomState(2), 400)
    got = (features(W, b, X, sf) * features(W, b, Y, sf)).sum(axis=0)
    ref = np.diag(camphor_ref(X, Y, ls, sf).numpy())
    assert np.abs(got - ref).max() <= 4.0 / np.sqrt(F) * sf * sf
    assert ref.std() > 0.1 * sf * sf                   # the pairs probe the kernel's range, not just its tails


def test_features_periodic_in_the_periodic_coordinates():
    W, b = spectral.draw_rff_basis("camphor_copper_kernel", 1000, 6, LS_ARD, np.random.RandomState(4))
    X = np.random.RandomState(5).rand(50, 6)
    base = features(W, b, X, 1.0)
    for d in range(6):
        Xs = X.copy()
        Xs[:, d] += 1.0
        diff = np.abs(features(W, b, Xs, 1.0) - base).max()
        if d in PERIODIC:
            assert diff <= 1e-12, d
        else:
            assert diff > 1e-3, d


def test_make_problem_camphor_basis():
    from ppbo_b200 import synthetic
    p = synthetic.make_problem("camphor6d", Q=30, F=400)
    assert p["W"].shape == (400, 6) and p["b"].shape == (400,)
    k = np.round(p["W"][:, PERIODIC] / (2 * np.pi))
    assert np.array_equal(p["W"][:, PERIODIC], 2 * np.pi * k)
    assert "W" not in synthetic.make_problem("camphor6d", Q=30)          # the config itself keeps F = 0
    q = synthetic.make_problem("camphor6d", Q=30)
    assert np.array_equal(q["X"], p["X"]) and np.array_equal(q["grids"], p["grids"])


# ----------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from ppbo_b200 import ops as _ops
    return _ops


def _np(t):
    return t.detach().cpu().numpy()


def _seam_points(rng, n):
    """points on [0,1]^6 with a third of the periodic coordinates on or next to the seam 0 = 1"""
    X = rng.rand(n, 6)
    sel = rng.rand(n, 6) < 1.0 / 3.0
    sel[:, 2] = False
    edge = rng.choice([0.0, 1.0, 1e-9, 1.0 - 1e-9, 0.004, 0.996], size=(n, 6))
    X[sel] = edge[sel]
    return X


def _materialised_mean(ops, X, ls, sf, alpha, Y):
    """the mean through the materialising path of ppbo_predict (tuning key 11: cross-covariance in the difference form + GEMV)"""
    from ppbo_b200 import _lib
    lib = _lib.load()
    N, P = X.shape[0], Y.shape[0]
    mu = torch.empty(P, dtype=torch.float64, device=X.device)
    ws = torch.empty(P * N + 64, dtype=torch.float64, device=X.device)
    lsh = np.ascontiguousarray(np.broadcast_to(np.asarray(ls, dtype=float), (6,)))
    lsp = lsh.ctypes.data_as(POINTER(c_double))
    lib.ppbo_set_tuning(11, 1)
    try:
        rc = lib.ppbo_predict(2, X.data_ptr(), N, 6, lsp, float(sf), 0.0, N, 0, alpha.data_ptr(), None, None, 0, None, 0,
                              Y.data_ptr(), P, 1, mu.data_ptr(), None, ws.data_ptr(), ws.numel() * 8,
                              torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
    finally:
        lib.ppbo_set_tuning(11, 0)
    assert rc == 0, lib.ppbo_last_error()
    return mu


@gpu
@pytest.mark.parametrize("ls", [0.26, LS_ARD], ids=["iso", "ard"])
@pytest.mark.parametrize("N", [26, 520, 5200])
def test_lifted_matvec(ops, N, ls):
    """camphor mean of ppbo_predict (lifted SE form, mat-vec mode) against the FP64 difference-form reference and against the
    materialising path, rows n1 across the 128-row tile edges, points on and across the seam:
    |mu - ref| <= 1e-12 sf^2 sum|alpha|"""
    rng = np.random.RandomState(N)
    sf = 0.7
    X = ops.to_dev(_seam_points(rng, N))
    alpha = ops.to_dev(rng.randn(N))
    bound = 1e-12 * sf * sf * float(alpha.abs().sum())
    for n1 in (1, 63, 64, 65, 127, 129, 6144, 20480):
        Yh = _seam_points(rng, n1)
        Yh[:min(n1, 8)] = _np(X[:min(n1, 8)])                   # coincident points: the largest entries
        Y = ops.to_dev(Yh)
        mu = ops.posterior_mean("camphor_copper_kernel", X, ls, sf, alpha, Y)
        ref = torch.cat([camphor_ref(Y[i:i + 4096], X, ls, sf) @ alpha for i in range(0, n1, 4096)])
        mat = _materialised_mean(ops, X, ls, sf, alpha, Y)
        assert float((mu - ref).abs().max()) <= bound, (n1, float((mu - ref).abs().max()), bound)
        assert float((mu - mat).abs().max()) <= bound, n1
        assert float((mat - ref).abs().max()) <= bound, n1


def _maximize(ops, W, b, sf, Om, X0, mask, max_iter=500, gtol=1e-9):
    return ops.rff_maximize(ops.to_dev(W), ops.to_dev(b), sf, ops.to_dev(Om), ops.to_dev(X0), max_iter=max_iter, gtol=gtol,
                            periodic_mask=mask)


MASK0_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rff_maximize", "mask0_parent.npz")


def rff_maximize_cases():
    """inputs of the mask-0 bit-identity test (recorded from the build before the periodic mask existed): the SE bases of the
    camel2d / hartmann6d goldens and a camphor basis, 16 random weight vectors, 8 starts each, two iteration limits"""
    from conftest import load_golden
    cases = []
    for name in ("camel2d", "hartmann6d"):
        g = load_golden(name)
        cases.append((name, g["rff_W"], g["rff_b"], g["theta"][2]))
    W, b = spectral.draw_rff_basis("camphor_copper_kernel", 500, 6, 0.26, np.random.RandomState(7))
    cases.append(("camphor", W, b, 0.1))
    out = []
    for name, W, b, sf in cases:
        rng = np.random.RandomState(len(name))
        Om = rng.randn(16, W.shape[0])
        X0 = rng.rand(16, 8, W.shape[1])
        X0[:, 0] = np.round(X0[:, 0])                       # starts on corners of the box
        for max_iter, gtol in ((500, 1e-9), (7, 0.0)):
            out.append(("%s_%d" % (name, max_iter), W, b, sf, Om, X0, max_iter, gtol))
    return out


@gpu
def test_maximize_mask0_bit_identical_to_box_maximiser(ops):
    z = np.load(MASK0_GOLDEN)
    for key, W, b, sf, Om, X0, max_iter, gtol in rff_maximize_cases():
        xb, fb = _maximize(ops, W, b, sf, Om, X0, 0, max_iter, gtol)
        assert np.array_equal(_np(xb), z[key + "_x"]), key
        assert np.array_equal(_np(fb), z[key + "_f"]), key


def _seam_function():
    """g(x) = sum_{d periodic} cos(2 pi (x_d - c_d)) + cos(3 (x_2 - 0.45)) as an RFF function (one feature per term, sf = 1):
    separable, so the maximum of a dense grid is the sum of the per-coordinate maxima of its 1-D grids.  c_0 = 0.985: started at
    x_0 = 0.03 the ascent runs into the seam; the maximum lies across it."""
    c = {0: 0.985, 1: 0.3, 3: 0.6, 4: 0.0, 5: 0.75}
    W = np.zeros((6, 6))
    b = np.zeros(6)
    for f, d in enumerate(PERIODIC):
        W[f, d] = 2 * np.pi
        b[f] = -2 * np.pi * c[d]
    W[5, 2], b[5] = 3.0, -3.0 * 0.45
    amp = np.sqrt(2.0 / 6)
    t = np.linspace(0, 1, 100001)
    grid_max = sum(np.cos(W[f, :].max() * t + b[f]).max() for f in range(6)) * amp
    return W, b, np.ones((1, 6)), grid_max, amp


@gpu
def test_maximize_wraps_across_the_seam(ops):
    W, b, Om, grid_max, amp = _seam_function()
    X0 = np.array([[[0.03, 0.2, 0.5, 0.5, 0.1, 0.8], [0.02, 0.5, 0.4, 0.7, 0.9, 0.6]]])
    xb, fb = _maximize(ops, W, b, 1.0, Om, X0, MASK)
    xb, fb = _np(xb)[0], float(_np(fb)[0])
    start = max(amp * np.cos(W @ x + b).sum() for x in X0[0])
    assert fb >= grid_max - 1e-9 and fb >= start
    assert abs(xb[0] - 0.985) < 1e-4 and np.all((xb >= 0) & (xb < 1))
    x0, f0 = _maximize(ops, W, b, 1.0, Om, X0, 0)            # the box maximiser from the same starts stops at the seam
    assert _np(x0)[0][0] == 0.0 and float(_np(f0)[0]) < grid_max - 1e-3


@gpu
def test_maximize_rejects_mask_beyond_D(ops):
    from ppbo_b200._lib import PPBOError
    W, b, Om, _, _ = _seam_function()
    with pytest.raises(PPBOError):
        _maximize(ops, W, b, 1.0, Om, np.zeros((1, 1, 6)), 1 << 6)


# ----------------------------------------------------------------------------------------------- run_iteration at the scaled shape
def _scaled_problem():
    from ppbo_b200 import synthetic
    return synthetic.make_problem("camphor6d", Q=200, S=32768, P=1024, F=1000)


def _run_steps(it, prob, Q0, steps, S, seed, overlap, cov, dev, batch=None):
    theta, m, name = prob["theta"], prob["m"], prob["kernel"]
    X = torch.from_numpy(prob["X"]).to(dev)
    W, b, grids = (torch.from_numpy(np.ascontiguousarray(prob[k])).to(dev) for k in ("W", "b", "grids"))
    saved = it.OVERLAP_SAMPLING
    out = []
    try:
        it.OVERLAP_SAMPLING = overlap
        state = it.IterationState(name, theta, 6, m, Q0 + steps, dev, W, b)
        for k in range(steps + 1):
            Q = Q0 + k
            if k == 0:
                d = {"X": X[:Q0 * (m + 1)].contiguous(), "W": W, "b": b, "grids": grids}
            else:
                d = {"block": X[(Q - 1) * (m + 1):Q * (m + 1)].contiguous(), "W": W, "b": b, "grids": grids}
            res = it.run_iteration(d, name, theta, Q, m, S, seed=seed, state=state, weight_covariance=cov, batch=batch)
            torch.cuda.synchronize()
            sums, gp, rff = res[:3]
            out.append(dict(sums=sums.clone(), omega=rff.omega_map.clone(), hd=rff.hess_diag.clone(), alpha=gp.alpha.clone(),
                            fmap=gp.f_map.clone(), L=None if rff.L is None else rff.L.clone(), pick=None if batch is None else res[3]))
    finally:
        it.OVERLAP_SAMPLING = saved
    return out


def _reference(prob, Q, step, S, seed, cov, dev):
    """FP64 sums of the sampled maxima on the same Philox normals, from the device's weight-space optimum (and, for the full
    covariance, the host Cholesky of the host-formed exact Hessian there); mu* from the device alpha with the difference-form kernel"""
    from oracle import ppbo_oracle as O
    from test_weight_covariance import hessian_full, sample_omega_full
    m, theta, F = prob["m"], prob["theta"], prob["F"]
    Xh = prob["X"][:Q * (m + 1)]
    w = _np(step["omega"])
    Z = O.philox_normals(seed, 0, 0, S * F).reshape(S, F)
    if cov == "full":
        PhiX = O.rff_features(prob["W"], prob["b"], Xh, theta[2])
        Om = sample_omega_full(w, -hessian_full(w, PhiX, Q, m, theta[0]), Z)
    else:
        Om = w[None, :] + Z / np.sqrt(-_np(step["hd"]))[None, :]
    Om = torch.from_numpy(Om).to(dev)
    X = torch.from_numpy(Xh).to(dev)
    mustar = float(step["fmap"].max())
    fmax, gap, arg = [], [], []
    for g in prob["grids"]:
        G = torch.from_numpy(g).to(dev)
        mustar = max(mustar, float((camphor_ref(G, X, theta[1], theta[2]) @ step["alpha"]).max()))
        Fs = Om @ torch.from_numpy(O.rff_features(prob["W"], prob["b"], g, theta[2])).to(dev)
        top2 = Fs.topk(2, dim=1)
        fmax.append(top2.values[:, 0])
        gap.append(top2.values[:, 0] - top2.values[:, 1])
        arg.append(top2.indices[:, 0])
    fmax = torch.stack(fmax)
    sums = torch.stack([(fmax - mustar).clamp(min=0).sum(dim=1), fmax.sum(dim=1), (fmax * fmax).sum(dim=1)], dim=1)
    return _np(sums), _np(fmax), mustar


@gpu
@pytest.mark.parametrize("cov", ["diag", "full"])
def test_run_iteration_camphor_scaled(ops, cov):
    """N = 5200, D = 6 lines of P = 1024, S = 32768, F = 1000: cold and three appended iterations; overlapped and sequential
    schedules bit-identical at every step, sums against the FP64 reference 1e-9 relative, q = 2 picks equal to the FP64 greedy
    selection on the device's per-sample maxima"""
    from ppbo_b200 import iteration as it
    from test_batch_queries import batch_qei_greedy
    prob = _scaled_problem()
    assert (prob["N"], prob["X"].shape[1], prob["grids"].shape[0]) == (5200, 6, 6)
    S, steps, seed = prob["S"], 3, 3
    Q0 = prob["Q"] - steps
    dev = torch.device("cuda", torch.cuda.current_device())
    ov = _run_steps(it, prob, Q0, steps, S, seed, True, cov, dev, batch=2)
    sq = _run_steps(it, prob, Q0, steps, S, seed, False, cov, dev, batch=2)
    for k in range(steps + 1):
        assert torch.equal(ov[k]["sums"], sq[k]["sums"]), k
        assert torch.equal(ov[k]["pick"][0], sq[k]["pick"][0]) and torch.equal(ov[k]["pick"][1], sq[k]["pick"][1]), k
        ref, fmax_ref, mustar = _reference(prob, Q0 + k, ov[k], S, seed, cov, dev)
        got = _np(ov[k]["sums"])
        for c in range(3):
            assert np.abs(got[:, c] - ref[:, c]).max() <= 1e-9 * np.abs(ref[:, c]).max(), (k, c)
        idx_ref, _ = batch_qei_greedy(fmax_ref, mustar, 2)
        assert np.array_equal(_np(ov[k]["pick"][0]), idx_ref), k


@gpu
def test_sampled_argmax_camphor_scaled(ops):
    """per-sample arg-max of the INT8 contraction on the camphor operands equals the dense FP64 one wherever it is decided"""
    from oracle import ppbo_oracle as O
    from ppbo_b200 import iteration as it
    prob = _scaled_problem()
    S, seed, dev = prob["S"], 3, torch.device("cuda", torch.cuda.current_device())
    out = _run_steps(it, prob, prob["Q"], 0, S, seed, True, "diag", dev)[0]
    r = it.RFFFit()
    r.omega_map, r.hess_diag = out["omega"], out["hd"]
    W, b = torch.from_numpy(prob["W"]).to(dev), torch.from_numpy(prob["b"]).to(dev)
    PhiT = it.rff_grid_features(W, b, prob["theta"][2], torch.from_numpy(prob["grids"]).to(dev))
    assert it.sampling_engine(S, PhiT.shape[1], prob["F"]) == "i8"
    fmax, arg = it.rff_sampled_maxima(r, PhiT, 0, S, seed=seed)
    Z = torch.from_numpy(O.philox_normals(seed, 0, 0, S * prob["F"]).reshape(S, prob["F"])).to(dev)
    Om = out["omega"][None, :] + Z / torch.sqrt(-out["hd"])[None, :]
    for bl in range(PhiT.shape[0]):
        Fs = Om @ PhiT[bl].T
        top2 = Fs.topk(2, dim=1)
        scale = float(top2.values[:, 0].abs().max())
        decided = _np(top2.values[:, 0] - top2.values[:, 1]) > 1e-9 * scale
        assert decided.mean() > 0.99
        assert np.array_equal(_np(arg[bl])[decided], _np(top2.indices[:, 0])[decided]), bl
        assert float((fmax[bl] - top2.values[:, 0]).abs().max()) <= 1e-10 * scale, bl


@gpu
@pytest.mark.parametrize("form", ["diag", "full"])
def test_hsampler_end_to_end_camphor_golden(ops, form):
    """the reference's Hsampler flow on the camphor6d golden model: basis, features, MAP fit, covariance, sampled maxima over the
    query grids, and the batched maximiser with the periodic coordinates wrapped: finite, inside [0,1]^6, no worse than its starts"""
    from conftest import load_golden
    from random_fourier_sampler import Hsampler
    from test_src_gpu import _model
    g = load_golden("camphor6d")
    _, gp = _model(g)
    np.random.seed(0)
    h = Hsampler(gp, nFeatures=500)
    h.covariance_form = form
    h.generate_basis()
    assert h.W.shape == (500, 6)
    h.update_phi_X()
    h.update_omega_MAP()
    h.update_covariancematrix()
    assert np.all(np.isfinite(h.omega_MAP))
    rng = np.random.RandomState(1)
    grids = rng.rand(6, 64, 6)
    fmax = h.sample_max_over_grids(grids, 256, float(g["mustar"]))
    assert np.all(np.isfinite(_np(fmax) if torch.is_tensor(fmax) else np.asarray(fmax, dtype=float)))
    idx, qei = h.select_batch_over_grids(grids, 256, float(g["mustar"]), 2)
    assert len(set(np.asarray(idx).tolist())) == 2
    om = h.sample_omegas(8)
    om = _np(om) if torch.is_tensor(om) else np.asarray(om)
    seen = {}
    real = ops.rff_maximize

    def spy(*a, **kw):
        seen["X0"], seen["mask"] = _np(a[4]), kw.get("periodic_mask")
        return real(*a, **kw)
    ops.rff_maximize = spy
    try:
        xs, vals = h.return_xstar_batch(om, n_restarts=8)
    finally:
        ops.rff_maximize = real
    assert seen["mask"] == MASK
    assert np.all(np.isfinite(xs)) and np.all((xs >= 0) & (xs <= 1))
    amp = np.sqrt(2.0 * g["theta"][2] ** 2 / h.W.shape[0])
    for s in range(om.shape[0]):
        starts = np.clip(seen["X0"][s], 0, 1)
        f_start = (amp * np.cos(starts @ h.W.T + h.b.ravel()[None, :]) @ om[s]).max()
        f_x = amp * np.cos(h.W @ xs[s] + h.b.ravel()) @ om[s]
        assert vals[s] >= f_start - 1e-12 * max(1.0, abs(f_start)), s
        assert abs(f_x - vals[s]) <= 1e-12 * max(1.0, abs(vals[s])), s
