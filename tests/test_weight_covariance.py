"""Full Laplace covariance of the weight-space posterior (opt-in; the reference's is diagonal, src/random_fourier_sampler.py:134-137).

H = -grad^2 S(omega_MAP) = I + Psi' diag(a) Psi with the SIGNED coefficients a, H = L L':
    omega_s = omega_MAP + L^-T z_s ,   f_s(x_p) = mu_p + z_s . Phi~_p ,   mu_p = phi(x_p)' omega_MAP ,   Phi~ = Phi L^-T.
The FP64 references live here (the shared oracle is used unchanged): the dense signed Hessian, the biased INT8 arg-max
(ozaki_matmul + bias, bit-exact because the scales are powers of two) and the full-covariance draw.
Host tests pin the references; GPU tests hold the device factor, the draws, the biased contraction and run_iteration to them."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import scipy.linalg

from oracle import ppbo_oracle as O

torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ----------------------------------------------------------------------------------------------- FP64 references
def hessian_full(omega, PhiX, Q, m, sigma):
    """exact Hessian of S (dense F x F): -I - sum_u a_u d_u d_u', a = -Delta phi~(Delta) / (2 m sigma^2) signed, d_u = phi_j - phi_i"""
    f = PhiX.T @ omega
    Dl = O.deltas(f, Q, m, sigma)
    c = -0.5 * Dl * O.var2_normal_pdf(Dl) / (m * sigma ** 2)
    d = O._rff_diffs(PhiX, Q, m).reshape(PhiX.shape[0], -1)
    return -np.eye(PhiX.shape[0]) - (d * c.ravel()) @ d.T


def sample_omega_full(omega_map, precision, Z):
    """omega_map + Z L^-1 with precision = L L'"""
    L = np.linalg.cholesky(precision)
    return omega_map[None, :] + scipy.linalg.solve_triangular(L, Z.T, lower=True, trans='T').T


def ozaki_eval_argmax_bias(A, Bm, slices, bias):
    Fs = O.ozaki_matmul(A, Bm, slices) + bias[None, :]
    return Fs.max(axis=1), Fs.argmax(axis=1).astype(np.int32), Fs


def _fit_problem(name, **kw):
    """synthetic problem, its design features and a host weight-space optimum (Newton with the clamped Hessian, as the device fit)"""
    from ppbo_b200 import synthetic
    p = synthetic.make_problem(name, **kw)
    PhiX = O.rff_features(p["W"], p["b"], p["X"], p["theta"][2])
    return p, PhiX


# ----------------------------------------------------------------------------------------------- host
def test_full_hessian_diagonal_is_reference_hess_diag():
    p, PhiX = _fit_problem("camel2d", Q=12, F=150)
    rng = np.random.RandomState(0)
    w = 0.5 * rng.randn(PhiX.shape[0])
    H = hessian_full(w, PhiX, p["Q"], p["m"], p["theta"][0])
    hd = O.rff_S_hess_diag(w, PhiX, p["Q"], p["m"], p["theta"][0])
    assert np.abs(np.diag(H) - hd).max() <= 1e-14 * np.abs(hd).max()
    assert np.abs(H - H.T).max() <= 1e-15 * np.abs(H).max()
    # the signed coefficients really are mixed here, so the exact Hessian is not the clamped one
    f = PhiX.T @ w
    Dl = O.deltas(f, p["Q"], p["m"], p["theta"][0])
    assert (Dl * O.var2_normal_pdf(Dl) > 0).any() and (Dl * O.var2_normal_pdf(Dl) < 0).any()


def test_biased_oracle_argmax_equals_dense_fp64():
    rng = np.random.RandomState(4)
    S, F, P = 400, 300, 150
    Z = rng.randn(S, F)
    Gt = 0.05 * rng.randn(P, F)
    mu = 0.3 * rng.randn(P)
    mx, am, Fs = ozaki_eval_argmax_bias(Z, Gt, 6, mu)
    ref = Z @ Gt.T + mu[None, :]
    tol = 1e-11 * np.abs(ref).max()
    assert np.abs(Fs - ref).max() <= tol
    idx = ref.argmax(axis=1)
    top = ref[np.arange(S), idx]
    r2 = ref.copy()
    r2[np.arange(S), idx] = -np.inf
    decided = top - r2.max(axis=1) > 4 * tol
    assert decided.mean() > 0.99
    assert np.array_equal(am[decided], idx[decided])
    # the offset is added after the exact power-of-two scaling: one rounding, the same bits as the plain sum
    assert np.array_equal(Fs, O.ozaki_matmul(Z, Gt, 6) + mu[None, :])


def test_host_rng_full_draw_equals_numpy_multivariate_normal():
    from random_fourier_sampler import legacy_mvn_draw
    rng = np.random.RandomState(5)
    F = 40
    A = rng.randn(F, F)
    cov = A @ A.T / F + 0.1 * np.eye(F)
    mean = rng.randn(F)
    np.random.seed(123)
    ref = np.random.multivariate_normal(mean, cov, size=7)
    st_ref = np.random.get_state()
    np.random.seed(123)
    got = legacy_mvn_draw(mean, cov, 7)
    st = np.random.get_state()
    assert np.abs(got - ref).max() <= 1e-12 * np.abs(ref).max()
    assert st[0] == st_ref[0] and np.array_equal(st[1], st_ref[1]) and st[2:] == st_ref[2:]


# ----------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from ppbo_b200 import ops as _ops
    return _ops


def _np(t):
    return t.detach().cpu().numpy()


def _device_fit(ops, p, PhiX):
    """device weight-space optimum of the problem (the omega the factor is taken at in the product path)"""
    Pd = ops.to_dev(PhiX)
    w, hd, st = ops.rff_fit(Pd, p["Q"], p["m"], p["theta"][0])
    assert st["info"] == 0
    return Pd, w, hd


@gpu
@pytest.mark.parametrize("name,kw", [("camel2d", {}), ("levy10d", {}), ("ackley20d", {}), ("levy10d", {"F": 1100, "Q": 30}),
                                     ("ackley20d", {"kernel": "Matern52_kernel", "Q": 60})])
def test_hessian_factor_matches_host_cholesky(ops, name, kw):
    """ppbo_rff_hessian_factor against the host Cholesky of the host-formed signed Hessian at the device optimum (1e-12 relative),
    at the camel2d / levy10d / bench shapes, across the 1024 block (F = 1100) and with a Matern-5/2 basis; the fit's factor cache
    is a different object (the clamped chord matrix)"""
    p, PhiX = _fit_problem(name, **kw)
    Q, m, sigma = p["Q"], p["m"], p["theta"][0]
    F = PhiX.shape[0]
    Pd, w, hd = _device_fit(ops, p, PhiX)
    wh = _np(w)
    H = -hessian_full(wh, PhiX, Q, m, sigma)
    Lh = np.linalg.cholesky(H)
    buf = ops.rff_hessian_factor_buffer(F, Pd.device)
    assert ops.rff_hessian_factor(Pd, Q, m, sigma, w, buf) == 0
    L, _ = ops.hessian_factor_views(buf, F)
    Ld = np.tril(_np(L))
    assert np.abs(Ld - Lh).max() <= 1e-12 * np.abs(Lh).max(), np.abs(Ld - Lh).max() / np.abs(Lh).max()
    assert np.abs(np.diag(H) + _np(hd)).max() <= 1e-12 * np.abs(np.diag(H)).max()
    if name == "ackley20d" and "kernel" not in kw:
        f = PhiX.T @ wh
        Dl = O.deltas(f, Q, m, sigma)
        assert (Dl * O.var2_normal_pdf(Dl) > 0).sum() > 100          # negative coefficients a: the clamped Hessian differs


@gpu
def test_full_draw_with_identity_normals_gives_inverse_hessian(ops):
    p, PhiX = _fit_problem("levy10d", Q=30)
    Q, m, sigma = p["Q"], p["m"], p["theta"][0]
    F = PhiX.shape[0]
    Pd, w, _ = _device_fit(ops, p, PhiX)
    buf = ops.rff_hessian_factor_buffer(F, Pd.device)
    assert ops.rff_hessian_factor(Pd, Q, m, sigma, w, buf) == 0
    Om = ops.rff_sample_omega_full(w, buf, F, Z=ops.to_dev(np.eye(F)))
    E = _np(Om) - _np(w)[None, :]
    Hinv = np.linalg.inv(-hessian_full(_np(w), PhiX, Q, m, sigma))
    assert np.abs(E.T @ E - Hinv).max() <= 1e-12 * np.abs(Hinv).max()
    # Philox draws: the oracle's normals through the same transform
    S = 300
    Z = O.philox_normals(9, 2, 5 * F, S * F).reshape(S, F)
    got = _np(ops.rff_sample_omega_full(w, buf, S, seed=9, stream_id=2, sample0=5))
    ref = sample_omega_full(_np(w), -hessian_full(_np(w), PhiX, Q, m, sigma), Z)
    assert np.abs(got - ref).max() <= 1e-12 * np.abs(ref).max()


@gpu
@pytest.mark.parametrize("S,F,sample0", [(128, 64, 0), (300, 1000, 0), (257, 333, 7), (8, 65, 1)])
def test_normal_slice_bit_identical(ops, S, F, sample0):
    dev = torch.device("cuda", torch.cuda.current_device())
    for slices in (5, 6, 7):
        Z = ops.normal_fill(42, 3, sample0 * F, S * F, dev).view(S, F)
        p0, s0 = ops.ozaki_slice(Z, 0, slices)
        p1, s1 = ops.ozaki_normal_slice(S, F, dev, seed=42, stream_id=3, sample0=sample0, slices=slices)
        assert torch.equal(s0, s1) and torch.equal(p0, p1)


def _biased_operands(S, F, P, B, seed):
    rng = np.random.RandomState(seed)
    Z = rng.randn(S, F)
    G = np.stack([0.04 * rng.randn(P, F) for _ in range(B)])
    mu = 0.2 * rng.randn(B, P)
    return Z, G, mu


def _rowmax_bias(ops, Z, G, mu, slices=6, want_full=True):
    S, F = Z.shape
    B, P, _ = G.shape
    ap, asc = ops.ozaki_slice(ops.to_dev(Z), 0, slices)
    bp, bsc = ops.ozaki_slice(ops.to_dev(G), 1, slices)
    err = torch.zeros(1, dtype=torch.int32, device=ap.device)
    out = ops.ozaki_rowmax(ap, asc, S, bp, bsc, P, B, F, slices, want_full=want_full, err=err, bias=ops.to_dev(mu))
    torch.cuda.synchronize()
    return [None if t is None else _np(t) for t in out]


@gpu
@pytest.mark.parametrize("slices", [5, 6, 7])
@pytest.mark.parametrize("S,F,P,B", [(128, 64, 64, 1), (300, 200, 100, 2), (129, 1000, 70, 3), (1000, 333, 257, 2)])
def test_rowmax_bias_bit_exact_vs_oracle(ops, slices, S, F, P, B):
    Z, G, mu = _biased_operands(S, F, P, B, seed=S + P)
    fmax, arg, full = _rowmax_bias(ops, Z, G, mu, slices)
    for b in range(B):
        mx, am, Fs = ozaki_eval_argmax_bias(Z, G[b], slices, mu[b])
        assert np.array_equal(full[b], Fs) and np.array_equal(fmax[b], mx) and np.array_equal(arg[b], am)


@gpu
def test_rowmax_bias_ties_groups_and_launch_shapes(ops):
    """planted ties (in one tile's two halves, across tiles, across column groups) resolve to the lowest column; column-group
    counts (tuning key 4) and reserved-SM launch shapes (key 14) give the same bits; the offset decides the arg-max where the
    products alone would not"""
    from ppbo_b200 import _lib
    S, F, P, B = 300, 128, 200, 3
    Z, G, mu = _biased_operands(S, F, P, B, seed=8)
    G[:] = G[0]
    mu[:] = 0.0
    G[0][5] = G[0][40] = G[0][70] = 3.0 * G[0][5]
    G[1][40] = G[1][70] = 3.0 * G[0][5]
    G[2][33] = G[2][199] = 3.0 * G[0][5]
    mu[0, [5, 40, 70]] = mu[1, [40, 70]] = mu[2, [33, 199]] = 0.25
    lib = _lib.load()
    outs = []
    for key, groups in ((0, 0), (-1, 0), (0, 2), (100, 4), (12, 1)):
        lib.ppbo_set_tuning(14, key)
        lib.ppbo_set_tuning(4, groups)
        try:
            outs.append(_rowmax_bias(ops, Z, G, mu))
        finally:
            lib.ppbo_set_tuning(14, 0)
            lib.ppbo_set_tuning(4, 0)
    for b, first in enumerate((5, 40, 33)):
        mx, am, Fs = ozaki_eval_argmax_bias(Z, G[b], 6, mu[b])
        assert (am == first).sum() > 20
        for fmax, arg, full in outs:
            assert np.array_equal(full[b], Fs) and np.array_equal(fmax[b], mx) and np.array_equal(arg[b], am)
    # an offset alone moves the arg-max: the bias is inside the max, not added to it
    mu2 = np.zeros((1, P))
    mu2[0, 150] = 1e3
    fmax, arg, _ = _rowmax_bias(ops, Z, G[:1], mu2, want_full=False)
    assert np.all(arg[0] == 150)


@gpu
def test_rowmax_bias_zero_equals_plain_rowmax(ops):
    S, F, P, B = 1000, 333, 257, 2
    Z, G, _ = _biased_operands(S, F, P, B, seed=1)
    fmax, arg, _ = _rowmax_bias(ops, Z, G, np.zeros((B, P)), want_full=False)
    f0, a0, _ = ops.rff_eval_argmax_i8(ops.to_dev(Z), ops.to_dev(G), slices=6)
    assert np.array_equal(fmax, _np(f0)) and np.array_equal(arg, _np(a0))


def _reference_sums(prob, Q, gp, w, S, seed):
    """FP64 host reference of the full-covariance sums on the same Philox normals: Omega = omega + Z L^-1 with L the host Cholesky
    of the host-formed exact Hessian at the device optimum w; mu* from the device GP fit's alpha (the GP side is tested elsewhere)"""
    m, theta = prob["m"], prob["theta"]
    N = Q * (m + 1)
    Xh = prob["X"][:N]
    PhiX = O.rff_features(prob["W"], prob["b"], Xh, theta[2])
    Hp = -hessian_full(w, PhiX, Q, m, theta[0])
    F = PhiX.shape[0]
    Z = O.philox_normals(seed, 0, 0, S * F).reshape(S, F)
    Omega = torch.from_numpy(sample_omega_full(w, Hp, Z)).cuda()
    alpha = _np(gp.alpha)
    mustar = float(_np(gp.f_map).max())
    fmax, gap = [], []
    for g in prob["grids"]:
        mustar = max(mustar, float((O.se_kernel(Xh, g, theta).T @ alpha).max()))
        Fs = Omega @ torch.from_numpy(O.rff_features(prob["W"], prob["b"], g, theta[2])).cuda()
        top2 = Fs.topk(2, dim=1).values
        fmax.append(top2[:, 0])
        gap.append(top2[:, 0] - top2[:, 1])
    fmax = torch.stack(fmax)
    sums = torch.stack([(fmax - mustar).clamp(min=0).sum(dim=1), fmax.sum(dim=1), (fmax * fmax).sum(dim=1)], dim=1)
    return _np(sums), _np(fmax), _np(torch.stack(gap)), Hp


def _cache_contents(rf, F):
    """what the weight-space fit defines in its factor cache: the lower factor, the inverted 128-blocks and, when the fit reports them
    valid, the 1024-block inverses Binv and BinvT (the padding doubles and the solves' scratch vector are never part of a result)"""
    from ppbo_b200 import _lib
    cache = rf.factor_cache
    nf = _lib.load().ppbo_factor_doubles(F)
    parts = [torch.tril(cache[:F * F].view(F, F)), cache[F * F:nf]]
    if rf.fit.stats.get("binv_cached", False):
        BI = 1024
        nbI = -(-F // BI)
        parts.append(cache[nf:nf + 2 * nbI * BI * BI])
    return torch.cat([t.reshape(-1) for t in parts]).clone()


def _run(it, prob, Q0, steps, S, seed, overlap, cov, dev):
    theta, m, name = prob["theta"], prob["m"], prob["kernel"]
    D = prob["X"].shape[1]
    X = torch.from_numpy(prob["X"]).to(dev)
    W, b, grids = (torch.from_numpy(np.ascontiguousarray(prob[k])).to(dev) for k in ("W", "b", "grids"))
    saved = it.OVERLAP_SAMPLING
    out = []
    try:
        it.OVERLAP_SAMPLING = overlap
        state = it.IterationState(name, theta, D, m, Q0 + steps, dev, W, b)
        for k in range(steps + 1):
            Q = Q0 + k
            if k == 0:
                d = {"X": X[:Q0 * (m + 1)].contiguous(), "W": W, "b": b, "grids": grids}
            else:
                d = {"block": X[(Q - 1) * (m + 1):Q * (m + 1)].contiguous(), "W": W, "b": b, "grids": grids}
            sums, gp, rff = it.run_iteration(d, name, theta, Q, m, S, seed=seed, state=state, weight_covariance=cov)
            torch.cuda.synchronize()
            F = rff.omega_map.shape[0]
            out.append(dict(sums=sums.clone(), omega=rff.omega_map.clone(), cache=_cache_contents(state.rff, F), gp=gp,
                            Lbuf=rff.L, L=None if rff.L is None else torch.tril(rff.L[:F * F].view(F, F)).clone()))
    finally:
        it.OVERLAP_SAMPLING = saved
    return out


@gpu
@pytest.mark.parametrize("name,kw,S,steps", [("levy10d", dict(Q=42, P=256, F=500), 4096, 2),
                                              ("ackley20d", dict(Q=202), None, 2)])
def test_run_iteration_full_covariance(ops, name, kw, S, steps):
    """run_iteration(weight_covariance="full"), cold and two appended iterations, on a reduced shape and at the bench shape:
    sums against the FP64 host reference on the same Philox normals (1e-9 relative), arg-max identical where decided,
    overlapped and sequential pipelines bit-identical, the exact-Hessian factor in its own buffer (the fit's factor_cache is
    bit-identical to that of a diagonal run)"""
    from ppbo_b200 import iteration as it
    from ppbo_b200 import synthetic
    prob = synthetic.make_problem(name, **kw)
    S = prob["S"] if S is None else S
    Q0 = prob["Q"] - steps
    dev = torch.device("cuda", torch.cuda.current_device())
    seed = 3
    full = _run(it, prob, Q0, steps, S, seed, True, "full", dev)
    seq = _run(it, prob, Q0, steps, S, seed, False, "full", dev)
    diag = _run(it, prob, Q0, steps, S, seed, True, "diag", dev)
    for k in range(steps + 1):
        assert torch.equal(full[k]["sums"], seq[k]["sums"]), k
        assert torch.equal(full[k]["L"], seq[k]["L"]), k
        assert torch.equal(full[k]["omega"], diag[k]["omega"]), k
        assert torch.equal(full[k]["cache"], diag[k]["cache"]), k        # the fit's chord factor is not the home of L
        assert not torch.equal(full[k]["sums"], diag[k]["sums"]), k
    Q = Q0 + steps
    ref, fmax_ref, gap, _ = _reference_sums(prob, Q, full[-1]["gp"], _np(full[-1]["omega"]), S, seed)
    got = _np(full[-1]["sums"])
    for c in range(3):
        assert np.abs(got[:, c] - ref[:, c]).max() <= 1e-9 * np.abs(ref[:, c]).max(), (c, np.abs(got[:, c] - ref[:, c]).max())
    # per-sample arg-max: the contraction itself on the iteration's operands against the dense FP64 one
    r = it.RFFFit()
    r.omega_map, r.L = full[-1]["omega"], full[-1]["Lbuf"]
    grids = torch.from_numpy(prob["grids"]).to(dev)
    PhiT = it.rff_grid_features(torch.from_numpy(prob["W"]).to(dev), torch.from_numpy(prob["b"]).to(dev), prob["theta"][2], grids)
    fmax, arg = it.rff_sampled_maxima(r, PhiT, 0, S, seed=seed, covariance="full")
    scale = np.abs(fmax_ref).max()
    assert np.abs(_np(fmax) - fmax_ref).max() <= 1e-10 * scale
    Z = O.philox_normals(seed, 0, 0, S * prob["F"]).reshape(S, prob["F"])
    Om = torch.from_numpy(sample_omega_full(_np(r.omega_map), -hessian_full(
        _np(r.omega_map), O.rff_features(prob["W"], prob["b"], prob["X"][:Q * (prob["m"] + 1)], prob["theta"][2]), Q, prob["m"],
        prob["theta"][0]), Z)).to(dev)
    decided = gap > 1e-9 * scale
    assert decided.mean() > 0.99
    for b in range(prob["grids"].shape[0]):
        am = _np((Om @ PhiT[b].T).argmax(dim=1))
        assert np.array_equal(_np(arg[b])[decided[b]], am[decided[b]]), b


@gpu
def test_levy10d_variance_closer_to_gp_than_diagonal(ops):
    """variance of the sampled function phi(x)' omega on the grid points, full covariance from the DEVICE factor against the GP's
    Laplace predictive variance (oracle): median ratio in [0.8, 1.25] and closer to 1 than the diagonal covariance's"""
    from ppbo_b200 import synthetic
    p = synthetic.make_problem("levy10d")
    X, Q, m, th = p["X"], p["Q"], p["m"], p["theta"]
    K = O.se_kernel(X, X, th)
    Sig = O.regularize_covariance(K, svd_roundtrip=False)
    f = O.fmap_tight(Sig, Q, m, th[0], np.zeros(X.shape[0]))
    Sinv = np.linalg.inv(Sig)
    Lam = O.create_Lambda(f, Q, m, th[0])
    post = np.linalg.inv(Sinv - Lam)
    G = p["grids"][:, ::32].reshape(-1, X.shape[1])
    _, Sp = O.mu_Sigma_pred(X, G, th, O.se_kernel, Sinv, f, post, svd_roundtrip=False)
    v_gp = np.diag(Sp)
    PhiX = O.rff_features(p["W"], p["b"], X, th[2])
    Pd, w, hd = _device_fit(ops, p, PhiX)
    F = PhiX.shape[0]
    buf = ops.rff_hessian_factor_buffer(F, Pd.device)
    assert ops.rff_hessian_factor(Pd, Q, m, th[0], w, buf) == 0
    L, _ = ops.hessian_factor_views(buf, F)
    Pg = O.rff_features(p["W"], p["b"], G, th[2])
    V = scipy.linalg.solve_triangular(np.tril(_np(L)), Pg, lower=True)
    v_full = (V * V).sum(axis=0)
    v_diag = (Pg * Pg / (-_np(hd))[:, None]).sum(axis=0)
    r_full, r_diag = np.median(v_full / v_gp), np.median(v_diag / v_gp)
    assert 0.8 <= r_full <= 1.25, r_full
    assert abs(np.log(r_full)) < abs(np.log(r_diag)), (r_full, r_diag)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


@gpu
def test_two_rank_full_covariance_equals_single_rank():
    """two ranks (the weight-space fit on rank 1 broadcasts L with omega_MAP and hess_diag): the sums of the per-sample maxima equal
    the one-rank run's, cold and after an appended comparison set"""
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "mgpu_weight_cov_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "MGPU_FULL_OK" in r.stdout
