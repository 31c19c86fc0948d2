"""The kernels that walk the comparison-set layout, against FP64 references written here in numpy / scipy.

Row q (m+1) of f is the winner of comparison set q and rows q (m+1) + 1 + j are its m pseudo-observations; u = q m + j indexes
the differences Delta_u = f[q (m+1) + 1 + j] - f[q (m+1)] and B (N x M, N = Q (m+1), M = Q m) is the incidence matrix with +1 at
the pseudo-observation and -1 at the winner of every column.  Every per-set kernel is one warp per set with a lane loop over j, so
the set size m is swept across the warp width (31, 32, 33, 63, 64, 65, 100) and the kernels that index u = q m + j see M on both
sides of the 128 and 256 tiles.  The predictive covariance is checked with planted signed coefficients: its exact Woodbury term
for the r < 0 coefficients at the shapes where its layout changes (r at the 128 edge, both 16-byte parities of the sub-buffers,
negatives at either end of the set range), and the case where the posterior precision is indefinite.

No reference goes through a ppbo_* entry point; modes are tightened with oracle.fmap_tight.  Device outputs with a capacity
(Sigma, G, Phi_X, the factor objects, Lambda, the evidence matrix) live in NaN-filled buffers whose leading dimension exceeds the
problem, and the NaNs outside the problem must keep their bits.
"""
import ctypes
import math

import numpy as np
import pytest
import scipy.special

from oracle import ppbo_oracle as O

U = 2.0 ** -53                       # unit roundoff of FP64
SIGMA = 0.5                          # likelihood noise of section A: a power of two, so Delta / sigma is exact
M_SWEEP = (1, 2, 31, 32, 33, 63, 64, 65, 100)
THETA = (0.09, 0.4, 1.0)             # (sigma, length-scale, sigma_f) of the SE designs of sections B-D
BORDER_MAX = 64                      # appended rows the warm fit carries as a border (laplace.cu)


def set_counts(m):
    """Q such that M = Q m lies on both sides of 128 and of 256"""
    return sorted({max(1, 127 // m), 128 // m + 1, max(1, 255 // m), 256 // m + 1})


# ------------------------------------------------------------------------------------------------ host references
def incidence(Q, m):
    """B [N x M]: column u = (q, j) has +1 at row q (m+1) + 1 + j and -1 at the winner row q (m+1)"""
    B = np.zeros((Q * (m + 1), Q * m))
    for q in range(Q):
        for j in range(m):
            B[q * (m + 1) + 1 + j, q * m + j] = 1.0
            B[q * (m + 1), q * m + j] = -1.0
    return B


def deltas(f, Q, m):
    F = np.asarray(f).reshape(Q, m + 1)
    return (F[:, 1:] - F[:, :1]).reshape(-1)


def lik_reference(f, Q, m, sigma):
    """the formulas of the header of laplace.cu for x = Delta / sigma:  Phi~(x) = erfc(-x/2) / 2,  phi~(x) = exp(-x^2/4) / sqrt(4 pi),
    a = -x phi~(x) / (2 m sigma^2) (signed arrow coefficient), beta = B g with g_u = -phi~(x_u) / (sigma m)"""
    x = deltas(f, Q, m) / sigma
    ph = np.exp(-0.25 * x * x) / math.sqrt(4.0 * math.pi)
    Phi = 0.5 * scipy.special.erfc(-0.5 * x)
    a = -0.5 * x * ph / (m * sigma * sigma)
    g = -ph / (sigma * m)
    beta = np.zeros(Q * (m + 1))
    beta.reshape(Q, m + 1)[:, 1:] = g.reshape(Q, m)
    beta.reshape(Q, m + 1)[:, 0] = -g.reshape(Q, m).sum(axis=1)
    return dict(x=x, ph=ph, Phi=Phi, a=a, g=g, beta=beta)


def planted_f(Q, m, seed=0):
    """f whose sets hold Delta = 0 exactly, +-2^-40 sigma, +-58 sigma (phi~ = 0 exactly, Phi~ saturated at 0 and 1) and dyadic
    values spread over +-40 sigma of both signs; the special values sit at lanes that move from set to set (lanes >= 32 too).
    Winners are multiples of 1/16 and every Delta / sigma is k / 64 or +-2^-40: f, Delta, Delta / sigma and (Delta / sigma)^2 are
    exact, so the only rounding the kernels and the references see is in the functions themselves."""
    rng = np.random.RandomState(seed)
    f = np.empty((Q, m + 1))
    for q in range(Q):
        pool = np.array([0.0, 2.0 ** -40, -(2.0 ** -40), 58.0 * (-1) ** q])
        if m >= pool.size:
            row = np.concatenate([pool, rng.randint(-40 * 64, 40 * 64 + 1, size=m - pool.size) / 64.0])
        else:
            row = np.roll(pool, -q)[:m]
        row = np.roll(row, (7 * q) % m)
        f[q, 0] = rng.randint(-64, 65) / 16.0
        f[q, 1:] = f[q, 0] + row * SIGMA
    return f.reshape(-1)


def dyadic_symmetric(n, rng, scale_bits=8):
    """symmetric matrix of multiples of 2^-scale_bits in [-1, 1]: every sum of a few of its entries is exact"""
    A = rng.randint(-(1 << scale_bits), (1 << scale_bits) + 1, size=(n, n)) / float(1 << scale_bits)
    return np.tril(A) + np.tril(A, -1).T


def se_design(Q, m, D=3, seed=0):
    return np.random.RandomState(seed).uniform(0.0, 1.0, (Q * (m + 1), D))


def reg_prior(X1, X2=None, theta=THETA):
    """regularised SE prior covariance (oracle closed form of the shrinkage, as the device applies it)"""
    if X2 is None:
        return O.regularize_covariance(O.se_kernel(X1, X1, theta), svd_roundtrip=False)
    return O.se_kernel(X1, X2, theta)


def neg_indices(r, placement, Q, m):
    """r consecutive indices u: from u = 0, ending at u = M - 1, starting at a set boundary (whole sets negative once r >= m) or
    straddling one"""
    M = Q * m
    if r == 0:
        return np.zeros(0, dtype=int)
    if placement == "u0":
        start = 0
    elif placement == "last":
        start = M - r
    elif placement == "set":
        start = min((Q // 3) * m, (M - r) // m * m)
    elif placement == "cross":
        start = min(max((Q // 2) * m - (r + 1) // 2, 0), M - r)
    else:
        raise ValueError(placement)
    return np.arange(start, start + r)


def planted_arrow(G, neg, seed=0, pos_scale=20.0, neg_scale=0.5):
    """signed coefficients: positives of up to pos_scale / lambda_max(G) and, on the indices `neg`, negatives of at most
    neg_scale / lambda_max(G) -- then diag(1 / |a_-|) - G[-, -] >= lambda_max(G) (2 - 1) I keeps the posterior precision positive
    definite with a margin, and I + G diag(a) is well conditioned"""
    rng = np.random.RandomState(seed)
    lmax = float(np.linalg.eigvalsh(G)[-1])
    a = rng.uniform(0.05, 1.0, G.shape[0]) * pos_scale / lmax
    a[neg] = -rng.uniform(0.1, 1.0, len(neg)) * neg_scale / lmax
    return a


def diffspace_covariance(Kss, D, G, a):
    """Sigma_p = reg(K**) - D diag(a) (I + G diag(a))^-1 D',  D = K*X B: the posterior covariance of the latent values at the
    prediction points for W = B diag(a) B' of any sign (push-through of K*X W (I + Sigma W)^-1 KX*); Kss [batch, P, P], D [batch P, M]"""
    batch, P, _ = Kss.shape
    A = np.eye(G.shape[0]) + G * a[None, :]
    Y = a[:, None] * np.linalg.solve(A, D.T)
    out = Kss.copy()
    for b in range(batch):
        out[b] -= D[b * P:(b + 1) * P] @ Y[:, b * P:(b + 1) * P]
    return out, float(np.linalg.cond(A))


def precision_covariance(Kss, Ks, Sigma, W):
    """the same covariance through the dense N x N posterior precision Sigma^-1 + W (W = B diag(a) B' is never invertible: every
    set's all-ones vector is in its null space)"""
    Si = np.linalg.inv(Sigma)
    Post = np.linalg.inv(Si + W)
    return Kss - Ks @ Si @ Ks.T + Ks @ Si @ Post @ Si @ Ks.T


def indefinite_threshold(G, a, j):
    """largest c for which a_j = -c keeps Sigma^-1 + W positive definite (all other a >= 0): 1 / c must exceed the variance of
    Delta_j under the positive coefficients, g = G_jj - G_j+ s (I + s G++ s)^-1 s G_+j, s = a+^1/2"""
    s = np.sqrt(np.maximum(a, 0.0))
    s[j] = 0.0
    A = np.eye(G.shape[0]) + s[:, None] * G * s[None, :]
    h = s * G[:, j]
    g = G[j, j] - h @ np.linalg.solve(A, h)
    return 1.0 / g


def sqrt_psd(S):
    w, V = np.linalg.eigh(S)
    return (V * np.sqrt(np.maximum(w, 0.0))) @ V.T


INDEFINITE_QM = (6, 4)


def indefinite_case(Q=INDEFINITE_QM[0], m=INDEFINITE_QM[1], seed=3):
    """design, Sigma, G and the index j of the planted negative coefficient; a_in / a_out put a_j at 1/2 / 2 times the threshold"""
    X = se_design(Q, m, seed=seed)
    Sigma = reg_prior(X)
    B = incidence(Q, m)
    G = B.T @ Sigma @ B
    a = planted_arrow(G, [], seed=seed)
    j = Q * m // 2 + 1
    c = indefinite_threshold(G, a, j)
    a_in, a_out = a.copy(), a.copy()
    a_in[j], a_out[j] = -0.5 * c, -2.0 * c
    return X, Sigma, B, G, a_in, a_out


# ------------------------------------------------------------------------------------------------ host checks of the constructions
@pytest.mark.parametrize("m", M_SWEEP)
def test_planted_differences_give_the_intended_signs(m):
    for Q in set_counts(m):
        f = planted_f(Q, m, seed=m)
        ref = lik_reference(f, Q, m, SIGMA)
        d, a = deltas(f, Q, m).reshape(Q, m), ref["a"].reshape(Q, m)
        live = ref["ph"].reshape(Q, m) > 0                  # at |Delta| = 58 sigma phi~ and a underflow to zero
        assert np.array_equal(np.sign(a[live]), -np.sign(d[live])), "a > 0 exactly where the pseudo-observation lies below its winner"
        assert np.all(a[d == 0.0] == 0.0) and np.all(a[~live] == 0.0)
        assert np.all(ref["ph"][np.abs(ref["x"]) == 58.0] == 0.0), "phi~ underflows to zero at |Delta| = 58 sigma"
        assert np.all(ref["Phi"][ref["x"] == 58.0] == 1.0) and np.all(ref["Phi"][ref["x"] == -58.0] == 0.0)
        if m >= 4:
            for q in range(Q):
                x = d[q] / SIGMA
                assert (x == 0.0).sum() >= 1 and (x == 2.0 ** -40).sum() >= 1 and (x == -(2.0 ** -40)).sum() >= 1, q
                assert (x > 1).any() and (x < -1).any(), q
        if m >= 40:
            assert np.abs(d / SIGMA).max() >= 58 and (np.abs(d / SIGMA) > 30).sum() >= Q


@pytest.mark.parametrize("r, placement", [(3, "u0"), (3, "last"), (6, "set"), (5, "cross")])
def test_difference_space_covariance_equals_dense_precision_form(r, placement):
    Q, m = 5, 3
    X = se_design(Q, m, seed=1)
    Xp = np.random.RandomState(2).uniform(0.0, 1.0, (7, X.shape[1]))
    Sigma = reg_prior(X)
    B = incidence(Q, m)
    G = B.T @ Sigma @ B
    a = planted_arrow(G, neg_indices(r, placement, Q, m), seed=r)
    Ks = reg_prior(Xp, X)
    Kss = reg_prior(Xp)[None]
    got, kappa = diffspace_covariance(Kss, Ks @ B, G, a)
    ref = precision_covariance(Kss[0], Ks, Sigma, B @ np.diag(a) @ B.T)
    # the dense form inverts Sigma (cond ~ 1e7 here): its own error dominates
    assert np.abs(got[0] - ref).max() <= 1e-6 * np.abs(Kss).max(), np.abs(got[0] - ref).max()
    assert kappa < 1e4


def test_planted_indefinite_case_is_indefinite_with_margin():
    X, Sigma, B, G, a_in, a_out = indefinite_case()
    S12 = sqrt_psd(Sigma)
    lam_in = np.linalg.eigvalsh(np.eye(len(Sigma)) + S12 @ B @ np.diag(a_in) @ B.T @ S12)[0]
    lam_out = np.linalg.eigvalsh(np.eye(len(Sigma)) + S12 @ B @ np.diag(a_out) @ B.T @ S12)[0]
    assert lam_out < -1e-3, lam_out
    assert lam_in > 1e-3, lam_in


# ------------------------------------------------------------------------------------------------ device helpers
@pytest.fixture(scope="module")
def env():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from ppbo_b200 import _lib, iteration, ops, synthetic
    return dict(torch=torch, lib=_lib.load(), ops=ops, it=iteration, syn=synthetic,
                dev=torch.device("cuda", torch.cuda.current_device()))


def nan_buffer(env, shape):
    shape = (shape,) if isinstance(shape, int) else shape
    return env["torch"].full(shape, float("nan"), dtype=env["torch"].float64, device=env["dev"])


def in_capacity(env, A, extra=(3, 5)):
    """host matrix -> view A [:n, :k] of a NaN-filled device buffer with `extra` more rows and columns"""
    n, k = A.shape
    buf = nan_buffer(env, (n + extra[0], k + extra[1]))
    buf[:n, :k] = env["torch"].as_tensor(A, device=env["dev"])
    return buf, buf[:n, :k]


def assert_nan_outside(buf, n, k, what):
    h = buf.detach().cpu().numpy()
    mask = np.ones(h.shape, dtype=bool)
    mask[:n, :k] = False
    bits = h.view(np.uint64)[mask]
    nan_bits = np.array([np.nan]).view(np.uint64)[0]
    assert np.all(bits == nan_bits), "%s: %d sentinel(s) outside the %d x %d problem were written" % (what, int((bits != nan_bits).sum()), n, k)


def _np(t):
    return t.detach().cpu().numpy()


def _p(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _stream(env):
    return ctypes.c_void_p(env["torch"].cuda.current_stream().cuda_stream)


def _ok(env, rc, what):
    assert rc == 0, "%s: rc %d (%s)" % (what, rc, env["lib"].ppbo_last_error().decode())


# ------------------------------------------------------------------------------------------------ A. element kernels over m
def _elem_tol(ref, k=16):
    """k ulp of the reference, with a floor at the bottom of the normal range: an exp or erfc that lands in the subnormals keeps
    fewer bits (two evaluations of at most a handful of roundings each, plus the last-ulp error of exp / erfc on either side)"""
    return k * U * np.abs(ref) + k * np.finfo(float).tiny


@pytest.mark.gpu
@pytest.mark.parametrize("m", M_SWEEP)
def test_lik_terms_and_set_sums(env, m):
    ops, torch = env["ops"], env["torch"]
    for Q in set_counts(m):
        f = planted_f(Q, m, seed=m)
        ref = lik_reference(f, Q, m, SIGMA)
        fd = ops.to_dev(f)
        s, beta, arrow = ops.lik_terms(fd, Q, m, SIGMA)
        sums = ops.lik_set_sums(fd, Q, m, SIGMA)
        torch.cuda.synchronize()
        what = "m = %d, Q = %d" % (m, Q)
        a, b = _np(arrow), _np(beta)
        assert np.all(np.abs(a - ref["a"]) <= _elem_tol(ref["a"])), "%s: arrow, worst %.3g ulp" % (
            what, np.max(np.abs(a - ref["a"]) / np.maximum(np.abs(ref["a"]), 1e-300)) / U)
        assert np.array_equal(np.signbit(a[ref["a"] != 0]), np.signbit(ref["a"][ref["a"] != 0])), what
        bp = b.reshape(Q, m + 1)[:, 1:].reshape(-1)
        assert np.all(np.abs(bp - ref["g"]) <= _elem_tol(ref["g"])), "%s: beta of the pseudo-observations" % what
        # winner rows: a warp sum of m terms -- at most m roundings on top of the per-term error
        abs_g = np.abs(ref["g"]).reshape(Q, m).sum(axis=1)
        bw = b.reshape(Q, m + 1)[:, 0]
        assert np.all(np.abs(bw - ref["beta"].reshape(Q, m + 1)[:, 0]) <= (m + 16) * U * abs_g + 16 * np.finfo(float).tiny), \
            "%s: beta of the winners" % what
        Phi_q = ref["Phi"].reshape(Q, m)
        ref_sums, abs_sums = Phi_q.sum(axis=1), np.abs(Phi_q).sum(axis=1)
        got = _np(sums)
        # m roundings of the warp sum on top of the per-term error of erfc: scipy's is up to 8 ulp on these arguments (against a
        # 120-bit evaluation), CUDA's is documented at 5
        assert np.all(np.abs(got - ref_sums) <= (m + 16) * U * abs_sums), "%s: set sums off by %.3g" % (
            what, np.abs(got - ref_sums).max())
        assert abs(float(_np(s)[0]) - ref_sums.sum()) <= (Q + m + 16) * U * abs_sums.sum(), "%s: likelihood sum" % what
        # lanes beyond m contribute nothing: changing every other set leaves a set's sum bit for bit
        f2 = f.reshape(Q, m + 1).copy()
        f2[1::2] = f2[1::2][:, ::-1] + 0.75
        sums2 = _np(ops.lik_set_sums(ops.to_dev(f2.reshape(-1)), Q, m, SIGMA))
        assert np.array_equal(sums2[0::2], got[0::2]), "%s: a set sum depends on another set's values" % what


def signed_coefficients(M, seed):
    rng = np.random.RandomState(seed)
    a = rng.randn(M)
    a[rng.rand(M) < 0.4] *= -1.0
    return a


@pytest.mark.gpu
@pytest.mark.parametrize("m", M_SWEEP)
def test_lambda_dense_and_evidence_matrix(env, m):
    lib, ops = env["lib"], env["ops"]
    rng = np.random.RandomState(100 + m)
    for Q in set_counts(m):
        N, M = Q * (m + 1), Q * m
        what = "m = %d, Q = %d" % (m, Q)
        a = signed_coefficients(M, seed=m + Q)
        B = incidence(Q, m)
        W = B @ np.diag(a) @ B.T
        Wabs = np.abs(B) @ np.diag(np.abs(a)) @ np.abs(B).T        # |B| |diag a| |B'|: scale of every entry's sum
        ad = ops.to_dev(a)
        # Lambda = -W: off the winner diagonal single products (exact); winner diagonal a sum of m terms
        Lbuf = nan_buffer(env, (N + 2, N + 7))
        _ok(env, lib.ppbo_lambda_dense(_p(ad), Q, m, _p(Lbuf), Lbuf.stride(0), _stream(env)), "ppbo_lambda_dense")
        L = _np(Lbuf)[:N, :N]
        assert np.all(np.abs(L + W) <= 2 * m * U * Wabs), "%s: Lambda" % what
        assert_nan_outside(Lbuf, N, N, what + ": Lambda")
        # I +- Sigma W for a symmetric Sigma of dyadic entries: each entry is a sum of at most m + 1 products
        Sbuf, S = in_capacity(env, dyadic_symmetric(N, rng))
        Sh = _np(S)
        bound = 4 * (m + 2) * U * (np.abs(Sh) @ Wabs)      # device and BLAS each within (m + 2) u; rounding to half-ulps
        for ref_sign, sign in ((0, 1.0), (1, -1.0)):
            Ebuf = nan_buffer(env, (N + 1, N + 9))
            _ok(env, lib.ppbo_evidence_matrix(_p(S), S.stride(0), Q, m, _p(ad), ref_sign, _p(Ebuf), Ebuf.stride(0), _stream(env)),
                "ppbo_evidence_matrix")
            E = _np(Ebuf)[:N, :N]
            ref = np.eye(N) + sign * (Sh @ W)
            err = np.abs(E - ref)
            assert np.all(err <= bound + 2 * U * np.abs(ref)), "%s, sign %+d: evidence matrix off by %.3g (worst ratio %.3g)" % (
                what, sign, err.max(), np.max(err / (bound + 2 * U * np.abs(ref) + 1e-300)))
            assert_nan_outside(Ebuf, N, N, what + ": evidence matrix")
        assert_nan_outside(Sbuf, N, N, what + ": Sigma")


@pytest.mark.gpu
@pytest.mark.parametrize("m", M_SWEEP)
def test_diffspace_gram_bit_exact_and_append(env, m):
    lib = env["lib"]
    rng = np.random.RandomState(200 + m)
    Qs = set_counts(m)
    Qmax = Qs[-1]
    Nmax, Mmax = Qmax * (m + 1), Qmax * m
    Sh = dyadic_symmetric(Nmax, rng)
    Sbuf, S = in_capacity(env, Sh)
    scratch = {}
    for Q in [0] + Qs:
        M = Q * m
        G = nan_buffer(env, (Mmax + 2, Mmax + 5))
        if Q:
            _ok(env, lib.ppbo_diffspace_gram(_p(S), S.stride(0), Q, m, _p(G), G.stride(0), _stream(env)), "ppbo_diffspace_gram")
            B = incidence(Q, m)
            ref = B.T @ Sh[:Q * (m + 1), :Q * (m + 1)] @ B           # dyadic entries: exact in any order
            assert np.array_equal(_np(G)[:M, :M], ref), "m = %d, Q = %d: G != B' Sigma B" % (m, Q)
        assert_nan_outside(G, M, M, "m = %d, Q = %d: G" % (m, Q))
        scratch[Q] = G
    for Q_old in [0] + Qs:
        for Q_new in Qs:
            if Q_new <= Q_old:
                continue
            G = scratch[Q_old].clone()
            _ok(env, lib.ppbo_diffspace_gram_append(_p(S), S.stride(0), Q_old, Q_new, m, _p(G), G.stride(0), _stream(env)),
                "ppbo_diffspace_gram_append")
            M = Q_new * m
            assert env["torch"].equal(G[:M, :M], scratch[Q_new][:M, :M]), "m = %d: G grown %d -> %d sets differs" % (m, Q_old, Q_new)
            assert_nan_outside(G, M, M, "m = %d: G grown %d -> %d sets" % (m, Q_old, Q_new))
    assert_nan_outside(Sbuf, Nmax, Nmax, "Sigma")


def weight_space_problem(Q, m, F, seed):
    """Phi_X [F x N] of a random Fourier basis with sigma_f^2 = sigma^2 / 4 (differences of O(sigma): signed a of both signs)
    and omega ~ N(0, I)"""
    rng = np.random.RandomState(seed)
    N, D = Q * (m + 1), 3
    X = rng.uniform(0, 1, (N, D))
    W = rng.randn(F, D) / 0.3
    b = rng.uniform(0, 2 * np.pi, F)
    sigma = 0.2
    Phi = O.rff_features(W, b, X, 0.5 * sigma)
    omega = rng.randn(F)
    return Phi, omega, sigma


def weight_space_reference(Phi, omega, Q, m, sigma):
    """f = Phi' omega; grad = -omega + Phi beta(f); hdiag = -1 - sum_u a_u d_u^2 and the signed Hessian I + Psi' diag(a) Psi with
    Psi[u] = Phi[:, r(u)] - Phi[:, w(u)]; plus the first-order sensitivities of a and g to an error in Delta"""
    F, N = Phi.shape
    f = Phi.T @ omega
    ref = lik_reference(f, Q, m, sigma)
    Fq = Phi.T.reshape(Q, m + 1, F)
    Psi = (Fq[:, 1:, :] - Fq[:, :1, :]).reshape(Q * m, F)
    a, x, ph = ref["a"], ref["x"], ref["ph"]
    ref["grad"] = -omega + Phi @ ref["beta"]
    ref["hdiag"] = -1.0 - (a[:, None] * Psi * Psi).sum(axis=0)
    ref["H"] = np.eye(F) + Psi.T @ (a[:, None] * Psi)
    ref["Psi"] = Psi
    ref["dg"] = np.abs(0.5 * x * ph) / (sigma * sigma * m)                          # |dg / dDelta|
    ref["da"] = np.abs(ph * (1.0 - 0.5 * x * x)) / (2.0 * m * sigma ** 3)          # |da / dDelta|
    eps_f = 2 * F * U * (np.abs(Phi.T) @ np.abs(omega))                            # error of the device f = Phi' omega
    eF = eps_f.reshape(Q, m + 1)
    ref["eps_delta"] = (eF[:, 1:] + eF[:, :1]).reshape(-1)
    return ref


@pytest.mark.gpu
@pytest.mark.parametrize("F", (96, 130))
@pytest.mark.parametrize("m", M_SWEEP)
def test_weight_space_per_set_kernels(env, m, F):
    ops, lib, torch = env["ops"], env["lib"], env["torch"]
    for Q in set_counts(m):
        what = "m = %d, Q = %d, F = %d" % (m, Q, F)
        N, M = Q * (m + 1), Q * m
        Phi, omega, sigma = weight_space_problem(Q, m, F, seed=m * 1000 + Q + F)
        ref = weight_space_reference(Phi, omega, Q, m, sigma)
        a, Psi = ref["a"], ref["Psi"]
        assert (a > 0).sum() > 0 and (a < 0).sum() > 0, what
        Pbuf, Pd = in_capacity(env, Phi, extra=(0, 6))
        od = ops.to_dev(omega)
        _, grad, hd = ops.rff_objective(Pd, Q, m, sigma, od, want_S=False)
        torch.cuda.synchronize()
        # gradient: N products summed, plus the first-order effect of the f error through g on both rows of every difference
        absPhi = np.abs(Phi)
        Fq = absPhi.T.reshape(Q, m + 1, F)
        pair = (Fq[:, 1:, :] + Fq[:, :1, :]).reshape(M, F)
        prop_g = pair.T @ (ref["dg"] * ref["eps_delta"])
        bound_g = 2 * (N + 16) * U * (absPhi @ np.abs(ref["beta"])) + U * np.abs(omega) + 2 * prop_g
        err = np.abs(_np(grad) - ref["grad"])
        assert np.all(err <= bound_g), "%s: gradient off by %.3g (worst ratio %.3g)" % (what, err.max(), np.max(err / bound_g))
        # Hessian diagonal: M terms a_u d_u^2
        ad2 = np.abs(a)[:, None] * Psi * Psi
        prop_h = (ref["da"] * ref["eps_delta"]) @ (Psi * Psi)
        bound_h = 2 * (M + 16) * U * ad2.sum(axis=0) + U + 2 * prop_h
        err = np.abs(_np(hd) - ref["hdiag"])
        assert np.all(err <= bound_h), "%s: Hessian diagonal off by %.3g (worst ratio %.3g)" % (what, err.max(), np.max(err / bound_h))
        # exact Hessian factor with signed a, in a factor object of leading dimension F + 3
        lam = np.linalg.eigvalsh(ref["H"])
        assert lam[0] > 0.05, "%s: construction: the signed Hessian must be positive definite (%.3g)" % (what, lam[0])
        ldl = F + 3
        Lbuf = nan_buffer(env, int(lib.ppbo_rff_hessian_factor_doubles(F, ldl)))
        wbytes = lib.ppbo_rff_hessian_factor_workspace_bytes(F, Q, m)
        ws = torch.empty(wbytes // 8 + 1, dtype=torch.float64, device=env["dev"])
        info = ctypes.c_int(-7)
        _ok(env, lib.ppbo_rff_hessian_factor(_p(Pd), Pd.stride(0), F, Q, m, float(sigma), _p(od), _p(Lbuf), ldl, _p(ws), wbytes,
                                             ctypes.byref(info), _stream(env)), "ppbo_rff_hessian_factor")
        assert info.value == 0, what
        Lfull = Lbuf[:F * ldl].view(F, ldl)
        L = np.tril(_np(Lfull)[:, :F])
        absPsi = np.abs(Psi)
        bound = (2 * (F + 1) * U * (np.abs(L) @ np.abs(L).T) + 2 * (M + 16) * U * (absPsi.T @ (np.abs(a)[:, None] * absPsi))
                 + 2 * absPsi.T @ ((ref["da"] * ref["eps_delta"])[:, None] * absPsi))
        err = np.abs(L @ L.T - ref["H"])
        assert np.all(err <= bound), "%s: |L L' - H| = %.3g (worst ratio %.3g)" % (what, err.max(), np.max(err / bound))
        assert_nan_outside(Lfull, F, F, what + ": Hessian factor")
        assert_nan_outside(Pbuf, F, N, what + ": Phi_X")


# ------------------------------------------------------------------------------------------------ B. the Laplace fit at large m
@pytest.mark.gpu
@pytest.mark.parametrize("m, Q", [(33, 4), (64, 3), (65, 3)])
def test_laplace_fit_and_single_set_border_at_large_m(env, m, Q):
    from test_steady_state import check_gp_factor
    ops, it, torch = env["ops"], env["it"], env["torch"]
    sigma = THETA[0]
    D = 4
    X, _, _ = env["syn"].make_design(D, Q + 1, m, seed=m)
    N0, N1 = Q * (m + 1), (Q + 1) * (m + 1)
    Xd = ops.to_dev(X)
    # cold ops.laplace_fit against the reference's trust-exact from zero, tightened by the oracle
    Sigma = ops.gram_regularized("SE_kernel", Xd[:N0].contiguous(), THETA[1], THETA[2], it.SHRINKAGE)
    Sh = _np(Sigma)
    f_te, _ = O.fmap_trust_exact(O.pd_inverse(Sh), Q, m, sigma, np.zeros(N0))
    f_ref = O.fmap_tight(Sh, Q, m, sigma, f_te)
    fit = ops.laplace_fit(Sigma, Q, m, sigma)
    torch.cuda.synchronize()
    assert fit.info == 0
    f = _np(fit.f_map)
    scale = np.abs(f_ref).max()
    assert np.abs(f - f_ref).max() <= 1e-9 * scale, "m = %d: cold mode off by %.3g relative" % (m, np.abs(f - f_ref).max() / scale)
    assert np.abs(Sh @ _np(fit.alpha) - f).max() <= 1e-9 * scale, "m = %d: Sigma alpha != f" % m
    assert np.array_equal(_np(fit.arrow), _np(ops.lik_terms(fit.f_map, Q, m, sigma)[2])), "arrow at the mode"
    # the same cold fit in a growing model, then one appended set: a border of m rows up to BORDER_MAX, a refactorisation above
    gp = it.GPState("SE_kernel", THETA, D, m, Q + 1, env["dev"])
    gp.cold(Xd[:N0].contiguous())
    torch.cuda.synchronize()
    check_gp_factor(gp, M_old=None, what="m = %d cold" % m)
    gp.append(Xd[N0:N1].contiguous())
    torch.cuda.synchronize()
    st = gp.lap.stats
    assert st["border_rows"] == (m if m <= BORDER_MAX else 0), (m, st)
    if m > BORDER_MAX:
        assert st["factorizations"] >= 1, st
    check_gp_factor(gp, M_old=Q * m, what="m = %d appended" % m)
    Sh1 = _np(gp.Sigma)
    # the reference's trust-exact from the padded previous mode, tightened: Newton on the fixed point alone can end on a saddle
    # of T here (it does for m = 65), so the reference is also checked to be a maximum (I + Sigma^1/2 W Sigma^1/2 > 0)
    f_pad = np.concatenate([f_ref, Sh1[N0:N1, :N0] @ O.lik_beta(f_ref, Q, m, sigma)])
    f_te1, _ = O.fmap_trust_exact(O.pd_inverse(Sh1), Q + 1, m, sigma, f_pad)
    f_ref1 = O.fmap_tight(Sh1, Q + 1, m, sigma, f_te1)
    S12, B1 = sqrt_psd(Sh1), incidence(Q + 1, m)
    a1 = lik_reference(f_ref1, Q + 1, m, sigma)["a"]
    assert np.linalg.eigvalsh(np.eye(N1) + S12 @ B1 @ np.diag(a1) @ B1.T @ S12)[0] > 0, "reference is not a maximum of T"
    f1 = _np(gp.f_map)
    scale = np.abs(f_ref1).max()
    assert np.abs(f1 - f_ref1).max() <= 1e-6 * scale, "m = %d: appended mode off by %.3g relative" % (
        m, np.abs(f1 - f_ref1).max() / scale)


# ------------------------------------------------------------------------------------------------ C. predictive covariance
def planted_fit(env, Sigma, Q, m, sigma, a, alpha, cap=None):
    """a LaplaceFit built without a fit: G = B' Sigma B from ppbo_diffspace_gram, planted signed coefficients and alpha; the factor
    at the mode is built on first read of Lfac (ppbo_laplace_refactor).  cap > M: G, the factor object and sa_fac in NaN-filled
    capacity buffers."""
    ops, lib = env["ops"], env["lib"]
    M = Q * m
    fit = ops.LaplaceFit()
    fit.Q, fit.m, fit.sigma = Q, m, float(sigma)
    if cap is None:
        fit.cap = fit.ldg = M
        fit.G = ops.diffspace_gram(Sigma, Q, m)
        fit._Lfac = env["torch"].empty(lib.ppbo_factor_doubles(M), dtype=env["torch"].float64, device=env["dev"])
        fit.sa_fac = env["torch"].empty(M, dtype=env["torch"].float64, device=env["dev"])
    else:
        fit.cap = fit.ldg = cap
        fit.G = nan_buffer(env, (cap, cap))
        _ok(env, lib.ppbo_diffspace_gram(_p(Sigma), Sigma.stride(0), Q, m, _p(fit.G), cap, _stream(env)), "ppbo_diffspace_gram")
        fit._Lfac = nan_buffer(env, int(lib.ppbo_factor_doubles(cap)))
        fit.sa_fac = nan_buffer(env, cap)
    fit.arrow, fit.alpha = ops.to_dev(a), ops.to_dev(alpha)
    fit.f_map, fit.stats, fit.info, fit.factor_state = None, {}, 0, 0
    fit.n_neg, fit._neg_idx, fit._neg_corr = 0, None, None
    fit.binv_cache, fit.binv_state = None, None
    return fit


def check_capacity_sentinels(fit, M, what):
    cap = fit.cap
    assert_nan_outside(fit.G, M, M, what + ": G")
    assert_nan_outside(fit._Lfac[:cap * cap].view(cap, cap), M, M, what + ": factor")
    assert_nan_outside(fit.sa_fac.view(1, cap), 1, M, what + ": sa_fac")


class PredictCase:
    """one design with its device Sigma and host references"""

    def __init__(self, env, Q, m, seed, X=None):
        self.Q, self.m, self.N, self.M = Q, m, Q * (m + 1), Q * m
        self.X = se_design(Q, m, D=3, seed=seed) if X is None else X
        self.Xd = env["ops"].to_dev(self.X)
        self.Sbuf, self.Sigma = in_capacity(env, np.zeros((self.N, self.N)), extra=(1, 4))
        env["ops"].gram_regularized("SE_kernel", self.Xd, THETA[1], THETA[2], env["it"].SHRINKAGE, out=self.Sigma)
        self.Sh = _np(self.Sigma)
        self.B = incidence(Q, m)
        self.G = self.B.T @ self.Sh @ self.B
        self.alpha = np.random.RandomState(seed + 1).randn(self.N)

    def reference(self, Xp, P, batch, a):
        Kss = (1.0 - O.SHRINKAGE) * np.stack([O.se_kernel(x, x, THETA) for x in Xp.reshape(batch, P, -1)]) + \
            O.SHRINKAGE * THETA[2] ** 2 * np.eye(P)[None]
        Ks = reg_prior(Xp, self.X)
        cov, kappa = diffspace_covariance(Kss, Ks @ self.B, self.G, a)
        return Ks @ self.alpha, np.abs(Ks) @ np.abs(self.alpha), cov, kappa, np.abs(Kss).max()


def check_prediction(env, case, fit, a, P, batch, seed, what):
    ops, torch = env["ops"], env["torch"]
    Xp = np.random.RandomState(seed).uniform(0.0, 1.0, (P * batch, case.X.shape[1]))
    mu, Sp = ops.predict("SE_kernel", case.Xd, THETA[1], THETA[2], env["it"].SHRINKAGE, fit, ops.to_dev(Xp), P, batch)
    torch.cuda.synchronize()
    mu_ref, mu_abs, cov_ref, kappa, kmax = case.reference(Xp, P, batch, a)
    assert kappa <= 1e4, "%s: construction: cond(I + G diag(a)) = %.3g" % (what, kappa)
    assert np.all(np.abs(_np(mu).reshape(-1) - mu_ref) <= 2 * (case.N + 4) * U * mu_abs + 1e-15 * np.abs(mu_ref).max()), \
        what + ": mean"
    Sp = _np(Sp)
    assert np.isfinite(Sp).all(), what + ": non-finite covariance"
    # Cholesky, triangular solves and products of length <= M + r are backward stable with errors of c n u relative to their
    # operands (n <= 600, n u <= 7e-14); the solve with I + G diag(a) amplifies them by at most its condition number kappa:
    # 1e-12 kappa max|reg(K**)| leaves a factor of about 10 above that estimate
    err = np.abs(Sp - cov_ref).max()
    assert err <= 1e-12 * kappa * kmax, "%s: covariance off by %.3g (bound %.3g, kappa %.3g)" % (what, err, 1e-12 * kappa * kmax, kappa)
    return err


PLACEMENTS = ("u0", "last", "set", "cross")
NEG_CASES = [(0, "none")] + [(r, p) for r in (1, 2, 127, 128, 129, 257) for p in PLACEMENTS]
GRIDS = [(P, batch) for P in (1, 63, 64, 65, 129) for batch in (1, 3)]


PREDICT_SETS = (62, 61)              # m = 5: M = 310 and 305


def factor_offset(r, M):
    """doubles in front of the r x r Woodbury factor in neg_corr: idx (r int32, padded to whole doubles), then Ht (r x M)"""
    return (r + 1) // 2 + r * M


def test_predictive_covariance_alignment_parities_covered():
    """both parities of the factor's offset inside neg_corr -- 16-byte aligned or not -- occur among the planted cases, for odd
    and for even r"""
    for rs in ([r for r, _ in NEG_CASES if r % 2], [r for r, _ in NEG_CASES if r and r % 2 == 0]):
        assert {factor_offset(r, Q * 5) % 2 for r in rs for Q in PREDICT_SETS} == {0, 1}


@pytest.fixture(scope="module")
def predict_cases(env):
    return {Q: PredictCase(env, Q, 5, seed=Q) for Q in PREDICT_SETS}


@pytest.mark.gpu
@pytest.mark.parametrize("r, placement", NEG_CASES, ids=["r%d-%s" % c for c in NEG_CASES])
def test_predictive_covariance_planted(env, predict_cases, r, placement):
    lib = env["lib"]
    for _, case in sorted(predict_cases.items()):
        Q, m, M = case.Q, case.m, case.M
        neg = neg_indices(r, placement, Q, m)
        a = planted_arrow(case.G, neg, seed=r + M)
        assert np.array_equal(np.flatnonzero(a < 0), neg)
        what = "r = %d (%s), M = %d, factor at an %s offset" % (r, placement, M, ("even", "odd")[factor_offset(r, M) % 2])
        fit = planted_fit(env, case.Sigma, Q, m, THETA[0], a, case.alpha)
        for P, batch in GRIDS:
            check_prediction(env, case, fit, a, P, batch, seed=P * 7 + batch, what="%s, P = %d, batch = %d" % (what, P, batch))
        assert fit.n_neg == r and list(fit._neg_idx[:r]) == list(neg), what
        if r:
            assert fit.neg_corr.numel() == lib.ppbo_neg_corr_doubles(M, r), what
        # the same fit in capacity buffers (cap > M)
        cap = M + 13
        fit_c = planted_fit(env, case.Sigma, Q, m, THETA[0], a, case.alpha, cap=cap)
        for P, batch in ((129, 3), (1, 1)):
            check_prediction(env, case, fit_c, a, P, batch, seed=P + batch, what="%s, cap %d, P = %d, batch = %d" % (what, cap, P, batch))
        check_capacity_sentinels(fit_c, M, what)
        assert_nan_outside(case.Sbuf, case.N, case.N, what + ": Sigma")


@pytest.mark.gpu
@pytest.mark.parametrize("cap_extra", (0, 11))
def test_indefinite_posterior_precision_refused(env, cap_extra):
    ops, torch = env["ops"], env["torch"]
    X, _, _, _, _, _ = indefinite_case()
    Q, m = INDEFINITE_QM
    case = PredictCase(env, Q, m, seed=5, X=X)
    a = planted_arrow(case.G, [], seed=3)           # the construction of indefinite_case on the device Sigma
    j = Q * m // 2 + 1
    c = indefinite_threshold(case.G, a, j)
    cap = case.M + cap_extra if cap_extra else None
    # just inside the margin: a valid covariance that matches the reference
    a_in = a.copy()
    a_in[j] = -0.5 * c
    fit = planted_fit(env, case.Sigma, Q, m, THETA[0], a_in, case.alpha, cap=cap)
    check_prediction(env, case, fit, a_in, 33, 2, seed=9, what="a_j = -c / 2")
    # beyond it: neg_corr leaves info > 0, predict raises and returns nothing
    a_out = a.copy()
    a_out[j] = -2.0 * c
    fit = planted_fit(env, case.Sigma, Q, m, THETA[0], a_out, case.alpha, cap=cap)
    _ = fit.neg_corr
    torch.cuda.synchronize()
    assert fit.info > 0, "an indefinite posterior precision must leave info > 0"
    Xp = ops.to_dev(np.random.RandomState(4).uniform(0.0, 1.0, (33, 3)))
    with pytest.raises(ops.PPBOError, match="not positive definite"):
        ops.predict("SE_kernel", case.Xd, THETA[1], THETA[2], env["it"].SHRINKAGE, fit, Xp, 33, 1)
    if cap:
        check_capacity_sentinels(fit, case.M, "indefinite, cap %d" % cap)


# ------------------------------------------------------------------------------------------------ D. launch shapes
@pytest.mark.gpu
@pytest.mark.parametrize("batch", (1023, 1024, 1025))
def test_predict_rows_beyond_the_grid_limit(env, batch):
    """P batch = 65472, 65536, 65600 prediction rows: one per grid row would exceed the 65535 limit of gridDim.y"""
    ops = env["ops"]
    case = PredictCase(env, 4, 5, seed=11)
    P = 64
    a = planted_arrow(case.G, neg_indices(3, "cross", case.Q, case.m), seed=batch)
    fit = planted_fit(env, case.Sigma, case.Q, case.m, THETA[0], a, case.alpha)
    try:
        check_prediction(env, case, fit, a, P, batch, seed=batch, what="P = %d, batch = %d" % (P, batch))
    except ops.PPBOError as e:                  # a refusal must be an argument check with a message, not a failed launch
        assert "(-1)" in str(e) and "bad argument" in str(e), str(e)
