"""The steady state: a model that grows by appended comparison sets, fit after fit, against references computed here in FP64.

An appended GP fit starts from the previous mode with the previous factor object (the bordered warm start of ppbo_laplace_fit),
grows that factor by the border rows when it ends, and keeps the 1024-block inverses of the factor's unchanged leading blocks
(`binv_cache` / `binv_state`) for the next fit.  An appended weight-space fit starts its chord steps on the factor (and block
inverses) the previous fit left in `RFFState.factor_cache`.  A chord iteration converges to the same fixed point with any factor,
so a wrongly grown factor or a stale block inverse leaves the mode right and only shows as slower contraction or a fall-back
factorisation.  The invariant checkers below therefore look at what one fit hands to the next, not only at the modes.

References never come from a ppbo_* entry point: the GP mode is tightened by the oracle's Newton iteration on f = Sigma beta(f)
(torch FP64 dense solves on the device at the bench size, numpy on the host below it), each from the previous REFERENCE mode padded
with its posterior mean; the weight-space mode by the reference's trust-exact from the previous reference, tightened by Newton with
the exact Hessian.
"""
import math

import numpy as np
import pytest

from conftest import load_oracle_full, relerr

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

BI, NB = 1024, 128          # block sizes of the 1024-block inverses and of the Cholesky's inverted diagonal blocks
BORDER_MAX = 64             # appended rows carried as a border (laplace.cu); more rows: the warm fit refactorises
F64 = torch.float64


def _np(t):
    return t.detach().cpu().numpy()


@pytest.fixture(scope="module")
def env():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from oracle import ppbo_oracle as O
    from ppbo_b200 import _lib, iteration, ops, synthetic
    return dict(O=O, lib=_lib.load(), it=iteration, ops=ops, syn=synthetic, dev=torch.device("cuda", torch.cuda.current_device()))


# ------------------------------------------------------------------------------------------------ invariant checkers
def _check_dinv(L, dinv, n, what):
    """every inverted 128 x 128 diagonal block of the factor tail inverts the matching diagonal block of L"""
    for b in range((n + NB - 1) // NB):
        j0 = b * NB
        jb = min(NB, n - j0)
        D = dinv[b * NB * NB:(b + 1) * NB * NB].view(NB, NB)[:jb, :jb]
        Lb = torch.tril(L[j0:j0 + jb, j0:j0 + jb])
        err = (D @ Lb - torch.eye(jb, dtype=F64, device=L.device)).abs().max().item()
        assert err <= 1e-10, "%s: inverted diagonal block %d off by %.3g" % (what, b, err)


def _check_blockinv(L, W, nbI, n, valid, what):
    """1024-block inverses (layout of linalg.cu blockinv_build: Binv, BinvT, Lpad, each nbI x 1024^2) of the factor L of order n:
    for every valid block J, Lpad_J is L_JJ's lower triangle padded with the identity, Binv_J Lpad_J = I and BinvT_J = Binv_J^T"""
    BB = BI * BI
    Binv = W[:nbI * BB].view(nbI, BI, BI)
    BinvT = W[nbI * BB:2 * nbI * BB].view(nbI, BI, BI)
    Lpad = W[2 * nbI * BB:3 * nbI * BB].view(nbI, BI, BI)
    eye = torch.eye(BI, dtype=F64, device=L.device)
    for J in range(valid):
        j0 = J * BI
        rows = min(BI, n - j0)
        ref = eye.clone()
        ref[:rows, :rows] = torch.tril(L[j0:j0 + rows, j0:j0 + rows])
        assert torch.equal(Lpad[J], ref), "%s: Lpad block %d is not L's diagonal block (identity padding)" % (what, J)
        err = (Binv[J] @ ref - eye).abs().max().item()
        assert err <= 1e-10, "%s: 1024-block inverse %d off by %.3g" % (what, J, err)
        assert torch.equal(BinvT[J], Binv[J].T), "%s: BinvT block %d is not the transpose of Binv" % (what, J)
        if rows < BI:                                              # padding of the last partial block: exactly the identity
            for name, X in (("Binv", Binv[J]), ("BinvT", BinvT[J])):
                assert torch.equal(X[rows:, :], eye[rows:, :]) and torch.equal(X[:, rows:], eye[:, rows:]), \
                    "%s: padding of %s block %d" % (what, name, J)


def check_gp_factor(gp, M_old=None, what="gp"):
    """Factor object and block-inverse cache that a GP fit leaves for the next one.  M_old: rows of the previous fit (an appended
    fit), None after a cold fit.  Reads the buffers directly: LaplaceFit.L / Lfac would rebuild the factor at the mode."""
    lap = gp.lap
    M, cap = lap.M, lap.cap
    assert lap.factor_state == 1, "%s: the fit left no factor for the next one (factor_state %d)" % (what, lap.factor_state)
    L = lap._Lfac[:cap * cap].view(cap, cap)[:M, :M]
    s = lap.sa_fac[:M]
    A = torch.eye(M, dtype=F64, device=L.device) + s[:, None] * lap.G[:M, :M] * s[None, :]
    Lt = torch.tril(L)
    err = (Lt @ Lt.T - A).abs().max().item()
    assert err <= 1e-12 * math.sqrt(M) * A.abs().max().item(), "%s: |L L' - (I + s G s)| = %.3g" % (what, err)
    _check_dinv(L, lap._Lfac[cap * cap:], M, what)
    state = (lap.binv_state[0], lap.binv_state[1])
    bordered = M_old is not None and lap.stats["border_rows"] > 0 and lap.stats["factorizations"] == 0
    if bordered:
        # built for the previous factor (M_old rows); the finalisation rewrote the rows from the last 128-boundary of M_old on
        assert state == ((M_old // NB) * NB, -(-M_old // BI)), "%s: binv_state %s after a bordered fit from %d rows" % (what, state, M_old)
        _check_blockinv(L, lap.binv_cache, state[1], M_old, state[0] // BI, what)
    elif state != (0, 0):                                         # (0, 0): the fit left no block inverses
        assert state == (M, -(-M // BI)), "%s: binv_state %s at M = %d" % (what, state, M)
        _check_blockinv(L, lap.binv_cache, state[1], M, state[1], what)
    return state


def check_rff_cache(env, cache, F, what="rff"):
    """factor of the weight-space Hessian in RFFState.factor_cache: [F x F lower factor | inverted 128-blocks | block inverses]"""
    L = cache[:F * F].view(F, F)
    _check_dinv(L, cache[F * F:], F, what)
    W = cache[env["lib"].ppbo_factor_doubles(F):]
    nbI = -(-F // BI)
    _check_blockinv(L, W, nbI, F, nbI, what)
    return L


# ------------------------------------------------------------------------------------------------ references
def _ref_omega(O, PhiX, Q, m, sigma, w0):
    """weight-space mode next to w0: Newton with the exact Hessian (make_full_fixtures.rff_tight) from w0.  After an append the
    exact Hessian at the previous mode can be indefinite (one set moves the mode of schedule A by 4x its size) and Newton runs off to
    a saddle; then the reference's trust-exact (diagonal Hessian) from w0 comes first, as for the committed fixtures.  The result
    must be a stationary point with a positive definite -Hessian (a local maximum of S)."""
    from oracle.make_full_fixtures import rff_tight
    F = PhiX.shape[0]
    D3 = O._rff_diffs(PhiX, Q, m).reshape(F, Q * m)

    def is_max(w):
        if not np.linalg.norm(O.rff_S_grad(w, PhiX, Q, m, sigma)) <= 1e-8 * max(1.0, np.abs(w).max()):
            return False
        a = O.arrow_coeffs(PhiX.T @ w, Q, m, sigma).ravel()
        try:
            np.linalg.cholesky(np.eye(F) + (D3 * a[None, :]) @ D3.T)
        except np.linalg.LinAlgError:
            return False
        return True
    w = rff_tight(PhiX, Q, m, sigma, w0, iters=10)          # (quadratic convergence from a start inside the basin)
    if not is_max(w):
        w_te, _ = O.rff_omega_map(PhiX, Q, m, sigma, w0)
        w = rff_tight(PhiX, Q, m, sigma, w_te)
        assert is_max(w), "weight-space reference is not a local maximum of S"
    return w


class TorchMode:
    """oracle.fmap_tight's Newton iteration on f = Sigma beta(f) with torch FP64 dense operations on the device (same formulas:
    W = -Lambda(f), f_new = Sigma (I + W Sigma)^-1 (W f + beta(f)))"""

    def __init__(self, Sigma, m, sigma):
        self.Sigma, self.m, self.sigma = Sigma, m, float(sigma)

    def parts(self, f, Q):
        m, s = self.m, self.sigma
        Fq = f.view(Q, m + 1)
        Dl = (Fq[:, 1:] - Fq[:, :1]) / s
        pdf = torch.exp(-0.25 * Dl * Dl) / math.sqrt(4.0 * math.pi)
        a = -0.5 * Dl * pdf / (m * s * s)
        ph = pdf / (s * m)
        beta = torch.cat([ph.sum(dim=1, keepdim=True), -ph], dim=1).reshape(-1)
        Wb = torch.zeros((Q, m + 1, m + 1), dtype=F64, device=f.device)
        Wb[:, 0, 0] = a.sum(dim=1)
        Wb[:, 0, 1:] = -a
        Wb[:, 1:, 0] = -a
        Wb[:, 1:, 1:] = torch.diag_embed(a)
        return Wb, beta

    def tight(self, f_start, Q, iters=60, tol=1e-13):
        N = Q * (self.m + 1)
        S = self.Sigma[:N, :N]
        f = f_start.clone()
        eye = torch.eye(N, dtype=F64, device=f.device)
        for _ in range(iters):
            Wb, beta = self.parts(f, Q)
            b = torch.bmm(Wb, f.view(Q, self.m + 1, 1)).reshape(-1) + beta
            WS = torch.bmm(Wb, S.reshape(Q, self.m + 1, N)).reshape(N, N)
            f_new = S @ torch.linalg.solve(eye + WS, b)
            step = (f_new - f).abs().max().item()
            f = f_new
            if step <= tol * max(1.0, f.abs().max().item()):
                break
        return f

    def pad(self, f_old, Q_old, Q_new):
        """previous mode, and its posterior mean Sigma[new, old] beta(f_old) on the appended rows (alpha = beta(f) at a mode)"""
        n0, n1 = Q_old * (self.m + 1), Q_new * (self.m + 1)
        _, beta = self.parts(f_old, Q_old)
        return torch.cat([f_old, self.Sigma[n0:n1, :n0] @ beta])


# ------------------------------------------------------------------------------------------------ per-fit checks
def _check_grown_matrices(env, gp, X, kernel, theta, Q, m):
    ops = env["ops"]
    N, M = Q * (m + 1), Q * m
    fresh = ops.gram_regularized(kernel, X[:N].contiguous(), theta[1], theta[2], env["it"].SHRINKAGE)
    assert torch.equal(gp.Sigma, fresh), "Sigma at Q = %d differs from a fresh build" % Q
    assert torch.equal(gp.lap.G[:M, :M], ops.diffspace_gram(fresh, Q, m)), "G at Q = %d differs from a fresh build" % Q


def _check_gp_mode(gp, f_ref, what):
    f = gp.f_map
    err = (f - f_ref).abs().max().item()
    assert err <= 1e-6 * f_ref.abs().max().item(), "%s: mode off by %.3g relative" % (what, err / f_ref.abs().max().item())
    Sa = gp.Sigma @ gp.alpha
    assert relerr(_np(Sa), _np(f)) < 1e-9, "%s: Sigma alpha != f" % what


def _check_rff_mode(env, r, w_ref, PhiX, Q, m, sigma, what):
    w = _np(r.omega_map)
    assert np.abs(w - w_ref).max() <= 1e-6 * np.abs(w_ref).max(), "%s: omega off by %.3g relative" % (
        what, np.abs(w - w_ref).max() / np.abs(w_ref).max())
    hd_ref = env["O"].rff_S_hess_diag(w, PhiX, Q, m, sigma)
    assert relerr(_np(r.hess_diag), hd_ref) <= 1e-12, "%s: hess_diag" % what


# ------------------------------------------------------------------------------------------------ 2. the bench's steady state
Q0, STEPS = 200, 13
# Weight-space fits of the sequence below, queries 201..213 (measured on a B200): factorisations and chord steps per appended fit.
# The factor kept from the previous fit is refreshed by a mid-fit factorisation in 6 of the 13 fits.
RFF_FACTORIZATIONS = [0, 1, 0, 0, 1, 0, 0, 1, 1, 1, 1, 0, 0]
RFF_CHORD_STEPS = [11, 9, 11, 13, 8, 10, 13, 8, 7, 11, 8, 10, 13]


def _steady_run(env, prob, S, seed, overlap, on_step=None):
    it, ops, dev = env["it"], env["ops"], env["dev"]
    kernel, theta, m = prob["kernel"], prob["theta"], prob["m"]
    B, P, D = prob["grids"].shape
    X = ops.to_dev(prob["X"])
    W, b, grids = ops.to_dev(prob["W"]), ops.to_dev(prob["b"]), ops.to_dev(prob["grids"])
    saved = it.OVERLAP_SAMPLING
    out = []
    try:
        it.OVERLAP_SAMPLING = overlap
        state = it.IterationState(kernel, theta, D, m, Q0 + STEPS, dev, W, b)
        n0 = Q0 * (m + 1)
        d = {"X": X[:n0].contiguous(), "W": W, "b": b, "grids": grids}
        for k in range(STEPS + 1):
            Q = Q0 + k
            if k > 0:
                d = {"block": X[(Q - 1) * (m + 1):Q * (m + 1)].contiguous(), "W": W, "b": b, "grids": grids}
            sums, gp, rff = it.run_iteration(d, kernel, theta, Q, m, S, seed=seed, state=state)
            torch.cuda.synchronize()
            out.append((sums.clone(), gp.f_map.clone(), rff.omega_map.clone()))
            if on_step is not None:
                on_step(k, Q, X, state, sums, gp, rff)
    finally:
        it.OVERLAP_SAMPLING = saved
    return out


def test_bench_steady_state_sequence(env):
    """Ackley-20D, queries 201..213 appended one at a time to the fitted 200-query model (bench.py steady_reset / steady_step), the
    overlapped one-GPU pipeline: after every fit the grown matrices, the factor objects and block-inverse caches handed to the next
    fit, both modes against references carried along the sequence, and the fit statistics; the sequential pipeline returns the same
    bits at every step; the last step's sampled acquisition against the FP64 contraction of the reference weight-space mode."""
    O, syn, ops = env["O"], env["syn"], env["ops"]
    prob = syn.make_problem("ackley20d", Q=Q0 + STEPS)
    fx = load_oracle_full("ackley20d")
    kernel, theta, m, Fdim = prob["kernel"], prob["theta"], prob["m"], prob["F"]
    sigma = theta[0]
    S, seed = int(fx["slice_samples"]), int(fx["seed"])
    Xh = prob["X"]
    Sigma_h = O.regularize_covariance(O.se_kernel(Xh, Xh, theta), svd_roundtrip=False)
    ref = TorchMode(ops.to_dev(Sigma_h), m, sigma)
    del Sigma_h
    # the torch reference itself: from the fixture's mode it must stay there
    f_ref = ref.tight(ops.to_dev(fx["f_tight"]), Q0)
    assert (f_ref - ops.to_dev(fx["f_tight"])).abs().max().item() <= 1e-9 * np.abs(fx["f_tight"]).max()
    w_ref = np.array(fx["omega_tight"])
    PhiX_all = O.rff_features(prob["W"], prob["b"], Xh, theta[2])
    refs = {}
    stats = []

    def on_step(k, Q, X, state, sums, gp, rff):
        nonlocal f_ref, w_ref
        N, M = Q * (m + 1), Q * m
        what = "Q = %d" % Q
        if k > 0:
            f_ref = ref.tight(ref.pad(f_ref, Q - 1, Q), Q)
            w_ref = _ref_omega(O, PhiX_all[:, :N], Q, m, sigma, w_ref)
        refs[k] = (f_ref, w_ref)
        _check_grown_matrices(env, gp, X, kernel, theta, Q, m)
        check_gp_factor(gp, M_old=None if k == 0 else M - m, what=what)
        _check_gp_mode(gp, f_ref, what)
        _check_rff_mode(env, rff, w_ref, PhiX_all[:, :N], Q, m, sigma, what)
        if rff.stats["binv_cached"]:
            check_rff_cache(env, state.rff.factor_cache, Fdim, what)
        st = gp.lap.stats
        stats.append((st["border_rows"], st["factorizations"], st["chord_steps"], rff.stats["factorizations"], rff.stats["chord_steps"]))
        if k > 0:
            assert st["converged"] == 1 and st["border_rows"] == m, (what, dict(st))
            if k >= 2:          # (the first append follows a cold fit, whose single factor is far from the mode: DESIGN.md 4)
                assert st["factorizations"] == 0 and 5 <= st["chord_steps"] <= 7, (what, dict(st))

    seq = _steady_run(env, prob, S, seed, True, on_step)
    plain = _steady_run(env, prob, S, seed, False)
    for k, (a, b_) in enumerate(zip(seq, plain)):
        for x, y, name in zip(a, b_, ("sums", "f_map", "omega_map")):
            assert torch.equal(x, y), "overlapped and sequential pipelines differ in %s at Q = %d" % (name, Q0 + k)
    # last step: the 2048-sample slice against the FP64 contraction of the reference omega, mu* from the reference mode
    Q = Q0 + STEPS
    N = Q * (m + 1)
    f_last, w_last = refs[STEPS]
    hd = O.rff_S_hess_diag(w_last, PhiX_all[:, :N], Q, m, sigma)
    Z = O.philox_normals(seed, 0, 0, S * Fdim).reshape(S, Fdim)
    Omega = ops.to_dev(O.rff_sample_omega(w_last, hd, Z))
    _, beta = ref.parts(f_last, Q)
    mustar = f_last.max().item()
    fmax = []
    for g in prob["grids"]:
        mustar = max(mustar, float((ops.to_dev(O.se_kernel(Xh[:N], g, theta)).T @ beta).max().item()))
        fmax.append((Omega @ ops.to_dev(O.rff_features(prob["W"], prob["b"], g, theta[2]))).max(dim=1).values)
    fmax = torch.stack(fmax)
    ref_sums = _np(torch.stack([(fmax - mustar).clamp(min=0).sum(dim=1), fmax.sum(dim=1), (fmax * fmax).sum(dim=1)], dim=1))
    got = _np(seq[-1][0])
    scale = float(fmax.abs().max().item())
    for c in range(3):
        assert np.abs(got[:, c] - ref_sums[:, c]).max() <= 1e-6 * max(np.abs(ref_sums[:, c]).max(), S * 1e-3 * scale), c
    it = env["it"]
    ei, _ = it.acquisition_values(got, S)
    ei_ref = ref_sums[:, 0] / S
    assert int(np.argmax(ei)) == int(np.argmax(ei_ref))
    assert np.abs(ei - ei_ref).max() <= 1e-6 * max(ei_ref.max(), 1e-300) + 1e-9 * scale
    # fit statistics of the appended weight-space fits
    rff_counts = [(s_[3], s_[4]) for s_ in stats[1:]]
    assert [c[0] for c in rff_counts] == RFF_FACTORIZATIONS and [c[1] for c in rff_counts] == RFF_CHORD_STEPS, \
        "(border rows, GP factorisations, GP chord steps, weight-space factorisations, chord steps) per fit: %s" % (stats,)


# ------------------------------------------------------------------------------------------------ 3. boundary schedules
ACKLEY_THETA = [0.09, 0.3, 0.5]
# name: D, m, theta, F, cold Q, comparison sets appended per fit
SCHEDULES = {
    # the 128 / 1024 edges of M and the border limit: M = 960 -> 1024 exactly in eight appends, 1032 (a second 1024-block), a border
    # of 64 rows (BORDER_MAX), 72 rows (the warm fit without a border), one more set
    "A": dict(D=20, m=8, theta=ACKLEY_THETA, F=1000, Q=120, appends=[1] * 8 + [1, 2, 8, 9, 1]),
    # F > 1024: two weight-space 1024-blocks and a second trip of every stride-1024 loop over F; M 1000 -> 1025 -> 1075 (border of
    # 50) -> 1150 (75 rows) -> 1175 (crosses 1152)
    "B": dict(D=20, m=25, theta=ACKLEY_THETA, F=1100, Q=40, appends=[1, 2, 3, 1]),
    # sharp likelihood (sigma = 1e-3): M 2000 -> 2025 -> 2050 (crosses 2048); the warm fits may fall back to a factorisation
    "C": dict(problem="levy10d", F=1000, Q=80, appends=[1, 1]),
    # Q > 1024 in every per-set loop of both fits (m = 1), F = 333 (not a multiple of 8), N = 2200 (not a multiple of 128)
    "D": dict(D=6, m=1, theta=ACKLEY_THETA, F=333, Q=1100, appends=[1, 1]),
}

# (GP, weight-space) factorisations per fit of each schedule, cold fit first (measured on a B200)
SCHEDULE_FACTORIZATIONS = {
    "A": [(1, 2), (1, 1), (0, 1), (0, 0), (0, 1), (0, 1), (0, 1), (0, 2), (0, 1), (0, 0), (0, 2), (0, 3), (3, 1), (0, 1)],
    "B": [(1, 2), (0, 1), (0, 3), (3, 3), (0, 1)],
    "C": [(6, 8), (3, 3), (1, 3)],
    "D": [(5, 4), (0, 0), (0, 0)],
}


def _schedule_problem(env, spec):
    syn = env["syn"]
    Q_end = spec["Q"] + sum(spec["appends"])
    if "problem" in spec:
        p = syn.make_problem(spec["problem"], Q=Q_end, F=spec["F"])
        return dict(X=p["X"], W=p["W"], b=p["b"], D=p["D"], m=p["m"], theta=p["theta"], kernel=p["kernel"], fixture=spec["problem"])
    X, _, _ = syn.make_design(spec["D"], Q_end, spec["m"], seed=0)
    rng = np.random.RandomState(1)
    W = rng.randn(spec["F"], spec["D"]) / spec["theta"][1]
    b = rng.uniform(0, 2 * np.pi, spec["F"])
    return dict(X=X, W=W, b=b, D=spec["D"], m=spec["m"], theta=spec["theta"], kernel="SE_kernel", fixture=None)


@pytest.mark.parametrize("name", sorted(SCHEDULES))
def test_boundary_schedule(env, name):
    """A persistent GP model and weight-space model grown by the sets of the schedule: after every fit the grown matrices, the
    factor object and block inverses handed on, the border statistics and both modes against host references (GP: the reference's
    trust-exact from zero at the cold size, then oracle.fmap_tight from the previous reference padded with its posterior mean;
    weight space: the reference's trust-exact from the previous reference, tightened by Newton with the exact Hessian)."""
    O, it, ops, dev = env["O"], env["it"], env["ops"], env["dev"]
    spec = SCHEDULES[name]
    p = _schedule_problem(env, spec)
    m, theta, kernel = p["m"], p["theta"], p["kernel"]
    sigma = theta[0]
    Xh = p["X"]
    Q_end = Xh.shape[0] // (m + 1)
    Sigma_h = O.regularize_covariance(O.se_kernel(Xh, Xh, theta), svd_roundtrip=False)
    PhiX_h = O.rff_features(p["W"], p["b"], Xh, theta[2])
    X, W, b = ops.to_dev(Xh), ops.to_dev(p["W"]), ops.to_dev(p["b"])
    gp = it.GPState(kernel, theta, p["D"], m, Q_end, dev)
    rf = it.RFFState(W, b, theta, m, Q_end)
    Q = spec["Q"]
    N = Q * (m + 1)
    if p["fixture"]:                    # the committed fixture holds exactly this cold reference (trust-exact from 0, tightened)
        fx = load_oracle_full(p["fixture"])
        f_ref, w_ref = np.array(fx["f_tight"]), np.array(fx["omega_tight"])
    else:
        f_te, _ = O.fmap_trust_exact(O.pd_inverse(Sigma_h[:N, :N]), Q, m, sigma, np.zeros(N))
        f_ref = O.fmap_tight(Sigma_h[:N, :N], Q, m, sigma, f_te)
        w_ref = _ref_omega(O, PhiX_h[:, :N], Q, m, sigma, np.zeros(spec["F"]))
    gp.cold(X[:N])
    r = rf.cold(X[:N])
    prev_M = None
    counts = []
    for step, q in enumerate([0] + spec["appends"]):
        if q:
            Q_old, Q = Q, Q + q
            n0, N = Q_old * (m + 1), Q * (m + 1)
            f_pad = np.concatenate([f_ref, Sigma_h[n0:N, :n0] @ O.lik_beta(f_ref, Q_old, m, sigma)])
            f_ref = O.fmap_tight(Sigma_h[:N, :N], Q, m, sigma, f_pad)
            w_ref = _ref_omega(O, PhiX_h[:, :N], Q, m, sigma, w_ref)
            gp.append(X[n0:N])
            r = rf.append(X[n0:N])
        torch.cuda.synchronize()
        M = Q * m
        what = "schedule %s, Q = %d (M = %d)" % (name, Q, M)
        st = dict(gp.lap.stats)
        if q:
            assert st["border_rows"] == (q * m if q * m <= BORDER_MAX else 0), (what, st)
        _check_grown_matrices(env, gp, X, kernel, theta, Q, m)
        check_gp_factor(gp, M_old=prev_M, what=what)
        _check_gp_mode(gp, ops.to_dev(f_ref), what)
        _check_rff_mode(env, r, w_ref, PhiX_h[:, :N], Q, m, sigma, what)
        if r.stats["binv_cached"]:
            check_rff_cache(env, rf.factor_cache, spec["F"], what)
        prev_M = M
        counts.append((st["factorizations"], r.stats["factorizations"]))
    # factorisations per fit (GP, weight space), cold fit first: a chord phase that stops contracting (a wrong iteration matrix or
    # acceptance test) shows here even though the modes stay right
    assert counts == SCHEDULE_FACTORIZATIONS[name], "(GP, weight-space) factorisations per fit: %s" % (counts,)


def test_weight_space_fit_below_feature_slices(env):
    """F = 7 < FV_SLICES = 8: the feature-sliced Phi' omega kernel has an empty slice; cold fit against the host optimum"""
    O, it, ops, syn = env["O"], env["it"], env["ops"], env["syn"]
    D, Q, m, F = 20, 40, 8, 7
    theta = ACKLEY_THETA
    Xh, _, _ = syn.make_design(D, Q, m, seed=0)
    rng = np.random.RandomState(2)
    Wh, bh = rng.randn(F, D) / theta[1], rng.uniform(0, 2 * np.pi, F)
    PhiX = O.rff_features(Wh, bh, Xh, theta[2])
    w_ref = _ref_omega(O, PhiX, Q, m, theta[0], np.zeros(F))
    r = it.rff_fit(ops.to_dev(Xh), ops.to_dev(Wh), ops.to_dev(bh), theta, Q, m, tol=1e-10)
    _check_rff_mode(env, r, w_ref, PhiX, Q, m, theta[0], "F = 7")

