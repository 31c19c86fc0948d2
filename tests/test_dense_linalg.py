"""The dense FP64 linear algebra (GEMM and row-max GEMM, blocked Cholesky, triangular solves, LU log-determinant, evidence matrix)
against references that are EXACT in FP64.

Every input is built from small integers or dyadic fractions with power-of-two scale factors, small enough that every
intermediate sum of the operation stays below 2^53.  The exact result is then representable, the float64 numpy / scipy result
is exact too, and an indexing, tie, swap or tile-edge error shows up as a bit difference instead of hiding under a relative
tolerance of 1e-13.  Where the device arithmetic itself rounds (the Cholesky of a dense factor goes through inverted
128 x 128 blocks) the test states a c n u bound.

Capacity regions around every written block are filled with NaN sentinels and must keep their bits.

The constructions are checked on the CPU by the tests that are not marked `gpu`."""
import ctypes
import functools

import numpy as np
import pytest
import scipy.linalg as sla
from scipy.linalg.lapack import dpotrf

U = np.finfo(np.float64).eps / 2          # unit round-off
NAN_BITS = int(np.array(np.nan).view(np.int64))


# ============================================================================================= exact constructions (numpy)
def int_matrix(rng, shape, lim):
    """integers in [-lim, lim] as float64"""
    return rng.randint(-lim, lim + 1, size=shape).astype(np.float64)


def gemm_reference(A, B, C, alpha, beta):
    """alpha A B^T + beta C for integer A, B, C (|a|, |b| <= 2^8, K <= 2^12: every partial sum is an integer below 2^53, so the
    float64 product is exact in any summation order); beta == 0: C is not read"""
    P = A @ B.T
    return alpha * P if beta == 0.0 else alpha * P + beta * C


def chol_factor0(n, seed):
    """dense dyadic lower factor: diagonal 2^e (e in {-1, 0, 1}), entries below it m / 1024 with |m| <= 3.  A = L0 L0^T is exact
    in float64 (multiples of 2^-20 below 2^3), and numpy's unblocked Cholesky recovers L0 bit for bit; cond2(A) is about 20 at
    every size used here"""
    rng = np.random.RandomState(seed)
    L = np.tril(rng.randint(-3, 4, size=(n, n)).astype(np.float64) / 1024, -1)
    L[np.diag_indices(n)] = 2.0 ** rng.randint(-1, 2, size=n)
    return L


@functools.lru_cache(maxsize=4)
def chol_case(n, seed=0):
    L0 = chol_factor0(n, seed)
    return L0, L0 @ L0.T


@functools.lru_cache(maxsize=4)
def chol_conditions(n):
    """(cond_inf(L0), cond_inf(A)) of chol_case(n)"""
    L0, A = chol_case(n)
    Li = sla.solve_triangular(L0, np.eye(n), lower=True)
    return (np.abs(L0).sum(1).max() * np.abs(Li).sum(1).max(), np.abs(A).sum(1).max() * np.abs(Li.T @ Li).sum(1).max())


def semidefinite_case(n, k, kind, seed=0):
    """A = L diag(d) L^T whose leading minor k (1-based) is the first that is not positive definite, the bad pivot EMERGING from
    elimination: L is unit lower with entries m / 8 (|m| <= 4) only in rows of the parity of k - 1 and columns of the other
    parity (and L[k-1, k-2] = 3/2), so E = L - I has E E = 0 and every block inverse (I - E), Schur complement and pivot of any
    blocked elimination is exact; d_i in {1, 4}.  kind: 'zero' (d_{k-1} = 0), 'negative' (d_{k-1} = -1) or 'nan' (A[k-1, k-1] = NaN)."""
    rng = np.random.RandomState(seed + 7 * k)
    b = k - 1
    i, j = np.indices((n, n))
    mask = (j < i) & (i % 2 == b % 2) & (j % 2 != b % 2)
    L = np.eye(n) + np.where(mask, rng.randint(-4, 5, size=(n, n)) / 8.0, 0.0)
    if b > 0:
        L[b, b - 1] = 1.5                  # A[b, b] >= 2.25 - 1 > 0: the bad pivot is not on the diagonal of A itself
    d = 4.0 ** rng.randint(0, 2, size=n)
    if kind == "zero":
        d[b] = 0.0
    elif kind == "negative":
        d[b] = -1.0
    A = (L * d) @ L.T
    if kind == "nan":
        A[b, b] = np.nan
    return A, L, d


def lu_case(n, seed, permute=True, ties=()):
    """A = P^T L0 U0: L0 unit lower with entries m / 8, |m| <= 7 (|l| < 1 strictly, so partial pivoting picks the planted row at
    every step and recovers P, L0, U0 exactly), U0 upper with entries m / 8 and diagonal +-2^e, e in {-1, 0, 1}; every product
    and partial sum is a multiple of 2^-6 below 2^12.  ties: (row i, column k, +-1) entries |l_ik| = 1, i.e. rows i and k of
    the Schur complement tie in column k (use with permute=False: the first index -- the pivot row k -- must win).
    Returns A, L0, U0, perm (A = (L0 U0)[perm]), sum of the exponents e, sign of det U0."""
    rng = np.random.RandomState(seed)
    L = np.tril(int_matrix(rng, (n, n), 7) / 8, -1) + np.eye(n)
    for i, k, s in ties:
        L[i, k] = s
    Uu = np.triu(int_matrix(rng, (n, n), 8) / 8, 1)
    e = rng.randint(-1, 2, size=n)
    sgn = np.where(rng.rand(n) < 0.5, -1.0, 1.0)
    Uu[np.diag_indices(n)] = sgn * 2.0 ** e
    perm = rng.permutation(n) if permute else np.arange(n)
    return (L @ Uu)[perm], L, Uu, perm, int(e.sum()), float(np.prod(sgn))


def perm_sign(perm):
    """sign of a permutation (cycle count)"""
    seen = np.zeros(len(perm), dtype=bool)
    s = 1
    for i in range(len(perm)):
        if not seen[i]:
            j, c = i, 0
            while not seen[j]:
                seen[j] = True
                j = perm[j]
                c += 1
            s *= -1 if c % 2 == 0 else 1
    return s


def lapack_split(lu, piv):
    """(sign det U, sign of the row interchanges) of a scipy.linalg.lu_factor result"""
    d = np.diag(lu)
    return float(np.prod(np.sign(d))), (-1.0) ** int(np.sum(piv != np.arange(len(piv))))


# tie pairs of the row-max layout: every tile configuration has 32-column warp slices (WN = 32) and lane t4 owns the column pairs
# (2 t4, 2 t4 + 1) of each 8-column group, so (c, c+1) and (c, c+8) are ONE lane, (c, c+2) / (c, c+6) two lanes of one warp, (c, c+32)
# two WARPS_N warps at the same lane, (c, c+128) two column tiles at the same lane and warp (BN = 64 or 128)
def tie_pairs(P):
    pairs = [(10, 11), (16, 24), (34, 36), (41, 47), (5, 37), (30, 33), (62, 64), (70, 198), (100, 228), (3, P - 1)]
    return [(a, b) for a, b in pairs if b < P]


def rowmax_case(B, S, P, K, seed, shared=False, with_mu=True):
    """integer Z [B,S,K] (or [S,K] shared by the batch entries), Fac [B,P,K], mu [B,P] with planted exact ties.
    Coordinates t < T select tie pair t (both of its columns get 2^16, so they are the row's maximum, with equal values: the
    pair's second column copies the first's Fac row and mu); coordinate T carries mu, and a row with Z[s, T] = -1 and no other
    entry cancels mu exactly (every column ties at 0, expected arg-max 0); the remaining coordinates are noise in [-2, 2].
    Row s: s % (T + 2) < T selects a pair, == T is an all-tie row, == T + 1 is noise only."""
    pairs = tie_pairs(P)
    T = len(pairs)
    assert K >= T + 2
    rng = np.random.RandomState(seed)
    Fac = int_matrix(rng, (B, P, K), 2)
    mu = int_matrix(rng, (B, P), 64) if with_mu else np.zeros((B, P))
    Fac[:, :, :T] = 0.0
    for t, (a, b) in enumerate(pairs):
        Fac[:, a, t] = Fac[:, b, t] = 2.0 ** 16
        Fac[:, b, T + 1:] = Fac[:, a, T + 1:]
        mu[:, b] = mu[:, a]
    Fac[:, :, T] = mu
    Zs = int_matrix(rng, (1 if shared else B, S, K), 2)
    Zs[:, :, :T + 1] = 0.0
    for s in range(S):
        r = s % (T + 2)
        if r < T:
            Zs[:, s, r] = 1.0
        elif r == T:
            Zs[:, s, :] = 0.0
            Zs[:, s, T] = -1.0
    V = np.matmul(np.broadcast_to(Zs, (B, S, K)), Fac.transpose(0, 2, 1)) + mu[:, None, :]
    return (Zs[0] if shared else Zs), Fac, mu, V


def evidence_reference(Sigma, Q, m, arrow, reference_sign):
    """dense I + s Sigma B diag(a) B^T, s = -1 (reference_sign) or +1; B [N x Qm]: column (q, j) is e_w - e_{w+1+j}, w = q (m + 1)"""
    N, M = Q * (m + 1), Q * m
    Bm = np.zeros((N, M))
    for q in range(Q):
        for j in range(m):
            Bm[q * (m + 1), q * m + j] = 1.0
            Bm[q * (m + 1) + 1 + j, q * m + j] = -1.0
    W = (Bm * arrow) @ Bm.T
    return np.eye(N) + (-1.0 if reference_sign else 1.0) * (Sigma @ W)


# ============================================================================================= CPU checks of the constructions
def test_gemm_reference_is_exact():
    rng = np.random.RandomState(0)
    A, B, C = int_matrix(rng, (65, 4096), 256), int_matrix(rng, (33, 4096), 256), int_matrix(rng, (65, 33), 256)
    exact = A.astype(np.int64) @ B.astype(np.int64).T
    assert np.abs(exact).max() < 2 ** 53 and 256 * 256 * 4096 <= 2 ** 28
    assert np.array_equal(gemm_reference(A, B, C, 1.0, 0.0), exact.astype(np.float64))
    assert np.array_equal(gemm_reference(A, B, C, -0.5, 0.5), (-exact + C.astype(np.int64)) / 2.0)


@pytest.mark.parametrize("n", [33, 257])
def test_chol_construction_is_exact(n):
    L0, A = chol_case(n)
    Li = (L0 * 2048).astype(np.int64)                      # 2^11 L0 is an integer matrix
    assert np.array_equal(Li.astype(np.float64), L0 * 2048)
    assert np.array_equal(A * 2.0 ** 22, (Li @ Li.T).astype(np.float64))
    assert np.array_equal(np.linalg.cholesky(A), L0)       # the exact factor is L0
    d = np.log2(np.diag(L0))
    assert np.array_equal(d, np.round(d))


@pytest.mark.parametrize("k", [1, 2, 5, 33, 130, 300])
@pytest.mark.parametrize("kind", ["zero", "negative", "nan"])
def test_semidefinite_construction(k, kind):
    n = 300
    A, L, d = semidefinite_case(n, k, kind)
    E = L - np.eye(n)
    assert not np.any(E @ E)                               # E^2 = 0: (I + E)^-1 = I - E exactly
    assert np.array_equal(A, A.T, equal_nan=True)
    if kind != "nan":
        assert np.array_equal(A, ((L * 4 * d) @ (L * 8).T) / 32)         # exact
        Lf, info = dpotrf(A, lower=1)
        assert info == k
        Lk = L[:k - 1, :k - 1] * np.sqrt(d[:k - 1])
        assert np.array_equal(np.tril(Lf[:k - 1, :k - 1]), Lk)           # exact factor of the leading minor
        # the pivot emerges from elimination: the diagonal entry itself is positive unless there is nothing to eliminate
        assert A[k - 1, k - 1] > 0 or k == 1
    else:
        assert np.isnan(A[k - 1, k - 1]) and np.sum(np.isnan(A)) == 1


@pytest.mark.parametrize("n", [1, 65, 129, 1025])
def test_lu_construction_recovers_factors(n):
    A, L0, U0, perm, esum, sgn = lu_case(n, n)
    P, L, Uf = sla.lu(A)
    assert np.array_equal(L, L0) and np.array_equal(Uf, U0)
    assert np.array_equal(P.T @ A, L0 @ U0) and np.array_equal(np.argmax(P, axis=1), perm)
    lu, piv = sla.lu_factor(A)
    su, sp = lapack_split(lu, piv)
    assert su == sgn and sp == perm_sign(perm)
    assert np.log(np.abs(np.diag(U0))).sum() == pytest.approx(esum * np.log(2.0), abs=1e-12 * n)


def lu_ties(n):
    """|l_ik| = 1 planted for the pivot search of lu_panel_kernel (thread tid takes rows col + tid + 1024 j): the tied row i
    sits in another lane (i - k < 32), another warp, or in the same thread one 1024-stride later"""
    out = []
    for k in (0, 7, 64, 130, 700):
        for d, s in ((1, 1.0), (31, -1.0), (32, 1.0), (100, -1.0), (1024, 1.0), (1056, -1.0)):
            if k + d < n:
                out.append((k + d, k, s))
    return out


def test_lu_ties_are_real_ties():
    n = 2080
    A, L0, U0, perm, _, _ = lu_case(n, 5, permute=False, ties=lu_ties(n))
    lu, piv = sla.lu_factor(A)
    assert np.array_equal(piv, np.arange(n))               # first index on ties: the diagonal row wins, no interchange
    assert np.array_equal(np.tril(lu, -1) + np.eye(n), L0) and np.array_equal(np.triu(lu), U0)
    for i, k, s in lu_ties(n):                             # column k of the Schur complement at step k: rows k and i tie
        S = L0[k:, k:k + 1] * U0[k, k]
        assert abs(S[0, 0]) == abs(S[i - k, 0]) == np.abs(S).max()


def test_rowmax_construction_has_planted_ties():
    B, S, P, K = 2, 40, 257, 24
    Z, Fac, mu, V = rowmax_case(B, S, P, K, 1)
    pairs = tie_pairs(P)
    T = len(pairs)
    for s in range(S):
        r = s % (T + 2)
        if r < T:
            a, b = pairs[r]
            assert np.all(V[:, s, a] == V[:, s, b]) and np.all(V[:, s, a] == V[:, s].max(axis=1))
            assert np.all(V[:, s].argmax(axis=1) == a)
            assert np.all(np.sort(V[:, s], axis=1)[:, -3] < V[:, s, a])      # exactly two maxima
        elif r == T:
            assert np.all(V[:, s] == 0.0)
    assert np.abs(V).max() < 2 ** 20
    Zs, _, _, Vs = rowmax_case(3, 30, 1037, 1024, 2, shared=True)
    assert Zs.ndim == 2 and np.abs(Vs).max() < 2 ** 18


def test_evidence_reference_matches_entry_formula():
    rng = np.random.RandomState(0)
    Q, m = 3, 4
    N = Q * (m + 1)
    Sigma, a = int_matrix(rng, (N, N), 16) / 8, int_matrix(rng, Q * m, 8) / 8
    for ref_sign in (0, 1):
        E = evidence_reference(Sigma, Q, m, a, ref_sign)
        s = -1.0 if ref_sign else 1.0
        for i in range(N):
            for c in range(N):
                q, rc = divmod(c, m + 1)
                w = q * (m + 1)
                if rc == 0:
                    v = sum(a[q * m + j] * (Sigma[i, w] - Sigma[i, w + 1 + j]) for j in range(m))
                else:
                    v = a[q * m + rc - 1] * (Sigma[i, c] - Sigma[i, w])
                assert E[i, c] == (1.0 if i == c else 0.0) + s * v


# ============================================================================================= GPU
torch = None


@pytest.fixture(scope="module")
def ops():
    global torch
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from ppbo_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def lib(ops):
    from ppbo_b200 import _lib
    return _lib.load()


class tuning:
    """ppbo_set_tuning(key, value) for the duration of a with-block"""

    def __init__(self, lib, key, value):
        self.lib, self.key, self.value = lib, key, value

    def __enter__(self):
        self.lib.ppbo_set_tuning(self.key, self.value)

    def __exit__(self, *exc):
        self.lib.ppbo_set_tuning(self.key, 0)


def _np(t):
    return t.detach().cpu().numpy()


def _sentinel(*shape):
    return torch.full(shape, float("nan"), dtype=torch.float64, device="cuda")


def _dev(a):
    return torch.as_tensor(np.ascontiguousarray(a), device="cuda")


def _outside_untouched(buf, inside):
    """every element of buf outside the boolean mask `inside` still holds the sentinel's bits"""
    return bool(((buf.view(torch.int64) == NAN_BITS) | inside).all())


def _region(buf, r0, r1, c0, c1):
    m = torch.zeros(buf.shape, dtype=torch.bool, device=buf.device)
    m[r0:r1, c0:c1] = True
    return m


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


# --------------------------------------------------------------------------------------------- 1. GEMM
DIMS = (0, 1, 7, 8, 9, 63, 64, 65, 127, 128, 129, 257)
ALPHA_BETA = ((1.0, 0.0), (-1.0, 1.0), (0.5, -1.0), (0.0, 0.5), (1.0, 0.5), (-1.0, 0.0))


def _gemm_shapes():
    """every (M, N) of DIMS x DIMS, K walking through DIMS"""
    return [(M, N, DIMS[(5 * i + 7 * j) % len(DIMS)]) for i, M in enumerate(DIMS) for j, N in enumerate(DIMS)]


def _operand(X, layout, rows_pad=1):
    """device copy of X as a strided view: 'even' (even ld > K), 'odd' (odd ld) or 'offset' (8 bytes past a 16-byte boundary);
    everything around it is NaN, so a read past K or past the last row poisons the result"""
    M, K = X.shape
    if layout == "even":
        buf = _sentinel(M + rows_pad, K + 2 - K % 2)
        v = buf[:M, :K]
    elif layout == "odd":
        buf = _sentinel(M + rows_pad, K + 1 + K % 2)
        v = buf[:M, :K]
    else:
        buf = _sentinel(M + rows_pad, K + 3)
        v = buf[:M, 1:K + 1]
    v.copy_(_dev(X))
    return v


def _run_gemm(ops, cfg, M, N, K, alpha, beta, layout, seed):
    rng = np.random.RandomState(seed)
    A, B, C = int_matrix(rng, (M, K), 256), int_matrix(rng, (N, K), 256), int_matrix(rng, (M, N), 256)
    Ad, Bd = _operand(A, layout), _operand(B, layout)
    ldc = N + 1 + seed % 2                                   # odd and even ldc > N
    Cbuf = _sentinel(M + 2, ldc + 1)
    Cd = Cbuf[1:M + 1, 1:N + 1] if layout == "offset" else Cbuf[1:M + 1, :N]
    if beta != 0.0:
        Cd.copy_(_dev(C))                                    # beta == 0: C stays NaN (it must not be read)
    if cfg is None:
        ops.gemm_nt(Ad, Bd, Cd, alpha=alpha, beta=beta)
    else:
        ops.gemm_nt_cfg(cfg, Ad, Bd, Cd, alpha=alpha, beta=beta)
    ref = gemm_reference(A, B, C, alpha, beta)
    c0 = 1 if layout == "offset" else 0
    inside = _region(Cbuf, 1, M + 1, c0, c0 + N)
    return np.array_equal(_np(Cd), ref), _outside_untouched(Cbuf, inside)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [0, 1, 2, 3, 4, 5])
def test_gemm_cfg_exact(ops, cfg):
    """every tile configuration (tuning entry: 16-byte aligned operands, even lda / ldb) bit for bit against the exact product"""
    bad = []
    for t, (M, N, K) in enumerate(_gemm_shapes()):
        alpha, beta = ALPHA_BETA[t % len(ALPHA_BETA)]
        ok, kept = _run_gemm(ops, cfg, M, N, K, alpha, beta, "even", t)
        if not (ok and kept):
            bad.append((M, N, K, alpha, beta, ok, kept))
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["even", "odd", "offset"])
def test_gemm_default_dispatch_exact(ops, layout):
    """the launcher's choice (CfgSmall / Tall3 when the operands allow 16-byte copies, the ...U variants otherwise), every shape
    of the grid plus products large enough for the non-small configurations"""
    bad = []
    shapes = _gemm_shapes() + [(1600, 1537, 65), (1601, 1543, 8), (2000, 1300, 257)]
    for t, (M, N, K) in enumerate(shapes):
        alpha, beta = ALPHA_BETA[(t + 3) % len(ALPHA_BETA)]
        ok, kept = _run_gemm(ops, None, M, N, K, alpha, beta, layout, t)
        if not (ok and kept):
            bad.append((M, N, K, alpha, beta, ok, kept))
    assert not bad, bad


@pytest.mark.gpu
def test_gemm_k0_scales_c(ops):
    """K = 0: C <- beta C (and alpha A B^T = 0), for every configuration"""
    for cfg in (None, 0, 1, 2, 3, 4, 5):
        for alpha, beta in ((1.0, 0.5), (-1.0, -1.0), (2.0, 0.0)):
            ok, kept = _run_gemm(ops, cfg, 70, 130, 0, alpha, beta, "even", 3)
            assert ok and kept, (cfg, alpha, beta)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 65, 127, 129, 1000, 1237, 1600])
def test_gemm_lower_exact(ops, N):
    """gemm_nt_lower: the lower triangle bit-identical to gemm_nt (and exact), nothing written strictly above the diagonal 128 x 128
    blocks (the tiles there are skipped), what is written above the diagonal inside them equal to the full product"""
    rng = np.random.RandomState(N)
    K = 37 if N < 1600 else 64
    A, B, C = int_matrix(rng, (N, K), 256), int_matrix(rng, (N, K), 256), int_matrix(rng, (N, N), 256)
    Ad, Bd = _operand(A, "even"), _operand(B, "even")
    for alpha, beta in ((1.0, 0.0), (-1.0, 0.5)):
        outs = []
        for lower in (False, True):
            buf = _sentinel(N + 1, N + 2)
            Cd = buf[:N, :N]
            if beta != 0.0:
                Cd.copy_(_dev(C))
            if lower:
                ops.gemm_nt_lower(Ad, Bd, Cd, alpha=alpha, beta=beta)
            else:
                ops.gemm_nt(Ad, Bd, Cd, alpha=alpha, beta=beta)
            outs.append((buf, Cd))
        (fbuf, full), (lbuf, low) = outs
        assert _outside_untouched(lbuf, _region(lbuf, 0, N, 0, N))
        ref = gemm_reference(A, B, C, alpha, beta)
        assert np.array_equal(_np(full), ref)
        il = torch.tril_indices(N, N, device="cuda")
        assert torch.equal(low[il[0], il[1]].view(torch.int64), full[il[0], il[1]].view(torch.int64))
        i = torch.arange(N, device="cuda")[:, None]
        j = torch.arange(N, device="cuda")[None, :]
        above_blocks = (j // 128) > (i // 128)
        low_bits, full_bits = low.view(torch.int64), full.view(torch.int64)
        init_bits = (_dev(C) if beta != 0.0 else _sentinel(N, N)).view(torch.int64)
        assert bool((low_bits == init_bits)[above_blocks].all())
        assert bool(((low_bits == init_bits) | (low_bits == full_bits))[j > i].all())


# --------------------------------------------------------------------------------------------- 2. row max / first arg-max
def _strided3(X, layout):
    """[B, R, K] device view with the row layout of _operand"""
    Bn, R, K = X.shape
    if layout == "even":
        buf = torch.full((Bn, R + 1, K + 2 - K % 2), float("nan"), dtype=torch.float64, device="cuda")
        v = buf[:, :R, :K]
    elif layout == "odd":
        buf = torch.full((Bn, R + 1, K + 1 + K % 2), float("nan"), dtype=torch.float64, device="cuda")
        v = buf[:, :R, :K]
    else:
        buf = torch.full((Bn, R + 1, K + 3), float("nan"), dtype=torch.float64, device="cuda")
        v = buf[:, :R, 1:K + 1]
    v.copy_(_dev(X))
    return v


def _check_rowmax(fmax, arg, V):
    return np.array_equal(_np(fmax), V.max(axis=2)) and np.array_equal(_np(arg), V.argmax(axis=2))


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["even", "odd", "offset"])
def test_mvn_rowmax_ties_exact(ops, layout):
    """first arg-max with exact ties inside one lane, across lanes, across WARPS_N warps and across column tiles (and rows where
    every column ties), S in {1, 127, 129, 1025}, batch 1-3, ldz > K"""
    bad = []
    for S in (1, 127, 129, 1025):
        for B in (1, 2, 3):
            for P in (257, 1037):
                K = 24 if layout == "even" else 25
                Z, Fac, mu, V = rowmax_case(B, S, P, K, S + 10 * B + P)
                fmax, arg = ops.mvn_rowmax(_strided3(Z, layout), _strided3(Fac, layout), _dev(mu))
                if not _check_rowmax(fmax, arg, V):
                    bad.append((S, B, P))
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["even", "odd", "offset"])
def test_rff_eval_argmax_ties_exact(ops, layout):
    """the same ties through ppbo_rff_eval_argmax (Omega shared by the batch entries, no bias; all-tie rows are Omega[s] = 0)"""
    bad = []
    for S in (1, 127, 129, 1025):
        for B in (1, 2, 3):
            P = 257 if S % 2 else 1037
            K = 24 if layout == "even" else 25
            Z, Fac, _, V = rowmax_case(B, S, P, K, S + B, shared=True, with_mu=False)
            fmax, arg, _ = ops.rff_eval_argmax(_operand(Z, layout), _strided3(Fac, layout))
            if not _check_rowmax(fmax, arg, V):
                bad.append((S, B, P))
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("key", [0, 1, 3])
def test_rowmax_large_configs_and_group_tail(ops, lib, key):
    """S = 6400, batch 3: ceil(S / 128) * batch >= 148 selects the non-small configurations (tuning key 0: 0 Tall3, 1 Big,
    3 Sq16); with K = 1024 a row-tile group holds 48 of the 50 row tiles, so the last group is a tail (tiles_m % group_m != 0)
    whenever the A operand is shared by the batch entries (rff_eval_argmax, and mvn_rowmax with a stride-0 Z)"""
    S, P, K, B = 6400, 257, 1024, 3
    Z, Fac, mu, V = rowmax_case(B, S, P, K, 11, shared=True)
    Zd, Facd, mud = _dev(Z), _dev(Fac), _dev(mu)
    with tuning(lib, 0, key):
        fmax, arg = ops.mvn_rowmax(Zd.expand(B, S, K), Facd, mud)                 # group tail
        assert _check_rowmax(fmax, arg, V)
        Zb, Facb, mub, Vb = rowmax_case(B, S, P, K, 12)
        fmax, arg = ops.mvn_rowmax(_dev(Zb), _dev(Facb), _dev(mub))               # per-entry Z: one group
        assert _check_rowmax(fmax, arg, Vb)
        Fac0 = Fac.copy()
        Fac0[:, :, len(tie_pairs(P))] = 0.0                                        # no bias: all-tie rows are 0
        V0 = np.matmul(Z, Fac0.transpose(0, 2, 1))
        fmax, arg, _ = ops.rff_eval_argmax(Zd, _dev(Fac0))
        assert _check_rowmax(fmax, arg, V0)
        if key == 0:                                                               # odd ld: CfgBigU
            fmax, arg, _ = ops.rff_eval_argmax(_operand(Z, "odd"), _strided3(Fac0, "odd"))
            assert _check_rowmax(fmax, arg, V0)


@pytest.mark.gpu
def test_mvn_rowmax_empty_rows(ops):
    """S = 0 is a no-op"""
    Z = torch.zeros((2, 0, 8), dtype=torch.float64, device="cuda")
    fmax, arg = ops.mvn_rowmax(Z, torch.zeros((2, 5, 8), dtype=torch.float64, device="cuda"),
                               torch.zeros((2, 5), dtype=torch.float64, device="cuda"))
    torch.cuda.synchronize()
    assert fmax.shape == (2, 0) and arg.shape == (2, 0)


# --------------------------------------------------------------------------------------------- 3. Cholesky
CHOL_SIZES = [1, 2, 3, 4, 5, 31, 32, 33, 127, 128, 129, 255, 257, 1023, 1025, 2049, 5200]


def _chol_params():
    out = []
    for n in CHOL_SIZES:
        ldas = ["n", "odd", "even"] if n <= 1025 else (["odd"] if n == 2049 else ["n", "even"])
        out += [(n, l) for l in ldas]
    return out


def _cap(n, lda):
    return {"n": n, "odd": n + 1 + n % 2, "even": n + 2 - n % 2}[lda]


def _factor_on_device(ops, A, cap):
    """A into the leading n x n block of an (n + 1) x cap NaN buffer (NaN above the diagonal too); potrf_lower on the view"""
    n = A.shape[0]
    buf = _sentinel(n + 1, cap)
    v = buf[:n, :n]
    v.copy_(_dev(np.tril(A) + np.triu(np.full((n, n), np.nan), 1)))
    info, ws = ops.potrf_lower(v)
    return info, ws, buf, v


def _upper_kept(buf, n):
    """the contract of ppbo_potrf_lower outside the factor: the capacity region and the strictly upper triangle outside the
    128 x 128 diagonal blocks keep their bits (inside those blocks the upper triangle is scratch)"""
    i = torch.arange(buf.shape[0], device="cuda")[:, None]
    j = torch.arange(buf.shape[1], device="cuda")[None, :]
    written = (i < n) & (j < n) & ((j <= i) | ((j // 128) == (i // 128)))
    return _outside_untouched(buf, written)


def _check_factor(L, L0, A, n):
    """backward error max|A - L L^T| <= 8 n u max(diag A) and forward error max|L - L0| <= 8 n u max|L0| (cond2(A) ~ 20)"""
    fwd = np.abs(L - L0).max()
    assert fwd <= 8 * n * U * np.abs(L0).max(), fwd
    if n <= 2049:
        bwd = np.abs(A - L @ L.T).max()
        assert bwd <= 8 * n * U * np.diag(A).max(), bwd


def _check_dinv(ws, L0):
    """the inverted 128 x 128 diagonal blocks potrf_lower leaves in its workspace, against inv(L0_jj); zero above the diagonal and
    beyond jb"""
    n = L0.shape[0]
    W = _np(ws)
    for b in range((n + 127) // 128):
        j0, jb = 128 * b, min(128, n - 128 * b)
        D = W[b * 16384:(b + 1) * 16384].reshape(128, 128)
        X0 = sla.solve_triangular(L0[j0:j0 + jb, j0:j0 + jb], np.eye(jb), lower=True)
        assert np.abs(D[:jb, :jb] - X0).max() <= 8 * jb * U * np.abs(X0).max()
        assert not np.any(np.triu(D, 1)) and not np.any(D[jb:]) and not np.any(D[:, jb:])


@pytest.mark.gpu
@pytest.mark.parametrize("n,lda", _chol_params())
def test_potrf_exact_factor(ops, n, lda):
    L0, A = chol_case(n)
    info, ws, buf, v = _factor_on_device(ops, A, _cap(n, lda))
    assert info == 0
    assert _upper_kept(buf, n)
    L = np.tril(_np(v))
    _check_factor(L, L0, A, n)
    _check_dinv(ws, L0)


@pytest.mark.gpu
@pytest.mark.parametrize("key,value", [(8, 1), (9, 1), (9, 2)])
@pytest.mark.parametrize("n", [1025, 2049])
def test_potrf_tuning_paths(ops, lib, n, key, value):
    """general GEMM kernel instead of the row-panel kernel (8 = 1) or the strip trailing update (9 = 1), one tile per CTA (9 = 2):
    the same bounds and contract, and close to the default path's factor"""
    L0, A = chol_case(n)
    _, _, _, v0 = _factor_on_device(ops, A, n + 2)
    with tuning(lib, key, value):
        info, ws, buf, v = _factor_on_device(ops, A, n + 2)
    assert info == 0 and _upper_kept(buf, n)
    L = np.tril(_np(v))
    _check_factor(L, L0, A, n)
    _check_dinv(ws, L0)
    assert np.abs(L - np.tril(_np(v0))).max() <= 8 * n * U * np.abs(L0).max()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2500, 5200])
def test_potrf_deterministic(ops, n):
    """two runs give the same bits (the bulk of the trailing update runs on a side stream at these sizes)"""
    L0, A = chol_case(n)
    res = []
    for _ in range(2):
        info, ws, buf, v = _factor_on_device(ops, A, n)
        assert info == 0
        res.append((torch.tril(v).clone(), ws[: ((n + 127) // 128) * 16384].clone()))
    assert torch.equal(res[0][0].view(torch.int64), res[1][0].view(torch.int64))
    assert torch.equal(res[0][1].view(torch.int64), res[1][1].view(torch.int64))


INFO_N = 1037


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["zero", "negative", "nan"])
@pytest.mark.parametrize("k", [1, 2, 4, 5, 32, 33, 128, 129, 130, 1000, INFO_N])
def test_potrf_info_first_bad_pivot(ops, k, kind):
    """leading minor k is the first that is not positive definite, its pivot produced by elimination (inside a delayed rank-4
    group of the warp Cholesky, at 32-column piece and 128-block boundaries, after the look-ahead); info equals LAPACK's.
    scipy's dpotrf (OpenBLAS) does not test for NaN and returns 0 for the NaN case; reference LAPACK (dpotrf2: ajj <= 0 or
    NaN) returns k, as the library does."""
    A, _, _ = semidefinite_case(INFO_N, k, kind)
    cap = INFO_N if k % 2 else INFO_N + 3
    info, _, buf, _ = _factor_on_device(ops, A, cap)
    if kind == "nan":
        assert info == k
    else:
        assert info == dpotrf(A, lower=1)[1] == k
    i = torch.arange(buf.shape[0], device="cuda")[:, None]
    j = torch.arange(buf.shape[1], device="cuda")[None, :]
    assert _outside_untouched(buf, (i < INFO_N) & (j < INFO_N))


# --------------------------------------------------------------------------------------------- 4. solves
def _factored(ops, n, cap):
    L0, A = chol_case(n)
    info, ws, buf, v = _factor_on_device(ops, A, cap)
    assert info == 0
    return L0, A, ws, v


@pytest.mark.gpu
@pytest.mark.parametrize("n", [129, 1025])
def test_trsm_right_lower(ops, n):
    """X L^-T for nrhs in {1, 37, 128, 129, 1000}, ldx > n, factor with lda > n: residual and forward error against the exact L0"""
    L0, _, ws, v = _factored(ops, n, n + 3)
    rng = np.random.RandomState(n)
    for nrhs in (1, 37, 128, 129, 1000):
        X = int_matrix(rng, (nrhs, n), 16)
        buf = _sentinel(nrhs + 1, n + 5)
        Xd = buf[:nrhs, :n]
        Xd.copy_(_dev(X))
        ops.trsm_right_lower(v, ws, Xd)
        Y = _np(Xd)
        Y0 = sla.solve_triangular(L0, X.T, lower=True).T
        assert np.abs(Y @ L0.T - X).max() <= 8 * n * U * (np.abs(Y) @ np.abs(L0).T).max(), nrhs
        assert np.abs(Y - Y0).max() <= 8 * n * U * chol_conditions(n)[0] * np.abs(Y0).max(), nrhs
        assert _outside_untouched(buf, _region(buf, 0, nrhs, 0, n))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1023, 1024, 1025, 2049])
def test_potrs_vec_chained_and_blockinv(ops, n):
    """(L L^T) x = b by the chained solve and by the 1024-block inverses, lda = cap > n"""
    L0, A, ws, v = _factored(ops, n, n + 1 + n % 2)
    rng = np.random.RandomState(n)
    b = int_matrix(rng, n, 64)
    x0 = sla.solve_triangular(L0.T, sla.solve_triangular(L0, b, lower=True), lower=False)
    W = ops.blockinv_build(v, ws)
    for x in (_np(ops.potrs_vec(v, ws, _dev(b))), _np(ops.potrs_vec_blockinv(v, W, _dev(b)))):
        assert np.abs(A @ x - b).max() <= 8 * n * U * (np.abs(A) @ np.abs(x)).max()
        assert np.abs(x - x0).max() <= 8 * n * U * chol_conditions(n)[1] * np.abs(x0).max()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [129, 1025])
def test_potri_lower_strided(ops, lib, n):
    """(L L^T)^-1 into an output with ldo > n (NaN sentinels around it): symmetric and a small residual"""
    _, A, ws, v = _factored(ops, n, n + 2)
    work = torch.empty((n, n), dtype=torch.float64, device="cuda")
    buf = _sentinel(n + 1, n + 3)
    out = buf[:n, :n]
    rc = lib.ppbo_potri_lower(ctypes.c_void_p(v.data_ptr()), v.stride(0), n, ctypes.c_void_p(ws.data_ptr()),
                              lib.ppbo_potrf_workspace_bytes(n), ctypes.c_void_p(work.data_ptr()),
                              ctypes.c_void_p(out.data_ptr()), out.stride(0), _stream())
    assert rc == 0
    X = _np(out)
    assert _outside_untouched(buf, _region(buf, 0, n, 0, n))
    assert np.abs(X - X.T).max() <= 4 * n * U * np.abs(X).max()
    assert np.abs(X @ A - np.eye(n)).max() <= 8 * n * U * chol_conditions(n)[1]


# --------------------------------------------------------------------------------------------- 5. LU log-determinant
def _lu_on_device(ops, A, cap):
    n = A.shape[0]
    buf = _sentinel(n + 1, cap)
    v = buf[:n, :n]
    v.copy_(_dev(A))
    res = ops.lu_logdet(v)
    return res, buf, v


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 63, 64, 65, 127, 129, 1000, 1025, 2080])
@pytest.mark.parametrize("wide", [False, True])
def test_lu_logdet_exact(ops, n, wide):
    """A = P^T L0 U0: the device LU is LAPACK's, bit for bit (the packed factors equal scipy.linalg.lu_factor's), sign det U and the
    permutation sign are the planted ones, log|det A| = sum e_i log 2"""
    A, L0, U0, perm, esum, sgn = lu_case(n, n + wide)
    (sign_u, logabs, sign_p, rc), buf, v = _lu_on_device(ops, A, n + 3 if wide else n)
    assert rc == 0
    lu, piv = sla.lu_factor(A)
    assert np.array_equal(_np(v), lu)
    assert (sign_u, sign_p) == (sgn, perm_sign(perm)) == lapack_split(lu, piv)
    assert abs(logabs - esum * np.log(2.0)) <= 4 * n * U * max(np.log(2.0) * n, 1.0)
    assert _outside_untouched(buf, _region(buf, 0, n, 0, n))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1025, 2080])
def test_lu_logdet_ties_first_index(ops, n):
    """|l| = 1 entries: the tied rows sit in other lanes, other warps and other 1024-strides of the pivot search; the first index
    (the diagonal row) must win as in dgetrf, so no row is interchanged"""
    A, L0, U0, perm, esum, sgn = lu_case(n, 5, permute=False, ties=lu_ties(n))
    (sign_u, logabs, sign_p, rc), _, v = _lu_on_device(ops, A, n + 1)
    lu, piv = sla.lu_factor(A)
    assert rc == 0
    assert np.array_equal(_np(v), lu)
    assert (sign_u, sign_p) == lapack_split(lu, piv) == (sgn, 1.0)


@pytest.mark.gpu
@pytest.mark.parametrize("what", ["zero_column_0", "zero_column_5", "zero_column_70", "zero_column_last", "duplicate_row"])
def test_lu_logdet_singular(ops, what):
    """exactly singular input: return value 1 and log|det| = -inf (dgetrf's rule: an exactly zero pivot column is not scaled)"""
    n = 300
    A, *_ = lu_case(n, 3)
    if what == "duplicate_row":
        A[200] = A[17]
    else:
        k = {"zero_column_0": 0, "zero_column_5": 5, "zero_column_70": 70, "zero_column_last": n - 1}[what]
        A[:, k] = 0.0
    (sign_u, logabs, sign_p, rc), _, _ = _lu_on_device(ops, A, n)
    assert rc == 1
    assert logabs == -np.inf
    assert sign_u in (1.0, -1.0) and sign_p in (1.0, -1.0)


@pytest.mark.gpu
@pytest.mark.parametrize("Q,m", [(5, 3), (40, 25), (80, 25)])
@pytest.mark.parametrize("reference_sign", [0, 1])
def test_evidence_matrix_exact(ops, lib, Q, m, reference_sign):
    """ppbo_evidence_matrix against the dense I +- Sigma B diag(a) B^T with signed arrow coefficients, lds and ldo > N"""
    N = Q * (m + 1)
    rng = np.random.RandomState(Q + m)
    Sigma = int_matrix(rng, (N, N), 16) / 8
    a = int_matrix(rng, Q * m, 8) / 8
    a[::7] = -np.abs(a[::7]) - 0.125                        # some negative coefficients
    sbuf = _sentinel(N + 1, N + 3)
    Sd = sbuf[:N, :N]
    Sd.copy_(_dev(Sigma))
    buf = _sentinel(N + 2, N + 5)
    out = buf[1:N + 1, :N]
    ad = _dev(a)
    rc = lib.ppbo_evidence_matrix(ctypes.c_void_p(Sd.data_ptr()), Sd.stride(0), Q, m, ctypes.c_void_p(ad.data_ptr()),
                                  reference_sign, ctypes.c_void_p(out.data_ptr()), out.stride(0), _stream())
    assert rc == 0
    assert np.array_equal(_np(out), evidence_reference(Sigma, Q, m, a, reference_sign))
    assert _outside_untouched(buf, _region(buf, 1, N + 1, 0, N))
