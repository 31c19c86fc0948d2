"""The half-triangle kernels of the two fits: the lower-only weight-space Hessian product (same bits below the diagonal as the full
product) and the symmetric mat-vec of the GP fit (lower triangle only, bits independent of the launch grid)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from ppbo_b200 import ops as _ops
    return _ops


@pytest.mark.parametrize("F,M", [(1000, 5000), (333, 1237)])
def test_hessian_lower_tiles_match_full_product(ops, F, M):
    """Psi' a+ Psi as launched by the weight-space fit (Psi^T stored F x M): the bench shape and an odd one"""
    g = torch.Generator(device="cuda").manual_seed(F)
    PsiT = torch.randn(F, M, dtype=torch.float64, device="cuda", generator=g)
    full = ops.gemm_nt(PsiT, PsiT)
    low = torch.full((F, F), float("nan"), dtype=torch.float64, device="cuda")
    ops.gemm_nt_lower(PsiT, PsiT, low)
    torch.cuda.synchronize()
    il = torch.tril_indices(F, F, device="cuda")
    assert torch.equal(low[il[0], il[1]], full[il[0], il[1]])


def _sym(n, ld, seed, upper_garbage=True):
    g = torch.Generator(device="cuda").manual_seed(seed)
    B = torch.randn(n, n, dtype=torch.float64, device="cuda", generator=g)
    S = (B + B.T) / 2
    A = torch.full((n, ld), float("nan"), dtype=torch.float64, device="cuda")
    A[:, :n] = S
    if upper_garbage:          # nothing above the diagonal may be read
        iu = torch.triu_indices(n, n, 1, device="cuda")
        A[iu[0], iu[1]] = float("nan")
    return A, S


@pytest.mark.parametrize("n", [1, 127, 128, 129, 1000, 5000, 5200])
def test_symv_lower_matches_gemv(ops, n):
    A, S = _sym(n, n, n)
    x = torch.randn(n, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(n + 1))
    y = ops.symv_lower(A, x)
    ref = ops.gemv(S.contiguous(), x)
    torch.cuda.synchronize()
    assert torch.isfinite(y).all()
    assert (torch.max(torch.abs(y - ref)) / torch.max(torch.abs(ref))).item() < 1e-14


def test_symv_lower_capacity_layout(ops):
    """lda > n, as for G and the factor in their capacity buffers"""
    n, ld = 1237, 1501
    A, S = _sym(n, ld, 7)
    x = torch.randn(n, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(8))
    y = ops.symv_lower(A, x)
    yc = ops.symv_lower(torch.tril(S).contiguous(), x)
    torch.cuda.synchronize()
    assert torch.equal(y, yc)
    ref = ops.gemv(S.contiguous(), x)
    assert (torch.max(torch.abs(y - ref)) / torch.max(torch.abs(ref))).item() < 1e-14


def test_symv_lower_bits_independent_of_grid(ops):
    """the tile kernel's grid (tuning key 15) leaves the bits alone: the GP fit runs it on whatever SMs the contraction leaves"""
    from ppbo_b200 import _lib
    lib = _lib.load()
    n = 5000
    A, _ = _sym(n, n, 11)
    x = torch.randn(n, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(12))
    outs = []
    try:
        for grid in (0, 1, 7, 16, 32, 148, 1000):
            lib.ppbo_set_tuning(15, grid)
            outs.append(ops.symv_lower(A, x).clone())
    finally:
        lib.ppbo_set_tuning(15, 0)
    torch.cuda.synchronize()
    for y in outs[1:]:
        assert torch.equal(y, outs[0])
    assert np.isfinite(outs[0].cpu().numpy()).all()
