"""Batch queries: q query lines per iteration by greedy joint expected improvement (q-EI) over the shared posterior draws.

q-EI of a set A of lines is E_s[max(max_{b in A} fmax[b][s] - mu*, 0)]; the maxima of all lines in one sample s come from the same
sampled function.  batch_qei_greedy below is the FP64 reference of the greedy selection.  The kernel tests use dyadic maxima, so
every sum is exact in any order and the device must give the reference's indices and values bit for bit."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from conftest import load_golden, relerr

torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def batch_qei_greedy(fmax, mustar, q):
    """(idx [q], qei [q]): step k takes the line with the largest joint EI together with the lines chosen so far, the lowest index
    on ties; qei[k] = the joint EI of the first k+1 picks"""
    fmax = np.asarray(fmax, dtype=float)
    B, S = fmax.shape
    cur = np.full(S, -np.inf)
    chosen = np.zeros(B, dtype=bool)
    idx, val = [], []
    for _ in range(q):
        gains = np.maximum(np.maximum(cur[None, :], fmax) - mustar, 0.0).sum(axis=1)
        gains[chosen] = -np.inf
        b = int(np.argmax(gains))                       # first maximum: the lowest index
        idx.append(b)
        val.append(gains[b] / S)
        chosen[b] = True
        cur = np.maximum(cur, fmax[b])
    return np.array(idx, dtype=np.int32), np.array(val)


def _dyadic(B, S, seed):
    """maxima k / 8 with |k| < 512: partial sums stay exact in FP64 in any order"""
    return np.random.RandomState(seed).randint(-511, 512, (B, S)) / 8.0


# ------------------------------------------------------------------------------------------------ reference (CPU)
def test_greedy_reference_properties():
    rng = np.random.RandomState(0)
    fmax = rng.randn(12, 500)
    fmax[9] = fmax[2] + 0.3                              # line 9 is the best one; line 4 reaches the same peaks
    fmax[4] = fmax[9]
    mustar = 0.5
    ei = np.maximum(fmax - mustar, 0).mean(axis=1)
    idx, qei = batch_qei_greedy(fmax, mustar, 6)
    assert idx[0] == int(np.argmax(ei)) == 4             # q = 1 is the EI arg-max (lowest index of the tied pair)
    assert 9 not in idx                                  # the duplicate adds nothing while any other line adds something
    assert len(set(idx.tolist())) == 6
    assert np.all(np.diff(qei) >= 0)
    assert qei[0] == ei[4]
    top = np.argsort(-ei, kind="stable")[:2]
    assert set(top.tolist()) == {4, 9}                   # top-q by marginal EI takes both


def test_greedy_reference_ties():
    f = np.zeros((5, 7))
    idx, qei = batch_qei_greedy(f, 1.0, 5)               # mu* above every sample: all gains zero
    assert idx.tolist() == [0, 1, 2, 3, 4] and np.all(qei == 0)


# ------------------------------------------------------------------------------------------------ kernels (GPU)
def _dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", torch.cuda.current_device())


def _select(fmax_h, mustar, q, dev):
    from ppbo_b200 import iteration
    fmax = torch.from_numpy(np.ascontiguousarray(fmax_h)).to(dev)
    idx, qei = iteration.select_batch(fmax, torch.tensor([float(mustar)], dtype=torch.float64, device=dev), q, fmax.shape[0])
    return idx.cpu().numpy(), qei.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 1023, 1025, 32768])
@pytest.mark.parametrize("B", [1, 2, 37, 300])
def test_select_exact(B, S):
    dev = _dev()
    f = _dyadic(B, S, B * 7 + S)
    for mustar in (0.25, -70.0):
        for q in sorted({1, min(3, B), B}):
            idx, qei = _select(f, mustar, q, dev)
            ref_idx, ref_qei = batch_qei_greedy(f, mustar, q)
            assert np.array_equal(idx, ref_idx), (mustar, q)
            assert np.array_equal(qei, ref_qei), (mustar, q)
            assert len(set(idx.tolist())) == q
    # planted ties: three identical best lines -> the lowest index first, and a copy only when nothing else is left to gain
    if B >= 12:
        g = f.copy()
        g[[3, 7, 11]] = f.max(axis=0) + 1.0
        idx, qei = _select(g, 0.25, 3, dev)
        assert idx[0] == 3 and 7 not in idx and 11 not in idx
        assert np.array_equal(idx, batch_qei_greedy(g, 0.25, 3)[0])
    # all gains zero (mu* above every sample): the lowest unchosen index wins every step
    q = min(B, 5)
    idx, qei = _select(f, 1e3, q, dev)
    assert idx.tolist() == list(range(q)) and np.all(qei == 0)


@pytest.mark.gpu
def test_select_argument_errors():
    from ppbo_b200 import iteration, ops
    from ppbo_b200._lib import PPBOError
    dev = _dev()
    f = torch.from_numpy(_dyadic(4, 100, 1)).to(dev)
    mu = torch.zeros(1, dtype=torch.float64, device=dev)
    idx = torch.empty(5, dtype=torch.int32, device=dev)
    val = torch.empty(5, dtype=torch.float64, device=dev)
    cur = torch.empty(100, dtype=torch.float64, device=dev)
    for q in (0, 5):
        with pytest.raises(PPBOError):
            ops.acq_batch_gain(f, mu, cur, 0, q)
        with pytest.raises(PPBOError):
            ops.acq_batch_pick(torch.zeros(5, dtype=torch.float64, device=dev), f, 0, q, idx, val, cur)
        with pytest.raises(PPBOError):
            iteration.select_batch(f, mu, q, 4)
    big = torch.zeros((65536, 1), dtype=torch.float64, device=dev)        # above the candidate limit
    with pytest.raises(PPBOError):
        ops.acq_batch_gain(big, mu, None, 0, 1)


# ------------------------------------------------------------------------------------------------ pipeline (GPU)
def _problem(dev, S):
    from ppbo_b200 import synthetic
    prob = synthetic.make_problem("levy10d", Q=41, P=256, F=500, S=S)
    t = {k: torch.from_numpy(np.ascontiguousarray(prob[k])).to(dev) for k in ("X", "W", "b", "grids")}
    return prob, t


def _run(prob, t, S, cov, batch=None, grids=None):
    from ppbo_b200 import iteration as it
    d = {"X": t["X"], "W": t["W"], "b": t["b"], "grids": t["grids"] if grids is None else grids}
    return it.run_iteration(d, prob["kernel"], prob["theta"], prob["Q"], prob["m"], S, seed=5, weight_covariance=cov, batch=batch)


@pytest.mark.gpu
def test_first_step_equals_reduction():
    from ppbo_b200 import iteration as it
    from ppbo_b200 import ops
    dev = _dev()
    S = 4096
    prob, t = _problem(dev, S)
    sums, gp, rff = _run(prob, t, S, "diag")
    B, P, D = t["grids"].shape
    PhiT = it.rff_grid_features(t["W"], t["b"], prob["theta"][2], t["grids"])
    fmax, _ = it.rff_sampled_maxima(rff, PhiT, 0, S, seed=5)
    mustar = it.mustar_over_candidates(gp, t["grids"].reshape(B * P, D))
    gain = ops.acq_batch_gain(fmax, mustar, None, 0, 1)
    col0 = ops.acq_reduce_dev(fmax, mustar)[:, 0]
    assert torch.equal(gain[:B], col0)
    assert torch.equal(col0, sums[:, 0])
    assert float(gain[B]) == S


@pytest.mark.gpu
@pytest.mark.parametrize("cov", ["diag", "full"])
@pytest.mark.parametrize("S", [4096, 64], ids=["i8", "f64"])
def test_run_iteration_batch(S, cov):
    from ppbo_b200 import iteration as it
    dev = _dev()
    prob, t = _problem(dev, S)
    q = 4
    assert it.sampling_engine(S, t["grids"].shape[1], prob["F"]) == ("i8" if S == 4096 else "f64")
    sums0, _, _ = _run(prob, t, S, cov)
    sums, gp, rff, (idx, qei) = _run(prob, t, S, cov, batch=q)
    assert torch.equal(sums, sums0)                          # the selection changes nothing of the sums
    B, P, D = t["grids"].shape
    PhiT = it.rff_grid_features(t["W"], t["b"], prob["theta"][2], t["grids"])
    fmax, _ = it.rff_sampled_maxima(rff, PhiT, 0, S, seed=5, covariance=cov)
    mustar = float(it.mustar_over_candidates(gp, t["grids"].reshape(B * P, D)))
    ref_idx, ref_qei = batch_qei_greedy(fmax.cpu().numpy(), mustar, q)
    assert np.array_equal(idx.cpu().numpy(), ref_idx)
    assert relerr(qei.cpu().numpy(), ref_qei) <= 1e-12
    assert np.array_equal(qei.cpu().numpy()[:1], sums.cpu().numpy()[ref_idx[:1], 0] / S)
    if S == 4096:                                            # the overlapped schedule against the sequential one
        saved = it.OVERLAP_SAMPLING
        try:
            it.OVERLAP_SAMPLING = False
            _, _, _, (idx_s, qei_s) = _run(prob, t, S, cov, batch=q)
        finally:
            it.OVERLAP_SAMPLING = saved
        assert torch.equal(idx_s, idx) and torch.equal(qei_s, qei)


@pytest.mark.gpu
def test_run_iteration_batch_skips_duplicate_line():
    """lines 3 and 7 made copies of the best line: top-q by marginal EI takes two copies, the joint selection one"""
    dev = _dev()
    S, q = 4096, 3
    prob, t = _problem(dev, S)
    sums, _, _ = _run(prob, t, S, "diag")
    best = int(torch.argmax(sums[:, 0]))
    grids = t["grids"].clone()
    grids[3] = t["grids"][best]
    grids[7] = t["grids"][best]
    copies = {3, 7, best}
    sums, _, _, (idx, _) = _run(prob, t, S, "diag", batch=q, grids=grids)
    ei = sums[:, 0].cpu().numpy()
    top = np.argsort(-ei, kind="stable")[:q]
    assert len(copies & set(top.tolist())) >= 2
    assert len(copies & set(idx.cpu().numpy().tolist())) == 1


# ------------------------------------------------------------------------------------------------ several ranks (GPU, NCCL)
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_n_rank_batch_equals_single_rank(world):
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "mgpu_batch_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "MGPU_BATCH_OK world=%d" % world in r.stdout


# ------------------------------------------------------------------------------------------------ reference API (GPU)
def _model(g):
    from gp_model import GPModel
    from ppbo_settings import PPBO_settings
    st = PPBO_settings(D=g["D"], bounds=g["bounds"], xi_acquisition_function="EI-EXT-FAST", m=g["m"],
                       theta_initial=list(g["theta"]), kernel=g["kernel"], verbose=False, alpha_grid_distribution="equispaced")
    gp = GPModel(st)
    np.random.seed(int(g["seed_design"]))
    gp.update_feedback_processing_object(g["X_obs"])
    gp.update_data()
    gp.turn_initialization_off()
    gp.set_theta()
    gp.update_Sigma(gp.theta)
    np.random.seed(int(g["seed_fit"]))
    gp.update_fMAP()
    gp.xstar, gp.mustar = g["xstar"].copy(), float(g["mustar"])
    gp.xstars_local = g["xstars_local"].copy()
    return st, gp


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["camel2d", "hartmann6d"])
def test_next_query_batch(name):
    import acquisition
    from oracle import ppbo_oracle as O
    _dev()
    g = load_golden(name)
    st, gp = _model(g)
    D, S, P = g["D"], st.mc_samples, acquisition.GRID_POINTS
    xis, pairs = acquisition._coordinate_pairs(gp)
    np.random.seed(21)
    fmax, grids, Z, mu, L = acquisition.sampled_max_joint(pairs, gp, S)
    fmax, mu, L = fmax.cpu().numpy(), mu.cpu().numpy(), L.cpu().numpy()
    # Joint covariance of the D*70 points: the oracle's prediction from the reference's own fit.  The lines all pass near x*, so the
    # matrix is numerically singular and two Cholesky factors of it (device, LAPACK) agree only to about sqrt(eps): the factor is
    # judged by L L' against the oracle's covariance, and the maxima against the FP64 product of that same factor with the same Z.
    Xp = grids.reshape(D * P, D)
    mu_o, Sp_o = O.mu_Sigma_pred(g["X"], Xp, g["theta"], O.se_kernel, g["Sigma_inv"], g["fMAP"], g["posterior_covariance"])
    sf2 = g["theta"][2] ** 2
    assert np.abs(L @ L.T - Sp_o).max() <= 2e-5 * sf2           # the factor (with its jitter) of the cross-grid covariance
    assert np.abs(mu - mu_o).max() <= 2e-5 * np.abs(mu_o).max()
    # the per-grid maxima of f = mu + L z over the shared draws, in FP64 on the host from the same factor and the same Z
    Fs = mu[None, :] + Z @ L.T
    ref = Fs.reshape(S, D, P).max(axis=2).T
    assert np.abs(fmax - ref).max() <= 1e-9 * np.abs(ref).max()
    # the public entry on the same stream: q distinct unit directions, the greedy picks, the generator where it should be
    q = D
    np.random.seed(21)
    out = acquisition.next_query_batch(st, gp, q, unscale=False)
    after = np.random.get_state()
    np.random.seed(21)
    for xi, x in pairs:
        gp.FP.xi_grid(xi=xi, x=x, alpha_grid_distribution='equispaced', alpha_star=None, m=P, is_scaled=True)
    np.random.standard_normal((S, D * P))
    expect = np.random.get_state()
    assert after[0] == expect[0] and np.array_equal(after[1], expect[1]) and after[2:] == expect[2:]
    ref_idx, _ = batch_qei_greedy(fmax, float(gp.mustar), q)
    assert [int(np.argmax(xi)) for xi, _ in out] == ref_idx.tolist()
    assert len({int(np.argmax(xi)) for xi, _ in out}) == q
    for xi, x in out:
        assert np.count_nonzero(xi) == 1 and xi.max() == 1.0 and x.shape == (D,)
    # the evaluators answer the q queries; the answers go in one at a time and the model refits
    np.random.seed(21)
    X_obs = g["X_obs"]
    for xi, x in acquisition.next_query_batch(st, gp, q, unscale=True):
        X_obs = np.vstack([X_obs, np.concatenate([0.5 * xi + x, xi, [0.5]])])
        gp.update_feedback_processing_object(X_obs)
        gp.update_data()
    gp.fMAP_random_initial_vector = False
    gp.update_model()
    assert gp.N == g["X"].shape[0] + q * (g["m"] + 1) and len(gp.fMAP) == gp.N


@pytest.mark.gpu
def test_hsampler_select_batch_over_grids():
    """the sampler's entry equals select_batch on the maxima of its own draws, and two 'ranks' without a process group see the
    same picks as one"""
    from random_fourier_sampler import Hsampler
    _dev()
    g = load_golden("camel2d")
    st, gp = _model(g)
    np.random.seed(int(g["seed_rff"]))
    h = Hsampler(gp, nFeatures=g["rff_W"].shape[0])
    h.generate_basis()
    h.update_phi_X()
    h.update_omega_MAP(omega_initial=g["rff_omega_MAP"])
    h.update_covariancematrix()
    grids = np.stack([g["rff_grid"], g["rff_grid"][::-1] * 0.9, g["rff_grid"] * 0.5 + 0.2])
    idx, qei = h.select_batch_over_grids(grids, 256, float(g["mustar"]), 2, seed=3)
    sums = h.sample_max_over_grids(grids, 256, float(g["mustar"]), seed=3)
    assert idx[0] == int(np.argmax(sums[:, 0])) and qei[0] == sums[idx[0], 0] / 256
    assert len(set(idx.tolist())) == 2 and qei[1] >= qei[0]
