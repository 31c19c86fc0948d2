"""CPU tests of the host side of the drop-in package src/ (no GPU): the design-matrix builder must consume the global
RNG exactly like the reference (golden X / X_full were produced by the executed reference), the settings object must
carry the reference's attributes, and the coordinate strategies of next_query are pure host logic."""
import os
import sys
import types

import numpy as np
import pytest

from conftest import load_golden, golden_names


def _settings(g, strategy="EI-EXT-FAST"):
    from ppbo_settings import PPBO_settings
    return PPBO_settings(D=g["D"], bounds=g["bounds"], xi_acquisition_function=strategy, m=g["m"],
                         theta_initial=list(g["theta"]), kernel=g["kernel"], verbose=False,
                         alpha_grid_distribution="equispaced")


def test_design_matrix_matches_reference(golden):
    """FeedbackProcessing.create_X with the reference's seed reproduces the reference's X bit for bit."""
    from feedback_processing import FeedbackProcessing
    g = golden
    fp = FeedbackProcessing(g["D"], g["m"], g["bounds"], "equispaced", 0.4)
    np.random.seed(int(g["seed_design"]))
    fp.initialize_data(g["X_obs"])
    assert np.array_equal(fp.X_full, g["X_full"])
    assert np.array_equal(fp.X, g["X"])
    assert fp.N == g["X"].shape[0]
    assert fp.obs_indices == [int(i) for i in g["obs_indices"]]
    assert fp.latest_obs_indices[:g["m"] + 2] == [0] * (g["m"] + 1) + [g["m"] + 1]
    assert len(fp.pseudobs_indices) == g["Q"] * g["m"]


def test_design_matrix_incremental_update(golden):
    """update_X keeps the earlier pseudo-observation grids and appends one block (src/feedback_processing.py:133-154)."""
    from feedback_processing import FeedbackProcessing
    g = golden
    fp = FeedbackProcessing(g["D"], g["m"], g["bounds"], "equispaced", 0.4)
    np.random.seed(3)
    fp.initialize_data(g["X_obs"][:-1])
    head = fp.X_full.copy()
    fp.update_data(g["X_obs"])
    assert fp.iter_number == 2
    assert np.array_equal(fp.X_full[:len(head)], head)
    assert fp.N == g["X"].shape[0]
    blk = fp.X_full[-(g["m"] + 1):]
    assert np.array_equal(blk[0, :g["D"]], g["X_obs"][-1, :g["D"]])
    assert np.array_equal(blk[:, 2 * g["D"]], np.r_[0, np.ones(g["m"])])


def test_scale_unscale_roundtrip(golden):
    from feedback_processing import FeedbackProcessing
    g = golden
    fp = FeedbackProcessing(g["D"], g["m"], g["bounds"], "equispaced", 0.4)
    rng = np.random.RandomState(0)
    lo = np.array([b[0] for b in g["bounds"]]); hi = np.array([b[1] for b in g["bounds"]])
    X = lo + rng.rand(7, g["D"]) * (hi - lo)
    assert np.allclose(fp.unscale(fp.scale(X)), X, rtol=0, atol=1e-12 * np.abs(hi - lo).max())
    Z = X.copy(); Z[:, 0] = 0
    assert np.all(fp.scale(Z, retain_0_values=True)[:, 0] == 0)
    assert np.all(fp.unscale(np.zeros((2, g["D"])), retain_0_values=True) == 0)


def test_xi_grid_shapes_and_bounds():
    from feedback_processing import FeedbackProcessing
    bounds = ((-3, 3), (-2, 2), (0, 5))
    fp = FeedbackProcessing(3, 10, bounds, "equispaced", 0.4)
    np.random.seed(0)
    g = fp.xi_grid(xi=[0, 2.0, 0], x=np.array([1.0, 0, 2.0]))
    assert g.shape == (10, 3) and np.all(g[:, 0] == 1.0) and np.all(np.abs(g[:, 1]) <= 2 + 1e-12)
    g2 = fp.xi_grid(xi=[0, 2.0, 0])                       # x=None: only the moving coordinate is returned
    assert g2.shape == (10, 1)
    g3 = fp.xi_grid(xi=[1, 0, 0], x=np.zeros(3), m=70, is_scaled=True)
    assert g3.shape == (70, 3) and g3[:, 0].min() >= 0 and g3[:, 0].max() <= 1 and np.all(np.diff(g3[:, 0]) > 0)
    for dist in ("Cauchy", "TGN"):
        g4 = fp.xi_grid(xi=[1, 0, 0], x=np.zeros(3), alpha_grid_distribution=dist, alpha_star=0.5)
        assert g4.shape == (10, 3) and g4[:, 0].min() >= -3 and g4[:, 0].max() <= 3


def test_alpha_bounds():
    from misc import alpha_bounds
    lo, hi = alpha_bounds([1, 0], [-3, -2], [3, 2])
    assert (lo, hi) == (-3, 3)
    lo, hi = alpha_bounds([0.5, -1.0], [-3, -2], [3, 2])
    assert lo == max(-3 / 0.5, 2 / -1.0) and hi == min(-2 / -1.0, 3 / 0.5)


@pytest.mark.parametrize("strategy", ["PCD", "EXT", "RAND", "EI", "EI-FIXEDX", "EXR", "EI-EXT", "EI-EXT-FAST", "EI-VARMAX",
                                      "EI-VARMAX-FAST", "COORDINATE-VARMAX"])
def test_settings_match_reference(strategy):
    """The attributes of the reference's PPBO_settings (its src/ppbo_settings.py:8-79) for these arguments, with their values,
    stored per strategy in tests/golden/settings_reference.json (tuples as JSON lists); the B200-path knobs are ours alone."""
    import json
    from conftest import GOLDEN_DIR
    from ppbo_settings import PPBO_settings
    with open(os.path.join(GOLDEN_DIR, "settings_reference.json")) as fh:
        rec = json.load(fh)
    kw = dict(rec["kwargs"], bounds=tuple(tuple(b) for b in rec["kwargs"]["bounds"]), xi_acquisition_function=strategy)
    ours = PPBO_settings(**kw)
    assert ours.n_pseudoobservations == 7 and ours.mc_samples == 150 and ours.BO_maxiter == 20
    assert ours.n_gausshermite_sample_points == 200 and ours.TGN_speed == 0.4 and ours.fMAP_optimizer == 'trust-exact'
    theirs = rec["attributes"][strategy]
    for k, v in theirs.items():
        assert json.loads(json.dumps(getattr(ours, k))) == v, k


def test_cyclic_strategies_match_golden(golden):
    """PCD / EXT are host logic on (settings, xstar, FP): three successive calls reproduce the reference's queries."""
    import acquisition
    from feedback_processing import FeedbackProcessing
    g = golden
    fp = FeedbackProcessing(g["D"], g["m"], g["bounds"], "equispaced", 0.4)
    model = types.SimpleNamespace(xstar=g["xstar"].copy(), FP=fp, verbose=False, D=g["D"])
    for strat in ("PCD", "EXT"):
        st = _settings(g, strat)
        for k in range(3):
            xi, x = acquisition.next_query(st, model, unscale=True)
            assert np.allclose(np.concatenate([xi, x]), g["next_" + strat][k], rtol=1e-12, atol=0)


def test_c_abi_exports_every_declared_symbol():
    """The shared library loads without a GPU and exports exactly the entry points include/ppbo_b200.h declares."""
    import os
    import re
    from ppbo_b200 import _lib
    from ppbo_b200 import build as _build
    _build.build()
    lib = _lib.load()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "ppbo_b200.h")).read()
    declared = set(re.findall(r"\b(ppbo_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(lib, name), "library lacks " + name
    assert declared == set(_lib.EXPORTED_SYMBOLS), declared ^ set(_lib.EXPORTED_SYMBOLS)
    assert lib.ppbo_version() >= 100
    assert lib.ppbo_factor_doubles(256) == 256 * 256 + 2 * 128 * 128


def test_no_cpu_fallback_without_gpu():
    import torch
    from ppbo_b200 import ops
    from ppbo_b200._lib import PPBOError
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(PPBOError):
        ops.device()


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs next to ours) on this host: one JSON line with the contract's keys"""
    import json
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "ppbo_iteration_ms" and line["unit"] == "ms"
    assert line["higher_is_better"] is False and line["value"] > 0 and line["steps"] == 1
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"]


def test_bench_refuses_to_run_our_arm_without_a_gpu():
    """no CPU fallback: our arm exits with an error when there is no CUDA device"""
    import subprocess
    import torch
    if torch.cuda.is_available():
        pytest.skip("needs a host without a GPU")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
