#!/usr/bin/env python
"""bench.py -- one PPBO iteration (GP Laplace fit + RFF acquisition over the xi-grids of every query direction).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config ackley20d] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is one full iteration on synthetic inputs of the named BASELINE.json shape (default: Ackley-20D, 200 queries x
m = 25 -> N = 5200 rows / 5000 pseudo-observations, F = 1000 features, 20 directions x 1024 grid points, 32768 samples):
  value : ms per iteration from a COLD start (f = 0, omega = 0 -- what the reference's default random start corresponds to),
          inputs already resident in HBM (max over ranks, CUDA events)
  e2e   : the same iteration through the public host API with pinned HOST buffers: H2D of the inputs and D2H of the
          per-direction sums inside the timed region, followed by the host arg-max over directions
  steady_state : what every iteration after the first costs: one comparison set is APPENDED to the fitted 200-query model
          (rows of Sigma and G, factor grown by 25 rows, chord iteration from the previous mode, warm weight-space fit), end to
          end with host buffers; K consecutive appends (queries 201 ... 200 + K)
  parity_gate : after the timed regions, the cold step's results against the committed oracle fixture
          (tests/golden/full_<config>.npz, made by oracle/make_full_fixtures.py on the host) and the host gradient formula
Only the Monte-Carlo samples (and, from 3 ranks on, the mu* candidates) are partitioned over the ranks (fixed total work ->
"scaling": "strong").  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")      # see ppbo_b200/__init__.py (before the CUDA context exists)

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ppbo_iteration_ms"
UNIT = "ms"
# FP64 tensor (DMMA) pipe peak measured on this pool's B200 by scratch/ubench.cu (profiles/r01_fp64_peaks_ubench.txt):
# register-resident mma.sync.m8n8k4.f64 loop, 37.1 TFLOP/s; MEASURED_PEAKS.json carries no FP64 figure.  The bench also measures
# its own FP64 GEMM rate (roofline.fp64_gemm_measured_tflops).
FP64_TENSOR_PEAK_TFLOPS = 37.1
SEED = 1234


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="ackley20d")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-api-leg", action="store_true", help="skip the src/ API timing at configs 1-3")
    ap.add_argument("--samples", type=int, default=None, help="override S (debug)")
    ap.add_argument("--profile", default=None, choices=[None, "cold", "steady"],
                    help="1 warm-up + --steps resident steps of the named kind, no JSON (for ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed resident step returned as DIR/<name>.npy (float64), to compare two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        # (every 200 ms: each query takes the driver's lock for a few ms; a host-synchronous step that meets one is a 20-90 ms
        # outlier in the per-step times, seen in ~1 of 150 steps at 100 ms)
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s in sm if s > 0]
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------- CPU reference arm
def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def blas_threads(n=None):
    """pin (n given) and report the BLAS/OpenMP thread count of numpy/scipy"""
    try:
        import threadpoolctl
        if n is not None:
            threadpoolctl.threadpool_limits(limits=n)
        info = threadpoolctl.threadpool_info()
        return max([i.get("num_threads", 1) for i in info] or [1])
    except Exception:
        return None


def recorded_outer_iterations(name):
    """outer-iteration count of the oracle's trust-exact fit at FULL N from the reference's random start, measured once in the build
    container by oracle/make_full_fixtures.py record (profiles/r02_reference_full_fit_<name>.json)"""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_reference_full_fit_%s.json" % name)) as fh:
            rec = json.load(fh)
        full = max(rec["runs"], key=lambda r: r["N"])
        return int(full["trust_exact_nit"]), "profiles/r02_reference_full_fit_%s.json (N=%d: %d outer iterations, %.1f s each on %d threads there)" % (
            name, full["N"], full["trust_exact_nit"], full["trust_exact_s_per_iteration"], rec.get("host_threads", 0))
    except Exception:
        return 12, "no record file: 12 outer iterations assumed (the count measured for ackley20d)"


class ReferenceArm:
    """The reference's algorithm (oracle port: numpy/scipy + multi-threaded BLAS) on the named workload at FULL size.

    One timed step = ONE real outer iteration of scipy trust-exact on the dense N x N Hessian at full N from the reference's random
    start (objective, gradient, Hessian assembly, More-Sorensen subproblem with its Cholesky factorisations) -- the unit the
    reference's fit repeats.  The one-off N^3 pieces (Sigma^-1 by dposv, posterior covariance), the weight-space fit and a bounded
    slice of the sampling contraction are timed once at start-up.  One full iteration = one-off pieces + per-iteration time x the
    outer-iteration count RECORDED from a complete run of the same fit (recorded_outer_iterations); that product is an
    extrapolation and is labelled as one."""

    def __init__(self, prob, s_sample=256):
        from oracle import ppbo_oracle as O
        self.O, self.prob = O, prob
        self.threads = blas_threads()
        D, Q, m, S, F = prob["D"], prob["Q"], prob["m"], prob["S"], prob["F"]
        theta, X = prob["theta"], prob["X"]
        self.parts = {}

        def timed(name, scale, fn):
            t0 = time.perf_counter()
            out = fn()
            self.parts[name] = (time.perf_counter() - t0) * scale * 1e3
            return out
        Sigma = timed("gram_regularize_closed_form", 1.0, lambda: O.regularize_covariance(O.se_kernel(X, X, theta), svd_roundtrip=False))
        self.Sinv = timed("Sigma_inverse_dposv", 1.0, lambda: O.pd_inverse(Sigma))
        rng = np.random.RandomState(0)
        self.f0 = np.linalg.cholesky(Sigma) @ rng.standard_normal(X.shape[0])          # f ~ N(0, Sigma), the reference's start (:374)
        timed("posterior_covariance_dposv", 1.0, lambda: O.posterior_covariance(self.Sinv, self.f0 * 0.0, Q, m, theta[0]))
        del Sigma
        if F:
            W, b = prob["W"], prob["b"]
            PhiX = timed("rff_features_design", 1.0, lambda: O.rff_features(W, b, X, theta[2]))
            t0 = time.perf_counter()
            _, res = O.rff_omega_map(PhiX, Q, m, theta[0], np.zeros(F))
            self.parts["rff_trust_exact_fit(%d outer iterations, measured in full)" % res.nit] = (time.perf_counter() - t0) * 1e3
            ss = min(S, s_sample)
            Omega = np.random.RandomState(1).randn(ss, F)

            def sampling():
                out = 0.0
                for d in range(prob["grids"].shape[0]):
                    mx, _ = O.rff_eval_argmax(Omega, O.rff_features(W, b, prob["grids"][d], theta[2]))
                    out += np.maximum(mx, 0).sum()
                return out
            timed("rff_sampling_gemm_rowmax(%d of %d samples, scaled)" % (ss, S), S / ss, sampling)
        self.nit, self.nit_source = recorded_outer_iterations(prob["name"])

    def step(self):
        """one real trust-exact outer iteration at full N; returns its wall time in ms"""
        import scipy.optimize
        O, p = self.O, self.prob
        Q, m, sigma = p["Q"], p["m"], p["theta"][0]
        t0 = time.perf_counter()
        scipy.optimize.minimize(lambda f: -O.T_value(f, self.Sinv, Q, m, sigma, quadrature=False), self.f0, method="trust-exact",
                                jac=lambda f: -O.T_grad(f, self.Sinv, Q, m, sigma), hess=lambda f: -O.T_hessian(f, self.Sinv, Q, m, sigma),
                                options={"maxiter": 1})
        return (time.perf_counter() - t0) * 1e3

    def iteration_ms(self, per_iteration_ms):
        return sum(self.parts.values()) + per_iteration_ms * self.nit

    def sample_text(self, per_iteration_ms):
        return ("oracle port (numpy/scipy, BLAS threads = %s of %d host threads) at FULL N = %d: one trust-exact outer iteration measured per "
                "step = %.0f ms; iteration = one-off parts + that x %d outer iterations [%s] -- EXTRAPOLATED by the recorded count; one-off "
                "parts ms: %s" % (self.threads, host_threads(), self.prob["N"], per_iteration_ms, self.nit, self.nit_source,
                                  {k: round(v, 1) for k, v in self.parts.items()}))


def single_thread_ratio(prob_name):
    """the reference's own policy is BLAS threads = 1 (numerical_experiments/run.slrm:6-9): ratio of one trust-exact outer iteration
    with 1 thread to all threads, measured at a quarter of the problem (N = 1300 for ackley20d)"""
    try:
        import threadpoolctl
        from ppbo_b200 import synthetic
        from oracle import ppbo_oracle as O
        import scipy.optimize
        cfg = synthetic.CONFIGS[prob_name]
        p = synthetic.make_problem(prob_name, Q=max(4, cfg["Q"] // 4), S=8, P=8)
        Sigma = O.regularize_covariance(O.se_kernel(p["X"], p["X"], p["theta"]), svd_roundtrip=False)
        Sinv = O.pd_inverse(Sigma)
        f0 = np.linalg.cholesky(Sigma) @ np.random.RandomState(0).standard_normal(p["N"])

        def one():
            t0 = time.perf_counter()
            scipy.optimize.minimize(lambda f: -O.T_value(f, Sinv, p["Q"], p["m"], p["theta"][0], quadrature=False), f0, method="trust-exact",
                                    jac=lambda f: -O.T_grad(f, Sinv, p["Q"], p["m"], p["theta"][0]),
                                    hess=lambda f: -O.T_hessian(f, Sinv, p["Q"], p["m"], p["theta"][0]), options={"maxiter": 1})
            return (time.perf_counter() - t0) * 1e3
        one()
        t_all = one()
        with threadpoolctl.threadpool_limits(limits=1):
            t_one = one()
        return {"N": p["N"], "outer_iteration_ms_all_threads": t_all, "outer_iteration_ms_1_thread": t_one, "ratio": t_one / t_all}
    except Exception as e:       # pragma: no cover
        return {"error": str(e)}


def run_reference(args):
    """--impl reference: the reference algorithm on the host cores (oracle port; the Python reference cannot travel)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from ppbo_b200 import synthetic
    prob = synthetic.make_problem(args.config, S=args.samples)
    arm = ReferenceArm(prob)
    per = []
    for i in range(args.warmup + args.steps):
        t = arm.step()
        if i >= args.warmup:
            per.append(t)
    per_it = float(np.mean(per))
    v = arm.iteration_ms(per_it)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": v, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(prob, args.gpus),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": arm.threads or host_threads(), "kind": "port", "sample": arm.sample_text(per_it)},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "extrapolated": True, "measured_step_ms": per_it, "measured_step": "one trust-exact outer iteration at full N",
            "outer_iterations_recorded": arm.nit, "one_off_parts_ms": {k: round(v_, 1) for k, v_ in arm.parts.items()},
            "blas_threads": arm.threads, "single_thread": single_thread_ratio(args.config)}
    print(json.dumps(line))


def iteration_slices():
    from ppbo_b200 import iteration
    return iteration.SAMPLING_SLICES


def iteration_reserved_sms():
    from ppbo_b200 import iteration
    return "%d (cold) / %d (appended)" % (iteration.OVERLAP_RESERVED_SMS_COLD, iteration.OVERLAP_RESERVED_SMS) if iteration.OVERLAP_SAMPLING else "0"


def workload_config(prob, n_gpus):
    return {"workload": "%s: D=%d, Q=%d queries x m=%d (N=%d rows, %d pseudo-observations), %s theta=%s, F=%d RFF features, "
                        "%d query directions x P=%d xi-grid points, S=%d samples" % (
                            prob["name"], prob["D"], prob["Q"], prob["m"], prob["N"], prob["Q"] * prob["m"], prob["kernel"],
                            prob["theta"], prob["F"], prob["grids"].shape[0], prob["P"], prob["S"]),
            "parallelism": ("one GPU, two concurrent chains: weight-space fit -> draws -> INT8 contraction (foreground streams, persistent "
                            "grid on all but %s SMs) || GP fit -> mu* (background thread, lowest stream priority, on the SMs left free); "
                            "only the reduction of 3 x directions sums needs both" % iteration_reserved_sms() if n_gpus == 1 else
                            "GP fit on rank 0, weight-space fit on rank 1, broadcast of (omega_MAP, diag Hessian); S sharded over the "
                            "ranks by measured stage times (rank 0 samples only if its fit ends before the others would); mu* candidates "
                            "sharded from 3 ranks on (all-reduce max); one all-reduce of 3 x directions doubles"),
            "l2_policy": "working set per step (Sigma, G, factor, Omega, PhiT: > 1 GB) exceeds the 126 MB L2; no explicit flush",
            "fit_start": "value / e2e: cold (GP Newton from f = 0; weight-space Newton from omega = 0); steady_state: warm (appended model)",
            "sampling_engine": "tcgen05 INT8, %d digit planes per operand (error-free splitting; FP64-GEMM accuracy)" % iteration_slices()}


# ------------------------------------------------------------------------------------------------- measured peaks
def measure_int8_peak(lib, torch, dev, sms):
    """INT8 tensor-pipe rate of back-to-back tcgen05.mma.kind::i8 on resident shared-memory operands, one issuing thread per SM,
    all SMs (ppbo_ozaki_mma_rate), timed with CUDA events: the pipe's own ceiling for the sampling kernel's instruction shape"""
    import ctypes
    best, best_cfg = 0.0, None
    out = torch.zeros(sms, dtype=torch.int64, device=dev)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for N, nacc in ((256, 1), (128, 3), (192 if False else 64, 6)):
        iters = 1 << 16
        for rep in range(3):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            rc = lib.ppbo_ozaki_mma_rate(N, 0, nacc, iters, sms, ctypes.c_void_p(out.data_ptr()), st)
            b.record()
            torch.cuda.synchronize()
            if rc != 0:
                break
            tops = sms * iters * 2.0 * 128 * N * 32 / (a.elapsed_time(b) * 1e-3) / 1e12
            if rep > 0 and tops > best:
                best, best_cfg = tops, "M=128 N=%d K=32, %d accumulators" % (N, nacc)
    return best, best_cfg


def measure_fp64_gemm(ops, torch, dev, n=4096):
    A = torch.randn((n, n), dtype=torch.float64, device=dev)
    B = torch.randn((n, n), dtype=torch.float64, device=dev)
    C = torch.empty((n, n), dtype=torch.float64, device=dev)
    best = 0.0
    for rep in range(4):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ops.gemm_nt(A, B, C)
        b.record()
        torch.cuda.synchronize()
        if rep:
            best = max(best, 2.0 * n ** 3 / (a.elapsed_time(b) * 1e-3) / 1e12)
    return best


def recorded_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture (profiles/traffic.json, written by
    scripts/ncu_summary.py from the .ncu-rep of the same launch); None when no capture is recorded for this shape"""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            rec = json.load(fh)
        e = rec.get(kernel_key)
        return (e["dram_bytes"], e["source"]) if e else (None, None)
    except Exception:
        return None, None


# ------------------------------------------------------------------------------------------------- parity gate
def parity_gate(prob, gp, rff, sums_full, S, iteration, ops, torch):
    """The timed cold iteration's results against the committed oracle fixture and the reference's gradient formula, on the host."""
    import scipy.linalg
    from oracle import ppbo_oracle as O
    path = os.path.join(ROOT, "tests", "golden", "full_%s.npz" % prob["name"])
    gate = {"fixture": os.path.relpath(path, ROOT) if os.path.exists(path) else None}
    X, theta, Q, m = prob["X"], prob["theta"], prob["Q"], prob["m"]
    f = gp.f_map.cpu().numpy()
    Sigma = O.regularize_covariance(O.se_kernel(X, X, theta), svd_roundtrip=False)
    a = scipy.linalg.cho_solve(scipy.linalg.cho_factor(Sigma, lower=True), f)
    gate["grad_norm_ref_formula"] = float(np.linalg.norm(-a + O.lik_beta(f, Q, m, theta[0])))      # src/gp_model.py:228-240
    ei_full, _ = iteration.acquisition_values(sums_full.cpu().numpy(), S)
    gate["direction_full_S"] = int(np.argmax(ei_full))
    if gate["fixture"] is None:
        return gate
    z = np.load(path)
    gate["mode_rel"] = float(np.abs(f - z["f_tight"]).max() / np.abs(z["f_tight"]).max())
    gate["grad_norm_oracle_mode"] = float(z["grad_norm_tight"])
    w = rff.omega_map.cpu().numpy()
    gate["omega_rel"] = float(np.abs(w - z["omega_tight"]).max() / np.abs(z["omega_tight"]).max())
    # sampled acquisition on the fixture's slice of the Philox stream, with the pipeline's own fits
    Ss = int(z["slice_samples"])
    dev = gp.f_map.device
    grids = ops.to_dev(prob["grids"])
    B, P, D = prob["grids"].shape
    PhiT = iteration.SlicedGrids(iteration.rff_grid_features(rff.W, rff.b, theta[2], grids))
    mustar = iteration.mustar_over_candidates(gp, grids.reshape(B * P, D))
    gate["mustar_rel"] = float(abs(float(mustar.cpu()[0]) - float(z["mustar"])) / abs(float(z["mustar"])))
    class _OneRank(iteration.Shard):          # the gate runs on rank 0 alone: no collective
        def __init__(self):
            self.dist, self.group, self.rank, self.world = None, None, 0, 1
    sums, fmax, arg = iteration.rff_acquisition(rff, PhiT, Ss, mustar, shard=_OneRank(), seed=int(z["seed"]), bounds=(0, Ss))
    sums = sums.cpu().numpy()
    ref = z["slice_sums"]
    gate["slice_samples"] = Ss
    gate["slice_sums_rel"] = float(np.abs(sums - ref).max() / np.abs(ref).max())
    gate["direction_slice"] = int(np.argmax(sums[:, 0]))
    gate["direction_oracle"] = int(z["slice_direction"])
    gate["direction_matches_oracle"] = bool(gate["direction_slice"] == gate["direction_oracle"])
    decided = z["slice_gap"] > 1e-9 * np.abs(z["slice_fmax"]).max()
    gate["argmax_identical_frac"] = float(np.mean(arg.cpu().numpy()[decided] == z["slice_arg"].astype(np.int32)[decided]))
    gate["pass"] = bool(gate["mode_rel"] <= 1e-6 and gate["omega_rel"] <= 1e-6 and gate["slice_sums_rel"] <= 1e-6 and
                        gate["direction_matches_oracle"] and gate["argmax_identical_frac"] == 1.0)
    return gate


# ------------------------------------------------------------------------------------------------- --dump-outputs
DUMP_MATRIX_BYTES = 16 << 20        # per matrix: the outputs stay far below 64 MB in all
DUMP_SEED = 0


def dump_outputs(dirname, sums, gp, rff):
    """What run_iteration returned to its caller, as DIR/<name>.npy in float64: the per-direction sums, the GP mode and
    alpha, the weight-space mode and its Hessian diagonal in full; of Sigma [N x N] and Phi_X [F x N] a fixed seeded sample of
    rows (the row numbers in <name>_index.npy).  The inputs and the sample depend only on the arguments, so two builds run
    with the same arguments can be compared file for file."""
    os.makedirs(dirname, exist_ok=True)
    arrays = {"sums": sums}
    if gp is not None:
        arrays.update(f_map=gp.f_map, alpha=gp.alpha, Sigma_rows=gp.Sigma)
    if rff is not None:
        arrays.update(omega_map=rff.omega_map, hess_diag=rff.hess_diag, Phi_X_rows=rff.Phi_X)
    for name, t in arrays.items():
        if t is None:
            continue
        a = t.detach().cpu().numpy().astype(np.float64)
        if name.endswith("_rows"):
            k = min(a.shape[0], max(1, DUMP_MATRIX_BYTES // (8 * a.shape[1])))
            idx = np.sort(np.random.RandomState(DUMP_SEED).choice(a.shape[0], k, replace=False))
            a = a[idx]
            np.save(os.path.join(dirname, name + "_index.npy"), idx.astype(np.float64))
        np.save(os.path.join(dirname, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------- src/ API leg (configs 1-3)
def api_leg(torch):
    """BASELINE configs 1-3 through the reference's own API (ppbo_numerical_main.py:102-124): update_feedback_processing_object ->
    update_data -> update_model -> next_query('EI-EXT-FAST'), host numpy arrays in and out, host wall clock.  The model is fitted
    on Q - 1 queries first, the timed iteration appends the last one (the warm start pads the previous mode, src/gp_model.py:375-377);
    a cold update_model at the full size is timed beside it."""
    src = os.path.join(ROOT, "src")
    if src not in sys.path:
        sys.path.insert(1, src)
    import acquisition
    from gp_model import GPModel
    from ppbo_settings import PPBO_settings
    from ppbo_b200 import synthetic
    out = {}
    for name in ("camel2d", "hartmann6d", "camphor6d"):
        cfg = synthetic.CONFIGS[name]
        D, Q, m = cfg["D"], cfg["Q"], cfg["m"]
        _, log, _ = synthetic.make_design(D, Q, m, seed=0)
        rows = np.array([np.concatenate([a * xi + x, xi, [a]]) for xi, x, a in log])           # bounds (0,1)^D: scaled == original units
        res = {"N": Q * (m + 1)}
        try:
            for mode in ("warmup", "cold", "append"):        # the first pass loads every kernel of the path (CUDA loads modules lazily)
                np.random.seed(0)
                st = PPBO_settings(D=D, bounds=((0, 1),) * D, xi_acquisition_function="EI-EXT-FAST", m=m, theta_initial=list(cfg["theta"]),
                                   kernel=cfg["kernel"], verbose=False, alpha_grid_distribution="equispaced")
                gp = GPModel(st)
                if mode == "append":
                    gp.update_feedback_processing_object(rows[:-1])
                    gp.update_data()
                    gp.turn_initialization_off()
                    gp.update_model()
                    gp.fMAP_random_initial_vector = False
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                gp.update_feedback_processing_object(rows)
                gp.update_data()
                if mode != "append":
                    gp.turn_initialization_off()
                t1 = time.perf_counter()
                calls0, launches0 = getattr(gp, "mu_pred_calls", 0), getattr(gp, "mu_star_launches", 0)
                gp.update_model()
                t2 = time.perf_counter()
                xi, x = acquisition.next_query(st, gp, unscale=True)
                t3 = time.perf_counter()
                if mode == "warmup":
                    continue
                res[mode] = {"total_ms": 1e3 * (t3 - t0), "feedback_ms": 1e3 * (t1 - t0), "update_model_ms": 1e3 * (t2 - t1),
                             "fit_ms": 1e3 * gp.timing.get("fit", float("nan")), "mu_star_ms": 1e3 * gp.timing.get("mu_star", float("nan")),
                             "mu_pred_evaluations": getattr(gp, "mu_pred_calls", 0) - calls0,
                             "mu_star_search": "%s, windows of %s" % (getattr(gp, "mustar_method", "?"), getattr(gp, "mustar_window", "?")),
                             "mu_star_launches": getattr(gp, "mu_star_launches", 0) - launches0, "next_query_ms": 1e3 * (t3 - t2),
                             "next_query_parts_ms": {k: round(1e3 * v_, 2) for k, v_ in gp.timing.items() if k.startswith("acq_")},
                             "fit_iterations": gp.fit_stats["iterations"], "selected_direction": int(np.argmax(xi != 0))}
        except Exception as e:       # the leg is a report, never a reason to lose the bench line
            res["error"] = "%s: %s" % (type(e).__name__, e)
        out[name] = res
    return out


# ------------------------------------------------------------------------------------------------- our arm
def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    import torch
    import torch.distributed as dist
    from ppbo_b200 import _lib, iteration, ops, synthetic

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=90))
    lib = _lib.load()
    shard = iteration.Shard()
    W_steps, K = max(args.warmup, 3), args.steps

    cfg = synthetic.CONFIGS[args.config]
    Q0 = cfg["Q"]
    n_extra = W_steps + K
    big = synthetic.make_problem(args.config, S=args.samples, Q=Q0 + n_extra)      # the first Q0 queries are the base problem
    prob = synthetic.make_problem(args.config, S=args.samples)
    kernel, theta, m, S = prob["kernel"], prob["theta"], prob["m"], prob["S"]
    n0 = Q0 * (m + 1)
    assert np.array_equal(big["X"][:n0], prob["X"])
    B, P, D = prob["grids"].shape
    Fdim = prob["F"]
    # f_init = None: cold start of the GP Newton iteration at f = 0; omega0 = None: weight-space Newton from omega = 0
    inputs = iteration.IterationInputs(prob["X"], None, prob["W"], prob["b"], None, prob["grids"])
    sums_host = torch.empty((B, 3), dtype=torch.float64).pin_memory()
    blocks_host = [torch.from_numpy(np.ascontiguousarray(big["X"][(Q0 + i) * (m + 1):(Q0 + i + 1) * (m + 1)])).pin_memory()
                   for i in range(n_extra)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    shares, smu = [None], [None]

    def step(resident=None, timers=None):
        d = resident if resident is not None else inputs.to_device(dev)
        sums, gp, rff = iteration.run_iteration(d, kernel, theta, Q0, m, S, shard=shard, seed=SEED, timers=timers, shares=shares[0],
                                                shard_mustar=smu[0])
        if resident is None:
            sums_host.copy_(sums, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            ei, var = iteration.acquisition_values(sums_host.numpy(), S)
            return int(np.argmax(ei)), gp, rff
        return sums, gp, rff

    step_marks = {}
    held = [None]

    def timed_run(resident):
        import gc
        gc.collect()
        gc.disable()                       # a generation-2 collection inside the timed region is a host hiccup, not the workload
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = lib.ppbo_launch_count()
        marks = [time.perf_counter()]
        e0.record()
        out, held[0] = held[0], None       # the previous step's products stay alive until the next step has replaced them,
        for _ in range(K):                 # in the warm-up as in the timed steps: the allocator pool is in its steady state
            out = step(resident)
            marks.append(time.perf_counter())      # host time after the step was issued (e2e: after its result arrived)
        held[0] = out
        e1.record()
        torch.cuda.synchronize()
        gc.enable()
        ms = e0.elapsed_time(e1)
        launches = lib.ppbo_launch_count() - l0
        step_marks["resident" if resident is not None else "e2e"] = [1e3 * (b - a) for a, b in zip(marks[:-1], marks[1:])]
        barrier()
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / K, launches, out

    def stage_times(run, reps):
        """mean ms between the stage marks of `reps` runs on this rank"""
        acc = {}
        for _ in range(reps):
            timers = []
            run(timers)
            torch.cuda.synchronize()
            for (n0_, a), (n1_, b_) in zip(timers[:-1], timers[1:]):
                acc.setdefault(n1_, []).append(a.elapsed_time(b_))
        return {k: float(np.mean(v)) for k, v in acc.items()}

    def all_gather_stage(local_dict):
        if world == 1:
            return [local_dict]
        out = [None] * world
        dist.all_gather_object(out, local_dict)
        return out

    # ---- steady state: a persistent model that grows by one comparison set per iteration
    state = [None]

    def steady_reset():
        state[0] = iteration.IterationState(kernel, theta, D, m, Q0 + n_extra, dev, resident["W"], resident["b"], shard=shard)
        iteration.run_iteration(resident, kernel, theta, Q0, m, S, shard=shard, seed=SEED, state=state[0], shares=shares[0])
        torch.cuda.synchronize()

    def steady_step(i, timers=None, host=True):
        """append query Q0 + i to the model and run the iteration; host=True: the block, the grids and the basis come from pinned
        host memory and the result goes back to the host (the e2e definition)"""
        if host:
            d = {"block": blocks_host[i].to(dev, non_blocking=True), "W": inputs.host["W"].to(dev, non_blocking=True),
                 "b": inputs.host["b"].to(dev, non_blocking=True), "grids": inputs.host["grids"].to(dev, non_blocking=True)}
        else:
            d = {"block": blocks_dev[i], "W": resident["W"], "b": resident["b"], "grids": resident["grids"]}
        sums, gp, rff = iteration.run_iteration(d, kernel, theta, Q0 + i + 1, m, S, shard=shard, seed=SEED, timers=timers,
                                                state=state[0], shares=steady_shares[0], shard_mustar=steady_smu[0])
        if host:
            sums_host.copy_(sums, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            ei, var = iteration.acquisition_values(sums_host.numpy(), S)
            return int(np.argmax(ei)), gp, rff
        return sums, gp, rff

    resident = inputs.to_device(dev)
    blocks_dev = [b_.to(dev) for b_ in blocks_host]
    steady_shares, steady_smu = [None], [None]

    def plan(st_all):
        """sample shares and the mu* mode from the per-rank stage times of one iteration with the default partition"""
        t_gp = st_all[0].get("gp_fit", 0.0) + st_all[0].get("mustar", 0.0)
        t_rff = st_all[1].get("rff_fit", 0.0)
        sh = iteration.plan_shares(world, t_gp, t_rff, t_sampling_all[0])
        others_done = t_rff + max(sh[1:])                   # when the ranks >= 1 finish their samples
        return sh, bool(world >= 3 and st_all[0].get("gp_fit", 0.0) >= others_done)
    t_sampling_all = [0.0]
    if args.profile:
        if args.profile == "cold":
            for _ in range(1 + K):
                step(resident)
        else:
            steady_reset()
            for i in range(min(n_extra, 1 + K)):
                steady_step(i, host=False)
        torch.cuda.synchronize()
        return

    # ---- calibration of the sample shares (several ranks): measured stage times of one cold iteration with the default partition
    for _ in range(2):
        held[0] = step(resident)
    if world > 1:
        st_all = all_gather_stage(stage_times(lambda tm: step(resident, tm), 2))
        # the default partition gives every rank >= 1 an equal share: the whole sample set costs the sum of their sampling stages
        t_sampling_all[0] = float(np.sum([s_.get("sampling", 0.0) for s_ in st_all[1:]]))
        shares[0], smu[0] = plan(st_all)
    # The clock sampler starts BEFORE the warm-up: the start-up of nvidia-smi (NVML initialisation, first query) holds driver locks
    # for 50-100 ms, and a host-synchronous step that meets it was a 70-110 ms outlier in the timed region (steps 1-4 of the first
    # timed run, whenever the process came up there).  Its periodic queries keep running through both timed regions.
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
        t_wait = time.perf_counter()
        while not clocks.rows and time.perf_counter() - t_wait < 3.0:      # first sample = start-up is over
            time.sleep(0.02)
    for _ in range(W_steps):
        held[0] = step(resident)           # (a warm-up that drops its products at once leaves the second timed step to
                                           # cudaMalloc a second set of 200 MB buffers: +1 ms on one GPU, up to +10 ms on two)
    ms_dev, launches, out = timed_run(resident)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *out)
    fit_stats = out[1].lap.stats if out[1] is not None else None
    rff_iters = out[2].stats["iterations"] if (out[2] is not None and out[2].stats) else None
    for _ in range(2):
        held[0] = step(None)
    ms_e2e, _, out2 = timed_run(None)
    clk = clocks.stop() if rank == 0 else None

    # stage breakdown of the cold iteration (every rank; rank 0 reports its own and the sampling ranks' mean)
    barrier()
    cold_stages = all_gather_stage(stage_times(lambda tm: step(resident, tm), max(3, min(K, 5))))

    # ---- steady state
    held[0] = None
    steady_reset()
    if world > 1:
        steady_step(0, host=False)            # (first append on a fresh process: one-time workspace growth; it also follows a cold
        steady_smu[0] = False                 # fit, whose single factor is stale: the calibration uses the second append)
        st_all = all_gather_stage(stage_times(lambda tm: steady_step(1, tm, host=False), 1))
        steady_shares[0], steady_smu[0] = plan(st_all)
        steady_reset()
    sel = []
    for i in range(W_steps):
        steady_step(i)
    import gc
    gc.collect()
    gc.disable()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = lib.ppbo_launch_count()
    e0.record()
    steady_fits, steady_marks = [], [time.perf_counter()]
    for i in range(W_steps, W_steps + K):
        o = steady_step(i)
        steady_marks.append(time.perf_counter())
        sel.append(o[0])
        if o[1] is not None:
            steady_fits.append(dict(o[1].lap.stats))
    e1.record()
    torch.cuda.synchronize()
    gc.enable()
    steady_launches = lib.ppbo_launch_count() - l0
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_steady = float(t.item()) / K
    # warm model against a cold fit at the final size (GPU against GPU: consistency of the incremental path, not an oracle check)
    warm_vs_cold = None
    if rank == 0:
        Qf = Q0 + n_extra
        gfin = iteration.gp_fit(ops.to_dev(big["X"]), kernel, theta, Qf, m, tol=1e-9)
        fw, fc = state[0].gp.f_map.cpu().numpy(), gfin.f_map.cpu().numpy()
        warm_vs_cold = float(np.abs(fw - fc).max() / np.abs(fc).max())
        del gfin
    # stage breakdown of a steady-state append: the SECOND append on a fresh state (the first one follows a cold fit, whose factor is
    # the stale one of its single factorisation)
    steady_reset()
    steady_step(0, host=False)
    steady_stages = all_gather_stage(stage_times(lambda tm: steady_step(1, tm, host=False), 1))
    state[0] = None

    # ---- acquisition stage alone: S samples x P points x B directions, even shares over ALL ranks (sample-points / s)
    rffs = out[2]
    if rffs is None or rffs.omega_map is None:
        raise SystemExit("no weight-space fit on this rank")
    lo, hi = shard.bounds(S)
    PhiT = iteration.rff_grid_features(resident["W"], resident["b"], theta[2], resident["grids"])
    engine = iteration.sampling_engine(hi - lo, P, Fdim)
    PhiS = iteration.SlicedGrids(PhiT) if engine == "i8" else PhiT
    mu_dev = torch.zeros(1, dtype=torch.float64, device=dev)
    acq_ms = []
    for i in range(3 + 5):
        barrier()
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        iteration.rff_acquisition(rffs, PhiS, S, mu_dev, shard=shard, seed=SEED, bounds=(lo, hi))
        b_.record()
        torch.cuda.synchronize()
        if i >= 3:
            acq_ms.append(a.elapsed_time(b_))
    t = torch.tensor([float(np.mean(acq_ms))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    acq_t = float(t.item())
    sample_points_per_s = S * P * B / (acq_t * 1e-3)

    # ---- the dominant kernel (sampling contraction with fused row max) timed with CUDA events on its stream
    ks = iteration.SAMPLING_SLICES
    Omega = ops.rff_sample_omega(rffs.omega_map, rffs.hess_diag, hi - lo, seed=SEED, sample0=lo)
    flops = 2.0 * (hi - lo) * Fdim * P * B                       # SURVEY.md 8d K3: 2 S F P per direction
    if engine == "i8":
        ap, asc = ops.ozaki_slice(Omega, 0, ks)
        fm = torch.empty((B, hi - lo), dtype=torch.float64, device=dev)
        am = torch.empty((B, hi - lo), dtype=torch.int32, device=dev)

        def dominant():
            ops.ozaki_rowmax(ap, asc, hi - lo, PhiS.planes, PhiS.scale, P, B, Fdim, ks, fmax=fm, arg=am)
    else:
        def dominant():
            ops.rff_eval_argmax(Omega, PhiT)
    gemm_ms = []
    for i in range(3 + 5):
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        dominant()
        b_.record()
        torch.cuda.synchronize()
        if i >= 3:
            gemm_ms.append(a.elapsed_time(b_))
    gemm_t = float(np.mean(gemm_ms))
    fp64_equiv = flops / (gemm_t * 1e-3) / 1e12

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    sms = lib.ppbo_device_sm_count(local)
    fp64_gemm = measure_fp64_gemm(ops, torch, dev)
    if engine == "i8":
        # KS (KS+1)/2 exact INT8 plane products per FP64 product
        ops_per_launch = flops * ks * (ks + 1) / 2
        achieved = ops_per_launch / (gemm_t * 1e-3) / 1e12
        peak, peak_cfg = measure_int8_peak(lib, torch, dev, sms)
        bf16 = None
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                bf16 = float(json.load(fh)["bf16_tflops"])
        except Exception:
            pass
        key = "ozaki_rowmax_kernel<%d,64>@%s/S=%d/P=%d/B=%d" % (ks, args.config, hi - lo, P, B)
        traffic, traffic_src = recorded_traffic(key)
        roof = {"kernel": "ozaki_rowmax_kernel<%d,64> (RFF sampling contraction on tcgen05.mma.kind::i8, %d digit planes per operand, "
                          "fused per-sample max/arg-max)" % (ks, ks),
                "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TOP/s", "frac": achieved / peak if peak else None,
                "peak_source": "measured in this run: back-to-back tcgen05.mma.kind::i8 on all %d SMs (ppbo_ozaki_mma_rate, %s)" % (sms, peak_cfg),
                "frac_of_2x_bf16_measured": achieved / (2 * bf16) if bf16 else None,
                "traffic": traffic, "traffic_unit": "bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum, ncu)",
                "traffic_source": traffic_src,
                "algorithmic_bytes": float(ap.numel() + PhiS.planes.numel()),      # every digit plane read once
                "kernel_ms": gemm_t, "ops_per_launch": ops_per_launch, "fp64_equivalent_tflops": fp64_equiv,
                "fp64_dmma_peak_tflops": FP64_TENSOR_PEAK_TFLOPS, "fp64_gemm_measured_tflops": fp64_gemm}
    else:
        achieved = fp64_equiv
        roof = {"kernel": "gemm_nt_rowmax_kernel (RFF sampling GEMM, fused per-sample max/arg-max)", "bound": "tensor",
                "achieved": achieved, "peak": FP64_TENSOR_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": achieved / FP64_TENSOR_PEAK_TFLOPS,
                "traffic": None, "kernel_ms": gemm_t, "flops_per_launch": flops, "fp64_gemm_measured_tflops": fp64_gemm,
                "peak_source": "FP64 DMMA pipe measured on this pool (profiles/r01_fp64_peaks_ubench.txt); "
                               "MEASURED_PEAKS.json has no FP64 figure"}

    def merge(stages):
        """rank 0's own stages plus the mean sampling time of the ranks that sample"""
        o = dict(stages[0])
        samp_ = [s_["sampling"] for s_ in stages[1:] if "sampling" in s_]
        if samp_:
            o["sampling_other_ranks_mean"] = float(np.mean(samp_))
        if len(stages) > 1 and "rff_fit" in stages[1]:
            o["rff_fit_rank1"] = stages[1]["rff_fit"]
        return o

    gate = parity_gate(prob, out[1], out[2], out[0], S, iteration, ops, torch) if out[1] is not None else None
    line = {
        "metric": METRIC, "value": ms_dev, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W_steps,
        "ms_per_step": ms_dev, "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload_config(prob, world),
        "e2e": {"value": ms_e2e, "unit": UNIT, "h2d_bytes_per_step": inputs.nbytes(), "d2h_bytes_per_step": B * 3 * 8,
                "selected_direction": out2[0]},
        "gpu_launches": int(launches),
        "clocks": clk,
        "roofline": roof,
        "stages_ms": merge(cold_stages),
        "stages_note": ("one GPU: rff_fit and sampling time the foreground chain (weight-space fit, then draws + INT8 contraction); the GP "
                        "fit and mu* run concurrently on the background thread, gp_tail is what is left of them when the contraction "
                        "has ended" if world == 1 else "rank 0's stages; sampling_other_ranks_mean / rff_fit_rank1 from the other ranks"),
        "steady_state": {"value": ms_steady, "unit": UNIT, "what": "e2e (pinned host buffers in, sums out) per appended query, queries %d..%d "
                         "appended to the fitted %d-query model" % (Q0 + W_steps + 1, Q0 + W_steps + K, Q0),
                         "h2d_bytes_per_step": int(blocks_host[0].numel() * 8 + sum(inputs.host[k].numel() * 8 for k in ("W", "b", "grids"))),
                         "d2h_bytes_per_step": B * 3 * 8, "gpu_launches": int(steady_launches), "stages_ms": merge(steady_stages),
                         "factorizations_per_step": [int(s_["factorizations"]) for s_ in steady_fits],
                         "chord_steps_per_step": [int(s_["chord_steps"]) for s_ in steady_fits],
                         "host_ms_per_step": [round(1e3 * (b_ - a_), 2) for a_, b_ in zip(steady_marks[:-1], steady_marks[1:])],
                         "selected_directions": sel, "warm_vs_cold_mode_rel": warm_vs_cold,
                         "sample_shares": steady_shares[0], "mustar_sharded": steady_smu[0]},
        "sample_shares": shares[0], "mustar_sharded": smu[0],
        # diagnostics: host time per issued step (resident steps are issued asynchronously, e2e steps end with the result on the host)
        "resident_host_ms_per_step": [round(t_, 2) for t_ in step_marks.get("resident", [])],
        "e2e_host_ms_per_step": [round(t_, 2) for t_ in step_marks.get("e2e", [])],
        "fit_newton_iterations": fit_stats["iterations"] if fit_stats else None,
        "fit_factorizations": fit_stats["factorizations"] if fit_stats else None,
        "rff_newton_iterations": rff_iters,
        "rff_sample_points_per_s": sample_points_per_s, "rff_sample_points_per_s_per_gpu": sample_points_per_s / world,
        "acquisition_stage_ms_even_shares": acq_t,
        "parity_gate": gate,
    }
    if world == 1 and not args.no_api_leg:
        line["e2e_api"] = api_leg(torch)
    if world == 1 and not args.no_cpu_baseline:
        arm = ReferenceArm(prob)
        per = [arm.step() for _ in range(2)]
        v = arm.iteration_ms(float(np.mean(per)))
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": arm.threads or host_threads(), "kind": "port",
                                "sample": arm.sample_text(float(np.mean(per))), "extrapolated": True}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
