#!/usr/bin/env python
"""bench.py -- DagmaLinear inner Adam iterations/second on the batched d=64 sweep.

Workload (BASELINE.json configs[3], "C4"): independent DagmaLinear l2 problems, ER4 graphs,
d=64, n=1000, 1024 seeds x lambda1 in {0.01, 0.02, 0.03, 0.05}; 4096 problems per GPU
(weak scaling: every rank owns its own 4096 problems, no data-path collective).

A "step" is one pass of the hot path over the batch: one `DagmaLinear.minimize` call of
`checkpoint` = 1000 inner iterations (mu=1, s=1, lr=3e-4; tol=0 so no problem stops early)
for every problem, i.e. 4096 x 1000 inner Adam iterations per GPU per step.

    value  : problem-iterations / s, inputs resident in HBM (CUDA events, max over ranks)
    e2e    : same metric through the public host API `minimize_batch` on pinned host
             buffers (H2D of W and cov, kernel, D2H of W inside the timed region)
    roofline: 4 d^3 flop per iteration (inverse 2d^3 + cov@(I-W) 2d^3) against the FP64
             pipe peak measured live with the DFMA/DMMA yardstick kernels
    cpu_baseline / --impl reference: the UNMODIFIED reference class (dagma.linear.DagmaLinear
             imported from /root/reference/src, kind "reference") when that tree exists, else the
             numpy restatement of it (oracle/linear_ref.py, bit-identical to it in the build
             container, kind "port" -- /root/reference does not exist on the GPU box); one
             single-threaded-BLAS process per host core, bounded sample.
    parity_sample: 24 of the 4096 problems of the full default fit against the fits of the unmodified
             reference recorded in tests/golden/fit_c4_sample24.npz (edge sets, |dW| next to the
             reference's own inv(M.T).T round-off envelope).
    --dump-outputs DIR: what the last timed step returned, as DIR/<name>.npy (W of a fixed, seeded sample of
             the problems, status and stage statistics of all of them), to compare two builds output for output;
             the inputs depend only on the arguments.
    c5 / c2 / c3 / c1: the other configs of BASELINE.json (own roofline / e2e / CPU sample each);
    with --gpus N > 1 also the row-sharded C2 / C3 iterations and a strong-scaling C4 step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the bench leaves the tree as it found it (it may be read-only): no byte-code caches beside the sources, also in the
# spawned CPU-baseline workers, which import this file first
sys.dont_write_bytecode = True

D, N_SAMPLES, K_EDGES = 64, 1000, 4
LAMBDAS = (0.01, 0.02, 0.03, 0.05)
ITERS_PER_STEP = 1000
FLOP_PER_ITER = 4.0 * D ** 3
DUMP_PROBLEMS = 512     # --dump-outputs: W of a fixed, seeded sample of the problems (512 x 64 x 64 float64 = 16.8 MB)


# --------------------------------------------------------------------------- data
def make_covs(n_seeds: int, seed0: int):
    """[n_seeds, n, d] synthetic ER4 gaussian SEM data (oracle/simulate.py is only a data generator here)."""
    import numpy as np
    from oracle import simulate
    X = np.empty((n_seeds, N_SAMPLES, D))
    for i in range(n_seeds):
        X[i], _ = simulate.make_linear_problem(D, K_EDGES, N_SAMPLES, "ER", "gauss", seed0 + i)
    return X


# --------------------------------------------------------------------------- CPU arm
REFERENCE_SRC = "/root/reference/src"


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_SRC, "dagma", "linear.py"))


class _Bar:
    def update(self, *_a, **_k):
        pass


def _reference_minimize(X, lam, iters):
    """`iters` inner iterations of the UNMODIFIED reference DagmaLinear.minimize (set-up as fit() does, linear.py:406-429)."""
    import numpy as np
    sys.dont_write_bytecode = True
    if REFERENCE_SRC not in sys.path:
        sys.path.insert(0, REFERENCE_SRC)
    from dagma.linear import DagmaLinear as RefLinear
    m = RefLinear("l2")
    m.X, m.lambda1, m.checkpoint = X, lam, ITERS_PER_STEP
    m.n, m.d = X.shape
    m.Id = np.eye(m.d)
    m.X -= X.mean(axis=0, keepdims=True)
    m.exc_r = m.exc_c = m.inc_r = m.inc_c = None
    m.cov = X.T @ X / float(m.n)
    calls = [0]
    adam = m._adam_update

    def tap(*a, **k):
        calls[0] += 1
        return adam(*a, **k)

    m._adam_update = tap
    t0 = time.perf_counter()
    m.minimize(np.zeros((m.d, m.d)), 1.0, iters, 1.0, lr=3e-4, tol=0.0, pbar=_Bar())
    return calls[0], time.perf_counter() - t0


def _cpu_worker(args):
    seed, lam, iters, kind = args
    import numpy as np
    from threadpoolctl import threadpool_limits
    from oracle import simulate
    with threadpool_limits(limits=1):
        X, _ = simulate.make_linear_problem(D, K_EDGES, N_SAMPLES, "ER", "gauss", seed)
        if kind == "reference":
            return _reference_minimize(X, lam, iters)
        from oracle.linear_ref import OracleLinear
        o = OracleLinear("l2").prepare(X, lam, checkpoint=ITERS_PER_STEP)
        t0 = time.perf_counter()
        o.minimize(np.zeros((D, D)), 1.0, iters, 1.0, 3e-4, tol=0.0)
        return o.last_iters, time.perf_counter() - t0


def cpu_kind() -> str:
    return "reference" if reference_available() else "port"


def cpu_what(kind: str) -> str:
    return ("the unmodified reference dagma.linear.DagmaLinear.minimize (numpy/scipy)" if kind == "reference" else
            "oracle/linear_ref.py (numpy/scipy restatement of the reference)")


def cpu_rate(iters: int, rounds: int = 1, kind: str = None):
    """problem-iterations/s of the CPU implementation with one single-thread process per host core."""
    import multiprocessing as mp
    kind = kind or cpu_kind()
    cores = len(os.sched_getaffinity(0))
    jobs = [(1000 + i, LAMBDAS[i % 4], iters, kind) for i in range(cores * rounds)]
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker, [(1000, 0.02, 5, kind)] * cores)    # spawn + import warm-up
        t0 = time.perf_counter()
        res = pool.map(_cpu_worker, jobs, chunksize=1)
        wall = time.perf_counter() - t0
    done = sum(r[0] for r in res)
    return done / wall, cores, done, wall


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    iters = 20000      # ~3 s of CPU work per core and step: the whole --steps 5 run stays well under a minute
    for _ in range(args.warmup):
        pass   # process-pool warm-up happens inside cpu_rate
    rates = []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        rate, cores, done, wall = cpu_rate(iters)
        rates.append((rate, done, wall))
    total_wall = sum(r[2] for r in rates)
    total_done = sum(r[1] for r in rates)
    value = total_done / total_wall
    kind = cpu_kind()
    sample = (f"{cores} problems (one per core) x {iters} inner iterations per step of {cpu_what(kind)}, "
              "single-thread BLAS per process")
    line = {
        "impl": "reference", "metric": "DagmaLinear inner Adam iters/sec (batched d=64)", "value": value,
        "unit": "problem-iterations/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total_wall / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "C4: DagmaLinear l2 minimize, ER4 d=64 n=1000, mu=1 s=1 lr=3e-4", "d": D,
                   "n": N_SAMPLES, "iters_per_problem_per_step": iters},
        "cpu_baseline": {"value": value, "unit": "problem-iterations/s", "cores": cores, "kind": kind,
                         "sample": sample},
        "e2e": {"value": value, "unit": "problem-iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        rows = [r.strip().split(", ") for r in self.f.read().splitlines() if r.count(",") >= 5]
        os.unlink(self.f.name)
        if not rows:
            return out
        sm = sorted(int(float(r[0])) for r in rows)
        out["sm_mhz"] = sm[len(sm) // 2]
        out["sm_max_mhz"] = int(float(rows[0][1]))
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for i, nme in enumerate(names):
            if any(r[2 + i].strip().lower().startswith("active") for r in rows):
                out["reasons"].append(nme)
        out["samples"] = len(rows)
        return out


# --------------------------------------------------------------------------- GPU arm
def fp64_peak_tflops(torch, _lib, sms):
    """FP64 pipe peak measured live (DFMA and DMMA.8x8x4 yardsticks; the larger is the denominator)."""
    lib = _lib.load()
    sink = torch.zeros(8, dtype=torch.float64, device="cuda")
    best = {}
    for name, fn, flops in (("dfma", lib.dagma_bench_fp64_fma, lambda c, t, i: c * t * i * 32.0),
                            ("dmma", lib.dagma_bench_fp64_dmma, lambda c, t, i: c * (t // 32) * i * 8 * 512.0)):
        ctas, threads, iters = sms * 4, 512, 4000 if name == "dfma" else 500
        fn(_lib.stream_ptr(), ctas, threads, iters, sink.data_ptr())
        torch.cuda.synchronize()
        tbest = 1e9
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn(_lib.stream_ptr(), ctas, threads, iters, sink.data_ptr())
            e1.record()
            torch.cuda.synchronize()
            tbest = min(tbest, e0.elapsed_time(e1) * 1e-3)
        best[name] = flops(ctas, threads, iters) / tbest / 1e12
    # cuBLAS DGEMM 8192^3 through torch.matmul: the practical FP64 tensor peak SURVEY.md 7.3 asks the bench to record
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    c = torch.empty(n, n, dtype=torch.float64, device="cuda")
    torch.matmul(a, b, out=c)
    torch.cuda.synchronize()
    tbest = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b, out=c)
        e1.record()
        torch.cuda.synchronize()
        tbest = min(tbest, e0.elapsed_time(e1) * 1e-3)
    best["cublas_dgemm_8192"] = 2.0 * n ** 3 / tbest / 1e12
    del a, b, c
    return best


def traffic_from_profile(kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of `kernel`, parsed from the committed ncu summary
    that profiles/roofline_sources.json names for it (None when there is no capture)."""
    import re
    try:
        src = json.load(open(os.path.join(ROOT, "profiles", "roofline_sources.json")))[kernel]
        text = open(os.path.join(ROOT, src["file"])).read()
    except (OSError, KeyError, ValueError):
        return None, None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    total = 0.0
    for name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
        m = re.search(re.escape(name) + r" \[(\w+)\] = ([0-9.,]+)", text)
        if not m:
            return None, None
        total += float(m.group(2).replace(",", "")) * unit[m.group(1)]
    return total, src


def parity_sample(W_raw, stage_iters):
    """The fitted W of the sampled problems of the 4096-batch against the full default fits of the UNMODIFIED
    reference (tests/golden/fit_c4_sample24.npz, oracle/make_golden_scale.py c4): per-problem edge-set identity,
    |dW| next to the reference's own round-off envelope (the same fit with inv(M.T).T, SURVEY.md 7.4)."""
    import numpy as np
    path = os.path.join(ROOT, "tests", "golden", "fit_c4_sample24.npz")
    if not os.path.exists(path):
        return None
    g = np.load(path)
    probs = [int(p) for p in g["problems"]]
    if max(probs) >= len(W_raw):
        return None
    Wr = g["W_reference"]
    rows, n_same, n_env_same = [], 0, 0
    for k, p in enumerate(probs):
        W = W_raw[p]
        e_gpu, e_ref = np.abs(W) >= 0.3, np.abs(Wr[k]) >= 0.3
        diff = int((e_gpu != e_ref).sum())
        env_diff = int(g["envelope_edge_diff"][k])
        n_same += diff == 0
        n_env_same += env_diff == 0
        ref_iters = [int(c[0]) for c in g["calls_reference"][k] if c[0] >= 0]
        row = {"problem": p, "edge_diff": diff, "max_abs_dW": float(np.abs(W - Wr[k]).max()),
               "envelope_max_abs_dW": float(g["envelope_max_abs_dW"][k]), "envelope_edge_diff": env_diff,
               "stage_iters": [int(x) for x in stage_iters[p]], "reference_stage_iters": ref_iters}
        if diff:
            bad = np.argwhere(e_gpu != e_ref)
            row["exceptions"] = [{"edge": [int(i), int(j)], "W_gpu": float(W[i, j]), "W_ref": float(Wr[k][i, j]),
                                  "margin_ref": float(abs(abs(Wr[k][i, j]) - 0.3))} for i, j in bad[:8]]
        rows.append(row)
    dws = np.array([r["max_abs_dW"] for r in rows])
    envs = np.array([r["envelope_max_abs_dW"] for r in rows])
    return {"problems": len(probs), "identical_edge_sets": int(n_same), "reference_envelope_identical_edge_sets": int(n_env_same),
            "max_abs_dW_median": float(np.median(dws)), "max_abs_dW_max": float(dws.max()),
            "envelope_median": float(np.median(envs)), "envelope_max": float(envs.max()),
            "same_stage_lengths": int(sum(r["stage_iters"] == r["reference_stage_iters"] for r in rows)),
            "source": "tests/golden/fit_c4_sample24.npz (unmodified reference; envelope = the reference with inv(M.T).T)",
            "per_problem": rows}


def bench_c5(torch, _lib, peak_tflops, with_cpu):
    """BASELINE.json configs[4]: one DagmaLinear l2 problem, SF4 d=2000 n=20000 -- inner iterations / s of the
    multi-CTA path (blocked DMMA inverse + cov@W DGEMM + fused update), each replayed as a CUDA graph and
    timed with CUDA events; the numpy restatement of the reference is timed beside it on a few iterations."""
    import numpy as np
    from oracle import simulate
    from midagma_b200 import DagmaLinear
    d, n = 2000, 20000
    X, _ = simulate.make_linear_problem(d, 4, n, "SF", "gauss", 0)
    model = DagmaLinear("l2")
    model.fit(X.copy(), lambda1=0.02, T=1, warm_iter=0, max_iter=0)        # centring + covariance on the GPU
    eng = model._large_engine()
    W = np.zeros((d, d))
    model.minimize(W, 1.0, 30, 1.0, lr=3e-4)                               # captures the iteration graph
    torch.cuda.synchronize()

    def graph_of(fn):
        fn()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
        return g

    def timed(g, reps=20):
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3 / reps

    t_it = timed(eng._graph)
    t_inv = timed(graph_of(lambda: eng._inverse(1.0)))
    t_gemm = timed(graph_of(lambda: eng._score_T()))
    inv_tf = 2.0 * d ** 3 / t_inv / 1e12
    traffic, src = traffic_from_profile("outer_step_kernel")
    out = {"workload": "C5: single DagmaLinear l2 problem, SF4 d=2000 n=20000, mu=1 s=1 lr=3e-4 (graph-replayed inner iteration)",
           "ms_per_iter": t_it * 1e3, "iters_per_s": 1.0 / t_it, "flop_per_iter": 4.0 * d ** 3,
           "tflops": 4.0 * d ** 3 / t_it / 1e12, "frac_of_fp64_peak": 4.0 * d ** 3 / t_it / 1e12 / peak_tflops,
           "inverse_ms": t_inv * 1e3, "inverse_tflops": inv_tf,
           "inverse_frac_of_fp64_peak": inv_tf / peak_tflops,
           "score_gemm_ms": t_gemm * 1e3, "score_gemm_tflops": 2.0 * d ** 3 / t_gemm / 1e12,
           "roofline": {"bound": "tensor", "achieved": inv_tf, "peak": peak_tflops, "unit": "TFLOP/s",
                        "frac": inv_tf / peak_tflops,
                        # per LAUNCH of outer_step_kernel (one of the 8 outer steps of an inverse): 2 d^3 / 8 flop
                        "traffic": traffic, "traffic_source": src,
                        "kernel": "outer_step_kernel x ceil(d / 256) launches = one blocked inverse (2 d^3 flop)",
                        "flop_per_unit": 2.0 * d ** 3, "units_per_launch": 1.0 / 8}}
    # ---- e2e: the call a reference user makes -- host X in, thresholded W_est out (reduced schedule of the parity
    # fixture: warm_iter = max_iter = 500; H2D of X, centring + covariance, 2500 iterations with their checkpoint
    # objective evaluations, D2H of W and of the centred X inside the timed region)
    del eng
    import gc
    gc.collect()                                  # the timing engine and its graphs go NOW, not inside the timed fit
    model = DagmaLinear("l2")
    Xh = X.copy()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    W_est = model.fit(Xh, lambda1=0.02, warm_iter=500, max_iter=500, s=[1.0, .9, .8, .7, .6])
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    iters = int(sum(model.stage_iters))
    out["e2e"] = {"value": iters / wall, "unit": "inner iterations/s", "wall_s": wall, "inner_iters": iters,
                  "h2d_bytes": int(X.nbytes), "d2h_bytes": int(X.nbytes + 8 * d * d * 6),
                  "what": "DagmaLinear('l2').fit(X, lambda1=0.02, warm_iter=500, max_iter=500) on host arrays"}
    gpath = os.path.join(ROOT, "tests", "golden", "fit_c5_reduced.npz")
    if os.path.exists(gpath):
        g = np.load(gpath)
        idx = np.cumsum(g["w_idx_delta"].astype(np.int64))         # flat indices of the entries |W_ref| >= 0.05
        edges_ref = np.zeros(d * d, dtype=bool)
        edges_ref[idx[g["w_edge"]]] = True
        sample = idx[g["w_sample_pos"]]
        out["parity"] = {"edge_set_distance": int(((W_est != 0).ravel() != edges_ref).sum()),
                         "edges": int((W_est != 0).sum()), "reference_edges": int(g["nnz_est"]),
                         "max_abs_dW_on_sampled_ref_entries_ge_0.05":
                             float(np.abs(model.W_raw.ravel()[sample] - g["w_sample_val"]).max()),
                         "stage_iters": model.stage_iters, "reference_wall_s": float(g["wall_s"]),
                         "source": "tests/golden/fit_c5_reduced.npz (the same fit by the unmodified reference)"}
        out["e2e"]["speedup_vs_reference_fit_wall"] = float(g["wall_s"]) / wall
    if with_cpu:
        from oracle.linear_ref import OracleLinear
        o = OracleLinear("l2").prepare(X, 0.02, checkpoint=1000)
        Wc = W.copy()
        o.minimize(Wc, 1.0, 1, 1.0, 3e-4, tol=0.0)
        n_cpu = 30
        t0 = time.perf_counter()
        o.minimize(Wc, 1.0, n_cpu, 1.0, 3e-4, tol=0.0)
        cpu = (time.perf_counter() - t0) / n_cpu
        out["cpu_ms_per_iter"] = cpu * 1e3
        out["cpu_sample"] = (f"{n_cpu} iterations of oracle/linear_ref.py with all host BLAS threads "
                             f"({len(os.sched_getaffinity(0))} cores)")
        out["speedup_vs_cpu"] = cpu / t_it
    return out


def bench_c2_c3(torch, with_cpu, peak_tflops=None):
    import gc
    """BASELINE.json configs[0] (full fit wall clock of the reference's own case), configs[1] and [2]: logistic DagmaLinear (ER2 d=100 n=10000) and DagmaMLP (d=40 m1=10 n=2000):
    wall clock per graph-replayed inner iteration (the host synchronises only at the checkpoints), the numpy
    restatement of the reference beside it on a few iterations."""
    import numpy as np
    from oracle import simulate
    from midagma_b200 import DagmaLinear
    from midagma_b200.nonlinear import DagmaMLP, DagmaNonlinear
    out = {}
    # ---- C1: the reference's own CPU-runnable case, full default fit (one launch of the on-chip kernel)
    X, W_true = simulate.config_c1(0)
    model = DagmaLinear("l2")
    model.fit(X.copy(), lambda1=0.02, s=[1.0, .9, .8, .7, .6])            # warm-up (library load, allocations)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    W_gpu = model.fit(X.copy(), lambda1=0.02, s=[1.0, .9, .8, .7, .6])
    torch.cuda.synchronize()
    t_fit = time.perf_counter() - t0
    iters = int(sum(model.stage_iters))
    c1 = {"workload": "C1: DagmaLinear l2 full default fit, ER2 d=20 n=500 (host arrays in, thresholded W_est out)",
          "fit_wall_s": t_fit, "inner_iters": iters, "us_per_iter": t_fit / iters * 1e6,
          "shd_vs_truth": int(simulate.count_accuracy(W_true != 0, W_gpu != 0)["shd"])}
    if with_cpu:
        from oracle.linear_ref import OracleLinear
        t0 = time.perf_counter()
        W_cpu = OracleLinear("l2").fit(X.copy(), lambda1=0.02)
        cpu = time.perf_counter() - t0
        c1.update({"cpu_fit_wall_s": cpu, "speedup_vs_cpu": cpu / t_fit,
                   "edge_set_distance_vs_cpu": int(simulate.edge_set_distance(W_gpu, W_cpu)),
                   "cpu_sample": "the same full default fit by oracle/linear_ref.py (bit-identical port of the reference)"})
    out["c1"] = c1
    # ---- C2
    X, _ = simulate.config_c2(0)
    d, n = X.shape[1], X.shape[0]
    m = DagmaLinear("logistic")
    m.fit(X.copy(), lambda1=0.02, T=1, warm_iter=0, max_iter=0)
    W = np.zeros((d, d))
    m.minimize(W, 1.0, 200, 1.0, lr=3e-4)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    m.minimize(W, 1.0, 4000, 1.0, lr=3e-4, tol=0.0)
    torch.cuda.synchronize()
    t = (time.perf_counter() - t0) / 4000
    flop = 4.0 * n * d * d + 2.0 * d ** 3
    c2 = {"workload": "C2: DagmaLinear logistic, ER2 d=100 n=10000, mu=1 s=1 lr=3e-4 (4000 inner iterations of DagmaLinear.minimize, "
                      "wall clock; one persistent kernel per checkpoint interval, csrc/lin_iter.cu)",
          "us_per_iter": t * 1e6, "iters_per_s": 1.0 / t, "flop_per_iter": flop, "tflops": flop / t / 1e12}
    if peak_tflops:
        c2["roofline"] = {"bound": "tensor", "achieved": flop / t / 1e12, "peak": peak_tflops, "unit": "TFLOP/s",
                          "frac": flop / t / 1e12 / peak_tflops, "traffic": None,
                          "note": "one persistent kernel: the iteration is bound by the on-chip inverse of the 100 x 100 matrix "
                                  "on ONE CTA (two 64-pivot sweeps + six 64^3 products), the score products of the other "
                                  "147 CTAs hide behind it: the fraction is reported, not a target"}
    gc.collect()                                            # engines / graphs of earlier sections are released NOW, not inside the timed fit
    # e2e: the call a reference user makes -- host X in, thresholded W_est out (reduced schedule T=2 x 1000 iterations)
    m2 = DagmaLinear("logistic")
    Xh = X.copy()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    m2.fit(Xh, lambda1=0.02, T=2, warm_iter=1000, max_iter=1000, s=[1.0, .9])
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    it2 = int(sum(m2.stage_iters))
    c2["e2e"] = {"value": it2 / wall, "unit": "inner iterations/s", "wall_s": wall, "inner_iters": it2,
                 "h2d_bytes": int(X.nbytes), "d2h_bytes": int(8 * d * d * 4),
                 "what": "DagmaLinear('logistic').fit(X, lambda1=0.02, T=2, warm_iter=1000, max_iter=1000) on host arrays"}
    del m2
    if with_cpu:
        from oracle.linear_ref import OracleLinear
        o = OracleLinear("logistic").prepare(X.copy(), 0.02, checkpoint=1000)
        Wc = np.zeros((d, d))
        o.minimize(Wc, 1.0, 1, 1.0, 3e-4, tol=0.0)
        t0 = time.perf_counter()
        o.minimize(Wc, 1.0, 10, 1.0, 3e-4, tol=0.0)
        cpu = (time.perf_counter() - t0) / 10
        c2.update({"cpu_ms_per_iter": cpu * 1e3, "speedup_vs_cpu": cpu / t,
                   "cpu_sample": f"10 iterations of oracle/linear_ref.py with all host BLAS threads ({len(os.sched_getaffinity(0))} cores)"})
    out["c2"] = c2
    # ---- mid-d l2 (64 < d <= 128): one persistent kernel per problem, problems of a batch side by side
    from midagma_b200 import fit_batch
    from midagma_b200.linear import _batch_lanes
    db, nb, itb = 128, 16, 3000
    rngb = np.random.default_rng(0)
    Xb = rngb.normal(size=(nb, 4 * db, db))
    kwb = dict(T=1, warm_iter=itb, max_iter=itb, checkpoint=1000, s=(1.0,), return_info=True)
    fit_batch(Xb[:2], 0.02, **dict(kwb, warm_iter=100, max_iter=100))     # warm-up
    gc.collect()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _, infob = fit_batch(Xb, 0.02, **kwb)
    torch.cuda.synchronize()
    wallb = time.perf_counter() - t0
    lanes = _batch_lanes(db, nb)
    out["mid_d_batch"] = {"workload": f"{nb} independent DagmaLinear l2 problems, d={db} n={4 * db}, one stage of up to {itb} "
                                      "iterations each (fit_batch; host arrays in, W_est out)",
                          "lanes": lanes, "cuda_device_max_connections": os.environ.get("CUDA_DEVICE_MAX_CONNECTIONS"),
                          "wall_s": wallb, "inner_iters": int(infob["total_iters"]),
                          "iters_per_s": infob["total_iters"] / wallb,
                          "us_per_iter_and_lane": wallb / infob["total_iters"] * lanes * 1e6,
                          "flop_per_iter": 4.0 * db ** 3,
                          "what": "every problem's iterations between two checkpoints are one persistent kernel of d/8 + 1 CTAs "
                                  "(csrc/lin_iter.cu); `lanes` problems run side by side, one stream and host thread each"}
    del Xb
    # ---- C3
    X, _ = simulate.config_c3(0)
    d, m1, n = X.shape[1], 10, X.shape[0]
    torch.manual_seed(0)
    model = DagmaMLP(dims=[d, m1, 1], bias=True)
    init = {k: v.detach().clone() for k, v in model.state_dict().items()}
    # the launch sequence DagmaNonlinear.minimize replays (one CUDA graph per iteration), timed with CUDA events
    from midagma_b200 import nonlinear as nlmod
    eng = nlmod._MlpEngine(model, torch.from_numpy(X).cuda())
    sh = eng.state_host
    sh.zero_()
    for f, val in ((nlmod.F_MU, 0.1), (nlmod.F_S, 1.0), (nlmod.F_LR, 2e-4), (nlmod.F_LAM1, 0.02), (nlmod.F_LAM2, 0.005),
                   (nlmod.F_B1, 0.99), (nlmod.F_B2, 0.999), (nlmod.F_GAMMA, 1.0)):
        sh[f] = float(val)
    eng.state.copy_(sh)
    eng.replay(1.0, 500)                                   # warm-up iteration, graph capture, 500 replays
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eng.replay(1.0, 4000)
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) * 1e-3 / 4000
    _, step, halted = eng.pull()
    flop = 2.0 * (2.0 * n * d * d * m1) + 6.0 * n * d * m1 + 2.0 * d ** 3
    c3 = {"workload": "C3: DagmaMLP [40, 10, 1] n=2000, mu=0.1 s=1 lr=2e-4 (4000 iterations of DagmaNonlinear.minimize's engine: "
                      "one persistent kernel, csrc/mlp_iter.cu; CUDA events)",
          "us_per_iter": t * 1e6, "iters_per_s": 1.0 / t, "flop_per_iter": flop, "tflops": flop / t / 1e12,
          "iterations_done": int(step), "halted": int(halted)}
    if peak_tflops:
        c3["roofline"] = {"bound": "tensor", "achieved": flop / t / 1e12, "peak": peak_tflops, "unit": "TFLOP/s",
                          "frac": flop / t / 1e12 / peak_tflops, "traffic": None,
                          "note": "one persistent kernel, two grid barriers per iteration; bound by the 40-pivot sweep of the h CTA "
                                  "and the barriers, not by throughput: the fraction is reported, not a target"}
    gc.collect()
    # e2e: DagmaNonlinear.fit on host X (reduced schedule T=2 x 1000 iterations), thresholded adjacency out
    torch.manual_seed(0)
    model_e = DagmaMLP(dims=[d, m1, 1], bias=True)
    eq = DagmaNonlinear(model_e)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    eq.fit(X.copy(), lambda1=0.02, lambda2=0.005, T=2, warm_iter=1000, max_iter=1000)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    it3 = int(sum(eq.stage_iters))
    c3["e2e"] = {"value": it3 / wall, "unit": "inner iterations/s", "wall_s": wall, "inner_iters": it3,
                 "h2d_bytes": int(X.nbytes), "d2h_bytes": int(8 * d * d),
                 "what": "DagmaNonlinear(DagmaMLP([40,10,1])).fit(X, T=2, warm_iter=1000, max_iter=1000) on a host array"}
    if with_cpu:
        from oracle.nonlinear_ref import OracleMLP, OracleNonlinear
        om = OracleMLP([d, m1, 1], {k: v.numpy() for k, v in init.items()})
        on = OracleNonlinear(om)
        on.minimize(X, 2, 2e-4, 0.02, 0.005, 0.1, 1.0, tol=0.0, checkpoint=10 ** 9)
        t0 = time.perf_counter()
        on.minimize(X, 20, 2e-4, 0.02, 0.005, 0.1, 1.0, tol=0.0, checkpoint=10 ** 9)
        cpu = (time.perf_counter() - t0) / 20
        c3.update({"cpu_ms_per_iter": cpu * 1e3, "speedup_vs_cpu": cpu / t,
                   "cpu_sample": "20 iterations of oracle/nonlinear_ref.py (closed-form numpy backward; the reference's torch-autograd "
                                 "iteration is 14.8 ms, SURVEY.md 6.2)"})
    out["c3"] = c3
    return out


def bench_sharded(torch, dist, rank, world, dev):
    """SURVEY.md 8e2 on N GPUs (every rank calls this): the row-sharded C2 (logistic d=100) and C3 (MLP [40,10,1])
    inner iterations -- rows of X split contiguously, ONE sum of the d x d (parameter-sized) partial gradient over the
    GPUs per iteration: C2 inside the persistent iteration kernel over NVLink peer memory when every GPU's rows fit its
    workers (csrc/lin_iter.cu), else and for C3 a NCCL all-reduce captured inside the iteration's CUDA graph -- timed
    with CUDA events (max over ranks)
    next to the same iterations un-sharded on one GPU, with |dW| between the two after the timed iterations; the C2
    pair is repeated at larger n (rows tiled) to locate the n above which sharding pays."""
    import numpy as np
    from oracle import simulate
    from midagma_b200 import DagmaLinear, parallel
    from midagma_b200.nonlinear import DagmaMLP, DagmaNonlinear

    def rmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def time_linear(X, shard, iters):
        m = DagmaLinear("logistic")
        Xl = X
        if shard:
            m.shard_rows()
            Xl = X[parallel.row_shard(X.shape[0], rank, world)]
        m.fit(np.ascontiguousarray(Xl), lambda1=0.02, T=1, warm_iter=0, max_iter=0, checkpoint=10 ** 9)
        d = X.shape[1]
        W = np.zeros((d, d))
        m.minimize(W, 1.0, 100, 1.0, lr=3e-4, tol=0.0)            # graph capture + warm-up
        W[...] = 0.0
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        m.minimize(W, 1.0, iters, 1.0, lr=3e-4, tol=0.0)
        e1.record()
        torch.cuda.synchronize()
        eng = m._large
        path = ("persistent kernel, cross-GPU sum over NVLink peer memory" if eng._peer is not None else
                "persistent kernel" if eng.one_kernel else
                "launch sequence" + (" + NCCL all-reduce in the CUDA graph" if shard else ""))
        t = rmax(e0.elapsed_time(e1) * 1e-3) / iters
        m.close()                                                 # peer mappings (collective)
        return t, W, path

    out = {"n_gpus": world, "all_reduce": "C2: summed inside the persistent kernel over NVLink peer memory (plain stores + "
                                          "sequence flags, rank order) when the rows fit, else NCCL; C3: torch.distributed NCCL sum "
                                          "all-reduce captured inside the iteration's CUDA graph"}
    X, _ = simulate.config_c2(0)
    rows = []
    for mult in (1, 2, 4, 8, 16, 64):
        Xn = np.tile(X, (mult, 1)) if mult > 1 else X
        iters = 1000 if mult <= 8 else 200
        t_sh, W_sh, p_sh = time_linear(Xn, True, iters)
        t_1, W_1, p_1 = time_linear(Xn, False, iters)
        rows.append({"n": int(Xn.shape[0]), "us_per_iter_sharded": t_sh * 1e6, "us_per_iter_one_gpu": t_1 * 1e6,
                     "speedup": t_1 / t_sh, "max_abs_dW_vs_one_gpu": float(np.abs(W_sh - W_1).max()), "iters": iters,
                     "sharded_path": p_sh, "one_gpu_path": p_1})
        del Xn
    out["c2_sharded"] = {"workload": "C2: DagmaLinear logistic d=100, rows sharded over the GPUs (n = 10 000 is BASELINE's size; "
                                     "larger n: the same rows tiled)",
                         "iters_per_s": 1e6 / rows[0]["us_per_iter_sharded"], "by_n": rows,
                         "crossover_n": next((r["n"] for r in rows if r["speedup"] >= 1.0), None)}
    # ---- C3
    Xn, _ = simulate.config_c3(0)
    n, d, m1 = Xn.shape[0], Xn.shape[1], 10

    def time_mlp(shard, iters):
        torch.manual_seed(0)
        model = DagmaMLP(dims=[d, m1, 1], bias=True)
        eq = DagmaNonlinear(model)
        Xl = Xn
        if shard:
            eq.group, eq.n_total = dist.group.WORLD, n
            Xl = Xn[parallel.row_shard(n, rank, world)]
        eq.X = torch.from_numpy(np.ascontiguousarray(Xl)).cuda()
        eq.checkpoint = 10 ** 9
        state = {k: v.detach().clone() for k, v in model.state_dict().items()}
        eq.minimize(100, 2e-4, 0.02, 0.005, 0.1, 1.0, tol=0.0)
        model.load_state_dict(state)
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eq.minimize(iters, 2e-4, 0.02, 0.005, 0.1, 1.0, tol=0.0)
        e1.record()
        torch.cuda.synchronize()
        eng = eq._engine
        path = ("persistent kernel, cross-GPU sum over NVLink peer memory" if eng._peer is not None else
                "persistent kernel" if eng.one_kernel else
                "launch sequence" + (" + NCCL all-reduce in the CUDA graph" if shard else ""))
        t = rmax(e0.elapsed_time(e1) * 1e-3) / iters
        w = model.fc1.weight.detach().clone()
        eq.close()                                                # peer mappings (collective)
        return t, w, path

    rows3 = []
    X3 = Xn
    for mult in (1, 4, 16):
        Xn = np.tile(X3, (mult, 1)) if mult > 1 else X3
        n = Xn.shape[0]
        t_sh, w_sh, p_sh = time_mlp(True, 1000)
        t_1, w_1, p_1 = time_mlp(False, 1000)
        rows3.append({"n": int(n), "us_per_iter_sharded": t_sh * 1e6, "us_per_iter_one_gpu": t_1 * 1e6, "speedup": t_1 / t_sh,
                      "max_abs_dfc1_vs_one_gpu": float((w_sh - w_1).abs().max().item()), "sharded_path": p_sh,
                      "one_gpu_path": p_1})
    out["c3_sharded"] = {"workload": "C3: DagmaMLP [40, 10, 1], rows sharded over the GPUs (n = 2000 is BASELINE's size; larger "
                                     "n: the same rows tiled)",
                         "iters_per_s": 1e6 / rows3[0]["us_per_iter_sharded"],
                         "us_per_iter_sharded": rows3[0]["us_per_iter_sharded"],
                         "us_per_iter_one_gpu": rows3[0]["us_per_iter_one_gpu"], "speedup": rows3[0]["speedup"],
                         "max_abs_dfc1_vs_one_gpu": rows3[0]["max_abs_dfc1_vs_one_gpu"], "by_n": rows3,
                         "crossover_n": next((r["n"] for r in rows3 if r["speedup"] >= 1.0), None)}
    return out


def dump_outputs(out_dir, res, W, rank, world):
    """What the last timed step returned to its caller (W is updated in place), as float64 `out_dir/<name>.npy`:
    W of a fixed, seeded sample of the problems, and status and stage statistics of every problem."""
    import numpy as np
    pick = np.sort(np.random.default_rng(0).choice(W.shape[0], min(DUMP_PROBLEMS, W.shape[0]), replace=False))
    arrays = {"W_sample": W[pick.tolist()].cpu().numpy(), "W_sample_problems": pick.astype(np.float64),
              "status": res.status.cpu().numpy().astype(np.float64), "stage_stats": res.stage_stats.cpu().numpy()}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + (f"_rank{rank}" if world > 1 else "") + ".npy"), a)


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from midagma_b200 import _lib, fit_batch
    from midagma_b200.linear import _run_small, center_cov

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    sms = _lib.require_device()
    dev = torch.device("cuda", local)

    nprob = args.problems
    n_seeds = max(nprob // len(LAMBDAS), 1)
    seed0 = 1000 + rank * n_seeds                       # every rank owns different problems
    t_gen = time.perf_counter()
    X = make_covs(n_seeds, seed0)
    Xd = torch.from_numpy(X).to(dev)
    cov_seed = center_cov(Xd, center=True)
    del Xd, X
    cov = cov_seed.repeat_interleave(len(LAMBDAS), dim=0)[:nprob].contiguous()
    lam = torch.tensor([LAMBDAS[i % 4] for i in range(nprob)], dtype=torch.float64, device=dev)
    t_gen = time.perf_counter() - t_gen

    W = torch.zeros(nprob, D, D, dtype=torch.float64, device=dev)

    def step():
        return _run_small(cov, W, lam, [1.0], [1.0], [ITERS_PER_STEP], lr=3e-4, tol=0.0, beta1=0.99, beta2=0.999,
                          checkpoint=ITERS_PER_STEP, retry=False, want_final=False)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    sync()
    sampler = ClockSampler(local) if rank == 0 else None
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    done = 0
    ev[0].record()
    results = []
    for k in range(args.steps):
        results.append(step())
        ev[k + 1].record()
    sync()
    clocks = sampler.stop() if sampler else None
    dt = ev[0].elapsed_time(ev[-1]) * 1e-3
    kernel_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
    done = sum(int(r.stage_stats[:, 0, 0].sum().item()) for r in results)
    assert done == nprob * ITERS_PER_STEP * args.steps, "a problem stopped early inside the timed region"
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, results[-1], W, rank, world)

    # ---- e2e: public host API, pinned host buffers, copies inside the timed region
    from midagma_b200 import minimize_batch
    W_host = torch.zeros(nprob, D, D, dtype=torch.float64).pin_memory()
    cov_host = cov.cpu().pin_memory()
    lam_host = lam.cpu().numpy()
    minimize_batch(W_host, cov_host, lam_host, 1.0, ITERS_PER_STEP, 1.0, 3e-4, tol=0.0,
                   checkpoint=ITERS_PER_STEP, device=dev)
    sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t_e2e = time.perf_counter()
    for _ in range(args.steps):
        W_host, ok, st = minimize_batch(W_host, cov_host, lam_host, 1.0, ITERS_PER_STEP, 1.0, 3e-4,
                                        tol=0.0, checkpoint=ITERS_PER_STEP, device=dev)
    e1.record()
    sync()
    dt_e2e = max(e0.elapsed_time(e1) * 1e-3, 0.0)
    dt_e2e_wall = time.perf_counter() - t_e2e

    # ---- max over ranks
    def rmax(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    dt, dt_e2e = rmax(dt), rmax(max(dt_e2e, dt_e2e_wall))
    total_iters = float(nprob) * ITERS_PER_STEP * args.steps * world
    value = total_iters / dt
    e2e_value = total_iters / dt_e2e

    # ---- the contract line is complete from here on; everything below adds keys to it.  A watchdog guarantees that
    # rank 0 prints it exactly once even if an extra section hangs (e.g. a collective after a failure on one rank) or
    # raises: the extras then carry an `extras_error` / `extras_timeout` note instead of values.
    import threading
    core = {
        "metric": "DagmaLinear inner Adam iters/sec (batched d=64)", "value": value,
        "unit": "problem-iterations/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "C4: batched DagmaLinear l2 minimize, ER4 d=64 n=1000, 1024 seeds x 4 lambda1",
                   "problems_per_gpu": nprob, "d": D, "n": N_SAMPLES, "iters_per_step": ITERS_PER_STEP,
                   "mu": 1.0, "s": 1.0, "lr": 3e-4, "l2_policy": "inputs exceed L2 (cov+W = 268 MB per GPU)",
                   "data_gen_s": round(t_gen, 1)},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "problem-iterations/s",
                "h2d_bytes_per_step": 2 * nprob * D * D * 8 + nprob * 8, "d2h_bytes_per_step": nprob * D * D * 8},
        "gpu_launches": args.steps,
    }
    extra = {}
    emit_lock, emitted = threading.Lock(), []

    def emit(note=None):
        with emit_lock:
            if emitted:
                return
            emitted.append(1)
            if rank == 0:
                line = dict(core)
                line.update(extra)
                if note:
                    line.update(note)
                print(json.dumps(line), flush=True)

    def on_timeout():
        emit({"extras_timeout": f"an extra section did not finish within {args.extras_timeout} s: keys after the last "
                                "completed section are missing"})
        os._exit(0)

    watchdog = threading.Timer(args.extras_timeout, on_timeout)
    watchdog.daemon = True
    watchdog.start()
    try:
        run_extras(args, torch, dist, _lib, fit_batch, _run_small, extra, locals())
    except BaseException as e:                            # noqa: BLE001 -- reported in the line, never lost
        extra["extras_error"] = f"{type(e).__name__}: {e}"[:500]
        if world > 1:
            watchdog.cancel()
            emit()
            os._exit(0)                                  # the other ranks may sit in a collective: their watchdogs end them
    watchdog.cancel()
    emit()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_extras(args, torch, dist, _lib, fit_batch, _run_small, extra, env):
    """Everything of the bench line beyond the contract keys (see the module docstring); `env` = the locals of run_b200."""
    import numpy as np                                    # noqa: F401
    world, rank, dev, sms, nprob = env["world"], env["rank"], env["dev"], env["sms"], env["nprob"]
    cov, lam, sync, rmax, kernel_ms = env["cov"], env["lam"], env["sync"], env["rmax"], env["kernel_ms"]
    W_host, cov_host = env["W_host"], env["cov_host"]
    if world > 1:
        # ---- strong scaling of the same workload: 4096 problems in total, 4096 / N per GPU (2 CTAs per SM: 512
        # equal-length problems are 1.73 waves of 296 resident CTAs -- the second wave bounds the step)
        n_loc = max(nprob // world, 1)
        Ws = torch.zeros(n_loc, D, D, dtype=torch.float64, device=dev)

        def sstep():
            return _run_small(cov[:n_loc], Ws, lam[:n_loc], [1.0], [1.0], [ITERS_PER_STEP], lr=3e-4, tol=0.0, beta1=0.99,
                              beta2=0.999, checkpoint=ITERS_PER_STEP, retry=False, want_final=False)
        sstep()
        sync()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(args.steps):
            sstep()
        s1.record()
        sync()
        dt_s = rmax(s0.elapsed_time(s1) * 1e-3)
        strong = {"problems_total": n_loc * world, "problems_per_gpu": n_loc,
                  "value": float(n_loc) * world * ITERS_PER_STEP * args.steps / dt_s, "unit": "problem-iterations/s",
                  "ms_per_step": 1e3 * dt_s / args.steps, "resident_ctas_per_gpu": 2 * sms,
                  "waves": n_loc / (2.0 * sms)}
        del Ws
        sharded = bench_sharded(torch, dist, rank, world, dev) if args.sharded else None
        if rank == 0:
            extra["strong_scaling"] = strong
            if sharded:
                extra.update({k: v for k, v in sharded.items() if k in ("c2_sharded", "c3_sharded")})
    if rank == 0:
        peaks = fp64_peak_tflops(torch, _lib, sms)
        peak = max(peaks.values())
        per_gpu_rate = nprob * ITERS_PER_STEP / (sum(kernel_ms) / len(kernel_ms) * 1e-3)
        achieved = per_gpu_rate * FLOP_PER_ITER / 1e12
        traffic, tsrc = traffic_from_profile("fit_small_dmma_kernel")
        if not (nprob == 4096 and ITERS_PER_STEP == 1000):
            traffic = None                       # the capture is of this configuration only
        extra["roofline"] = {
            "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
            # dram__bytes_read.sum + dram__bytes_write.sum of one launch of this configuration (4096 problems x 1000
            # iterations), parsed from the committed ncu --set full summary named in profiles/roofline_sources.json
            "traffic": traffic, "traffic_source": tsrc,
            "traffic_unit": "bytes per launch (algorithmic I/O: cov + W in, W out = 402.7e6)",
            "kernel": "fit_small_dmma_kernel (one launch per step)",
            "peak_source": "measured live: FP64 pipe yardsticks and cuBLAS DGEMM 8192^3 "
                           + json.dumps({k: round(v, 2) for k, v in peaks.items()})
                           + " TFLOP/s; denominator = the largest (MEASURED_PEAKS.json has no FP64 entry; FP64 tensor = "
                             "FP64 FMA rate on B200)",
            "fp64_peaks_tflops": {k: round(v, 3) for k, v in peaks.items()},
            "flop_per_unit": FLOP_PER_ITER, "units_per_launch": nprob * ITERS_PER_STEP,
        }
        if args.cpu_baseline:
            kind = cpu_kind()
            rate, cores, cdone, cwall = cpu_rate(args.cpu_iters, kind=kind)
            extra["cpu_baseline"] = {
                "value": rate, "unit": "problem-iterations/s", "cores": cores, "kind": kind,
                "sample": f"{cores} problems (one per core) x {args.cpu_iters} iterations, {cwall:.1f} s wall, "
                          f"{cpu_what(kind)}, 1 BLAS thread per process"}
        if args.full_fit and world == 1:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            W_est, info = fit_batch(cov=cov, lambda1=lam, return_info=True, device=dev)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            extra["full_fit"] = {"problems": nprob, "wall_s": wall, "total_inner_iters": info["total_iters"],
                                 "iters_per_s": info["total_iters"] / wall,
                                 "status_nonzero": int((info["status"] != 0).sum()),
                                 "mean_edges": float((W_est != 0).sum(axis=(1, 2)).mean())}
            ps = parity_sample(info["W_raw"], info["stage_iters"])
            if ps is not None:
                extra["parity_sample"] = ps
            del W_est, info

        if args.c5 and world == 1:
            del W_host, cov_host
            env.pop("W_host", None)
            env.pop("cov_host", None)
            extra["c5"] = bench_c5(torch, _lib, peak, args.cpu_baseline)
            extra.update(bench_c2_c3(torch, args.cpu_baseline, peak))



def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--problems", type=int, default=4096, help="problems per GPU")
    ap.add_argument("--cpu-iters", type=int, default=100000, help="oracle iterations per core (~15 s)")
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--no-full-fit", dest="full_fit", action="store_false")
    ap.add_argument("--no-c5", dest="c5", action="store_false", help="skip the single d=2000 problem (C5)")
    ap.add_argument("--no-sharded", dest="sharded", action="store_false",
                    help="N > 1: skip the row-sharded C2 / C3 iterations")
    ap.add_argument("--extras-timeout", type=float, default=1500.0,
                    help="seconds after which the contract line is printed without the unfinished extra keys")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float64, about 17 MB)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
