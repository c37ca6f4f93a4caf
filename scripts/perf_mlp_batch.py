"""Batched nonlinear minimize (csrc/mlp_batch.cu) against the per-problem loop a user has without it.

Shapes ([d, m1, 1] MLPs from the reference start -- fc1 = 0, fc2 as DagmaMLP initialises it -- on Gaussian data, which
the timing does not depend on):
  C3: 296 x (d = 40, m1 = 10, n = 2000)   -- two problems per SM, the benchmark's C3 configuration
  B : 1024 x (d = 20, m1 = 10, n = 1000)
  C : 2048 x (d = 10, m1 = 10, n = 500)
For each: one minimize pass of ITERS iterations on device-resident inputs (warmed up, CUDA events around the launch),
problem-iterations/s, achieved FP64 FLOP/s from 4 n d^2 m1 + 2 d^3 per iteration and its share of the FP64 peak
measured in the same run (bench.py's yardsticks); the loop DagmaNonlinear.minimize on LOOP_PROBLEMS of the problems
(wall clock ending in a synchronise) and the largest relative parameter difference between the two.
Usage: perf_mlp_batch.py --out DIR   (writes DIR/perf_mlp_batch.json, nothing else)"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

SHAPES = {"C3": (296, 40, 10, 2000), "B": (1024, 20, 10, 1000), "C": (2048, 10, 10, 500)}
ITERS, LOOP_PROBLEMS = 100, 4
LR, LAM1, LAM2, MU, S = 2e-4, 0.02, 0.005, 0.1, 1.0


def flop_per_iter(d, m1, n):
    return 4.0 * n * d * d * m1 + 2.0 * d ** 3


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def make_models(torch, batch, d, m1):
    from midagma_b200.nonlinear import DagmaMLP
    torch.manual_seed(0)
    return [DagmaMLP([d, m1, 1]) for _ in range(batch)]


def batched(torch, models, Xd):
    from midagma_b200.nonlinear import _MlpBatch
    B = len(models)
    bt = _MlpBatch(models, Xd)
    full = lambda x: np.full(B, x)                              # noqa: E731
    args = (full(LR), full(LAM1), full(LAM2), full(MU), full(S), full(False), 1e-6, 1000)
    snap = bt.theta.clone()
    bt.run(np.arange(B), 5, *args)                              # warm-up
    bt.theta.copy_(snap)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ok, its = bt.run(np.arange(B), ITERS, *args)
    e1.record()
    torch.cuda.synchronize()
    return bt.theta.cpu().numpy(), ok, e0.elapsed_time(e1) * 1e-3, int(its.sum())


def loop(torch, models, Xd):
    import copy
    from midagma_b200.nonlinear import DagmaNonlinear
    thetas, t_total, iters = [], 0.0, 0
    for b in range(LOOP_PROBLEMS):
        if b == 0:                                              # warm-up of this shape
            eq = DagmaNonlinear(copy.deepcopy(models[0]))
            eq.X, eq.checkpoint = Xd[0], 1000
            eq.minimize(5, LR, LAM1, LAM2, MU, S)
        eq = DagmaNonlinear(models[b])
        eq.X, eq.checkpoint = Xd[b], 1000
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        eq.minimize(ITERS, LR, LAM1, LAM2, MU, S)
        torch.cuda.synchronize()
        t_total += time.perf_counter() - t0
        iters += eq.n_iters
        thetas.append(models[b].pack().cpu().numpy())
    return np.stack(thetas), t_total, iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "perf_mlp_batch.json")
    import torch
    from midagma_b200 import _lib
    import bench
    _lib.require_device()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    res = {"device": device_info(), "iterations": ITERS, "lr": LR, "lambda1": LAM1, "lambda2": LAM2, "mu": MU, "s": S,
           "fp64_peaks_tflops": {k: round(v, 3) for k, v in bench.fp64_peak_tflops(torch, _lib, sms).items()}}
    peak = max(res["fp64_peaks_tflops"].values())
    res["fp64_peak_tflops"] = peak

    def dump():
        with open(path, "w") as f:
            json.dump(res, f, indent=1)

    dump()
    for name, (batch, d, m1, n) in SHAPES.items():
        g = torch.Generator(device="cuda").manual_seed(7)
        Xd = torch.randn(batch, n, d, dtype=torch.float64, device="cuda", generator=g)
        models = make_models(torch, batch, d, m1)
        thb, okb, t, iters = batched(torch, models, Xd)
        rate = iters / t
        tflops = rate * flop_per_iter(d, m1, n) / 1e12
        thl, tl, itl = loop(torch, models, Xd)
        lrate = itl / tl
        r = {"batch": batch, "d": d, "m1": m1, "n": n, "batched_seconds": t, "batched_problem_iters": iters,
             "batched_problem_iters_per_s": rate, "flop_per_iter": flop_per_iter(d, m1, n),
             "achieved_fp64_tflops": tflops, "share_of_fp64_peak": tflops / peak, "failed_problems": int((~okb).sum()),
             "loop_problems": LOOP_PROBLEMS, "loop_seconds": tl, "loop_problem_iters_per_s": lrate,
             "loop_achieved_fp64_tflops": lrate * flop_per_iter(d, m1, n) / 1e12,
             "speedup_vs_loop": rate / lrate,
             "parity_max_rel_dtheta_loop_vs_batched": float(np.abs(thl - thb[:LOOP_PROBLEMS]).max()
                                                            / np.abs(thl).max())}
        res[f"shape_{name}"] = r
        print(name, json.dumps(r), flush=True)
        dump()
        del Xd


if __name__ == "__main__":
    main()
