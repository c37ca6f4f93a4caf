"""Batched logistic fits (csrc/small_fit_logistic.cu) against the per-problem loop a user has without them.

Shapes (logistic ER2 SEM, binary data, seeds from 1000, lambda1 cycling 0.01, 0.02, 0.03, 0.05):
  A: 1024 x (d = 64, n = 1000)  -- X is 524 MB, more than the 126 MB of L2
  B: 4096 x (d = 20, n = 500)   -- X is 328 MB
For each: one minimize_batch(loss_type="logistic") pass of 1000 iterations on device-resident inputs (warmed up, CUDA
events), problem-iterations/s, achieved FP64 FLOP/s from 4 n d^2 + 2 d^3 per iteration and its share of the FP64 peak
measured in the same run (bench.py's yardsticks); the loop DagmaLinear("logistic").minimize on 8 of the problems
(wall clock ending in a synchronise) and max|dW| between the two; then a full default fit_batch on shape B.
Usage: perf_logistic_batch.py --out DIR   (writes DIR/perf_logistic_batch.json, nothing else)"""
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

LAMBDAS = (0.01, 0.02, 0.03, 0.05)
SHAPES = {"A": (1024, 64, 1000), "B": (4096, 20, 500)}
ITERS, LOOP_PROBLEMS, MU, S, LR = 1000, 8, 1.0, 1.0, 3e-4


def make_data(batch, d, n):
    from oracle import simulate
    return np.stack([simulate.make_linear_problem(d, 2, n, "ER", "logistic", 1000 + p)[0] for p in range(batch)])


def flop_per_iter(d, n):
    return 4.0 * n * d * d + 2.0 * d ** 3


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def batched_rate(torch, Xd, lam, d):
    from midagma_b200 import minimize_batch
    batch = Xd.shape[0]
    from midagma_b200.linear import center_cov
    cov = center_cov(Xd, center=False)
    W = torch.zeros(batch, d, d, dtype=torch.float64, device="cuda")
    minimize_batch(W[:64].clone(), cov[:64], lam[:64], MU, 50, S, LR, loss_type="logistic", X=Xd[:64])   # warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    W, ok, st = minimize_batch(W, cov, lam, MU, ITERS, S, LR, loss_type="logistic", X=Xd)
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) * 1e-3
    iters = float(st[:, 0, 0].sum().item())
    return W.cpu().numpy(), ok.cpu().numpy(), t, iters


def loop_rate(torch, Xs, lam):
    from midagma_b200 import DagmaLinear
    d = Xs.shape[2]
    Ws, t_total, iters = [], 0.0, 0
    for b in range(LOOP_PROBLEMS):
        m = DagmaLinear("logistic")
        m.fit(Xs[b].copy(), lambda1=float(lam[b]), T=1, warm_iter=0, max_iter=0, checkpoint=1000)
        if b == 0:
            m.minimize(np.zeros((d, d)), MU, 50, S, lr=LR)                     # warm-up of this shape
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        W, _ = m.minimize(np.zeros((d, d)), MU, ITERS, S, lr=LR)
        torch.cuda.synchronize()
        t_total += time.perf_counter() - t0
        iters += m.last_iters
        Ws.append(W)
    return np.stack(Ws), t_total, iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--skip-full-fit", action="store_true")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "perf_logistic_batch.json")
    import torch
    from midagma_b200 import _lib
    import bench
    _lib.require_device()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    res = {"device": device_info(), "iterations": ITERS, "mu": MU, "s": S, "lr": LR,
           "fp64_peaks_tflops": {k: round(v, 3) for k, v in bench.fp64_peak_tflops(torch, _lib, sms).items()}}
    peak = max(res["fp64_peaks_tflops"].values())
    res["fp64_peak_tflops"] = peak

    def dump():
        with open(path, "w") as f:
            json.dump(res, f, indent=1)

    dump()
    for name, (batch, d, n) in SHAPES.items():
        t0 = time.perf_counter()
        Xs = make_data(batch, d, n)
        lam = np.array([LAMBDAS[p % len(LAMBDAS)] for p in range(batch)])
        gen = time.perf_counter() - t0
        Xd = torch.as_tensor(Xs).cuda()
        lamd = torch.as_tensor(lam).cuda()
        Wb, okb, t, iters = batched_rate(torch, Xd, lamd, d)
        rate = iters / t
        tflops = rate * flop_per_iter(d, n) / 1e12
        Wl, tl, itl = loop_rate(torch, Xs, lam)
        loop = itl / tl
        r = {"batch": batch, "d": d, "n": n, "X_MB": Xs.nbytes / 1e6, "data_gen_s": round(gen, 1),
             "batched_seconds": t, "batched_problem_iters": iters, "batched_problem_iters_per_s": rate,
             "flop_per_iter": flop_per_iter(d, n), "achieved_fp64_tflops": tflops, "share_of_fp64_peak": tflops / peak,
             "failed_problems": int((~okb).sum()),
             "loop_problems": LOOP_PROBLEMS, "loop_seconds": tl, "loop_problem_iters_per_s": loop,
             "speedup_vs_loop": rate / loop,
             "parity_max_abs_dW_loop_vs_batched": float(np.abs(Wl - Wb[:LOOP_PROBLEMS]).max())}
        res[f"shape_{name}"] = r
        print(name, json.dumps(r), flush=True)
        dump()
        del Xd
        if name == "B" and not args.skip_full_fit:
            from midagma_b200 import fit_batch
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, info = fit_batch(Xs, lam, loss_type="logistic", return_info=True)
            torch.cuda.synchronize()
            tf = time.perf_counter() - t0
            si = info["stage_iters"]
            res["full_fit_B"] = {"seconds": tf, "total_iters": int(si.sum()),
                                 "problem_iters_per_s": float(si.sum()) / tf,
                                 "retry_limit_problems": int(((info["status"] & _lib.ST_RETRY_LIMIT) != 0).sum()),
                                 "stage_iters_percentiles": {
                                     f"stage_{k}": np.percentile(si[:, k], [0, 10, 50, 90, 100]).tolist()
                                     for k in range(si.shape[1])},
                                 "retries_total": int(info["stage_stats"][:, :, 6].sum())}
            print("full fit B", json.dumps(res["full_fit_B"]), flush=True)
            dump()


if __name__ == "__main__":
    main()
