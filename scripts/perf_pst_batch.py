"""Batched PST ``inv`` / ``exp`` or spectral TCC fits (csrc/small_fit_pst.cu) against the plain l2 batch and the
per-problem loop a user has without them.

Shapes (Gaussian ER2 SEM, seeds from 2000, lambda1 = 0.02): 1024 x (d = 20, n = 500) and 1024 x (d = 64, n = 1000);
each problem's pair set I is the no-trek pairs of its true graph, PST ``--seq`` / mean, weight 0.1.  For each shape:
  * minimize_batch(trek_reg=[...]) with tol = 0 (every problem runs every iteration) on device-resident inputs, warmed
    up, timed by CUDA events: problem-iterations/s, achieved FP64 TFLOP/s from the flop model below and its share of the
    FP64 peak measured in the same run (bench.py's yardsticks);
  * the same call without trek_reg (the plain l2 kernel): what the trek term costs;
  * DagmaLinear("l2", trek_reg=...).minimize on 4 of the problems (wall clock ending in a synchronise) and max|dW|.
Flop model per iteration: 4 d^3 for the l2 iteration (inverse + cov W); for the trek term 8 d^3 with inv (second
inverse, three products) and 234 d^3 with exp (117 products: 29 for expm, one for F G_S, 87 for the coupled Frechet
chain); the pair values (2 d per pair, at checkpoints only for inv / mean) are left out.
--seq tcc: TCCRegularizer(I, weight 0.1) with the reference's dispatch (spectral, approx_trek_graph, eig: the Perron
pair iterated until it stops moving).  Its cost is the number of power steps, a chain of latency-bound steps, so no flop
model or FP64 share is reported; instead the mean power steps per Perron solve, from the kernel's perron_steps counter of
an untimed repeat of the batched call (the kernel is deterministic) over its solves (iterations + the final checkpoint
+ back-tracking steps per problem).
Usage: perf_pst_batch.py --out DIR [--seq inv|exp|tcc]   (writes DIR/perf_pst_batch.json for inv,
DIR/perf_pst_exp_batch.json for exp, DIR/perf_tcc_batch.json for tcc, nothing else)"""
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

SHAPES = {"d20": (1024, 20, 500), "d64": (1024, 64, 1000)}
ITERS, LOOP_PROBLEMS, MU, S, LR, LAM, WEIGHT, CKPT = 1000, 4, 1.0, 1.0, 3e-4, 0.02, 0.1, 100


def no_trek_pairs(B):
    """(i, j), i < j, with no trek in the DAG B: no node reaches both (a node reaches itself)."""
    d = B.shape[0]
    R = np.eye(d, dtype=bool) | (B != 0)
    for _ in range(d):
        R = R | ((R.astype(np.int64) @ R.astype(np.int64)) > 0)
    trek = (R.T.astype(np.int64) @ R.astype(np.int64)) > 0
    return np.array([(i, j) for i in range(d) for j in range(i + 1, d) if not trek[i, j]], dtype=np.int64).reshape(-1, 2)


def make_data(batch, d, n):
    from oracle import simulate
    Xs, pairs = [], []
    for p in range(batch):
        X, W_true = simulate.make_linear_problem(d, 2, n, "ER", "gauss", 2000 + p)
        Xs.append(X - X.mean(axis=0, keepdims=True))
        pairs.append(no_trek_pairs(W_true))
    return np.stack(Xs), pairs


TREK_FLOP = {"inv": 8.0, "exp": 234.0}       # per d^3 and iteration, see the docstring


def flop_per_iter(d, trek, seq="inv"):
    return (4.0 + (TREK_FLOP[seq] if trek else 0.0)) * d ** 3


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def batched(torch, cov, d, regs):
    from midagma_b200 import minimize_batch
    batch = cov.shape[0]
    W = torch.zeros(batch, d, d, dtype=torch.float64, device="cuda")
    minimize_batch(W[:64].clone(), cov[:64], LAM, MU, 50, S, LR, tol=0.0, checkpoint=CKPT,
                   trek_reg=regs[:64] if regs else None)                                  # warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    W, ok, st = minimize_batch(W, cov, LAM, MU, ITERS, S, LR, tol=0.0, checkpoint=CKPT, trek_reg=regs)
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) * 1e-3
    return W.cpu().numpy(), ok.cpu().numpy(), t, float(st[:, 0, 0].sum().item())


def perron_steps(torch, cov, d, regs):
    """Mean power steps per Perron solve of the batched call (an untimed repeat through its launcher)."""
    from midagma_b200.linear import _run_small, _tcc_dev, _trek_batch
    batch = cov.shape[0]
    W = torch.zeros(batch, d, d, dtype=torch.float64, device="cuda")
    tcc = _tcc_dev(_trek_batch(regs, batch, d, "l2", "perf")[1], "cuda")
    lam = torch.full((batch,), LAM, dtype=torch.float64, device="cuda")
    res = _run_small(cov, W, lam, [MU], [S], [ITERS], lr=LR, tol=0.0, beta1=0.99, beta2=0.999, checkpoint=CKPT,
                     retry=False, want_final=False, tcc=tcc)
    st = res.stage_stats.cpu().numpy()
    steps = tcc.perron_steps.cpu().numpy()
    solves = st[:, 0, 0] + 1 + st[:, 0, 7]
    return float(steps.sum() / solves.sum()), int(steps.max()), int(((res.status.cpu().numpy() & 8) != 0).sum())


def loop(torch, cov, d, regs):
    from midagma_b200 import DagmaLinear
    Ws, t_total, iters = [], 0.0, 0
    for b in range(LOOP_PROBLEMS):
        m = DagmaLinear("l2", trek_reg=regs[b])
        m._fit_from_cov(cov[b], LAM, T=1, warm_iter=0, max_iter=0, checkpoint=CKPT)
        if b == 0:
            m.minimize(np.zeros((d, d)), MU, 50, S, lr=LR, tol=0.0)                 # warm-up of this shape
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        W, _ = m.minimize(np.zeros((d, d)), MU, ITERS, S, lr=LR, tol=0.0)
        torch.cuda.synchronize()
        t_total += time.perf_counter() - t0
        iters += m.last_iters
        Ws.append(W)
    return np.stack(Ws), t_total, iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--seq", choices=("inv", "exp", "tcc"), default="inv")
    args = ap.parse_args()
    seq = args.seq
    tcc = seq == "tcc"
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, {"inv": "perf_pst_batch.json", "exp": "perf_pst_exp_batch.json",
                                   "tcc": "perf_tcc_batch.json"}[seq])
    import torch
    from midagma_b200 import _lib
    from midagma_b200.linear import center_cov
    from midagma_b200.notreks import PSTRegularizer, TCCRegularizer
    import bench
    _lib.require_device()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    res = {"device": device_info(), "iterations": ITERS, "tol": 0.0, "mu": MU, "s": S, "lr": LR, "lambda1": LAM}
    if tcc:
        res["tcc"] = {"weight": WEIGHT, "I": "no-trek pairs of the true graph",
                      "dispatch": "reference default: spectral, approx_trek_graph, eig (converged Perron pair)"}
    else:
        res.update({"pst": {"seq": seq, "agg": "mean", "weight": WEIGHT, "I": "no-trek pairs of the true graph"},
                    "flop_model": f"{TREK_FLOP[seq] + 4:g} d^3 per iteration with the trek term, 4 d^3 without",
                    "fp64_peaks_tflops": {k: round(v, 3) for k, v in bench.fp64_peak_tflops(torch, _lib, sms).items()}})
        peak = max(res["fp64_peaks_tflops"].values())
        res["fp64_peak_tflops"] = peak

    def dump():
        with open(path, "w") as f:
            json.dump(res, f, indent=1)

    dump()
    for name, (batch, d, n) in SHAPES.items():
        Xs, pairs = make_data(batch, d, n)
        if tcc:
            regs = [TCCRegularizer(I=p, weight=WEIGHT, mode="opt") for p in pairs]
        else:
            regs = [PSTRegularizer(I=p, seq=seq, weight=WEIGHT, mode="opt", kwargs={"agg": "mean"}) for p in pairs]
        cov = center_cov(torch.as_tensor(Xs).cuda(), center=False)
        Wb, okb, t, iters = batched(torch, cov, d, regs)
        _, okp, tp, itp = batched(torch, cov, d, None)
        Wl, tl, itl = loop(torch, cov, d, regs)
        rate, plain, lrate = iters / t, itp / tp, itl / tl
        key = "tcc" if tcc else "pst"
        r = {"batch": batch, "d": d, "n": n, "mean_pairs": float(np.mean([len(p) for p in pairs])),
             f"{key}_seconds": t, f"{key}_problem_iters": iters, f"{key}_problem_iters_per_s": rate}
        if tcc:
            mean_steps, max_steps, capped = perron_steps(torch, cov, d, regs)
            r.update({"mean_power_steps_per_solve": mean_steps, "max_power_steps_per_problem": max_steps,
                      "problems_with_capped_solve": capped})
        else:
            tflops = rate * flop_per_iter(d, True, seq) / 1e12
            r.update({"pst_achieved_fp64_tflops": tflops, "pst_share_of_fp64_peak": tflops / peak})
        r.update({f"{key}_failed_problems": int((~okb).sum()),
                  "plain_seconds": tp, "plain_problem_iters_per_s": plain,
                  "plain_achieved_fp64_tflops": plain * flop_per_iter(d, False) / 1e12,
                  "trek_cost_factor": plain / rate,
                  "loop_problems": LOOP_PROBLEMS, "loop_seconds": tl, "loop_problem_iters_per_s": lrate,
                  "speedup_vs_loop": rate / lrate,
                  "parity_max_abs_dW_loop_vs_batched": float(np.abs(Wl - Wb[:LOOP_PROBLEMS]).max())})
        res[f"shape_{name}"] = r
        print(name, json.dumps(r), flush=True)
        dump()


if __name__ == "__main__":
    main()
