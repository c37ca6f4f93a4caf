"""DagmaLinear's multi-CTA path at every shape it accepts, against the float64 oracle (``oracle.linear_ref``), numpy
and LAPACK.

* The persistent iteration kernel (csrc/lin_iter.cu, d <= 128) splits a problem over workers (``li_plan``): logistic
  workers keep up to 72 rows of X each, l2 workers own 8 rows of T = cov W, and the staged operands are padded to
  ``kd`` and ``ldx``.  A Python restatement of that plan is checked against the library, and the shape lists below are
  checked to reach every edge of it: one to three workers (fewer than the four lanes of the fixed-order reduction of
  ``part``), every worker full, a last worker with one row, d on every residue mod 4 and mod 16, a partial last l2
  worker and a second pivot block of 1 ... 64 columns.
* The launch sequence (csrc/large.cu, _large.py) serves l2 beyond d = 128 and logistic problems beyond the kernel's
  rows: the blocked inverse on both sides of its single-level / two-level switch, the update and objective kernels
  at d not a multiple of 32 and with more rows than CTAs, the logistic loss, split-K X^T R, every GEMM route inside a
  real iteration, back-tracking inside a checkpoint interval longer than the probe interval of the graph path, and
  the flow kernel (DAGMA_LOOKAHEAD=2) with its rider cov @ W.
* The blocked inverse through its C ABI: every scale branch (s outside (0.5, 1] is scaled by a power of two), padded
  leading dimensions whose padding must stay untouched, each output alone, and a batch.
* ``dagma_gemm_f64`` on each of its routes (balanced and queued TMA kernels, cp.async with and without split-K), with
  the route restated in Python and checked against the kernels a call launches.

Starts are generic (a seeded W0 with a zero diagonal, DESIGN.md 2), so no Adam sign tie decides a comparison.  Every
oracle trajectory runs once per module (``_oracle_run``)."""
import collections
import functools
import json
import math
import os
import subprocess
import sys
import tempfile
import zlib

import numpy as np
import pytest
import torch

from oracle.linear_ref import OracleLinear

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F64 = dict(dtype=torch.float64, device="cuda")
W_RTOL = 1e-9            # max |W - W_ref| / max |W_ref|
CKPT_RTOL = 1e-9         # objective, score and h of every checkpoint


def _cdiv(a, b):
    return -(-a // b)


def _relmax(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _close(a, b, rtol, floor=1e-6):
    return abs(a - b) <= rtol * max(abs(b), floor)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# n of a shape as a function of the SM count S of the device (the worker plan depends on it)
N_SPECS = {
    "8(S-1)-1": lambda S: 8 * (S - 1) - 1,
    "8(S-1)": lambda S: 8 * (S - 1),
    "8(S-1)+1": lambda S: 8 * (S - 1) + 1,
    "72(S-2)+1": lambda S: 72 * (S - 2) + 1,
    "72(S-1)-1": lambda S: 72 * (S - 1) - 1,
    "72(S-1)": lambda S: 72 * (S - 1),
    "72(S-1)+1": lambda S: 72 * (S - 1) + 1,
}


def _n(spec, sms):
    return N_SPECS[spec](sms) if isinstance(spec, str) else int(spec)


# =====================================================================================================================
# the plans, restated
# =====================================================================================================================
DMMA_SMEM_TOTAL = 2 * 64 * 68 + 2 * 8 * 68 + 2 * 64 * 8 + 2 * 64 + 64 + 96 + 2     # DmmaSmem::total (small_dmma.cuh)
INV2_SMEM_TOTAL = ((DMMA_SMEM_TOTAL + 1) & ~1) + 3 * 64 * 68 + 2 * 64                # Inv2Smem::total (small_inv2.cuh)
LI_RB = 72                                                                          # rows of X a worker keeps


def li_plan(logistic, n, d, sms):
    """``li_plan`` of csrc/lin_iter.cu with DAGMA_LIN_STREAM unset; None where the persistent kernel does not run."""
    if not (1 <= d <= 128) or sms < 3:
        return None
    ldx, kd = 16 * _cdiv(d, 16) + 4, 4 * _cdiv(d, 4)
    if logistic:
        if n < 1:
            return None
        NR = 8 * _cdiv(_cdiv(n, sms - 1), 8)
        if NR > LI_RB:                       # rows that do not fit are streamed only on request
            return None
        NW = _cdiv(n, NR)
        total = max(kd, NR) * ldx + NR * ldx + 2
        last = n - (NW - 1) * NR             # rows of the last worker
    else:
        NR, NW = 0, _cdiv(d, 8)
        if NW > sms - 1:
            return None
        total = kd * ldx + 2
        last = d - 8 * (NW - 1)              # rows of T of the last worker
    smem = max(total, DMMA_SMEM_TOTAL if d <= 64 else INV2_SMEM_TOTAL)
    if smem * 8 > 227 * 1024:
        return None
    return dict(logistic=logistic, n=n, d=d, S=sms, G=NW + 1, NW=NW, NR=NR, kd=kd, ldx=ldx, last=last,
                ws=(NW * d * d if logistic else 0) + 8)


def gemm_route(trans_a, M, N, K, lda, ldb, a_aligned, b_aligned, beta, epi, ws_bytes, sms):
    """``gemm_launch`` of csrc/large.cu at the defaults (DAGMA_TMA = 5, no forced mode, 64 x 64 cp.async tile):
    ("balanced" | "queue", None) for the 128 x 128 TMA kernel, ("cp.async", splits) for the cp.async kernel."""
    if M <= 0 or N <= 0:
        return ("none", None)
    tma_ok = (not trans_a and K > 0 and lda % 2 == 0 and ldb % 2 == 0 and a_aligned and b_aligned
              and _cdiv(M, 64) * _cdiv(N, 64) >= 296)
    if tma_ok:                                                   # gemm_tma_sched
        t128 = _cdiv(M, 128) * _cdiv(N, 128)
        plain = beta == 0.0 and epi == 0
        sched = None
        if plain and t128 >= 148 and K >= 512:
            sched = "balanced"
        elif t128 >= 4 * 148 and K >= 1024:
            sched = "queue"
        if sched == "balanced":                                  # gemm_tma_launch_cfg: every range a tile long
            grid, nk = min(t128, sms), _cdiv(K, 16)
            if not (t128 * nk // grid >= nk):
                sched = "queue"
        if sched is not None:
            return (sched, None)
    tm, tn, ktiles = _cdiv(M, 64), _cdiv(N, 64), _cdiv(K, 16)    # gemm_launch_tile<64, 64, 2, 2>
    splits, slots = 1, 148 * 4 * 64 * 64 // (128 * 64)
    if tm * tn < slots // 2 and ktiles >= 8 and ws_bytes is not None:
        splits = min(slots // (tm * tn), ktiles // 4)
        while splits > 1 and splits * M * N * 8 > ws_bytes:
            splits -= 1
        splits = max(splits, 1)
    if ktiles == 0:
        return ("cp.async", 1)
    kchunk = _cdiv(ktiles, splits)
    return ("cp.async", _cdiv(ktiles, kchunk))


# ---------------------------------------------------------------------------------------------------- shape lists
# persistent kernel, logistic: (d, n, what the pair covers)
FUSED_LOGISTIC = [
    (1, 1, "d = 1, n = 1: one worker holding one row"),
    (2, 7, "one worker, a partial 8-row tile"),
    (3, 9, "two workers, the last with one row"),
    (4, 17, "three workers, the last with one row"),
    (5, 25, "four workers, the last with one row"),
    (15, "8(S-1)", "NR = 8, S - 1 full workers"),
    (16, "8(S-1)+1", "NR = 16, d = 0 mod 16"),
    (17, "72(S-2)+1", "NR = 72, the last worker holds one row"),
    (33, "72(S-1)-1", "NR = 72, the last worker one row short"),
    (63, "72(S-1)", "the largest resident grid, d = 3 mod 4"),
    (64, "8(S-1)", "d = 64, the last on-chip-sweep inverse"),
    (65, "8(S-1)-1", "d = 65: the two-block inverse, last worker 7 rows"),
    (100, "72(S-1)", "d = 100, every worker full"),
    (127, "72(S-2)+1", "d = 127, last worker one row"),
    (128, "72(S-1)", "d = 128: the largest kernel shape"),
    (128, 25, "d = 128 on four workers (kd > NR)"),
    (127, 7, "d = 127 on one worker"),
    (100, 1, "d = 100, n = 1"),
    (64, 17, "d = 64 on three workers"),
    (33, 1, "d = 33, n = 1"),
    (5, "72(S-1)", "d = 5 on the largest grid"),
    (1, "72(S-1)-1", "d = 1 on the largest grid"),
    (2, "8(S-1)+1", "d = 2, NR = 16"),
    (3, "72(S-1)", "d = 3 on the largest grid"),
    (66, "72(S-2)+1", "d = 2 mod 16 beyond 64, last worker one row"),
]
# persistent kernel, l2: partial last 8-row worker, second pivot block of 1 ... 64 columns; below 64 forced
FUSED_L2 = [65, 66, 71, 73, 79, 80, 97, 120, 121, 127, 128]
FUSED_L2_FORCED = [1, 3, 17, 63, 64]
# launch sequence
SEQ_L2 = [129, 160, 255, 256, 257, 300, 511, 513, 600]
SEQ_LOGISTIC = [(129, 500), (200, 10000), (257, 4097), (100, "72(S-1)+1"), (101, 20001), (520, 19999), (1030, 9473)]

LI_EDGES = {
    "logistic: one worker": lambda p: p["logistic"] and p["NW"] == 1,
    "logistic: 2 or 3 workers (fewer than the 4 reduction lanes)": lambda p: p["logistic"] and 2 <= p["NW"] <= 3,
    "logistic: n < 8 (a partial row tile)": lambda p: p["logistic"] and p["n"] < 8,
    "logistic: NR = 8, S - 1 full workers": lambda p: p["logistic"] and p["NR"] == 8 and p["NW"] == p["S"] - 1 and p["last"] == 8,
    "logistic: NR = 8, S - 1 workers, the last one row short": lambda p: p["logistic"] and p["NR"] == 8 and p["NW"] == p["S"] - 1 and p["last"] == 7,
    "logistic: NR = 16": lambda p: p["logistic"] and p["NR"] == 16,
    "logistic: NR = 72, last worker one row": lambda p: p["logistic"] and p["NR"] == 72 and p["last"] == 1,
    "logistic: NR = 72, last worker 71 rows": lambda p: p["logistic"] and p["NR"] == 72 and p["last"] == 71,
    "logistic: NR = 72, every worker full": lambda p: p["logistic"] and p["NR"] == 72 and p["last"] == 72,
    "logistic: NR > kd (R spills past the staged W)": lambda p: p["logistic"] and p["NR"] > p["kd"],
    "logistic: kd > NR": lambda p: p["logistic"] and p["kd"] > p["NR"],
    "l2: partial last worker (d not a multiple of 8)": lambda p: not p["logistic"] and p["last"] < 8,
    "l2: last worker with one row": lambda p: not p["logistic"] and p["last"] == 1,
    "l2: full last worker": lambda p: not p["logistic"] and p["last"] == 8,
    "l2: second pivot block of 1 column": lambda p: not p["logistic"] and p["d"] == 65,
    "l2: second pivot block of 64 columns": lambda p: not p["logistic"] and p["d"] == 128,
    "l2: d <= 64 (tensor-core sweep)": lambda p: not p["logistic"] and p["d"] <= 64,
    "d = 1": lambda p: p["d"] == 1,
    "d = 128": lambda p: p["d"] == 128,
    **{f"d = {r} mod 4": (lambda r: lambda p: p["d"] % 4 == r)(r) for r in range(4)},
    **{f"d = {r} mod 16": (lambda r: lambda p: p["d"] % 16 == r)(r) for r in (0, 1, 2, 3, 15)},
}


# ---------------------------------------------------------------------------------------------------- GEMM cases
GemmCase = collections.namedtuple("GemmCase", "name trans M N K alpha beta epi lda_pad ldb_pad a_off b_off ws")
_MN = 100 * 100
GEMM_CASES = [
    # balanced 128 x 128 TMA: beta = 0, no epilogue, >= 148 tiles of 128 x 128, K >= 512
    GemmCase("balanced-partial-tiles-K16k+1", False, 1537, 1551, 513, 1.3, 0.0, 0, 1, 1, 0, 0, None),
    GemmCase("balanced-K16k-1", False, 1664, 1600, 527, -0.7, 0.0, 0, 1, 0, 0, 0, None),
    GemmCase("balanced-K1024-padded-ld", False, 1540, 1544, 1024, 1.0, 0.0, 0, 2, 4, 0, 0, None),
    # the same products with an odd lda or a misaligned operand: back to cp.async
    GemmCase("odd-lda-falls-back", False, 1537, 1550, 514, 1.0, 0.0, 0, 1, 0, 0, 0, None),
    GemmCase("odd-ldb-falls-back", False, 1537, 1550, 514, 1.0, 0.0, 0, 0, 1, 0, 0, None),
    GemmCase("A-offset-falls-back", False, 1537, 1550, 514, 1.0, 0.0, 0, 0, 0, 1, 0, None),
    GemmCase("B-offset-falls-back", False, 1537, 1550, 514, 1.0, 0.0, 0, 0, 0, 0, 1, None),
    # queued 128 x 128 TMA: beta != 0 or an epilogue, >= 592 tiles, K >= 1024
    GemmCase("queue-alpha=beta=1", False, 3073, 3000, 1025, 1.0, 1.0, 0, 1, 0, 0, 0, None),
    GemmCase("queue-general-K16k-1", False, 3073, 3000, 1039, 0.7, -1.3, 0, 1, 0, 0, 0, None),
    GemmCase("queue-sigmoid", False, 3073, 3000, 1040, 0.01, 0.0, 1, 0, 0, 0, 0, None),
    # cp.async, no split
    GemmCase("K0-beta0", False, 130, 77, 0, 1.0, 0.0, 0, 0, 0, 0, 0, None),
    GemmCase("K0-beta0.5", False, 130, 77, 0, 1.0, 0.5, 0, 0, 0, 0, 0, None),
    GemmCase("K0-beta0-sigmoid", False, 130, 77, 0, 0.7, 0.0, 1, 0, 0, 0, 0, None),
    GemmCase("K0-beta0.5-sigmoid", False, 130, 77, 0, -2.0, 0.5, 1, 0, 0, 0, 0, None),
    GemmCase("K0-trans-split-ws", True, 100, 100, 0, 1.0, 0.5, 0, 0, 0, 0, 0, 148 * _MN),
    GemmCase("K1", False, 130, 77, 1, 0.7, -1.3, 0, 0, 0, 0, 0, None),
    GemmCase("K15-alpha=beta=1", False, 130, 77, 15, 1.0, 1.0, 0, 0, 0, 0, 0, None),
    GemmCase("K17-sigmoid", False, 130, 77, 17, 0.3, 0.5, 1, 0, 0, 0, 0, None),
    GemmCase("K1000-odd-lda-B-offset", False, 130, 77, 1000, 0.7, -1.3, 0, 1, 0, 0, 1, None),
    GemmCase("trans-K33", True, 130, 77, 33, 0.7, -1.3, 0, 0, 0, 0, 0, None),
    GemmCase("trans-alpha=beta=1", True, 65, 7, 31, 1.0, 1.0, 0, 0, 0, 0, 0, None),
    # cp.async, split-K (4 output tiles, 257 k-tiles)
    GemmCase("split-ws-all", False, 100, 100, 4097, 0.7, -1.3, 0, 0, 0, 0, 0, 148 * _MN),
    GemmCase("split-ws-three", False, 100, 100, 4097, 0.7, -1.3, 0, 0, 0, 0, 0, 3 * _MN),
    GemmCase("split-ws-below-two", False, 100, 100, 4097, 0.7, -1.3, 0, 0, 0, 0, 0, 3 * _MN // 2),
    GemmCase("split-alpha=beta=1", False, 100, 100, 4095, 1.0, 1.0, 0, 1, 0, 0, 0, 148 * _MN),
    GemmCase("split-trans-sigmoid", True, 100, 100, 4097, 0.01, 0.0, 1, 0, 0, 0, 0, 148 * _MN),
    GemmCase("split-trans-beta-sigmoid", True, 100, 100, 4111, 0.01, -0.5, 1, 0, 0, 1, 0, 148 * _MN),
]


def _lda(c):
    return max((c.M if c.trans else c.K) + c.lda_pad, 1)


def _ldb(c):
    return c.N + c.ldb_pad


def _case_route(c, sms):
    return gemm_route(c.trans, c.M, c.N, c.K, _lda(c), _ldb(c), c.a_off % 2 == 0, c.b_off % 2 == 0, c.beta, c.epi,
                      c.ws * 8 if c.ws is not None else None, sms)


def _products_in_iterations(sms):
    """The GEMMs the launch sequence issues at the shapes of SEQ_L2 / SEQ_LOGISTIC: (product, d, n, route)."""
    out = []
    for d in SEQ_L2 + [1600]:
        out.append(("cov @ W", d, 0, gemm_route(False, d, d, d, d, d, True, True, 0.0, 0, None, sms)))
    for d, nspec in SEQ_LOGISTIC:
        n = _n(nspec, sms)
        out.append(("sigmoid(X @ W)", d, n, gemm_route(False, n, d, d, d, d, True, True, 0.0, 1, None, sms)))
        out.append(("X @ W of the loss", d, n, gemm_route(False, n, d, d, d, d, True, True, 0.0, 0, None, sms)))
        out.append(("X^T R", d, n, gemm_route(True, d, d, n, d, d, True, True, 0.0, 0, (148 * d * d + 8) * 8, sms)))
    return out


GEMM_EDGES = {
    "balanced TMA route": lambda c, r: r[0] == "balanced",
    "balanced, K not a multiple of 16 (zero-filled slab)": lambda c, r: r[0] == "balanced" and c.K % 16 != 0,
    "balanced, partial M and N tiles": lambda c, r: r[0] == "balanced" and c.M % 128 and c.N % 128,
    "queued TMA route": lambda c, r: r[0] == "queue",
    "queued, alpha = beta = 1": lambda c, r: r[0] == "queue" and c.alpha == 1.0 and c.beta == 1.0,
    "queued, sigmoid epilogue": lambda c, r: r[0] == "queue" and c.epi == 1,
    "queued, K not a multiple of 16": lambda c, r: r[0] == "queue" and c.K % 16 != 0,
    "TMA-sized product with an odd lda on cp.async": lambda c, r: r[0] == "cp.async" and _lda(c) % 2 == 1 and c.M * c.N > 10 ** 6,
    "TMA-sized product with an odd ldb on cp.async": lambda c, r: r[0] == "cp.async" and _ldb(c) % 2 == 1 and c.M * c.N > 10 ** 6,
    "TMA-sized product with A off by one double on cp.async": lambda c, r: r[0] == "cp.async" and c.a_off and c.M * c.N > 10 ** 6,
    "TMA-sized product with B off by one double on cp.async": lambda c, r: r[0] == "cp.async" and c.b_off and c.M * c.N > 10 ** 6,
    "cp.async, K = 0, beta = 0": lambda c, r: c.K == 0 and c.beta == 0.0 and c.epi == 0,
    "cp.async, K = 0, beta = 0.5": lambda c, r: c.K == 0 and c.beta == 0.5 and c.epi == 0,
    "cp.async, K = 0, sigmoid": lambda c, r: c.K == 0 and c.epi == 1,
    "cp.async, alpha = beta = 1 (accumulators read from C)": lambda c, r: r == ("cp.async", 1) and c.alpha == 1.0 and c.beta == 1.0,
    "cp.async, sigmoid epilogue": lambda c, r: r == ("cp.async", 1) and c.epi == 1 and c.K > 0,
    "cp.async, trans_a": lambda c, r: r == ("cp.async", 1) and c.trans and c.K > 0,
    "split-K, ws for every split": lambda c, r: r[0] == "cp.async" and r[1] > 3,
    "split-K, ws for only three splits": lambda c, r: r == ("cp.async", 3),
    "split-K refused, ws for fewer than two": lambda c, r: c.ws is not None and c.K > 0 and r == ("cp.async", 1),
    "split-K, alpha = beta = 1": lambda c, r: r[0] == "cp.async" and r[1] > 1 and c.alpha == 1.0 and c.beta == 1.0,
    "split-K, trans_a with sigmoid": lambda c, r: r[0] == "cp.async" and r[1] > 1 and c.trans and c.epi == 1,
    "partial M and N tiles on cp.async": lambda c, r: r[0] == "cp.async" and c.M % 64 and c.N % 64,
}
ITER_GEMM_EDGES = {
    "cov @ W on the balanced route inside an iteration": lambda p, d, n, r: p == "cov @ W" and r[0] == "balanced",
    "the loss's X @ W on the balanced route, partial K slab":
        lambda p, d, n, r: p == "X @ W of the loss" and r[0] == "balanced" and d % 16 != 0,
    "sigmoid(X @ W) on the queued route, d >= 1024": lambda p, d, n, r: p == "sigmoid(X @ W)" and r[0] == "queue" and d >= 1024,
    "sigmoid(X @ W) of a TMA-sized product on cp.async because lda = d is odd":
        lambda p, d, n, r: p == "sigmoid(X @ W)" and r[0] == "cp.async" and d % 2 == 1 and _cdiv(n, 64) * _cdiv(d, 64) >= 296,
    "X^T R with split-K": lambda p, d, n, r: p == "X^T R" and r[0] == "cp.async" and r[1] > 1,
}


def _default_env_or_skip(*names):
    for k in names:
        if os.environ.get(k) not in (None, ""):
            pytest.skip(f"{k} is set: the restatement describes the defaults")


def test_li_plan_restatement_matches_library():
    from midagma_b200 import _lib
    _default_env_or_skip("DAGMA_LIN_STREAM")
    lib, sms = _lib.load(), _sms()
    _lib.require_device()
    ns = sorted({1, 2, 7, 8, 9, 16, 17, 24, 25, 33, 100, 1000, 10 ** 5} | {f(sms) for f in N_SPECS.values()})
    for d in range(1, 130):
        p = li_plan(0, 0, d, sms)
        assert bool(lib.dagma_linear_iter_supported(0, 0, d)) == (p is not None), ("l2", d)
        assert lib.dagma_linear_iter_workspace_doubles(0, 0, d) == (p["ws"] if p else 0), ("l2", d)
        for n in ns:
            p = li_plan(1, n, d, sms)
            assert bool(lib.dagma_linear_iter_supported(1, n, d)) == (p is not None), ("logistic", n, d)
            assert lib.dagma_linear_iter_workspace_doubles(1, n, d) == (p["ws"] if p else 0), ("logistic", n, d)


def _kernels_of(fn):
    """(name, grid) of every kernel that ``fn`` launches, from a torch.profiler trace."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    ks = [(e["name"], e.get("args", {}).get("grid")) for e in events if e.get("cat") == "kernel"]
    assert all(g is not None for _, g in ks), "the profiler trace carries no grid dimensions"
    return [(name, tuple(g)) for name, g in ks]


def test_gemm_route_restatement_matches_library():
    """The kernels a call launches are the ones the restated route names: the zeroing kernel and the TMA kernel for
    the balanced schedule, the TMA kernel alone for the queue, the cp.async kernel with grid.z = splits (and the
    fixed-order reduction when splits > 1)."""
    _default_env_or_skip("DAGMA_TMA", "DAGMA_TMA_GEMM_MODE", "DAGMA_GEMM_TILE")
    sms = _sms()
    for c in GEMM_CASES:
        route, splits = _case_route(c, sms)
        call = _GemmCall(c)
        ks = _kernels_of(call.run)
        names = [k[0] for k in ks]
        tma = [k for k in ks if "gemm_tma_kernel" in k[0]]
        zero = [k for k in ks if "gemm_tma_zero_shared_kernel" in k[0]]
        tile = [k for k in ks if "gemm_f64_kernel" in k[0]]
        red = [k for k in ks if "splitk_reduce_kernel" in k[0]]
        print(c.name, route, splits, names)
        if route == "balanced":
            assert len(tma) == 1 and len(zero) == 1 and not tile and "TmaCfg<128" in tma[0][0].replace(" ", ""), names
        elif route == "queue":
            assert len(tma) == 1 and not zero and not tile and "TmaCfg<128" in tma[0][0].replace(" ", ""), names
        else:
            assert not tma and not zero and len(tile) == 1, names
            assert tile[0][1][2] == splits, (c.name, tile[0][1], splits)
            assert len(red) == (1 if splits > 1 else 0), names


def test_shape_lists_reach_every_plan_edge():
    sms = _sms()
    plans = [li_plan(1, _n(n, sms), d, sms) for d, n, _ in FUSED_LOGISTIC]
    plans += [li_plan(0, 0, d, sms) for d in FUSED_L2 + FUSED_L2_FORCED]
    assert all(p is not None for p in plans)
    hit = {name: [f"{'logistic' if p['logistic'] else 'l2'} d={p['d']} n={p['n']}" for p in plans if pred(p)]
           for name, pred in LI_EDGES.items()}
    for c in GEMM_CASES:
        r = _case_route(c, sms)
        for name, pred in GEMM_EDGES.items():
            if pred(c, r):
                hit.setdefault(name, []).append(f"gemm {c.name} -> {r}")
    for prod, d, n, r in _products_in_iterations(sms):
        for e, pred in ITER_GEMM_EDGES.items():
            if pred(prod, d, n, r):
                hit.setdefault(e, []).append(f"{prod} at d={d} n={n} -> {r}")
    for name in list(GEMM_EDGES) + list(ITER_GEMM_EDGES):
        hit.setdefault(name, [])
    # the launch-sequence logistic shapes really leave the persistent kernel
    for d, nspec in SEQ_LOGISTIC:
        assert li_plan(1, _n(nspec, sms), d, sms) is None, (d, nspec)
    missing = [k for k, v in hit.items() if not v]
    print("\n".join(f"{k}: {v[0]}" for k, v in hit.items() if v))
    assert not missing, f"no shape reaches {missing}"


# =====================================================================================================================
# problems, starts, the oracle (cached) and the device runs
# =====================================================================================================================
Run = collections.namedtuple("Run", "loss d n seed lam lr calls checkpoint exclude include")
# (mu, s, iterations, chained): K = 1, then two chained stages with checkpoints inside
CALLS = ((1.0, 1.0, 1, False), (1.0, 1.0, 30, False), (0.1, 0.8, 20, True))
CALLS_SHORT = ((1.0, 1.0, 1, False), (1.0, 1.0, 12, False), (0.1, 0.8, 8, True))
CALLS_TINY = ((1.0, 1.0, 1, False), (1.0, 1.0, 2, False), (0.1, 0.8, 1, True))
Result = collections.namedtuple("Result", "W ok iters ckpts last_lr halved")


def _data(loss, d, n, seed):
    rng = np.random.default_rng(seed)
    if loss == "l2":                     # a sparse upper-triangular SEM
        B = np.triu(rng.normal(size=(d, d)) * (rng.random((d, d)) < 2.0 / max(d, 2)), 1)
        return rng.normal(size=(n, d)) @ np.linalg.inv(np.eye(d) - B)
    z = rng.normal(size=(n, 1)) + 0.5 * rng.normal(size=(1, d))          # correlated binary columns
    return (rng.random((n, d)) < 1.0 / (1.0 + np.exp(-z))).astype(np.float64)


def _w0(d, seed):
    """Generic start: entries ~ N(0, 0.2 / d) (row sums of W o W ~ 0.2, inside the domain at s = 0.8), zero
    diagonal, no ties."""
    W = np.random.default_rng(seed + 7).normal(size=(d, d)) * math.sqrt(0.2 / d)
    np.fill_diagonal(W, 0.0)
    return W


@functools.lru_cache(maxsize=None)
def _oracle_run(run):
    X = _data(run.loss, run.d, run.n, run.seed)
    o = OracleLinear(run.loss).prepare(X, run.lam, checkpoint=run.checkpoint, exclude_edges=run.exclude,
                                       include_edges=run.include)
    W0 = _w0(run.d, run.seed)
    out, W = [], W0
    for mu, s, iters, chain in run.calls:
        ev = len(o.events)
        W, ok = o.minimize((W if chain else W0).copy(), mu, iters, s, run.lr)
        halved = sum(1 for e in o.events[ev:] if e[0] == "lr_halved")
        out.append(Result(W.copy(), ok, o.last_iters, [c[:4] for c in o.checkpoints], o.last_lr if ok else None, halved))
    return out


def _model(run, monkeypatch, force=False):
    from midagma_b200 import DagmaLinear
    monkeypatch.delenv("DAGMA_LIN_FUSED", raising=False)
    if force:
        monkeypatch.setattr(DagmaLinear, "_small_ok", lambda self: False)
    m = DagmaLinear(run.loss)
    m.fit(_data(run.loss, run.d, run.n, run.seed), lambda1=run.lam, T=1, warm_iter=0, max_iter=0,
          checkpoint=run.checkpoint, exclude_edges=run.exclude, include_edges=run.include)
    return m


def _device_run(m, run):
    W0 = _w0(run.d, run.seed)
    out, W = [], W0
    for mu, s, iters, chain in run.calls:
        m.checkpoint_log = []
        W, ok = m.minimize((W if chain else W0).copy(), mu, iters, s, lr=run.lr)
        last_lr = m._large.last_lr
        halved = round(math.log2(run.lr / last_lr)) if ok else None
        out.append(Result(W.copy(), ok, m.last_iters, [tuple(r[1:5]) for r in m.checkpoint_log], last_lr if ok else None,
                          halved))
    return out


_WORST = collections.defaultdict(lambda: (0.0, None))


def _record(section, err, where):
    if err > _WORST[section][0]:
        _WORST[section] = (err, where)


def _elimination_growth(M):
    """max |entry| met by Gaussian elimination without pivoting, over max |M| (the blocked inverse does not pivot)."""
    A, g = M.copy(), np.abs(M).max()
    for k in range(A.shape[0] - 1):
        A[k + 1:, k:] -= np.outer(A[k + 1:, k] / A[k, k], A[k, k:])
        g = max(g, np.abs(A[k + 1:, k + 1:]).max())
    return g / np.abs(M).max()


def _ckpt_rtol(W, s):
    """CKPT_RTOL inside the domain.  A step can leave it (lr = 1: sI - W o W is no M-matrix, the next iteration
    backs off): the objective of such a W is reported, and log|det| from elimination without pivoting is then only as
    good as its element growth allows (1e-12 growth: 5e7 at the lr = 1 shapes below, measured error <= 1.6e-5)."""
    M = s * np.eye(W.shape[0]) - W * W
    if not np.any(np.linalg.inv(M) < 0.0):
        return CKPT_RTOL
    return max(CKPT_RTOL, 1e-12 * _elimination_growth(M))


def _compare(got, ref, label, section, run):
    for k, (g, r) in enumerate(zip(got, ref)):
        s = run.calls[k][1]
        where = f"{label} call {k}"
        assert g.ok == r.ok and g.iters == r.iters, (where, g.ok, r.ok, g.iters, r.iters)
        err = _relmax(g.W, r.W)
        _record(section + " W", err, where)
        assert err <= W_RTOL, (where, err)
        if r.ok:
            assert g.last_lr == r.last_lr and g.halved == r.halved, (where, g.last_lr, r.last_lr, r.halved)
        assert len(g.ckpts) == len(r.ckpts), (where, len(g.ckpts), len(r.ckpts))
        for j, ((it, obj, score, h), (it_r, obj_r, score_r, h_r)) in enumerate(zip(g.ckpts, r.ckpts)):
            assert int(it) == it_r, (where, it, it_r)
            # the last checkpoint of a call is at the returned W (earlier ones: W inside the domain, it went on)
            rtol = _ckpt_rtol(r.W, s) if j == len(r.ckpts) - 1 else CKPT_RTOL
            tag = "" if rtol == CKPT_RTOL else " (W outside the domain)"
            for name, a, b in (("obj", obj, obj_r), ("score", score, score_r), ("h", h, h_r)):
                e = abs(a - b) / max(abs(b), 1e-6)
                _record(section + " checkpoint " + name + tag, e, f"{where} iter {it_r}")
                assert e <= rtol, (where, name, it_r, a, b, rtol)
    print(label, {k: f"{v[0]:.2e}" for k, v in _WORST.items()})


def _masks(d, rows_from):
    """Exclude / include edges in the rows from ``rows_from`` on, in the last column and in the last (partly padded)
    16-wide column tile; none on the diagonal, the two sets disjoint."""
    t = 16 * ((d - 1) // 16)                 # first column of the last 16-wide tile
    exc = [(d - 1, 0), (rows_from, t), (0, d - 1), (d - 2, d - 1)]
    inc = [(d - 1, t + 1 if t + 1 < d - 1 else 1), (rows_from, d - 2), (1, d - 1), (d - 2, t)]
    exc = [e for e in dict.fromkeys(exc) if e[0] != e[1]]
    inc = [e for e in dict.fromkeys(inc) if e[0] != e[1] and e not in exc]
    return tuple(exc), tuple(inc)


def _check_masks(got, run):
    for g in got:
        for (i, j) in run.exclude or ():
            assert g.W[i, j] == 0.0


# =====================================================================================================================
# persistent kernel against the oracle
# =====================================================================================================================
@pytest.mark.parametrize("d,nspec,what", FUSED_LOGISTIC, ids=[f"d{d}-n{n}" for d, n, _ in FUSED_LOGISTIC])
def test_persistent_logistic(monkeypatch, d, nspec, what):
    n = _n(nspec, _sms())
    run = Run("logistic", d, n, 1000 + d, 0.02, 3e-4, CALLS, 12, None, None)
    m = _model(run, monkeypatch)
    assert m._large_engine().one_kernel
    _compare(_device_run(m, run), _oracle_run(run), f"persistent logistic d={d} n={n} ({what})", "persistent", run)


@pytest.mark.parametrize("d", FUSED_L2 + FUSED_L2_FORCED)
def test_persistent_l2(monkeypatch, d):
    run = Run("l2", d, 200, 2000 + d, 0.02, 3e-4, CALLS, 12, None, None)
    m = _model(run, monkeypatch, force=d <= 64)
    assert m._large_engine().one_kernel
    _compare(_device_run(m, run), _oracle_run(run), f"persistent l2 d={d}", "persistent", run)


@pytest.mark.parametrize("loss,d,nspec", [("l2", 73, 0), ("l2", 121, 0), ("logistic", 65, "8(S-1)+1"),
                                          ("logistic", 127, 9)])
def test_persistent_masks(monkeypatch, loss, d, nspec):
    sms = _sms()
    n = _n(nspec, sms) if loss == "logistic" else 200
    p = li_plan(1 if loss == "logistic" else 0, n, d, sms)
    rows_from = 8 * (p["NW"] - 1) if loss == "l2" else d - 2       # l2: the last worker's rows of T
    exc, inc = _masks(d, rows_from)
    run = Run(loss, d, n, 3000 + d, 0.05, 3e-4, CALLS, 12, exc, inc)
    m = _model(run, monkeypatch)
    assert m._large_engine().one_kernel
    got = _device_run(m, run)
    _compare(got, _oracle_run(run), f"persistent {loss} d={d} masks", "persistent", run)
    _check_masks(got, run)


@pytest.mark.parametrize("loss,d,n", [("l2", 65, 130), ("l2", 128, 256), ("logistic", 33, 500)])
def test_persistent_backtracking(monkeypatch, loss, d, n):
    """lr = 1: the inverse turns infeasible inside a launch; the host halves lr as the oracle does."""
    run = Run(loss, d, n, 4000 + d, 0.02, 1.0, CALLS, 12, None, None)
    ref = _oracle_run(run)
    assert ref[1].halved > 0
    m = _model(run, monkeypatch)
    assert m._large_engine().one_kernel
    _compare(_device_run(m, run), ref, f"persistent {loss} d={d} lr=1", "persistent", run)


# =====================================================================================================================
# launch sequence against the oracle
# =====================================================================================================================
def _check_pieces(m, run, label):
    """_score, _h and _func at a generic W against the oracle's score, h and func (1e-12 relative)."""
    o = OracleLinear(run.loss).prepare(_data(run.loss, run.d, run.n, run.seed), run.lam, checkpoint=run.checkpoint)
    W = _w0(run.d, run.seed + 1) * 1.5
    for s in (1.0, 0.9):
        loss, G = m._score(W)
        loss_r, G_r = o.score(W)
        h, Gh = m._h(W, s)
        h_r, Gh_r = o.h(W, s)
        obj, score, h2, _ = m._func(W, 0.3, s)
        obj_r, score_r, h2_r, _ = o.func(W, 0.3, s)
        # h = -log|det| + d log s: at s < 1 both terms are of size d |log s| and h is their small difference
        hs = max(abs(h_r), run.d * abs(math.log(s)))
        errs = dict(score=abs(loss - loss_r) / abs(loss_r), grad=_relmax(G, G_r), h=abs(h - h_r) / hs,
                    h_grad=_relmax(Gh, Gh_r), obj=abs(obj - obj_r) / max(abs(obj_r), hs),
                    func_h=abs(h2 - h2_r) / hs)
        for k, e in errs.items():
            _record("pieces " + k, e, f"{label} s={s}")
        assert max(errs.values()) <= 1e-12, (label, s, errs)


@pytest.mark.parametrize("d", SEQ_L2 + [1600])
def test_launch_sequence_l2(monkeypatch, d):
    calls = CALLS if d <= 300 else CALLS_SHORT if d <= 600 else ((1.0, 1.0, 1, False), (1.0, 1.0, 4, False),
                                                                   (0.1, 0.8, 2, True))
    run = Run("l2", d, max(200, d), 5000 + d, 0.02, 3e-4, calls, 12 if d <= 300 else 5 if d <= 600 else 2, None, None)
    m = _model(run, monkeypatch)
    assert not m._large_engine().one_kernel
    _compare(_device_run(m, run), _oracle_run(run), f"launch sequence l2 d={d}", "launch sequence", run)
    _check_pieces(m, run, f"l2 d={d}")


@pytest.mark.parametrize("d,nspec", SEQ_LOGISTIC, ids=[f"d{d}-n{n}" for d, n in SEQ_LOGISTIC])
def test_launch_sequence_logistic(monkeypatch, d, nspec):
    n = _n(nspec, _sms())
    calls, ck = (CALLS, 12) if d <= 257 else (CALLS_SHORT, 5) if d < 1024 else (CALLS_TINY, 2)
    run = Run("logistic", d, n, 6000 + d, 0.02, 3e-4, calls, ck, None, None)
    m = _model(run, monkeypatch)
    assert not m._large_engine().one_kernel
    _compare(_device_run(m, run), _oracle_run(run), f"launch sequence logistic d={d} n={n}", "launch sequence", run)
    _check_pieces(m, run, f"logistic d={d} n={n}")


@pytest.mark.parametrize("loss,d,n", [("l2", 257, 300), ("logistic", 129, 500)])
def test_launch_sequence_masks(monkeypatch, loss, d, n):
    exc, inc = _masks(d, d - 2)
    run = Run(loss, d, n, 7000 + d, 0.05, 3e-4, CALLS, 12, exc, inc)
    m = _model(run, monkeypatch)
    assert not m._large_engine().one_kernel
    got = _device_run(m, run)
    _compare(got, _oracle_run(run), f"launch sequence {loss} d={d} masks", "launch sequence", run)
    _check_masks(got, run)


@pytest.mark.parametrize("d", [130, 300])
def test_launch_sequence_halt_in_long_interval(monkeypatch, d):
    """Back-tracking in the graph path when the checkpoint interval (80) is longer than the probe interval of the
    latch (64): the halt at iteration 2 stops the replays at the first probe, the rest of the interval resumes."""
    from midagma_b200._large import LargeLinearEngine
    assert LargeLinearEngine.PROBE == 64
    run = Run("l2", d, 2 * d, 8000 + d, 0.02, 0.3, ((1.0, 1.0, 80, False),), 80, None, None)
    ref = _oracle_run(run)
    assert ref[0].halved > 0 and ref[0].ok
    m = _model(run, monkeypatch)
    assert not m._large_engine().one_kernel
    _compare(_device_run(m, run), ref, f"launch sequence l2 d={d} halt", "launch sequence", run)


@pytest.mark.parametrize("loss,d,n", [("l2", 130, 260), ("logistic", 129, 500)])
def test_launch_sequence_infeasible_start_and_out_of_domain(monkeypatch, loss, d, n):
    run = Run(loss, d, n, 9000 + d, 0.02, 0.3, ((1.0, 0.8, 40, False),), 20, None, None)
    m = _model(run, monkeypatch)
    assert not m._large_engine().one_kernel
    if loss == "l2":                     # a halt at s <= 0.9 after a feasible first iteration: ST_OUT_OF_DOMAIN
        ref = _oracle_run(run)
        assert not ref[0].ok and ref[0].iters >= 1
        _compare(_device_run(m, run), ref, f"launch sequence {loss} d={d} out of domain", "launch sequence", run)
    W0 = np.zeros((d, d))
    W0[0, 1] = W0[1, 0] = 1.5
    W1, ok = m.minimize(W0.copy(), 1.0, 10, 1.0, lr=3e-4)
    assert not ok and np.array_equal(W1, W0) and m.last_iters == 0


@pytest.mark.skipif(os.environ.get("DAGMA_LOOKAHEAD") == "2", reason="already the flow kernel")
def test_launch_sequence_flow_kernel():
    """The l2 cases at even d > 256 once more with DAGMA_LOOKAHEAD=2: the inverse as one dependency-driven kernel
    carrying cov @ W as its rider (the switch is read once per process, hence the subprocess)."""
    even = [d for d in SEQ_L2 + [1600] if d > 256 and d % 2 == 0]
    ids = [f"{os.path.abspath(__file__)}::test_launch_sequence_l2[{d}]" for d in even]
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider", *ids],
                       env=dict(os.environ, DAGMA_LOOKAHEAD="2"), cwd=ROOT, capture_output=True, text=True,
                       timeout=1200)
    assert r.returncode == 0 and f"{len(even)} passed" in r.stdout, r.stdout[-3000:] + r.stderr[-2000:]


# =====================================================================================================================
# the blocked inverse through its C ABI
# =====================================================================================================================
def _inv_problem(d, s, square, seed):
    rng = np.random.default_rng(seed)
    A = rng.normal(size=(d, d)) * (rng.random((d, d)) < 0.05)
    if not square:
        A = np.abs(A)
    B = A * A if square else A
    rho = max(np.abs(np.linalg.eigvals(B)).max(), 1e-12)
    A *= np.sqrt(0.7 * s / rho) if square else 0.7 * s / rho
    return A


def _inv_expect(A, s, square):
    d = A.shape[0]
    M = s * np.eye(d) - (A * A if square else A)
    Minv = np.linalg.inv(M)
    minors_pos = all(np.linalg.slogdet(M[:k, :k])[0] > 0 for k in [1, 2, 3, 4] + list(range(8, d + 1, max(1, d // 16))) + [d])
    info0 = minors_pos and Minv.min() + 1e-16 >= 0.0
    return M, Minv, np.linalg.slogdet(M)[1], (2 * A * Minv.T if square else Minv.T), info0


def _padded(X, ld, fill=float("nan")):
    rows, cols = X.shape[-2:]
    buf = torch.full(X.shape[:-2] + (rows, ld), fill, **F64)
    buf[..., :cols] = torch.from_numpy(X)
    return buf


@pytest.mark.parametrize("s", [0.3, 0.5, 0.9, 1.0, 2.5])
@pytest.mark.parametrize("d", [129, 200, 256, 257, 300])
def test_blocked_inverse_abi(d, s):
    """dagma_logdet_inv_ws_f64 with lda = d + 3, ldo = d + 5 (NaN padding untouched): inverse only, gradient only,
    both, square_input = 0; every scale branch (s = 0.3 and 0.5: scale 1/2, 0.9 and 1: 1, 2.5: 4)."""
    from midagma_b200 import _lib
    lib = _lib.load()
    lda, ldo = d + 3, d + 5
    ws = torch.empty(lib.dagma_large_workspace_bytes(d) // 8 + 8, **F64)
    for mode in ("inv", "grad", "both", "both-unsquared"):
        square = mode != "both-unsquared"
        A = _inv_problem(d, s, square, d * 10 + int(10 * s))
        M, Minv, lad, G, info0 = _inv_expect(A, s, square)
        Ad = _padded(A, lda)
        minv = torch.full((d, ldo), float("nan"), **F64) if mode != "grad" else None
        grad = torch.full((d, ldo), float("nan"), **F64) if mode != "inv" else None
        sc = torch.full((4,), float("nan"), **F64)
        info = torch.full((1,), -7, dtype=torch.int32, device="cuda")
        _lib.check(lib.dagma_logdet_inv_ws_f64(
            _lib.stream_ptr(), d, s, Ad.data_ptr(), lda, int(square), sc.data_ptr(), sc.data_ptr() + 8,
            minv.data_ptr() if minv is not None else None, grad.data_ptr() if grad is not None else None, ldo,
            sc.data_ptr() + 16, info.data_ptr(), ws.data_ptr(), ws.numel() * 8), "dagma_logdet_inv_ws_f64")
        torch.cuda.synchronize()
        assert (int(info.item()) == 0) == info0 and info0
        scv = sc.cpu().numpy()
        assert abs(scv[0] - lad) <= 1e-10 * max(1.0, abs(lad)), (mode, scv[0], lad)
        assert abs(scv[1] - (-lad + d * np.log(s))) <= 1e-10 * max(1.0, abs(lad)), (mode, scv[1])
        assert abs(scv[2] - Minv.min()) <= 1e-10 * np.abs(Minv).max(), (mode, scv[2], Minv.min())
        _record("inverse log|det|", abs(scv[0] - lad) / max(1.0, abs(lad)), f"d={d} s={s} {mode}")
        for out, ref in ((minv, Minv), (grad, G)):
            if out is None:
                continue
            o = out.cpu().numpy()
            assert np.isnan(o[:, d:]).all(), "padding written"
            e = _relmax(o[:, :d], ref)
            _record("inverse outputs", e, f"d={d} s={s} {mode}")
            assert e <= 1e-10, (mode, e)
        assert np.isnan(Ad.cpu().numpy()[:, d:]).all()
    # outside the domain: flagged
    A = _inv_problem(d, s, True, d)
    A[0, 1] = A[1, 0] = 3.0 * math.sqrt(s)
    *_, info0 = _inv_expect(A, s, True)
    info = torch.full((1,), -7, dtype=torch.int32, device="cuda")
    Ad = _padded(A, lda)
    _lib.check(lib.dagma_logdet_inv_ws_f64(_lib.stream_ptr(), d, s, Ad.data_ptr(), lda, 1, None, None, None, None, ldo,
                                           None, info.data_ptr(), ws.data_ptr(), ws.numel() * 8), "dagma_logdet_inv_ws_f64")
    assert not info0 and int(info.item()) != 0


@pytest.mark.parametrize("d,s", [(200, 0.3), (257, 2.5)])
def test_blocked_inverse_batch(d, s):
    """dagma_logdet_inv_f64 with a batch of 3 and padded leading dimensions."""
    from midagma_b200 import _lib
    lib = _lib.load()
    lda, ldo, B = d + 3, d + 5, 3
    As = np.stack([_inv_problem(d, s, True, 77 + b) for b in range(B)])
    Ad = _padded(As, lda)
    minv, grad = torch.full((B, d, ldo), float("nan"), **F64), torch.full((B, d, ldo), float("nan"), **F64)
    lad, h, mn = (torch.full((B,), float("nan"), **F64) for _ in range(3))
    info = torch.full((B,), -7, dtype=torch.int32, device="cuda")
    _lib.check(lib.dagma_logdet_inv_f64(_lib.stream_ptr(), B, d, s, Ad.data_ptr(), lda, 1, lad.data_ptr(), h.data_ptr(),
                                        minv.data_ptr(), grad.data_ptr(), ldo, mn.data_ptr(), info.data_ptr()),
               "dagma_logdet_inv_f64")
    torch.cuda.synchronize()
    for b in range(B):
        M, Minv, lad_r, G, info0 = _inv_expect(As[b], s, True)
        assert info0 and int(info[b].item()) == 0
        assert abs(lad[b].item() - lad_r) <= 1e-10 * max(1.0, abs(lad_r))
        assert abs(h[b].item() - (-lad_r + d * np.log(s))) <= 1e-10 * max(1.0, abs(lad_r))
        assert abs(mn[b].item() - Minv.min()) <= 1e-10 * np.abs(Minv).max()
        for out, ref in ((minv[b], Minv), (grad[b], G)):
            o = out.cpu().numpy()
            assert np.isnan(o[:, d:]).all()
            assert _relmax(o[:, :d], ref) <= 1e-10


# =====================================================================================================================
# dagma_gemm_f64 on every route
# =====================================================================================================================
class _GemmCall:
    """Operands of a GemmCase on the device (padding and offsets as the case says, NaN in the padding and in C
    when beta = 0) and the float64 reference."""

    def __init__(self, c):
        from midagma_b200 import _lib
        self.c, self.lib, self._lib = c, _lib.load(), _lib
        rng = np.random.default_rng(zlib.crc32(c.name.encode()))
        Ashape = (c.K, c.M) if c.trans else (c.M, c.K)
        self.A, self.B = rng.normal(size=Ashape), rng.normal(size=(c.K, c.N))
        self.C0 = rng.normal(size=(c.M, c.N)) if c.beta != 0.0 else np.full((c.M, c.N), np.nan)
        self.lda, self.ldb = _lda(c), _ldb(c)
        self.Ab = self._buf(self.A, self.lda, c.a_off)
        self.Bb = self._buf(self.B, self.ldb, c.b_off)
        self.Cd = torch.from_numpy(self.C0.copy()).cuda()
        self.ws = torch.empty(c.ws, **F64) if c.ws is not None else None

    @staticmethod
    def _buf(X, ld, off):
        rows, cols = X.shape
        buf = torch.full((off + max(rows, 1) * ld,), float("nan"), **F64)     # never empty: K = 0 still passes A
        if rows and cols:
            buf[off:].view(rows, ld)[:, :cols] = torch.from_numpy(X)
        return buf

    def run(self):
        c = self.c
        self.Cd.copy_(torch.from_numpy(self.C0))
        rc = self.lib.dagma_gemm_f64(self._lib.stream_ptr(), int(c.trans), c.M, c.N, c.K, c.alpha,
                                     self.Ab.data_ptr() + 8 * c.a_off, self.lda, self.Bb.data_ptr() + 8 * c.b_off,
                                     self.ldb, c.beta, self.Cd.data_ptr(), c.N, c.epi,
                                     self.ws.data_ptr() if self.ws is not None else None,
                                     self.ws.numel() * 8 if self.ws is not None else 0)
        self._lib.check(rc, "dagma_gemm_f64")
        return self.Cd.cpu().numpy()

    def check(self, C):
        c = self.c
        opA = self.A.T if c.trans else self.A
        z = c.alpha * (opA @ self.B) if c.K else np.zeros((c.M, c.N))
        bound = 1e-13 * abs(c.alpha) * (np.abs(opA) @ np.abs(self.B)) if c.K else np.zeros((c.M, c.N))
        if c.beta != 0.0:
            z = z + c.beta * self.C0
            bound = bound + 1e-13 * abs(c.beta) * np.abs(self.C0)
        if c.epi == 1:
            z, bound = 1.0 / (1.0 + np.exp(-z)), 0.25 * bound + 1e-15      # the sigmoid is 1/4-Lipschitz
        assert np.isfinite(C).all(), c.name
        err = np.abs(C - z)
        worst = float((err / np.maximum(bound, 1e-300)).max())
        _record("gemm |dC| / bound", worst, c.name)
        assert (err <= bound).all(), (c.name, float(err.max()), worst)
        if c.K == 0 and c.epi == 0:                                         # BLAS: exactly beta C
            assert np.array_equal(C, c.beta * self.C0 if c.beta != 0.0 else np.zeros_like(C)), c.name


@pytest.mark.parametrize("case", GEMM_CASES, ids=[c.name for c in GEMM_CASES])
def test_gemm_routes(case):
    call = _GemmCall(case)
    C = call.run()
    call.check(C)
    if _case_route(case, _sms())[0] == "balanced":                         # two calls, bit for bit
        assert np.array_equal(call.run(), C)


def test_gemm_rejects_short_leading_dimensions():
    from midagma_b200 import _lib
    lib = _lib.load()
    A, B, C = (torch.zeros(64 * 64, **F64) for _ in range(3))
    call = lambda trans, M, N, K, lda: lib.dagma_gemm_f64(_lib.stream_ptr(), trans, M, N, K, 1.0, A.data_ptr(), lda,  # noqa: E731
                                                          B.data_ptr(), N, 0.0, C.data_ptr(), N, 0, None, 0)
    assert call(0, 8, 8, 10, 9) != 0 and call(1, 10, 8, 8, 9) != 0
    assert call(0, 8, 8, 10, 10) == 0 and call(1, 10, 8, 8, 10) == 0 and call(0, 8, 8, 0, 1) == 0
    torch.cuda.synchronize()


def test_zz_report_largest_errors():
    """Largest error per section over the tests of this module that ran (printed with -s)."""
    for k, (e, where) in sorted(_WORST.items()):
        print(f"{k}: {e:.2e} at {where}")
