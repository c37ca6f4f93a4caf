"""The on-chip kernels at every size they accept, against float64 references.

* The batched l2 fit (``fit_batch`` / ``minimize_batch``, d <= 64) runs on three kernels picked by d in
  csrc/small_fit.cu: the scalar rank-1 sweep with ``Cfg<1,1,16,16>`` (d <= 16) and ``Cfg<2,2,16,16>`` (d <= 32), and
  the tensor-core kernel of csrc/small_fit_dmma.cu (identity padded to 64, 8 x 8 pivot blocks, fraction-free groups
  of four pivots).  Sizes on both sides of every edge, and padded tensor-core sizes (d % 8 != 0), are compared with
  the numpy oracle (``oracle.linear_ref.OracleLinear``): W, iteration counts, the kernel's checkpoint log, the cold
  branches, and the independence of a problem's result from the CTA that ran it and what that CTA ran before.
* The stand-alone batched slogdet + inverse (csrc/small_inv.cu, ``dagma_logdet_inv_f64``) against LAPACK at every
  path's edges, with batches in which every CTA handles several problems, several s, strided operands, both
  ``info`` codes and the M-matrix boundary.
* ``center_cov`` (csrc/cov.cu) against numpy, and batches beyond the 65 535 limit of a grid's y / z extent.
The A/B switches ``DAGMA_SMALL_CFG`` and ``DAGMA_SMALL_INV_DMMA`` are read once per process: their re-runs are
subprocesses."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import simulate
from oracle.linear_ref import OracleLinear

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _relmax(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


# =====================================================================================================================
# l2 batched fit: helpers
# =====================================================================================================================
def _l2_data(d, n, seed):
    if d == 1:                                      # no graph to simulate: plain Gaussian data
        return np.random.default_rng(seed).normal(size=(n, 1))
    return simulate.make_linear_problem(d, 2, n, "ER", "gauss", seed)[0]


def _generic_start(d, seed, scale=0.05):
    """0.05 N(0, 1) with a zero diagonal: no exact ties in the l1 sign terms (DESIGN.md 2), inside the domain."""
    W0 = np.random.default_rng(seed).normal(size=(d, d)) * scale
    np.fill_diagonal(W0, 0.0)
    assert not np.any(np.linalg.inv(np.eye(d) - W0 * W0) + 1e-16 < 0), "start must be feasible"
    return W0


def _near_boundary_start(d, seed, t=0.999):
    """W0 o W0 = t P with P dense and row-stochastic (Perron root t): a step of lr = 1e-2 leaves the domain for these
    problems when the score gradient dominates (data scaled by 30), and lr is halved."""
    rng = np.random.default_rng(seed)
    P = rng.random((d, d))
    P /= P.sum(axis=1, keepdims=True)
    return np.sqrt(t * P)


def _run(cov, W0, lam, mus, ss, iters, *, lr=3e-4, tol=1e-6, checkpoint=40, retry=False, masks=(None, None)):
    """``_run_small`` (the launcher of fit_batch / minimize_batch) with its checkpoint log, on host arrays:
    (W, status, stage_stats, [per problem: checkpoint rows (stage, iter, obj, score, h, lr)])."""
    import torch
    from midagma_b200.linear import _batch_masks, _run_small
    batch, d, _ = cov.shape
    covd = torch.as_tensor(np.ascontiguousarray(cov)).cuda()
    Wd = torch.as_tensor(np.ascontiguousarray(W0, dtype=np.float64)).cuda()
    lamd = torch.as_tensor(np.broadcast_to(np.asarray(lam, dtype=np.float64), (batch,)).copy()).cuda()
    exc, inc = _batch_masks(*masks, d, "cuda")
    cap = sum(int(k) // checkpoint + 2 for k in iters)
    res = _run_small(covd, Wd, lamd, list(mus), list(ss), [int(k) for k in iters], lr=lr, tol=tol, beta1=0.99,
                     beta2=0.999, checkpoint=checkpoint, retry=retry, want_final=False, mask_exc=exc, mask_inc=inc,
                     ckpt_log_cap=cap)
    log, cnt = res.ckpt_log.cpu().numpy(), res.ckpt_count.cpu().numpy()
    return (Wd.cpu().numpy(), res.status.cpu().numpy(), res.stage_stats.cpu().numpy(),
            [log[b, :cnt[b]] for b in range(batch)])


def _check_vs_oracle(o, W_ref, ok_ref, W, status, st, log, what):
    """One problem of a ``_run`` (one stage) against the oracle's minimize call."""
    d = W.shape[-1]
    assert ((status & 1) == 0) == ok_ref, what
    assert int(st[0]) == o.last_iters, (what, st[0], o.last_iters)
    err = _relmax(W, W_ref)
    assert err <= 1e-9, (what, err)
    ref = np.array(o.checkpoints)
    assert len(log) == len(ref) and np.array_equal(log[:, 1], ref[:, 0]), (what, log[:, 1], ref[:, 0])
    for col, name in ((2, "obj"), (3, "score"), (4, "h")):
        # h is a sum of d logs of pivots, each with an absolute round-off of a few eps on either side: near W = 0 (h
        # of order lr^2 after one step) that, not the 1e-9 relative bar, is the accuracy of both routes
        floor = 4 * d * EPS if col == 4 else 0.0
        tol = 1e-9 * np.abs(ref[:, col - 1]) + floor
        assert np.all(np.abs(log[:, col] - ref[:, col - 1]) <= tol), (what, name, log[:, col], ref[:, col - 1])
    return err


# =====================================================================================================================
# 1. l2 batched fit vs the oracle at every kernel configuration
# =====================================================================================================================
FIT_D = [1, 2, 3, 8, 15, 16, 17, 24, 31, 32, 33, 34, 36, 39, 41, 47, 49, 56, 57, 62, 63, 64]


@pytest.mark.parametrize("d", FIT_D)
def test_l2_fit_vs_oracle(d):
    """K = 1 and K = 100 iterations of minimize (mu = 1, s = 1, checkpoint every 40) from a generic start, then a
    chained stage at mu = 0.1, s = 0.8 (s / 2^e pre-scaling, log|det| at s != 1): W to 1e-9 max-norm relative,
    iteration counts, and the objective / score / h of every checkpoint the kernel logged."""
    X = _l2_data(d, 200, 700 + d)
    lam = 0.05
    o = OracleLinear("l2").prepare(X.copy(), lam, checkpoint=40)
    cov = o.cov[None]
    W0 = _generic_start(d, 900 + d)[None] if d > 1 else np.zeros((1, 1, 1))
    errs = []
    for K in (1, 100):
        W_ref, ok_ref = o.minimize(W0[0].copy(), 1.0, K, 1.0, 3e-4)
        W, status, st, log = _run(cov, W0, lam, [1.0], [1.0], [K])
        errs.append(_check_vs_oracle(o, W_ref, ok_ref, W[0], status[0], st[0, 0], log[0], (d, K)))
    W2_ref, ok2_ref = o.minimize(W_ref.copy(), 0.1, 100, 0.8, 3e-4)
    W2, status, st, log = _run(cov, W, lam, [0.1], [0.8], [100])
    errs.append(_check_vs_oracle(o, W2_ref, ok2_ref, W2[0], status[0], st[0, 0], log[0], (d, "mu=0.1 s=0.8")))
    print(f"l2 fit d={d}: max-norm rel |dW| K=1 {errs[0]:.1e}, K=100 {errs[1]:.1e}, second stage {errs[2]:.1e}")


# =====================================================================================================================
# 2. cold branches at the configuration edges
# =====================================================================================================================
COLD_D = [16, 17, 32, 33, 63]


@pytest.mark.parametrize("d", COLD_D)
def test_cold_backtracking(d):
    """lr = 1 at s = 1 leaves the domain: lr is halved and the step re-taken (linear.py:235-241); the halving count,
    the final lr (exactly) and W match the oracle."""
    X, _ = simulate.make_linear_problem(d, 2, 300, "ER", "gauss", 4)
    o = OracleLinear("l2").prepare(X, 0.0, checkpoint=50)
    W_ref, ok_ref = o.minimize(np.zeros((d, d)), 1.0, 40, 1.0, 1.0)
    n_halved = sum(1 for e in o.events if e[0] == "lr_halved")
    assert n_halved > 0, "test input must exercise back-tracking"
    W, status, st, _ = _run(o.cov[None], np.zeros((1, d, d)), 0.0, [1.0], [1.0], [40], lr=1.0, checkpoint=50)
    err = np.abs(W[0] - W_ref).max()
    print(f"d={d}: halvings oracle {n_halved} gpu {st[0, 0, 7]:.0f}, lr {o.last_lr} / {st[0, 0, 1]}, max|dW| {err:.1e}")
    assert ((status[0] & 1) == 0) == ok_ref
    assert int(st[0, 0, 7]) == n_halved and int(st[0, 0, 0]) == o.last_iters
    assert st[0, 0, 1] == o.last_lr
    assert err <= 1e-6


@pytest.mark.parametrize("d", COLD_D)
def test_cold_infeasible_start(d):
    """A start outside the domain returns (W, False) at iteration 0, alone and in the middle of a batch, and leaves
    its neighbours untouched."""
    from midagma_b200 import minimize_batch
    X, _ = simulate.make_linear_problem(d, 2, 100, "ER", "gauss", 0)
    o = OracleLinear("l2").prepare(X, 0.02, checkpoint=1000)
    cov = o.cov[None]
    W0 = np.zeros((1, d, d))
    W0[0, 0, d - 1], W0[0, d - 1, 0] = 1.5, 1.5
    W, ok, st = minimize_batch(W0.copy(), cov, 0.02, 1.0, 50, 1.0, 3e-4)
    assert not ok[0] and int(st[0, 0, 0]) == 0 and np.array_equal(W, W0)
    W_ref, _ = o.minimize(np.zeros((d, d)), 1.0, 50, 1.0, 3e-4)
    Wb = np.concatenate([np.zeros((1, d, d)), W0, np.zeros((1, d, d))])
    W, ok, st = minimize_batch(Wb.copy(), np.repeat(cov, 3, axis=0), 0.02, 1.0, 50, 1.0, 3e-4)
    assert ok.tolist() == [True, False, True] and st[:, 0, 0].tolist() == [50, 0, 50]
    assert np.array_equal(W[1], W0[0]) and np.array_equal(W[0], W[2])
    assert np.abs(W[0] - W_ref).max() <= 1e-9 * np.abs(W_ref).max()


def _edge_edges(d):
    """Mask entries at tile and mask-word edges: (0, d-1), (d-1, 0), (15, 16), (16, 15), (31, 32), (32, 31),
    (d-1, d-2), where they exist."""
    cand = [(0, d - 1), (d - 1, 0), (15, 16), (16, 15), (31, 32), (32, 31), (d - 1, d - 2)]
    out = []
    for e in cand:
        if max(e) < d and e[0] != e[1] and e not in out:
            out.append(e)
    return out


@pytest.mark.parametrize("flip", [False, True], ids=["set-a", "set-b"])
@pytest.mark.parametrize("d", COLD_D)
def test_cold_masks(d, flip):
    """Exclude / include masks at tile and word edges through fit_batch against OracleLinear.fit; each edge is
    excluded in one parametrisation and included in the other."""
    from midagma_b200 import fit_batch
    X, _ = simulate.make_linear_problem(d, 2, 300, "ER", "gauss", 9)
    edges = _edge_edges(d)
    exc = tuple(e for k, e in enumerate(edges) if (k % 2 == 0) != flip)
    inc = tuple(e for k, e in enumerate(edges) if (k % 2 == 0) == flip)
    kw = dict(lambda1=0.03, T=2, warm_iter=400, max_iter=300, checkpoint=100)
    o = OracleLinear("l2")
    o.fit(X.copy(), s=[1.0, 0.9], exclude_edges=exc, include_edges=inc, **kw)
    _, info = fit_batch(np.stack([X, X]), s=(1.0, 0.9), exclude_edges=exc, include_edges=inc, return_info=True, **kw)
    err = np.abs(info["W_raw"][0] - o.W_raw).max()
    print(f"d={d} masks exc {exc} inc {inc}: max|dW| {err:.1e}, stage iters {info['stage_iters'][0]} {o.stage_iters}")
    assert info["stage_iters"][0].tolist() == o.stage_iters
    assert err <= 1e-8
    assert np.array_equal(info["W_raw"][0], info["W_raw"][1])
    for (i, j) in exc:
        assert info["W_raw"][0][i, j] == 0.0
    for (i, j) in inc:
        assert info["W_raw"][0][i, j] != 0.0


# =====================================================================================================================
# 3. l2 scheduling independence
# =====================================================================================================================
def _mixed_batch(d, batch, seed):
    """Unequal problems: 16 data sets cycled (every fourth scaled by 30), lambda1 in [0.005, 0.1], generic starts; a
    few infeasible starts (return at iteration 0) and a few near-boundary starts on scaled data (the score gradient
    pushes them out of the domain at lr = 1e-2 and they back-track)."""
    rng = np.random.default_rng(seed)
    covs = []
    for k in range(16):
        X = _l2_data(d, 120, 50 + k) * (30.0 if k % 4 == 3 else 1.0)
        covs.append(X.T @ X / 120)
    cov = np.stack([covs[b % 16] for b in range(batch)])
    lam = rng.uniform(0.005, 0.1, size=batch)
    W0 = rng.normal(size=(batch, d, d)) * 0.02
    W0[:, np.arange(d), np.arange(d)] = 0.0
    infeasible = [2, batch // 3 + 1, batch - 7]
    for b in infeasible:
        W0[b] = 0.0
        W0[b, 0, d - 1] = W0[b, d - 1, 0] = 1.5
    backtrack = [x - x % 16 + 3 for x in (16, batch // 2, batch - 32)]          # data sets scaled by 30
    assert not set(infeasible) & set(backtrack)
    for b in backtrack:
        W0[b] = _near_boundary_start(d, b)
    return cov, lam, W0, infeasible, backtrack


def _assert_alone_equal(cov, lam, W0, batched, picks, **kw):
    W, status, st, log = batched
    for b in picks:
        Wa, sa, sta, loga = _run(cov[b:b + 1], W0[b:b + 1], lam[b:b + 1], **kw)
        assert np.array_equal(Wa[0], W[b]), b
        assert sa[0] == status[b] and np.array_equal(sta[0], st[b]), (b, sta[0], st[b])
        assert np.array_equal(loga[0], log[b]), b


@pytest.mark.parametrize("d", [9, 24, 37, 64])
def test_l2_scheduling_independence(d):
    """Three times the resident CTAs, problems of unequal lengths, infeasible and back-tracking problems among them:
    each of the chosen problems gets bit for bit the W, stage statistics and checkpoint log it gets alone (the Adam
    moments in tensor memory and the mask bits are reused from problem to problem)."""
    from midagma_b200.linear import _resident_ctas
    batch = 3 * _resident_ctas()
    cov, lam, W0, infeasible, backtrack = _mixed_batch(d, batch, d)
    kw = dict(mus=[1.0], ss=[1.0], iters=[300], lr=1e-2, tol=3e-3, checkpoint=10)
    W, status, st, log = out = _run(cov, W0, lam, **kw)
    iters = st[:, 0, 0]
    for b in infeasible:
        assert status[b] & 1 and iters[b] == 0 and np.array_equal(W[b], W0[b])
    assert all(st[b, 0, 7] > 0 for b in backtrack), st[backtrack, 0, 7]
    feasible = np.setdiff1d(np.arange(batch), infeasible)
    assert len(np.unique(iters[feasible])) > 3, "problems must stop at different checkpoints"
    picks = sorted({0, batch - 1, int(feasible[np.argmin(iters[feasible])]), int(np.argmax(iters)),
                    infeasible[1] + 1, backtrack[1]})
    print(f"d={d}: batch {batch}, iterations {iters.min():.0f}..{iters.max():.0f}, picks {picks}")
    _assert_alone_equal(cov, lam, W0, out, picks, **kw)


@pytest.mark.parametrize("d", [9, 24, 37, 64])
def test_l2_scheduling_independence_with_retries(d):
    """The same property for a fit whose second stage (s = 0.3) fails and is retried with lr / 2, s + 0.1."""
    from midagma_b200.linear import _resident_ctas
    batch = 3 * _resident_ctas()
    cov, lam, _, _, _ = _mixed_batch(d, batch, 100 + d)
    W0 = np.zeros((batch, d, d))
    kw = dict(mus=[1.0, 0.1], ss=[1.0, 0.3], iters=[200, 200], lr=0.01, checkpoint=50, retry=True)
    W, status, st, log = out = _run(cov, W0, lam, **kw)
    retries = st[:, 1, 6]
    assert retries.max() > 0 and len(np.unique(retries)) > 1, "stages must retry, unequally"
    total = st[:, :, 0].sum(axis=1)
    picks = sorted({0, batch - 1, int(np.argmin(total)), int(np.argmax(total)), int(np.argmax(retries)),
                    int(np.argmin(retries))})
    print(f"d={d}: retries {retries.min():.0f}..{retries.max():.0f}, picks {picks}")
    _assert_alone_equal(cov, lam, W0, out, picks, **kw)


# =====================================================================================================================
# 4. logdet_inv (csrc/small_inv.cu) at every size, s, stride and batch
# =====================================================================================================================
INV_D = [1, 2, 16, 17, 32, 33, 39, 64, 65, 71, 100, 127, 128]
INV_S = [1.0, 0.5, 2.0, 0.25, 0.3, 0.6, 1.7]
INV_S_D = [2, 17, 39, 71, 128]


def _inv_batch_size():
    from midagma_b200 import _lib
    return 5 * _lib.require_device() + 3            # every CTA of every path (grid <= 4 x SMs) does >= 2 problems


def _scaled(B, target):
    """The factor that puts the Perron root of B >= 0 at target (B's largest entry, if B is nilpotent)."""
    rho = np.abs(np.linalg.eigvals(B)).max()
    return target / (rho if rho > 1e-6 * B.max() else B.max())


POOL = 41      # distinct problems per batch, cycled: the grid strides of the paths (SMs, 2 SMs, 4 SMs) are no multiple


def _inv_problems(d, s, square, seed):
    """A pool of POOL problems [POOL, d, d] and their kinds: kind 0 well-conditioned (Perron root of B = 0.6 s, sparse,
    B = A o A or |A|), kind 1 a Z-matrix s I - B with B >= 0 dense and rho(B) = 1.5 s (a non-positive pivot), kind 2
    (square_input = 0 only) signed dense A with rho(|A|) = 0.6 s (positive pivots, negative entries in the inverse)."""
    rng = np.random.default_rng(seed)
    kinds = np.resize((0, 1, 0, 0) if square else (0, 1, 0, 2), POOL)
    A = np.empty((POOL, d, d))
    for b in range(POOL):
        k = kinds[b]
        a = rng.normal(size=(d, d))
        if k == 0:
            a *= rng.random((d, d)) < 0.3
            a[0, 0] += 0.5                          # never all zero
        if k != 2 and not square:
            a = np.abs(a)
        B = a * a if square else np.abs(a)
        f = _scaled(B, (1.5 if k == 1 else 0.6) * s)
        A[b] = a * (np.sqrt(f) if square else f)
    return A, kinds


def _lu_pivots(M):
    """Pivots of the no-pivoting LU of each M [batch, d, d]; after the first non-positive pivot they are not needed."""
    U = M.copy()
    d = M.shape[-1]
    piv = np.empty(M.shape[:-1])
    with np.errstate(divide="ignore", invalid="ignore"):
        for k in range(d):
            p = U[:, k, k].copy()
            piv[:, k] = p
            if k + 1 < d:
                L = U[:, k + 1:, k] / p[:, None]
                U[:, k + 1:, k + 1:] -= L[:, :, None] * U[:, k, None, k + 1:]
    return piv


def _host_info(M, z_matrix):     # z_matrix: [batch] bool
    """The kernel's info code on the host: 1 iff a pivot of the no-pivot LU is <= 0; else 2 iff min(inv) + 1e-16 < 0.
    For a Z-matrix with positive pivots (a nonsingular M-matrix) the exact inverse is >= 0, so 0 (LAPACK leaves
    round-off negatives at its structural zeros, which the predicate must not see)."""
    piv = _lu_pivots(M)
    first_bad = np.argmax(~(piv > 0), axis=1)
    bad = ~np.all(piv > 0, axis=1)
    info = np.zeros(len(M), dtype=np.int64)
    for b in range(len(M)):
        if bad[b]:
            # the decision is not a round-off call: every pivot up to the first bad one is clear of 0
            assert np.abs(piv[b, :first_bad[b] + 1]).min() > 1e-6 * np.abs(M[b]).max(), b
            info[b] = 1
        elif not z_matrix[b]:
            mn = np.linalg.inv(M[b]).min()
            assert not (-1e-12 < mn < 0), (b, mn)
            info[b] = 2 if mn + 1e-16 < 0 else 0
    return info


def _logdet_inv_c(A, s, square, lda, ldo):
    """``dagma_logdet_inv_f64`` through the C ABI with row strides lda (input) and ldo (outputs); the padding of A
    and of the outputs is NaN.  Returns host arrays (minv and grad [batch, d, ldo] with their padding)."""
    import torch
    from midagma_b200 import _lib
    batch, d, _ = A.shape
    Ap = np.full((batch, d, lda), np.nan)
    Ap[:, :, :d] = A
    Ad = torch.as_tensor(Ap).cuda()
    minv = torch.full((batch, d, ldo), float("nan"), dtype=torch.float64, device="cuda")
    grad = torch.full((batch, d, ldo), float("nan"), dtype=torch.float64, device="cuda")
    lad, h, mn = (torch.full((batch,), float("nan"), dtype=torch.float64, device="cuda") for _ in range(3))
    info = torch.full((batch,), -1, dtype=torch.int32, device="cuda")
    _lib.check(_lib.load().dagma_logdet_inv_f64(_lib.stream_ptr(), batch, d, float(s), Ad.data_ptr(), lda, int(square),
                                                lad.data_ptr(), h.data_ptr(), minv.data_ptr(), grad.data_ptr(), ldo,
                                                mn.data_ptr(), info.data_ptr()), "dagma_logdet_inv_f64")
    return {k: v.cpu().numpy() for k, v in dict(logabsdet=lad, h=h, minv=minv, grad=grad, min_entry=mn,
                                                   info=info).items()}


def _check_logdet_inv(A, s, square, out, kinds, idx):
    """Every problem of a batch A[idx] against numpy: info against the host predicate; for problems with positive pivots,
    slogdet, inv, the gradient, min_entry and h with the tolerances of test_small_gpu.py::test_logdet_inv_vs_numpy.
    Copies of a problem get the same bits wherever they run."""
    d = A.shape[-1]
    B = A * A if square else A
    M = s * np.eye(d) - B
    info = _host_info(M, z_matrix=square | (kinds != 2))
    assert np.array_equal(out["info"], info[idx]), (np.flatnonzero(out["info"] != info[idx]), out["info"][:8])
    first = np.arange(len(idx)) < POOL
    for k in ("logabsdet", "h", "min_entry", "minv", "grad"):
        v = out[k]
        assert np.array_equal(v, v[first][idx], equal_nan=True), k
    ok = info != 1
    Minv = np.linalg.inv(M[ok])
    lad = np.linalg.slogdet(M[ok])[1]
    G = 2 * A[ok] * np.swapaxes(Minv, 1, 2) if square else np.swapaxes(Minv, 1, 2)
    o = {k: v[:POOL][ok] for k, v in out.items()}
    scale = np.maximum(1.0, np.abs(lad))
    rel = lambda x, r: (np.abs(x[:, :, :d] - r).max(axis=(1, 2)) / np.abs(r).max(axis=(1, 2))).max()  # noqa: E731
    err = dict(lad=np.max(np.abs(o["logabsdet"] - lad) / scale),
               h=np.max(np.abs(o["h"] - (-lad + d * np.log(s))) / scale),
               minv=rel(o["minv"], Minv), grad=rel(o["grad"], G),
               min_entry=np.max(np.abs(o["min_entry"] - Minv.min(axis=(1, 2))) / np.abs(Minv).max(axis=(1, 2))))
    assert err["lad"] <= 1e-11 and err["h"] <= 1e-11, err
    assert err["minv"] <= 1e-11 and err["grad"] <= 1e-11, err
    assert err["min_entry"] <= 1e-12, err
    return err, np.bincount(info[idx], minlength=3)


@pytest.mark.parametrize("square", [True, False], ids=["square", "plain"])
@pytest.mark.parametrize("d,s", [(d, 0.9) for d in INV_D] + [(d, s) for d in INV_S_D for s in INV_S])
def test_logdet_inv_batch_vs_numpy(d, s, square):
    """A batch of 5 SMs + 3 mixed problems (every CTA of every path handles at least two: mbarrier phase, pivots and
    identity padding carried over), checked problem by problem; s = 1, 0.5, 2 hit the f == 0.5 case of the
    power-of-two pre-scaling."""
    import torch
    from midagma_b200.linear import logdet_inv
    A, kinds = _inv_problems(d, s, square, seed=1000 * d + int(100 * s) + square)
    idx = np.arange(_inv_batch_size()) % POOL
    o = logdet_inv(torch.as_tensor(A[idx]).cuda(), s=s, square_input=square, want_inv=True, want_grad=True)
    out = {k: v.cpu().numpy() for k, v in o.items()}
    err, counts = _check_logdet_inv(A, s, square, out, kinds, idx)
    print(f"d={d} s={s} square={square}: info counts {counts.tolist()}, " + ", ".join(f"{k} {v:.1e}" for k, v in err.items()))
    assert counts[1] > 0 and counts[0] > 0
    if not square and d > 1:
        assert counts[2] > 0


@pytest.mark.parametrize("d", INV_D)
def test_logdet_inv_strided(d):
    """lda = d + 3, ldo = d + 5 through the C ABI: the same bits as the packed call, the NaN padding of the input is
    never read and that of the outputs never written."""
    import torch
    from midagma_b200.linear import logdet_inv
    idx = np.arange(_inv_batch_size()) % POOL
    for square in (True, False):
        s = 0.8
        A, kinds = _inv_problems(d, s, square, seed=7 * d + square)
        out = _logdet_inv_c(A[idx], s, square, d + 3, d + 5)
        assert np.isnan(out["minv"][:, :, d:]).all() and np.isnan(out["grad"][:, :, d:]).all()
        packed = {k: v.cpu().numpy() for k, v in logdet_inv(torch.as_tensor(A[idx]).cuda(), s=s, square_input=square,
                                                             want_inv=True, want_grad=True).items()}
        for k in ("logabsdet", "h", "min_entry", "info"):
            assert np.array_equal(out[k], packed[k], equal_nan=True), k
        for k in ("minv", "grad"):
            assert np.array_equal(out[k][:, :, :d], packed[k], equal_nan=True), k
        _check_logdet_inv(A, s, square, out, kinds, idx)


def _stochastic_w(d, t, seed):
    """W o W = t P, P dense and row-stochastic (Perron root exactly 1): s I - W o W is a nonsingular M-matrix iff t < s,
    with an entrywise positive inverse that grows like 1 / (s - t)."""
    rng = np.random.default_rng(seed)
    P = rng.random((d, d)) + 0.05
    P /= P.sum(axis=1, keepdims=True)
    return np.sqrt(t * P)


@pytest.mark.parametrize("d", INV_D)
def test_logdet_inv_m_matrix_boundary(d):
    """Perron root of W o W at s (1 - 1e-7): info 0, min_entry > 0 and a residual |M X - I| of the GPU inverse at most
    2x LAPACK's (the bar of the d = 2000 test); at s (1 + 1e-7): flagged."""
    import torch
    from midagma_b200.linear import logdet_inv
    s = 0.8
    W = np.stack([_stochastic_w(d, s * (1 - 1e-7), d), _stochastic_w(d, s * (1 + 1e-7), d)])
    out = logdet_inv(torch.as_tensor(W).cuda(), s=s, square_input=True, want_inv=True, want_grad=True)
    info = out["info"].cpu().numpy()
    assert info[0] == 0 and info[1] != 0, info
    M = s * np.eye(d) - W[0] * W[0]
    Minv = np.linalg.inv(M)
    X = out["minv"][0].cpu().numpy()
    assert Minv.min() > 0 and out["min_entry"][0].item() > 0
    res_gpu, res_ref = np.abs(M @ X - np.eye(d)).max(), np.abs(M @ Minv - np.eye(d)).max()
    lad = np.linalg.slogdet(M)[1]
    print(f"d={d}: max(Minv) {Minv.max():.1e}, residual gpu {res_gpu:.1e} lapack {res_ref:.1e}, "
          f"max-norm rel err {_relmax(X, Minv):.1e}, log|det| {out['logabsdet'][0].item():.10f} / {lad:.10f}")
    # the bar of the d = 2000 test, with a floor of one rounding of the largest entry of |M| |X|: at d = 2 every entry
    # of M X - I is a sum of two rounded products, and which of two correct routes lands closer is rounding luck
    assert res_gpu <= max(2.0 * res_ref, EPS * (np.abs(M) @ np.abs(X)).max())
    # log|det| = sum log(pivots); the last pivot is ~1e-7 s and carries an absolute error of ~cond * eps
    assert abs(out["logabsdet"][0].item() - lad) <= 1e-6


# =====================================================================================================================
# A/B switches: the scalar fallbacks of the fit (DAGMA_SMALL_CFG) and of the inverse (DAGMA_SMALL_INV_DMMA)
# =====================================================================================================================
def _rerun(env, expr):
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-m", "gpu", os.path.abspath(__file__), "-k", expr],
                       env=dict(os.environ, **env), cwd=ROOT, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


@pytest.mark.parametrize("cfg", ["10", "11", "12"])
def test_env_small_cfg(cfg):
    """Sections 1-2 with the scalar rank-1 kernels for 33 <= d <= 64 (C48 up to 48, then C64 / C64B / C64C)."""
    _rerun({"DAGMA_SMALL_CFG": cfg}, "l2_fit_vs_oracle or cold_")


def test_env_small_inv_dmma0():
    """Section 4 with the scalar sweep for 33 <= d <= 128."""
    _rerun({"DAGMA_SMALL_INV_DMMA": "0"}, "logdet_inv")


# =====================================================================================================================
# 5. center_cov and batches beyond 65 535
# =====================================================================================================================
@pytest.mark.parametrize("center", [True, False], ids=["centred", "raw"])
@pytest.mark.parametrize("d", [1, 31, 32, 33, 64, 100])
@pytest.mark.parametrize("n", [1, 5, 31, 32, 33, 1000])
def test_center_cov_vs_numpy(n, d, center):
    """(X - mean)^T (X - mean) / n or X^T X / n against numpy, the in-place centring of X, exact symmetry.  Bound: a
    recursive sum of n products is within n eps sum|x_i x_j| of the exact one, and sum|x_i x_j| / n <= max diag."""
    import torch
    from midagma_b200.linear import center_cov
    rng = np.random.default_rng(n * 1000 + d)
    X = rng.normal(size=(3, n, d)) + rng.normal(size=(3, 1, d)) * 3.0       # non-zero column means
    Xd = torch.as_tensor(X).cuda()
    cov = center_cov(Xd, center=center).cpu().numpy()
    Xg = Xd.cpu().numpy()
    Xc = X - X.mean(axis=1, keepdims=True) if center else X
    ref = np.einsum("bni,bnj->bij", Xc, Xc) / n
    print(f"center_cov n={n} d={d} center={center}: max|dcov| / max|cov| {_relmax(cov, ref):.1e}")
    for b in range(3):
        scale = max(np.abs(ref[b]).max(), np.abs(X[b]).max() ** 2)
        assert np.abs(cov[b] - ref[b]).max() <= 4 * (n + 2) * EPS * scale, b
        assert np.array_equal(cov[b], cov[b].T), b
        assert np.abs(Xg[b] - Xc[b]).max() <= 4 * (n + 2) * EPS * np.abs(X[b]).max(), b
    if not center:
        assert np.array_equal(Xg, X)
    if n == 1 and center:
        assert not cov.any()


def test_batches_beyond_65535():
    """65 541 problems (d = 3, n = 16): center_cov, an l2 fit_batch and a logistic minimize_batch run, and problems
    0, 65 535 and 65 540 are bit for bit what they are alone (the batch is not bounded by a grid dimension)."""
    import torch
    from midagma_b200 import fit_batch, minimize_batch
    from midagma_b200.linear import center_cov
    batch, n, d = 65536 + 5, 16, 3
    picks = [0, 65535, 65540]
    rng = np.random.default_rng(5)
    X = rng.normal(size=(batch, n, d)) + rng.normal(size=(batch, 1, d))
    X[:, :, 1] += 0.8 * X[:, :, 0]
    for center in (True, False):
        Xd = torch.as_tensor(X).cuda()
        cov = center_cov(Xd, center=center).cpu().numpy()
        Xg = Xd.cpu().numpy()
        for b in picks:
            Xa = torch.as_tensor(X[b:b + 1]).cuda()
            assert np.array_equal(center_cov(Xa, center=center).cpu().numpy()[0], cov[b]), (center, b)
            assert np.array_equal(Xa.cpu().numpy()[0], Xg[b]), (center, b)
        Xc = X[picks] - X[picks].mean(axis=1, keepdims=True) if center else X[picks]
        ref = np.einsum("bni,bnj->bij", Xc, Xc) / n
        assert np.abs(cov[picks] - ref).max() <= 1e-13 * np.abs(ref).max()
    kw = dict(T=2, warm_iter=20, max_iter=20, checkpoint=10, s=(1.0, 0.9), return_info=True)
    _, info = fit_batch(X, 0.02, **kw)
    assert (info["status"] == 0).all()
    for b in picks:
        _, one = fit_batch(X[b:b + 1], 0.02, **kw)
        assert np.array_equal(one["W_raw"][0], info["W_raw"][b]) and np.array_equal(one["stage_stats"][0],
                                                                                      info["stage_stats"][b]), b
    Xb = (X > 0.3).astype(np.float64)
    W, ok, st = minimize_batch(np.zeros((batch, d, d)), None, 0.02, 1.0, 20, 1.0, 3e-4, checkpoint=10,
                               loss_type="logistic", X=Xb)
    assert ok.all() and (st[:, 0, 0] == 20).all()
    for b in picks:
        W1, ok1, st1 = minimize_batch(np.zeros((1, d, d)), None, 0.02, 1.0, 20, 1.0, 3e-4, checkpoint=10,
                                      loss_type="logistic", X=Xb[b:b + 1])
        assert np.array_equal(W1[0], W[b]) and np.array_equal(st1[0], st[b]), b
