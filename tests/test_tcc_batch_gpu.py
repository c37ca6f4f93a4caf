"""Batched spectral-TCC fits on the one-CTA-per-problem kernel (csrc/small_fit_pst.cu, the TCC instantiation) against
the reference's recorded trajectory, the per-problem ``DagmaLinear(trek_reg=...)`` (launch sequence + PerronSolver),
and solo runs of the same problems."""
import numpy as np
import pytest
import torch

from oracle import simulate
from oracle.linear_ref import OracleLinear

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps


def _tcc(pairs, weight=0.5, mode="opt", **kw):
    from midagma_b200.notreks import TCCRegularizer
    return TCCRegularizer(I=np.asarray(pairs, dtype=np.int64).reshape(-1, 2), weight=weight, mode=mode, **kw)


@pytest.fixture
def on_chip_only(monkeypatch):
    """The batched entry points must not fall back to the per-problem route."""
    from midagma_b200 import linear

    def refuse(*a, **k):
        raise AssertionError("TCC batch went to the per-problem route")
    monkeypatch.setattr(linear, "_minimize_batch_large", refuse)
    monkeypatch.setattr(linear, "_fit_batch_large", refuse)


def _run(cov, W0, lam, regs, mus, ss, iters, *, lr=3e-4, tol=1e-6, checkpoint=40, retry=False, masks=(None, None)):
    """``_run_small`` with the TCC inputs of ``regs`` (one per problem) and its checkpoint log, on host arrays:
    (W, status, stage_stats, [per problem: checkpoint rows (stage, iter, obj, score, h, lr)], perron_steps)."""
    from midagma_b200.linear import _batch_masks, _TccBatch, _run_small, _tcc_dev, _trek_batch
    batch, d, _ = cov.shape
    _, plan = _trek_batch(regs, batch, d, "l2", "test")
    assert isinstance(plan, _TccBatch)
    tcc = _tcc_dev(plan, "cuda")
    covd = torch.as_tensor(np.ascontiguousarray(cov)).cuda()
    Wd = torch.as_tensor(np.ascontiguousarray(W0, dtype=np.float64)).cuda()
    lamd = torch.as_tensor(np.broadcast_to(np.asarray(lam, dtype=np.float64), (batch,)).copy()).cuda()
    exc, inc = _batch_masks(*masks, d, "cuda")
    cap = sum(int(k) // checkpoint + 2 for k in iters) * (8 if retry else 1)
    res = _run_small(covd, Wd, lamd, list(mus), list(ss), [int(k) for k in iters], lr=lr, tol=tol, beta1=0.99,
                     beta2=0.999, checkpoint=checkpoint, retry=retry, want_final=False, mask_exc=exc, mask_inc=inc,
                     ckpt_log_cap=cap, tcc=tcc)
    log, cnt = res.ckpt_log.cpu().numpy(), res.ckpt_count.cpu().numpy()
    return (Wd.cpu().numpy(), res.status.cpu().numpy(), res.stage_stats.cpu().numpy(),
            [log[b, :cnt[b]] for b in range(batch)], tcc.perron_steps.cpu().numpy())


def _per_problem(cov, W0, lam, reg, mu, iters, s, *, lr=3e-4, tol=1e-6, checkpoint=40, masks=(None, None)):
    """``DagmaLinear("l2", trek_reg=reg).minimize`` on one problem: (W, ok, iterations, checkpoint rows)."""
    from midagma_b200 import DagmaLinear
    m = DagmaLinear("l2", trek_reg=reg)
    m._fit_from_cov(torch.as_tensor(np.ascontiguousarray(cov)).cuda(), float(lam), T=1, warm_iter=0, max_iter=0,
                    checkpoint=checkpoint, exclude_edges=masks[0], include_edges=masks[1])
    m.checkpoint_log = []
    W, ok = m.minimize(np.array(W0, dtype=np.float64), mu, int(iters), s, lr=lr, tol=tol)
    return W, ok, m.last_iters, np.array(m.checkpoint_log, dtype=np.float64).reshape(-1, 6)


def _relmax(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1.0))


def _check(W, status, st, log, ref, what):
    """One problem against the per-problem class: ok, iterations, W, every checkpoint's obj / score / h."""
    W_ref, ok_ref, it_ref, log_ref = ref
    d = W.shape[-1]
    assert ((status & 1) == 0) == ok_ref, what
    assert int(st[0]) == it_ref, (what, st[0], it_ref)
    err = _relmax(W, W_ref)
    assert err <= 1e-9, (what, err)
    assert len(log) == len(log_ref) and np.array_equal(log[:, 1], log_ref[:, 1]), (what, log[:, 1], log_ref[:, 1])
    for col in (2, 3, 4):
        floor = 4 * d * EPS if col == 4 else 0.0          # h near W = 0: a sum of d logs of pivots (absolute round-off)
        tol = 1e-9 * np.abs(log_ref[:, col]) + floor
        assert np.all(np.abs(log[:, col] - log_ref[:, col]) <= tol), (what, col, log[:, col], log_ref[:, col])
    return err


def _generic_start(d, seed, t=0.3):
    rng = np.random.default_rng(seed)
    P = rng.random((d, d))
    P /= P.sum(axis=1, keepdims=True)
    return np.sqrt(t * P) * rng.choice([-1.0, 1.0], size=(d, d))


def _pairs(d, seed, frac=0.15):
    """Random pairs with a duplicate, a reversed pair, a diagonal entry and a negative index."""
    rng = np.random.default_rng(seed)
    allp = [(i, j) for i in range(d) for j in range(d) if i != j] or [(0, 0)]
    k = max(1, int(frac * d * d))
    p = [allp[i] for i in rng.choice(len(allp), size=min(k, len(allp)), replace=False)]
    p += [p[0], (p[-1][1], p[-1][0]), (d // 2, d // 2), (-1, 0)]
    return np.array(p, dtype=np.int64)


def _cov(d, seed, n=200):
    X, _ = simulate.make_linear_problem(d, 2, n, "ER", "gauss", seed) if d > 1 else (
        np.random.default_rng(seed).normal(size=(n, 1)), None)
    X = X - X.mean(axis=0, keepdims=True)
    return X.T @ X / n


def no_trek_pairs(B):
    """(i, j), i < j, with no trek in the DAG B: no node reaches both (a node reaches itself)."""
    d = B.shape[0]
    R = np.eye(d, dtype=bool) | (B != 0)
    for _ in range(d):
        R = R | ((R.astype(np.int64) @ R.astype(np.int64)) > 0)
    trek = (R.T.astype(np.int64) @ R.astype(np.int64)) > 0
    return np.array([(i, j) for i in range(d) for j in range(i + 1, d) if not trek[i, j]], dtype=np.int64).reshape(-1, 2)


# =====================================================================================================================
# 1. the reference's recorded TCC trajectory, inside a batch
# =====================================================================================================================
def test_reference_tcc_in_batch(golden, on_chip_only):
    """The two chained minimize stages of tests/golden/tcc_spectral.npz (TCC weight 0.5, w 0.7, n_iter 10, the
    reference's dispatch: approx_trek_graph / eig, lambda1 0.02, checkpoint 100) from W = 0, as three copies inside a
    batch of 11 TCC problems with their own pairs, weights and w: W within 1e-8 of the reference, the recorded ok."""
    from midagma_b200 import minimize_batch
    g = golden("tcc_spectral")
    X = g["fit_X"]
    d = X.shape[1]
    cov_fix = OracleLinear("l2").prepare(X.copy(), 0.02).cov
    batch, where = 11, (0, 5, 10)
    covs, regs = [], []
    for b in range(batch):
        if b in where:
            covs.append(cov_fix)
            regs.append(_tcc(g["pairs"], weight=0.5, w=0.7, n_iter=10))
        else:
            covs.append(_cov(d, 300 + b))
            regs.append(_tcc(_pairs(d, b), weight=0.1 * b, w=0.3 + 0.1 * b))
    W = np.zeros((batch, d, d))
    for si, (mu, iters, s, lr) in enumerate(g["stages"]):
        W, ok, _ = minimize_batch(W, np.stack(covs), 0.02, mu, int(iters), s, lr, checkpoint=100, trek_reg=regs)
        for b in where:
            assert bool(ok[b]) == bool(g["fit_ok"][si])
            err = np.abs(W[b] - g["fit_W"][si]).max()
            assert err <= 1e-8, (si, b, err)


# =====================================================================================================================
# 2. against the per-problem class, every version / method the kernel takes
# =====================================================================================================================
@pytest.mark.parametrize("d", [1, 5, 12, 33, 64])
@pytest.mark.parametrize("version,method", [("approx_trek_graph", "eig_numpy"), ("DAG_learning", "eig_numpy"),
                                            ("approx_trek_graph", "power"), ("DAG_learning", "power")])
def test_against_per_problem_class(d, version, method, monkeypatch):
    """Three problems with their own pairs, weight, w, eps (and n_iter for power) from a generic start, 120 iterations
    with checkpoints every 40: iterations, ok, W (1e-9 relative) and every checkpoint's obj / score / h match
    ``DagmaLinear("l2", trek_reg=reg).minimize``.  Anything but the reference's dispatch goes through the forward
    flag."""
    from midagma_b200 import notreks
    monkeypatch.setattr(notreks, "FORWARD_TCC_CONFIG", (version, method) != ("approx_trek_graph", "eig_numpy"))
    batch = 3
    regs = [_tcc(_pairs(d, 10 * d + b), weight=(0.2, 0.5, 1.0)[b], w=(1.0, 0.7, 0.4)[b], eps=(1e-12, 1e-10, 1e-8)[b],
                 n_iter=(10, 4, 25)[b], version=version, method=method) for b in range(batch)]
    cov = np.stack([_cov(d, 50 * d + b) for b in range(batch)])
    W0 = np.stack([_generic_start(d, 7 * d + b) for b in range(batch)])
    W, status, st, logs, steps = _run(cov, W0, 0.02, regs, [1.0], [1.0], [120], checkpoint=40)
    assert np.all(steps > 0)
    for b in range(batch):
        ref = _per_problem(cov[b], W0[b], 0.02, regs[b], 1.0, 120, 1.0, checkpoint=40)
        _check(W[b], int(status[b]), st[b, 0], logs[b], ref, (d, version, method, b))


# =====================================================================================================================
# 3. the nilpotent start
# =====================================================================================================================
@pytest.mark.parametrize("d", [4, 12])
def test_nilpotent_start_matches_per_problem_class(d):
    """W = 0 with strictly upper-triangular pairs: the block matrix is nilpotent, so the first solves take the
    rho0 <= 1e-200 branch (d = 4: A^8 = 0) or run into the chunk cap (d = 12: long chains); the batch follows the
    per-problem class through both."""
    pairs = np.array([(i, j) for i in range(d) for j in range(i + 1, d)], dtype=np.int64)
    regs = [_tcc(pairs, weight=0.3, w=0.5), _tcc(pairs[::2], weight=0.6, w=1.0)]
    cov = np.stack([_cov(d, 900 + b) for b in range(2)])
    W0 = np.zeros((2, d, d))
    W, status, st, logs, steps = _run(cov, W0, 0.02, regs, [1.0], [1.0], [30], checkpoint=10)
    for b in range(2):
        ref = _per_problem(cov[b], W0[b], 0.02, regs[b], 1.0, 30, 1.0, checkpoint=10)
        _check(W[b], int(status[b]), st[b, 0], logs[b], ref, ("nilpotent", d, b))


# =====================================================================================================================
# 4. scheduling independence
# =====================================================================================================================
def test_problem_gives_the_same_bits_alone_and_in_any_batch():
    """A problem alone and at several positions of shuffled batches (two stages, retries on, s = 0.5 so stages retry):
    bit-identical W, stage statistics, checkpoint log and power-step count."""
    d = 12
    rng = np.random.default_rng(5)
    probe_reg = _tcc(_pairs(d, 77), weight=0.8, w=0.6)
    probe_cov, probe_W = _cov(d, 77), _generic_start(d, 77, t=0.6)
    kw = dict(mus=[1.0, 0.1], ss=[0.5, 0.9], iters=[80, 80], checkpoint=20, retry=True, lr=1e-2)
    alone = _run(probe_cov[None], probe_W[None], 0.02, [probe_reg], **kw)
    for trial in range(3):
        batch = 9
        pos = int(rng.integers(batch))
        regs = [_tcc(_pairs(d, 100 + trial * 10 + b), weight=0.1 + 0.1 * b, w=0.5) for b in range(batch)]
        cov = np.stack([_cov(d, 500 + trial * 10 + b) for b in range(batch)])
        W0 = np.stack([_generic_start(d, 600 + trial * 10 + b, t=0.6) for b in range(batch)])
        regs[pos], cov[pos], W0[pos] = probe_reg, probe_cov, probe_W
        res = _run(cov, W0, 0.02, regs, **kw)
        assert np.array_equal(res[0][pos], alone[0][0]), trial
        assert res[1][pos] == alone[1][0]
        assert np.array_equal(res[2][pos], alone[2][0])
        assert np.array_equal(res[3][pos], alone[3][0])
        assert res[4][pos] == alone[4][0]


# =====================================================================================================================
# 5. full fits
# =====================================================================================================================
def test_fit_batch_against_per_problem_fit(on_chip_only):
    """fit_batch(trek_reg=[...]) of 16 problems, T = 3 short stages, the no-trek pairs of each true graph, one None and
    one mode-"log" entry: stage iterations, W_raw (1e-9) and the support match ``DagmaLinear(...).fit``."""
    from midagma_b200 import DagmaLinear, fit_batch
    batch, d, n = 16, 10, 300
    Xs, regs = [], []
    for b in range(batch):
        X, B = simulate.make_linear_problem(d, 2, n, "ER", "gauss", 4000 + b)
        Xs.append(X)
        regs.append(_tcc(no_trek_pairs(B), weight=0.2 + 0.05 * b, w=0.7))
    regs[3] = None
    regs[7] = _tcc(regs[6].cfg["I"], mode="log")
    Xs = np.stack(Xs)
    kw = dict(lambda1=0.02, T=3, warm_iter=300, max_iter=400, checkpoint=100)
    W_est, info = fit_batch(Xs.copy(), return_info=True, trek_reg=regs, **kw)
    # a problem solves Perron pairs iff its term changes W (a true graph may have no no-trek pair at all)
    active = [r is not None and r.mode == "opt" and len(r.cfg["I"]) > 0 for r in regs]
    assert info["perron_steps"].shape == (batch,) and ((info["perron_steps"] > 0) == active).all()
    assert not active[3] and not active[7] and sum(active) >= 8
    for b in range(batch):
        m = DagmaLinear("l2", trek_reg=regs[b])
        W_ref = m.fit(Xs[b].copy(), **kw)
        assert list(info["stage_iters"][b]) == list(m.stage_iters), b
        err = _relmax(info["W_raw"][b], m.W_raw)
        assert err <= 1e-9, (b, err)
        assert np.array_equal(W_est[b] != 0, W_ref != 0), b


# =====================================================================================================================
# 6. masks and an infeasible start
# =====================================================================================================================
def test_masks_and_infeasible_start():
    """Exclude / include masks, and a start outside the M-matrix domain (W o W with spectral radius > s): W, status
    bits and iterations match the per-problem class."""
    d = 8
    masks = (((0, 1), (2, 3), (7, 7)), ((4, 5), (1, 0)))
    regs = [_tcc(_pairs(d, 31), weight=0.5, w=0.8), _tcc(_pairs(d, 32), weight=0.3, w=1.0)]
    cov = np.stack([_cov(d, 33), _cov(d, 34)])
    W0 = np.stack([_generic_start(d, 35), _generic_start(d, 36, t=3.0)])
    W, status, st, logs, _ = _run(cov, W0, 0.02, regs, [1.0], [1.0], [100], checkpoint=25, masks=masks)
    assert status[1] & 1                                     # the infeasible start is out of domain, as in the reference
    for b in range(2):
        ref = _per_problem(cov[b], W0[b], 0.02, regs[b], 1.0, 100, 1.0, checkpoint=25, masks=masks)
        _check(W[b], int(status[b]), st[b, 0], logs[b], ref, ("masks", b))
