"""Batched PST ``seq="exp"`` fits on the one-CTA-per-problem kernel (csrc/small_fit_pst.cu, the exp instantiation)
against the reference's recorded trajectory, the float64 oracle with the PST exp term added, solo runs of the same
problems, and the per-problem ``DagmaLinear`` on the reference's own smoke configuration."""
import numpy as np
import pytest
import torch

from oracle import notreks_ref, simulate
from oracle.linear_ref import OracleLinear

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps


class TrekOracle(OracleLinear):
    """``OracleLinear`` with the PST ``exp`` term of linear.py:251-258 / 122-133: ``weight * grad`` joins Gobj before the
    Adam step, ``weight * value`` joins the checkpoint objective.  ``minimize`` updates its ``W`` in place, so the W the
    gradient is taken at is the array the call was given."""

    def __init__(self, pairs, weight, agg):
        super().__init__("l2")
        self.tk = (np.asarray(pairs, dtype=np.int64).reshape(-1, 2), float(weight), agg)

    def minimize(self, W, *a, **k):
        self._W = W
        return super().minimize(W, *a, **k)

    def adam_update(self, grad, it, b1, b2):
        pairs, w, agg = self.tk
        if len(pairs):
            grad = grad + w * notreks_ref.pst_value_grad(self._W, pairs, seq="exp", agg=agg)[1]
        return super().adam_update(grad, it, b1, b2)

    def func(self, W, mu, s=1.0):
        obj, score, h, _ = super().func(W, mu, s)
        pairs, w, agg = self.tk
        v = notreks_ref.pst_value_grad(W, pairs, seq="exp", agg=agg)[0] if len(pairs) else 0.0
        return obj + w * v, score, h, v


def _pst(pairs, weight, agg="mean", mode="opt", **kw):
    from midagma_b200.notreks import PSTRegularizer
    return PSTRegularizer(I=np.asarray(pairs, dtype=np.int64).reshape(-1, 2), seq="exp", weight=weight, mode=mode,
                          kwargs={"agg": agg, **kw})


@pytest.fixture
def on_chip_only(monkeypatch):
    """The batched entry points must not fall back to the per-problem route."""
    from midagma_b200 import linear

    def refuse(*a, **k):
        raise AssertionError("PST exp batch went to the per-problem route")
    monkeypatch.setattr(linear, "_minimize_batch_large", refuse)
    monkeypatch.setattr(linear, "_fit_batch_large", refuse)


def _run(cov, W0, lam, regs, mus, ss, iters, *, lr=3e-4, tol=1e-6, checkpoint=40, retry=False, masks=(None, None)):
    """``_run_small`` with the PST inputs of ``regs`` (one per problem) and its checkpoint log, on host arrays:
    (W, status, stage_stats, [per problem: checkpoint rows (stage, iter, obj, score, h, lr)])."""
    from midagma_b200.linear import _batch_masks, _pst_dev, _run_small, _trek_batch
    batch, d, _ = cov.shape
    _, onchip = _trek_batch(regs, batch, d, "l2", "test")
    assert onchip is not None and onchip[4] is None
    covd = torch.as_tensor(np.ascontiguousarray(cov)).cuda()
    Wd = torch.as_tensor(np.ascontiguousarray(W0, dtype=np.float64)).cuda()
    lamd = torch.as_tensor(np.broadcast_to(np.asarray(lam, dtype=np.float64), (batch,)).copy()).cuda()
    exc, inc = _batch_masks(*masks, d, "cuda")
    cap = sum(int(k) // checkpoint + 2 for k in iters) * (8 if retry else 1)
    res = _run_small(covd, Wd, lamd, list(mus), list(ss), [int(k) for k in iters], lr=lr, tol=tol, beta1=0.99,
                     beta2=0.999, checkpoint=checkpoint, retry=retry, want_final=False, mask_exc=exc, mask_inc=inc,
                     ckpt_log_cap=cap, pst=_pst_dev(onchip, "cuda"))
    log, cnt = res.ckpt_log.cpu().numpy(), res.ckpt_count.cpu().numpy()
    return (Wd.cpu().numpy(), res.status.cpu().numpy(), res.stage_stats.cpu().numpy(),
            [log[b, :cnt[b]] for b in range(batch)])


def _relmax(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1.0))


def _check(o, W_ref, ok_ref, W, status, st, log, what):
    """One problem, one stage, against the oracle's minimize call: ok, iterations, W, every checkpoint's obj/score/h."""
    d = W.shape[-1]
    assert ((status & 1) == 0) == ok_ref, what
    assert int(st[0]) == o.last_iters, (what, st[0], o.last_iters)
    err = _relmax(W, W_ref)
    assert err <= 1e-9, (what, err)
    ref = np.array(o.checkpoints)
    assert len(log) == len(ref) and np.array_equal(log[:, 1], ref[:, 0]), (what, log[:, 1], ref[:, 0])
    for col in (2, 3, 4):
        floor = 4 * d * EPS if col == 4 else 0.0          # h near W = 0: a sum of d logs of pivots (absolute round-off)
        tol = 1e-9 * np.abs(ref[:, col - 1]) + floor
        assert np.all(np.abs(log[:, col] - ref[:, col - 1]) <= tol), (what, col, log[:, col], ref[:, col - 1])
    return err


def _generic_start(d, seed, t=0.3):
    rng = np.random.default_rng(seed)
    P = rng.random((d, d))
    P /= P.sum(axis=1, keepdims=True)
    return np.sqrt(t * P) * rng.choice([-1.0, 1.0], size=(d, d))


def _pairs(d, seed, frac=0.2):
    rng = np.random.default_rng(seed)
    allp = [(i, j) for i in range(d) for j in range(d)]
    k = max(1, int(frac * d * d))
    p = [allp[i] for i in rng.choice(len(allp), size=k, replace=False)]
    p += [p[0]] + [(p[-1][1], p[-1][0])]                  # a duplicate and a reversed pair
    return np.array(p, dtype=np.int64)


def no_trek_pairs(B):
    """(i, j), i < j, with no trek in the DAG B: no node reaches both (a node reaches itself)."""
    d = B.shape[0]
    R = np.eye(d, dtype=bool) | (B != 0)
    for _ in range(d):
        R = R | ((R.astype(np.int64) @ R.astype(np.int64)) > 0)
    trek = (R.T.astype(np.int64) @ R.astype(np.int64)) > 0
    return np.array([(i, j) for i in range(d) for j in range(i + 1, d) if not trek[i, j]], dtype=np.int64).reshape(-1, 2)


# =====================================================================================================================
# 1. the reference's recorded exp trajectory, inside a batch
# =====================================================================================================================
def test_reference_exp_mean_in_batch(golden, on_chip_only):
    """The two chained minimize stages of ``exp_mean`` in tests/golden/pst_series.npz (PST exp / mean, weight 0.7,
    lambda1 0.02, checkpoint 100) from W = 0, as three copies inside a batch of 33 exp problems with their own pairs and
    weights: W within 1e-9 of the reference, same ok flags."""
    from midagma_b200 import minimize_batch
    g = golden("pst_series")
    pairs = g["pairs"]
    X = g["exp_mean_X"]
    d = X.shape[1]
    cov_fix = OracleLinear("l2").prepare(X.copy(), 0.02).cov
    batch, where = 33, (0, 16, 32)
    covs, regs = [], []
    for b in range(batch):
        if b in where:
            covs.append(cov_fix)
            regs.append(_pst(pairs, 0.7))
        else:
            Xo, _ = simulate.make_linear_problem(d, 2, 200, "ER", "gauss", 100 + b)
            covs.append(OracleLinear("l2").prepare(Xo, 0.02).cov)
            regs.append(None if b % 7 == 3 else _pst(_pairs(d, b), 0.05 * (b % 5)))
    W = np.zeros((batch, d, d))
    for si, (mu, iters, s, lr) in enumerate(g["stages"]):
        W, ok, _ = minimize_batch(W, np.stack(covs), 0.02, float(mu), int(iters), float(s), float(lr), checkpoint=100,
                                  trek_reg=regs)
        for b in where:
            assert bool(ok[b]) == bool(g["exp_mean_ok"][si])
            assert np.abs(W[b] - g["exp_mean_W"][si]).max() <= 1e-9, (si, b, np.abs(W[b] - g["exp_mean_W"][si]).max())


# =====================================================================================================================
# 2. the oracle at every size, every aggregation
# =====================================================================================================================
ORACLE_D = [1, 2, 12, 31, 32, 33, 48, 63, 64]


@pytest.mark.parametrize("agg", ["mean", "sum", "max", "lse"])
@pytest.mark.parametrize("d", ORACLE_D)
def test_vs_oracle(d, agg):
    """From a generic start and from W = 0 (two problems of one batch): a first stage that runs all its iterations and
    a chained second one that stops on the tolerance test.  W within 1e-9, iteration counts equal, every checkpoint's
    objective (with the trek term), score and h within 1e-9 relative.  ``max`` from W = 0 gets one pair, its duplicate
    and its reverse, as in the inv tests: round-off alone would otherwise pick among pair values equal in exact
    arithmetic."""
    X, _ = simulate.make_linear_problem(d, 2, 200, "ER", "gauss", 300 + d)
    lam, w = 0.03, {"mean": 0.5, "sum": 0.02, "max": 0.3, "lse": 0.2}[agg]
    pairs = _pairs(d, 50 + d) if d > 1 else np.array([(0, 0), (0, 0)])
    p1 = pairs if agg != "max" else np.array([pairs[1], pairs[1], pairs[1][::-1]])
    oracles = [TrekOracle(p, w, agg).prepare(X.copy(), lam, checkpoint=40) for p in (pairs, p1)]
    cov = np.stack([oracles[0].cov] * 2)
    W0 = np.stack([_generic_start(d, 900 + d), np.zeros((d, d))])
    regs = [_pst(pairs, w, agg), _pst(p1, w, agg)]
    W1, status, st, log = _run(cov, W0, lam, regs, [1.0], [1.0], [100], tol=0.0)
    # tol 0.999: the first checkpoint, compared with obj_prev = 1e16, cannot pass the test; the second one does
    W2, status2, st2, log2 = _run(cov, W1, lam, regs, [0.1], [0.9], [400], tol=0.999)
    stopped_early = False
    for b, o in enumerate(oracles):
        W_ref, ok_ref = o.minimize(W0[b].copy(), 1.0, 100, 1.0, 3e-4, tol=0.0)
        _check(o, W_ref, ok_ref, W1[b], status[b], st[b, 0], log[b], (d, agg, b, 1))
        W2_ref, ok2_ref = o.minimize(W_ref.copy(), 0.1, 400, 0.9, 3e-4, tol=0.999)
        _check(o, W2_ref, ok2_ref, W2[b], status2[b], st2[b, 0], log2[b], (d, agg, b, 2))
        stopped_early |= o.last_iters < 400
    assert stopped_early, "the second stage must end on the tolerance test"


@pytest.mark.parametrize("d", [12, 33])
def test_max_tie_between_a_pair_and_its_reverse(d):
    """H = F^T F is symmetric, so (i, j) and (j, i) tie exactly for the maximum and share its gradient."""
    X, _ = simulate.make_linear_problem(d, 2, 200, "ER", "gauss", 17)
    pairs = np.array([(0, 1), (1, 0)])
    o = TrekOracle(pairs, 0.4, "max").prepare(X.copy(), 0.02, checkpoint=40)
    W0 = _generic_start(d, 5)
    W_ref, ok_ref = o.minimize(W0.copy(), 1.0, 120, 1.0, 3e-4, tol=0.0)
    W, status, st, log = _run(o.cov[None], W0[None], 0.02, [_pst(pairs, 0.4, "max")], [1.0], [1.0], [120], tol=0.0)
    _check(o, W_ref, ok_ref, W[0], status[0], st[0, 0], log[0], ("tie", d))


# =====================================================================================================================
# 3. back-tracking, infeasible starts, stage retries, masks -- with the trek term active
# =====================================================================================================================
@pytest.mark.parametrize("d,agg", [(16, "lse"), (33, "mean"), (63, "max")])
def test_backtracking(d, agg):
    X, _ = simulate.make_linear_problem(d, 2, 300, "ER", "gauss", 4)
    pairs = _pairs(d, d)
    o = TrekOracle(pairs, 0.5, agg).prepare(X, 0.0, checkpoint=50)
    W_ref, ok_ref = o.minimize(np.zeros((d, d)), 1.0, 40, 1.0, 1.0)
    n_halved = sum(1 for e in o.events if e[0] == "lr_halved")
    assert n_halved > 0, "test input must exercise back-tracking"
    W, status, st, _ = _run(o.cov[None], np.zeros((1, d, d)), 0.0, [_pst(pairs, 0.5, agg)], [1.0], [1.0], [40],
                            lr=1.0, checkpoint=50)
    assert ((status[0] & 1) == 0) == ok_ref
    assert int(st[0, 0, 7]) == n_halved and int(st[0, 0, 0]) == o.last_iters and st[0, 0, 1] == o.last_lr
    assert np.abs(W[0] - W_ref).max() <= 1e-6          # lr = 1: the steps amplify round-off (see test_onchip_sizes_gpu)


@pytest.mark.parametrize("d", [16, 40])
def test_infeasible_start_mid_batch(d):
    X, _ = simulate.make_linear_problem(d, 2, 200, "ER", "gauss", 8)
    cov = OracleLinear("l2").prepare(X, 0.02).cov
    pairs = _pairs(d, 3)
    W0 = np.stack([_generic_start(d, k) for k in range(5)])
    W0[2] *= 4.0                                       # (W o W) row sums 4.8: outside the domain at s = 1
    regs = [_pst(pairs, 0.3, "lse")] * 5
    W, status, st, log = _run(np.stack([cov] * 5), W0, 0.02, regs, [1.0], [1.0], [80])
    assert (status[2] & 1) and int(st[2, 0, 0]) == 0 and np.array_equal(W[2], W0[2])
    for b in (1, 3):
        Ws, ss_, sts, logs = _run(cov[None], W0[b:b + 1], 0.02, regs[:1], [1.0], [1.0], [80])
        assert np.array_equal(W[b], Ws[0]) and np.array_equal(st[b], sts[0]) and np.array_equal(log[b], logs[0])


@pytest.mark.parametrize("d,agg", [(12, "mean"), (33, "lse"), (64, "sum")])
def test_fit_retries_with_masks(d, agg):
    """Two stages under ``fit`` semantics, the second at s = 0.3 so that it restarts with lr / 2 and s + 0.1; include and
    exclude edges next to the trek term: W, stage iterations and retry counts against the oracle's fit."""
    X, W_true = simulate.make_linear_problem(d, 2, 300, "ER", "gauss", 21)
    edges = np.argwhere(W_true != 0)
    inc = ((int(edges[0][0]), int(edges[0][1])),)
    exc = ((int(edges[1][0]), int(edges[1][1])), (0, d - 1))
    pairs = _pairs(d, 9)
    o = TrekOracle(pairs, 0.1, agg)
    o.fit(X.copy(), lambda1=0.02, T=2, warm_iter=200, max_iter=200, checkpoint=50, s=[1.0, 0.3], lr=0.01,
          w_threshold=0.0, exclude_edges=exc, include_edges=inc)
    n_retry = sum(1 for e in o.events if e[0] == "out_of_domain")
    assert n_retry > 0, "test input must retry a stage"
    W, status, st, _ = _run(o.cov[None], np.zeros((1, d, d)), 0.02, [_pst(pairs, 0.1, agg)], [1.0, 0.1], [1.0, 0.3],
                            [200, 200], lr=0.01, checkpoint=50, retry=True, masks=(exc, inc))
    assert [int(x) for x in st[0, :, 0]] == o.stage_iters and int(st[0, :, 6].sum()) == n_retry
    assert _relmax(W[0], o.W_raw) <= 1e-9


# =====================================================================================================================
# 4. scheduling independence
# =====================================================================================================================
def _mixed_pairs(d, b):
    kind = b % 6
    if kind == 0:
        return np.array([(b % d, (3 * b + 1) % d)])                          # m = 1
    if kind == 1:
        return np.array([(0, 1), (0, 1), (1, 0), (2, 5), (0, 1)])            # duplicates
    if kind == 2:
        return np.array([(i, i) for i in range(0, d, 3)])                    # diagonal pairs
    if kind == 3:
        return np.array([(i, j) for i in range(d) for j in range(d)])        # m = d^2
    if kind == 4:
        return np.zeros((0, 2), dtype=np.int64)                              # m = 0
    return _pairs(d, b, 0.1)


@pytest.mark.parametrize("agg", ["mean", "max", "lse"])
def test_scheduling_independence(agg):
    """Three waves of resident CTAs (one per SM) + 7 problems with their own pair sets and weights, unequal lengths and
    stage retries: picked problems are bit for bit what they are alone (W, stage statistics, checkpoint log)."""
    d = 24
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    batch = 3 * sms + 7
    covs = []
    for k in range(9):
        X, _ = simulate.make_linear_problem(d, 2, 150, "ER", "gauss", 600 + k)
        covs.append(OracleLinear("l2").prepare(X, 0.02).cov)
    cov = np.stack([covs[b % 9] for b in range(batch)])
    regs = [_pst(_mixed_pairs(d, b), 0.05 + 0.1 * (b % 4), agg) for b in range(batch)]
    lam = 0.01 + 0.01 * (np.arange(batch) % 3)
    kw = dict(mus=[1.0, 0.1], ss=[1.0, 0.3], iters=[150, 150], lr=0.01, tol=0.03, checkpoint=10, retry=True)
    W, status, st, log = _run(cov, np.zeros((batch, d, d)), lam, regs, **kw)
    assert st[:, 1, 6].max() > 0 and len(np.unique(st[:, :, 0].sum(axis=1))) > 1
    for b in (0, 1, 2, 3, sms + 4, 2 * sms + 5, batch - 1):     # (an m = 0 problem alone has no trek term to batch)
        Ws, ss_, sts, logs = _run(cov[b:b + 1], np.zeros((1, d, d)), lam[b], [regs[b]], **kw)
        assert np.array_equal(W[b], Ws[0]), b
        assert np.array_equal(st[b], sts[0]) and status[b] == ss_[0] and np.array_equal(log[b], logs[0]), b


# =====================================================================================================================
# 5. the reference's smoke configuration: fit_batch against the per-problem class
# =====================================================================================================================
def test_reference_smoke_configuration(on_chip_only):
    """ER d = 20 (20 edges), n = 500, Gaussian noise, ``I`` = the no-trek pairs of each true graph,
    ``PSTRegularizer(seq="exp", weight=0.1)`` and lambda1 = 0.02 as in the reference's ``dagma.linear.test()``, over a
    short schedule: ``fit_batch(trek_reg=[...])`` against ``DagmaLinear("l2", trek_reg=...).fit`` problem by problem --
    equal stage iterations and support, W_raw, h_final and score_final within 1e-9."""
    from midagma_b200 import DagmaLinear, fit_batch
    d, n, batch = 20, 500, 6
    Xs, regs = [], []
    for b in range(batch):
        rng = np.random.default_rng(1 + b)
        B = simulate.simulate_dag(d, d, "ER", rng)
        W_true = simulate.simulate_parameter(B, rng=rng)
        Xs.append(simulate.simulate_linear_sem(W_true, n, "gauss", rng=rng))
        regs.append(_pst(no_trek_pairs(B), 0.1))
    Xs = np.stack(Xs)
    kw = dict(lambda1=0.02, T=3, warm_iter=300, max_iter=500, checkpoint=100)
    W_est, info = fit_batch(Xs.copy(), return_info=True, trek_reg=regs, s=[1.0, 0.9, 0.8], **kw)
    for b in range(batch):
        m = DagmaLinear("l2", trek_reg=regs[b])
        Wb = m.fit(Xs[b].copy(), s=[1.0, 0.9, 0.8], **kw)    # a fresh list: retries add 0.1 to it in place (Q9)
        assert list(info["stage_iters"][b]) == list(m.stage_iters), b
        assert np.array_equal(W_est[b] != 0, Wb != 0), b
        assert np.abs(info["W_raw"][b] - m.W_raw).max() <= 1e-9, b
        assert abs(info["h_final"][b] - m.h_final) <= 1e-9 * max(1.0, abs(m.h_final)), b
        assert abs(info["score_final"][b] - m.score_final) <= 1e-9 * max(1.0, abs(m.score_final)), b
