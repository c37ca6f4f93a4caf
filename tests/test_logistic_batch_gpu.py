"""Batched logistic fits on the one-CTA-per-problem kernel (csrc/small_fit_logistic.cu): ``fit_batch`` /
``minimize_batch`` with ``loss_type="logistic"`` against the reference fixture, the per-problem GPU path
(``DagmaLinear("logistic")``, csrc/lin_iter.cu) and the numpy oracle of src/dagma/linear.py."""
import numpy as np
import pytest

from oracle import simulate
from oracle.linear_ref import OracleLinear

STAGES = ((1.0, 1.0, 130), (0.1, 0.9, 90))        # (mu, s, iterations): two chained minimize calls, checkpoints inside


def _data(d, n, seed):
    if d == 1:                                      # no graph to simulate: random binary data
        return (np.random.default_rng(seed).random((n, 1)) < 0.4).astype(np.float64)
    return simulate.make_linear_problem(d, 2, n, "ER", "logistic", seed)[0]


def _per_problem(X, lam, stages=STAGES, checkpoint=50, lr=3e-4, W0=None, masks=None):
    """Chained ``DagmaLinear("logistic").minimize`` calls: [(W, ok, iterations, checkpoint objectives, final lr)]."""
    from midagma_b200 import DagmaLinear
    m = DagmaLinear("logistic")
    m.fit(X.copy(), lambda1=lam, T=1, warm_iter=0, max_iter=0, checkpoint=checkpoint, **(masks or {}))
    d = X.shape[1]
    W = np.zeros((d, d)) if W0 is None else W0.copy()
    out = []
    for mu, s, iters in stages:
        m.checkpoint_log = []
        W, ok = m.minimize(W.copy(), mu, iters, s, lr=lr)
        out.append((W.copy(), ok, m.last_iters, [row[2] for row in m.checkpoint_log], m._large.last_lr))
    return out


def _batched(Xs, lam, stages=STAGES, checkpoint=50, lr=3e-4, W0=None, masks=None):
    """The same chain through the batched kernel (with its checkpoint log): per stage, per problem
    [(W, ok, iterations, checkpoint objectives, final lr)]."""
    import torch
    from midagma_b200.linear import _run_small, _batch_masks, center_cov
    Xd = torch.as_tensor(np.ascontiguousarray(Xs)).cuda()
    cov = center_cov(Xd, center=False)
    batch, _, d = Xs.shape
    W = torch.zeros(batch, d, d, dtype=torch.float64, device="cuda") if W0 is None else torch.as_tensor(W0).cuda()
    lamd = torch.as_tensor(np.broadcast_to(np.asarray(lam, dtype=np.float64), (batch,)).copy()).cuda()
    exc, inc = _batch_masks(*(masks or {}).get("edges", (None, None)), d, "cuda")
    out = []
    for mu, s, iters in stages:
        res = _run_small(cov, W, lamd, [mu], [s], [iters], lr=lr, tol=1e-6, beta1=0.99, beta2=0.999,
                         checkpoint=checkpoint, retry=False, want_final=False, mask_exc=exc, mask_inc=inc,
                         ckpt_log_cap=iters // checkpoint + 2, X=Xd)
        st, log, cnt = res.stage_stats.cpu().numpy(), res.ckpt_log.cpu().numpy(), res.ckpt_count.cpu().numpy()
        ok = (res.status.cpu().numpy() & 1) == 0
        Wn = W.cpu().numpy()
        out.append([(Wn[b].copy(), bool(ok[b]), int(st[b, 0, 0]), list(log[b, :cnt[b], 2]), float(st[b, 0, 1]))
                    for b in range(batch)])
    return out


@pytest.mark.gpu
def test_reference_fixture_in_a_batch(golden):
    """The stages of the reference-recorded fixture (chained from W = 0), as 8 copies inside a batch of 32."""
    from midagma_b200 import minimize_batch
    g = golden("linear_logistic_d12")
    X = g["X"]
    n, d = X.shape
    Xs = np.stack([X if b % 4 == 0 else _data(d, n, 300 + b) for b in range(32)])
    copies = np.arange(0, 32, 4)
    W = np.zeros((32, d, d))
    for si, (mu, s, iters, lr) in enumerate(g["stages"]):
        W, ok, st = minimize_batch(W, None, float(g["lambda1"]), mu, int(iters), s, lr, checkpoint=int(g["checkpoint"]),
                                   loss_type="logistic", X=Xs)
        ref = g[f"W_after_{si}"]
        for b in copies:
            assert bool(ok[b]) == bool(g[f"ok_{si}"]) and int(st[b, 0, 0]) == int(g[f"iters_{si}"])
            err = np.abs(W[b] - ref).max()
            assert err <= 1e-8, (si, b, err)
            assert abs(st[b, 0, 3] - float(g[f"obj_{si}"])) <= 1e-9 * abs(float(g[f"obj_{si}"]))
            assert np.array_equal(W[b], W[copies[0]])
        print("fixture stage", si, "max|dW| =", np.abs(W[copies[0]] - ref).max())


@pytest.mark.gpu
@pytest.mark.parametrize("d,n", [(1, 40), (5, 40), (12, 300), (20, 500), (33, 1000), (48, 777), (64, 2000)])
def test_matches_per_problem_path(d, n):
    """Two chained stages from W = 0 against DagmaLinear("logistic") (the persistent per-problem kernel)."""
    X = _data(d, n, 100 + d)
    a = _per_problem(X, 0.02)
    b = _batched(X[None], 0.02)
    for (Wa, oka, ita, obja, _), [(Wb, okb, itb, objb, _)] in zip(a, b):
        assert oka == okb and ita == itb
        err = np.abs(Wa - Wb).max()
        print("logistic", d, n, "max|dW| per-problem vs batched =", err)
        assert err <= 1e-11
        assert len(obja) == len(objb) and np.allclose(obja, objb, rtol=1e-11, atol=0)


@pytest.mark.gpu
def test_vs_oracle_generic_start():
    from midagma_b200 import minimize_batch
    d = 30
    X = _data(d, 800, 5)
    W0 = np.random.default_rng(1).normal(size=(d, d)) * 0.05       # a generic start (no exact-tie entries, DESIGN.md 2)
    np.fill_diagonal(W0, 0.0)
    Wg, okg, st = minimize_batch(W0[None].copy(), None, 0.02, 1.0, 100, 1.0, 3e-4, checkpoint=40,
                                 loss_type="logistic", X=X[None])
    o = OracleLinear("logistic").prepare(X.copy(), 0.02, checkpoint=40)
    Wr, okr = o.minimize(W0.copy(), 1.0, 100, 1.0, 3e-4)
    assert bool(okg[0]) == okr and int(st[0, 0, 0]) == o.last_iters
    err = np.abs(Wg[0] - Wr).max()
    print("logistic d=30 vs oracle max|dW| =", err)
    assert err <= 1e-9


@pytest.mark.gpu
def test_full_fits_match_per_problem_fits():
    from midagma_b200 import DagmaLinear, fit_batch
    d, n, batch = 20, 500, 16
    Xs = np.stack([_data(d, n, 1000 + b) for b in range(batch)])
    lam = np.array([0.01, 0.02, 0.03, 0.05] * 4)
    kw = dict(T=3, warm_iter=300, max_iter=500, checkpoint=100)
    W_est, info = fit_batch(Xs, lam, loss_type="logistic", return_info=True, s=(1.0, .9, .8), **kw)
    for b in range(batch):
        m = DagmaLinear("logistic")
        Wb = m.fit(Xs[b].copy(), lambda1=float(lam[b]), s=[1.0, .9, .8], **kw)
        assert info["stage_iters"][b].tolist() == list(m.stage_iters), b
        err = np.abs(info["W_raw"][b] - m.W_raw).max()
        assert err <= 1e-9, (b, err)
        assert np.array_equal(W_est[b] != 0, Wb != 0), b
        assert abs(info["h_final"][b] - m.h_final) <= 1e-9 * max(abs(m.h_final), 1e-12), b
        assert abs(info["score_final"][b] - m.score_final) <= 1e-9 * abs(m.score_final), b


@pytest.mark.gpu
def test_backtracking_and_infeasible_start():
    """lr = 1: the inverse turns infeasible, lr is halved and the step re-taken (linear.py:230-241), as on the
    per-problem path; an infeasible start leaves W untouched and reports failure."""
    from midagma_b200 import minimize_batch
    d = 12
    X = _data(d, 300, 4)
    stages = ((1.0, 1.0, 30),)
    [(Wa, oka, ita, _, lra)] = _per_problem(X, 0.0, stages=stages, checkpoint=20, lr=1.0)
    [[(Wb, okb, itb, _, lrb)]] = _batched(X[None], 0.0, stages=stages, checkpoint=20, lr=1.0)
    assert oka == okb and ita == itb and lra == lrb and lra < 1.0
    assert np.abs(Wa - Wb).max() <= 1e-9
    W0 = np.zeros((1, d, d))
    W0[0, 0, 1] = W0[0, 1, 0] = 1.5
    W1, ok, _ = minimize_batch(W0.copy(), None, 0.02, 1.0, 10, 1.0, 3e-4, loss_type="logistic", X=X[None])
    assert not ok[0] and np.array_equal(W1, W0)


@pytest.mark.gpu
def test_stage_retry():
    """A stage at s = 0.3 goes out of domain and is retried with lr / 2, s + 0.1 (linear.py:446-451)."""
    from midagma_b200 import DagmaLinear, fit_batch
    d = 10
    X = _data(d, 300, 4)
    kw = dict(lambda1=0.01, T=2, warm_iter=300, max_iter=300, lr=0.05, checkpoint=100)
    o = OracleLinear("logistic")
    o.fit(X.copy(), s=[1.0, 0.3], **kw)
    fails = [e for e in o.events if e[0] == "out_of_domain"]
    assert fails, "test input must exercise the retry path"
    s_list = [1.0, 0.3]
    m = DagmaLinear("logistic")
    m.fit(X.copy(), s=s_list, **kw)
    lam = kw.pop("lambda1")
    _, info = fit_batch(X[None], lam, s=(1.0, 0.3), loss_type="logistic", return_info=True, **kw)
    retries = info["stage_stats"][0, :, 6]
    print("retries oracle", len(fails), "batched", retries, "per-problem s", s_list)
    assert int(retries.sum()) == len(fails)
    assert abs(info["stage_stats"][0, 1, 2] - s_list[1]) < 1e-12
    assert info["stage_iters"][0].tolist() == list(m.stage_iters)
    assert np.abs(info["W_raw"][0] - m.W_raw).max() <= 1e-9


@pytest.mark.gpu
def test_masks():
    d = 40
    X = _data(d, 600, 7)
    exc, inc = ((0, 1), (5, 2), (d - 1, 0)), ((3, 4), (1, d - 2))
    a = _per_problem(X, 0.05, masks=dict(exclude_edges=exc, include_edges=inc))
    b = _batched(X[None], 0.05, masks={"edges": (exc, inc)})
    for (Wa, *_), [(Wb, *_)] in zip(a, b):
        assert np.abs(Wa - Wb).max() <= 1e-11
        assert Wb[0, 1] == 0.0 and Wb[5, 2] == 0.0 and Wb[d - 1, 0] == 0.0


@pytest.mark.gpu
def test_scheduling_independence():
    """Three times the resident CTAs, problems of unequal lengths: each problem gets bit for bit the W it gets alone."""
    from midagma_b200 import minimize_batch
    from midagma_b200.linear import _resident_ctas
    d, n = 8, 96
    batch = 3 * _resident_ctas()
    rng = np.random.default_rng(11)
    Xs = (rng.random((batch, n, d)) < rng.uniform(0.2, 0.6, size=(batch, 1, d))).astype(np.float64)
    lam = rng.uniform(0.005, 0.1, size=batch)
    W, ok, st = minimize_batch(np.zeros((batch, d, d)), None, lam, 1.0, 600, 1.0, 3e-3, checkpoint=50,
                               loss_type="logistic", X=Xs)
    iters = st[:, 0, 0]
    assert len(np.unique(iters)) > 1, "problems must have unequal lengths"
    for b in [0, 1, batch // 2, batch - 1, int(np.argmin(iters)), int(np.argmax(iters))]:
        W1, ok1, st1 = minimize_batch(np.zeros((1, d, d)), None, lam[b:b + 1], 1.0, 600, 1.0, 3e-3, checkpoint=50,
                                      loss_type="logistic", X=Xs[b:b + 1])
        assert np.array_equal(W1[0], W[b]) and st1[0, 0, 0] == iters[b], b


@pytest.mark.gpu
def test_mid_d_logistic_batch_runs_side_by_side(monkeypatch):
    """d = 72 > 64: one DagmaLinear("logistic") per problem, several at once -- bit for bit the sequential result."""
    from midagma_b200 import fit_batch
    from midagma_b200.linear import _batch_lanes
    d, n, batch = 72, 300, 4
    Xs = np.stack([_data(d, n, 60 + p) for p in range(batch)])
    lam = np.linspace(0.01, 0.05, batch)
    kw = dict(T=2, warm_iter=200, max_iter=300, checkpoint=100, s=(1.0, .9), return_info=True, loss_type="logistic")
    monkeypatch.delenv("DAGMA_BATCH_LANES", raising=False)
    assert _batch_lanes(d, batch, n) > 1
    _, par = fit_batch(Xs, lam, **kw)
    monkeypatch.setenv("DAGMA_BATCH_LANES", "1")
    _, seq = fit_batch(Xs, lam, **kw)
    assert np.array_equal(par["W_raw"], seq["W_raw"])
    assert par["stage_iters"].tolist() == seq["stage_iters"].tolist()
    assert np.array_equal(par["h_final"], seq["h_final"])


@pytest.mark.gpu
def test_sharded_wrapper_passes_the_loss():
    from midagma_b200 import fit_batch
    from midagma_b200.parallel import fit_batch_sharded
    d, n = 12, 300
    Xs = np.stack([_data(d, n, 500 + p) for p in range(6)])
    kw = dict(T=2, warm_iter=200, max_iter=300, checkpoint=100, s=(1.0, .9), loss_type="logistic")
    assert np.array_equal(fit_batch_sharded(Xs, 0.02, **kw), fit_batch(Xs, 0.02, **kw))


def test_argument_checks_without_a_device():
    from midagma_b200 import _lib, fit_batch, minimize_batch
    cov = np.eye(4)[None]
    X = np.zeros((1, 10, 4))
    with pytest.raises(ValueError):
        fit_batch(cov=cov, loss_type="logistic")
    with pytest.raises(ValueError):
        fit_batch(X, 0.02, cov=cov, loss_type="logistic")
    with pytest.raises(ValueError):
        fit_batch(X, 0.02, loss_type="poisson")
    with pytest.raises(ValueError):
        minimize_batch(np.zeros((1, 4, 4)), cov, 0.02, 1.0, 10, 1.0, 3e-4, loss_type="logistic")
    with pytest.raises(ValueError):
        minimize_batch(np.zeros((1, 4, 4)), cov, 0.02, 1.0, 10, 1.0, 3e-4, loss_type="poisson")
    with pytest.raises(ValueError):
        fit_batch(X[0], 0.02, loss_type="logistic")           # X must be [batch, n, d]
    import os
    header = open(os.path.join(os.path.dirname(__file__), "..", "include", "dagma_b200.h")).read()
    assert "dagma_linear_fit_small_logistic_f64" in header
    assert "dagma_linear_fit_small_logistic_f64" in _lib.EXPORTS
