"""Batched nonlinear fits (nonlinear.fit_batch / minimize_batch on csrc/mlp_batch.cu), built up layer by layer: one
iteration against the launch sequence of _MlpEngine, minimize against DagmaNonlinear.minimize and the oracle, the
reference fixtures inside batches, infeasible starts, scheduling independence, fit against DagmaNonlinear.fit, and the
shapes that run one problem after the other.  The argument checks at the end need no GPU."""
import copy

import numpy as np
import pytest
import torch

from oracle.nonlinear_ref import OracleMLP, OracleNonlinear

gpu = pytest.mark.gpu


def _relmax(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _model(dims, seed, fc1_std=None):
    from midagma_b200.nonlinear import DagmaMLP
    torch.manual_seed(seed)
    model = DagmaMLP(list(dims))
    d = dims[0]
    with torch.no_grad():
        model.fc1.weight.normal_(0.0, fc1_std if fc1_std is not None else 0.4 / np.sqrt(d * dims[1]))
        model.fc1.bias.normal_(0.0, 0.1)
    return model


def _data(batch, n, d, seed):
    g = np.random.default_rng(seed)
    return g.normal(size=(batch, n, d)) * g.uniform(0.5, 2.0, size=(batch, 1, d))


def _theta(model):
    return model.pack().cpu().numpy()


def _fixture_model(g):
    from midagma_b200.nonlinear import DagmaMLP
    model = DagmaMLP([int(x) for x in g["dims"]])
    model.load_state_dict({k[5:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("init.")})
    return model


# ------------------------------------------------------------------------------------------ 1. one iteration
ONE_ITER_SHAPES = [(1, 1, 1), (2, 3, 15), (7, 10, 16), (8, 40, 17), (9, 3, 33), (16, 10, 500), (17, 1, 33),
                   (33, 3, 17), (40, 10, 2000), (63, 1, 15), (64, 40, 16), (64, 3, 500), (9, 40, 1), (8, 5, 2000)]


@gpu
@pytest.mark.parametrize("d,m1,n", ONE_ITER_SHAPES, ids=[f"d{d}-m{m}-n{n}" for d, m, n in ONE_ITER_SHAPES])
def test_one_iteration_vs_engine(d, m1, n):
    """Objective, S, h and one Adam step against _MlpEngine.evaluate + the Adam kernel, at every DMMA edge of d, every
    row-tile edge of n and every slice edge of d * m1 against 40."""
    from midagma_b200.nonlinear import (_MlpBatch, _MlpEngine, F_MU, F_S, F_LR, F_LAM1, F_LAM2, F_B1, F_B2, F_GAMMA,
                                        F_OBJ, F_H, F_SS)
    B = 3
    models = [_model([d, m1, 1], 100 * d + 10 * m1 + b) for b in range(B)]
    X = torch.from_numpy(_data(B, n, d, d * n + m1))
    lam1 = np.array([0.02, 0.05, 0.01])
    bt = _MlpBatch(models, X)
    full = lambda x: np.full(B, x)                              # noqa: E731
    ok, its = bt.run(np.arange(B), 1, full(2e-3), lam1, full(0.005), full(0.1), full(1.0), full(False), 1e-6, 1000)
    assert ok.all() and (its == 1).all()
    st = bt.state.cpu().numpy()
    for b in range(B):
        eng = _MlpEngine(models[b], X[b].cuda())
        sh = eng.state_host
        sh.zero_()
        for f, val in ((F_MU, 0.1), (F_S, 1.0), (F_LR, 2e-3), (F_LAM1, lam1[b]), (F_LAM2, 0.005), (F_B1, 0.99),
                       (F_B2, 0.999), (F_GAMMA, 1.0)):
            sh[f] = float(val)
        eng.state.copy_(sh)
        eng.iteration(1.0)
        ref, _, _ = eng.pull()
        for f in (F_OBJ, F_SS, F_H):
            assert abs(st[b, f] - float(ref[f])) <= 1e-11 * max(abs(float(ref[f])), 1e-3), (b, f, st[b, f], float(ref[f]))
        assert _relmax(bt.theta[b].cpu().numpy(), eng.theta.cpu().numpy()) <= 1e-11, b
        assert _relmax(bt.m[b].cpu().numpy(), eng.m.cpu().numpy()) <= 1e-11, b


# ------------------------------------------------------------------------------------------ 2. minimize
def _solo_minimize(model, X, K, lr, lam1, lam2, mu, s, tol=1e-6, checkpoint=50, lr_decay=False):
    from midagma_b200.nonlinear import DagmaNonlinear, F_OBJ
    eq = DagmaNonlinear(model)
    eq.X, eq.checkpoint = torch.as_tensor(X).cuda(), checkpoint
    ok = eq.minimize(K, lr, lam1, lam2, mu, s, lr_decay, tol)
    return ok, eq.n_iters, float(eq._engine.pull()[0][F_OBJ])


@gpu
@pytest.mark.parametrize("d,m1,n,tol", [(7, 5, 50, 1e-6), (20, 10, 300, 1e-6), (40, 10, 2000, 1e-6), (13, 4, 77, 3e-3)])
def test_minimize_batch_vs_per_problem(d, m1, n, tol):
    """K = 200 iterations, checkpoint = 50: success flags, iteration counts, the objective at every checkpoint (the
    last iteration of a run of 1, 51, 101, 151, 200) and the parameters against DagmaNonlinear.minimize."""
    from midagma_b200.nonlinear import _MlpBatch, F_OBJ
    B = 5
    base = [_model([d, m1, 1], 7 * d + b) for b in range(B)]
    X = _data(B, n, d, 3 * d + n)
    lam1 = np.array([0.02, 0.01, 0.05, 0.0, 0.03])
    for K in (1, 51, 101, 151, 200):
        models = [copy.deepcopy(m) for m in base]
        bt = _MlpBatch(models, torch.from_numpy(X))
        full = lambda x: np.full(B, x)                          # noqa: E731
        ok, its = bt.run(np.arange(B), K, full(2e-3), lam1, full(0.005), full(0.1), full(1.0), full(False), tol, 50)
        bt.write_back()
        objs = bt.state[:, F_OBJ].cpu().numpy()
        for b in range(B):
            ref_model = copy.deepcopy(base[b])
            ok_r, it_r, obj_r = _solo_minimize(ref_model, X[b], K, 2e-3, float(lam1[b]), 0.005, 0.1, 1.0, tol=tol)
            assert bool(ok[b]) == ok_r and int(its[b]) == it_r, (K, b, ok[b], ok_r, its[b], it_r)
            assert abs(objs[b] - obj_r) <= 1e-10 * abs(obj_r), (K, b, objs[b], obj_r)
            assert _relmax(_theta(models[b]), _theta(ref_model)) <= 1e-9, (K, b)


@gpu
@pytest.mark.parametrize("d,m1,n", [(5, 3, 40), (12, 6, 90)])
def test_minimize_batch_vs_oracle(d, m1, n):
    from midagma_b200.nonlinear import minimize_batch
    B = 3
    models = [_model([d, m1, 1], 31 * d + b) for b in range(B)]
    refs = [OracleMLP([d, m1, 1], {k: v.numpy().copy() for k, v in m.state_dict().items()}) for m in models]
    X = _data(B, n, d, 5 * d)
    lam1 = np.array([0.02, 0.04, 0.01])
    ok = minimize_batch(models, X, 200, 2e-3, lam1, 0.005, 0.1, 1.0, checkpoint=50)
    for b in range(B):
        o = OracleNonlinear(refs[b])
        ok_r = o.minimize(X[b], 200, 2e-3, float(lam1[b]), 0.005, 0.1, 1.0, checkpoint=50)
        assert bool(ok[b]) == ok_r
        for k, p in models[b].state_dict().items():
            assert _relmax(p.numpy(), refs[b].p[k].reshape(p.shape)) <= 1e-9, (b, k)


# ------------------------------------------------------------------------------------------ 3. fixtures in a batch
def _fillers(g, count, seed):
    dims = [int(x) for x in g["dims"]]
    X0 = g["X"]
    models = [_model(dims, seed + b) for b in range(count)]
    rng = np.random.default_rng(seed)
    Xs = [X0[rng.permutation(X0.shape[0])] + 0.1 * rng.normal(size=X0.shape) for _ in range(count)]
    return models, Xs


@gpu
@pytest.mark.parametrize("name", ["mlp_d7", "mlp_d40"])
def test_minimize_fixture_inside_batch(golden, name):
    from midagma_b200.nonlinear import minimize_batch
    g = golden(name)
    lambda1, lambda2, mu, s, lr = (float(x) for x in g["hyper"])
    steps = int(g["steps"])
    models, Xs = _fillers(g, 8, 11)
    at = (1, 5)
    for p in at:
        models[p], Xs[p] = _fixture_model(g), g["X"].copy()
    ok = minimize_batch(models, np.stack(Xs), steps, lr, lambda1, lambda2, mu, s, checkpoint=10 ** 9)
    for p in at:
        assert bool(ok[p]) == bool(g["ok"])
        for k, prm in models[p].state_dict().items():
            assert _relmax(prm.numpy(), g[f"after{steps}.{k}"]) <= 1e-9, (p, k)


@gpu
@pytest.mark.parametrize("name", ["mlp_fit_d5", "mlp_fit_retry_d5", "mlp_fit_retry2_d5", "mlp_fit_retry_decay_d5"])
def test_fit_fixture_inside_batch(golden, name):
    from midagma_b200.nonlinear import fit_batch
    g = golden(name)
    T, warm, mx, ck = (int(x) for x in g["kw"])
    lr = float(g["lr"]) if "lr" in g.files else 2e-4
    tol = 1e-8 if name == "mlp_fit_d5" else 1e-6
    models, Xs = _fillers(g, 7, 23)
    at = (0, 3, 6)
    for p in at:
        models[p], Xs[p] = _fixture_model(g), g["X"].copy()
    W, info = fit_batch(models, np.stack(Xs), lambda1=0.02, lambda2=0.005, T=T, warm_iter=warm, max_iter=mx, lr=lr,
                        checkpoint=ck, return_info=True)
    for p in at:
        if "calls" in g.files:
            assert np.array_equal(np.array(info["minimize_calls"][p], dtype=np.float64), g["calls"])
        assert np.abs(info["W_raw"][p] - g["W_raw"]).max() <= tol
        assert np.array_equal(W[p] != 0, g["W_est"] != 0)
        for k, prm in models[p].state_dict().items():
            assert np.abs(prm.numpy() - g["final." + k]).max() <= tol, (p, k)


# ------------------------------------------------------------------------------------------ 4. h < 0 starts
@gpu
def test_infeasible_start_alone_and_mid_batch():
    from midagma_b200.nonlinear import minimize_batch
    d, m1, n = 6, 3, 64
    X = _data(5, n, d, 99)

    def bad():
        m = _model([d, m1, 1], 0)
        with torch.no_grad():
            m.fc1.weight.fill_(0.8)
        return m

    solo = bad()
    before = _theta(solo)
    assert not minimize_batch([solo], X[2:3], 20, 1e-3, 0.02, 0.005, 0.1, 1.0, checkpoint=10)[0]
    assert np.array_equal(_theta(solo), before)
    models = [_model([d, m1, 1], 40 + b) for b in range(5)]
    models[2] = bad()
    alone = [copy.deepcopy(m) for m in models]
    ok = minimize_batch(models, X, 20, 1e-3, 0.02, 0.005, 0.1, 1.0, checkpoint=10)
    assert not ok[2] and np.array_equal(_theta(models[2]), before)
    for b in (0, 1, 3, 4):
        ok_b = minimize_batch([alone[b]], X[b:b + 1], 20, 1e-3, 0.02, 0.005, 0.1, 1.0, checkpoint=10)
        assert ok[b] and ok_b[0]
        assert np.array_equal(_theta(models[b]), _theta(alone[b])), b


# ------------------------------------------------------------------------------------------ 5. scheduling independence
@gpu
def test_scheduling_independence(golden):
    """A batch of 3 x the resident CTAs mixing different lambda1 (unequal lengths), infeasible starts and retries with
    ExponentialLR active: six chosen problems equal their solo runs bit for bit."""
    from midagma_b200.nonlinear import fit_batch
    g = golden("mlp_fit_retry_decay_d5")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = 3 * 2 * sms
    models, Xs = _fillers(g, B, 1000)
    for b in range(B):
        if b % 3 == 0:
            models[b] = _fixture_model(g)
            with torch.no_grad():
                models[b].fc2[0].weight.mul_(1.0 + 0.01 * (b % 17))
        if b % 97 == 5:
            with torch.no_grad():
                models[b].fc1.weight.fill_(0.8)
    X = np.stack(Xs)
    lam1 = 0.005 + 0.03 * np.random.default_rng(5).random(B)
    kw = dict(lambda2=0.005, T=2, warm_iter=150, max_iter=1300, lr=0.05, checkpoint=400, return_info=True)
    start = [copy.deepcopy(m) for m in models]
    _, info = fit_batch(models, X, lambda1=lam1, **kw)
    calls = info["minimize_calls"]
    assert any(c[3] == 1 and c[2] == 1 for cs in calls for c in cs), "no successful retry with ExponentialLR"
    assert any(all(c[2] == 0 for c in cs) for cs in calls), "no infeasible start"
    assert len(set(info["n_iters"].tolist())) > 10, "lengths should differ"
    chosen = [0, 5, 97 + 5, B // 2 + 1, B - 3, B - 1]
    for b in chosen:
        m = start[b]
        _, si = fit_batch([m], X[b:b + 1], lambda1=lam1[b:b + 1], **kw)
        assert np.array_equal(_theta(m), _theta(models[b])), b
        assert si["stage_iters"][0] == info["stage_iters"][b] and si["minimize_calls"][0] == calls[b], b
        assert int(si["n_iters"][0]) == int(info["n_iters"][b])


# ------------------------------------------------------------------------------------------ 6. fit vs the loop
@gpu
def test_fit_batch_vs_loop(golden):
    from midagma_b200.nonlinear import DagmaNonlinear, fit_batch
    g = golden("mlp_fit_retry_d5")
    B = 12
    models, Xs = _fillers(g, B, 500)
    models[4], Xs[4] = _fixture_model(g), g["X"].copy()
    with torch.no_grad():
        models[9].fc1.weight.fill_(0.8)
    lam1 = np.linspace(0.01, 0.04, B)
    loop_models = [copy.deepcopy(m) for m in models]
    kw = dict(lambda2=0.005, T=2, warm_iter=120, max_iter=160, lr=0.05, checkpoint=40)
    W, info = fit_batch(models, np.stack(Xs), lambda1=lam1, return_info=True, **kw)
    assert any(c[2] == 0 for cs in info["minimize_calls"] for c in cs), "no retry"
    # a failed call that took steps before h < 0: stage_iters counts the stage's last call only, n_iters every call
    assert any(sum(info["stage_iters"][b]) < info["n_iters"][b] for b in range(B)), "no failed call with steps"
    for b in range(B):
        eq = DagmaNonlinear(loop_models[b])
        Wl = eq.fit(Xs[b], lambda1=float(lam1[b]), **kw)
        assert info["stage_iters"][b] == eq.stage_iters and info["n_iters"][b] == eq.n_iters, b
        assert info["minimize_calls"][b] == eq.minimize_calls, b
        assert np.abs(info["W_raw"][b] - loop_models[b].fc1_to_adj()).max() <= 1e-8, b
        assert np.array_equal(W[b] != 0, Wl != 0), b
        for k, p in models[b].state_dict().items():
            assert np.abs(p.numpy() - loop_models[b].state_dict()[k].numpy()).max() <= 1e-8, (b, k)


# ------------------------------------------------------------------------------------------ 7. other shapes
@gpu
@pytest.mark.parametrize("dims", [[6, 5, 3, 1], [65, 2, 1], [4, 41, 1], [5, 1]], ids=["deep", "d65", "m41", "d-1"])
def test_unsupported_shapes_run_the_loop(dims):
    from midagma_b200.nonlinear import DagmaMLP, DagmaNonlinear, fit_batch, minimize_batch
    B, n, d = 3, 30, dims[0]
    torch.manual_seed(3)
    models = []
    for b in range(B):
        m = DagmaMLP(list(dims))
        with torch.no_grad():
            m.fc1.weight.normal_(0.0, 0.05)
        models.append(m)
    X = _data(B, n, d, 17)
    ref = [copy.deepcopy(m) for m in models]
    ok = minimize_batch(models, X, 30, 1e-3, 0.02, 0.005, 0.1, 1.0, checkpoint=10)
    for b in range(B):
        eq = DagmaNonlinear(ref[b])
        eq.X, eq.checkpoint = torch.from_numpy(X[b]).cuda(), 10
        assert ok[b] == eq.minimize(30, 1e-3, 0.02, 0.005, 0.1, 1.0)
        assert np.array_equal(_theta(models[b]), _theta(ref[b]))
    W, info = fit_batch(models, X, T=2, warm_iter=20, max_iter=30, checkpoint=10, return_info=True)
    for b in range(B):
        eq = DagmaNonlinear(ref[b])
        Wl = eq.fit(X[b], T=2, warm_iter=20, max_iter=30, checkpoint=10)
        assert np.array_equal(W[b], Wl) and info["minimize_calls"][b] == eq.minimize_calls
        assert np.array_equal(_theta(models[b]), _theta(ref[b]))


# ------------------------------------------------------------------------------------------ argument checks (CPU)
def test_argument_checks():
    from midagma_b200.nonlinear import DagmaMLP, fit_batch, minimize_batch
    a, b = DagmaMLP([4, 3, 1]), DagmaMLP([4, 2, 1])
    X = np.zeros((2, 10, 4))
    with pytest.raises(ValueError, match="same dims"):
        minimize_batch([a, b], X, 10, 1e-3, 0.02, 0.005, 0.1, 1.0)
    with pytest.raises(ValueError, match="non-empty"):
        fit_batch([], X)
    with pytest.raises(ValueError, match=r"\[batch, n, d\]"):
        fit_batch([a, copy.deepcopy(a)], np.zeros((2, 10, 5)))
    with pytest.raises(ValueError, match=r"\[batch, n, d\]"):
        fit_batch([a], X)
    with pytest.raises(ValueError, match="no rows"):
        fit_batch([a, copy.deepcopy(a)], np.zeros((2, 0, 4)))
    with pytest.raises(ValueError, match="lambda1"):
        fit_batch([a, copy.deepcopy(a)], X, lambda1=[0.1, 0.2, 0.3])
    with pytest.raises(ValueError, match="lambda2"):
        minimize_batch([a, copy.deepcopy(a)], X, 10, 1e-3, 0.02, np.zeros((2, 2)), 0.1, 1.0)
    with pytest.raises(ValueError, match="s should be"):
        fit_batch([a, copy.deepcopy(a)], X, s="x")
