"""GPU parity of the DagmaMLP / DagmaNonlinear path against the fixtures recorded from the
reference (torch autograd + torch.optim.Adam) and against the numpy oracle."""
import numpy as np
import pytest
import torch

from oracle import simulate
from oracle.nonlinear_ref import OracleMLP, OracleNonlinear

pytestmark = pytest.mark.gpu


def _relmax(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _checksum(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return np.array([a.sum(), np.abs(a).sum(), (a * a).sum(), a.ravel()[:: max(a.size // 97, 1)].sum()])


def _model_from(g, prefix="init."):
    from midagma_b200.nonlinear import DagmaMLP
    dims = [int(x) for x in g["dims"]]
    model = DagmaMLP(dims=dims, bias=True, dtype=torch.double)
    sd = {k[len(prefix):]: torch.from_numpy(g[k]) for k in g.files if k.startswith(prefix)}
    model.load_state_dict(sd)          # same parameter names and shapes as the reference
    return model


@pytest.mark.parametrize("name", ["mlp_d7", "mlp_d40", "mlp_c3_n2000", "mlp_deep_d6", "mlp_deep4_d5", "mlp_lin_d6"])
def test_mlp_value_grad_steps_vs_reference(golden, name):
    from midagma_b200.nonlinear import DagmaNonlinear, _MlpEngine, F_MU, F_S, F_LAM1, F_LAM2, F_OBJ, F_SCORE, F_H
    g = golden(name)
    lambda1, lambda2, mu, s, lr = (float(x) for x in g["hyper"])
    model = _model_from(g)
    if "X" in g.files:
        X, X_hat_ref = g["X"], g["X_hat"]
    else:
        # at n = 2000 the fixture keeps the seed of X (checksum of the arrays the reference was fed) and a fixed
        # sample of the rows of X_hat
        X, _ = simulate.config_c3(int(g["seed"]), n=int(g["n"]), d=int(g["dims"][0]))
        assert np.allclose(_checksum(X), g["x_checksum"], rtol=1e-13, atol=0), "not the arrays the reference was fed"
        X_hat_ref = None
    rows = g["X_hat_rows"] if "X_hat_rows" in g.files else slice(None)
    # public surface: forward, h_func, l1, adjacency
    X_hat = model.forward(torch.from_numpy(X))
    assert _relmax(X_hat.numpy()[rows], g["X_hat"]) <= 1e-12
    assert abs(model.h_func(s).item() - float(g["h"])) <= 1e-9 * max(abs(float(g["h"])), 1e-3)
    assert _relmax(model.fc1_to_adj(), g["adj"]) <= 1e-13
    ref_l1 = np.abs(g["init.fc1.weight"]).sum()
    assert abs(model.fc1_l1_reg().item() - ref_l1) <= 1e-12 * ref_l1
    eq = DagmaNonlinear(model)
    X_hat = X_hat if X_hat_ref is None else torch.from_numpy(X_hat_ref)
    assert abs(eq.log_mse_loss(X_hat, torch.from_numpy(X)).item() - float(g["score"])) \
        <= 1e-12 * abs(float(g["score"]))
    # one evaluation: objective pieces and every gradient within 1e-9 relative (north_star)
    eng = _MlpEngine(model, torch.from_numpy(X).cuda())
    sh = eng.state_host
    sh.zero_()
    sh[F_MU], sh[F_S], sh[F_LAM1], sh[F_LAM2] = mu, s, lambda1, lambda2
    eng.state.copy_(sh)
    eng.evaluate(s)
    st, _, halted = eng.pull()
    assert not halted
    for f, key in ((F_OBJ, "obj"), (F_SCORE, "score"), (F_H, "h")):
        assert abs(float(st[f]) - float(g[key])) <= 1e-9 * max(abs(float(g[key])), 1e-3), key
    grads = eng.grads_scaled()
    for k, gk in grads.items():
        ref = g["grad." + k].reshape(gk.shape)
        assert _relmax(gk, ref) <= 1e-9, k
    # `steps` iterations of minimize: parameters match torch.optim.Adam
    steps = int(g["steps"])
    eq.X = torch.from_numpy(X).cuda()
    eq.checkpoint = 10 ** 9
    ok = eq.minimize(steps, lr, lambda1, lambda2, mu, s)
    assert ok == bool(g["ok"]) and eq.n_iters == steps
    for k, p in model.state_dict().items():
        ref = g[f"after{steps}.{k}"]
        assert _relmax(p.numpy(), ref) <= 1e-9, k


def test_mlp_short_fit_vs_reference(golden):
    from midagma_b200.nonlinear import DagmaNonlinear
    g = golden("mlp_fit_d5")
    T, warm, mx, ck = (int(x) for x in g["kw"])
    model = _model_from(g)
    eq = DagmaNonlinear(model)
    W = eq.fit(g["X"], lambda1=0.02, lambda2=0.005, T=T, warm_iter=warm, max_iter=mx, checkpoint=ck)
    assert np.abs(model.fc1_to_adj() - g["W_raw"]).max() <= 1e-8
    assert np.array_equal(W != 0, g["W_est"] != 0)
    for k, p in model.state_dict().items():
        assert np.abs(p.numpy() - g["final." + k]).max() <= 1e-8, k


def test_mlp_h_negative_returns_false():
    """fc1 large enough that sI - A leaves the M-matrix domain -> minimize returns False (nonlinear.py:215)."""
    from midagma_b200.nonlinear import DagmaMLP, DagmaNonlinear
    torch.manual_seed(0)
    d, m1, n = 6, 3, 64
    model = DagmaMLP([d, m1, 1])
    with torch.no_grad():
        model.fc1.weight.fill_(0.8)
    eq = DagmaNonlinear(model)
    eq.X = torch.randn(n, d, dtype=torch.float64).cuda()
    eq.checkpoint = 10
    before = model.fc1.weight.clone()
    assert eq.minimize(20, 1e-3, 0.02, 0.005, 0.1, 1.0) is False
    assert torch.equal(model.fc1.weight, before)
    # and the oracle agrees
    o = OracleMLP([d, m1, 1], {k: v.numpy() for k, v in model.state_dict().items()})
    assert OracleNonlinear(o).minimize(eq.X.cpu().numpy(), 20, 1e-3, 0.02, 0.005, 0.1, 1.0) is False


def test_locally_connected_forward():
    from midagma_b200.nonlinear import LocallyConnected
    torch.manual_seed(1)
    lc = LocallyConnected(5, 4, 3)
    x = torch.randn(17, 5, 4, dtype=torch.float64)
    ref = torch.matmul(x.unsqueeze(2), lc.weight.detach().unsqueeze(0)).squeeze(2) + lc.bias.detach()
    assert _relmax(lc(x).numpy(), ref.numpy()) <= 1e-14


@pytest.mark.parametrize("d,m1,n,iters", [(40, 10, 2000, 25), (5, 3, 50, 40), (64, 7, 333, 12), (17, 40, 1000, 12),
                                          (8, 4, 100000, 6), (33, 16, 4099, 8)],
                         ids=["c3", "tiny", "d64-m7", "m1-40", "streamed-samples", "odd"])
def test_one_kernel_iteration_vs_launch_sequence(d, m1, n, iters, monkeypatch):
    """The persistent one-kernel iteration (csrc/mlp_iter.cu) against the launch sequence of csrc/mlp.cu on the same
    start: parameters, Adam moments and the state block after `iters` iterations (different summation orders only),
    for shapes that exercise one and several node slices, padded m-tiles, the last partial sample group and sample
    groups that do not fit in shared memory (streamed in sub-groups)."""
    from midagma_b200.nonlinear import (DagmaMLP, _MlpEngine, F_MU, F_S, F_LR, F_LAM1, F_LAM2, F_B1, F_B2, F_GAMMA, F_OBJ,
                                        F_SCORE, F_H, F_SS, F_L1)
    torch.manual_seed(d * 1000 + m1)
    model = DagmaMLP([d, m1, 1], bias=True, dtype=torch.double)
    with torch.no_grad():
        model.fc1.weight.mul_(0.5).add_(0.02 * torch.randn_like(model.fc1.weight))
        model.fc1.bias.add_(0.1 * torch.randn_like(model.fc1.bias))
    X = torch.randn(n, d, dtype=torch.float64).cuda()
    out = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("DAGMA_MLP_FUSED", mode)
        eng = _MlpEngine(model, X)
        assert eng.one_kernel == (mode == "1")
        sh = eng.state_host
        sh.zero_()
        for f, val in ((F_MU, 0.1), (F_S, 1.0), (F_LR, 2e-3), (F_LAM1, 0.02), (F_LAM2, 0.005), (F_B1, 0.99), (F_B2, 0.999),
                       (F_GAMMA, 1.0)):
            sh[f] = val
        eng.state.copy_(sh)
        eng.replay(1.0, iters - 3)
        eng.replay(1.0, 3)                       # a second launch continues from the state the first one left
        st, step, halted = eng.pull()
        assert step == iters and not halted
        out[mode] = (eng.theta.cpu().numpy(), eng.m.cpu().numpy(), eng.v.cpu().numpy(), st.clone().numpy())
    for a, b, what in zip(out["1"][:3], out["0"][:3], ("theta", "m", "v")):
        assert _relmax(a, b) <= 1e-11, (what, _relmax(a, b))
    for f in (F_OBJ, F_SCORE, F_H, F_SS, F_L1):
        assert abs(out["1"][3][f] - out["0"][3][f]) <= 1e-11 * max(abs(out["0"][3][f]), 1e-3), f
