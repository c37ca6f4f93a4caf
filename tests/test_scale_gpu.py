"""Parity at the sizes BASELINE.json quotes (round 2): C5 (l2, SF4, d = 2000), C2 (logistic, d = 100, n = 10 000),
C3 (MLP [40, 10, 1], n = 2000).  Fixtures were recorded from the unmodified reference by
oracle/make_golden_scale.py; the big inputs are regenerated from their seeds and proven identical by checksum.

Tolerances (SURVEY.md 7.4): per-call h / inverse / gradient 1e-9 max-norm relative where the reference route itself is
that accurate; where LAPACK's own error (cond * eps) is larger, the GPU inverse must be at least as close to the exact
inverse as LAPACK's (residual test) -- "measure cond on snapshots first".  Short-horizon fits: identical edge set and
|dW| <= 1e-6."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import simulate

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def _relmax(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _checksum(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return np.array([a.sum(), np.abs(a).sum(), (a * a).sum(), a.ravel()[:: max(a.size // 97, 1)].sum()])


# --------------------------------------------------------------------------------------------- C5: the inverse
def _sf4_w(alpha, eps, density=0.01):
    """A late-stage-like iterate: the (scaled) true SF4 weights plus small dense noise that closes cycles."""
    d = 2000
    rng = np.random.default_rng(0)
    W_true = simulate.simulate_parameter(simulate.simulate_dag(d, 4 * d, "SF", rng), rng)
    nr = np.random.default_rng(1)
    return alpha * W_true + eps * nr.normal(size=(d, d)) * (nr.random((d, d)) < density)


def _stochastic_w(t, seed=3):
    """W with W o W = t * P, P row-stochastic (Perron root exactly 1): sI - W o W is a nonsingular M-matrix iff
    t < s, and its inverse blows up like 1 / (s - t) at the boundary."""
    d = 2000
    rng = np.random.default_rng(seed)
    P = rng.random((d, d)) * (rng.random((d, d)) < 0.004)
    P[np.arange(d), rng.integers(d, size=d)] += 0.5          # no empty row
    P /= P.sum(axis=1, keepdims=True)
    return np.sqrt(t * P)


C5_CASES = {
    # name: (W factory, s, feasible?, tolerance vs LAPACK).  Measured on the LAPACK side (build container):
    #   benign             cond_1 2e1,  max(M^-1) 1.2,   residual 2e-15
    #   late_stage_s0.7_a  cond_1 1e9,  max(M^-1) 1.9e5, residual 2e-10, min entry +3.5e-15
    #   late_stage_s0.7_b  cond_1 4e10, max(M^-1) 5.7e6, residual 5e-9,  min entry +6.0e-16
    #   dag_exact_zeros    an exact DAG: the true inverse has exact zeros; LAPACK returns entries down to -3e-12 there,
    #                      i.e. the REFERENCE's predicate any(inv + 1e-16 < 0) fires on round-off (SURVEY 7.4 (2)); the
    #                      no-pivot elimination of a Z-matrix cannot produce a negative entry, so the GPU says feasible
    #   boundary_*         Perron root of W o W at s (1 -+ 1e-7): max(M^-1) 2e4 / negative inverse
    "benign": (lambda: _benign_w(), 0.9, True, 1e-10),
    "late_stage_s0.7_a": (lambda: _sf4_w(0.55, 1e-3), 0.7, True, 1e-9),
    "late_stage_s0.7_b": (lambda: _sf4_w(0.6, 5e-4), 0.7, True, 1e-7),
    "dag_exact_zeros": (lambda: _sf4_w(0.45, 0.0), 0.6, "lapack-noise", 1e-9),
    "boundary_inside": (lambda: _stochastic_w(0.8 * (1 - 1e-7)), 0.8, True, 1e-6),
    "boundary_outside": (lambda: _stochastic_w(0.8 * (1 + 1e-7)), 0.8, False, None),
}


def _benign_w():
    d = 2000
    rng = np.random.default_rng(d)
    A = rng.normal(size=(d, d)) * (rng.random((d, d)) < 0.02)
    v = np.ones(d)
    B = A * A
    for _ in range(200):                                      # Perron root by power iteration (B >= 0)
        v = B @ v
        rho = np.linalg.norm(v)
        v /= rho
    return A * np.sqrt(0.7 / rho)


@pytest.mark.parametrize("case", list(C5_CASES))
def test_c5_inverse_d2000(case):
    """The blocked two-level inverse at the size of config 5 (DagmaLinear._h / the per-iteration inverse,
    linear.py:113-115, 226): value, inverse, gradient, min entry and the feasibility predicate."""
    from midagma_b200.linear import logdet_inv
    make, s, feasible, tol = C5_CASES[case]
    W = make()
    d = W.shape[0]
    out = logdet_inv(torch.from_numpy(np.ascontiguousarray(W[None])).cuda(), s=s, square_input=True, want_inv=True,
                     want_grad=True)
    info = int(out["info"][0].item())
    M = s * np.eye(d) - W * W
    Minv = np.linalg.inv(M)                                    # LAPACK getrf + getri, the reference's route
    if not feasible:
        assert np.any(Minv + 1e-16 < 0), "test matrix must be outside the M-matrix domain"
        assert info != 0
        return
    X = out["minv"][0].cpu().numpy()
    Id = np.eye(d)
    res_gpu, res_ref = np.abs(M @ X - Id).max(), np.abs(M @ Minv - Id).max()
    err = _relmax(X, Minv)
    cond1 = np.abs(M).sum(0).max() * np.abs(Minv).sum(0).max()
    lad = np.linalg.slogdet(M)[1]
    print(f"{case}: cond_1 {cond1:.2e} max(Minv) {Minv.max():.2e} min(Minv) ref {Minv.min():.2e} gpu "
          f"{out['min_entry'][0].item():.2e} | max-norm rel err {err:.2e} | residual gpu {res_gpu:.2e} lapack {res_ref:.2e}")
    if feasible is True:
        assert not np.any(Minv + 1e-16 < 0), "test matrix must be inside the domain for the reference"
    else:                                                      # exact DAG: the negative LAPACK entries are round-off
        assert Minv.min() > -1e-9 * Minv.max() and simulate.is_dag(W)
    assert info == 0
    assert out["min_entry"][0].item() + 1e-16 >= 0            # the literal predicate of linear.py:226-230
    assert abs(out["min_entry"][0].item() - X.min()) <= 1e-12 * np.abs(X).max()
    assert err <= tol
    assert res_gpu <= 2.0 * res_ref + 1e-13                   # at least as close to the exact inverse as LAPACK
    assert abs(out["logabsdet"][0].item() - lad) <= 1e-10 * max(1.0, abs(lad))
    assert abs(out["h"][0].item() - (-lad + d * np.log(s))) <= 1e-9 * max(1.0, abs(lad))
    # gradient 2 W o M^{-T}: absolute scale max|2W| max|M^-1| (for the exact DAG the true gradient is identically zero)
    gerr = np.abs(out["grad"][0].cpu().numpy() - 2 * W * Minv.T).max()
    assert gerr <= max(tol, 1e-10) * 2 * np.abs(W).max() * np.abs(Minv).max()


# --------------------------------------------------------------------------------------------- C5: reduced fit
def test_c5_reduced_fit_vs_reference(golden):
    """`fit(X, lambda1=0.02, warm_iter=500, max_iter=500)` on the SF4 d = 2000, n = 20 000 problem of config 5
    (linear.py:335-462) against the run of the unmodified reference: identical thresholded edge set, |dW| reported."""
    from midagma_b200 import DagmaLinear
    g = golden("fit_c5_reduced")
    X, W_true = simulate.config_c5(int(g["seed"]))
    assert np.allclose(_checksum(X), g["x_checksum"], rtol=1e-13, atol=0), "not the arrays the reference was fed"
    model = DagmaLinear("l2")
    W_est = model.fit(X, lambda1=float(g["lambda1"]), warm_iter=int(g["warm_iter"]), max_iter=int(g["max_iter"]),
                      s=[1.0, .9, .8, .7, .6])
    d = 2000
    W = model.W_raw
    ref_calls = g["calls"]
    assert model.stage_iters == [int(c[0]) for c in ref_calls] and all(int(c[1]) == 1 for c in ref_calls)
    # pre-threshold W of the reference: every entry with |W| >= 0.05 (flat indices, delta-coded) and whether it is an
    # edge (|W| >= 0.3); the values of a fixed, seeded sample of those entries
    idx = np.cumsum(g["w_idx_delta"].astype(np.int64))
    big = np.zeros(d * d, dtype=bool)
    big[idx] = True
    big = big.reshape(d, d)
    edges_ref = np.zeros(d * d, dtype=bool)
    edges_ref[idx[g["w_edge"]]] = True
    edges_ref = edges_ref.reshape(d, d)
    sample, w_ref = idx[g["w_sample_pos"]], g["w_sample_val"]
    err_big = np.abs(W.ravel()[sample] - w_ref).max()
    err_small = np.abs(W)[~big].max()                          # the reference has |W| < 0.05 there
    edges = W_est != 0
    margin = np.abs(np.abs(w_ref) - 0.3).min()
    print(f"C5 reduced fit: stage iters {model.stage_iters}, edges {int(edges.sum())} (reference {int(g['nnz_est'])}), "
          f"edge-set distance {int((edges != edges_ref).sum())}, max|dW| on sampled |W_ref|>=0.05: {err_big:.2e}, "
          f"max|W| elsewhere {err_small:.3f}, closest sampled |W_ref| to the threshold {margin:.2e}, "
          f"h_final {model.h_final:.6e} (ref {float(g['h_final']):.6e})")
    assert int(edges_ref.sum()) == int(g["nnz_est"])
    assert int((edges != edges_ref).sum()) == 0
    assert err_big <= 1e-6 and err_small < 0.05 + 1e-6
    assert abs(np.linalg.norm(W) - float(g["w_fro"])) <= 1e-7 * float(g["w_fro"])
    assert abs(np.abs(W).sum() - float(g["w_abssum"])) <= 1e-7 * float(g["w_abssum"])
    assert abs(model.h_final - float(g["h_final"])) <= 1e-7 * max(abs(float(g["h_final"])), 1e-3)
    assert abs(model.score_final - float(g["score_final"])) <= 1e-9 * abs(float(g["score_final"]))


# --------------------------------------------------------------------------------------------- C2
def test_c2_logistic_stages_vs_reference(golden):
    """Config 2 at size: logistic loss, d = 100, n = 10 000 binary data (linear.py:165-333 with the score of :90-92,
    :246) against trajectories of the unmodified reference.

    * From a generic (seeded random) W0: 100 iterations, every entry within 1e-9.
    * From W = 0, two chained stages: with binary data some entries have an EXACTLY zero gradient at W = 0 (integer
      ties 2 #(x_i x_j) = #(x_i), about 1 % of the pairs at n = 10 000).  The reference computes
      `(1/n * X.T) @ expit(.) - cov` there, i.e. pure round-off (+-1e-15) whose sign starts the l1 chatter of that
      entry (amplitude ~ lr); `X.T @ expit(.) / n - cov` -- what the kernels compute -- is exactly 0.  Those entries are
      round-off driven in the reference itself (SURVEY.md 7.4) and are graded at the chatter amplitude; every other
      entry at the short-horizon bar 1e-6."""
    from midagma_b200 import DagmaLinear
    g = golden("linear_logistic_c2")
    X, _ = simulate.config_c2(int(g["seed"]))
    assert np.allclose(_checksum(X), g["x_checksum"], rtol=1e-13, atol=0)
    model = DagmaLinear("logistic")
    model.fit(X, lambda1=float(g["lambda1"]), T=1, warm_iter=0, max_iter=0, checkpoint=int(g["checkpoint"]))
    assert _relmax(model.cov, X.T @ X / float(X.shape[0])) <= 1e-13
    d = model.d
    # ---- generic start
    W, ok = model.minimize(g["W0_random"].copy(), 1.0, int(g["iters_random"]), 1.0, lr=3e-4)
    err = np.abs(W - g["W_random_after"]).max()
    print("C2 random start: max|dW| =", err)
    assert ok == bool(g["ok_random"]) and model.last_iters == int(g["iters_random"])
    assert err <= 1e-9
    # ---- zero start
    cnt = X.T @ X                                              # exact integers
    ties = (2.0 * cnt == np.diag(cnt)[:, None])
    print("exact-tie entries at W = 0:", int(ties.sum()))
    assert ties.sum() > 0
    # the reference's own round-off envelope: the oracle (bit-identical to the reference) against itself with the
    # score gradient summed first and scaled afterwards -- the same mathematics, different rounding of the tie entries
    from oracle.linear_ref import OracleLinear
    mu0, s0, it0, lr0 = g["stages"][0]
    o_ref = OracleLinear("logistic").prepare(X.copy(), float(g["lambda1"]), checkpoint=int(g["checkpoint"]))
    W_a, _ = o_ref.minimize(np.zeros((d, d)), mu0, int(it0), s0, lr0)
    # (in the build container the oracle reproduces the fixture bit for bit; on another host the threaded BLAS may sum
    # in another order, which is one more sample of the same envelope)
    print("oracle on this host vs the reference fixture: max|dW|", np.abs(W_a - g["W_after_0"]).max())
    o_alt = OracleLinear("logistic").prepare(X.copy(), float(g["lambda1"]), checkpoint=int(g["checkpoint"]))
    o_alt.logistic_route = "sum-then-scale"
    W_b, _ = o_alt.minimize(np.zeros((d, d)), mu0, int(it0), s0, lr0)
    env = np.maximum(np.abs(W_b - W_a), np.abs(W_b - g["W_after_0"]))
    print("reference round-off envelope after stage 0: max|dW|", env.max(), "entries > 1e-8:", int((env > 1e-8).sum()))
    W = np.zeros((d, d))
    for si, (mu, s, iters, lr) in enumerate(g["stages"]):
        W, ok = model.minimize(W.copy(), mu, int(iters), s, lr=lr)
        assert ok == bool(g[f"ok_{si}"]) and model.last_iters == int(g[f"iters_{si}"])
        e = np.abs(W - g[f"W_after_{si}"])
        _, _, obj, score, h, _ = model.checkpoint_log[-1]
        print("C2 stage", si, "max|dW|", e.max(), "entries > 1e-8:", int((e > 1e-8).sum()), "obj", obj, "ref",
              float(g[f"obj_{si}"]))
        # inside the envelope: the chatter amplitude (a few lr) bounds every entry, most entries are untouched, and
        # the objective agrees to 1e-6
        assert e.max() <= max(2.0 * env.max(), 1e-6) and e.max() <= 2e-3, (si, e.max(), env.max())
        assert (e > 1e-8).mean() <= 0.15
        assert abs(obj - float(g[f"obj_{si}"])) <= 1e-6 * abs(float(g[f"obj_{si}"]))
        assert abs(score - float(g[f"score_{si}"])) <= 1e-6 * abs(float(g[f"score_{si}"]))
    # ---- per-call parity at the reference's last W (1e-9 relative)
    Wl = g[f"W_after_{len(g['stages']) - 1}"]
    sv, sg = model._score(Wl)
    assert abs(sv - float(g["score_val"])) <= 1e-9 * abs(float(g["score_val"]))
    assert _relmax(sg, g["score_grad"]) <= 1e-9
    hv, hg = model._h(Wl, 0.9)
    assert abs(hv - float(g["h_val"])) <= 1e-9 * max(abs(float(g["h_val"])), 1e-3)
    assert _relmax(hg, g["h_grad"]) <= 1e-9


# --------------------------------------------------------------------------------------------- C3: fit retry path
@pytest.mark.parametrize("name", ["mlp_fit_retry_d5", "mlp_fit_retry2_d5", "mlp_fit_retry_decay_d5"])
def test_mlp_fit_retry_path_vs_reference(golden, name):
    """DagmaNonlinear.fit through its failure branch (nonlinear.py:316-327): h < 0 -> parameters restored, lr halved
    (and the halving persists into later stages), ExponentialLR(0.8) switched on, s_cur = 1."""
    from midagma_b200.nonlinear import DagmaMLP, DagmaNonlinear
    g = golden(name)
    dims = [int(x) for x in g["dims"]]
    model = DagmaMLP(dims=dims, bias=True, dtype=torch.double)
    model.load_state_dict({k[5:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("init.")})
    T, warm, mx, ck = (int(x) for x in g["kw"])
    eq = DagmaNonlinear(model)
    W = eq.fit(g["X"], lambda1=0.02, lambda2=0.005, lr=float(g["lr"]), T=T, warm_iter=warm, max_iter=mx,
               checkpoint=ck)
    calls = np.array(eq.minimize_calls, dtype=np.float64)
    print(name, "calls (lr, s, ok, decay):", calls.tolist(), "max|dW_raw|", np.abs(model.fc1_to_adj() - g["W_raw"]).max())
    assert calls.shape == g["calls"].shape and np.array_equal(calls, g["calls"])
    assert (g["calls"][:, 2] == 0).any(), "fixture must exercise the retry path"
    assert np.abs(model.fc1_to_adj() - g["W_raw"]).max() <= 1e-6
    assert np.array_equal(W != 0, g["W_est"] != 0)
    for k, p in model.state_dict().items():
        assert np.abs(p.numpy() - g["final." + k]).max() <= 1e-6, k


def test_locally_connected_without_bias():
    """LocallyConnected(bias=False) (locally_connected.py:38-43, 72-74)."""
    from midagma_b200.nonlinear import LocallyConnected
    torch.manual_seed(2)
    lc = LocallyConnected(6, 5, 2, bias=False)
    assert lc.bias is None and [k for k, _ in lc.named_parameters()] == ["weight"]
    x = torch.randn(33, 6, 5, dtype=torch.float64)
    ref = torch.matmul(x.unsqueeze(2), lc.weight.detach().unsqueeze(0)).squeeze(2)
    assert _relmax(lc(x).numpy(), ref.numpy()) <= 1e-14


# --------------------------------------------------------------------------------------------- host-pointer C entry
def test_host_pointer_entry_matches_fit_batch():
    """dagma_linear_fit_small_host_f64 (the entry INTEGRATION.md shows a C caller): host pointers in, host results
    out, against fit_batch on the same problems."""
    import ctypes as C
    from midagma_b200 import _lib, fit_batch
    lib = _lib.load()
    d, batch = 40, 3
    covs, lams = [], np.array([0.02, 0.03, 0.05])
    for p in range(batch):
        X, _ = simulate.make_linear_problem(d, 2, 300, "ER", "gauss", 20 + p)
        X -= X.mean(axis=0, keepdims=True)
        covs.append(X.T @ X / 300)
    cov = np.ascontiguousarray(np.stack(covs))
    kw = dict(T=3, warm_iter=300, max_iter=400, checkpoint=100)
    W_ref, info = fit_batch(None, lams, cov=cov, s=(1.0, .9, .8), return_info=True, **kw)
    a = _lib.SmallFitArgs()
    a.batch, a.d, a.n_stages, a.checkpoint, a.retry_on_fail, a.ckpt_log_cap = batch, d, 3, 100, 1, 0
    a.lr, a.tol, a.beta1, a.beta2 = 3e-4, 1e-6, 0.99, 0.999
    mu = 1.0
    for t, s in enumerate((1.0, .9, .8)):
        a.mu[t], a.s[t], a.iters[t] = mu, s, 400 if t == 2 else 300
        mu *= 0.1
    W = np.zeros((batch, d, d))
    status = np.full(batch, -1, dtype=np.int32)
    stats = np.full((batch, 3, 8), np.nan)
    final = np.full((batch, 2), np.nan)
    count = np.full(batch, -1, dtype=np.int32)
    ptr = lambda x: x.ctypes.data_as(C.c_void_p)  # noqa: E731
    a.cov, a.lambda1, a.w = ptr(cov), ptr(lams), ptr(W)
    a.status, a.stage_stats, a.final, a.ckpt_count = ptr(status), ptr(stats), ptr(final), ptr(count)
    _lib.check(lib.dagma_linear_fit_small_host_f64(None, C.byref(a)), "dagma_linear_fit_small_host_f64")
    assert status.tolist() == [0, 0, 0]
    assert np.array_equal(W, info["W_raw"])
    assert np.array_equal(stats[:, :, 0].astype(np.int64), info["stage_iters"])
    assert np.array_equal(final[:, 0], info["h_final"]) and np.array_equal(final[:, 1], info["score_final"])
    W[np.abs(W) < 0.3] = 0
    assert np.array_equal(W, W_ref)
    # T = 0: outputs of stages that never run read as zero, not as device garbage (the block is memset)
    a.n_stages = 0
    W0 = np.zeros((batch, d, d))
    stats0 = np.full((batch, 1, 8), np.nan)
    a.w, a.stage_stats = ptr(W0), ptr(stats0)
    _lib.check(lib.dagma_linear_fit_small_host_f64(None, C.byref(a)), "dagma_linear_fit_small_host_f64")
    assert status.tolist() == [0, 0, 0] and np.all(stats0 == 0) and np.all(np.isfinite(final))
    assert np.all(final[:, 0] == 0.0)                                      # h(0) = 0
    assert np.allclose(final[:, 1], 0.5 * np.trace(cov, axis1=1, axis2=2), rtol=1e-13)
