"""DagmaNonlinear at every shape it accepts, against the float64 oracle (``oracle.nonlinear_ref``).

* The persistent ``[d, m1, 1]`` kernel (csrc/mlp_iter.cu, d <= 64, m1 <= 40) cuts a problem into node slices and
  sample groups (``mi_plan``) and stages ``fc1.weight`` for its h CTA in node chunks.  A Python restatement of that
  plan is checked against the library, and the shape list below is checked to reach every edge of it: partial node
  slices, padded m- and n-tiles, padded and one-sample sample groups, samples streamed in sub-groups, odd rows of
  ``fc1.weight`` and a partial last staged chunk.
* The launch sequence (csrc/mlp.cu) serves ``DAGMA_MLP_FUSED=0``, d > 64, m1 > 40, deeper stacks and ``[d, 1]``:
  one evaluation (objective, score, h, every gradient) and K steps, at n on both sides of the 256-sample chunks, with
  the on-chip inverse up to d = 128 and the blocked inverse above.
* Halting: infeasible starts, a halt in the middle of a launch, and ``sI - A`` outside the M-matrix domain with
  ``h > 0``, where the reference keeps stepping.
* Split launches, ExponentialLR across launch boundaries, short full fits and the public helpers at scale.

Starts are generic (random ``fc1.weight``, perturbed biases), so no Adam sign tie decides a comparison."""
import math

import numpy as np
import pytest
import torch

from oracle.nonlinear_ref import OracleMLP, OracleNonlinear

pytestmark = pytest.mark.gpu

LAM1, LAM2, MU = 0.02, 0.005, 0.1


def _relmax(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _close(a, b, rtol, floor=1e-3):
    return abs(a - b) <= rtol * max(abs(b), floor)


# =====================================================================================================================
# the plan of csrc/mlp_iter.cu, restated
# =====================================================================================================================
MI_PR, MI_KSL = 40, 4
MI_SMEM_CAP_D = 200 * 1024 // 8                 # MI_SMEM_CAP in doubles
DMMA_SMEM_TOTAL = 2 * 64 * 68 + 2 * 8 * 68 + 2 * 64 * 8 + 2 * 64 + 64 + 96 + 2   # DmmaSmem::total (small_dmma.cuh)
MI_H_STAGE = (DMMA_SMEM_TOTAL + 1) & ~1


def _cdiv(a, b):
    return -(-a // b)


def _tdiv(a, b):                                 # C integer division (truncates toward zero)
    q = abs(a) // abs(b)
    return q if (a >= 0) == (b > 0) else -q


def mi_plan(n, d, m1, sms):
    """``mi_plan`` + the h-CTA staging of ``mlp_iter_launch``; None where the kernel does not run the shape."""
    if not (1 <= d <= 64 and 1 <= m1 <= MI_PR and n >= 1 and sms >= 2):
        return None
    JN = min(MI_PR // m1, d)
    JS = _cdiv(d, JN)
    if JS > sms - 1:
        return None
    SG = (sms - 1) // JS
    NSG = 16 * _cdiv(_cdiv(n, SG), 16)
    SG = _cdiv(n, NSG)
    ldx = 16 * _cdiv(d, 16) + 4
    NT, MT = _cdiv(d, 8), _cdiv(JN * m1, 8)
    fixed = 8 * MT * ldx + 2 * MI_PR + JN + (2 * MI_PR + JN + 2) + MI_KSL * MT * NT * 64 + 96 + 16
    per_sample = ldx + 8 * MT + JN
    cap = _tdiv(_tdiv(MI_SMEM_CAP_D - fixed - 8 * MT * 4, per_sample), 16) * 16
    if cap < 16:
        return None
    NSUB = min(NSG, cap)
    ldh = NSUB + 4
    o_tail = 8 * MT * ldx + NSUB * ldx + 8 * MT * ldh + JN * NSUB + 2 * MI_PR + JN
    total = ((o_tail + 2 * MI_PR + JN + 2) & ~1) + MI_KSL * MT * NT * 64 + 96
    if total > MI_SMEM_CAP_D:
        return None
    w1, node = d * m1 * d, m1 * d
    stage = max(min(MI_SMEM_CAP_D - MI_H_STAGE, w1), node)
    stage = (stage + 1) & ~1
    jc = max(1, stage // node)
    W = w1 + 2 * d * m1 + d
    return dict(n=n, d=d, m1=m1, JN=JN, JS=JS, SG=SG, NSG=NSG, NSUB=NSUB, MT=MT, jc=jc, ws=SG * W + SG * JS + 8)


def _last_sub(p):
    """samples of the last sub-group of the last sample group"""
    last = p["n"] - (p["SG"] - 1) * p["NSG"]
    return last - ((last - 1) // p["NSUB"]) * p["NSUB"]


PLAN_EDGES = {
    "d = 0 mod 4": lambda p: p["d"] % 4 == 0,
    "d = 1 mod 4": lambda p: p["d"] % 4 == 1,
    "d = 2 mod 4": lambda p: p["d"] % 4 == 2,
    "d = 3 mod 4": lambda p: p["d"] % 4 == 3,
    "d not a multiple of 8": lambda p: p["d"] % 8 != 0,
    "d = 1": lambda p: p["d"] == 1,
    "d = 64": lambda p: p["d"] == 64,
    "JN m1 not a multiple of 8 (padded m-tile)": lambda p: (p["JN"] * p["m1"]) % 8 != 0,
    "JS > 1 with a partial last slice": lambda p: p["JS"] > 1 and p["d"] % p["JN"] != 0,
    "m1 = 1": lambda p: p["m1"] == 1,
    "m1 = 40": lambda p: p["m1"] == 40,
    "n = 1": lambda p: p["n"] == 1,
    "n < 16": lambda p: p["n"] < 16,
    "n = SG NSG": lambda p: p["n"] == p["SG"] * p["NSG"] and p["SG"] > 1,
    "n = SG NSG - 1": lambda p: p["n"] == p["SG"] * p["NSG"] - 1 and p["SG"] > 1,
    "n = SG NSG + 1 (last sample group holds one sample)": lambda p: p["SG"] > 1 and p["n"] == (p["SG"] - 1) * p["NSG"] + 1,
    "NSUB < NSG, last sub-group partial and not a multiple of 16":
        lambda p: p["NSUB"] < p["NSG"] and _last_sub(p) < p["NSUB"] and _last_sub(p) % 16 != 0,
    "m1 d odd (scalar staging loads)": lambda p: (p["m1"] * p["d"]) % 2 == 1,
    "m1 d even (cp.async staging)": lambda p: (p["m1"] * p["d"]) % 2 == 0,
    "fc1.weight in one staged chunk": lambda p: p["jc"] >= p["d"],
    "fc1.weight in several staged chunks, the last partial": lambda p: p["jc"] < p["d"] and p["d"] % p["jc"] != 0,
}

# (d, m1, n, s) of the persistent-kernel comparisons (section 2); which plan edge each one reaches is asserted by
# test_shape_list_reaches_every_plan_edge
FUSED_SHAPES = [
    (1, 1, 1, 1.0), (2, 7, 15, 0.8), (3, 13, 50, 3.0), (5, 9, 200, 1.0), (5, 2, 2352, 0.8), (8, 8, 256, 3.0),
    (8, 13, 700, 1.0), (9, 3, 300, 0.8), (9, 40, 160, 3.0), (15, 2, 1000, 1.0), (15, 39, 90, 0.8), (16, 20, 700, 3.0),
    (17, 3, 333, 1.0), (17, 9, 463, 0.8), (31, 39, 1500, 3.0), (32, 1, 2000, 1.0), (32, 3, 97, 0.8),
    (33, 7, 1200, 3.0), (33, 20, 449, 1.0), (40, 7, 500, 0.8), (40, 9, 900, 3.0), (63, 13, 500, 1.0),
    (64, 1, 147, 0.8), (64, 40, 1000, 3.0), (2, 1, 7, 1.0),
]


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _sid(shape):
    d, m1, n, s = shape
    return f"d{d}-m{m1}-n{n}-s{s}"


def test_plan_restatement_matches_library():
    from midagma_b200 import _lib
    lib, sms = _lib.load(), _sms()
    _lib.require_device()
    grid = [(n, d, m1) for d in (1, 2, 3, 5, 8, 9, 16, 17, 31, 32, 33, 40, 63, 64, 65)
            for m1 in (1, 2, 3, 7, 8, 13, 20, 39, 40, 41) for n in (1, 15, 16, 17, 255, 1000, 4099, 100000, 1000003)]
    for n, d, m1 in grid + [(s[2], s[0], s[1]) for s in FUSED_SHAPES]:
        p = mi_plan(n, d, m1, sms)
        assert bool(lib.dagma_mlp_iter_supported(n, d, m1)) == (p is not None), (n, d, m1)
        assert lib.dagma_mlp_iter_workspace_doubles(n, d, m1) == (p["ws"] if p else 0), (n, d, m1)


def test_shape_list_reaches_every_plan_edge():
    sms = _sms()
    plans = [mi_plan(n, d, m1, sms) for d, m1, n, _ in FUSED_SHAPES]
    assert all(p is not None for p in plans)
    hit = {}
    for name, pred in PLAN_EDGES.items():
        who = [f"[{p['d']}, {p['m1']}, 1] n={p['n']}" for p in plans if pred(p)]
        hit[name] = who
    missing = [k for k, v in hit.items() if not v]
    print("\n".join(f"{k}: {v[0]}" for k, v in hit.items() if v))
    assert not missing, f"no shape of FUSED_SHAPES reaches {missing}"


# =====================================================================================================================
# helpers
# =====================================================================================================================
def _start(dims, seed, a_row=0.2):
    """A generic start: fc1.weight ~ N(0, a_row / (d m1)) (A's row sums ~ a_row, well inside the domain at s >= 0.8,
    no zero or tied entries), fc1.bias perturbed, the LocallyConnected layers at their default initialisation."""
    from midagma_b200.nonlinear import DagmaMLP
    torch.manual_seed(seed)
    model = DagmaMLP(list(dims), bias=True, dtype=torch.double)
    d, m1 = dims[0], dims[1]
    with torch.no_grad():
        model.fc1.weight.copy_(math.sqrt(a_row / (d * m1)) * torch.randn_like(model.fc1.weight))
        model.fc1.bias.add_(0.1 * torch.randn_like(model.fc1.bias))
    return model


def _params(model):
    return {k: v.detach().numpy().copy() for k, v in model.state_dict().items()}


def _data(n, d, seed):
    return np.random.default_rng(seed).normal(size=(n, d))


def _oracle(model):
    return OracleNonlinear(OracleMLP(list(model.dims), _params(model)))


def _minimize_both(model, X, K, lr, s, checkpoint, lr_decay=False):
    """DagmaNonlinear.minimize and OracleNonlinear.minimize from the same start, tol = 0 (no early stop)."""
    from midagma_b200.nonlinear import DagmaNonlinear
    o = _oracle(model)
    o.trace = []
    ok_ref = o.minimize(X, K, lr, LAM1, LAM2, MU, s, lr_decay=lr_decay, tol=0.0, checkpoint=checkpoint)
    eq = DagmaNonlinear(model)
    eq.X, eq.checkpoint = torch.from_numpy(X).cuda(), checkpoint
    ok = eq.minimize(K, lr, LAM1, LAM2, MU, s, lr_decay=lr_decay, tol=0.0)
    return eq, ok, o, ok_ref


def _check_params(model, o, rtol, what):
    worst = 0.0
    for k, p in model.state_dict().items():
        err = _relmax(p.numpy(), o.model.p[k])
        worst = max(worst, err)
        assert err <= rtol, (what, k, err)
    return worst


def _check_state(eq, o, rtol, what):
    from midagma_b200.nonlinear import F_OBJ, F_SCORE, F_H
    st, _, _ = eq._engine.pull()
    last = o.trace[-1]
    for f, key in ((F_OBJ, "obj"), (F_SCORE, "score"), (F_H, "h")):
        assert _close(float(st[f]), last[key], rtol), (what, key, float(st[f]), last[key])


# =====================================================================================================================
# section 2: the persistent kernel against the oracle
# =====================================================================================================================
@pytest.mark.parametrize("K", [1, 30], ids=lambda k: f"K{k}")
@pytest.mark.parametrize("shape", FUSED_SHAPES, ids=_sid)
def test_persistent_kernel_vs_oracle(shape, K, monkeypatch):
    monkeypatch.setenv("DAGMA_MLP_FUSED", "1")
    d, m1, n, s = shape
    model = _start([d, m1, 1], seed=100 * d + m1)
    X = _data(n, d, seed=n + d)
    eq, ok, o, ok_ref = _minimize_both(model, X, K, 2e-3, s, checkpoint=7)
    assert eq._engine.one_kernel
    assert ok is True and ok_ref is True
    assert eq.n_iters == o.n_iters == K
    err = _check_params(model, o, 1e-9, _sid(shape))
    _check_state(eq, o, 1e-9, _sid(shape))
    print(f"{_sid(shape)} K={K}: max rel |d param| = {err:.2e}")


# =====================================================================================================================
# section 3: the launch sequence against the oracle, one evaluation and K steps
# =====================================================================================================================
# (dims, n, s)
SEQ_SHAPES = [
    # [d, m1, 1] on mlp_forward_kernel / mlp_backward_kernel (DAGMA_MLP_FUSED=0)
    ([1, 1, 1], 1, 1.0), ([3, 13, 1], 255, 0.8), ([8, 8, 1], 256, 3.0), ([17, 3, 1], 257, 1.0),
    ([31, 39, 1], 1000, 0.8), ([33, 20, 1], 449, 3.0), ([64, 40, 1], 1000, 1.0), ([5, 9, 1], 1000, 1.0),
    # d > 64: the on-chip inverse up to d = 128, the blocked inverse above
    ([65, 4, 1], 257, 1.0), ([100, 3, 1], 255, 0.8), ([128, 2, 1], 300, 1.0), ([129, 2, 1], 256, 1.0),
    ([200, 2, 1], 1000, 3.0),
    # m1 > 40
    ([4, 41, 1], 257, 1.0), ([9, 64, 1], 1000, 0.8),
    # deeper stacks: a layer of width >= 4 leaves a partial group of three outputs in lc_backward_kernel
    ([5, 3, 1, 1], 255, 1.0), ([5, 4, 2, 1], 1, 1.0), ([5, 2, 3, 1], 256, 0.8), ([5, 3, 4, 1], 257, 1.0),
    ([5, 3, 7, 1], 1000, 3.0),
    ([33, 2, 1, 1], 256, 1.0), ([33, 3, 2, 1], 300, 0.8), ([33, 2, 3, 1], 257, 1.0), ([33, 3, 4, 1], 1000, 1.0),
    ([33, 2, 7, 1], 255, 3.0),
    ([70, 2, 1, 1], 257, 1.0), ([70, 2, 2, 1], 100, 1.0), ([70, 2, 3, 1], 256, 0.8), ([70, 3, 4, 1], 255, 1.0),
    ([70, 2, 7, 1], 1000, 1.0),
    ([7, 5, 4, 3, 1], 257, 1.0), ([9, 2, 7, 5, 1], 1000, 0.8),
    # [d, 1]: x_hat = fc1(x)
    ([1, 1], 1, 1.0), ([6, 1], 257, 1.0), ([65, 1], 1000, 0.8),
]


def _dims_id(dims, n, s):
    return "x".join(str(x) for x in dims) + f"-n{n}-s{s}"


@pytest.mark.parametrize("dims,n,s", SEQ_SHAPES, ids=[_dims_id(*c) for c in SEQ_SHAPES])
def test_launch_sequence_vs_oracle(dims, n, s, monkeypatch):
    from midagma_b200.nonlinear import _MlpEngine, F_MU, F_S, F_LAM1, F_LAM2, F_OBJ, F_SCORE, F_H
    monkeypatch.setenv("DAGMA_MLP_FUSED", "0")
    d = dims[0]
    model = _start(dims, seed=7 * d + len(dims) + dims[1])
    X = _data(n, d, seed=3 * n + d)
    # one evaluation
    o = _oracle(model)
    obj, score, h, grads = o.model.obj_and_grads(X, LAM1, MU, s)
    eng = _MlpEngine(model, torch.from_numpy(X).cuda())
    assert not eng.one_kernel
    sh = eng.state_host
    sh.zero_()
    sh[F_MU], sh[F_S], sh[F_LAM1], sh[F_LAM2] = MU, s, LAM1, LAM2
    eng.state.copy_(sh)
    eng.evaluate(s)
    st, _, halted = eng.pull()
    assert not halted
    for f, ref, key in ((F_OBJ, obj, "obj"), (F_SCORE, score, "score"), (F_H, h, "h")):
        assert _close(float(st[f]), ref, 1e-9), (key, float(st[f]), ref)
    worst = 0.0
    for k, g in eng.grads_scaled().items():
        err = _relmax(g, grads[k].reshape(g.shape))
        worst = max(worst, err)
        assert err <= 1e-9, (k, err)
    # K steps over several launches
    K = 20
    eq, ok, o, ok_ref = _minimize_both(model, X, K, 2e-3, s, checkpoint=6)
    assert ok is True and ok_ref is True and eq.n_iters == o.n_iters == K
    errp = _check_params(model, o, 1e-9, _dims_id(dims, n, s))
    _check_state(eq, o, 1e-9, _dims_id(dims, n, s))
    print(f"{_dims_id(dims, n, s)}: grads {worst:.2e}, params after {K} steps {errp:.2e}")


# =====================================================================================================================
# section 4: halting and the M-matrix boundary
# =====================================================================================================================
def _engines_for(d):
    return ["1", "0"] if d <= 64 else ["0"]


def _infeasible_start(d, m1, seed):
    """A = 3 P with P dense and row-stochastic: det(I - A) ~ 1 - 3 (the other eigenvalues of P are small), so
    |det(I - A)| > 1 and h < 0 at iteration 0."""
    model = _start([d, m1, 1], seed)
    rng = np.random.default_rng(seed)
    P = rng.random((d, d)) + 0.5
    P /= P.sum(axis=1, keepdims=True)
    A = 3.0 * P                                                     # A[i, j] = sum_k w[j, k, i]^2
    w = np.sqrt(A.T[:, None, :] / m1) * rng.choice([-1.0, 1.0], size=(d, m1, d)) * (1 + 0.01 * rng.random((d, m1, d)))
    with torch.no_grad():
        model.fc1.weight.copy_(torch.from_numpy(w.reshape(d * m1, d)))
    return model


@pytest.mark.parametrize("fused", ["1", "0"], ids=["mlp_iter", "launch-seq"])
@pytest.mark.parametrize("d", [2, 17, 33, 64, 70, 129], ids=lambda d: f"d{d}")
def test_infeasible_start(d, fused, monkeypatch):
    if fused not in _engines_for(d):
        pytest.skip("d > 64 runs the launch sequence only")
    monkeypatch.setenv("DAGMA_MLP_FUSED", fused)
    m1, n = 3, 100
    model = _infeasible_start(d, m1, seed=d)
    X = _data(n, d, seed=d)
    assert OracleMLP([d, m1, 1], _params(model)).h_func(1.0) < -1e-6
    before = _params(model)
    eq, ok, o, ok_ref = _minimize_both(model, X, 20, 1e-3, 1.0, checkpoint=5)
    assert eq._engine.one_kernel == (fused == "1")
    assert ok is False and ok_ref is False
    assert eq.n_iters == o.n_iters == 0
    for k, p in model.state_dict().items():
        assert np.array_equal(p.numpy(), before[k]), k


# (d, m1, n, seed, t, lr, K): a start with A = t P (P dense and row-stochastic) and a large lr.  Adam's first steps
# move every weight by about lr, past zero, and the oracle's h turns negative at an iteration k with 3 <= k <= K - 3
# (found with the oracle; the test re-derives k and checks the margins of h on both sides of it)
HALT_CASES = [
    (5, 3, 64, 0, 0.9, 0.2, 20),
    (17, 3, 100, 1, 0.9, 0.1, 20),
    (33, 3, 200, 0, 0.97, 0.1, 20),
    (64, 2, 300, 0, 0.97, 0.05, 20),
    (70, 2, 200, 0, 0.97, 0.05, 20),
]


def _near_boundary_start(d, m1, seed, t):
    model = _start([d, m1, 1], seed)
    rng = np.random.default_rng(seed + 1000)
    P = rng.random((d, d)) + 0.5
    P /= P.sum(axis=1, keepdims=True)
    w = np.sqrt(t * P.T[:, None, :] / m1) * rng.choice([-1.0, 1.0], size=(d, m1, d)) * (1 + 0.01 * rng.random((d, m1, d)))
    with torch.no_grad():
        model.fc1.weight.copy_(torch.from_numpy(w.reshape(d * m1, d)))
    return model


@pytest.mark.parametrize("fused", ["1", "0"], ids=["mlp_iter", "launch-seq"])
@pytest.mark.parametrize("case", HALT_CASES, ids=lambda c: f"d{c[0]}-m{c[1]}-n{c[2]}")
def test_halt_inside_a_launch(case, fused, monkeypatch):
    d, m1, n, seed, t, lr, K = case
    if fused not in _engines_for(d):
        pytest.skip("d > 64 runs the launch sequence only")
    monkeypatch.setenv("DAGMA_MLP_FUSED", fused)
    model = _near_boundary_start(d, m1, seed, t)
    X = _data(n, d, seed)
    eq, ok, o, ok_ref = _minimize_both(model, X, K, lr, 1.0, checkpoint=K)      # one launch up to the halt
    k = o.n_iters
    hs = [t["h"] for t in o.trace]
    h_k = OracleMLP([d, m1, 1], o.model.p).h_func(1.0)
    assert ok_ref is False and 3 <= k <= K - 3, (k, hs)
    assert hs[-1] >= 1e-6 and h_k <= -1e-6, (hs[-1], h_k)          # no tie at k - 1 or k
    assert eq._engine.one_kernel == (fused == "1")
    assert ok is False and eq.n_iters == k
    _check_params(model, o, 1e-9, f"halt d={d}")


def _cycle_start(d, m1, seed, prod=1.5):
    """fc1 with a two-node cycle A[0, 1] A[1, 0] = prod and every other entry of A small: det(I - A) ~ 1 - prod < 0
    (outside the M-matrix domain), h = -log|det| ~ log 2 > 0, pivots far from zero."""
    model = _start([d, m1, 1], seed, a_row=0.02)
    w = model.fc1.weight.detach().numpy().reshape(d, m1, d).copy()      # w[j, k, i]: A[i, j] = sum_k w[j, k, i]^2
    w[1, 0, 0] = w[0, 0, 1] = prod ** 0.25
    with torch.no_grad():
        model.fc1.weight.copy_(torch.from_numpy(w.reshape(d * m1, d)))
    return model


@pytest.mark.parametrize("d", [5, 33, 70, 129], ids=lambda d: f"d{d}")
def test_outside_domain_with_positive_h(d, monkeypatch):
    """The reference halts only when h < 0 (nonlinear.py:215-217) and h takes log |det|: outside the M-matrix domain
    with |det(sI - A)| < s^d it keeps stepping with M^-1.  d <= 64: mlp_iter; 70: small_inv; 129: blocked inverse."""
    monkeypatch.setenv("DAGMA_MLP_FUSED", "1")
    m1, n, K = 3, 200, 20
    model = _cycle_start(d, m1, seed=d)
    X = _data(n, d, seed=d + 1)
    o0 = OracleMLP([d, m1, 1], _params(model))
    sign, _ = np.linalg.slogdet(np.eye(d) - o0.adj_sq())
    assert sign < 0 and o0.h_func(1.0) > 0.3
    eq, ok, o, ok_ref = _minimize_both(model, X, K, 1e-3, 1.0, checkpoint=7)
    assert eq._engine.one_kernel == (d <= 64)
    hs = np.array([t["h"] for t in o.trace])
    assert ok_ref is True and hs.min() > 1e-3                    # the reference steps through: no tie with h = 0
    assert ok is True and eq.n_iters == o.n_iters == K
    _check_params(model, o, 1e-9, f"cycle d={d}")
    _check_state(eq, o, 1e-9, f"cycle d={d}")


# =====================================================================================================================
# section 5: split launches, ExponentialLR, short fits
# =====================================================================================================================
@pytest.mark.parametrize("d,m1,n", [(9, 40, 160), (33, 7, 1200), (64, 40, 1000)], ids=["d9-m40", "d33-m7", "d64-m40"])
def test_split_launches_bit_identical(d, m1, n, monkeypatch):
    """Every sum of the persistent kernel has a fixed order: where the launches end changes no bit."""
    from midagma_b200.nonlinear import DagmaNonlinear, _MlpEngine, F_MU, F_S, F_LR, F_LAM1, F_LAM2, F_B1, F_B2, F_GAMMA
    monkeypatch.setenv("DAGMA_MLP_FUSED", "1")
    K = 25
    X = torch.from_numpy(_data(n, d, seed=d)).cuda()
    out = []
    for ck in (1, 7, K):
        model = _start([d, m1, 1], seed=d)
        eq = DagmaNonlinear(model)
        eq.X, eq.checkpoint = X, ck
        assert eq.minimize(K, 2e-3, LAM1, LAM2, MU, 1.0, tol=0.0) is True and eq.n_iters == K
        assert eq._engine.one_kernel
        out.append(torch.cat([p.reshape(-1) for p in model.state_dict().values()]).numpy())
    assert np.array_equal(out[0], out[1]) and np.array_equal(out[0], out[2])
    res = []
    for split in ((10, 15), (25,)):
        eng = _MlpEngine(_start([d, m1, 1], seed=d), X)
        sh = eng.state_host
        sh.zero_()
        for f, val in ((F_MU, MU), (F_S, 1.0), (F_LR, 2e-3), (F_LAM1, LAM1), (F_LAM2, LAM2), (F_B1, 0.99),
                       (F_B2, 0.999), (F_GAMMA, 1.0)):
            sh[f] = val
        eng.state.copy_(sh)
        for a in split:
            eng.replay(1.0, a)
        st, step, halted = eng.pull()
        assert step == K and not halted
        res.append((eng.theta.cpu().numpy(), eng.m.cpu().numpy(), eng.v.cpu().numpy()))
    for a, b in zip(*res):
        assert np.array_equal(a, b)
    assert np.array_equal(res[0][0], out[0])


@pytest.mark.parametrize("dims,fused", [([5, 4, 1], "1"), ([6, 3, 4, 1], "0")], ids=["mlp_iter-d5", "deep-d6"])
def test_exponential_lr_inside_launches(dims, fused, monkeypatch):
    """2100 iterations, checkpoint = 700: the decays after iterations 1000 and 2000 fall inside launches."""
    from midagma_b200.nonlinear import F_LR
    monkeypatch.setenv("DAGMA_MLP_FUSED", fused)
    d, n, K, lr = dims[0], 64, 2100, 1e-3
    model = _start(dims, seed=11)
    X = _data(n, d, seed=12)
    eq, ok, o, ok_ref = _minimize_both(model, X, K, lr, 1.0, checkpoint=700, lr_decay=True)
    assert eq._engine.one_kernel == (fused == "1")
    assert ok is True and ok_ref is True and eq.n_iters == o.n_iters == K
    lr_ref = lr
    for i in range(K):                                           # the oracle's schedule (ExponentialLR(gamma = .8))
        if (i + 1) % 1000 == 0:
            lr_ref *= 0.8
    st, _, _ = eq._engine.pull()
    assert float(st[F_LR]) == lr_ref
    _check_params(model, o, 1e-8, f"lr decay {dims}")


class _RecordingOracle(OracleNonlinear):
    """OracleNonlinear.fit that keeps (lr, s, success, lr_decay) of every minimize call, as DagmaNonlinear does."""

    def __init__(self, model):
        super().__init__(model)
        self.minimize_calls = []

    def minimize(self, X, max_iter, lr, lambda1, lambda2, mu, s, lr_decay=False, tol=1e-6, checkpoint=1000):
        ok = super().minimize(X, max_iter, lr, lambda1, lambda2, mu, s, lr_decay, tol, checkpoint)
        self.minimize_calls.append((float(lr), float(s), int(bool(ok)), int(bool(lr_decay))))
        return ok


FIT_CASES = [([17, 3, 1], 300), ([64, 40, 1], 1000), ([70, 4, 1], 200), ([6, 3, 4, 1], 100)]


@pytest.mark.parametrize("dims,n", FIT_CASES, ids=["x".join(map(str, c[0])) for c in FIT_CASES])
def test_short_fit_vs_oracle(dims, n):
    from midagma_b200.nonlinear import DagmaNonlinear
    d = dims[0]
    model = _start(dims, seed=21 + d)
    X = _data(n, d, seed=22 + d)
    kw = dict(lambda1=LAM1, lambda2=LAM2, T=2, warm_iter=40, max_iter=60, lr=2e-3, checkpoint=15, s=[1.0, 0.9])
    o = _RecordingOracle(OracleMLP(dims, _params(model)))
    W_ref = o.fit(X, **kw)
    eq = DagmaNonlinear(model)
    W = eq.fit(X, **kw)
    assert eq.minimize_calls == o.minimize_calls
    assert np.array_equal(W != 0, W_ref != 0)
    err = np.abs(model.fc1_to_adj() - o.model.fc1_to_adj()).max()
    assert err <= 1e-6, err
    print(f"fit {dims}: max |d W_raw| = {err:.2e}")


# =====================================================================================================================
# section 6: the public surface at scale
# =====================================================================================================================
SURFACE = [([1, 1, 1], 1), ([17, 9, 1], 463), ([64, 40, 1], 1000), ([129, 2, 1], 256), ([9, 2, 7, 5, 1], 1000),
           ([65, 1], 300), ([33, 3, 4, 1], 257)]


@pytest.mark.parametrize("dims,n", SURFACE, ids=["x".join(map(str, c[0])) + f"-n{c[1]}" for c in SURFACE])
def test_public_surface_vs_oracle(dims, n):
    from midagma_b200.nonlinear import DagmaNonlinear
    d = dims[0]
    model = _start(dims, seed=31 + d)
    X = _data(n, d, seed=32 + d)
    om = OracleMLP(dims, _params(model))
    assert _relmax(model.forward(torch.from_numpy(X)).numpy(), om.forward(X)) <= 1e-12
    for s in (1.0, 0.8, 3.0):
        assert _close(model.h_func(s).item(), om.h_func(s), 1e-12), s
    assert _relmax(model.fc1_to_adj(), om.fc1_to_adj()) <= 1e-12
    assert _close(model.fc1_l1_reg().item(), om.fc1_l1_reg(), 1e-12)
    Y = X + 0.1 * _data(n, d, seed=33 + d)
    ref = 0.5 * d * np.log(((Y - X) ** 2).sum() / n)
    got = DagmaNonlinear(model).log_mse_loss(torch.from_numpy(Y), torch.from_numpy(X)).item()
    assert _close(got, ref, 1e-12)


def test_log_mse_loss_many_elements():
    """more elements than the 592 x 256 threads of sumsq_diff_kernel: its grid-stride loop runs several passes"""
    from midagma_b200.nonlinear import DagmaNonlinear
    n, d = 2000, 100
    X, Y = _data(n, d, seed=1), _data(n, d, seed=2)
    assert n * d > 592 * 256
    ref = 0.5 * d * np.log(((Y - X) ** 2).sum() / n)
    got = DagmaNonlinear(_start([d, 1], seed=1)).log_mse_loss(torch.from_numpy(Y), torch.from_numpy(X)).item()
    assert _close(got, ref, 1e-12)


@pytest.mark.parametrize("bias", [True, False], ids=["bias", "no-bias"])
@pytest.mark.parametrize("n,d,m1,m2", [(7000, 100, 4, 1), (2100, 100, 4, 3)], ids=["m2-1", "m2-3"])
def test_locally_connected_grid_stride(n, d, m1, m2, bias):
    """n d m2 > 2368 x 256: the grid-stride loop of locally_connected_kernel runs more than one pass"""
    from midagma_b200.nonlinear import LocallyConnected
    assert n * d * m2 > 2368 * 256
    torch.manual_seed(m2)
    lc = LocallyConnected(d, m1, m2, bias=bias)
    x = torch.randn(n, d, m1, dtype=torch.float64)
    ref = np.einsum("njk,jkm->njm", x.numpy(), lc.weight.detach().numpy())
    if bias:
        ref = ref + lc.bias.detach().numpy()
    assert _relmax(lc(x).numpy(), ref) <= 1e-12
