"""Argument handling of ``fit_batch`` / ``minimize_batch(trek_reg=...)`` that needs no GPU: every regulariser is
validated before a device is looked for, with the errors ``DagmaLinear(trek_reg=...)`` raises, and
``fit_batch_sharded`` hands each rank the regularisers of its own problems."""
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp


def _pst(**kw):
    from midagma_b200.notreks import PSTRegularizer
    return PSTRegularizer(I=kw.pop("I", [(0, 1)]), seq=kw.pop("seq", "inv"), weight=kw.pop("weight", 0.5), **kw)


BAD = [
    lambda: _pst(seq="cos"),
    lambda: _pst(kwargs={"agg": "median"}),
    lambda: _pst(kwargs={"agg": "none"}),
    lambda: _pst(kwargs={"eps_inv": -1.0}),
    lambda: _pst(kwargs={"bogus": 1}),
    lambda: _pst(I=[(0, 1, 2)]),
    lambda: _pst(name="nope"),
]


@pytest.mark.parametrize("k", range(len(BAD)))
@pytest.mark.parametrize("who", ["fit_batch", "minimize_batch"])
def test_bad_regulariser_raises_before_the_device(k, who):
    """The same exception type and message as the per-problem class, shared or as one entry of a per-problem list."""
    from midagma_b200 import DagmaLinear, fit_batch, minimize_batch
    reg = BAD[k]()
    with pytest.raises(Exception) as want:
        DagmaLinear("l2", trek_reg=reg)
    d, batch = 4, 3
    for tr in (reg, [None, reg, None]):
        with pytest.raises(want.type) as got:
            if who == "fit_batch":
                fit_batch(cov=np.tile(np.eye(d), (batch, 1, 1)), trek_reg=tr)
            else:
                minimize_batch(np.zeros((batch, d, d)), np.tile(np.eye(d), (batch, 1, 1)), 0.02, 1.0, 10, 1.0, 3e-4,
                               trek_reg=tr)
        assert str(got.value) == str(want.value)


@pytest.mark.parametrize("n", [2, 4])
def test_per_problem_list_of_wrong_length(n):
    from midagma_b200 import fit_batch, minimize_batch
    regs = [_pst()] * n
    with pytest.raises(ValueError, match="trek_reg has"):
        fit_batch(np.zeros((3, 10, 4)), trek_reg=regs)
    with pytest.raises(ValueError, match="trek_reg has"):
        minimize_batch(np.zeros((3, 4, 4)), np.zeros((3, 4, 4)), 0.02, 1.0, 10, 1.0, 3e-4, trek_reg=regs)


def test_pair_index_out_of_range():
    from midagma_b200 import fit_batch
    with pytest.raises(IndexError, match="pair index"):
        fit_batch(cov=np.tile(np.eye(4), (2, 1, 1)), trek_reg=[_pst(I=[(0, 4)]), None])


def test_plan_of_a_batch():
    """What the on-chip launch is given: CSR pairs (negative indices wrapped), zero weight and no pairs for entries that
    do not change W, and the per-problem route for anything but PST inv with one agg / eps_inv on l2 at d <= 64."""
    from midagma_b200.linear import _trek_batch
    from midagma_b200.notreks import TCCRegularizer
    mean = _pst(I=[(0, 1), (-1, 2)], weight=0.7)
    log = _pst(I=[(0, 1)], mode="log")
    off_ = _pst(I=[(0, 1)], weight=0.0)
    regs, (off, pairs, w, agg, eps) = _trek_batch([mean, None, log, off_, _pst(I=np.zeros((0, 2)))], 5, 4, "l2", "t")
    assert off.tolist() == [0, 2, 2, 2, 2, 2] and pairs.tolist() == [[0, 1], [3, 2]]
    assert w.tolist() == [0.7, 0, 0, 0, 0] and agg == 0 and eps == 1e-8 and regs[1] is None
    assert _trek_batch(None, 3, 4, "l2", "t") is None
    assert _trek_batch([None, log], 2, 4, "l2", "t") is None
    for args in (([mean, _pst(kwargs={"agg": "sum"})], 2, 4, "l2"),
                 ([mean, _pst(kwargs={"eps_inv": 1e-6})], 2, 4, "l2"),
                 ([mean, _pst(seq="exp")], 2, 4, "l2"),
                 ([mean, TCCRegularizer(I=[(0, 1)])], 2, 4, "l2"),
                 (mean, 2, 4, "logistic"),
                 (mean, 2, 65, "l2")):
        regs, onchip = _trek_batch(*args, "t")
        assert onchip is None and len(regs) == 2


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, ws, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=ws)
    from midagma_b200 import parallel
    n_prob, d = 5, 3
    covs = np.stack([np.eye(d) * (p + 1) for p in range(n_prob)])
    regs = [None if p == 2 else _pst(weight=0.1 * (p + 1)) for p in range(n_prob)]
    seen = {}

    def solver(X, lam, cov=None, trek_reg=None, **k):
        for c, tr in zip(cov, trek_reg):
            seen[int(c[0, 0]) - 1] = tr
        return np.stack([c * (0.0 if tr is None else tr.weight) for c, tr in zip(cov, trek_reg)])

    W = parallel.fit_batch_sharded(cov=covs, lambda1=0.02, solver=solver, trek_reg=regs)
    mine = parallel.problem_shard(n_prob, rank, ws)
    assert sorted(seen) == mine.tolist() and all(seen[p] is regs[p] for p in mine)
    want = np.stack([c * (0.0 if tr is None else tr.weight) for c, tr in zip(covs, regs)])
    assert np.array_equal(W, want)
    shared = _pst(weight=0.3)                   # one regulariser for the batch is passed through as it is
    seen.clear()
    parallel.fit_batch_sharded(cov=covs, lambda1=0.02, solver=lambda X, lam, cov=None, trek_reg=None, **k: (
        seen.update(shared_ok=trek_reg is shared) or np.zeros((len(cov), d, d))), trek_reg=shared)
    assert seen["shared_ok"]
    dist.barrier()
    open(os.path.join(out_dir, f"ok{rank}"), "w").close()
    dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_sharded_per_problem_trek_reg(tmp_path):
    ws = 2
    mp.spawn(_worker, args=(ws, _free_port(), str(tmp_path)), nprocs=ws, join=True)
    assert all((tmp_path / f"ok{r}").exists() for r in range(ws))
