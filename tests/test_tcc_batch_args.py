"""Routing of ``fit_batch`` / ``minimize_batch(trek_reg=...)`` with spectral TCC regularisers that needs no GPU: which
batches the on-chip TCC kernel takes and what it is given, that the header and ``_tcc`` run the same Perron schedule,
and the warning of the chunk cap."""
import os
import re
import warnings

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _tcc(**kw):
    from midagma_b200.notreks import TCCRegularizer
    return TCCRegularizer(I=kw.pop("I", [(0, 1)]), weight=kw.pop("weight", 0.5), **kw)


def test_tcc_plan_of_a_batch():
    """CSR pairs (negative indices wrapped, duplicates kept so m counts them), the per-problem weight / w / eps / n_iter
    and flags of the default dispatch (approx_trek_graph, eig), and no pairs for entries that do not change W."""
    from midagma_b200.linear import _TccBatch, _trek_batch
    from midagma_b200.notreks import PSTRegularizer
    a = _tcc(I=[(0, 1), (-1, 2), (0, 1)], weight=0.7, w=0.3, eps=1e-10, n_iter=7)
    b = _tcc(I=[(2, 2)], weight=0.1)
    log = _tcc(I=[(0, 1)], mode="log")
    off_ = _tcc(I=[(0, 1)], weight=0.0)
    regs, plan = _trek_batch([a, None, log, b, _tcc(I=np.zeros((0, 2))), off_], 6, 4, "l2", "t")
    assert isinstance(plan, _TccBatch) and regs[1] is None and regs[0] is a
    assert plan.pair_off.tolist() == [0, 3, 3, 3, 4, 4, 4]
    assert plan.pairs.tolist() == [[0, 1], [3, 2], [0, 1], [2, 2]]
    assert plan.pair_off.dtype == np.int32 and plan.pairs.dtype == np.int32
    assert np.diff(plan.pair_off).tolist() == [3, 0, 0, 1, 0, 0]          # m of each problem, the duplicate counted
    assert plan.weight.tolist() == [0.7, 0, 0, 0.1, 0, 0]
    assert plan.w[0] == 0.3 and plan.w[3] == 1.0
    assert plan.eps[0] == 1e-10 and plan.eps[3] == 1e-12
    assert plan.n_iter[0] == 7 and plan.n_iter[3] == 10
    assert plan.flags.tolist() == [0] * 6 and plan.n_iter.dtype == np.int32 and plan.flags.dtype == np.int32
    # a PST-only batch keeps its five-field plan
    _, pst = _trek_batch(PSTRegularizer(I=[(0, 1)], seq="inv", weight=0.1), 2, 4, "l2", "t")
    assert not isinstance(pst, _TccBatch) and len(pst) == 5


def test_tcc_no_op_and_out_of_range_entries():
    """A batch whose TCC terms all leave W alone has no trek plan; an index outside [-d, d) is an IndexError before any
    device is needed."""
    from midagma_b200 import fit_batch, minimize_batch
    from midagma_b200.linear import _trek_batch
    assert _trek_batch([None, _tcc(mode="log"), _tcc(weight=0.0), _tcc(I=[])], 4, 4, "l2", "t") is None
    with pytest.raises(IndexError, match="pair index"):
        _trek_batch([_tcc(I=[(0, 4)]), None], 2, 4, "l2", "t")
    with pytest.raises(IndexError, match="pair index"):
        _trek_batch([_tcc(I=[(-5, 1)])], 1, 4, "l2", "t")
    with pytest.raises(IndexError, match="pair index"):
        minimize_batch(np.zeros((2, 4, 4)), np.tile(np.eye(4), (2, 1, 1)), 0.02, 1.0, 10, 1.0, 3e-4,
                       trek_reg=[None, _tcc(I=[(1, 9)])])
    with pytest.raises(IndexError, match="pair index"):
        fit_batch(cov=np.tile(np.eye(4), (2, 1, 1)), trek_reg=_tcc(I=[(0, 4)]))


def test_forward_flag_switches_version_and_method(monkeypatch):
    """With notreks.FORWARD_TCC_CONFIG the regulariser's own version / method reach the kernel, per problem; without
    it every problem runs the reference's dispatch (approx_trek_graph, eig) whatever it says."""
    from midagma_b200 import notreks
    from midagma_b200.linear import _TCC_DAG_LEARNING, _TCC_POWER, _trek_batch
    regs = [_tcc(version="DAG_learning", method="power", n_iter=5), _tcc(version="approx_trek_graph", method="power"),
            _tcc(version="DAG_learning", method="eig_numpy"), _tcc(method="eig_troch"), _tcc(method="eig_torch")]
    monkeypatch.setattr(notreks, "FORWARD_TCC_CONFIG", False)
    assert _trek_batch(regs, 5, 4, "l2", "t")[1].flags.tolist() == [0] * 5
    monkeypatch.setattr(notreks, "FORWARD_TCC_CONFIG", True)
    plan = _trek_batch(regs, 5, 4, "l2", "t")[1]
    assert plan.flags.tolist() == [_TCC_POWER | _TCC_DAG_LEARNING, _TCC_POWER, _TCC_DAG_LEARNING, 0, 0]
    assert plan.n_iter.tolist()[:2] == [5, 10]


def test_tcc_routes_to_the_per_problem_class(monkeypatch):
    """exact_trek_graph (a second Perron pair), logdet, the logistic loss, d > 64 and a PST + TCC mix run one problem
    after the other."""
    from midagma_b200 import notreks
    from midagma_b200.linear import _trek_batch
    from midagma_b200.notreks import PSTRegularizer
    t = _tcc()
    for args in ((t, 2, 4, "logistic"),
                 (t, 2, 65, "l2"),
                 ([t, PSTRegularizer(I=[(0, 1)], seq="inv", weight=0.1)], 2, 4, "l2"),
                 ([t, PSTRegularizer(I=[(0, 1)], seq="exp", weight=0.1)], 2, 4, "l2")):
        regs, onchip = _trek_batch(*args, "t")
        assert onchip is None and len(regs) == 2
    monkeypatch.setattr(notreks, "FORWARD_TCC_CONFIG", True)
    for other in (_tcc(version="exact_trek_graph", method="power"), _tcc(cycle_penalty="logdet",
                                                                           version="DAG_learning")):
        regs, onchip = _trek_batch([t, other], 2, 4, "l2", "t")
        assert onchip is None and regs[1] is other


def _header_value(name):
    src = open(os.path.join(ROOT, "include", "dagma_b200.h")).read()
    m = re.search(rf"#define\s+{name}\s+([0-9.eE+-]+)", src)
    assert m, name
    return float(m.group(1))


def test_tcc_constants_match_the_header():
    """The on-chip kernel (header) and PerronSolver.converged run the same schedule; the status bit and flags agree."""
    from midagma_b200 import _lib, _tcc, linear
    assert _header_value("DAGMA_TCC_EIG_WARMUP") == _tcc.EIG_WARMUP == 8
    assert _header_value("DAGMA_TCC_EIG_CHUNK") == _tcc.EIG_CHUNK
    assert _header_value("DAGMA_TCC_EIG_MAX_CHUNKS") == _tcc.EIG_MAX_CHUNKS
    assert _header_value("DAGMA_TCC_EIG_TOL") == _tcc.EIG_TOL
    assert _header_value("DAGMA_TCC_EIG_SHIFT") == _tcc.EIG_SHIFT == 0.25
    assert _header_value("DAGMA_TCC_EIG_NILPOTENT") == _tcc.EIG_NILPOTENT
    assert _header_value("DAGMA_ST_PERRON_CAP") == _lib.ST_PERRON_CAP
    assert (_header_value("DAGMA_TCC_POWER"), _header_value("DAGMA_TCC_DAG_LEARNING")) == (
        linear._TCC_POWER, linear._TCC_DAG_LEARNING)


def test_perron_cap_warns_once_per_call():
    """A status with the cap bit on several problems gives exactly one RuntimeWarning; without it, none."""
    from midagma_b200 import _lib
    from midagma_b200.linear import _warn_perron_cap
    cap = _lib.ST_PERRON_CAP
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        _warn_perron_cap(torch.tensor([cap, 0, cap | _lib.ST_OUT_OF_DOMAIN, _lib.ST_LR_UNDERFLOW], dtype=torch.int32))
    assert len(rec) == 1 and issubclass(rec[0].category, RuntimeWarning) and "2 problem(s)" in str(rec[0].message)
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        _warn_perron_cap(torch.tensor([0, _lib.ST_OUT_OF_DOMAIN, _lib.ST_RETRY_LIMIT], dtype=torch.int32))
    assert not rec
