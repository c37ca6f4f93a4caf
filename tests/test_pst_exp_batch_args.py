"""Routing of ``fit_batch`` / ``minimize_batch(trek_reg=...)`` with PST ``seq="exp"`` that needs no GPU: which batches the
on-chip exp kernel takes and what it is given, and that the header, the launch-sequence engine and the oracle agree on
the Taylor degree and the number of squarings of the fixed-scaling expm."""
import inspect
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _pst(**kw):
    from midagma_b200.notreks import PSTRegularizer
    return PSTRegularizer(I=kw.pop("I", [(0, 1)]), seq=kw.pop("seq", "exp"), weight=kw.pop("weight", 0.5), **kw)


def test_exp_plan_of_a_batch():
    """CSR pairs (negative indices wrapped), the weight of each problem, no pairs and zero weight for entries that do not
    change W, the shared agg, and no eps_inv (the series has none)."""
    from midagma_b200.linear import _PST_AGGS, _trek_batch
    a = _pst(I=[(0, 1), (-1, 2), (1, 0)], weight=0.7, kwargs={"agg": "lse"})
    b = _pst(I=[(2, 2)], weight=0.1, kwargs={"agg": "lse"})
    log = _pst(I=[(0, 1)], mode="log")
    regs, (off, pairs, w, agg, eps) = _trek_batch([a, None, log, b, _pst(I=np.zeros((0, 2)))], 5, 4, "l2", "t")
    assert off.tolist() == [0, 3, 3, 3, 4, 4] and pairs.tolist() == [[0, 1], [3, 2], [1, 0], [2, 2]]
    assert w.tolist() == [0.7, 0, 0, 0.1, 0] and agg == _PST_AGGS["lse"] and eps is None and regs[1] is None
    assert off.dtype == np.int32 and pairs.dtype == np.int32
    # the default regulariser of the fork is PST exp / mean: shared by the batch
    regs, (off, pairs, w, agg, eps) = _trek_batch(_pst(I=[(0, 3)], weight=0.2), 3, 4, "l2", "t")
    assert off.tolist() == [0, 1, 2, 3] and w.tolist() == [0.2] * 3 and agg == _PST_AGGS["mean"] and eps is None


def test_exp_batch_with_mixed_eps_inv_and_K_log_goes_on_chip():
    """eps_inv and K_log never reach the exp series: problems that differ only in them share one launch."""
    from midagma_b200.linear import _trek_batch
    regs = [_pst(), _pst(kwargs={"eps_inv": 1e-6}), _pst(kwargs={"K_log": 5}), _pst(kwargs={"eps_inv": 0.5, "K_log": 2})]
    _, onchip = _trek_batch(regs, 4, 8, "l2", "t")
    assert onchip is not None and onchip[4] is None and onchip[0].tolist() == [0, 1, 2, 3, 4]


def test_exp_routes_to_the_per_problem_class():
    """A mix of series, a mix of aggregations, the logistic loss and d > 64 run one problem after the other."""
    from midagma_b200.linear import _trek_batch
    from midagma_b200.notreks import TCCRegularizer
    e = _pst(I=[(0, 1)])
    for args in (([e, _pst(seq="inv")], 2, 4, "l2"),
                 ([e, _pst(seq="log")], 2, 4, "l2"),
                 ([e, _pst(kwargs={"agg": "max"})], 2, 4, "l2"),
                 ([e, TCCRegularizer(I=[(0, 1)])], 2, 4, "l2"),
                 (e, 2, 4, "logistic"),
                 (e, 2, 65, "l2")):
        regs, onchip = _trek_batch(*args, "t")
        assert onchip is None and len(regs) == 2
    # inv keeps its own plan: a float eps_inv in the fifth field
    _, onchip = _trek_batch([_pst(seq="inv"), _pst(seq="inv")], 2, 4, "l2", "t")
    assert onchip[4] == 1e-8
    # log / binom alone are not carried on chip either
    for seq in ("log", "binom"):
        assert _trek_batch(_pst(seq=seq), 2, 4, "l2", "t")[1] is None


def _header_define(name):
    src = open(os.path.join(ROOT, "include", "dagma_b200.h")).read()
    m = re.search(rf"#define\s+{name}\s+(\d+)", src)
    assert m, name
    return int(m.group(1))


def test_exp_constants_match_the_header():
    """The on-chip kernel (header), the launch sequence (_pst) and the float64 oracle run the same expm."""
    from midagma_b200 import _pst
    from oracle import notreks_ref
    deg, sq = _header_define("DAGMA_PST_EXP_DEGREE"), _header_define("DAGMA_PST_EXP_SQUARINGS")
    assert (_pst.EXP_DEGREE, _pst.EXP_SQUARINGS) == (deg, sq) == (18, 12)
    sig = inspect.signature(notreks_ref._expm_taylor).parameters
    assert (sig["degree"].default, sig["squarings"].default) == (deg, sq)
