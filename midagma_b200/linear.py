"""Drop-in ``DagmaLinear`` on the B200 kernels (reference: src/dagma/linear.py).

Same constructor, methods, defaults, return values and side effects as the
reference class (numpy in / numpy out, ``minimize`` mutates and returns its ``W``,
``fit`` centres the caller's ``X`` in place for the l2 loss, failure is a return
flag).  All arithmetic is done by libdagma_b200.so:

* d <= 64, l2 loss: one persistent CTA runs whole ``minimize`` stages -- and for
  ``fit`` the whole path-following loop including retries -- in one kernel launch
  (``dagma_linear_fit_small_f64``).
* larger d and the logistic loss: the multi-CTA path in ``_large.py`` (blocked
  inverse + score GEMMs + fused Adam), one CUDA-graph replay per inner iteration.

``fit_batch`` / ``minimize_batch`` are the batched entry points (independent
problems: seeds, lambda1 grids, bootstrap replicates) that the reference can only
express as a Python loop over ``DagmaLinear.fit``.
"""
from __future__ import annotations

import ctypes as C
import time
import typing

import numpy as np
import torch

from . import _lib

__all__ = ["DagmaLinear", "fit_batch", "minimize_batch"]


def _mu_schedule(mu_init: float, mu_factor: float, T: int) -> list:
    mus, mu = [], mu_init
    for _ in range(int(T)):
        mus.append(mu)
        mu *= mu_factor                     # repeated multiplication (linear.py:453, Q7)
    return mus


def _edge_mask(edges, d: int, device) -> typing.Optional[torch.Tensor]:
    if edges is None:
        return None
    m = np.zeros((d, d), dtype=np.uint8)
    r, c = zip(*edges)
    m[list(r), list(c)] = 1
    return torch.from_numpy(m).to(device)


class SmallFitResult(typing.NamedTuple):
    W: torch.Tensor             # [batch, d, d] raw (un-thresholded) result, device
    status: torch.Tensor        # [batch] int32
    stage_stats: torch.Tensor   # [batch, n_stages, 8]
    final: torch.Tensor         # [batch, 2] (h(W, s=1), score(W))
    ckpt_log: typing.Optional[torch.Tensor]
    ckpt_count: typing.Optional[torch.Tensor]
    ckpt_diag: typing.Optional[torch.Tensor] = None   # [batch, cap, 11] telemetry rows (include/dagma_b200.h)


def _run_small(cov: torch.Tensor, W: torch.Tensor, lambda1: torch.Tensor, mus, ss, iters, *, lr, tol,
               beta1, beta2, checkpoint, retry, mask_exc=None, mask_inc=None, ckpt_log_cap=0,
               want_final=True, want_diag=False, X=None, pst=None, tcc=None) -> SmallFitResult:
    """Launch ``dagma_linear_fit_small_f64`` on device tensors (W is updated in place).  With ``X`` ([batch, n, d]
    device tensor; ``cov`` = its un-centred X^T X / n) the logistic loss: ``dagma_linear_fit_small_logistic_f64``.
    With ``pst`` (a ``_PstBatch``) the l2 loss plus the PST term: ``dagma_linear_fit_small_pst_f64`` for ``inv``,
    ``dagma_linear_fit_small_pst_exp_f64`` for ``exp``.  With ``tcc`` (a ``_TccBatch`` of device tensors) the l2 loss
    plus the spectral TCC term: ``dagma_linear_fit_small_tcc_f64``; the power steps of each problem are added to
    ``tcc.perron_steps``."""
    _lib.require_device()
    lib = _lib.load()
    batch, d, _ = cov.shape
    T = len(mus)
    if T > _lib.MAX_STAGES:
        return _run_small_chunked(cov, W, lambda1, mus, ss, iters, lr=lr, tol=tol, beta1=beta1, beta2=beta2,
                                  checkpoint=checkpoint, retry=retry, mask_exc=mask_exc, mask_inc=mask_inc,
                                  ckpt_log_cap=ckpt_log_cap, want_final=want_final, want_diag=want_diag, X=X, pst=pst,
                                  tcc=tcc)
    assert cov.is_cuda and W.is_cuda and cov.dtype == torch.float64 and W.dtype == torch.float64
    assert cov.is_contiguous() and W.is_contiguous() and lambda1.is_contiguous()
    dev = cov.device
    a = _lib.SmallFitArgs()
    a.batch, a.d, a.n_stages, a.checkpoint = batch, d, T, int(checkpoint)
    a.retry_on_fail, a.ckpt_log_cap = int(bool(retry)), int(ckpt_log_cap)
    a.lr, a.tol, a.beta1, a.beta2 = float(lr), float(tol), float(beta1), float(beta2)
    for t in range(T):
        a.mu[t], a.s[t], a.iters[t] = float(mus[t]), float(ss[t]), int(iters[t])
    status = torch.zeros(batch, dtype=torch.int32, device=dev)
    stats = torch.zeros(batch, max(T, 1), 8, dtype=torch.float64, device=dev)
    final = torch.zeros(batch, 2, dtype=torch.float64, device=dev)
    counter = torch.zeros(16, dtype=torch.int32, device=dev)
    log = cnt = diag = None
    if ckpt_log_cap > 0:
        log = torch.zeros(batch, ckpt_log_cap, 6, dtype=torch.float64, device=dev)
        cnt = torch.zeros(batch, dtype=torch.int32, device=dev)
        if want_diag:
            diag = torch.zeros(batch, ckpt_log_cap, _lib.DIAG_COLS, dtype=torch.float64, device=dev)
    a.ckpt_diag = diag.data_ptr() if diag is not None else None
    a.cov, a.lambda1, a.w = cov.data_ptr(), lambda1.data_ptr(), W.data_ptr()
    a.mask_exc = mask_exc.data_ptr() if mask_exc is not None else None
    a.mask_inc = mask_inc.data_ptr() if mask_inc is not None else None
    a.status, a.stage_stats = status.data_ptr(), stats.data_ptr()
    a.final = final.data_ptr() if want_final else None
    a.ckpt_log = log.data_ptr() if log is not None else None
    a.ckpt_count = cnt.data_ptr() if cnt is not None else None
    a.work_counter = counter.data_ptr()
    if tcc is not None:
        assert X is None and pst is None and tcc.pair_off.shape[0] == batch + 1
        steps = torch.zeros(batch, dtype=torch.int64, device=dev)
        _lib.check(lib.dagma_linear_fit_small_tcc_f64(_lib.stream_ptr(), C.byref(a), tcc.pair_off.data_ptr(),
                                                      tcc.pairs.data_ptr(), tcc.weight.data_ptr(), tcc.w.data_ptr(),
                                                      tcc.eps.data_ptr(), tcc.n_iter.data_ptr(), tcc.flags.data_ptr(),
                                                      steps.data_ptr()), "dagma_linear_fit_small_tcc_f64")
        tcc.perron_steps.add_(steps)
    elif pst is not None and pst.eps_inv is None:
        assert X is None and pst.pair_off.shape[0] == batch + 1
        _lib.check(lib.dagma_linear_fit_small_pst_exp_f64(_lib.stream_ptr(), C.byref(a), pst.pair_off.data_ptr(),
                                                          pst.pairs.data_ptr(), pst.weight.data_ptr(), pst.agg),
                   "dagma_linear_fit_small_pst_exp_f64")
    elif pst is not None:
        assert X is None and pst.pair_off.shape[0] == batch + 1
        _lib.check(lib.dagma_linear_fit_small_pst_f64(_lib.stream_ptr(), C.byref(a), pst.pair_off.data_ptr(),
                                                      pst.pairs.data_ptr(), pst.weight.data_ptr(), pst.agg,
                                                      pst.eps_inv), "dagma_linear_fit_small_pst_f64")
    elif X is None:
        _lib.check(lib.dagma_linear_fit_small_f64(_lib.stream_ptr(), C.byref(a)), "dagma_linear_fit_small_f64")
    else:
        assert X.is_cuda and X.dtype == torch.float64 and X.is_contiguous() and X.shape[0] == batch and X.shape[2] == d
        _lib.check(lib.dagma_linear_fit_small_logistic_f64(_lib.stream_ptr(), C.byref(a), X.shape[1], X.data_ptr()),
                   "dagma_linear_fit_small_logistic_f64")
    return SmallFitResult(W, status, stats, final, log, cnt, diag)


def _run_small_chunked(cov, W, lambda1, mus, ss, iters, *, ckpt_log_cap=0, want_final=True, **kw) -> SmallFitResult:
    """More stages than one launch carries (DAGMA_MAX_STAGES): the stages of ``fit`` only communicate through W
    (linear.py:441-453), so the schedule is cut into consecutive launches; the final h / score come from the last."""
    T, step = len(mus), _lib.MAX_STAGES
    parts = []
    for lo in range(0, T, step):
        hi = min(lo + step, T)
        parts.append(_run_small(cov, W, lambda1, mus[lo:hi], ss[lo:hi], iters[lo:hi], ckpt_log_cap=ckpt_log_cap,
                                want_final=want_final and hi == T, **kw))
    status = parts[0].status.clone()
    for p in parts[1:]:
        status |= p.status
    stats = torch.cat([p.stage_stats for p in parts], dim=1)
    log = cnt = diag = None
    if ckpt_log_cap > 0:
        # rows keep their launch-local stage index; shift it to the global one and pack the launches back to back
        batch = cov.shape[0]
        log = torch.zeros(batch, ckpt_log_cap * len(parts), 6, dtype=torch.float64, device=cov.device)
        cnt = torch.zeros(batch, dtype=torch.int32, device=cov.device)
        if parts[0].ckpt_diag is not None:
            diag = torch.zeros(batch, ckpt_log_cap * len(parts), _lib.DIAG_COLS, dtype=torch.float64, device=cov.device)
        for k, p in enumerate(parts):
            rows = p.ckpt_log.clone()
            rows[:, :, 0] += k * step
            for b in range(batch):
                n, c = int(p.ckpt_count[b]), int(cnt[b])
                log[b, c:c + n] = rows[b, :n]
                if diag is not None:
                    diag[b, c:c + n] = p.ckpt_diag[b, :n]
                cnt[b] = c + n
    return SmallFitResult(W, status, stats, parts[-1].final, log, cnt, diag)


def center_cov(X: torch.Tensor, center: bool) -> torch.Tensor:
    """cov = X^T X / n on device ([batch, n, d] -> [batch, d, d]); X centred in place if asked."""
    _lib.require_device()
    assert X.is_cuda and X.dtype == torch.float64 and X.is_contiguous() and X.dim() == 3
    batch, n, d = X.shape
    cov = torch.empty(batch, d, d, dtype=torch.float64, device=X.device)
    _lib.check(_lib.load().dagma_center_cov_f64(_lib.stream_ptr(), batch, n, d, X.data_ptr(), int(center),
                                                cov.data_ptr()), "dagma_center_cov_f64")
    return cov


def logdet_inv(A: torch.Tensor, s: float = 1.0, square_input: bool = True, want_inv=False, want_grad=True):
    """Fused slogdet + inverse of ``sI - A∘A`` (or ``sI - A``) for a batch ``[b, d, d]`` on device.

    Returns dict(logabsdet, h, minv, grad, min_entry, info) of device tensors."""
    _lib.require_device()
    assert A.is_cuda and A.dtype == torch.float64 and A.dim() == 3 and A.is_contiguous()
    b, d, _ = A.shape
    dev = A.device
    out = {
        "logabsdet": torch.empty(b, dtype=torch.float64, device=dev),
        "h": torch.empty(b, dtype=torch.float64, device=dev),
        "minv": torch.empty(b, d, d, dtype=torch.float64, device=dev) if want_inv else None,
        "grad": torch.empty(b, d, d, dtype=torch.float64, device=dev) if want_grad else None,
        "min_entry": torch.empty(b, dtype=torch.float64, device=dev),
        "info": torch.empty(b, dtype=torch.int32, device=dev),
    }
    ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
    _lib.check(_lib.load().dagma_logdet_inv_f64(
        _lib.stream_ptr(), b, d, float(s), A.data_ptr(), d, int(bool(square_input)),
        ptr(out["logabsdet"]), ptr(out["h"]), ptr(out["minv"]), ptr(out["grad"]), d,
        ptr(out["min_entry"]), ptr(out["info"])), "dagma_logdet_inv_f64")
    return out


# =============================================================================
# batched entry points
# =============================================================================
def _warn_retry_limit(status: torch.Tensor) -> None:
    """The reference keeps retrying a failing stage for ever (linear.py:446-451); the kernels give up after 64
    retries of one stage and say so."""
    n = int(((status & _lib.ST_RETRY_LIMIT) != 0).sum().item())
    if n:
        import warnings
        warnings.warn(f"{n} problem(s) hit the stage-retry limit (64 retries with lr/2, s+0.1): their W is the last "
                      "restart point, not a converged solution", RuntimeWarning, stacklevel=3)


def _warn_perron_cap(status: torch.Tensor) -> None:
    """One warning per call when a TCC problem's Perron iteration hit the chunk cap, as ``_tcc.PerronSolver.converged``
    warns for one solve."""
    n = int(((status & _lib.ST_PERRON_CAP) != 0).sum().item())
    if n:
        import warnings
        warnings.warn(f"{n} problem(s): the Perron iteration of the TCC penalty did not converge in some evaluation "
                      "(Perron root not simple / tiny spectral gap): the vectors are the last iterate", RuntimeWarning,
                      stacklevel=3)



def _as_dev(x, device, dtype=torch.float64) -> torch.Tensor:
    if isinstance(x, torch.Tensor):
        return x.to(device=device, dtype=dtype).contiguous()
    a = np.ascontiguousarray(x)
    if not a.flags.writeable:            # e.g. a broadcast view: torch refuses to alias read-only memory quietly
        a = a.copy()
    return torch.as_tensor(a, dtype=dtype).to(device)


def _lam_dev(lambda1, batch: int, device) -> torch.Tensor:
    if isinstance(lambda1, torch.Tensor):
        lam = lambda1.to(device=device, dtype=torch.float64).reshape(-1)
        return (lam.expand(batch) if lam.numel() == 1 else lam).contiguous()
    return _as_dev(np.broadcast_to(np.asarray(lambda1, dtype=np.float64), (batch,)), device)


_LOSSES = ("l2", "logistic")


def _logistic_inputs(loss_type, X, who: str) -> bool:
    """Argument checks of the batched entry points that need no device; True for the logistic loss."""
    if loss_type not in _LOSSES:
        raise ValueError(f"{who}: loss_type should be one of {list(_LOSSES)}, got {loss_type!r}")
    if loss_type == "l2":
        return False
    if X is None:
        raise ValueError(f"{who}(loss_type='logistic') needs the data X [batch, n, d]: the logistic score is not a "
                         "function of the covariance")
    if np.ndim(X) != 3:
        raise ValueError(f"{who}(loss_type='logistic'): X must be [batch, n, d], got shape {tuple(np.shape(X))}")
    return True


def _batch_masks(exclude_edges, include_edges, d, device):
    """Edge lists shared by the whole batch -> the [d, d] byte masks of the kernels.  Same acceptance rule as the
    reference (linear.py:416-426, Q5): anything but a tuple of 2-tuples is silently ignored."""
    out = []
    for edges in (exclude_edges, include_edges):
        ok = (edges is not None and type(edges) is tuple and len(edges) > 0 and type(edges[0]) is tuple
              and bool(np.all(np.array([len(e) for e in edges]) == 2)))
        out.append(_edge_mask(edges, d, device) if ok else None)
    return out


_PST_AGGS = {"mean": 0, "sum": 1, "max": 2, "lse": 3}       # DAGMA_PST_* of include/dagma_b200.h


class _PstBatch(typing.NamedTuple):
    """Pair sets of an on-chip PST batch in the CSR form of ``dagma_linear_fit_small_pst_f64`` (``inv``) /
    ``dagma_linear_fit_small_pst_exp_f64`` (``exp``).  The series is told by ``eps_inv``: a float for ``inv``, None
    for ``exp`` (a series without that parameter)."""
    pair_off: torch.Tensor      # [batch + 1] int32
    pairs: torch.Tensor         # [max(total, 1), 2] int32
    weight: torch.Tensor        # [batch] float64
    agg: int
    eps_inv: typing.Optional[float]


class _TccBatch(typing.NamedTuple):
    """Pair sets and per-problem parameters of an on-chip TCC batch (``dagma_linear_fit_small_tcc_f64``): numpy arrays
    from ``_trek_batch``, device tensors after ``_tcc_dev``.  m of problem b = pair_off[b + 1] - pair_off[b]
    (duplicates counted, as ``SpectralTcc.n_vals``)."""
    pair_off: typing.Any        # [batch + 1] int32
    pairs: typing.Any           # [max(total, 1), 2] int32
    weight: typing.Any          # [batch] float64
    w: typing.Any               # [batch] float64, weight of the S block
    eps: typing.Any             # [batch] float64
    n_iter: typing.Any          # [batch] int32, steps of method "power"
    flags: typing.Any           # [batch] int32, _TCC_POWER | _TCC_DAG_LEARNING
    perron_steps: typing.Any = None   # [batch] int64 device tensor: power steps of all solves, summed over launches


_TCC_POWER, _TCC_DAG_LEARNING = 1, 2           # DAGMA_TCC_* of include/dagma_b200.h


def _pair_csr(plans, batch: int, d: int, who: str):
    """CSR form of the problems' pair sets (None: no pairs) and their weights; negative indices wrapped."""
    off = np.zeros(batch + 1, dtype=np.int64)
    weight = np.zeros(batch)
    parts = []
    for b, p in enumerate(plans):
        I = p["I"] if p is not None else np.zeros((0, 2), dtype=np.int64)
        if I.size and (I.min() < -d or I.max() >= d):
            raise IndexError(f"{who}: trek_reg of problem {b} has a pair index outside [-{d}, {d})")
        parts.append(I % d)                       # negative indices count from the end, as H[rows, cols] does
        off[b + 1] = off[b] + len(I)
        weight[b] = p["weight"] if p is not None else 0.0
    if off[-1] >= 2 ** 31:
        raise ValueError(f"{who}: {off[-1]} trek pairs in one batch (at most 2^31 - 1)")
    pairs = np.concatenate(parts).astype(np.int32) if off[-1] else np.zeros((1, 2), dtype=np.int32)
    return off.astype(np.int32), pairs, weight


def _tcc_batch(plans, batch: int, d: int, who: str) -> typing.Optional[_TccBatch]:
    """The on-chip TCC plan, or None when some problem's term, resolved as ``DagmaLinear`` resolves it
    (``_large._trek_setup``), is not spectral approx_trek_graph / DAG_learning with a method the kernel runs."""
    from . import notreks
    w, eps = np.ones(batch), np.full(batch, 1e-12)
    n_iter, flags = np.zeros(batch, dtype=np.int32), np.zeros(batch, dtype=np.int32)
    for b, p in enumerate(plans):
        if p is None:
            continue
        kw = notreks._tcc_call_args(p["reg"], notreks.FORWARD_TCC_CONFIG)
        version, method = kw.get("version", "approx_trek_graph"), kw.get("method", "eig_numpy")
        if (kw.get("cycle_penalty", "spectral") != "spectral" or version not in ("approx_trek_graph", "DAG_learning")
                or (method == "power" and not 0 <= kw["n_iter"] < 2 ** 31)):
            return None
        w[b], eps[b], n_iter[b] = kw["w"], kw["eps"], kw["n_iter"]
        flags[b] = (_TCC_POWER if method == "power" else 0) | (_TCC_DAG_LEARNING if version == "DAG_learning" else 0)
    off, pairs, weight = _pair_csr(plans, batch, d, who)
    return _TccBatch(off, pairs, weight, w, eps, n_iter, flags)


def _trek_batch(trek_reg, batch: int, d: int, loss_type: str, who: str):
    """``trek_reg`` of a batched call, checked without a device: one regulariser for the whole batch or a sequence with
    one regulariser (or None) per problem, each validated as ``DagmaLinear(trek_reg=...)`` validates it.

    Returns None when no problem carries a term that changes W (None, disabled, empty ``I``, mode "log": the reference
    only logs such a value, linear.py:122-133, 251-258).  Otherwise ``(regs, onchip)``: ``regs`` one regulariser per
    problem; ``onchip`` the host arrays of the on-chip PST kernels -- l2, d <= 64, every term PST ``inv`` with one
    ``agg`` and ``eps_inv``, or every term PST ``exp`` with one ``agg`` -- or None when the problems run one after the
    other as ``DagmaLinear(trek_reg=regs[b])``.  ``onchip = (pair_off, pairs, weight, agg, eps_inv)``; ``eps_inv`` is
    None for ``exp`` (``eps_inv`` and ``K_log`` never reach that series, so problems that differ only in them share a
    launch).  When every term is TCC and resolves to spectral approx_trek_graph / DAG_learning, ``onchip`` is a
    ``_TccBatch`` (problems with different w, eps, n_iter, method and version share the launch)."""
    if trek_reg is None:
        return None
    regs = list(trek_reg) if isinstance(trek_reg, (list, tuple)) else [trek_reg] * batch
    if len(regs) != batch:
        raise ValueError(f"{who}: trek_reg has {len(regs)} entries for a batch of {batch} problems")
    plans = [_trek_plan(r) for r in regs]
    plans = [p if p is not None and p["mode"] == "opt" else None for p in plans]
    active = [p for p in plans if p is not None]
    if not active:
        return None
    keys = {(p["kind"], p.get("seq"), p.get("agg"), p.get("eps_inv") if p.get("seq") == "inv" else None)
            for p in active}
    if loss_type == "l2" and d <= _lib.SMALL_MAX_D and keys == {("tcc", None, None, None)}:
        return regs, _tcc_batch(plans, batch, d, who)
    if (loss_type != "l2" or d > _lib.SMALL_MAX_D or len(keys) != 1
            or next(iter(keys))[:2] not in (("pst", "inv"), ("pst", "exp"))):
        return regs, None
    _, _, agg, eps_inv = keys.pop()
    off, pairs, weight = _pair_csr(plans, batch, d, who)
    return regs, (off, pairs, weight, _PST_AGGS[agg], None if eps_inv is None else float(eps_inv))


def _pst_dev(onchip, device) -> _PstBatch:
    off, pairs, weight, agg, eps_inv = onchip
    dev = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(device)  # noqa: E731
    return _PstBatch(dev(off), dev(pairs), dev(weight), agg, eps_inv)


def _tcc_dev(plan: _TccBatch, device) -> _TccBatch:
    dev = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(device)  # noqa: E731
    return _TccBatch(*(dev(a) for a in plan[:7]), torch.zeros(len(plan.weight), dtype=torch.int64, device=device))


def _onchip_trek(trek, device) -> dict:
    """The ``pst=`` / ``tcc=`` argument of ``_run_small`` for a batch that ``_trek_batch`` sends on chip."""
    if trek is None:
        return {}
    if isinstance(trek[1], _TccBatch):
        return {"tcc": _tcc_dev(trek[1], device)}
    return {"pst": _pst_dev(trek[1], device)}


def minimize_batch(W, cov, lambda1, mu, max_iter, s, lr, *, tol=1e-6, beta_1=0.99, beta_2=0.999,
                   checkpoint=1000, device=None, exclude_edges=None, include_edges=None, loss_type="l2", X=None,
                   trek_reg=None):
    """One ``DagmaLinear(loss_type).minimize`` call (linear.py:165-333) for a batch of
    independent problems.  ``W``/``cov``: [batch, d, d] numpy arrays or torch tensors on
    host (pinned or not) or device.  ``loss_type="logistic"`` needs the data ``X`` [batch, n, d]
    (not centred, not modified); ``cov`` is then its X^T X / n and may be None (computed from X).
    ``trek_reg``: one trek regulariser for the batch, or a sequence of one regulariser (or None)
    per problem -- what ``DagmaLinear(loss_type, trek_reg=...)`` would carry.  l2 problems with
    d <= 64 whose terms are all PST ``seq="inv"`` with one ``agg`` and ``eps_inv``, or all PST
    ``seq="exp"`` with one ``agg``, or all spectral TCC (``approx_trek_graph`` / ``DAG_learning``
    as ``DagmaLinear`` resolves them, any mix of w / eps / n_iter / method), run in one launch;
    other regularisers (a mix of series or of PST and TCC, ``log`` / ``binom``, the other TCC
    versions, the logistic loss, d > 64) run the problems one after the other through
    ``DagmaLinear``.
    Like the reference, ``W`` is updated in place and returned.
    Returns ``(W, success[batch], stage_stats[batch, 1, 8])``."""
    logistic = _logistic_inputs(loss_type, X, "minimize_batch")
    trek = _trek_batch(trek_reg, np.shape(W)[0], np.shape(W)[-1], loss_type, "minimize_batch")
    _lib.require_device()
    device = torch.device(device or "cuda")
    on_device = isinstance(W, torch.Tensor) and W.is_cuda
    if trek is None and _host_pipeline_ok(W, cov, loss_type):
        return _minimize_batch_host_pipelined(W, cov, lambda1, mu, max_iter, s, lr, tol=tol, beta_1=beta_1, beta_2=beta_2,
                                              checkpoint=checkpoint, device=device, exclude_edges=exclude_edges,
                                              include_edges=include_edges)
    Wd = W if on_device and W.dtype == torch.float64 and W.is_contiguous() else _as_dev(W, device)
    Xd = _as_dev(X, device) if logistic else None
    covd = center_cov(Xd, center=False) if logistic and cov is None else _as_dev(cov, device)
    batch, d, _ = covd.shape
    if Xd is not None and (Xd.shape[0] != batch or Xd.shape[2] != d):
        raise ValueError(f"minimize_batch: X {tuple(Xd.shape)} does not match W / cov [{batch}, {d}, {d}]")
    if d > _lib.SMALL_MAX_D or (trek is not None and trek[1] is None):
        return _minimize_batch_large(W, covd, lambda1, mu, max_iter, s, lr, tol=tol, beta_1=beta_1, beta_2=beta_2,
                                     checkpoint=checkpoint, exclude_edges=exclude_edges, include_edges=include_edges,
                                     Xd=Xd, treks=trek[0] if trek is not None else None)
    lam = _lam_dev(lambda1, batch, device)
    mask_exc, mask_inc = _batch_masks(exclude_edges, include_edges, d, device)
    res = _run_small(covd, Wd, lam, [mu], [s], [int(max_iter)], lr=lr, tol=tol, beta1=beta_1, beta2=beta_2,
                     checkpoint=checkpoint, retry=False, want_final=False, mask_exc=mask_exc, mask_inc=mask_inc, X=Xd,
                     **_onchip_trek(trek, device))
    _warn_perron_cap(res.status)
    ok = (res.status & _lib.ST_OUT_OF_DOMAIN) == 0
    if on_device:
        if Wd is not W:
            W.copy_(Wd)
        return W, ok, res.stage_stats
    if isinstance(W, torch.Tensor):
        W.copy_(res.W)                       # D2H into the caller's (possibly pinned) buffer
    else:
        W[...] = res.W.cpu().numpy()
    return W, ok.cpu().numpy(), res.stage_stats.cpu().numpy()


_COPY_STREAMS: dict = {}       # device index -> (H2D stream, D2H stream) of the pipelined host path


def _host_pipeline_ok(W, cov, loss_type="l2") -> bool:
    """Pinned host tensors of an l2 batch that spans several waves of resident CTAs: worth overlapping the copies."""
    import os
    if loss_type != "l2" or os.environ.get("DAGMA_HOST_PIPELINE", "1") == "0":
        return False
    ok = all(isinstance(t, torch.Tensor) and not t.is_cuda and t.is_pinned() and t.dtype == torch.float64
             and t.is_contiguous() and t.dim() == 3 for t in (W, cov))
    return ok and 32 < cov.shape[1] <= _lib.SMALL_MAX_D and cov.shape[0] >= 4 * _resident_ctas()


def _resident_ctas() -> int:
    """CTAs of the tensor-core fit kernel that are resident at once (two per SM)."""
    return 2 * torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _pipeline_chunks(batch: int, wave: int) -> list:
    """[lo, hi) ranges of the pipelined host path: a first chunk of two waves of resident CTAs (its H2D is the part of
    the copies that stays exposed), then chunks of four waves; a remainder of less than one wave joins the chunk in
    front of it.  Whole waves: k x `wave` equal-length problems take k wave-times alone or as part of the batch."""
    bounds, lo = [], 0
    for size in [2 * wave] + [4 * wave] * (batch // max(wave, 1) + 1):
        if lo >= batch:
            break
        hi = min(batch, lo + size)
        if batch - hi < wave:                     # no sliver at the end
            hi = batch
        bounds.append((lo, hi))
        lo = hi
    return bounds


def _minimize_batch_host_pipelined(W, cov, lambda1, mu, max_iter, s, lr, *, tol, beta_1, beta_2, checkpoint, device,
                                   exclude_edges, include_edges):
    """``minimize_batch`` on pinned host buffers with the copies hidden behind the kernel: the batch is cut into chunks of
    whole waves of resident CTAs (a chunk of k x 296 equal-length problems takes k wave-times whether it is launched
    alone or as part of the batch), H2D of chunk c + 1 and D2H of chunk c - 1 run on copy streams while chunk c
    computes.  What stays exposed is the H2D of a first, short chunk and the D2H of the last one."""
    batch, d, _ = cov.shape
    bounds = _pipeline_chunks(batch, _resident_ctas())
    lam = _lam_dev(lambda1, batch, device)
    mask_exc, mask_inc = _batch_masks(exclude_edges, include_edges, d, device)
    cur = torch.cuda.current_stream()
    key = torch.device(device).index or 0
    if key not in _COPY_STREAMS:
        _COPY_STREAMS[key] = (torch.cuda.Stream(), torch.cuda.Stream())
    s_in, s_out = _COPY_STREAMS[key]
    # the device buffers come from the CALLER's stream pool (reused from call to call: a buffer allocated under a copy
    # stream would be a fresh cudaMalloc every time); the copy streams are told about them with record_stream
    Wall = torch.empty(batch, d, d, dtype=torch.float64, device=device)
    call = torch.empty(batch, d, d, dtype=torch.float64, device=device)
    Wall.record_stream(s_in)
    Wall.record_stream(s_out)
    call.record_stream(s_in)
    s_in.wait_stream(cur)
    s_out.wait_stream(cur)
    bufs, results = [], []
    with torch.cuda.stream(s_in):                 # every H2D is queued up front; the chunks' kernels wait for their event
        for lo, hi in bounds:
            Wd, cd = Wall[lo:hi], call[lo:hi]
            Wd.copy_(W[lo:hi], non_blocking=True)
            cd.copy_(cov[lo:hi], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(s_in)
            bufs.append((Wd, cd, ev))
    for (lo, hi), (Wd, cd, ev) in zip(bounds, bufs):
        cur.wait_event(ev)
        res = _run_small(cd, Wd, lam[lo:hi].contiguous(), [mu], [s], [int(max_iter)], lr=lr, tol=tol, beta1=beta_1,
                         beta2=beta_2, checkpoint=checkpoint, retry=False, want_final=False, mask_exc=mask_exc,
                         mask_inc=mask_inc)
        done = torch.cuda.Event()
        done.record(cur)
        s_out.wait_event(done)
        with torch.cuda.stream(s_out):
            W[lo:hi].copy_(Wd, non_blocking=True)
        results.append(res)
    cur.wait_stream(s_out)
    status = torch.cat([r.status for r in results])
    stats = torch.cat([r.stage_stats for r in results])
    ok = ((status & _lib.ST_OUT_OF_DOMAIN) == 0).cpu().numpy()        # (synchronises: every copy has landed)
    torch.cuda.current_stream().synchronize()
    return W, ok, stats.cpu().numpy()


def fit_batch(X=None, lambda1=0.03, *, cov=None, w_threshold=0.3, T=5, mu_init=1.0, mu_factor=0.1,
              s=(1.0, .9, .8, .7, .6), warm_iter=3e4, max_iter=6e4, lr=0.0003, checkpoint=1000,
              beta_1=0.99, beta_2=0.999, tol=1e-6, device=None, return_info=False,
              exclude_edges=None, include_edges=None, loss_type="l2", trek_reg=None):
    """``DagmaLinear(loss_type).fit`` (linear.py:335-462) for a batch of independent problems.

    l2: ``X``: [batch, n, d] (centred on device, the caller's array is not modified) or
    ``cov``: [batch, d, d].  logistic: ``X`` [batch, n, d] only (not centred, not modified; the
    covariance is its X^T X / n).  ``lambda1``: scalar or [batch].  Each problem follows the
    reference schedule independently (own convergence checks, retries, back-tracking);
    problems are pulled from a device-side work queue by persistent CTAs.
    ``exclude_edges`` / ``include_edges``: tuples of 2-tuples shared by the batch (linear.py:416-426).
    ``trek_reg``: as in ``minimize_batch`` (one regulariser, or one per problem); l2 batches at
    d <= 64 whose terms are all PST ``inv`` (one ``agg`` / ``eps_inv``), all PST ``exp`` (one
    ``agg``) or all spectral TCC (``approx_trek_graph`` / ``DAG_learning``) run in one launch,
    other regularisers one problem after the other.
    Returns thresholded ``W_est`` [batch, d, d] as numpy (+ info dict; an on-chip TCC batch adds
    ``perron_steps`` [batch], the power steps of all Perron solves of each problem)."""
    logistic = _logistic_inputs(loss_type, X, "fit_batch")
    if logistic and cov is not None:
        raise ValueError("fit_batch(loss_type='logistic') takes X only: the covariance is computed from it")
    src = X if cov is None else cov
    trek = _trek_batch(trek_reg, np.shape(src)[0], np.shape(src)[-1], loss_type, "fit_batch")
    _lib.require_device()
    device = torch.device(device or "cuda")
    Xd = None
    if logistic:
        Xd = _as_dev(X, device)
        covd = center_cov(Xd, center=False)
    elif cov is None:
        Xc = _as_dev(X, device)
        if Xc.data_ptr() == (X.data_ptr() if isinstance(X, torch.Tensor) else 0):
            Xc = Xc.clone()
        covd = center_cov(Xc, center=True)
        del Xc
    else:
        covd = _as_dev(cov, device)
    batch, d, _ = covd.shape
    if d > _lib.SMALL_MAX_D or (trek is not None and trek[1] is None):
        return _fit_batch_large(covd, lambda1, w_threshold=w_threshold, T=T, mu_init=mu_init, mu_factor=mu_factor, s=s,
                                warm_iter=warm_iter, max_iter=max_iter, lr=lr, checkpoint=checkpoint, beta_1=beta_1,
                                beta_2=beta_2, return_info=return_info, exclude_edges=exclude_edges,
                                include_edges=include_edges, Xd=Xd, treks=trek[0] if trek is not None else None)
    lam = _lam_dev(lambda1, batch, device)
    T = int(T)
    ss = list(s) if isinstance(s, (list, tuple)) else T * [s]
    if len(ss) < T:
        ss = ss + (T - len(ss)) * [ss[-1]]
    mus = _mu_schedule(mu_init, mu_factor, T)
    iters = [int(max_iter) if i == T - 1 else int(warm_iter) for i in range(T)]
    Wd = torch.zeros(batch, d, d, dtype=torch.float64, device=device)
    mask_exc, mask_inc = _batch_masks(exclude_edges, include_edges, d, device)
    onchip = _onchip_trek(trek, device)
    res = _run_small(covd, Wd, lam, mus, ss[:T], iters, lr=lr, tol=tol, beta1=beta_1, beta2=beta_2,
                     checkpoint=checkpoint, retry=True, mask_exc=mask_exc, mask_inc=mask_inc, X=Xd, **onchip)
    _warn_retry_limit(res.status)
    _warn_perron_cap(res.status)
    W_raw = res.W.cpu().numpy()
    W_est = W_raw.copy()
    W_est[np.abs(W_est) < w_threshold] = 0
    if not return_info:
        return W_est
    stats = res.stage_stats.cpu().numpy()
    fin = res.final.cpu().numpy()
    info = {"W_raw": W_raw, "status": res.status.cpu().numpy(), "stage_iters": stats[:, :, 0].astype(np.int64),
            "stage_stats": stats, "h_final": fin[:, 0], "score_final": fin[:, 1],
            "total_iters": int(stats[:, :, 0].sum())}
    if "tcc" in onchip:
        info["perron_steps"] = onchip["tcc"].perron_steps.cpu().numpy()
    return W_est, info


def _batch_lanes(d: int, batch: int, n: typing.Optional[int] = None) -> int:
    """How many problems of a d > 64 batch run side by side.  For d <= 128 a problem's inner iterations are one
    persistent kernel (csrc/lin_iter.cu) of ceil(d / 8) + 1 CTAs for l2, and for the logistic loss (``n`` rows of X)
    of one CTA per block of rows plus the inverse CTA, each alone on its SM, so several problems fit on the
    device at once -- one host thread and one CUDA stream per lane (DAGMA_BATCH_LANES overrides; 1 = one after the
    other).  Beyond d = 128 the blocked inverse fills the device by itself."""
    import os
    env = os.environ.get("DAGMA_BATCH_LANES")
    if env:
        return max(1, min(int(env), batch))
    lib = _lib.load()
    logistic = n is not None
    if (d > 128 or not lib.dagma_linear_iter_supported(int(logistic), n or 0, d)
            or os.environ.get("DAGMA_LIN_FUSED", "1") == "0"):
        return 1
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    if logistic:
        # li_plan: the rows are spread over the SMs but one, in blocks of a multiple of 8 rows per worker CTA
        per = -(-n // (sms - 1))
        rows = 8 * -(-per // 8)
        ctas = -(-n // rows) + 1
    else:
        ctas = (d + 7) // 8 + 1
    return max(1, min((sms - 12) // ctas, 8, batch))       # a dozen SMs stay free for the checkpoint kernels of all lanes


_LANE_STREAMS: dict = {}       # device index -> raw streams of the batch lanes (created once, reused)


def _run_lanes(batch: int, d: int, solve, device, n: typing.Optional[int] = None) -> None:
    """``solve(b)`` for every problem of a d > 64 batch, ``_batch_lanes`` of them at a time: one host thread and one
    CUDA stream per lane (the caller's stream is waited for first; every lane is synchronised before returning)."""
    lanes = _batch_lanes(d, batch, n)
    if lanes <= 1:
        for b in range(batch):
            solve(b)
        return
    import ctypes as C
    import threading
    lib = _lib.load()
    main = torch.cuda.current_stream()
    todo = iter(range(batch))
    lock = threading.Lock()
    errors = []
    # one stream of its own per lane, created back to back: consecutive hardware work queues (streams from torch's pool
    # were created long ago, interleaved with others; several can share a queue and serialise the lanes' persistent
    # kernels).  The streams live as long as the process and are reused by later batches, so the caching allocator's
    # blocks of a lane stay usable and no stream it has seen is ever destroyed.
    raw = _LANE_STREAMS.setdefault(torch.device(device).index or 0, [])
    while len(raw) < lanes:
        p = C.c_void_p()
        _lib.check(lib.dagma_stream_create(C.byref(p)), "dagma_stream_create")
        raw.append(p)

    def lane(k):
        torch.cuda.set_device(device)
        st = torch.cuda.ExternalStream(raw[k].value, device=device)
        st.wait_stream(main)
        with torch.cuda.stream(st):
            while not errors:
                with lock:
                    b = next(todo, None)
                if b is None:
                    break
                try:
                    solve(b)
                except BaseException as e:                        # noqa: BLE001 -- re-raised on the caller's thread
                    errors.append(e)
            st.synchronize()

    threads = [threading.Thread(target=lane, args=(k,), daemon=True) for k in range(lanes)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]


def _minimize_batch_large(W, covd, lambda1, mu, max_iter, s, lr, *, tol, beta_1, beta_2, checkpoint, exclude_edges,
                          include_edges, Xd=None, treks=None):
    """``minimize_batch`` beyond the on-chip size: one ``DagmaLinear.minimize`` per problem on the multi-CTA engine, for
    d <= 128 several problems side by side (one persistent kernel each, csrc/lin_iter.cu).  With ``treks`` (one trek
    regulariser or None per problem) the problems run one after the other as ``DagmaLinear(trek_reg=treks[b])``: the
    lane count is sized for csrc/lin_iter.cu, which a trek regulariser turns off."""
    batch, d, _ = covd.shape
    lam = np.broadcast_to(np.asarray(lambda1.cpu() if isinstance(lambda1, torch.Tensor) else lambda1,
                                     dtype=np.float64), (batch,))
    W_np = W.detach().cpu().numpy() if isinstance(W, torch.Tensor) else np.asarray(W)
    W_out = np.array(W_np, dtype=np.float64, copy=True)
    ok = np.zeros(batch, dtype=bool)
    stats = np.zeros((batch, 1, 8))

    def solve(b):
        m = DagmaLinear("l2" if Xd is None else "logistic", trek_reg=treks[b] if treks is not None else None)
        m._fit_from_cov(covd[b], float(lam[b]), T=1, warm_iter=0, max_iter=0, checkpoint=checkpoint,
                        exclude_edges=exclude_edges, include_edges=include_edges,
                        X_dev=Xd[b] if Xd is not None else None)
        _, ok[b] = m.minimize(W_out[b], mu, int(max_iter), s, lr=lr, tol=tol, beta_1=beta_1, beta_2=beta_2)
        stats[b, 0, 0] = m.last_iters
        stats[b, 0, 1], stats[b, 0, 2] = (m._large.last_lr if m._large is not None else lr), s
        if m.checkpoint_log:
            stats[b, 0, 3:6] = m.checkpoint_log[-1][2:5]

    if treks is not None:
        for b in range(batch):
            solve(b)
    else:
        _run_lanes(batch, d, solve, covd.device, Xd.shape[1] if Xd is not None else None)
    if isinstance(W, torch.Tensor):
        W.copy_(torch.from_numpy(W_out))
        return W, (torch.from_numpy(ok).to(W.device) if W.is_cuda else ok), (torch.from_numpy(stats).to(W.device) if W.is_cuda else stats)
    W[...] = W_out
    return W, ok, stats


def _fit_batch_large(covd, lambda1, *, w_threshold, return_info, Xd=None, treks=None, **fit_kw):
    """``fit_batch`` beyond the on-chip size (d > 64): every problem runs on the multi-CTA engine -- the same code path
    as ``DagmaLinear.fit`` at that size, fed with the covariance instead of the data -- and ``_batch_lanes`` problems
    run concurrently, each on its own stream (for d <= 128 the inner iterations of a problem are one persistent kernel
    on a handful of SMs).  With ``treks`` the problems run one after the other as ``DagmaLinear(trek_reg=treks[b])``
    (see ``_minimize_batch_large``)."""
    batch, d, _ = covd.shape
    lam = np.broadcast_to(np.asarray(lambda1.cpu() if isinstance(lambda1, torch.Tensor) else lambda1,
                                     dtype=np.float64), (batch,))
    W_raw = np.empty((batch, d, d))
    stage_iters, h_fin, sc_fin = [None] * batch, [None] * batch, [None] * batch

    def solve(b):
        m = DagmaLinear("l2" if Xd is None else "logistic", trek_reg=treks[b] if treks is not None else None)
        kw = dict(fit_kw)
        kw["s"] = list(kw["s"]) if isinstance(kw["s"], (list, tuple)) else kw["s"]
        m._fit_from_cov(covd[b], float(lam[b]), X_dev=Xd[b] if Xd is not None else None, **kw)
        W_raw[b] = m.W_raw
        stage_iters[b], h_fin[b], sc_fin[b] = m.stage_iters, m.h_final, m.score_final

    if treks is not None:
        for b in range(batch):
            solve(b)
    else:
        _run_lanes(batch, d, solve, covd.device, Xd.shape[1] if Xd is not None else None)
    W_est = W_raw.copy()
    W_est[np.abs(W_est) < w_threshold] = 0
    if not return_info:
        return W_est
    si = np.array(stage_iters, dtype=np.int64)
    return W_est, {"W_raw": W_raw, "status": np.zeros(batch, dtype=np.int32), "stage_iters": si,
                   "h_final": np.array(h_fin), "score_final": np.array(sc_fin), "total_iters": int(si.sum())}


# =============================================================================
# the drop-in class
def _trek_plan(tr) -> typing.Optional[dict]:
    """Which trek regulariser the accelerated path carries (SURVEY.md 8f3): PST with any series (``inv``, ``log``,
    ``exp``, ``binom``) and any scalar aggregation (``mean``, ``sum``, ``max``, ``lse``)
    (src/notreks/notreks.py:454-619), or TCC (spectral by the reference's dispatch, notreks.py:699-707), in mode "opt"
    or "log".  A disabled regulariser or an empty pair list is the reference's no-op branch (notreks.py:684-689)."""
    if tr is None or not tr.enabled():
        return None
    I = tr.cfg.get("I") if tr.cfg is not None else None
    if I is None or len(I) == 0:
        return None
    name = tr.name.lower().strip()
    if name == "tcc":
        I_np = np.asarray(I, dtype=np.int64)
        if I_np.ndim != 2 or I_np.shape[1] != 2:
            raise ValueError("I must be array-like of shape (m,2)")
        return {"kind": "tcc", "I": I_np, "weight": float(tr.weight), "mode": tr.mode, "reg": tr}
    if name != "pst":
        raise ValueError(f"Unknown trek regularizer: {tr.name}. Has to be in ['pst', 'tcc']")   # notreks.py:664
    kwargs = dict(tr.cfg.get("kwargs", {}) or {})
    seq = str(tr.cfg.get("seq", "exp")).lower().strip()
    agg = str(kwargs.pop("agg", "mean")).lower().strip()
    eps_inv = float(kwargs.pop("eps_inv", 1e-8))
    K_log = kwargs.pop("K_log", None)
    kwargs.pop("s", None)                       # never reaches any series (notreks.py:509-513 vs 521-525, Q14)
    if kwargs:
        raise TypeError(f"pst() got unexpected keyword arguments {sorted(kwargs)}")
    if seq not in ("exp", "log", "inv", "binom"):
        raise ValueError("seq must be one of {'exp','log','inv','binom'}")
    if agg == "none":
        raise RuntimeError("agg='none' is not a scalar penalty (the reference fails in .item())")
    if agg not in ("mean", "sum", "max", "lse"):
        raise ValueError("agg must be one of {'mean','sum','max','lse','none'}")
    if eps_inv < 0:
        raise ValueError("eps_inv must be >= 0")
    I_np = np.asarray(I, dtype=np.int64)
    if I_np.ndim != 2 or I_np.shape[1] != 2:
        raise ValueError("I must be array-like of shape (m,2)")
    return {"kind": "pst", "I": I_np, "seq": seq, "agg": agg, "eps_inv": eps_inv, "K_log": K_log,
            "weight": float(tr.weight), "mode": tr.mode}


# =============================================================================
class DagmaLinear:
    """DAGMA for linear SEMs on B200 (same surface as the reference class, linear.py:20)."""

    def __init__(self, loss_type: str, verbose: bool = False, dtype: type = np.float64, *,
                 trek_reg=None, logger=None, log_cfg=None) -> None:
        losses = ['l2', 'logistic']
        assert loss_type in losses, f"loss_type should be one of {losses}"     # linear.py:52-53
        self.loss_type = loss_type
        self.dtype = dtype
        self.vprint = print if verbose else lambda *a, **k: None
        self.trek_reg = trek_reg
        self._trek_plan = _trek_plan(trek_reg)          # None, or the PST / TCC plan
        self._torch_dtype = torch.double
        self._device = torch.device("cuda")
        # telemetry: same defaults as the reference (linear.py:65-67) -- a logger that is silent unless verbose
        import logging
        from .logger import LogConfig, StructuredLogger, build_default_logger
        self._logger = logger or build_default_logger(level=logging.INFO if verbose else logging.WARNING)
        self._log_cfg = log_cfg or LogConfig(enabled=verbose)
        self._slog = StructuredLogger(self._logger, self._log_cfg)
        self._large = None
        self._group = None                  # torch.distributed group when the rows of X are sharded
        self.checkpoint_log = []            # rows (stage, iter, obj, score, h, lr) of the last calls

    def shard_rows(self, group=None) -> "DagmaLinear":
        """Declare that the ``X`` given to ``fit`` is this rank's contiguous row shard of the data
        (SURVEY.md 8e2): cov, the column means and the score gradient are then sum all-reduced over
        ``group``; every rank holds identical parameters and returns the identical ``W_est``."""
        import torch.distributed as dist
        self._group = group if group is not None else dist.group.WORLD
        return self

    # ------------------------------------------------------------------ helpers
    def _dev(self, x) -> torch.Tensor:
        return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64)).to(self._device)

    def _small_ok(self) -> bool:
        # the one-launch on-chip path; telemetry rows are produced inside the kernel at the checkpoint iterations, so
        # logging does not change the route -- only a trek regulariser does (its series need the multi-CTA GEMMs)
        return (self.loss_type == 'l2' and self.d <= _lib.SMALL_MAX_D and self._group is None
                and self._trek_plan is None)

    def _large_engine(self):
        from ._large import LargeLinearEngine
        if self._large is None or self._large.stale(self):
            if self._large is not None:
                self._large.close()              # peer mappings of a row-sharded engine (collective)
            self._large = LargeLinearEngine(self, group=self._group)
        return self._large

    def close(self) -> None:
        """Release what the multi-CTA engine holds beyond plain device memory (the NVLink peer mappings of a
        row-sharded logistic model: collective over the group).  Optional for un-sharded models."""
        if self._large is not None:
            self._large.close()
            self._large = None

    # ------------------------------------------------------------------ _score (linear.py:70-94)
    def _score(self, W: np.ndarray) -> typing.Tuple[float, np.ndarray]:
        loss, G = self._large_engine().score(self._dev(W))
        return loss, G.cpu().numpy()

    # ------------------------------------------------------------------ _h (linear.py:97-116)
    def _h(self, W: np.ndarray, s: float = 1.0) -> typing.Tuple[float, np.ndarray]:
        out = logdet_inv(self._dev(W)[None], s=s, square_input=True, want_inv=False, want_grad=True)
        return float(out["h"].item()), out["grad"][0].cpu().numpy()

    # ------------------------------------------------------------------ _func (linear.py:118-135)
    def _func(self, W: np.ndarray, mu: float, s: float = 1.0):
        score, _ = self._score(W)
        h, _ = self._h(W, s)
        obj = mu * (score + self.lambda1 * np.abs(W).sum()) + h
        trek_val = 0.0
        if self._trek_plan is not None:
            eng = self._large_engine()
            eng.W.copy_(self._dev(W))
            trek_val = eng._trek_value()
            if self._trek_plan["mode"] == "opt":
                obj = obj + self._trek_plan["weight"] * trek_val
        return obj, score, h, trek_val

    # ------------------------------------------------------------------ _adam_update (linear.py:138-163)
    def _adam_update(self, grad: np.ndarray, iter: int, beta_1: float, beta_2: float) -> np.ndarray:
        g = self._dev(grad)
        if not isinstance(getattr(self, "opt_m", 0), torch.Tensor):      # reference resets to scalar 0 (:215)
            self.opt_m, self.opt_v = torch.zeros_like(g), torch.zeros_like(g)
        out = torch.empty_like(g)
        _lib.check(_lib.load().dagma_adam_direction_f64(
            _lib.stream_ptr(), g.numel(), g.data_ptr(), self.opt_m.data_ptr(), self.opt_v.data_ptr(),
            float(beta_1), float(beta_2), 1 - beta_1 ** iter, 1 - beta_2 ** iter, out.data_ptr()),
            "dagma_adam_direction_f64")
        return out.cpu().numpy()

    # ------------------------------------------------------------------ minimize (linear.py:165-333)
    def minimize(self, W: np.ndarray, mu: float, max_iter: int, s: float, lr: float, tol: float = 1e-6,
                 beta_1: float = 0.99, beta_2: float = 0.999, pbar=None) -> typing.Tuple[np.ndarray, bool]:
        self.vprint(f'\n\nMinimize with -- mu:{mu} -- lr: {lr} -- s: {s} -- l1: {self.lambda1} for {max_iter} max iterations')
        if self._small_ok():
            Wd = self._dev(W)[None].contiguous()
            res = _run_small(self._cov_dev[None], Wd, self._lam_dev, [mu], [s], [int(max_iter)], lr=lr, tol=tol,
                             beta1=beta_1, beta2=beta_2, checkpoint=self.checkpoint, retry=False,
                             mask_exc=self._mask_exc, mask_inc=self._mask_inc,
                             ckpt_log_cap=int(max_iter) // max(int(self.checkpoint), 1) + 2, want_final=False,
                             want_diag=self._log_cfg.enabled)
            W[...] = res.W[0].cpu().numpy()
            status = int(res.status.item())
            iters_done = int(res.stage_stats[0, 0, 0].item())
            self._record_log(res, [mu], [s])
        else:
            log = []
            status, iters_done = self._large_engine().minimize(
                W, mu, int(max_iter), s, lr, tol, beta_1, beta_2, self.lambda1, int(self.checkpoint), log,
                telemetry=self._checkpoint_emitter(mu, s) if self._log_cfg.enabled else None)
            self.checkpoint_log.extend(log)
        self.last_iters = iters_done
        success = (status & _lib.ST_OUT_OF_DOMAIN) == 0
        if not success:
            self.vprint(f'W went out of domain for s={s} at iteration {iters_done + 1}')
        if pbar is not None:
            pbar.update(int(max_iter))
        return W, success

    def _checkpoint_emitter(self, mu: float, s: float):
        """The 25-key ``minimize.checkpoint`` row of the reference (linear.py:279-326)."""
        t0 = time.time()
        stage = getattr(self, "_stage", 0)
        tr = self.trek_reg
        trek_cfg = {k: v for k, v in tr.cfg.items() if k != "I"} if tr is not None else {}

        def emit(diag, it, obj, score, h, trek_val, lr):
            self._slog.emit("minimize.checkpoint", {
                "iter": int(it), "stage": int(stage), "elapsed_sec": float(time.time() - t0),
                "obj_total": float(obj), "score_datafit": float(score),
                "reg_dag_name": "dagma_logdet", "reg_dag_value": float(h), "reg_dag_cfg": {"s": float(s)},
                "reg_trek_name": tr.name if tr is not None else "none", "reg_trek_value": float(trek_val),
                "reg_trek_cfg": trek_cfg, "trek_mode": tr.mode if tr is not None else "off",
                "trek_weight": float(tr.weight) if tr is not None else 0.0,
                "mu": float(mu), "lr": float(lr),
                "w_norm": diag["w_norm"], "w_abs_sum": diag["w_abs_sum"], "max_abs_w": diag["max_abs_w"],
                "min_abs_w_nonzero": diag["min_abs_w_nonzero"],
                "grad_raw_norm": diag["grad_raw_norm"], "grad_step_norm": diag["grad_step_norm"],
                "step_norm": float(lr * diag["grad_step_norm"]), "grad_score_norm": diag["grad_score_norm"],
                "grad_dag_norm": diag["grad_dag_norm"], "grad_l1_norm": diag["grad_l1_norm"],
                "grad_inc_norm": diag["grad_inc_norm"], "grad_trek_norm": diag["grad_trek_norm"],
            })
        return emit

    def _record_log(self, res: SmallFitResult, mus=None, ss=None) -> None:
        """Checkpoint rows of an on-chip run: the (stage, iter, obj, score, h, lr) log and, with logging enabled, the
        fork's 25-key ``minimize.checkpoint`` event per row (linear.py:279-326) from the kernel's telemetry rows."""
        if res.ckpt_log is None:
            return
        n = int(res.ckpt_count[0].item())
        rows = res.ckpt_log[0, :n].cpu().numpy()
        self.checkpoint_log.extend(map(tuple, rows))
        diag = res.ckpt_diag[0, :n].cpu().numpy() if res.ckpt_diag is not None else None
        for k, (st, it, obj, score, h, lr) in enumerate(rows):
            self.vprint(f'\nInner iteration {int(it)}\n\th(W_est): {h:.4e}\n\tscore(W_est): {score:.4e}\n\tobj: {obj:.4e}')
            if diag is None or not self._log_cfg.enabled:
                continue
            dg = diag[k]
            t = min(int(st), len(mus) - 1)
            # the value of s a retried stage ended with is what its later rows ran at; rows of failed attempts carry
            # the s of that attempt only up to the 0.1 steps of the retries (the kernel reports the final one)
            self._slog.emit("minimize.checkpoint", {
                "iter": int(it), "stage": int(getattr(self, "_stage", 0)), "elapsed_sec": float(dg[10]),
                "obj_total": float(obj), "score_datafit": float(score),
                "reg_dag_name": "dagma_logdet", "reg_dag_value": float(h), "reg_dag_cfg": {"s": float(ss[t])},
                "reg_trek_name": self.trek_reg.name if self.trek_reg is not None else "none", "reg_trek_value": 0.0,
                "reg_trek_cfg": ({k_: v for k_, v in self.trek_reg.cfg.items() if k_ != "I"}
                                 if self.trek_reg is not None else {}),
                "trek_mode": self.trek_reg.mode if self.trek_reg is not None else "off",
                "trek_weight": float(self.trek_reg.weight) if self.trek_reg is not None else 0.0,
                "mu": float(mus[t]), "lr": float(lr),
                "w_norm": float(dg[6]), "w_abs_sum": float(dg[7]), "max_abs_w": float(dg[8]),
                "min_abs_w_nonzero": float(dg[9]),
                "grad_raw_norm": float(dg[0]), "grad_step_norm": float(dg[5]), "step_norm": float(lr * dg[5]),
                "grad_score_norm": float(dg[1]), "grad_dag_norm": float(dg[2]), "grad_l1_norm": float(dg[3]),
                "grad_inc_norm": float(dg[4]), "grad_trek_norm": 0.0,
            })

    def _fit_from_cov(self, cov_dev: torch.Tensor, lambda1: float, *, T=5, mu_init=1.0, mu_factor=0.1,
                      s=(1.0, .9, .8, .7, .6), warm_iter=3e4, max_iter=6e4, lr=0.0003, checkpoint=1000, beta_1=0.99,
                      beta_2=0.999, exclude_edges=None, include_edges=None, X_dev=None) -> np.ndarray:
        """The path-following loop of ``fit`` from a device covariance instead of the data (batched entry points);
        the logistic loss also needs the data itself, ``X_dev`` [n, d] on the device (cov = X^T X / n, un-centred)."""
        assert self.loss_type == 'l2' or X_dev is not None
        self.X, self.lambda1, self.checkpoint = None, lambda1, checkpoint
        self.d = int(cov_dev.shape[0])
        self.n = self._n_total = int(X_dev.shape[0]) if X_dev is not None else 0
        self.Id = np.eye(self.d).astype(self.dtype)
        self.checkpoint_log = []
        self._X_dev = X_dev.contiguous() if X_dev is not None else None
        self._cov_dev = cov_dev.contiguous()
        self.cov = self._cov_dev.cpu().numpy()
        self._run_path(lambda1, T, mu_init, mu_factor, s, warm_iter, max_iter, lr, checkpoint, beta_1, beta_2,
                       exclude_edges, include_edges)
        self.W_raw = self.W_est.copy()
        return self.W_raw

    def _run_path(self, lambda1, T, mu_init, mu_factor, s, warm_iter, max_iter, lr, checkpoint, beta_1, beta_2,
                  exclude_edges, include_edges) -> None:
        """linear.py:413-457: masks, the (mu, s) schedule, the stage loop with retries, final h / score."""
        self.exc_r, self.exc_c = None, None
        self.inc_r, self.inc_c = None, None
        if exclude_edges is not None:
            if type(exclude_edges) is tuple and type(exclude_edges[0]) is tuple and \
                    np.all(np.array([len(e) for e in exclude_edges]) == 2):
                self.exc_r, self.exc_c = zip(*exclude_edges)
            else:
                ValueError("blacklist should be a tuple of edges, e.g., ((1,2), (2,3))")   # not raised (Q5)
        if include_edges is not None:
            if type(include_edges) is tuple and type(include_edges[0]) is tuple and \
                    np.all(np.array([len(e) for e in include_edges]) == 2):
                self.inc_r, self.inc_c = zip(*include_edges)
            else:
                ValueError("whitelist should be a tuple of edges, e.g., ((1,2), (2,3))")
        self._mask_exc = _edge_mask(list(zip(self.exc_r, self.exc_c)) if self.exc_c is not None else None,
                                    self.d, self._device)
        self._mask_inc = _edge_mask(list(zip(self.inc_r, self.inc_c)) if self.inc_c is not None else None,
                                    self.d, self._device)
        self._lam_dev = torch.tensor([float(lambda1)], dtype=torch.float64, device=self._device)

        self.W_est = np.zeros((self.d, self.d)).astype(self.dtype)
        if type(s) == list:
            if len(s) < T:
                self.vprint(f"Length of s is {len(s)}, using last value in s for iteration t >= {len(s)}")
                s = s + (T - len(s)) * [s[-1]]
        elif type(s) in [int, float]:
            s = T * [s]
        else:
            ValueError("s should be a list, int, or float.")
        T = int(T)
        mus = _mu_schedule(mu_init, mu_factor, T)
        iters = [int(max_iter) if i == T - 1 else int(warm_iter) for i in range(T)]

        if self._small_ok():
            # the whole path-following loop (stages, retries, back-tracking) in one launch
            Wd = torch.zeros(1, self.d, self.d, dtype=torch.float64, device=self._device)
            cap = sum(it // max(int(checkpoint), 1) + 2 for it in iters)
            res = _run_small(self._cov_dev[None], Wd, self._lam_dev, mus, s[:T], iters, lr=lr, tol=1e-6,
                             beta1=beta_1, beta2=beta_2, checkpoint=checkpoint, retry=True,
                             mask_exc=self._mask_exc, mask_inc=self._mask_inc, ckpt_log_cap=min(cap, 4096),
                             want_diag=self._log_cfg.enabled)
            stats = res.stage_stats[0].cpu().numpy()
            for i in range(T):
                if stats[i, 6] > 0:
                    s[i] = float(stats[i, 2])           # s[i] += 0.1 per retry mutates the list (Q9)
            self.stage_iters = [int(x) for x in stats[:, 0]]
            self.stage_stats = stats
            self.status = int(res.status.item())
            _warn_retry_limit(res.status)
            self._record_log(res, mus, [float(x) for x in stats[:, 2]])
            self.W_est = res.W[0].cpu().numpy().astype(self.dtype)
            fin = res.final[0].cpu().numpy()
            self.h_final, self.score_final = float(fin[0]), float(fin[1])
        else:
            eng = self._large_engine()
            self.stage_iters = []
            mu = mu_init
            for i in range(T):
                self.vprint(f'\nIteration -- {i+1}:')
                lr_adam, success = lr, False
                while success is False:
                    W_temp, success = self.minimize(self.W_est.copy(), mu, iters[i], s[i], lr=lr_adam,
                                                    beta_1=beta_1, beta_2=beta_2)
                    if success is False:
                        self.vprint('Retrying with larger s')
                        lr_adam *= 0.5
                        s[i] += 0.1
                self.stage_iters.append(self.last_iters)
                self.W_est = W_temp
                mu *= mu_factor
            self.h_final, _ = self._h(self.W_est)
            self.score_final, _ = self._score(self.W_est)
            del eng

    # ------------------------------------------------------------------ fit (linear.py:335-462)
    def fit(self, X: np.ndarray, lambda1: float = 0.03, w_threshold: float = 0.3, T: int = 5,
            mu_init: float = 1.0, mu_factor: float = 0.1,
            s: typing.Union[typing.List[float], float] = [1.0, .9, .8, .7, .6],
            warm_iter: int = 3e4, max_iter: int = 6e4, lr: float = 0.0003, checkpoint: int = 1000,
            beta_1: float = 0.99, beta_2: float = 0.999,
            exclude_edges: typing.Optional[typing.List[typing.Tuple[int, int]]] = None,
            include_edges: typing.Optional[typing.List[typing.Tuple[int, int]]] = None) -> np.ndarray:
        _lib.require_device()
        t0 = time.time()
        self.X, self.lambda1, self.checkpoint = X, lambda1, checkpoint
        self.n, self.d = X.shape
        self.Id = np.eye(self.d).astype(self.dtype)
        self.checkpoint_log = []

        # centring + covariance on device; the centred X is copied back into the caller's
        # array to keep the reference's in-place side effect (linear.py:410-411, Q8)
        Xd = self._dev(X)[None].contiguous()
        self._n_total = self.n
        if self._group is None:
            cov = center_cov(Xd, center=(self.loss_type == 'l2'))
        else:                                   # row-sharded: global n, global column means, summed cov
            from .parallel import allreduce_sum_
            nt = allreduce_sum_(torch.tensor([float(self.n)], dtype=torch.float64, device=self._device), self._group)
            self._n_total = int(nt.item())
            if self.loss_type == 'l2':
                mean = allreduce_sum_(Xd[0].sum(dim=0), self._group) / self._n_total
                Xd[0] -= mean
            cov = center_cov(Xd, center=False)
            cov *= self.n / self._n_total
            allreduce_sum_(cov, self._group)
        if self.loss_type == 'l2':
            self.X[...] = Xd[0].cpu().numpy()
        self._X_dev = Xd[0]
        self._cov_dev = cov[0]
        self.cov = cov[0].cpu().numpy()

        self._run_path(lambda1, T, mu_init, mu_factor, s, warm_iter, max_iter, lr, checkpoint, beta_1, beta_2,
                       exclude_edges, include_edges)
        self.W_raw = self.W_est.copy()
        self.W_est[np.abs(self.W_est) < w_threshold] = 0
        self._slog.close()                                  # linear.py:460
        self.fit_seconds = time.time() - t0
        return self.W_est
