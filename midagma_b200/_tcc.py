"""Spectral trek-cycle-coupling penalty on device (reference: src/notreks/notreks.py:156-239, 291-378).

penalty = rho(A) - baseline,  A = [[W o W, w S], [I, (W o W)^T]]  (2d x 2d, S the indicator of the pair set I),
rho the Perron root;  d rho / dA = u v^T / (u.v + eps) with the left / right Perron vectors, folded back onto W through
the blocks A11 = W o W and A22 = (W o W)^T  =>  gradW = 2 W o (u1 v1^T + v2 u2^T) / (u.v + eps).

``method="power"`` follows the reference step by step (n_iter products from the all-ones vector, :178-194).  The eig
methods (``eig_numpy`` -- what ``trek_value_grad`` uses --, ``eig_torch``) return the Perron pair of a dense
eigendecomposition (LAPACK geev) in the reference; here the same pair is reached by iterating the power step on
A + shift I until the vectors stop moving (||dv|| <= 1e-13).  That is the same answer whenever the Perron root is
simple -- the ``DAG_learning`` and ``approx_trek_graph`` versions, which only need the pair of A.  It is NOT offered
for ``exact_trek_graph``: the baseline matrix B = [[W o W, 0], [I, (W o W)^T]] carries every eigenvalue twice and is
defective, its eigenvectors are whatever geev returns (numpy and torch disagree by 1e-3 on the reference's own
gradient, tests/golden/tcc_spectral.npz), so there is nothing to be in parity with.  ``exact_original_graph`` fails in
the reference (shape error in ``_gradW2_from_gradA``, :285-287) and fails here the same way.
"""
from __future__ import annotations

import warnings

import numpy as np
import torch

from . import _lib

# the schedule of ``PerronSolver.converged``; the on-chip TCC fit (DAGMA_TCC_EIG_* of include/dagma_b200.h) runs the same
EIG_WARMUP = 8           # unshifted steps from the all-ones vectors
EIG_NILPOTENT = 1e-200   # |rho| of the warm-up vectors at or below which A is taken as nilpotent
EIG_SHIFT = 0.25         # the chunks iterate on A + EIG_SHIFT * rho0 I
EIG_TOL = 1e-13          # ||v_k - v_{k-chunk}|| at which the iterated Perron pair is taken as converged
EIG_CHUNK = 64
EIG_MAX_CHUNKS = 600


class PerronSolver:
    """Perron pair (rho, u, v) of an n x n non-negative device matrix; every buffer is allocated once."""

    def __init__(self, n: int):
        _lib.require_device()
        self.lib = _lib.load()
        self.n = n
        f64 = dict(dtype=torch.float64, device="cuda")
        self.v, self.u = torch.empty(n, **f64), torch.empty(n, **f64)
        self.scal = torch.zeros(4, **f64)                       # rho, u.v, u.u, v.v
        self.ws = torch.empty(self.lib.dagma_power_workspace_bytes(n) // 8 + 8, **f64)
        self._prev = torch.empty(n, **f64)
        self._d4 = torch.empty(4, **f64)

    def _run(self, A, square, shift, n_iter, eps, start):
        _lib.check(self.lib.dagma_perron_power_f64(
            _lib.stream_ptr(), self.n, A.data_ptr(), A.stride(0), int(square), float(shift), int(n_iter), float(eps),
            int(start), self.v.data_ptr(), self.u.data_ptr(), self.scal.data_ptr(), self.ws.data_ptr(),
            self.ws.numel() * 8), "dagma_perron_power_f64")

    def power(self, A: torch.Tensor, n_iter: int, eps: float, square: bool = False):
        """notreks.py:178-194; no host synchronisation (CUDA-graph capturable)."""
        self._run(A, square, 0.0, n_iter, eps, 0)

    def converged(self, A: torch.Tensor, eps: float, square: bool = False) -> int:
        """The Perron pair a dense eigensolver returns, by power steps on A + shift I; returns the iterations used."""
        self._run(A, square, 0.0, EIG_WARMUP, eps, 0)
        rho0 = abs(float(self.scal[0].item()))
        if not rho0 > EIG_NILPOTENT:
            # nilpotent matrix (e.g. the block matrix at W = 0 with an acyclic pair set): rho = 0, the iterates vanish
            # and every eigenvector choice gives the same (zero) fold-back 2 W o (...) -- nothing to converge to
            return EIG_WARMUP
        shift = EIG_SHIFT * rho0                                # breaks periodicity, keeps most of the spectral gap
        total = EIG_WARMUP
        for _ in range(EIG_MAX_CHUNKS):
            self._prev.copy_(self.v)
            self._run(A, square, shift, EIG_CHUNK, eps, 1)
            total += EIG_CHUNK
            _lib.check(self.lib.dagma_vec_dots_f64(_lib.stream_ptr(), self.n, self.v.data_ptr(), self._prev.data_ptr(),
                                                   self._d4.data_ptr()), "dagma_vec_dots_f64")
            if float(self._d4[3].item()) <= EIG_TOL * EIG_TOL:
                return total
        warnings.warn("Perron iteration did not converge (Perron root not simple / tiny spectral gap): the vectors "
                      "are the last iterate", RuntimeWarning, stacklevel=3)
        return total


class SpectralTcc:
    """value and gradW of the spectral TCC penalty for one (d, I, w, version, method)."""

    VERSIONS = ("DAG_learning", "exact_trek_graph", "exact_original_graph", "approx_trek_graph")

    def __init__(self, d: int, I, *, w: float = 1.0, version: str = "approx_trek_graph", method: str = "eig_numpy",
                 n_iter: int = 50, eps: float = 1e-12):
        if method not in ("power", "eig_torch", "eig_numpy"):
            raise ValueError("method must be one of {'power','eig_torch','eig_numpy'}")
        if version not in self.VERSIONS:
            raise ValueError("version must be one of {TCCVersion} for spectral")
        if version == "exact_original_graph":
            # the reference folds a d x d gradient as if it were 2d x 2d: (d, d) + (0, 0)^T (notreks.py:285-287, 358)
            raise RuntimeError("The size of tensor a (%d) must match the size of tensor b (0) at non-singleton "
                               "dimension 1 (the reference fails here: exact_original_graph, spectral)" % d)
        if version == "exact_trek_graph" and method != "power":
            raise NotImplementedError(
                "exact_trek_graph with an eig method is ill-posed: the baseline block matrix is defective (every "
                "eigenvalue twice), its eigenvectors depend on the LAPACK build; use method='power'")
        _lib.require_device()
        self.lib = _lib.load()
        I_np = np.asarray(I, dtype=np.int64)
        if I_np.ndim != 2 or I_np.shape[1] != 2:
            raise ValueError("I must be array-like of shape (m,2)")
        self.d, self.w, self.version, self.method = d, float(w), version, method
        self.n_iter, self.eps, self.n_vals = int(n_iter), float(eps), int(I_np.shape[0])
        f64 = dict(dtype=torch.float64, device="cuda")
        S = torch.zeros(d, d, dtype=torch.float64)
        S[I_np[:, 0], I_np[:, 1]] = 1.0
        self.S = S.cuda()
        self.A = torch.empty(2 * d, 2 * d, **f64)
        self.solA = PerronSolver(2 * d)
        self.B = self.solB = None
        if version in ("exact_trek_graph", "approx_trek_graph"):
            self.B = torch.empty(2 * d, 2 * d, **f64)
        if version == "exact_trek_graph":
            self.solB = PerronSolver(2 * d)
        self.Bu = torch.empty(2 * d, **f64)
        self.d4 = torch.zeros(4, **f64)
        self.grad = torch.empty(d, d, **f64)
        self.iterations = 0

    def _assemble(self, W, dst, with_s):
        _lib.check(self.lib.dagma_tcc_assemble_f64(_lib.stream_ptr(), self.d, W.data_ptr(), self.S.data_ptr(), self.w,
                                                   int(with_s), dst.data_ptr()), "dagma_tcc_assemble_f64")

    def _solve(self, sol, M):
        if self.method == "power":
            sol.power(M, self.n_iter, self.eps)
        else:
            self.iterations = sol.converged(M, self.eps)

    def _fold(self, W, a1, b1, a2, b2, num, den, accumulate, out):
        _lib.check(self.lib.dagma_rank2_fold_f64(
            _lib.stream_ptr(), self.d, W.data_ptr() if W is not None else None, a1.data_ptr(), b1.data_ptr(),
            a2.data_ptr(), b2.data_ptr(), float(num), den.data_ptr(), self.eps, int(accumulate), out.data_ptr()),
            "dagma_rank2_fold_f64")

    def compute(self, W: torch.Tensor, out: torch.Tensor = None, fold_w: bool = True) -> torch.Tensor:
        """gradW (``fold_w``) or d penalty / d (W o W) transposed (the form the fused update kernel takes) into
        ``out``; with ``method="power"`` nothing synchronises with the host."""
        d, out = self.d, self.grad if out is None else out
        Wf = W if fold_w else None
        self._assemble(W, self.A, 1)
        self._solve(self.solA, self.A)
        u, v = self.solA.u, self.solA.v
        u1, u2, v1, v2 = u[:d], u[d:], v[:d], v[d:]
        inv_n = 1.0 / self.n_vals
        den_uv = self.solA.scal[1:2]
        # (G11 + G22^T) = (u1 v1^T + v2 u2^T) / (u.v + eps); transposed for the update kernel: (v1 u1^T + u2 v2^T)
        if fold_w:
            self._fold(Wf, u1, v1, v2, u2, inv_n, den_uv, 0, out)
        else:
            self._fold(None, v1, u1, u2, v2, inv_n, den_uv, 0, out)
        if self.version == "exact_trek_graph":
            self._assemble(W, self.B, 0)
            self._solve(self.solB, self.B)
            p, q = self.solB.u, self.solB.v
            den_b = self.solB.scal[1:2]
            if fold_w:
                self._fold(Wf, p[:d], q[:d], q[d:], p[d:], -inv_n, den_b, 1, out)
            else:
                self._fold(None, q[:d], p[:d], p[d:], q[d:], -inv_n, den_b, 1, out)
        elif self.version == "approx_trek_graph":
            # Rayleigh lower bound of rho(B) at uA and its gradient (u1 u1^T + u2 u2^T) / (u.u + eps)   :365-371
            self._assemble(W, self.B, 0)
            _lib.check(self.lib.dagma_matvec_f64(_lib.stream_ptr(), 2 * d, self.B.data_ptr(), 2 * d, 0, u.data_ptr(),
                                                 self.Bu.data_ptr()), "dagma_matvec_f64")
            _lib.check(self.lib.dagma_vec_dots_f64(_lib.stream_ptr(), 2 * d, u.data_ptr(), self.Bu.data_ptr(),
                                                   self.d4.data_ptr()), "dagma_vec_dots_f64")   # [u.Bu, u.u, ., .]
            self._fold(Wf, u1, u1, u2, u2, -inv_n, self.d4[1:2], 1, out)
        return out

    def value(self) -> torch.Tensor:
        """Penalty of the last ``compute`` as a 0-dim device tensor."""
        rho_a = self.solA.scal[0]
        if self.version == "DAG_learning":
            pen = rho_a
        elif self.version == "exact_trek_graph":
            pen = rho_a - self.solB.scal[0]
        else:
            pen = rho_a - self.d4[0] / (self.d4[1] + self.eps)
        return pen / self.n_vals
