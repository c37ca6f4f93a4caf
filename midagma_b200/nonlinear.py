"""Drop-in ``DagmaMLP`` / ``DagmaNonlinear`` / ``LocallyConnected`` on the B200 kernels
(reference: src/dagma/nonlinear.py, src/dagma/locally_connected.py).

Same class names, constructor arguments, parameter names and shapes (``fc1.weight
[d*m1, d]``, ``fc1.bias``, ``fc2.0.weight [d, m1, 1]``, ``fc2.0.bias``) so ``state_dict``s
interchange with the reference; same defaults and failure behaviour (``minimize`` returns
``False`` when ``h < 0``; ``fit`` restores the stage-start parameters, halves ``lr``, turns on
the exponential decay and retries with ``s = 1``).  The reference differentiates with torch
autograd on the CPU; here one inner iteration is a fixed sequence of hand-written kernels
(closed-form backward, see csrc/mlp.cu) replayed as a CUDA graph, and the host only
synchronises at the convergence checkpoints.  ``dims = [d, m1, 1]`` (the reference's and
BASELINE.json's configuration) runs on fused forward / backward kernels; any other stack
``[d, m1, ..., 1]`` (and the degenerate ``[d, 1]``) runs layer by layer on the generic
LocallyConnected kernels.

``fit_batch`` / ``minimize_batch`` run many independent ``[d, m1, 1]`` problems of one shape (d <= 64, m1 <= 40) in
one launch, one CTA per problem (csrc/mlp_batch.cu); other shapes run one ``DagmaNonlinear`` after the other.
"""
from __future__ import annotations

import copy
import typing

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from ._large import gemm

__all__ = ["DagmaMLP", "DagmaNonlinear", "LocallyConnected", "fit_batch", "minimize_batch"]

ST_DOUBLES = 17
(F_MU, F_S, F_LR, F_LAM1, F_LAM2, F_B1, F_B2, F_LAD, F_H, F_MIN, F_SS, F_L1, F_OBJ, F_SCORE, F_GAMMA) = range(15)
I_STEP, I_HALTED, I_INFO = 0, 1, 2


def _cuda64(x) -> torch.Tensor:
    _lib.require_device()
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(x)
    return x.detach().to(device="cuda", dtype=torch.float64).contiguous()


class LocallyConnected(nn.Module):
    """d independent ``m1 -> m2`` linear maps (locally_connected.py:6); forward runs on the GPU."""

    def __init__(self, num_linear: int, input_features: int, output_features: int, bias: bool = True):
        super().__init__()
        self.num_linear, self.input_features, self.output_features = num_linear, input_features, output_features
        self.weight = nn.Parameter(torch.Tensor(num_linear, input_features, output_features))
        if bias:
            self.bias = nn.Parameter(torch.Tensor(num_linear, output_features))
        else:
            self.register_parameter('bias', None)
        self.reset_parameters()

    @torch.no_grad()
    def reset_parameters(self):
        bound = (1.0 / self.input_features) ** 0.5            # locally_connected.py:49-53
        nn.init.uniform_(self.weight, -bound, bound)
        if self.bias is not None:
            nn.init.uniform_(self.bias, -bound, bound)

    @torch.no_grad()
    def forward(self, input: torch.Tensor) -> torch.Tensor:
        _lib.require_device()
        x = _cuda64(input)
        n, d, m1 = x.shape
        out = torch.empty(n, d, self.output_features, dtype=torch.float64, device="cuda")
        b = _cuda64(self.bias) if self.bias is not None else None
        _lib.check(_lib.load().dagma_locally_connected_f64(
            _lib.stream_ptr(), n, d, m1, self.output_features, x.data_ptr(), _cuda64(self.weight).data_ptr(),
            b.data_ptr() if b is not None else None, out.data_ptr()), "dagma_locally_connected_f64")
        return out.to(input.device)

    def extra_repr(self) -> str:
        return 'num_linear={}, in_features={}, out_features={}, bias={}'.format(
            self.num_linear, self.input_features, self.output_features, self.bias is not None)


class DagmaMLP(nn.Module):
    """Structural equations as MLPs (nonlinear.py:14)."""

    def __init__(self, dims: typing.List[int], bias: bool = True, dtype: torch.dtype = torch.double):
        torch.set_default_dtype(dtype)                          # global side effect kept (Q13)
        super().__init__()
        assert len(dims) >= 2
        assert dims[-1] == 1
        self.dims, self.d = dims, dims[0]
        self.I = torch.eye(self.d)
        self.fc1 = nn.Linear(self.d, self.d * dims[1], bias=bias)
        nn.init.zeros_(self.fc1.weight)
        nn.init.zeros_(self.fc1.bias)
        layers = []
        for l in range(len(dims) - 2):
            layers.append(LocallyConnected(self.d, dims[l + 1], dims[l + 2], bias=bias))
        self.fc2 = nn.ModuleList(layers)

    # ---- flat parameter vector  theta = [W1 | b1 | fc2.0.weight | fc2.0.bias | fc2.1.weight | ...]
    def _params(self):
        # bias=False never gets here: like the reference, the constructor fails in nn.init.zeros_(self.fc1.bias)
        # (nonlinear.py:38, AttributeError) -- DagmaMLP only exists with biases; LocallyConnected alone takes bias=False
        out = [self.fc1.weight, self.fc1.bias]
        for fc in self.fc2:
            out += [fc.weight, fc.bias]
        return out

    def pack(self) -> torch.Tensor:
        return torch.cat([_cuda64(p).reshape(-1) for p in self._params()])

    @torch.no_grad()
    def unpack(self, theta: torch.Tensor) -> None:
        off = 0
        for p in self._params():
            k = p.numel()
            p.copy_(theta[off:off + k].reshape(p.shape).to(p.device, p.dtype))
            off += k

    @torch.no_grad()
    def forward(self, x: torch.Tensor) -> torch.Tensor:       # [n, d] -> [n, d]
        eng = _MlpEngine(self, _cuda64(x))
        return eng.forward().to(x.device)

    def _aux(self) -> "_MlpEngine":
        """One data-less engine per model for the helper calls below (its buffers -- among them the workspace of the
        inverse -- are allocated once); the parameters are re-read on every call.

        These helpers run under ``torch.no_grad()`` and return tensors detached from the parameters: the kernels carry
        the closed-form backward, there is no autograd graph (``model.h_func(s).backward()`` as in reference-style
        user code is not supported; ``DagmaNonlinear.minimize`` / ``fit`` is the optimiser)."""
        eng = self.__dict__.get("_aux_engine")
        if eng is None:
            eng = _MlpEngine(self, None)
            self.__dict__["_aux_engine"] = eng             # not a module attribute: stays out of state_dict / deepcopy
        else:
            eng.theta.copy_(self.pack())
        return eng

    def __deepcopy__(self, memo):
        import copy as _copy
        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k != "_aux_engine":
                new.__dict__[k] = _copy.deepcopy(v, memo)
        return new

    @torch.no_grad()
    def h_func(self, s: float = 1.0) -> torch.Tensor:
        eng = self._aux()
        eng.h(s)
        st = eng.pull()[0]
        return torch.tensor(float(st[F_H]), dtype=torch.float64)

    @torch.no_grad()
    def fc1_l1_reg(self) -> torch.Tensor:
        return torch.tensor(self._aux().l1(), dtype=torch.float64)

    @torch.no_grad()
    def fc1_to_adj(self) -> np.ndarray:                        # [j * m1, i] -> [i, j]
        eng = self._aux()
        eng.adj()
        return np.sqrt(eng.A.cpu().numpy())


class _MlpEngine:
    """Device buffers + launch sequences for one (model, X) pair."""

    def __init__(self, model: DagmaMLP, X: typing.Optional[torch.Tensor], group=None, n_total=None, peer_cache=None):
        _lib.require_device()
        self.lib = _lib.load()
        self.model = model
        self.d, self.m1 = model.d, model.dims[1]
        d, P = self.d, self.d * self.m1
        self.P = P
        self.widths = [int(w) for w in model.dims[1:]]         # LC layer l maps widths[l] -> widths[l + 1]
        self.L = len(self.widths) - 1
        self.fused = (self.L == 1)                             # [d, m1, 1]: fused forward / backward kernels
        self.lc_off, off = [], P * d + P                       # (offset of fc2.l.weight, of fc2.l.bias) in theta
        for l in range(self.L):
            mi, mo = self.widths[l], self.widths[l + 1]
            self.lc_off.append((off, off + d * mi * mo))
            off += d * mi * mo + d * mo
        f64 = dict(dtype=torch.float64, device="cuda")
        self.theta = model.pack()
        self.total = self.theta.numel()
        assert self.total == off, (self.total, off)
        self.m = torch.zeros_like(self.theta)
        self.v = torch.zeros_like(self.theta)
        self.grads = torch.zeros_like(self.theta)
        self.A = torch.empty(d, d, **f64)
        self.Minv = torch.empty(d, d, **f64)
        self.l1_partial = torch.zeros((d * d + 255) // 256, **f64)
        self.state = torch.zeros(ST_DOUBLES, **f64)
        self.state_host = torch.zeros(ST_DOUBLES, dtype=torch.float64).pin_memory()
        self.ws = torch.empty(self.lib.dagma_large_workspace_bytes(d) // 8 + 8, **f64)
        self.group, self.graph = group, None
        self.one_kernel = False
        self._peer = None
        # NCCL all-reduces are captured inside the iteration graph (DAGMA_GRAPH_NCCL=0: eager launches)
        self._graph_collectives = False
        if group is not None:
            import os
            import torch.distributed as dist
            self._graph_collectives = (dist.get_backend(group) == "nccl"
                                       and os.environ.get("DAGMA_GRAPH_NCCL", "1") != "0")
        self._side = None
        if X is not None:
            self.X = X
            self.n = X.shape[0]
            self.n_total = n_total or self.n
            self.Xt = X.t().contiguous()
            self.Zt = torch.empty(P, self.n, **f64)
            self.res = torch.empty(d, self.n, **f64)
            chunks = (self.n + 255) // 256
            self.S_partial = torch.empty(chunks * d, **f64)
            width = 2 * P + d
            if not self.fused:                                 # activations of every layer, [d * width][n]
                self.acts = [self.Zt] + [torch.empty(d * w, self.n, **f64) for w in self.widths[1:]]
                width = max([d * self.widths[l] * self.widths[l + 1] + d * self.widths[l + 1]
                             for l in range(self.L)] + [1])
            self.part = torch.empty(chunks * width, **f64)
            self.kws = torch.empty(148 * P * d + 8, **f64)
            # [d, m1, 1] on one GPU: the whole iteration (and every iteration up to the next checkpoint) as one
            # persistent kernel, csrc/mlp_iter.cu (DAGMA_MLP_FUSED=0: the launch sequence below, replayed as a graph)
            # Rows sharded over the GPUs of one box: the same kernel on every GPU, the gradient sums and S summed INSIDE it
            # over NVLink peer memory (DAGMA_MLP_PEER=0: launch sequence + NCCL all-reduces)
            import os
            self.one_kernel = (self.fused and os.environ.get("DAGMA_MLP_FUSED", "1") != "0"
                               and bool(self.lib.dagma_mlp_iter_supported(self.n, d, self.m1)))
            if group is not None:
                # the exchange buffers outlive the engine (DagmaNonlinear re-creates it per minimize call, Q13): they
                # are created once per (shape, group) and handed on through `peer_cache`; every rank decides alike
                from ._peer import PeerExchange
                import torch.distributed as dist
                want = self.one_kernel and os.environ.get("DAGMA_MLP_PEER", "1") != "0"
                key = (d, self.m1, dist.get_world_size(group))
                cache = peer_cache if peer_cache is not None else {}
                if key not in cache:
                    nbytes = self.lib.dagma_mlp_iter_exchange_bytes(d, self.m1, key[2]) if self.fused else 0
                    cache[key] = PeerExchange.create(group, nbytes, torch.device("cuda", torch.cuda.current_device()), True)
                ok = PeerExchange._agree(group, torch.device("cuda", torch.cuda.current_device()),
                                         want and cache[key] is not None)
                self._peer = cache[key] if ok else None
                self.one_kernel = self._peer is not None
            if self.one_kernel:
                self.iter_ws = torch.empty(self.lib.dagma_mlp_iter_workspace_doubles(self.n, d, self.m1), **f64)
                self.iter_sync = torch.zeros(4, dtype=torch.int32, device="cuda")

    def _sptr(self, f):
        return self.state.data_ptr() + 8 * f

    def _iptr(self, slot):
        return self.state.data_ptr() + 8 * 15 + 4 * slot

    def pull(self):
        self.state_host.copy_(self.state)
        ints = self.state_host[15:].view(torch.int32)
        if int(ints[I_INFO]) == 99:
            raise _lib.DagmaB200Error("dagma_mlp_iter_f64: a grid barrier timed out (the grid was not co-resident)")
        return self.state_host, int(ints[I_STEP]), int(ints[I_HALTED])

    # ---- pieces
    def adj(self):
        _lib.check(self.lib.dagma_mlp_adj_f64(_lib.stream_ptr(), self.d, self.m1, self.theta.data_ptr(),
                                              self.A.data_ptr(), self.l1_partial.data_ptr()), "dagma_mlp_adj_f64")

    def l1(self) -> float:
        self.adj()
        return float(self.l1_partial.sum().item())

    def h(self, s: float):
        self.adj()
        self._h_inverse(s)

    def _h_inverse(self, s: float):
        _lib.check(self.lib.dagma_logdet_inv_ws_f64(
            _lib.stream_ptr(), self.d, float(s), self.A.data_ptr(), self.d, 0, self._sptr(F_LAD), self._sptr(F_H),
            self.Minv.data_ptr(), None, self.d, self._sptr(F_MIN), self._iptr(I_INFO), self.ws.data_ptr(),
            self.ws.numel() * 8), "dagma_logdet_inv_ws_f64")

    def _tptr(self, off):
        return self.theta.data_ptr() + 8 * off

    def _forward_stack(self, out=None):
        """Layer-by-layer forward of a general LocallyConnected stack (nonlinear.py:60-65)."""
        d, n, P, S = self.d, self.n, self.P, _lib.stream_ptr()
        optr = out.data_ptr() if out is not None else None
        if self.L == 0:                                        # dims = [d, 1]: x_hat = fc1(x)
            _lib.check(self.lib.dagma_mlp_residual_f64(
                S, n, d, self.Zt.data_ptr(), self._tptr(P * d), self.Xt.data_ptr(), self.res.data_ptr(), optr,
                self.S_partial.data_ptr(), self.l1_partial.data_ptr(), self.state.data_ptr()), "dagma_mlp_residual_f64")
            return
        for l in range(self.L):
            ow, ob = self.lc_off[l]
            _lib.check(self.lib.dagma_lc_forward_f64(
                S, n, d, self.widths[l], self.widths[l + 1], self.acts[l].data_ptr(),
                self._tptr(P * d) if l == 0 else None, self._tptr(ow), self._tptr(ob), self.acts[l + 1].data_ptr()),
                "dagma_lc_forward_f64")
        _lib.check(self.lib.dagma_mlp_residual_f64(
            S, n, d, self.acts[self.L].data_ptr(), None, self.Xt.data_ptr(), self.res.data_ptr(), optr,
            self.S_partial.data_ptr(), self.l1_partial.data_ptr(), self.state.data_ptr()), "dagma_mlp_residual_f64")

    def _backward_stack(self):
        """Closed-form backward of the stack: un-scaled sums into self.grads (all but fc1.weight)."""
        d, n, P, S = self.d, self.n, self.P, _lib.stream_ptr()
        dzn = self.res
        for l in reversed(range(self.L)):
            ow, _ = self.lc_off[l]
            _lib.check(self.lib.dagma_lc_backward_f64(
                S, n, d, self.widths[l], self.widths[l + 1], self.acts[l].data_ptr(), dzn.data_ptr(), self._tptr(ow),
                self.part.data_ptr(), self.grads.data_ptr() + 8 * ow), "dagma_lc_backward_f64")
            dzn = self.acts[l]
        _lib.check(self.lib.dagma_row_sums_f64(S, P, n, dzn.data_ptr(), self.grads.data_ptr() + 8 * P * d),
                   "dagma_row_sums_f64")
        return dzn

    def _forward(self, out=None):
        W1 = self.theta[:self.P * self.d].view(self.P, self.d)
        gemm(W1, self.Xt, self.Zt)
        if not self.fused:
            return self._forward_stack(out)
        _lib.check(self.lib.dagma_mlp_forward_f64(
            _lib.stream_ptr(), self.n, self.d, self.m1, self.Zt.data_ptr(), self.theta.data_ptr(), self.Xt.data_ptr(),
            self.res.data_ptr(), out.data_ptr() if out is not None else None, self.S_partial.data_ptr(),
            self.l1_partial.data_ptr(), self.state.data_ptr()), "dagma_mlp_forward_f64")

    def forward(self) -> torch.Tensor:
        out = torch.empty(self.n, self.d, dtype=torch.float64, device="cuda")
        self.adj()
        self._forward(out)
        return out

    def iteration(self, s: float):
        self.evaluate(s)
        _lib.check(self.lib.dagma_mlp_adam_ex_f64(
            _lib.stream_ptr(), self.d, self.m1, self.total, self.state.data_ptr(), self.theta.data_ptr(),
            self.grads.data_ptr(), self.m.data_ptr(), self.v.data_ptr(), self.Minv.data_ptr()), "dagma_mlp_adam_ex_f64")

    def evaluate(self, s: float):
        """h, forward, objective and the (un-scaled) gradient sums at the current parameters."""
        # the on-chip inverse of sI - A (one CTA, a serial pivot chain) runs on a side stream beside the forward pass;
        # they meet again at the objective (captured as parallel graph branches)
        self.adj()
        if self._side is None:
            self._side = torch.cuda.Stream()
        cur = torch.cuda.current_stream()
        self._side.wait_stream(cur)
        with torch.cuda.stream(self._side):
            self._h_inverse(s)
        self._forward()
        cur.wait_stream(self._side)
        if self.group is not None:
            torch.distributed.all_reduce(self.state[F_SS:F_SS + 1], group=self.group)
        _lib.check(self.lib.dagma_mlp_objective_f64(_lib.stream_ptr(), self.state.data_ptr(), self.n_total, self.d),
                   "dagma_mlp_objective_f64")
        dZt = self.Zt
        if self.fused:
            _lib.check(self.lib.dagma_mlp_backward_f64(
                _lib.stream_ptr(), self.n, self.d, self.m1, self.Zt.data_ptr(), self.theta.data_ptr(), self.res.data_ptr(),
                self.part.data_ptr(), self.grads.data_ptr() + 8 * self.P * self.d), "dagma_mlp_backward_f64")
        else:
            dZt = self._backward_stack()
        gW1 = self.grads[:self.P * self.d].view(self.P, self.d)
        gemm(dZt, self.X, gW1, ws=self.kws)
        if self.group is not None:
            torch.distributed.all_reduce(self.grads, group=self.group)

    def replay(self, s: float, n: int):
        if self.one_kernel and self._peer is not None:
            _lib.check(self.lib.dagma_mlp_iter_sharded_f64(
                _lib.stream_ptr(), self.n, self.n_total, self.d, self.m1, int(n), self.state.data_ptr(),
                self.theta.data_ptr(), self.m.data_ptr(), self.v.data_ptr(), self.X.data_ptr(), self.iter_ws.data_ptr(),
                self.Minv.data_ptr(), self.iter_sync.data_ptr(), self._peer.rank, self._peer.world, self._peer.ptrs),
                "dagma_mlp_iter_sharded_f64")
            return
        if self.one_kernel:
            _lib.check(self.lib.dagma_mlp_iter_f64(
                _lib.stream_ptr(), self.n, self.n_total, self.d, self.m1, int(n), self.state.data_ptr(),
                self.theta.data_ptr(), self.m.data_ptr(), self.v.data_ptr(), self.X.data_ptr(), self.iter_ws.data_ptr(),
                self.Minv.data_ptr(), self.iter_sync.data_ptr()), "dagma_mlp_iter_f64")
            return
        if self.group is not None and not self._graph_collectives:
            for _ in range(n):
                self.iteration(s)
            return
        if self.graph is None:
            snap = (self.theta.clone(), self.m.clone(), self.v.clone(), self.state.clone())
            self.iteration(s)                                  # warm-up
            torch.cuda.synchronize()
            for dst, src in zip((self.theta, self.m, self.v, self.state), snap):
                dst.copy_(src)
            from ._large import capture_graph
            self.graph = capture_graph(lambda: self.iteration(s))
        for _ in range(n):
            self.graph.replay()

    def grads_scaled(self) -> dict:
        """Gradients of mu*(score + lambda1 |fc1|) + h as the reference's autograd returns them
        (before weight decay): used by the parity tests."""
        st, _, _ = self.pull()
        mu, lam1 = float(st[F_MU]), float(st[F_LAM1])
        gs = mu * self.d / float(st[F_SS])
        g = (gs * self.grads).clone()
        P, d, m1 = self.P, self.d, self.m1
        w1 = self.theta[:P * d].view(d, m1, d)
        g[:P * d] += (mu * lam1 * torch.sign(w1) + 2.0 * w1 * self.Minv[:, None, :]).reshape(-1)
        names = ["fc1.weight", "fc1.bias"]
        for l in range(self.L):
            names += [f"fc2.{l}.weight", f"fc2.{l}.bias"]
        out, off = {}, 0
        for nme, prm in zip(names, self.model._params()):
            k = prm.numel()
            out[nme] = g[off:off + k].cpu().numpy().reshape(tuple(prm.shape))
            off += k
        return out


class DagmaNonlinear:
    """DAGMA with MLP structural equations (nonlinear.py:118)."""

    def __init__(self, model: nn.Module, verbose: bool = False, dtype: torch.dtype = torch.double):
        self.vprint = print if verbose else lambda *a, **k: None
        self.model = model
        self.dtype = dtype
        self.group = None            # torch.distributed group when the rows of X are sharded across ranks
        self.n_total = None
        self.n_iters = 0

    @torch.no_grad()
    def log_mse_loss(self, output: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
        _lib.require_device()
        n, d = target.shape
        a, b = _cuda64(output), _cuda64(target)
        partial = torch.empty(592, dtype=torch.float64, device="cuda")
        out = torch.empty(1, dtype=torch.float64, device="cuda")
        _lib.check(_lib.load().dagma_sumsq_diff_f64(_lib.stream_ptr(), a.numel(), a.data_ptr(), b.data_ptr(),
                                                    partial.data_ptr(), 592, out.data_ptr()), "dagma_sumsq_diff_f64")
        return (0.5 * d * torch.log(out[0] / n)).cpu()

    def minimize(self, max_iter: float, lr: float, lambda1: float, lambda2: float, mu: float, s: float,
                 lr_decay: float = False, tol: float = 1e-6, pbar=None) -> bool:
        self.vprint(f'\nMinimize s={s} -- lr={lr}')
        if getattr(self, "_peer_cache", None) is None:
            self._peer_cache = {}
        eng = _MlpEngine(self.model, self.X, self.group, self.n_total, peer_cache=self._peer_cache)   # optimizer re-created (Q13)
        sh = eng.state_host
        sh.zero_()
        for f, val in ((F_MU, mu), (F_S, s), (F_LR, lr), (F_LAM1, lambda1), (F_LAM2, lambda2), (F_B1, 0.99),
                       (F_B2, 0.999), (F_GAMMA, 0.8 if lr_decay is True else 1.0)):
            sh[f] = float(val)
        eng.state.copy_(sh)
        self._engine = eng
        max_iter = int(max_iter)
        obj_prev, i_next, ok = 1e16, 0, True
        while i_next < max_iter:
            # run up to and including the next checkpoint iteration (i % checkpoint == 0 or the last one)
            i_ck = i_next if i_next % self.checkpoint == 0 else min((i_next // self.checkpoint + 1) * self.checkpoint,
                                                                    max_iter - 1)
            i_ck = min(i_ck, max_iter - 1)
            eng.replay(s, i_ck - i_next + 1)
            st, step, halted = eng.pull()
            self.n_iters += step - i_next
            if halted:                                         # nonlinear.py:215-217
                self.vprint(f'Found h negative {float(st[F_H])} at iter {step}')
                ok = False
                break
            i_next = i_ck + 1
            obj_new = float(st[F_OBJ])
            self.vprint(f"\nInner iteration {i_ck}\n\th(W(model)): {float(st[F_H])}\n\tscore(model): {obj_new}")
            if np.abs((obj_prev - obj_new) / obj_prev) <= tol:  # nonlinear.py:231
                break
            obj_prev = obj_new
        self.model.unpack(eng.theta)
        if pbar is not None:
            pbar.update(max_iter)
        return ok

    def close(self) -> None:
        """Release the NVLink peer mappings of a row-sharded model (collective over the group; optional otherwise)."""
        cache, self._peer_cache = getattr(self, "_peer_cache", None) or {}, {}
        self._engine = None
        for px in cache.values():
            if px is not None:
                px.close()

    def fit(self, X: typing.Union[torch.Tensor, np.ndarray], lambda1: float = .02, lambda2: float = .005,
            T: int = 4, mu_init: float = .1, mu_factor: float = .1, s: float = 1.0, warm_iter: int = 5e4,
            max_iter: int = 8e4, lr: float = .0002, w_threshold: float = 0.3, checkpoint: int = 1000) -> np.ndarray:
        _lib.require_device()
        torch.set_default_dtype(self.dtype)
        if type(X) == torch.Tensor:
            self.X = _cuda64(X)
        elif type(X) == np.ndarray:
            self.X = _cuda64(torch.from_numpy(X))
        else:
            ValueError("X should be numpy array or torch Tensor.")
        self.checkpoint = checkpoint
        mu = mu_init
        if type(s) == list:
            if len(s) < T:
                self.vprint(f"Length of s is {len(s)}, using last value in s for iteration t >= {len(s)}")
                s = s + (T - len(s)) * [s[-1]]
        elif type(s) in [int, float]:
            s = T * [s]
        else:
            ValueError("s should be a list, int, or float.")
        self.stage_iters = []
        self.minimize_calls = []          # (lr, s, success, lr_decay) of every minimize call, retries included
        for i in range(int(T)):
            self.vprint(f'\nDagma iter t={i+1} -- mu: {mu}', 30 * '-')
            success, s_cur = False, s[i]
            inner_iter = int(max_iter) if i == T - 1 else int(warm_iter)
            model_copy = copy.deepcopy(self.model)
            lr_decay = False
            while success is False:
                before = self.n_iters
                success = self.minimize(inner_iter, lr, lambda1, lambda2, mu, s_cur, lr_decay)
                self.minimize_calls.append((float(lr), float(s_cur), int(bool(success)), int(bool(lr_decay))))
                if success is False:
                    self.model.load_state_dict(model_copy.state_dict().copy())
                    lr *= 0.5
                    lr_decay = True
                    if lr < 1e-10:
                        break
                    s_cur = 1
            self.stage_iters.append(self.n_iters - before)
            mu *= mu_factor
        W_est = self.model.fc1_to_adj()
        W_est[np.abs(W_est) < w_threshold] = 0
        return W_est


# ------------------------------------------------------------------------------------------------ batched problems
def _batch_inputs(models, X, fname):
    if not isinstance(models, (list, tuple)) or len(models) == 0:
        raise ValueError(f"{fname}: models must be a non-empty list of DagmaMLP")
    dims = list(models[0].dims)
    if any(list(m.dims) != dims for m in models):
        raise ValueError(f"{fname}: every model must have the same dims (got {dims} and others)")
    if isinstance(X, np.ndarray):
        X = torch.from_numpy(X)
    if not isinstance(X, torch.Tensor) or X.dim() != 3 or X.shape[0] != len(models) or X.shape[2] != dims[0]:
        raise ValueError(f"{fname}: X must be [batch, n, d] = [{len(models)}, n, {dims[0]}], "
                         f"got {tuple(X.shape) if hasattr(X, 'shape') else type(X)}")
    if X.shape[1] < 1:
        raise ValueError(f"{fname}: X has no rows")
    return dims, X


def _per_problem(x, batch, name):
    a = np.asarray(x, dtype=np.float64)
    if a.ndim == 0:
        return np.full(batch, float(a))
    if a.shape != (batch,):
        raise ValueError(f"{name} must be a scalar or [{batch}], got shape {a.shape}")
    return a.copy()


class _MlpBatch:
    """Device buffers of a batch of [d, m1, 1] problems on the one-CTA-per-problem kernel (csrc/mlp_batch.cu)."""

    def __init__(self, models, X: torch.Tensor):
        self.lib = _lib.load()
        self.models = models
        self.B, self.n, self.d = X.shape
        self.m1 = int(models[0].dims[1])
        self.X = _cuda64(X)
        self.theta = torch.stack([m.pack() for m in models])
        self.W = self.theta.shape[1]
        self.m = torch.zeros_like(self.theta)
        self.v = torch.zeros_like(self.theta)
        self.grad = torch.empty_like(self.theta)
        self.state = torch.zeros(self.B, ST_DOUBLES, dtype=torch.float64, device="cuda")
        self.iters = torch.zeros(self.B, dtype=torch.int32, device="cuda")
        self.counter = torch.zeros(1, dtype=torch.int32, device="cuda")

    def run(self, idx, max_iter, lr, lambda1, lambda2, mu, s, lr_decay, tol, checkpoint):
        """One minimize call (fresh Adam state) for the problems `idx`; per-problem arrays are indexed by problem.
        Returns (success, iterations) of those problems."""
        idx = np.asarray(idx, dtype=np.int64)
        if idx.size == 0:
            return np.zeros(0, dtype=bool), np.zeros(0, dtype=np.int64)
        sh = np.zeros((idx.size, ST_DOUBLES))
        for f, val in ((F_MU, mu), (F_S, s), (F_LR, lr), (F_LAM1, lambda1), (F_LAM2, lambda2)):
            sh[:, f] = np.asarray(val, dtype=np.float64)[idx]
        sh[:, F_B1], sh[:, F_B2] = 0.99, 0.999
        sh[:, F_GAMMA] = np.where(np.asarray(lr_decay)[idx], 0.8, 1.0)
        rows = torch.from_numpy(idx).cuda()
        self.state[rows] = torch.from_numpy(sh).cuda()          # step = halted = 0
        self.m[rows] = 0.0                                     # optimizer re-created per call (Q13)
        self.v[rows] = 0.0
        full = idx.size == self.B and np.array_equal(idx, np.arange(self.B))
        idx_dev = None if full else rows.to(torch.int32)
        _lib.check(self.lib.dagma_mlp_minimize_batch_f64(
            _lib.stream_ptr(), self.B, self.n, self.d, self.m1, int(max_iter), int(checkpoint), float(tol),
            idx_dev.data_ptr() if idx_dev is not None else None, int(idx.size), self.state.data_ptr(),
            self.theta.data_ptr(), self.m.data_ptr(), self.v.data_ptr(), self.X.data_ptr(), self.grad.data_ptr(),
            self.iters.data_ptr(), self.counter.data_ptr()), "dagma_mlp_minimize_batch_f64")
        halted = self.state[:, 15:].contiguous().view(torch.int32)[:, I_HALTED]
        ok = (halted[rows] == 0).cpu().numpy()
        return ok, self.iters[rows].cpu().numpy().astype(np.int64)

    def write_back(self):
        for b, model in enumerate(self.models):
            model.unpack(self.theta[b])


def _supported(dims, n) -> bool:
    return len(dims) == 3 and bool(_lib.load().dagma_mlp_batch_supported(int(n), int(dims[0]), int(dims[1])))


@torch.no_grad()
def minimize_batch(models, X, max_iter, lr, lambda1, lambda2, mu, s, lr_decay=False, tol=1e-6,
                   checkpoint=1000) -> np.ndarray:
    """``DagmaNonlinear(model).minimize(...)`` for every model, with ``X[b]`` as that model's data
    (nonlinear.py:161-236).  ``models``: DagmaMLP objects of identical ``dims``, updated in place; ``X``: [batch, n, d]
    (host or device, not modified); ``lambda1`` / ``lambda2``: scalar or [batch].  Returns ``success`` [batch].
    ``[d, m1, 1]`` with d <= 64, m1 <= 40 runs in one launch (csrc/mlp_batch.cu); other shapes one model at a time."""
    dims, X = _batch_inputs(models, X, "minimize_batch")
    B, n = X.shape[0], X.shape[1]
    lam1, lam2 = _per_problem(lambda1, B, "lambda1"), _per_problem(lambda2, B, "lambda2")
    _lib.require_device()
    if not _supported(dims, n):
        out = np.zeros(B, dtype=bool)
        for b, model in enumerate(models):
            eq = DagmaNonlinear(model)
            eq.X, eq.checkpoint = _cuda64(X[b]), checkpoint
            out[b] = eq.minimize(max_iter, lr, float(lam1[b]), float(lam2[b]), mu, s, lr_decay, tol)
        return out
    bt = _MlpBatch(models, X)
    full = lambda x: np.full(B, x)                              # noqa: E731
    ok, _ = bt.run(np.arange(B), int(max_iter), full(float(lr)), lam1, lam2, full(float(mu)), full(float(s)),
                   full(lr_decay is True), tol, checkpoint)
    bt.write_back()
    return ok


@torch.no_grad()
def fit_batch(models, X, lambda1=.02, lambda2=.005, T=4, mu_init=.1, mu_factor=.1, s=1.0, warm_iter=5e4, max_iter=8e4,
              lr=2e-4, w_threshold=.3, checkpoint=1000, return_info=False, device=None):
    """``DagmaNonlinear(model).fit(X[b], ...)`` for every model (nonlinear.py:486-530): the same stage loop per
    problem -- a failed minimize restores the stage-start parameters, halves that problem's lr (for the rest of its
    fit), turns on ExponentialLR and retries with s = 1 -- with every minimize call of a stage run for all problems in
    one launch and the retries relaunched for the failed problems only.  ``models`` are updated in place; returns
    W_est [batch, d, d] and, with ``return_info``, a dict of ``W_raw``, ``stage_iters`` (the iterations of each stage's
    last minimize call), ``n_iters`` (of every call) and ``minimize_calls`` (per problem, (lr, s, success, lr_decay)
    of every call), as DagmaNonlinear keeps them.  ``device``: the CUDA device to run on (default: the current one)."""
    if device is not None:
        with torch.cuda.device(torch.device(device)):
            return fit_batch(models, X, lambda1, lambda2, T, mu_init, mu_factor, s, warm_iter, max_iter, lr,
                             w_threshold, checkpoint, return_info)
    dims, X = _batch_inputs(models, X, "fit_batch")
    B, n = X.shape[0], X.shape[1]
    lam1, lam2 = _per_problem(lambda1, B, "lambda1"), _per_problem(lambda2, B, "lambda2")
    T = int(T)
    if isinstance(s, list):
        s = s + (T - len(s)) * [s[-1]] if len(s) < T else s
    elif isinstance(s, (int, float)):
        s = T * [s]
    else:
        raise ValueError("s should be a list, int, or float.")
    _lib.require_device()
    if not _supported(dims, n):
        eqs = []
        for b, model in enumerate(models):
            eq = DagmaNonlinear(model)
            eq.fit(X[b], lambda1=float(lam1[b]), lambda2=float(lam2[b]), T=T, mu_init=mu_init, mu_factor=mu_factor,
                   s=list(s), warm_iter=warm_iter, max_iter=max_iter, lr=lr, w_threshold=w_threshold,
                   checkpoint=checkpoint)
            eqs.append(eq)
        stage_iters = [list(eq.stage_iters) for eq in eqs]
        calls = [list(eq.minimize_calls) for eq in eqs]
        n_iters = np.array([eq.n_iters for eq in eqs], dtype=np.int64)
    else:
        bt = _MlpBatch(models, X)
        lr_b = np.full(B, float(lr))
        n_iters = np.zeros(B, dtype=np.int64)
        stage_iters = [[] for _ in range(B)]
        calls = [[] for _ in range(B)]
        mu = mu_init
        for i in range(T):
            inner = int(max_iter) if i == T - 1 else int(warm_iter)
            snap = bt.theta.clone()
            s_cur = np.full(B, float(s[i]))
            decay = np.zeros(B, dtype=bool)
            last = np.zeros(B, dtype=np.int64)
            todo = np.arange(B)
            while todo.size:
                ok, its = bt.run(todo, inner, lr_b, lam1, lam2, np.full(B, float(mu)), s_cur, decay, 1e-6, checkpoint)
                n_iters[todo] += its
                last[todo] = its
                for b, good in zip(todo, ok):
                    calls[b].append((float(lr_b[b]), float(s_cur[b]), int(good), int(decay[b])))
                failed = todo[~ok]
                if failed.size:
                    rows = torch.from_numpy(failed).cuda()
                    bt.theta[rows] = snap[rows]
                    lr_b[failed] *= 0.5
                    decay[failed] = True
                    s_cur[failed] = 1.0
                todo = failed[lr_b[failed] >= 1e-10]
            for b in range(B):                     # the stage's last minimize call, as DagmaNonlinear.fit counts it
                stage_iters[b].append(int(last[b]))
            mu *= mu_factor
        bt.write_back()
    W_raw = np.stack([model.fc1_to_adj() for model in models])
    W_est = W_raw.copy()
    W_est[np.abs(W_est) < w_threshold] = 0
    if not return_info:
        return W_est
    return W_est, {"W_raw": W_raw, "stage_iters": stage_iters, "n_iters": n_iters, "minimize_calls": calls}
