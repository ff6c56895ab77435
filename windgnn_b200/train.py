"""Training step of the GCN-GRU on the GPU (BASELINE.json configs[4]).

Mirrors the body of the reference's training loop, ``src/main.py:64-77``::

    outputs = model(adj_matrix, batch_x)          # :66
    optimizer.zero_grad()                         # :69
    loss = lossFunction(outputs, batch_y)         # :72   nn.MSELoss(), :49
    loss.backward()                               # :76
    optimizer.step()                              # :77   torch.optim.Adam(lr=1e-3), :52

Two ways in:

* ``GCN_GRU.forward`` under ``torch.enable_grad()`` goes through ``GcnGruFunction`` — an ordinary
  ``torch.autograd.Function`` whose forward / backward are the library's
  ``wg_gcn_gru_forward_train_f32`` / ``wg_gcn_gru_backward_f32`` — so the reference's loop runs
  unchanged with ``torch.optim.Adam``.
* ``Trainer.step(x, y)`` is the fused step: forward, MSE loss + its gradient, backward into ONE flat
  gradient bucket, one all-reduce of that bucket across the data-parallel ranks (NCCL over NVLink;
  identity for a single process), one fused Adam kernel over the flat parameter buffer.
* Windows over one table (``table[starts[n] : starts[n] + L]``) train without being materialised:
  ``GCN_GRU.forward_windows`` under grad mode (``GcnGruWindowsFunction``) and ``Trainer.step_table``, whose
  loss reads the targets from the table.  GCN, input projection and their gradients run once per table row
  (``wg_gcn_gru_forward_train_windows_f32`` / ``wg_gcn_gru_backward_windows_f32``, DESIGN.md section 10).

PyTorch is plumbing here (device memory, streams, ``torch.distributed``); every arithmetic step is a
kernel of ``libwindgnn_b200.so``.  CUDA only — no CPU fallback.
"""

from __future__ import annotations

from typing import Optional, Sequence

import torch

from . import _lib
from .ops import _attr_shape, _forecast_starts, _graph, _param_dims, _params, _require_cuda_f32, _table_shape


def _stream(dev: torch.device) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def forward_train(adj, x, params: Sequence[torch.Tensor]):
    """Forward that keeps what the backward needs.  Returns ``(out [B,T,H], workspace)``."""
    lib = _lib.load()
    x = _require_cuda_f32("attr_matrix", x)
    dev = x.device
    B, T, S, F_in = _attr_shape(x)
    (adj,) = _graph(adj, S, dev)
    params = _params(params, dev)
    F_hid, F_out, H = _param_dims(S, F_in, params)
    out = torch.empty((B, T, H), dtype=torch.float32, device=dev)
    # 0 bytes: the shape is rejected, and the call below returns the library's code and reason without launching
    nbytes = lib.wg_gcn_gru_train_workspace_bytes(B, T, S, F_in, F_hid, F_out, H)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    _lib.check(lib.wg_gcn_gru_forward_train_f32(
        adj.data_ptr(), x.data_ptr(), *(p.data_ptr() for p in params), out.data_ptr(),
        B, T, S, F_in, F_hid, F_out, H, ws.data_ptr(), ws.numel(), dev.index or 0, _stream(dev)))
    return out, ws


def _grads_bucket(lib, dims, dev, grads: Optional[torch.Tensor]) -> torch.Tensor:
    """``grads``, checked, or a new flat gradient bucket for the model of ``dims = (S, F_in, F_hid, F_out, H)``."""
    n = lib.wg_gcn_gru_param_count(*dims)
    if grads is None:
        return torch.empty(n, dtype=torch.float32, device=dev)
    if grads.numel() != n or not grads.is_cuda or grads.dtype != torch.float32 or not grads.is_contiguous():
        raise RuntimeError(f"grads must be a contiguous CUDA float32 buffer of {n} elements")
    return grads


def backward(adj, x, params: Sequence[torch.Tensor], out, d_out, ws, grads: Optional[torch.Tensor] = None):
    """Flat gradient bucket (state_dict order) of the loss w.r.t. the eight parameter tensors."""
    lib = _lib.load()
    x = _require_cuda_f32("attr_matrix", x)
    dev = x.device
    B, T, S, F_in = _attr_shape(x)
    (adj,) = _graph(adj, S, dev)
    params = _params(params, dev)
    F_hid, F_out, H = _param_dims(S, F_in, params)
    out = _require_cuda_f32("out", out, dev)
    d_out = _require_cuda_f32("d_out", d_out, dev)
    if out.shape != (B, T, H) or d_out.shape != (B, T, H):
        raise RuntimeError(f"out / d_out must be [{B}, {T}, {H}]")
    grads = _grads_bucket(lib, (S, F_in, F_hid, F_out, H), dev, grads)
    w1, b1, w2, b2, w_ih, w_hh, _, _ = params
    _lib.check(lib.wg_gcn_gru_backward_f32(
        adj.data_ptr(), x.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(),
        w_ih.data_ptr(), w_hh.data_ptr(), out.data_ptr(), d_out.data_ptr(), grads.data_ptr(),
        B, T, S, F_in, F_hid, F_out, H, ws.data_ptr(), ws.numel(), dev.index or 0, _stream(dev)))
    return grads


def _table_args(adj, table, params):
    """The checked table, ``(adj,)``, parameters and dims ``(S, F_in, F_hid, F_out, H)`` of a table-window call."""
    table = _require_cuda_f32("table", table)
    dev = table.device
    _, S, F_in = _table_shape(table)
    (adj,) = _graph(adj, S, dev)
    params = _params(params, dev)
    return table, adj, params, (S, F_in, *_param_dims(S, F_in, params))


def forward_train_windows(adj, table, starts, params: Sequence[torch.Tensor], seq_length: int):
    """``forward_train`` of the windows ``table[starts[n] : starts[n] + seq_length]`` of ``table [Ttot, S, F_in]``
    without materialising them: GCN and input projection run once per table row the windows cover.  ``starts``:
    int64 first rows (any order, repeats allowed; read from the host).  Returns ``(out [N, L, H], workspace)``."""
    lib = _lib.load()
    table, adj, params, dims = _table_args(adj, table, params)
    starts = _forecast_starts(starts)
    N, Ttot, dev = starts.numel(), table.shape[0], table.device
    out = torch.empty((N, max(seq_length, 0), dims[-1]), dtype=torch.float32, device=dev)
    # 0 bytes: the shape is rejected, and the call below returns the library's code and reason without launching
    nbytes = lib.wg_gcn_gru_train_windows_workspace_bytes(N, Ttot, seq_length, *dims)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    _lib.check(lib.wg_gcn_gru_forward_train_windows_f32(
        adj.data_ptr(), table.data_ptr(), starts.data_ptr(), *(p.data_ptr() for p in params), out.data_ptr(),
        N, Ttot, seq_length, *dims, ws.data_ptr(), ws.numel(), dev.index or 0, _stream(dev)))
    return out, ws


def backward_windows(adj, table, starts, params: Sequence[torch.Tensor], out, d_out, ws, seq_length: int,
                     grads: Optional[torch.Tensor] = None):
    """``backward`` after ``forward_train_windows`` (the same ``starts`` and workspace): the flat gradient bucket.
    The input-gate gradients are summed per table row, and dW_ih, dU and the GCN backward run once per row."""
    lib = _lib.load()
    table, adj, params, dims = _table_args(adj, table, params)
    starts = _forecast_starts(starts)
    N, Ttot, dev, H = starts.numel(), table.shape[0], table.device, dims[-1]
    out = _require_cuda_f32("out", out, dev)
    d_out = _require_cuda_f32("d_out", d_out, dev)
    if out.shape != (N, seq_length, H) or d_out.shape != (N, seq_length, H):
        raise RuntimeError(f"out / d_out must be [{N}, {seq_length}, {H}]")
    grads = _grads_bucket(lib, dims, dev, grads)
    w1, b1, w2, b2, w_ih, w_hh, _, _ = params
    _lib.check(lib.wg_gcn_gru_backward_windows_f32(
        adj.data_ptr(), table.data_ptr(), starts.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(),
        b2.data_ptr(), w_ih.data_ptr(), w_hh.data_ptr(), out.data_ptr(), d_out.data_ptr(), grads.data_ptr(),
        N, Ttot, seq_length, *dims, ws.data_ptr(), ws.numel(), dev.index or 0, _stream(dev)))
    return grads


def split_flat(flat: torch.Tensor, shapes):
    """Views of a flat buffer, one per shape, in order."""
    views, o = [], 0
    for shp in shapes:
        n = 1
        for d in shp:
            n *= d
        views.append(flat[o:o + n].view(shp))
        o += n
    if o != flat.numel():
        raise RuntimeError(f"flat buffer has {flat.numel()} elements, shapes need {o}")
    return views


class GcnGruWindowsFunction(torch.autograd.Function):
    """autograd bridge of the table windows: ``forward_train_windows`` + ``backward_windows``."""

    @staticmethod
    def forward(ctx, adj, table, starts, seq_length, *params):
        out, ws = forward_train_windows(adj, table, starts, [p.detach() for p in params], seq_length)
        ctx.save_for_backward(adj, table, *params, out)
        ctx.starts, ctx.seq_length, ctx.ws = starts, seq_length, ws
        return out

    @staticmethod
    def backward(ctx, d_out):
        adj, table, *rest = ctx.saved_tensors
        params, out = rest[:8], rest[8]
        flat = backward_windows(adj, table, ctx.starts, [p.detach() for p in params], out, d_out.contiguous(),
                                ctx.ws, ctx.seq_length)
        ctx.ws = None
        grads = split_flat(flat, [p.shape for p in params])
        return (None, None, None, None, *grads)


class GcnGruFunction(torch.autograd.Function):
    """autograd bridge: library forward (saving gates) + library backward."""

    @staticmethod
    def forward(ctx, adj, x, *params):
        out, ws = forward_train(adj, x, [p.detach() for p in params])
        ctx.save_for_backward(adj, x, *params, out)
        ctx.ws = ws
        return out

    @staticmethod
    def backward(ctx, d_out):
        adj, x, *rest = ctx.saved_tensors
        params, out = rest[:8], rest[8]
        flat = backward(adj, x, [p.detach() for p in params], out, d_out.contiguous(), ctx.ws)
        ctx.ws = None
        grads = split_flat(flat, [p.shape for p in params])
        return (None, None, *grads)


def mse_loss_grad(out: torch.Tensor, y: torch.Tensor, want_grad: bool = True):
    """``(loss, d_out)``: mean squared error over all elements (``nn.MSELoss()``, main.py:49) as a
    device scalar and ``2 (out - y) / n``."""
    lib = _lib.load()
    out = _require_cuda_f32("out", out)
    y = _require_cuda_f32("y", y, out.device)
    if y.numel() != out.numel():
        raise RuntimeError(f"target has {y.numel()} elements, output {out.numel()}")
    dev = out.device
    d_out = torch.empty_like(out) if want_grad else None
    loss = torch.empty((), dtype=torch.float32, device=dev)
    ws = torch.empty(lib.wg_mse_workspace_bytes(), dtype=torch.uint8, device=dev)
    _lib.check(lib.wg_mse_loss_grad_f32(out.data_ptr(), y.data_ptr(), out.numel(),
                                        d_out.data_ptr() if want_grad else None, loss.data_ptr(), ws.data_ptr(),
                                        ws.numel(), dev.index or 0, _stream(dev)))
    return loss, d_out


def mse_window_labels(out: torch.Tensor, table: torch.Tensor, starts, seq_length: int, label_feature: int = 11,
                      horizons: int = 3, want_grad: bool = True):
    """``mse_loss_grad`` of ``out [N, L, horizons * S]`` against the targets of the windows ``table[starts[n] :
    starts[n] + L]``, read from the table in place: ``y[n, l, k*S + s] = table[starts[n] + l + 1 + k, s,
    label_feature]``, what ``create_sequences`` builds for ``starts[n] = n L``.  The same loss bit for bit."""
    lib = _lib.load()
    out = _require_cuda_f32("out", out)
    dev = out.device
    table = _require_cuda_f32("table", table, dev)
    Ttot, S, F = _table_shape(table)
    starts = _forecast_starts(starts)
    N = starts.numel()
    if out.shape != (N, seq_length, horizons * S):
        raise RuntimeError(f"out must be [{N}, {seq_length}, {horizons * S}], got {tuple(out.shape)}")
    d_out = torch.empty_like(out) if want_grad else None
    loss = torch.empty((), dtype=torch.float32, device=dev)
    ws = torch.empty(max(lib.wg_mse_window_labels_workspace_bytes(N), 1), dtype=torch.uint8, device=dev)
    _lib.check(lib.wg_mse_window_labels_f32(out.data_ptr(), table.data_ptr(), starts.data_ptr(), N, seq_length, Ttot,
                                            S, F, label_feature, horizons, d_out.data_ptr() if want_grad else None,
                                            loss.data_ptr(), ws.data_ptr(), ws.numel(), dev.index or 0, _stream(dev)))
    return loss, d_out


def allreduce_mean_(flat: torch.Tensor, group=None) -> float:
    """Sum all-reduce of the flat gradient bucket across the data-parallel ranks, in place.  Returns
    the factor the optimiser must still apply (``1 / world``; the mean is folded into the Adam
    kernel).  Identity (factor 1) without an initialised process group."""
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()):
        return 1.0
    world = dist.get_world_size(group)
    if world == 1:
        return 1.0
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    return 1.0 / world


def shard_weight(local_batch: int, global_batch: int, group=None) -> float:
    """Weight of a rank's local-mean gradient in the average over ranks that reproduces the global mean:
    ``local_batch * world / global_batch`` (1 for equal shards or a single process)."""
    import torch.distributed as dist

    world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
    if global_batch <= 0:
        raise ValueError("global_batch must be positive")
    return float(local_batch) * world / float(global_batch)


class Trainer:
    """Fused data-parallel training step for a ``windgnn_b200.GCN_GRU`` on one GPU per process.

    The eight parameters are re-pointed at views of ONE flat buffer (state_dict order, keys and
    shapes unchanged, so ``state_dict()`` / ``load_state_dict()`` / ``torch.save`` keep working as
    in main.py:84,99); Adam's moments are flat buffers of the same size.
    """

    def __init__(self, model, adj: torch.Tensor, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8,
                 group=None):
        self.model = model
        self.adj = _require_cuda_f32("adj_matrix", adj)
        self.lr, self.betas, self.eps, self.group = float(lr), (float(betas[0]), float(betas[1])), float(eps), group
        self.step_count = 0
        self.params = list(model._params())
        dev = self.adj.device
        _params(self.params, dev)
        shapes = [tuple(p.shape) for p in self.params]
        n = sum(p.numel() for p in self.params)
        self.flat = torch.empty(n, dtype=torch.float32, device=dev)
        with torch.no_grad():
            for view, p in zip(split_flat(self.flat, shapes), self.params):
                view.copy_(p)
                p.data = view
        self.grads = torch.zeros_like(self.flat)
        self.exp_avg = torch.zeros_like(self.flat)
        self.exp_avg_sq = torch.zeros_like(self.flat)

    @torch.no_grad()
    def step(self, x: torch.Tensor, y: torch.Tensor, global_batch: Optional[int] = None) -> torch.Tensor:
        """One optimisation step on this rank's shard ``x [B,T,S,F]``, ``y [B,T,H]``.  Returns the
        local loss (device scalar; no host synchronisation).

        The ranks' gradients of their LOCAL mean losses are averaged, which is the gradient of the global
        mean-squared error when every rank holds the same number of windows.  For uneven shards pass
        ``global_batch`` (the number of windows over all ranks): this rank's upstream gradient is then
        weighted by ``B_local * world / global_batch`` so that the average is the global gradient."""
        ps = [p.data for p in self.params]
        out, ws = forward_train(self.adj, x, ps)
        loss, d_out = mse_loss_grad(out, y)
        if global_batch is not None:
            w = shard_weight(x.shape[0], global_batch, self.group)
            if w != 1.0:
                d_out.mul_(w)
        backward(self.adj, x, ps, out, d_out, ws, self.grads)
        self._update()
        return loss

    @torch.no_grad()
    def step_table(self, table: torch.Tensor, starts, seq_length: int = 168, label_feature: int = 11,
                   horizons: int = 3, global_batch: Optional[int] = None) -> torch.Tensor:
        """``step`` on this rank's windows ``table[starts[n] : starts[n] + seq_length]`` of ``table [Ttot, S, F]``,
        without materialising them: the targets are ``create_sequences``' (``label_feature`` ``1 .. horizons``
        rows after each step), read from the table, and GCN, input projection and their gradients run once per
        table row the windows cover.  The model's ``H`` must be ``horizons * S``.  Same all-reduce, ``global_batch``
        weighting and Adam update as ``step``; for ``starts[n] = n seq_length`` the same result bit for bit."""
        ps = [p.data for p in self.params]
        S, H = _table_shape(table)[1], ps[5].shape[1]
        if H != horizons * S:
            raise RuntimeError(f"step_table: the model's H = {H} is not horizons * S = {horizons} * {S}")
        starts = _forecast_starts(starts)
        out, ws = forward_train_windows(self.adj, table, starts, ps, seq_length)
        loss, d_out = mse_window_labels(out, table, starts, seq_length, label_feature, horizons)
        if global_batch is not None:
            w = shard_weight(starts.numel(), global_batch, self.group)
            if w != 1.0:
                d_out.mul_(w)
        backward_windows(self.adj, table, starts, ps, out, d_out, ws, seq_length, self.grads)
        self._update()
        return loss

    def _update(self) -> None:
        """All-reduce of the gradient bucket, then one Adam step over the flat parameters."""
        lib = _lib.load()
        dev = self.flat.device
        scale = allreduce_mean_(self.grads, self.group)
        self.step_count += 1
        _lib.check(lib.wg_adam_step_f32(
            self.flat.data_ptr(), self.grads.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(),
            self.flat.numel(), self.lr, self.betas[0], self.betas[1], self.eps, self.step_count, scale,
            dev.index or 0, _stream(dev)))
