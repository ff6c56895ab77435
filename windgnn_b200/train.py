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

PyTorch is plumbing here (device memory, streams, ``torch.distributed``); every arithmetic step is a
kernel of ``libwindgnn_b200.so``.  CUDA only — no CPU fallback.
"""

from __future__ import annotations

from typing import Optional, Sequence

import torch

from . import _lib
from .ops import _dims, _require_cuda_f32

PARAM_NAMES = (
    "conv1.weight", "conv1.bias", "conv2.weight", "conv2.bias",
    "gru.weight_ih_l0", "gru.weight_hh_l0", "gru.bias_ih_l0", "gru.bias_hh_l0",
)


def _stream(dev: torch.device) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def forward_train(adj, x, params: Sequence[torch.Tensor]):
    """Forward that keeps what the backward needs.  Returns ``(out [B,T,H], workspace)``."""
    lib = _lib.load()
    x = _require_cuda_f32("attr_matrix", x)
    dev = x.device
    adj = _require_cuda_f32("adj_matrix", adj, dev)
    params = [_require_cuda_f32(n, p, dev) for n, p in zip(PARAM_NAMES, params)]
    B, T, S, F_in, F_hid, F_out, H = _dims(adj, x, *params)
    out = torch.empty((B, T, H), dtype=torch.float32, device=dev)
    # 0 bytes: the shape is rejected, and the call below returns the library's code and reason without launching
    nbytes = lib.wg_gcn_gru_train_workspace_bytes(B, T, S, F_in, F_hid, F_out, H)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    _lib.check(lib.wg_gcn_gru_forward_train_f32(
        adj.data_ptr(), x.data_ptr(), *(p.data_ptr() for p in params), out.data_ptr(),
        B, T, S, F_in, F_hid, F_out, H, ws.data_ptr(), ws.numel(), dev.index or 0, _stream(dev)))
    return out, ws


def backward(adj, x, params: Sequence[torch.Tensor], out, d_out, ws, grads: Optional[torch.Tensor] = None):
    """Flat gradient bucket (state_dict order) of the loss w.r.t. the eight parameter tensors."""
    lib = _lib.load()
    x = _require_cuda_f32("attr_matrix", x)
    dev = x.device
    adj = _require_cuda_f32("adj_matrix", adj, dev)
    params = [_require_cuda_f32(n, p, dev) for n, p in zip(PARAM_NAMES, params)]
    out = _require_cuda_f32("out", out, dev)
    d_out = _require_cuda_f32("d_out", d_out, dev)
    B, T, S, F_in, F_hid, F_out, H = _dims(adj, x, *params)
    if out.shape != (B, T, H) or d_out.shape != (B, T, H):
        raise RuntimeError(f"out / d_out must be [{B}, {T}, {H}]")
    n = lib.wg_gcn_gru_param_count(S, F_in, F_hid, F_out, H)
    if grads is None:
        grads = torch.empty(n, dtype=torch.float32, device=dev)
    elif grads.numel() != n or not grads.is_cuda or grads.dtype != torch.float32 or not grads.is_contiguous():
        raise RuntimeError(f"grads must be a contiguous CUDA float32 buffer of {n} elements")
    w1, b1, w2, b2, w_ih, w_hh, _, _ = params
    _lib.check(lib.wg_gcn_gru_backward_f32(
        adj.data_ptr(), x.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(),
        w_ih.data_ptr(), w_hh.data_ptr(), out.data_ptr(), d_out.data_ptr(), grads.data_ptr(),
        B, T, S, F_in, F_hid, F_out, H, ws.data_ptr(), ws.numel(), dev.index or 0, _stream(dev)))
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
        self.params = [
            model.conv1.weight, model.conv1.bias, model.conv2.weight, model.conv2.bias,
            model.gru.weight_ih_l0, model.gru.weight_hh_l0, model.gru.bias_ih_l0, model.gru.bias_hh_l0,
        ]
        dev = self.adj.device
        for n, p in zip(PARAM_NAMES, self.params):
            _require_cuda_f32(n, p, dev)
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
        lib = _lib.load()
        dev = self.flat.device
        ps = [p.data for p in self.params]
        out, ws = forward_train(self.adj, x, ps)
        loss, d_out = mse_loss_grad(out, y)
        if global_batch is not None:
            w = shard_weight(x.shape[0], global_batch, self.group)
            if w != 1.0:
                d_out.mul_(w)
        backward(self.adj, x, ps, out, d_out, ws, self.grads)
        scale = allreduce_mean_(self.grads, self.group)
        self.step_count += 1
        _lib.check(lib.wg_adam_step_f32(
            self.flat.data_ptr(), self.grads.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(),
            self.flat.numel(), self.lr, self.betas[0], self.betas[1], self.eps, self.step_count, scale,
            dev.index or 0, _stream(dev)))
        return loss
