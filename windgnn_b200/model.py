"""Drop-in ``nn.Module`` mirrors of the reference model classes.

Same constructor signatures, same parameter names (so the shipped ``wind_gnn_7.pth`` /
``wind_gnn_34.pth`` state_dicts load with ``strict=True``), same ``forward(adj_matrix,
attr_matrix)`` — but ``forward`` runs the fused sm_100a path through the C-ABI library.

Reference: ``GraphConvLayer`` src/step5_gcn_layer_model.py:5-23,
           ``GCN_GRU``        src/step6_gcn_gru_combined_model.py:6-27.
"""

from __future__ import annotations

import torch
import torch.nn as nn

from . import ops
from .graph import CsrGraph


class _InferenceOnly(torch.autograd.Function):
    """Forward of a path that has no backward in the library: the result still takes part in autograd (so a
    forward under grad mode behaves like the reference's), and backward() raises with the reason."""

    @staticmethod
    def forward(ctx, message, fn, *params):
        ctx.message = message
        return fn()

    @staticmethod
    def backward(ctx, *grads):
        raise RuntimeError(ctx.message)


class GraphConvLayer(nn.Module):
    """``relu((adj @ attr) @ weight + bias)`` — step5:13-23.  Init as step5:8-10."""

    def __init__(self, input_dim, output_dim):
        super().__init__()
        self.weight = nn.Parameter(torch.randn(input_dim, output_dim))
        self.bias = nn.Parameter(torch.zeros(output_dim))

    def forward(self, adj_matrix, attr_matrix):
        if torch.is_grad_enabled() and any(
                t.requires_grad for t in (self.weight, self.bias, attr_matrix, adj_matrix)):
            # the stand-alone layer op has no backward (training goes through GCN_GRU, train.py): the forward
            # still works under grad mode, and a later backward() says why it cannot
            return _InferenceOnly.apply(
                "windgnn_b200.GraphConvLayer has no autograd formula: train through windgnn_b200.GCN_GRU, whose "
                "forward records the library backward, or call the layer under torch.no_grad()",
                lambda: ops.gcn_layer(adj_matrix.detach(), attr_matrix.detach(), self.weight.detach(),
                                      self.bias.detach()),
                self.weight, self.bias)
        return ops.gcn_layer(adj_matrix, attr_matrix, self.weight, self.bias)


class GCN_GRU(nn.Module):
    """conv1 -> conv2 -> flatten -> GRU, every hidden state returned (step6:13-27).

    ``attr_matrix`` is ``[B, T, S, F_in]``.  The reference accepts ``B == 1`` only and
    returns ``[T, H]`` (``squeeze(0)``, step6:26); that is reproduced, and ``B > 1`` returns
    ``[B, T, H]`` (sequences are independent, ``h0 = 0`` each).

    ``self.gru`` is a real ``nn.GRU`` used purely as the parameter container so that the
    state_dict keys (``gru.weight_ih_l0`` ...) match the reference's.
    """

    DENSE_MAX_STATIONS = 128  # above this the adjacency is handed to the library as CSR

    def __init__(self, input_dim, hidden_dim, output_dim, gru_input, gru_hidden_dim):
        super().__init__()
        self.conv1 = GraphConvLayer(input_dim, hidden_dim)
        self.conv2 = GraphConvLayer(hidden_dim, output_dim)
        self.gru = nn.GRU(gru_input, gru_hidden_dim, batch_first=True)
        self.chunk = 0  # sequences per internal pass; 0 = library default
        # "fp32": every contraction as FP32 FMA.  "tensor": the GRU input projection and the recurrent product
        # on the tcgen05 tensor cores with error-compensated fp16 split operands (same 1e-5 parity bar, see
        # inproj_tc2.cuh / recur_tc.cuh)
        self.precision = "fp32"
        self._csr_cache = None  # (key, (rowptr, colidx, vals)) of the last large adjacency seen

    def forward(self, adj_matrix, attr_matrix):
        if attr_matrix.dim() != 4:
            # the reference raises RuntimeError from view() for anything but [1, T, S, F] (step6:20)
            raise RuntimeError(
                f"attr_matrix must be [B, T, S, F_in], got {tuple(attr_matrix.shape)}"
            )
        params = (
            self.conv1.weight, self.conv1.bias, self.conv2.weight, self.conv2.bias,
            self.gru.weight_ih_l0, self.gru.weight_hh_l0, self.gru.bias_ih_l0, self.gru.bias_hh_l0,
        )
        widths = (self.conv1.weight.shape[0], self.conv1.weight.shape[1], self.conv2.weight.shape[1])
        needs_grad = torch.is_grad_enabled() and any(p.requires_grad for p in params)
        is_csr = isinstance(adj_matrix, CsrGraph)
        if torch.is_grad_enabled() and (attr_matrix.requires_grad or (not is_csr and adj_matrix.requires_grad)):
            # the reference never differentiates w.r.t. its data (main.py:66-77); the library has no such gradient
            raise RuntimeError("windgnn_b200.GCN_GRU: gradients w.r.t. attr_matrix / adj_matrix are not implemented")
        csr = self._csr_of(adj_matrix)
        if csr is not None:
            if needs_grad:
                # forward works under grad mode (main.py:66 style calls); backward() explains the limit
                out = _InferenceOnly.apply(
                    "windgnn_b200.GCN_GRU: training is implemented for dense graphs with at most "
                    f"{self.DENSE_MAX_STATIONS} stations and GCN widths <= 16 (got {adj_matrix.shape[0]} stations, "
                    f"widths {widths}); the scaled shapes are inference-only",
                    lambda: ops.gcn_gru_forward_csr(*csr, attr_matrix, *[p.detach() for p in params], self.chunk,
                                                    self._flags()),
                    *params)
            else:
                out = ops.gcn_gru_forward_csr(*csr, attr_matrix, *params, self.chunk, self._flags())
        elif needs_grad:
            # training (main.py:66 runs with grad enabled): forward that saves the gate values, library
            # backward (train.py); FP32 path only
            from .train import GcnGruFunction

            out = GcnGruFunction.apply(adj_matrix, attr_matrix, *params)
        else:
            out = ops.gcn_gru_forward(adj_matrix, attr_matrix, *params, self.chunk, self._flags())
        return out.squeeze(0)  # step6:26 — a no-op unless B == 1

    @torch.no_grad()
    def forward_host(self, adj_matrix, attr_host, out_host=None, last_step_range=None):
        """Host-buffer end-to-end forward (H2D, compute, D2H overlapped chunk by chunk).  With
        ``last_step_range=(wind_min, wind_max)`` only the de-normalised last timestep ``[B, 3S]`` comes back
        (the evaluation of main.py:101-116 in one call)."""
        params = (
            self.conv1.weight, self.conv1.bias, self.conv2.weight, self.conv2.bias,
            self.gru.weight_ih_l0, self.gru.weight_hh_l0, self.gru.bias_ih_l0, self.gru.bias_hh_l0,
        )
        return ops.gcn_gru_forward_host(adj_matrix, attr_host, [p.detach() for p in params], out_host, self.chunk,
                                        flags=self._flags(), last_step_range=last_step_range)

    @torch.no_grad()
    def forecast(self, adj_matrix, table, starts=None, seq_length=168, stride=1, last_step_range=None):
        """Rolling forecasts from one table: the last hidden state ``[N, H]`` of every window
        ``table[starts[n] : starts[n] + seq_length]`` of ``table [Ttot, S, F_in]`` (on the GPU), without
        materialising the windows: GCN and input projection run once per table row.  Row ``n`` is bit-identical to
        ``self(adj_matrix, window_n)[-1]`` under ``torch.no_grad()``.

        ``starts``: int64 first rows (any order, repeats allowed); ``None`` = every ``stride``-th window,
        ``window_starts(Ttot, seq_length, stride)``.  Same adjacency forms, routing, ``precision`` and ``chunk`` as
        ``forward``.  ``last_step_range=(wind_min, wind_max)``: de-normalised as ``denormalise_last_step`` does
        (src/main.py:103,116)."""
        from .sequences import denormalise_last_step, window_starts

        if starts is None:
            starts = window_starts(table.shape[0], seq_length, stride)
        params = [p.detach() for p in (
            self.conv1.weight, self.conv1.bias, self.conv2.weight, self.conv2.bias,
            self.gru.weight_ih_l0, self.gru.weight_hh_l0, self.gru.bias_ih_l0, self.gru.bias_hh_l0,
        )]
        csr = self._csr_of(adj_matrix)
        if csr is not None:
            out = ops.gcn_gru_forecast_csr(*csr, table, starts, *params, seq_length, self.chunk, self._flags())
        else:
            out = ops.gcn_gru_forecast(adj_matrix, table, starts, *params, seq_length, self.chunk, self._flags())
        if last_step_range is not None:
            out = denormalise_last_step(out.unsqueeze(1), *last_step_range)
        return out

    def _csr_of(self, adj_matrix):
        """The CSR arrays the library takes for ``adj_matrix``, or ``None`` for the dense path: a ``CsrGraph``, more
        than DENSE_MAX_STATIONS stations or GCN widths above 16 (the scaled shapes) go to CSR, a dense matrix
        through a cached conversion."""
        widths = (self.conv1.weight.shape[0], self.conv1.weight.shape[1], self.conv2.weight.shape[1])
        if isinstance(adj_matrix, CsrGraph):
            return (adj_matrix.rowptr, adj_matrix.colidx, adj_matrix.vals)
        if adj_matrix.shape[0] <= self.DENSE_MAX_STATIONS and max(widths) <= 16:
            return None
        key = (adj_matrix.data_ptr(), adj_matrix._version, tuple(adj_matrix.shape))
        if self._csr_cache is None or self._csr_cache[0] != key:
            self._csr_cache = (key, ops.dense_to_csr(adj_matrix))
        return self._csr_cache[1]

    def _flags(self) -> int:
        from . import _lib

        if self.precision == "fp32":
            return 0
        if self.precision in ("tensor", "tf32x3"):   # "tf32x3": the round-1 name of the tensor path
            return _lib.FLAG_TENSOR_CORES
        raise ValueError(f"precision must be 'fp32' or 'tensor', got {self.precision!r}")
